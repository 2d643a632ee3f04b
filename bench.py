#!/usr/bin/env python
"""Benchmark of the wav2sleep forward hot path on B200 (BASELINE.json metric: recording-hours/sec, forward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]              # reference algorithm on host CPU cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N   # N > 1, one rank per GPU

Workload (config.workload): BASELINE.json configs[2] - cardio model (ABD, THX, ECG, PPG; 4 classes), batch of
16 synthetic 10-hour nights per GPU (S = 1200 epochs; ECG/PPG 1 228 800 samples, ABD/THX 307 200 samples per
night, N(0,1) fp32), random-init weights.  Recordings are independent, so N GPUs = N replicas on disjoint shards
with no data-path collective ("scaling": "weak").

One "step" = one forward pass (signal encoders -> epoch mixer -> sequence mixer -> classifier -> argmax) over one
batch, through ``Wav2Sleep.predict_async`` (the forward runs on streams owned by the engine; results are awaited in
order).  `value` times K steps with inputs resident in HBM (CUDA events, barrier + synchronize on both sides, max
over ranks).  `e2e` times the same K steps with HOST (pinned) inputs: every step copies its 196.6 MB of inputs
host->device (copy stream, two batches ahead) and reads the int64 predictions back, all inside the timed region.
Inputs (196.6 MB/step) and activations (GBs) exceed the 126 MB L2, so no explicit L2 flush is needed
("l2": "inputs+activations > L2").

Secondary objects on the same JSON line, each with its own clock samples:
  train           BASELINE configs[3]: cardio training step (polarity flip + config masker + forward + CE + loss-scaled
                  backward + bucketed all-reduce + fused clip/AdamW), 16 nights per GPU; per-rank times and, for N > 1,
                  the same step with identical masks on every rank (mask stragglers vs communication)
  train_ecg_only  BASELINE configs[4]: the same step at batch 32 with PPG / ABD / THX missing for every night
  eog             BASELINE configs[1]: EOG model, 16 x 14-h nights, 1 GPU (N = 1 only)
  e2e_staged      the e2e loop with int16 transport + on-device z-score (SURVEY 8f N1)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CARDIO = {"ABD": "ABD", "THX": "THX", "ECG": "ECG", "PPG": "PPG"}
SPE = {"ABD": 256, "THX": 256, "ECG": 1024, "PPG": 1024}
S_EPOCHS = 1200          # 10-hour night
HOURS_PER_NIGHT = 10.0
BATCH = 16               # nights per GPU per step
METRIC = "recording-hours/sec fwd"
UNIT = "recording-hours/s"
WORKLOAD = "cardio 4-signal (ABD,THX,ECG,PPG) 4-class inference, 16 synthetic 10-h nights per GPU (BASELINE configs[2])"


def make_night_batch(B, seed, pin=False):
    g = torch.Generator().manual_seed(seed)
    x = {}
    for name in CARDIO:
        t = torch.randn(B, S_EPOCHS * SPE[name], generator=g)
        x[name] = t.pin_memory() if pin else t
    return x


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))), "measured"
    return 6650.0, 1400.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([f.strip() for f in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.02)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = max((int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(self.samples)}


def cpu_reference_time(steps, warmup, nights_per_step=1):
    """The reference algorithm (oracle port, same torch CPU kernels as the reference) on the host cores."""
    from oracle import wav2sleep_oracle as oracle
    from wav2sleep_b200 import build_default
    torch.set_num_threads(os.cpu_count() or 1)
    model = build_default(CARDIO, 4, seed=0)
    sd = model.state_dict()
    cfg = oracle.cardio_config()
    x = make_night_batch(nights_per_step, seed=42)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        oracle.forward(x, sd, cfg).argmax(-1)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    times.sort()
    med = times[len(times) // 2]
    return {"value": nights_per_step * HOURS_PER_NIGHT / med, "unit": UNIT, "cores": torch.get_num_threads(),
            "kind": "port", "s_per_step": med,
            "sample": f"{nights_per_step} night(s) of the workload per step (B={nights_per_step}, S={S_EPOCHS}), "
                      f"fp32 torch CPU, median of {steps} after {warmup} warm-up"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_time(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["s_per_step"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "nights_per_step": 1, "epochs_per_night": S_EPOCHS},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the tensors the timed path handed back in its last step, as <out_dir>/<name>.npy (float32), so
    that two builds run with the same arguments (hence the same seeded inputs) can be compared output for output."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        np.save(d / f"{name}.npy", t.detach().to("cpu", torch.float32).numpy())


def collect_profile(lib):
    n = lib.w2s_profile_count()
    recs = []
    buf = C.create_string_buffer(128)
    ms, by, fl = C.c_float(), C.c_double(), C.c_double()
    for i in range(n):
        if lib.w2s_profile_get(i, buf, 128, C.byref(ms), C.byref(by), C.byref(fl)) == 0:
            recs.append((buf.value.decode(), ms.value, by.value, fl.value))
    return recs


def run_cuda(args):
    import torch.distributed as dist
    from wav2sleep_b200 import _lib, build_default

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run --nproc-per-node N")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # Multi-rank runs: every rank stages its pinned host batches on the NUMA node of its own GPU (placement only; the
    # single-GPU run keeps all host cores for its cpu_baseline leg).
    host_cpus = 0
    if world > 1:
        from wav2sleep_b200 import hostmem
        host_cpus = hostmem.bind_to_gpu_numa(local_rank)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator is created: route fd 1 to stderr while that
        # happens so that stdout carries exactly one JSON line.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.load()
    hbm_peak, tf_peak, peak_src = measured_peaks()

    model = build_default(CARDIO, 4, seed=0).to(dev).eval()
    # two distinct host batches (pinned) so that consecutive steps never reuse data
    host = [make_night_batch(BATCH, seed=42 + rank * 2 + i, pin=True) for i in range(2)]
    devb = [{k: v.to(dev, non_blocking=True) for k, v in h.items()} for h in host]
    h2d_bytes = sum(v.numel() * 4 for v in host[0].values())
    d2h_bytes = BATCH * S_EPOCHS * 8
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def run_steps(n, batches):
        """n forward steps through the public throughput API (Wav2Sleep.predict_async: the forward runs on the engine's
        own streams and the caller awaits results in order, up to two outstanding; every step does all of its work and
        the last results are awaited before returning)."""
        pend, out = [], None
        for i in range(n):
            pend.append(model.predict_async(batches[i % 2]))
            if len(pend) > 2:
                out = pend.pop(0).wait()
        for q in pend:
            out = q.wait()
        return out

    # ---------------- device-resident timing ----------------
    with torch.inference_mode():
        run_steps(args.warmup, devb)
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        l0 = lib.w2s_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pred = run_steps(args.steps, devb)
        e1.record()
        barrier()
        launches = lib.w2s_launch_count() - l0 + model._get_engine().replayed_launches
        ms_dev = max_over_ranks(e0.elapsed_time(e1))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"predictions" if world == 1 else f"predictions_rank{rank}": pred})

        # ---------------- end-to-end timing: pinned host inputs -> predictions on host ----------------
        copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream()
        NS = 3  # staging buffers: uploads run two batches ahead of the forward that is starting
        stage = [{k: torch.empty_like(v) for k, v in devb[0].items()} for _ in range(NS)]
        out_host = [torch.empty(BATCH, S_EPOCHS, dtype=torch.int64).pin_memory() for _ in range(NS)]
        ready = [torch.cuda.Event() for _ in range(NS)]
        sig_ready = [{k: torch.cuda.Event() for k in devb[0]} for _ in range(NS)]  # per signal: its copy has landed
        free = [None] * NS  # event after which staging buffer b may be overwritten

        def pipelined(n, upload_one, make_inputs, per_signal=False):
            """Every step: H2D copy of its inputs (copy stream, pinned source) -> forward (predict_async, two in
            flight) -> D2H copy of its predictions; all inside the caller's timed region.  per_signal: every signal's
            encoder waits for its own copy only (largest signals are uploaded first), instead of the whole batch."""
            for b in range(NS):
                free[b] = None

            def upload(i):
                with torch.cuda.stream(copy_stream):
                    if free[i % NS] is not None:
                        copy_stream.wait_event(free[i % NS])
                    upload_one(i)
                    ready[i % NS].record(copy_stream)

            for i in range(min(2, n)):
                upload(i)
            pend = []
            for i in range(n):
                if not per_signal:
                    main.wait_event(ready[i % NS])
                x, released = make_inputs(i)
                p = model.predict_async(x, ready=sig_ready[i % NS] if per_signal else None)
                free[i % NS] = released if released is not None else p.done
                pend.append((p, i, x))
                if i + 2 < n:
                    upload(i + 2)
                if len(pend) > 1:  # the previous batch's predictions go back to the host while this batch runs
                    q, j, _ = pend.pop(0)
                    out_host[j % NS].copy_(q.wait(), non_blocking=True)
            for q, j, _ in pend:
                out_host[j % NS].copy_(q.wait(), non_blocking=True)
            torch.cuda.synchronize()

        def upload_f32(i):
            for k in sorted(stage[i % NS], key=lambda k: -stage[i % NS][k].numel()):  # longest encoder chains first
                stage[i % NS][k].copy_(host[i % 2][k], non_blocking=True)
                sig_ready[i % NS][k].record(copy_stream)

        def e2e_loop(n):
            pipelined(n, upload_f32, lambda i: (stage[i % NS], None), per_signal=True)

        e2e_loop(min(args.warmup, 3))
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        e2e_loop(args.steps)
        t1.record()
        barrier()
        ms_e2e = max_over_ranks(t0.elapsed_time(t1))
        sampler.stop_flag.set()
        sampler.join(timeout=3)

        # ---------------- same loop with int16 transport + on-device z-score (SURVEY 8f N1, secondary number) ----------
        from wav2sleep_b200.staging import zscore_on_device
        host16 = [{k: (v * 1000.0).round().clamp(-32000, 32000).to(torch.int16).pin_memory() for k, v in hb.items()}
                  for hb in host]
        stage16 = [{k: torch.empty(v.shape, dtype=torch.int16, device=dev) for k, v in host16[0].items()} for _ in range(NS)]

        def upload_i16(i):
            for k in stage16[i % NS]:
                stage16[i % NS][k].copy_(host16[i % 2][k], non_blocking=True)

        def zscored(i):
            # normalised inputs go into the (now unused) fp32 staging buffers: no allocation in the loop
            x = {k: zscore_on_device(v, out=stage[i % NS][k]) for k, v in stage16[i % NS].items()}
            ev = torch.cuda.Event()
            ev.record(main)  # the int16 buffer is free again once the z-score has read it
            return x, ev

        def staged_loop(n):
            pipelined(n, upload_i16, zscored)

        staged_loop(3)
        barrier()
        t0.record()
        staged_loop(args.steps)
        t1.record()
        barrier()
        ms_staged = max_over_ranks(t0.elapsed_time(t1))

        # ---------------- per-kernel profile (CUDA events around every launch, 2 extra steps) ----------------
        prof = []
        if rank == 0:
            eng = model._get_engine()
            # isolated per-kernel durations of exactly the launches of a timed step (paired encoder launches included):
            # the encoder streams run one after the other
            eng.serial_groups = True
            model.predict(devb[0])
            lib.w2s_profile_enable(1)
            for i in range(2):
                model.predict(devb[i % 2])
            torch.cuda.synchronize()
            prof = collect_profile(lib)
            lib.w2s_profile_enable(0)
            eng.serial_groups = False
            eng._release_buffers()

    del stage, stage16, host16, devb
    model._get_engine()._release_buffers()
    torch.cuda.empty_cache()
    train = train_ecg = eog = None
    if not args.no_train:
        train = time_train_step(model, dev, world, rank, barrier, max_over_ranks, lib)
        # the same step with every rank drawing the SAME modality masks: separates mask stragglers from communication
        train["same_mask_on_all_ranks"] = time_train_step(model, dev, world, rank, barrier, max_over_ranks, lib,
                                                          same_seed=True)["ms_per_step"] if world > 1 else None
        torch.cuda.empty_cache()
        train_ecg = time_train_step(model, dev, world, rank, barrier, max_over_ranks, lib, batch=32, only=("ECG",))
        torch.cuda.empty_cache()
    if not args.no_eog and world == 1:
        eog = time_eog(dev, lib, hbm_peak, tf_peak)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hours_per_step = BATCH * HOURS_PER_NIGHT * world
    value = hours_per_step * args.steps / (ms_dev * 1e-3)
    e2e_value = hours_per_step * args.steps / (ms_e2e * 1e-3)

    # aggregate the profile by kernel label: share of the step and achieved algorithmic bandwidth / flop rate
    agg = {}
    for label, ms, by, fl in prof:
        a = agg.setdefault(label, [0.0, 0.0, 0.0, 0])
        a[0] += ms; a[1] += by; a[2] += fl; a[3] += 1
    total_ms = sum(a[0] for a in agg.values()) or 1.0
    kernels = []
    for label, (ms, by, fl, n) in sorted(agg.items(), key=lambda kv: -kv[1][0]):
        kernels.append({"kernel": label, "launches_per_step": n // 2, "share": ms / total_ms,
                        "avg_ms": ms / n, "algo_bytes": by / n, "algo_GBps": by / ms * 1e-6 if ms > 0 else None,
                        "algo_TFLOPs": fl / ms * 1e-9 if ms > 0 else None})
    if args.kernels_out:
        Path(args.kernels_out).write_text(json.dumps(kernels, indent=1))
    roofline = None
    if kernels:
        # The dominant kernel is a kernel FUNCTION (template instantiation), as in the ncu launch list under profiles/:
        # all its launches of the step together (the labels above also carry the batch / length of each launch, which
        # splits one function over several lines).  bytes per launch and launch duration are averages over its launches.
        import re
        fn = {}
        for label, (ms, by, fl, n) in agg.items():
            a = fn.setdefault(re.sub(r" B\d+ L\d+$", "", label), [0.0, 0.0, 0.0, 0])
            a[0] += ms; a[1] += by; a[2] += fl; a[3] += n
        key, (ms, by, fl, n) = max(fn.items(), key=lambda kv: kv[1][0])
        k = {"kernel": key, "algo_GBps": by / ms * 1e-6, "algo_bytes": by / n, "share": ms / total_ms, "avg_ms": ms / n,
             "launches_per_step": n // 2}
        # DRAM traffic per launch of that kernel from the committed `ncu --set full` capture (profiles/), if any
        traffic = None
        tf = ROOT / "profiles" / "traffic.json"
        if tf.exists():
            traffic = json.loads(tf.read_text()).get(k["kernel"], {}).get("dram_bytes_per_launch")
        big = kernels[0]  # the largest single launch shape, for continuity with round 1 (block-0 fused conv2)
        roofline = {"bound": "hbm", "achieved": k["algo_GBps"], "peak": hbm_peak, "unit": "GB/s",
                    "frac": k["algo_GBps"] / hbm_peak, "traffic": traffic, "kernel": k["kernel"],
                    "launches_per_step": k["launches_per_step"],
                    "algo_bytes_per_launch": k["algo_bytes"],
                    "share_of_step": k["share"], "avg_launch_ms": k["avg_ms"], "peak_source": peak_src,
                    "largest_launch_shape": {"kernel": big["kernel"], "share_of_step": big["share"],
                                             "achieved": big["algo_GBps"], "frac": big["algo_GBps"] / hbm_peak,
                                             "avg_launch_ms": big["avg_ms"]},
                    "whole_step": {"algo_GBps": sum(a[1] for a in agg.values()) / total_ms * 1e-6,
                                   "algo_TFLOPs": sum(a[2] for a in agg.values()) / total_ms * 1e-9,
                                   "kernel_ms_per_step": total_ms / 2}}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_time(steps=3, warmup=1)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "nights_per_gpu_per_step": BATCH, "epochs_per_night": S_EPOCHS,
                   "parallelism": f"replicas x{world} (no data-path collective)",
                   "api": "Wav2Sleep.predict_async (engine-owned streams, results awaited in order)",
                   "l2": "inputs+activations > L2, 2 alternating batches",
                   "host_affinity": f"rank bound to {host_cpus} GPU-local CPUs" if host_cpus else "unbound"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": ms_e2e / args.steps},
        "e2e_staged": {"value": hours_per_step * args.steps / (ms_staged * 1e-3), "unit": UNIT,
                       "h2d_bytes_per_step": h2d_bytes // 2, "d2h_bytes_per_step": d2h_bytes,
                       "ms_per_step": ms_staged / args.steps,
                       "transport": "int16 raw samples + on-device whole-night z-score (SURVEY 8f N1), then the same forward"},
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        "roofline": roofline,
        "kernels": kernels[:8],
        "cpu_baseline": cpu,
        "train": train,
        "train_ecg_only": train_ecg,
        "eog": eog,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def clocks_during(fn, index):
    """Run fn() while sampling nvidia-smi clocks; returns (result, clocks summary)."""
    sampler = ClockSampler(index)
    sampler.start()
    try:
        out = fn()
    finally:
        sampler.stop_flag.set()
        sampler.join(timeout=3)
    return out, sampler.summary()


def time_train_step(model, dev, world, rank, barrier, max_over_ranks, lib, steps=5, warmup=3, batch=BATCH, only=None,
                    same_seed=False):
    """Secondary metric (BASELINE.json "train step ms").  configs[3]: cardio training step at 16 nights per GPU = polarity
    flip + config masker + forward (activations kept, dropout 0.1 in both mixers) + CE + loss-scaled fp16 backward +
    bucketed gradient all-reduce + fused clip + AdamW.  configs[4] (``only=("ECG",)``, batch 32): the same 4-signal model
    with PPG / ABD / THX missing for every night (rows of -inf, what the masker emits), no random masking."""
    import torch.distributed as dist
    from wav2sleep_b200.optim import FusedAdamW
    from wav2sleep_b200.trainer import SignalMasker, SleepLightningModule
    torch.manual_seed(1234 + (0 if same_seed else rank))
    masker = None if only else SignalMasker({"ABD": 0.7, "THX": 0.7, "ECG": 0.5, "PPG": 0.1}, backups=["ECG", "PPG"])
    pl = SleepLightningModule(model, optimizer=lambda ps: FusedAdamW(ps, lr=1e-3, weight_decay=1e-4, max_grad_norm=1.0),
                              num_classes=4, masker=masker)
    pl.setup_training()
    src = {k: v.to(dev) for k, v in make_night_batch(batch, seed=7 + rank).items()}
    if only:
        for k in src:
            if k not in only:
                src[k].fill_(float("-inf"))
    y = torch.randint(0, 4, (batch, S_EPOCHS), device=dev)
    y[torch.rand(batch, S_EPOCHS, device=dev) < 0.05] = -1

    def one():
        x = {k: v.clone() for k, v in src.items()}
        return pl.fit_step((x, y))

    for _ in range(warmup):
        one()
    barrier()
    l0 = lib.w2s_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed():
        e0.record()
        for _ in range(steps):
            loss = one()
        e1.record()
        barrier()
        return loss

    loss, clocks = clocks_during(timed, dev.index or 0)
    own = e0.elapsed_time(e1) / steps
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    per_rank = [own]
    if world > 1:
        t = torch.tensor([own], device=dev, dtype=torch.float64)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = [float(v.item()) for v in allt]
    eng = model._get_engine()
    eng.bucket_hooks = []
    model.eval()
    return {"ms_per_step": ms, "nights_per_gpu": batch, "n_gpus": world, "steps": steps, "warmup": warmup,
            "recording_hours_per_s": batch * HOURS_PER_NIGHT * world / (ms * 1e-3),
            "per_rank_ms": per_rank, "last_loss": float(loss),
            "gpu_launches_per_step": int((lib.w2s_launch_count() - l0) / steps),
            "signals": list(only) if only else "all four, config masker cardiorespiratory/all.yaml (ABD .7, THX .7, ECG .5, "
                                               "PPG .1; backups ECG, PPG)",
            "loss_scale": eng.last_loss_scale, "grad_dtype": "f16 activations (loss-scaled), f32 parameters",
            "dropout": float(model.epoch_mixer.dropout), "optimizer": "fused clip(1.0) + AdamW(lr 1e-3, wd 1e-4)",
            "clocks": clocks}


def time_eog(dev, lib, hbm_peak, tf_peak, steps=5, warmup=3):
    """BASELINE configs[1]: wav2sleep-eog (EOG-L + EOG-R, 4096 samples per epoch, 10-block encoders, 5 classes), batch of
    16 synthetic 14-h nights (S = 1680) on one GPU, inputs resident in HBM.  Same metric as the headline."""
    from wav2sleep_b200 import build_default
    S, B, hours = 1680, 16, 14.0
    model = build_default({"EOG-L": "EOG-L", "EOG-R": "EOG-R"}, 5, seed=0).to(dev).eval()
    g = torch.Generator().manual_seed(42)
    xs = [{k: torch.randn(B, S * 4096, generator=g).to(dev) for k in ("EOG-L", "EOG-R")} for _ in range(2)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.inference_mode():
        for i in range(warmup):
            model.predict_async(xs[i % 2]).wait()
        torch.cuda.synchronize()
        l0 = lib.w2s_launch_count()

        def timed():
            e0.record()
            pend = []
            for i in range(steps):
                pend.append(model.predict_async(xs[i % 2]))
                if len(pend) > 2:
                    pend.pop(0).wait()
            for q in pend:
                q.wait()
            e1.record()
            torch.cuda.synchronize()

        _, clocks = clocks_during(timed, dev.index or 0)
        launches = lib.w2s_launch_count() - l0
        ms = e0.elapsed_time(e1) / steps
        eng = model._get_engine()
        eng.enc_streams = False
        model.predict(xs[0])
        lib.w2s_profile_enable(1)
        model.predict(xs[1])
        torch.cuda.synchronize()
        prof = collect_profile(lib)
        lib.w2s_profile_enable(0)
    kms = sum(r[1] for r in prof) or 1.0
    by, fl = sum(r[2] for r in prof), sum(r[3] for r in prof)
    wide = [int(e.wide_blocks) for e in model.signal_encoders.encoders.values()]
    del xs, model
    torch.cuda.empty_cache()
    return {"metric": METRIC, "value": B * hours / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
            "warmup": warmup, "gpu_launches": int(launches), "clocks": clocks,
            "config": {"workload": "wav2sleep-eog (EOG-L, EOG-R) 5-class inference, 16 synthetic 14-h nights on 1 GPU "
                                   "(BASELINE configs[1])", "epochs_per_night": S, "wide_blocks": wide},
            "roofline": {"bound": "hbm", "achieved": by / kms * 1e-6, "peak": hbm_peak, "unit": "GB/s",
                         "frac": by / kms * 1e-6 / hbm_peak, "scope": "whole step, algorithmic bytes of every launch / "
                         "summed kernel time", "algo_TFLOPs": fl / kms * 1e-9, "kernel_ms_per_step": kms}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the secondary train-step timings")
    ap.add_argument("--no-eog", action="store_true", help="skip the secondary EOG-model timing (BASELINE configs[1])")
    ap.add_argument("--kernels-out", default=None, help="also write the full per-kernel profile (JSON list) to this file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the int64 [16, 1200] predictions of the last timed step (as float32) to DIR/predictions.npy"
                         " (DIR/predictions_rank<r>.npy for N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs applies to the CUDA path only")
    args.warmup = max(args.warmup, 3) if args.impl == "cuda" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
