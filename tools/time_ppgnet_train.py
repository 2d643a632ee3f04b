"""Train-step timing of SleepPPGNet on the general CUDA path (train-mode BatchNorm, general.py + csrc/general_bwd.cuh).

Default SleepPPGNet (leaky ReLU, feature_dim 128, dropout 0.2) on B full 10-h nights (1228800 PPG samples each); one
``SleepLightningModule.fit_step`` = forward + cross entropy + backward + clip + FusedAdamW, timed with device events
around warmed-up steps, then split into forward / backward / optimizer with events between the phases.  Then one step
under the library's per-launch CUDA-event profile: the largest kernels, and the two train-mode BatchNorm kernels
(w2s_gen_bn_stats, w2s_gen_bn_update_running) with their time and bandwidth (algorithmic bytes: one read of the
[B * L, C] fp32 tensor).  Prints the card and its power limit.

    python tools/time_ppgnet_train.py [--batch B] [--steps K]
"""
import argparse
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from wav2sleep_b200 import _lib  # noqa: E402
from wav2sleep_b200.optim import FusedAdamW  # noqa: E402
from wav2sleep_b200.ppgnet import SleepPPGNet  # noqa: E402
from wav2sleep_b200.trainer import SleepLightningModule  # noqa: E402

HBM_PEAK_GBS = 6551.0  # measured copy bandwidth of the B200 (DESIGN section 6)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    print(f"device: {torch.cuda.get_device_name(dev)}; nvidia-smi: {smi.stdout.strip() or smi.stderr.strip()}", flush=True)
    torch.manual_seed(0)
    model = SleepPPGNet().to(dev).train()
    pl = SleepLightningModule(model, optimizer=lambda ps: FusedAdamW(ps, lr=1e-3, weight_decay=1e-4, max_grad_norm=1.0),
                              num_classes=4, flip_polarity=False)
    pl.setup_training()
    B, T = args.batch, SleepPPGNet.INPUT_LENGTH
    x = torch.randn(B, T, generator=torch.Generator().manual_seed(7)).to(dev)
    y = torch.randint(0, 4, (B, 1200), device=dev)
    batch = ({"PPG": x}, y)
    for _ in range(2):
        pl.fit_step(batch)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = pl.fit_step(batch)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    print(f"SleepPPGNet, B={B} nights: fit_step {ms:.1f} ms = {B * 10 / ms * 1e3:.0f} recording-hours/s trained, loss "
          f"{float(loss):.3f}, peak memory {torch.cuda.max_memory_allocated(dev) / 2**30:.2f} GiB "
          f"({torch.cuda.max_memory_allocated(dev) / 2**30 / B:.2f} GiB per night)", flush=True)

    # the same step in phases (fit_step without the polarity flip it is configured without)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    phase = torch.zeros(3, dtype=torch.float64)
    for _ in range(args.steps):
        model.train()
        pl._opt.zero_grad()
        ev[0].record()
        loss = pl.training_step(batch)
        ev[1].record()
        loss.backward()
        ev[2].record()
        pl._opt.step()
        ev[3].record()
        torch.cuda.synchronize()
        phase += torch.tensor([ev[i].elapsed_time(ev[i + 1]) for i in range(3)], dtype=torch.float64)
    phase /= args.steps
    print(f"phases: forward + loss {phase[0]:.1f} ms, backward {phase[1]:.1f} ms, clip + AdamW {phase[2]:.2f} ms")

    lib = _lib.load()
    lib.w2s_profile_enable(1)
    pl.fit_step(batch)
    torch.cuda.synchronize()
    recs = bench.collect_profile(lib)
    lib.w2s_profile_enable(0)
    agg = {}
    for label, t, by, _ in recs:
        a = agg.setdefault(label, [0.0, 0, 0.0])
        a[0] += t
        a[1] += 1
        a[2] += by
    tot = sum(a[0] for a in agg.values())
    print(f"kernel time {tot:.1f} ms over {len(recs)} library launches; largest:")
    for k, (t, n, by) in sorted(agg.items(), key=lambda kv: -kv[1][0])[:12]:
        print(f"  {k:24s} n={n:5d} {t:9.2f} ms {100 * t / tot:5.1f}%")
    for label in ("gen_bn_stats", "gen_bn_running"):
        t, n, by = agg.get(label, (0.0, 0, 0.0))
        print(f"{label}: {n} launches, {t:.3f} ms in all, {by / 1e9 / max(t, 1e-9) * 1e3:.0f} GB/s over all launches")
    block0 = B * T * 16 * 4.0
    for label, t, by, _ in recs:
        if label == "gen_bn_stats" and by == block0:
            gbs = by / 1e9 / (t * 1e-3)
            print(f"gen_bn_stats at block 0 (rows {B * T}, C 16, {by / 1e6:.0f} MB): {t * 1e3:.1f} us, {gbs:.0f} GB/s = "
                  f"{100 * gbs / HBM_PEAK_GBS:.0f}% of the measured {HBM_PEAK_GBS:.0f} GB/s HBM peak")


if __name__ == "__main__":
    main()
