"""Cost of an input-attribution pass on the fast path: cardio, 16 full nights (bench.make_night_batch), default model,
every parameter frozen, eval().  Three legs, timed with CUDA events in alternating rounds:
  infer    : model(x) under no_grad (the fused inference kernels)
  saliency : logits = model(x) with x requiring grad, then logits[..., c].sum() backward into x
  train    : one training step of bench.py's train leg (fwd + CE + bwd + clip + AdamW, dropout on, parameters trainable)
then one profiled saliency pass, its time split by kernel (library launch profile).  Prints the card and its power limit
beside the numbers."""
import ctypes as C
import subprocess
import sys
from collections import defaultdict
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from wav2sleep_b200 import _lib, build_default  # noqa: E402
from wav2sleep_b200.optim import FusedAdamW  # noqa: E402
from wav2sleep_b200.trainer import SleepLightningModule  # noqa: E402

B, ROUNDS, REPS = 16, 5, 3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown card"


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_input_gradients: needs a CUDA device")
    dev = torch.device("cuda:0")
    src = {k: v.to(dev) for k, v in bench.make_night_batch(B, seed=7).items()}
    frozen = build_default(bench.CARDIO, 4, seed=0).to(dev).eval()
    for p in frozen.parameters():
        p.requires_grad_(False)

    def infer():
        with torch.no_grad():
            frozen(src)

    def saliency():
        x = {k: v.detach().requires_grad_(True) for k, v in src.items()}
        frozen(x)[..., 2].sum().backward()
        return x

    trained = build_default(bench.CARDIO, 4, seed=0).to(dev)
    pl = SleepLightningModule(trained, optimizer=lambda ps: FusedAdamW(ps, lr=1e-3, weight_decay=1e-4, max_grad_norm=1.0),
                              num_classes=4)
    pl.setup_training()
    y = torch.randint(0, 4, (B, bench.S_EPOCHS), device=dev)
    train = lambda: pl.fit_step(({k: v.clone() for k, v in src.items()}, y))

    legs = {"infer": infer, "saliency": saliency, "train": train}
    for fn in legs.values():  # warm every shape the timed rounds use
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    times = defaultdict(list)
    for _ in range(ROUNDS):
        for name, fn in legs.items():
            times[name].append(timed(fn, REPS))
    print(f"card: {card()}; cardio B={B} full nights (S={bench.S_EPOCHS}); {ROUNDS} alternating rounds x {REPS} calls")
    for name, ts in times.items():
        ts = sorted(ts)
        print(f"  {name:9s} median {ts[len(ts) // 2]:7.2f} ms  (min {ts[0]:.2f}, max {ts[-1]:.2f})")
    x = saliency()
    print(f"  saliency gradients finite: {all(bool(torch.isfinite(v.grad).all()) for v in x.values())}, "
          f"loss scale {frozen._get_engine().last_loss_scale:g}")

    lib = _lib.load()
    torch.cuda.synchronize()
    lib.w2s_profile_enable(1)
    saliency()
    torch.cuda.synchronize()
    per = defaultdict(lambda: [0, 0.0])
    buf, ms = C.create_string_buffer(96), C.c_float()
    for i in range(lib.w2s_profile_count()):
        _lib.check(lib.w2s_profile_get(i, buf, 96, C.byref(ms), None, None))
        key = buf.value.decode().split(" ")[0]
        per[key][0] += 1
        per[key][1] += ms.value
    lib.w2s_profile_enable(0)
    total = sum(v[1] for v in per.values())
    print(f"  profiled saliency pass: sum of library kernel times {total:.2f} ms (profiled run, events per launch)")
    for key, (n, t) in sorted(per.items(), key=lambda kv: -kv[1][1]):
        print(f"    {key:22s} {n:4d} launches {t:8.3f} ms  {100 * t / total:5.1f} %")

    # w2s_first_conv_dgrad by itself at the ECG shape of the batch (16 x 1 228 800 samples; 1.1 GB per call, > L2)
    T = src["ECG"].shape[1]
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(B, T, device=dev, generator=g)
    dy1 = torch.randn(B, T, 16, device=dev, generator=g).half()
    dr = torch.randn(B, T // 2, 16, device=dev, generator=g).half()
    w1, wds = torch.randn(16, 3, device=dev, generator=g), torch.randn(16, device=dev, generator=g)
    mask, dx = torch.zeros(B, dtype=torch.uint8, device=dev), torch.empty(B, T, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    call = lambda: _lib.check(lib.w2s_first_conv_dgrad(x.data_ptr(), dy1.data_ptr(), dr.data_ptr(), w1.data_ptr(),
                                                       wds.data_ptr(), mask.data_ptr(), dx.data_ptr(), B, T, 0.5, st))
    for _ in range(3):
        call()
    ms_k = timed(call, 50)
    nbytes = B * T * (32 + 16 + 4 + 4)
    print(f"  first_conv_dgrad alone, B={B} T={T}: {ms_k * 1e3:.1f} us, {nbytes / ms_k * 1e-9:.2f} TB/s of "
          f"{nbytes / 1e9:.2f} GB algorithmic traffic (dy1 32 + dr 16 + x 4 + dx 4 B per sample)")


if __name__ == "__main__":
    main()
