"""Cost of integrated_gradients (wav2sleep_b200/attribution.py):
  cardio : 16 full cardio nights (bench.make_night_batch), default model on the fast path, 32 steps, zero baseline
  ppgnet : one full SleepPPGNet night (general path), 32 steps
Wall time per call (host clock around the call, which ends with a device synchronise), then one profiled call per
workload: the share of the library kernel time taken by w2s_ig_path_inputs and w2s_ig_accumulate, and their achieved
bandwidth from their algorithmic bytes.  Prints the card and its power limit beside the numbers."""
import ctypes as C
import subprocess
import sys
import time
from collections import defaultdict
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from wav2sleep_b200 import _lib, build_default, integrated_gradients  # noqa: E402
from wav2sleep_b200.ppgnet import SleepPPGNet  # noqa: E402

STEPS, REPS = 32, 3


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown card"


def wall(fn, reps):
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3)
    return sorted(out)


def profile(lib, fn):
    lib.w2s_profile_enable(1)
    try:
        fn()
        torch.cuda.synchronize()
        per = defaultdict(lambda: [0, 0.0, 0.0])
        buf, ms, nbytes = C.create_string_buffer(96), C.c_float(), C.c_double()
        for i in range(lib.w2s_profile_count()):
            _lib.check(lib.w2s_profile_get(i, buf, 96, C.byref(ms), C.byref(nbytes), None))
            key = buf.value.decode().split(" ")[0]
            per[key][0] += 1
            per[key][1] += ms.value
            per[key][2] += nbytes.value
        return per
    finally:
        lib.w2s_profile_enable(0)


def report(name, lib, fn):
    fn()  # warm every shape
    ts = wall(fn, REPS)
    print(f"  {name}: wall per call median {ts[len(ts) // 2]:.1f} ms (min {ts[0]:.1f}, max {ts[-1]:.1f}; {REPS} calls)")
    per = profile(lib, fn)
    total = sum(v[1] for v in per.values())
    print(f"    profiled call: sum of library kernel times {total:.1f} ms")
    for key in ("ig_path_inputs", "ig_accumulate"):
        n, t, b = per.get(key, (0, 0.0, 0.0))
        bw = b / (t * 1e-3) / 1e12 if t > 0 else float("nan")
        print(f"    {key:15s} {n:4d} launches {t:8.3f} ms = {100 * t / total:6.3f} % of kernel time, {bw:.2f} TB/s "
              f"({b / 1e9:.2f} GB algorithmic)")
    for key, (n, t, _) in sorted(per.items(), key=lambda kv: -kv[1][1])[:6]:
        print(f"    top: {key:22s} {n:5d} launches {t:9.2f} ms  {100 * t / total:5.1f} %")


def main():
    if not torch.cuda.is_available():
        raise SystemExit("time_attribution: needs a CUDA device")
    dev = torch.device("cuda:0")
    lib = _lib.load()
    print(f"card: {card()}; integrated_gradients, {STEPS} Gauss-Legendre steps, default internal_batch_size (16)")
    x = {k: v.to(dev) for k, v in bench.make_night_batch(16, seed=7).items()}
    model = build_default(bench.CARDIO, 4, seed=0).to(dev).eval()
    report(f"cardio fast path, 16 nights x S={bench.S_EPOCHS}", lib, lambda: integrated_gradients(model, x, 2, steps=STEPS))
    attr, delta = integrated_gradients(model, x, 2, steps=STEPS)
    total = delta + sum(a.double().sum(dim=1) for a in attr.values())
    print(f"    completeness: max |delta| / |F(x) - F(x0)| = {(delta.abs() / total.abs()).max().item():.3e}")
    del attr, model, x
    torch.manual_seed(0)
    ppg = SleepPPGNet().to(dev).eval()
    xp = torch.randn(1, SleepPPGNet.INPUT_LENGTH, device=dev)
    report("SleepPPGNet, 1 night", lib, lambda: integrated_gradients(ppg, xp, 2, steps=STEPS))


if __name__ == "__main__":
    main()
