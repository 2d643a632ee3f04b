"""Launch one encoder conv layer at bench-like shapes (for ncu captures and quick timing).

    python tools/profile_conv.py --cin 16 --cout 16 --stride 1 --B 16 --L 1228800 [--ds] [--impl 0|1] [--iters 5]
"""
import argparse
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import gpu_utils as G  # noqa: E402
from wav2sleep_b200 import _lib  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--cin", type=int, default=16)
ap.add_argument("--cout", type=int, default=16)
ap.add_argument("--stride", type=int, default=1)
ap.add_argument("--B", type=int, default=16)
ap.add_argument("--L", type=int, default=1228800)
ap.add_argument("--ds", action="store_true")
ap.add_argument("--impl", type=int, default=0)
ap.add_argument("--iters", type=int, default=5)
ap.add_argument("--reps", type=int, default=1, help="launches between the two events")
ap.add_argument("--fir", action="store_true", help="block-0 fusion prologue (input = raw signal, conv1 recomputed)")
a = ap.parse_args()

dev = torch.device("cuda:0")
lib = _lib.load()
lib.w2s_set_conv_impl(a.impl)
torch.manual_seed(0)
y = torch.randn(a.B, a.L, a.cin, device=dev, dtype=torch.float16)
r = torch.randn(a.B, a.L, a.cin, device=dev, dtype=torch.float16) if a.ds else None
w = torch.randn(a.cout, a.cin, 3, device=dev) / (3 * a.cin) ** 0.5
wd = torch.randn(a.cout, a.cin, 1, device=dev) / a.cin ** 0.5 if a.ds else None
L_out = (a.L - 1) // a.stride + 1
out = torch.empty(a.B, L_out, a.cout, dtype=torch.float16, device=dev)
out_ds = torch.empty(a.B, L_out // 2, a.cout, dtype=torch.float16, device=dev) if a.ds else None
stats = torch.zeros(a.B, a.cout, 2, device=dev, dtype=torch.float64)
split = G.uses_split(a.cin, a.cout)
kw = dict(cin=a.cin, cout=a.cout, taps=3, stride=a.stride, dilation=1, pad=1,
          prologue=_lib.PRO_NORM_RES if a.ds else _lib.PRO_NORM, epilogue=_lib.EPI_STATS, has_ds=int(a.ds), B=a.B,
          L_in=a.L, L_out=L_out, in_res=r, in_stats=G.sums(y), w=G.pack_conv(w, split=split),
          w_ds=G.pack_conv(wd, split=split) if a.ds else None, out=out, out_ds=out_ds, out_stats=stats, in_eps=1e-2)
kw["in"] = y
if a.fir:
    x = torch.randn(a.B, a.L, device=dev)
    w1 = torch.randn(16, 3, device=dev) / 1.7
    y1 = torch.nn.functional.conv1d(x[:, None], w1[:, None], padding=1).transpose(1, 2).contiguous()
    kw.update(prologue=_lib.PRO_FIR, x_raw=x, w_first=w1.contiguous(), T_raw=a.L,
              in_stats=torch.stack([y1.double().sum(1), (y1.double() ** 2).sum(1)], -1).contiguous())
G.run_conv(**kw)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
ts = []
for _ in range(a.iters):
    e0.record()
    for _ in range(a.reps):
        G.run_conv(**kw)
    e1.record()
    torch.cuda.synchronize()
    ts.append(e0.elapsed_time(e1) / a.reps)
byt = a.B * a.L * a.cin * 2 * (2 if a.ds else 1) + a.B * L_out * a.cout * 2 * (1.5 if a.ds else 1)
ms = sorted(ts)[len(ts) // 2]
print(f"cin={a.cin} cout={a.cout} s={a.stride} ds={a.ds} impl={a.impl}: {ms:.3f} ms  {byt / ms * 1e-6:.0f} GB/s algorithmic")

import os
if int(os.environ.get("W2S_DEBUG_FLAGS", "0")) & 64:
    import ctypes
    buf = (ctypes.c_uint64 * 16)()
    torch.cuda.synchronize()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record(); G.run_conv(**kw); t1.record(); torch.cuda.synchronize()
    cta = (ctypes.c_uint64 * 1024)()
    lib.w2s_debug_timestamps(buf, cta)
    import numpy as np
    ct = np.array(cta[:2 * 148], dtype=np.int64).reshape(148, 2)
    t00 = ct[:, 0].min()
    st, en = (ct[:, 0] - t00) / 1e3, (ct[:, 1] - t00) / 1e3
    print("CTA entry (us): min %.1f med %.1f max %.1f | exit: min %.1f med %.1f max %.1f | duration: min %.1f med %.1f max %.1f"
          % (st.min(), np.median(st), st.max(), en.min(), np.median(en), en.max(), (en - st).min(), np.median(en - st),
             (en - st).max()))
    order = np.argsort(en)
    print("slowest CTAs:", [(int(i), round(float(en[i]), 1)) for i in order[-6:]], "fastest:", [(int(i), round(float(en[i]), 1)) for i in order[:4]])
    names = ["entry", "tmem_alloc", "setup_done", "xform_start", "xform_raw_ready", "xform_first_done", "epi_first_full",
             "epi_loop_done", "epi_flushed", "teardown_sync"]
    tot = max(buf[15], 1)
    print("blocked in mbarrier waits (%% of the CTA's %d cycles): MMA(t_empty) %.0f%%, "
          "epilogue(t_full) %.0f%%, transform: raw_full %.0f%% + a_empty %.0f%%"
          % (tot, 100 * buf[12] / tot, 100 * buf[13] / tot, 100 * buf[10] / tot, 100 * buf[14] / tot))
    base = buf[0]
    print("event-timed %.1f us; CTA0 milestones (us since entry): " % (t0.elapsed_time(t1) * 1e3)
          + ", ".join(f"{n}={(buf[i] - base) / 1e3:.1f}" for i, n in enumerate(names)))
