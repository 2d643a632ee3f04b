"""Train-step timing of a non-default configuration on the general CUDA path (general.py + csrc/general_bwd.cuh).

Architecture of tests/golden/general_causalconv_layer_silu (causal convolutions, layer norm, SiLU, feature_dim 32,
post-LN mixer, causal sequence mixer with its reference dropout 0.2) on full 10-h nights (S = 1200, ABD + ECG), one
``SleepLightningModule.fit_step`` = forward + cross entropy + backward + clip + FusedAdamW.  Then one step under the
library's per-launch CUDA-event profile, split into forward kernels, backward kernels and the rest.

    python tools/time_general_train.py [--batch B] [--steps K]
"""
import argparse
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from oracle import make_golden_general as G  # noqa: E402
from wav2sleep_b200 import _lib  # noqa: E402
from wav2sleep_b200 import model as M  # noqa: E402
from wav2sleep_b200.optim import FusedAdamW  # noqa: E402
from wav2sleep_b200.trainer import SleepLightningModule  # noqa: E402

FWD = ("gen_conv", "gen_stats", "gen_norm_consts", "gen_affine_act", "gen_rownorm", "gen_attn")
BWD = ("gen_conv_dgrad", "gen_conv_wgrad", "gen_affine_act_bwd", "gen_norm_bwd", "gen_rownorm_bwd", "gen_attn_bwd")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    case = G.CASES["general_causalconv_layer_silu"]
    model = G.build(M, case).to(dev).train()
    pl = SleepLightningModule(model, optimizer=lambda ps: FusedAdamW(ps, lr=1e-3, weight_decay=1e-4, max_grad_norm=1.0),
                              num_classes=case["num_classes"], masker=None)
    pl.setup_training()
    B, S = args.batch, bench.S_EPOCHS
    g = torch.Generator().manual_seed(7)
    src = {k: torch.randn(B, S * G.SPE[k], generator=g).to(dev) for k in case["signal_map"]}
    y = torch.randint(0, case["num_classes"], (B, S), device=dev)
    step = lambda: pl.fit_step(({k: v.clone() for k, v in src.items()}, y))
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    print(f"{torch.cuda.get_device_name(dev)}: general_causalconv_layer_silu, B={B} nights x S={S}: {ms:.1f} ms/step "
          f"= {B * 10 / ms * 1e3:.0f} recording-hours/s trained, loss {float(loss):.3f}, peak memory "
          f"{torch.cuda.max_memory_allocated(dev) / 2**30:.1f} GiB", flush=True)
    lib = _lib.load()
    lib.w2s_profile_enable(1)
    step()
    torch.cuda.synchronize()
    recs = bench.collect_profile(lib)
    lib.w2s_profile_enable(0)
    agg, split = {}, {"forward": 0.0, "backward": 0.0, "other": 0.0}
    for label, t, _, _ in recs:
        a = agg.setdefault(label, [0.0, 0])
        a[0] += t
        a[1] += 1
        split["forward" if label in FWD else "backward" if label in BWD else "other"] += t
    tot = sum(split.values())
    print(f"kernel time {tot:.1f} ms over {len(recs)} launches: forward {split['forward']:.1f} ms, backward "
          f"{split['backward']:.1f} ms ({split['backward'] / max(split['forward'], 1e-9):.1f}x), other "
          f"{split['other']:.1f} ms (dropout, clip + AdamW)")
    for k, (t, n) in sorted(agg.items(), key=lambda kv: -kv[1][0]):
        print(f"  {k:24s} n={n:5d} {t:9.2f} ms {100 * t / tot:5.1f}%")


if __name__ == "__main__":
    main()
