"""-m gpu: the stream kernels' transform on interior and edge tiles.

Interior tiles (no zero-padding rows, whole raw-signal window staged) take a fully unrolled path with per-thread
shared-memory offsets; edge tiles keep the bounds checks.  These tests put tiles on both paths in one launch: lengths
that are not a multiple of the tile, tiles at both ends of a sample, samples split over CTA ranges, a masked sample
between live ones, and -inf samples inside live raw-signal rows for the fused block-0 prologues (PRO_FIR, PRO_NORM_RES_X),
on both halves of a paired launch.
"""
import pytest
import torch

import gpu_utils as G
from wav2sleep_b200 import _lib

pytestmark = pytest.mark.gpu


def rel_err(a, b):
    return ((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-6)).item()


def _conv(impl, cin, cout, stride, has_ds, y, r, w, wd, mask):
    lib = _lib.load()
    lib.w2s_set_conv_impl(impl)
    try:
        B, L = y.shape[0], y.shape[1]
        L_out = (L - 1) // stride + 1
        dev = y.device
        out = torch.zeros(B, L_out, cout, dtype=torch.float16, device=dev)
        out_ds = torch.zeros(B, L_out // 2, cout, dtype=torch.float16, device=dev) if has_ds else None
        stats = torch.zeros(B, cout, 2, device=dev, dtype=torch.float64)
        split = G.uses_split(cin, cout)
        G.run_conv(cin=cin, cout=cout, taps=3, stride=stride, dilation=1, pad=1,
                   prologue=_lib.PRO_NORM_RES if has_ds else _lib.PRO_NORM, epilogue=_lib.EPI_STATS, has_ds=has_ds,
                   B=B, L_in=L, L_out=L_out, **{"in": y}, in_res=r, in_stats=G.sums(y), w=G.pack_conv(w, split=split),
                   w_ds=G.pack_conv(wd, split=split) if has_ds else None, out=out, out_ds=out_ds, out_stats=stats,
                   row_mask=mask, in_eps=1e-2)
        torch.cuda.synchronize()
        return out, out_ds, stats
    finally:
        lib.w2s_set_conv_impl(0)


# the default 16- and 32-channel ring-path instantiations; lengths are not a multiple of the tile (1024 / 512 / 256
# output rows) and give each sample several interior tiles plus an edge tile at either end
@pytest.mark.parametrize("cin,cout,stride,has_ds,B,L", [
    (16, 16, 1, 0, 5, 9000), (16, 16, 2, 0, 5, 9001), (16, 16, 1, 1, 5, 5000), (16, 32, 1, 1, 5, 4100),
    (32, 32, 1, 0, 5, 4097), (32, 32, 2, 0, 5, 3001), (32, 32, 1, 1, 5, 2999),
])
def test_stream_transform_matches_tile_kernel(cuda_device, cin, cout, stride, has_ds, B, L):
    """Stream kernel == tile-per-CTA kernel (same prologue math and operands) and the fp32 reference; the masked sample
    in the middle stays untouched."""
    torch.manual_seed(cin * 7 + cout + stride * 3 + has_ds + L)
    dev = cuda_device
    y = (torch.randn(B, L, cin, device=dev) * 1.3 + 0.2).half()
    r = torch.randn(B, L, cin, device=dev).half() if has_ds else None
    w = torch.randn(cout, cin, 3, device=dev) / (3 * cin) ** 0.5
    wd = torch.randn(cout, cin, 1, device=dev) / cin ** 0.5 if has_ds else None
    mask = torch.zeros(B, dtype=torch.uint8, device=dev)
    mask[2] = 1
    s_out, s_ds, s_st = _conv(0, cin, cout, stride, has_ds, y, r, w, wd, mask)
    t_out, t_ds, t_st = _conv(1, cin, cout, stride, has_ds, y, r, w, wd, mask)
    live = [b for b in range(B) if b != 2]
    split = G.uses_split(cin, cout)
    ref = G.conv_ref(G.prologue_ref(y, r), w, stride=stride, split=split)
    assert s_out[2].abs().max().item() == 0 and s_st[2].abs().max().item() == 0
    assert not torch.isnan(s_out.float()).any()
    # same fp16 operands, fp32 accumulation in both kernels: only the accumulation order of the MMAs may differ
    assert rel_err(s_out[live], t_out[live]) < 1e-3
    assert rel_err(s_out[live], ref[live]) < (1e-3 if split else 4e-3)
    assert torch.allclose(s_st[live], t_st[live], rtol=1e-4, atol=1e-2 * L ** 0.5)
    if has_ds:
        assert rel_err(s_ds[live], t_ds[live]) < 1e-3


def test_fused_block0_with_scattered_neg_inf(cuda_device):
    """Whole cardio forward (ECG + PPG and ABD + THX paired) against the oracle with -inf samples scattered inside
    live rows: the block-0 kernels that recompute conv1 from the raw signal (PRO_FIR) and add the raw-signal 1x1
    branch (PRO_NORM_RES_X) replace each of them by 0, on interior and edge tiles, in both halves of a paired launch;
    night 2 is masked on THX."""
    from oracle import wav2sleep_oracle as oracle
    from wav2sleep_b200 import build_default

    smap = {"ABD": "ABD", "THX": "THX", "ECG": "ECG", "PPG": "PPG"}
    spe = {"ABD": 256, "THX": 256, "ECG": 1024, "PPG": 1024}
    model = build_default(smap, 4, seed=5)
    g = torch.Generator().manual_seed(11)
    B, E = 4, 13
    x = {k: torch.randn(B, E * spe[k], generator=g) for k in smap}
    for k, n in (("ECG", 300), ("PPG", 200), ("ABD", 50)):
        T = E * spe[k]
        for b in range(B):
            idx = torch.randint(1, T, (n,), generator=g)
            idx = torch.cat([idx, torch.tensor([1, 2, T - 1, T - 2, 1023, 1024, 1025, 2047, 2048])])
            x[k][b, idx.clamp(1, T - 1)] = float("-inf")
    x["THX"][2] = float("-inf")
    ref = oracle.forward(x, model.state_dict(), oracle.cardio_config())
    model = model.to(cuda_device).eval()
    with torch.inference_mode():
        out = model({k: v.to(cuda_device) for k, v in x.items()})
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    err = (out.float().cpu() - ref).abs().max().item()
    assert err < 2e-2, f"logits differ from the oracle by {err}"
