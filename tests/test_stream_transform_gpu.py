"""-m gpu: the fused block-0 prologues inside whole-model forwards.

The stream kernels' interior tiles (no zero-padding rows, whole raw-signal window staged) take a fully unrolled path
and edge tiles keep the bounds checks; test_encoder_fwd_kernels_gpu.py holds each kernel to an fp64 reference on both.
Here -inf samples scattered inside live raw-signal rows go through a whole cardio forward, on both halves of a paired
launch.
"""
import pytest
import torch


pytestmark = pytest.mark.gpu


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
