"""Not-gpu: the SleepPPGNet training oracle (oracle/ppgnet_oracle.py) is tied to the reference.

``ppgnet_forward`` in eval mode must reproduce the real reference's logits in tests/golden/general_ppgnet.npz, and
``batch_norm_train`` must be ``nn.BatchNorm1d`` in ``train()`` - output and all three buffers, call after
call.  The GPU training tests (tests/test_ppgnet_training_gpu.py) then compare the CUDA path with this oracle.
"""
import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import ppgnet_oracle as PO
from oracle import make_golden_general as G


def test_ppgnet_oracle_reproduces_reference_logits():
    from wav2sleep_b200.ppgnet import SleepPPGNet
    model = G.build_ppgnet(SleepPPGNet)
    G.perturb(model, G.PPG_SEED)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    with torch.no_grad():
        got = PO.ppgnet_forward(G.ppg_input(), sd, "leaky")
    ref = torch.from_numpy(np.load(GOLDEN / "general_ppgnet.npz")["logits"])
    err = (got - ref).abs().max().item()
    print(f"SleepPPGNet oracle vs reference: max-abs logit error {err:.3e}")
    assert got.shape == ref.shape and err <= 1e-5


@pytest.mark.parametrize("momentum", [0.1, None])
def test_train_mode_batchnorm_equals_torch_batchnorm(momentum):
    g = torch.Generator().manual_seed(0 if momentum is None else 1)
    Cc = 5
    bn = torch.nn.BatchNorm1d(Cc, momentum=momentum).train()
    with torch.no_grad():
        bn.weight.copy_(1 + 0.3 * torch.randn(Cc, generator=g))
        bn.bias.copy_(0.3 * torch.randn(Cc, generator=g))
    sd = {f"n.{k}": v.detach().clone() for k, v in bn.state_dict().items()}
    for call in range(3):
        x = 3.0 + (call + 1) * torch.randn(4 - call, Cc, 37 + call, generator=g)
        upd = {}
        got = PO.batch_norm_train(x, sd, "n", upd, momentum=momentum)
        want = bn(x)
        torch.testing.assert_close(got, want, rtol=1e-6, atol=1e-6)
        for k, v in bn.state_dict().items():
            if k in ("weight", "bias"):
                continue
            o = upd[f"n.{k}"]
            if k == "num_batches_tracked":
                assert int(o) == int(v) == call + 1
            else:
                torch.testing.assert_close(o, v, rtol=1e-6, atol=1e-7)
        sd.update(upd)
