"""Not-gpu: the general-path gradient oracle (oracle/general_oracle.py) is tied to the reference model.

Its eval forward must reproduce the REAL reference's logits stored in tests/golden/general_*.npz for every case of
oracle/make_golden_general.CASES (same parameters: the case's seed + ``perturb``; same inputs).  The GPU training tests
then compare the CUDA backward with this oracle's autograd, so a gradient error cannot hide behind a shared mistake in
the forward restatement.
"""
import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import general_oracle as GO
from oracle import make_golden_general as G
from wav2sleep_b200 import model as M


@pytest.mark.parametrize("name", list(G.CASES))
def test_general_oracle_reproduces_reference_logits(name):
    case = G.CASES[name]
    model = G.build(M, case)
    G.perturb(model, case["seed"])
    sd = {k: v.detach().to(torch.float32) for k, v in model.state_dict().items()}
    with torch.no_grad():
        got = GO.forward(G.make_inputs(case), sd, GO.config(case))
    ref = torch.from_numpy(np.load(GOLDEN / f"{name}.npz")["logits"])
    err = (got - ref).abs().max().item()
    print(f"{name}: oracle vs reference max-abs logit error {err:.3e}")
    assert got.shape == ref.shape and err <= 1e-5
