"""CPU tests of integrated_gradients' host logic: the Gauss-Legendre rule, target parsing, the pass plan, and argument
errors raised before the CUDA library is loaded."""
import numpy as np
import pytest
import torch

import wav2sleep_b200
from wav2sleep_b200 import attribution as A
from wav2sleep_b200 import build_default
from wav2sleep_b200.ppgnet import SleepPPGNet


@pytest.mark.parametrize("steps", [1, 2, 7, 32, 64])
def test_gauss_legendre_on_unit_interval(steps):
    a, w = A.gauss_legendre(steps)
    assert a.dtype == np.float64 and a.shape == w.shape == (steps,)
    assert (a > 0).all() and (a < 1).all() and (np.diff(a) > 0).all() and (w > 0).all()
    assert abs(w.sum() - 1.0) < 1e-14
    for deg in range(2 * steps):  # exact for every polynomial of degree <= 2 K - 1
        assert abs((w * a ** deg).sum() - 1.0 / (deg + 1)) < 1e-13, deg
    if steps > 1:  # left-point Riemann weights (the plausible wrong rule) are not exact on the same polynomials
        left = np.full(steps, 1.0 / steps)
        assert abs((left * (np.arange(steps) / steps) ** 3).sum() - 0.25) > 1e-3


@pytest.mark.parametrize("bad", [0, -3, 2.5, True, None, "8"])
def test_gauss_legendre_refuses_bad_steps(bad):
    with pytest.raises(ValueError, match="steps"):
        A.gauss_legendre(bad)


def test_parse_target_forms():
    t = A.parse_target(2, 3, 4, 5)
    assert t.dtype == torch.int64 and t.shape == (3, 4) and (t == 2).all()
    t = A.parse_target(torch.tensor([0, -1, 4]), 3, 4, 5)
    assert t.tolist() == [[0] * 4, [-1] * 4, [4] * 4]
    full = torch.randint(-1, 5, (3, 4), generator=torch.Generator().manual_seed(0))
    assert torch.equal(A.parse_target(full.int(), 3, 4, 5), full)
    assert A.parse_target(np.int64(1), 1, 2, 2).tolist() == [[1, 1]]


@pytest.mark.parametrize("bad, exc, text", [
    (5, ValueError, "outside"), (-1, ValueError, "outside"), (True, TypeError, "bool"), (1.0, TypeError, "int"),
    (torch.tensor([0.0, 1.0, 2.0]), TypeError, "integer"), (torch.tensor([0, 1]), ValueError, r"\[B\]"),
    (torch.zeros(3, 5, dtype=torch.int64), ValueError, "got"), (torch.tensor([0, 5, 1]), ValueError, "lie in"),
    (torch.tensor([0, -2, 1]), ValueError, "lie in"), (torch.tensor([True, False, True]), TypeError, "integer"),
])
def test_parse_target_refuses(bad, exc, text):
    with pytest.raises(exc, match=text):
        A.parse_target(bad, 3, 4, 5)


@pytest.mark.parametrize("B, K, ibs", [(1, 1, 1), (2, 32, 16), (16, 32, 16), (3, 7, 4), (5, 8, 2), (20, 3, 16),
                                       (4, 64, 1), (2, 2, 16)])
def test_pass_plan_covers_every_step_once(B, K, ibs):
    plan = A.passes(B, K, ibs)
    seen = np.zeros((B, K), dtype=int)
    last_k = {}
    for b0, b1, k0, k1 in plan:
        assert 0 <= b0 < b1 <= B and 0 <= k0 < k1 <= K
        assert (b1 - b0) * (k1 - k0) <= ibs
        seen[b0:b1, k0:k1] += 1
        assert last_k.get(b0, 0) == k0  # steps of a night range in order: first = 1 exactly at k0 = 0
        last_k[b0] = k1
    assert (seen == 1).all()


def test_lazy_top_level_export():
    assert wav2sleep_b200.integrated_gradients is A.integrated_gradients
    assert "integrated_gradients" in wav2sleep_b200.__all__


@pytest.fixture
def no_library(monkeypatch):
    """Every argument error below is raised before the CUDA library is loaded (so before any launch)."""
    def refuse(*a, **k):
        raise AssertionError("the CUDA library was loaded before the arguments were checked")
    monkeypatch.setattr(A._lib, "load", refuse)


def test_argument_errors_before_any_launch(no_library):
    model = build_default({"ECG": "ECG", "THX": "THX"}, 4, seed=0)
    x = {"ECG": torch.zeros(2, 3 * 1024), "THX": torch.zeros(2, 3 * 256)}
    with pytest.raises(TypeError, match="Wav2Sleep or a SleepPPGNet"):
        A.integrated_gradients(torch.nn.Linear(2, 2), x, 0)
    with pytest.raises(ValueError, match="steps"):
        A.integrated_gradients(model, x, 0, steps=0)
    with pytest.raises(ValueError, match="internal_batch_size"):
        A.integrated_gradients(model, x, 0, internal_batch_size=0)
    with pytest.raises(TypeError, match="dict"):
        A.integrated_gradients(model, x["ECG"], 0)
    with pytest.raises(KeyError, match="EEG"):
        A.integrated_gradients(model, {"EEG": torch.zeros(2, 1024)}, 0)
    with pytest.raises(RuntimeError, match="CUDA"):  # no CPU fallback
        A.integrated_gradients(model, x, 0)
    ppg = SleepPPGNet(feature_dim=16)
    with pytest.raises(ValueError, match="1228800"):
        A.integrated_gradients(ppg, torch.zeros(1, 1000), 0)
    with pytest.raises(TypeError, match="SleepPPGNet takes"):
        A.integrated_gradients(ppg, {"x": torch.zeros(1, 1228800)}, 0)
    # the model's state is untouched by a refused call
    assert model.training and all(p.requires_grad for p in model.parameters())
