"""-m gpu: integrated gradients (wav2sleep_b200/attribution.py) and SleepPPGNet input gradients.

Kernels: ``w2s_ig_path_inputs`` / ``w2s_ig_accumulate`` against fp64 numpy.  IG: against an independent loop that builds
the same path points with torch, takes each input gradient with the models' attribution path and sums in fp64; against
fp64 autograd of the oracles at small sizes; completeness, invariants and side effects.  Bounds are at most 3x the
error measured on an NVIDIA B200 (power limit 1000 W); the measured values are in DESIGN.md section 4.3.2.  Every
comparison also checks that a plausible wrong reference misses its bound by at least 10x."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gpu_utils as GU
from conftest import make_inputs
from oracle import general_oracle as GO
from oracle import make_golden_general as G
from oracle import ppgnet_oracle as PO
from test_general_training_gpu import CASES as GENERAL_CASES
from test_input_gradients_gpu import _BN_CASE, _oracle_logits, _profile_labels
from test_input_gradients_gpu import CARDIO
from oracle import wav2sleep_oracle as oracle
from wav2sleep_b200 import _lib, build_default, integrated_gradients
from wav2sleep_b200 import attribution as A
from wav2sleep_b200 import model as M
from wav2sleep_b200.ppgnet import SleepPPGNet

pytestmark = pytest.mark.gpu
T_PPG = SleepPPGNet.INPUT_LENGTH

# measured on a B200 at 1000 W (DESIGN.md 4.3.2); each bound <= 3x the measurement
KERNEL_PATH = 2.5e-7   # w2s_ig_path_inputs, max abs error / max |reference| (measured 8.6e-8)
KERNEL_ACC = 1e-6       # w2s_ig_accumulate, max abs error / max |reference| (measured 3.5e-7 at K = 64)
LOOP_GEN = 2.1e-7     # IG against the independent loop, general path, rel L2 per signal (measured 7.3e-8)
LOOP_FAST = 2e-7      # fast path, same passes as the loop (measured 6.7e-8)
LOOP_PPG = 1.2e-7     # SleepPPGNet (measured 4.1e-8)
ORACLE_GEN = 1.4e-5    # IG against fp64 oracle autograd, general path (measured 4.8e-6)
ORACLE_FAST = 6e-2     # fast path, fp16 activations and activation gradients (measured 2.9e-2)
ORACLE_PPG = 3e-6      # SleepPPGNet (measured 1.1e-6)
IBS_FAST = 1.5e-2      # fast path, internal_batch_size 1 against 16: the B = 16 vs B = 2 bound of
                       # test_input_gradients_gpu (batch composition may change kernel schedules); measured 0 here
PPG_EVAL = 1.9e-6      # SleepPPGNet input gradients against fp64 oracle autograd, eval() (measured 6.5e-7)
PPG_TRAIN = 1.5e-4     # train(), batch statistics (measured 5.2e-5)


def _rel(g, r):
    g, r = g.detach().double().cpu().reshape(-1), r.detach().double().cpu().reshape(-1)
    return ((g - r).norm() / r.norm()).item()


def _worst_rel(got, ref):
    return max(_rel(got[n], ref[n]) for n in ref)


def _assert_zero_where_missing(x, attr):
    for n in x:
        xc, a = x[n].detach().cpu(), attr[n].detach().cpu()
        assert (a[~torch.isfinite(xc)] == 0).all(), n
        assert (a[torch.isinf(xc[:, 0])] == 0).all(), n


# ------------------------------------------------------------------------------------------------ kernels
def _path(lib, x, x0, alphas, K, out=None, guard=0):
    B, T = x.shape
    buf = torch.full((K * B * T + 2 * guard,), 12345.0, device=x.device) if out is None else out
    _lib.check(lib.w2s_ig_path_inputs(x.data_ptr(), None if x0 is None else x0.data_ptr(), alphas.data_ptr(), K, B, T,
                                      buf.data_ptr() + 4 * guard, GU.stream()))
    return buf


def _acc(lib, grads, w, K, x, x0, attr, first):
    B, T = x.shape
    _lib.check(lib.w2s_ig_accumulate(grads.data_ptr(), w.data_ptr(), K, x.data_ptr(), None if x0 is None else x0.data_ptr(),
                                     B, T, attr.data_ptr(), first, GU.stream()))


def _kernel_inputs(K, baseline, B=3, T=4099, seed=0):
    g = torch.Generator().manual_seed(seed + K)
    x = torch.randn(B, T, generator=g, dtype=torch.float64).float()
    x[1] = float("-inf")                                  # missing row
    x[0, 5], x[0, 6], x[2, 7], x[2, T - 1] = float("inf"), float("-inf"), float("nan"), float("nan")
    x0 = torch.randn(B, T, generator=g).float() if baseline else None
    a, w = A.gauss_legendre(K)
    return x, x0, a, w


@pytest.mark.parametrize("baseline", [False, True])
@pytest.mark.parametrize("K", [1, 7, 64])
def test_ig_path_inputs_matches_fp64(cuda_device, K, baseline):
    lib, dev = _lib.load(), cuda_device
    x, x0, a, _ = _kernel_inputs(K, baseline)
    B, T = x.shape
    guard = 1000
    buf = _path(lib, x.to(dev), None if x0 is None else x0.to(dev), torch.tensor(a, dtype=torch.float32).to(dev), K,
                guard=guard).cpu()
    assert (buf[:guard] == 12345.0).all() and (buf[-guard:] == 12345.0).all()  # nothing written outside [K * B, T]
    got = buf[guard:-guard].view(K, B, T).double()
    xd = x.double().numpy()
    x0d = np.zeros_like(xd) if x0 is None else x0.double().numpy()
    fin = np.isfinite(xd)
    ref = x0d[None] + np.asarray(a, dtype=np.float32).astype(np.float64)[:, None, None] * (xd - x0d)[None]
    g = got.numpy()
    nf = ~fin
    assert np.array_equal(g[:, nf], np.broadcast_to(xd[nf], (K, int(nf.sum()))), equal_nan=True)  # copied unchanged
    assert np.isneginf(g[:, 1, 0]).all()  # the missing row stays missing at every step
    scale = np.abs(ref[:, fin]).max()
    err = np.abs(g[:, fin] - ref[:, fin]).max() / scale
    print(f"MEASURED ig_path_inputs K={K} baseline={baseline}: {err:.3e}")
    assert err <= KERNEL_PATH, err
    # wrong references: the baseline not added back (a (x - x0)), or the path run the other way (a -> 1 - a)
    af = np.asarray(a)[:, None, None]
    wrong = af * (xd - x0d)[None] if x0 is not None else (1 - af) * xd[None]
    if x0 is not None or K > 1:  # (one node at a = 1/2 with a zero baseline is symmetric)
        miss = np.abs(g[:, fin] - wrong[:, fin]).max() / scale
        assert miss >= 10 * KERNEL_PATH, miss


@pytest.mark.parametrize("baseline", [False, True])
@pytest.mark.parametrize("K", [1, 7, 64])
def test_ig_accumulate_matches_fp64_over_three_calls(cuda_device, K, baseline):
    lib, dev = _lib.load(), cuda_device
    x, x0, _, w = _kernel_inputs(K, baseline, seed=1)
    B, T = x.shape
    g = torch.randn(K * B, T, generator=torch.Generator().manual_seed(7))
    xd_, x0d_ = x.to(dev), None if x0 is None else x0.to(dev)
    wt = torch.tensor(w, dtype=torch.float32).to(dev)
    gd = g.to(dev)
    one = torch.full((B, T), float("nan"), device=dev)
    _acc(lib, gd, wt, K, xd_, x0d_, one, 1)
    # the same steps split over three calls (first = 1, 0, 0): bitwise the one-call sum
    cuts = sorted({0, K // 3, (2 * K) // 3, K})
    three = torch.full((B, T), float("nan"), device=dev)
    for i, (k0, k1) in enumerate(zip(cuts[:-1], cuts[1:])):
        _acc(lib, gd[k0 * B:k1 * B], wt[k0:], k1 - k0, xd_, x0d_, three, int(i == 0))
    torch.cuda.synchronize()
    assert torch.equal(one, three)
    got = one.cpu().double().numpy()
    xd = x.double().numpy()
    x0d = np.zeros_like(xd) if x0 is None else x0.double().numpy()
    fin = np.isfinite(xd)
    wf = np.asarray(w, dtype=np.float32).astype(np.float64)
    s = np.einsum("k,kbt->bt", wf, g.double().view(K, B, T).numpy())
    d = np.where(fin, xd - x0d, 0.0)
    ref = d * s
    assert (got[~fin] == 0).all()  # exactly 0 at non-finite x, the missing row included
    err = np.abs(got - ref).max() / np.abs(ref).max()
    print(f"MEASURED ig_accumulate K={K} baseline={baseline}: {err:.3e}")
    assert err <= KERNEL_ACC, err
    for what, bad in (("no (x - x0) factor", np.where(fin, s, 0.0)),
                      ("left-point weights", d * np.einsum("kbt->bt", g.double().view(K, B, T).numpy()) / K)):
        if what == "left-point weights" and K == 1:
            continue  # one node of weight 1 either way
        miss = np.abs(bad - ref).max() / np.abs(ref).max()
        assert miss >= 10 * KERNEL_ACC, (what, miss)


def test_ig_kernels_past_2_31_elements(cuda_device):
    """K * B * T = 64 x 28 ECG nights = 2.2e9 elements (8.8 GB): 64-bit indexing in both kernels."""
    lib, dev = _lib.load(), cuda_device
    K, B, T = 64, 28, 1200 * 1024
    assert K * B * T > 2 ** 31
    g = torch.Generator(device=dev).manual_seed(3)
    x = torch.randn(B, T, device=dev, generator=g)
    x[5] = float("-inf")
    x0 = torch.randn(B, T, device=dev, generator=g)
    a, w = A.gauss_legendre(K)
    at, wt = torch.tensor(a, dtype=torch.float32).to(dev), torch.tensor(w, dtype=torch.float32).to(dev)
    out = torch.empty(K * B * T, device=dev)
    _path(lib, x, x0, at, K, out=out)
    out = out.view(K * B, T)
    attr = torch.empty(B, T, device=dev)
    _acc(lib, out, wt, K, x, x0, attr, 1)  # grads = the path points themselves: sum_k w_k (x0 + a_k d)
    torch.cuda.synchronize()
    ad = at.double()
    for k, b in ((0, 0), (K - 1, B - 1), (K // 2, 17)):  # the last plane lies past 2^31
        ref = x0[b].double() + ad[k] * (x[b].double() - x0[b].double())
        err = ((out[k * B + b].double() - ref).abs().max() / ref.abs().max()).item()
        assert err <= KERNEL_PATH, (k, b, err)
    assert torch.isinf(out[(K - 1) * B + 5]).all()
    d = torch.where(torch.isfinite(x), x - x0, torch.zeros_like(x)).double()
    ref = d * (x0.double() * wt.double().sum() + d * (wt.double() * ad).sum())
    err = ((attr.double() - ref).abs().max() / ref.abs().max()).item()
    print(f"MEASURED ig kernels past 2^31: accumulate {err:.3e}")
    assert err <= KERNEL_ACC and (attr[5] == 0).all()
    del out


def test_ig_kernels_refuse_bad_arguments(cuda_device):
    lib, dev = _lib.load(), cuda_device
    x, out, a = torch.zeros(2, 5, device=dev), torch.zeros(6, 5, device=dev), torch.zeros(3, device=dev)
    p = lambda t: None if t is None else t.data_ptr()
    for K, B, T, text in ((0, 2, 5, b"K=0"), (3, 0, 5, b"B=0"), (3, 2, 0, b"T=0"), (-1, 2, 5, b"K=-1"), (3, 2, -7, b"T=-7")):
        assert lib.w2s_ig_path_inputs(p(x), None, p(a), K, B, T, p(out), GU.stream()) != 0
        assert text in lib.w2s_last_error(), lib.w2s_last_error()
        assert lib.w2s_ig_accumulate(p(out), p(a), K, p(x), None, B, T, p(x), 1, GU.stream()) != 0
        assert text in lib.w2s_last_error(), lib.w2s_last_error()
    for ops in ((None, a, out), (x, None, out), (x, a, None)):
        assert lib.w2s_ig_path_inputs(p(ops[0]), None, p(ops[1]), 3, 2, 5, p(ops[2]), GU.stream()) != 0
        assert b"NULL operand" in lib.w2s_last_error()
    for i in range(4):
        ops = [out, a, x, x]
        ops[i] = None
        assert lib.w2s_ig_accumulate(p(ops[0]), p(ops[1]), 3, p(ops[2]), None, 2, 5, p(ops[3]), 1, GU.stream()) != 0
        assert b"NULL operand" in lib.w2s_last_error()
    assert lib.w2s_ig_accumulate(p(out), p(a), 3, p(x), None, 2, 5, p(x), 2, GU.stream()) != 0
    assert b"first=2" in lib.w2s_last_error()
    assert lib.w2s_ig_path_inputs(p(x), None, p(a), 3, 2, 5, p(out), GU.stream()) == 0
    assert lib.w2s_ig_accumulate(p(out), p(a), 3, p(x), p(x), 2, 5, p(out), 0, GU.stream()) == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ IG against a loop
def _onehot(tgt, n_classes, dev):
    oh = torch.zeros(*tgt.shape, n_classes, dtype=torch.float64)
    oh.scatter_(2, tgt.clamp(min=0).unsqueeze(-1), (tgt >= 0).double().unsqueeze(-1))
    return oh.to(dev)


def _call(model, xs):
    return model(xs["x"]) if isinstance(model, SleepPPGNet) else model(xs)


def _loop_ig(model, x, x0, tgt, steps, rule="gl", missing="keep"):
    """Independent IG: torch path points, one model call per step through the attribution path, fp64 sums.
    rule "left": left-point Riemann weights; missing "baseline": non-finite samples replaced by the baseline."""
    dev = next(iter(x.values())).device
    if rule == "gl":
        a, w = np.polynomial.legendre.leggauss(steps)
        a, w = (a + 1) / 2, w / 2
    else:
        a, w = np.arange(steps) / steps, np.full(steps, 1.0 / steps)
    model.eval()
    req = [p.requires_grad for p in model.parameters()]
    for p in model.parameters():
        p.requires_grad_(False)
    n_classes = model.classifier.out_features
    sums = {n: torch.zeros(v.shape, dtype=torch.float64, device=dev) for n, v in x.items()}
    try:
        for ak, wk in zip(a, w):
            xs = {}
            for n, v in x.items():
                # fp64 from the fp32 difference, rounded once: the points the kernel's fmaf gives
                pt = (x0[n].double() + float(np.float32(ak)) * (v - x0[n]).double()).float()
                pt = torch.where(torch.isfinite(v), pt, x0[n] if missing == "baseline" else v)
                xs[n] = pt.detach().requires_grad_(True)
            lo = _call(model, xs)
            (lo.double() * _onehot(tgt, n_classes, dev)).sum().backward()
            for n in x:
                sums[n] += float(wk) * xs[n].grad.double()
    finally:
        for p, r in zip(model.parameters(), req):
            p.requires_grad_(r)
    return {n: torch.where(torch.isfinite(x[n]), (x[n] - x0[n]).double() * sums[n], torch.zeros_like(sums[n])) for n in x}


def _drop_factor(ref, x, x0):
    """The wrong reference without the (x - x0) factor: sum_k w_k dF/dx at the path points."""
    out = {}
    for n, v in ref.items():
        d = (x[n] - x0[n]).double().to(v.device)
        out[n] = torch.where(torch.isfinite(d) & (d != 0), v / d, torch.zeros_like(v))
    return out


def _check_against(attr, x, ref_fn, bound, label):
    """attr vs ref_fn() within bound; the three wrong references of the issue miss it by >= 10x."""
    ref = ref_fn()
    _assert_zero_where_missing(x, attr)
    err = _worst_rel(attr, ref)
    print(f"MEASURED {label}: {err:.3e}")
    assert err <= bound, (label, err)
    return ref


def _misses(attr, wrongs, bound, label):
    for what, bad in wrongs:
        miss = _worst_rel(attr, bad)
        print(f"{label} wrong reference {what}: {miss:.3e}")
        assert miss >= 10 * bound, (label, what, miss)


def _general_setup(case, dev, seed=0):
    model = G.build(M, case)
    G.perturb(model, case["seed"])
    model = model.to(dev).eval()
    x = G.make_inputs(case)
    names = sorted(x)
    if not any(torch.isinf(v[:, 0]).any() for v in x.values()) and len(names) > 1:
        x[names[-1]][case["B"] - 1] = float("-inf")  # a missing row
    x[names[0]][0, 3] = float("inf")                  # isolated non-finite samples
    g = torch.Generator().manual_seed(seed + 100)
    x0 = {n: 0.5 * torch.randn(v.shape, generator=g) for n, v in x.items()}
    tgt = torch.randint(0, case["num_classes"], (case["B"], case["S"]), generator=g)
    tgt[0, 0] = -1
    return model, {n: v.to(dev) for n, v in x.items()}, {n: v.to(dev) for n, v in x0.items()}, tgt


@pytest.mark.parametrize("name", list(GENERAL_CASES))
def test_general_path_ig_matches_independent_loop(cuda_device, name):
    model, x, x0, tgt = _general_setup(GENERAL_CASES[name], cuda_device)
    attr, delta = integrated_gradients(model, x, tgt, baseline=x0, steps=8)
    assert delta.dtype == torch.float64 and delta.shape == (GENERAL_CASES[name]["B"],) and torch.isfinite(delta).all()
    _check_against(attr, x, lambda: _loop_ig(model, x, x0, tgt, 8), LOOP_GEN, f"general {name} vs loop")
    ref = _loop_ig(model, x, x0, tgt, 8)
    _misses(attr, [("no (x - x0)", _drop_factor(ref, x, x0)), ("left Riemann", _loop_ig(model, x, x0, tgt, 8, rule="left")),
                   ("baseline on -inf rows", _loop_ig(model, x, x0, tgt, 8, missing="baseline"))], LOOP_GEN, name)


def _fast_setup(dev, B=2, S=24, seed=5):
    model = build_default(CARDIO, 4, seed=0).to(dev).eval()
    x = make_inputs(CARDIO, B, S, masked=[("ABD", 0)], seed=seed)
    x["ECG"][0, 1000] = float("inf")
    x["THX"][1, 77] = float("-inf")
    g = torch.Generator().manual_seed(seed + 1)
    x0 = {n: 0.5 * torch.randn(v.shape, generator=g) for n, v in x.items()}
    tgt = torch.randint(0, 4, (B, S), generator=g)
    tgt[1, ::5] = -1
    return model, {n: v.to(dev) for n, v in x.items()}, {n: v.to(dev) for n, v in x0.items()}, tgt


def test_fast_path_ig_matches_independent_loop(cuda_device):
    model, x, x0, tgt = _fast_setup(cuda_device)
    attr, delta = integrated_gradients(model, x, tgt, baseline=x0, steps=8, internal_batch_size=2)  # the loop's passes
    assert torch.isfinite(delta).all()
    ref = _check_against(attr, x, lambda: _loop_ig(model, x, x0, tgt, 8), LOOP_FAST, "fast cardio vs loop")
    _misses(attr, [("no (x - x0)", _drop_factor(ref, x, x0)), ("left Riemann", _loop_ig(model, x, x0, tgt, 8, rule="left")),
                   ("baseline on -inf rows", _loop_ig(model, x, x0, tgt, 8, missing="baseline"))], LOOP_FAST, "fast")


def _ppg_model(dev, act="silu", seed=11):
    torch.manual_seed(seed)
    m = SleepPPGNet(activation=act, dropout=0.0)
    G.perturb(m, seed)
    return m.to(dev).eval()


def test_ppgnet_ig_matches_independent_loop(cuda_device):
    model = _ppg_model(cuda_device)
    g = torch.Generator().manual_seed(2)
    x = torch.randn(1, T_PPG, generator=g).to(cuda_device)
    x0 = (0.5 * torch.randn(1, T_PPG, generator=g)).to(cuda_device)
    tgt = torch.tensor([2])
    attr, delta = integrated_gradients(model, x, tgt, baseline=x0, steps=4)
    assert attr.shape == x.shape and attr.dtype == torch.float32 and torch.isfinite(delta).all()
    xs, x0s = {"x": x}, {"x": x0}
    ref = _check_against({"x": attr}, xs, lambda: _loop_ig(model, xs, x0s, tgt.view(1, 1).expand(1, 1200), 4), LOOP_PPG,
                         "ppgnet vs loop")
    _misses({"x": attr}, [("no (x - x0)", _drop_factor(ref, xs, x0s)),
                          ("left Riemann", _loop_ig(model, xs, x0s, tgt.view(1, 1).expand(1, 1200), 4, rule="left"))],
            LOOP_PPG, "ppgnet")


# ------------------------------------------------------------------------------------------------ IG against fp64 oracles
def _oracle_ig(logits_fn, x, x0, tgt, n_classes, steps, rule="gl"):
    """fp64 CPU autograd of an oracle along the same path (non-finite samples kept)."""
    if rule == "gl":
        a, w = A.gauss_legendre(steps)
    else:
        a, w = np.arange(steps) / steps, np.full(steps, 1.0 / steps)
    xd = {n: v.detach().cpu().double() for n, v in x.items()}
    x0d = {n: v.detach().cpu().double() for n, v in x0.items()}
    oh = _onehot(tgt, n_classes, "cpu")
    sums = {n: torch.zeros_like(v) for n, v in xd.items()}
    for ak, wk in zip(a, w):
        pts = {n: torch.where(torch.isfinite(v), x0d[n] + float(ak) * (v - x0d[n]), v).requires_grad_(True)
               for n, v in xd.items()}
        (logits_fn(pts) * oh).sum().backward()
        for n in xd:
            sums[n] += float(wk) * pts[n].grad
    return {n: torch.where(torch.isfinite(v), (v - x0d[n]) * sums[n], torch.zeros_like(v)) for n, v in xd.items()}


def test_ig_matches_fp64_oracle_autograd(cuda_device):
    dev = cuda_device
    # general path
    case = GENERAL_CASES["general_causalconv_layer_silu"]
    model, x, x0, tgt = _general_setup(case, dev)
    sd = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    attr, _ = integrated_gradients(model, x, tgt, baseline=x0, steps=4)
    fn = lambda pts: GO.forward(pts, sd, GO.config(case))
    ref = _check_against(attr, x, lambda: _oracle_ig(fn, x, x0, tgt, case["num_classes"], 4), ORACLE_GEN,
                         "general vs fp64 oracle")
    _misses(attr, [("no (x - x0)", _drop_factor(ref, x, x0))], ORACLE_GEN, "general")
    # fast path
    model, x, x0, tgt = _fast_setup(dev, B=2, S=4)
    params = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    attr, _ = integrated_gradients(model, x, tgt, baseline=x0, steps=4)
    fn = lambda pts: _oracle_logits(pts, params, oracle.cardio_config())
    ref = _check_against(attr, x, lambda: _oracle_ig(fn, x, x0, tgt, 4, 4), ORACLE_FAST, "fast vs fp64 oracle")
    _misses(attr, [("no (x - x0)", _drop_factor(ref, x, x0))], ORACLE_FAST, "fast")
    # SleepPPGNet
    model = _ppg_model(dev)
    g = torch.Generator().manual_seed(4)
    x, x0 = {"x": torch.randn(1, T_PPG, generator=g).to(dev)}, {"x": torch.zeros(1, T_PPG, device=dev)}
    tgt = torch.full((1, 1200), 1, dtype=torch.int64)
    tgt[0, :300] = -1
    sd = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    attr, _ = integrated_gradients(model, x["x"], tgt, steps=2)
    fn = lambda pts: PO.ppgnet_forward(pts["x"], sd, "silu")
    ref = _check_against({"x": attr}, x, lambda: _oracle_ig(fn, x, x0, tgt, 4, 2), ORACLE_PPG, "ppgnet vs fp64 oracle")
    _misses({"x": attr}, [("no (x - x0)", _drop_factor(ref, x, x0))], ORACLE_PPG, "ppgnet")


# ------------------------------------------------------------------------------------------------ completeness
def test_completeness_gap_falls_with_steps_on_general_path(cuda_device):
    """Instance-norm encoders: F is smooth along a path between two random signals.  (An encoder whose first norm is
    per time step, such as LayerNorm over the channels of a bias-free Cin = 1 conv, sees only the sign of each sample:
    F then steps wherever a sample crosses 0 on the path, and no quadrature closes the gap.)"""
    model, x, x0, tgt = _general_setup(GENERAL_CASES["chunk_causal_instance"], cuda_device)
    gaps = {}
    for steps in (8, 32, 64):
        attr, delta = integrated_gradients(model, x, tgt, baseline=x0, steps=steps)
        total = delta + sum(a.double().sum(dim=1) for a in attr.values())  # F(x) - F(x0)
        gaps[steps] = (delta.abs().max().item(), total.abs().min().item())
        print(f"MEASURED completeness general steps={steps}: max |delta| {gaps[steps][0]:.3e}, "
              f"min |F(x) - F(x0)| {gaps[steps][1]:.3e}")
    # measured 3.3, 1.3, 0.38 against min |F(x) - F(x0)| = 0.17 (DESIGN.md 4.3.2)
    assert gaps[32][0] < gaps[8][0] and gaps[64][0] < gaps[32][0]


def test_completeness_on_a_full_cardio_night_fast_path(cuda_device):
    model = build_default(CARDIO, 4, seed=0).to(cuda_device).eval()
    x = {n: v.to(cuda_device) for n, v in make_inputs(CARDIO, 1, 1200, seed=11).items()}
    attr, delta = integrated_gradients(model, x, 0, steps=32)
    total = delta + sum(a.double().sum(dim=1) for a in attr.values())
    print(f"MEASURED completeness fast full night: delta {delta.item():.4e}, F(x) - F(x0) {total.item():.4e}, "
          f"ratio {abs(delta.item()) / abs(total.item()):.3e}")
    # recorded, not bounded: the encoders' InstanceNorm makes F(a x) flat in a except near a = 0, where the integrand
    # of a zero baseline concentrates in a sliver that 32 nodes do not resolve (DESIGN.md 4.3.2)
    assert torch.isfinite(delta).all() and torch.isfinite(total).all()


# ------------------------------------------------------------------------------------------------ invariants
def test_internal_batch_size_invariance(cuda_device):
    model, x, x0, tgt = _general_setup(GENERAL_CASES["general_shared_embed_registers"], cuda_device)
    ref, dref = integrated_gradients(model, x, tgt, baseline=x0, steps=5)
    for ibs in (1, 3, 16):
        got, d = integrated_gradients(model, x, tgt, baseline=x0, steps=5, internal_batch_size=ibs)
        assert all(torch.equal(got[n], ref[n]) for n in x), ibs  # bitwise on the general path
        assert torch.equal(d, dref), ibs
    model, x, x0, tgt = _fast_setup(cuda_device, B=2, S=8)
    a16, _ = integrated_gradients(model, x, tgt, baseline=x0, steps=8)
    a1, _ = integrated_gradients(model, x, tgt, baseline=x0, steps=8, internal_batch_size=1)
    err = _worst_rel(a1, {n: v.double() for n, v in a16.items()})
    print(f"MEASURED fast internal_batch_size 1 vs 16: {err:.3e}")
    assert err <= IBS_FAST


def test_no_parameter_gradient_optimizer_or_buffer_is_touched(cuda_device):
    from wav2sleep_b200.optim import FusedAdamW
    dev = cuda_device
    # fast path: p.grad None before and after; training flag and requires_grad pattern kept
    model, x, x0, tgt = _fast_setup(dev, B=2, S=4)
    model.train()
    frozen = set(n for n, _ in list(model.named_parameters())[::3])
    for n, p in model.named_parameters():
        p.requires_grad_(n not in frozen)
    integrated_gradients(model, x, tgt, baseline=x0, steps=3)
    assert model.training and all(m.training for m in model.modules())
    assert all(p.grad is None for p in model.parameters())
    assert all(p.requires_grad == (n not in frozen) for n, p in model.named_parameters())
    # flat optimizer buffers after a training step: bitwise unchanged
    for p in model.parameters():
        p.requires_grad_(True)
    opt = FusedAdamW(model.parameters(), lr=1e-3)
    F.cross_entropy(model(x).reshape(-1, 4), tgt.clamp(min=0).to(dev).reshape(-1)).backward()
    opt.step()
    bufs = {k: getattr(opt, k).clone() for k in ("flat_param", "flat_grad", "exp_avg", "exp_avg_sq")}
    integrated_gradients(model, x, tgt, steps=3)
    torch.cuda.synchronize()
    for k, v in bufs.items():
        assert torch.equal(getattr(opt, k), v), k
    assert all(p.grad is not None and p.grad.data_ptr() >= opt.flat_grad.data_ptr() for p in model.parameters())
    # general path with BatchNorm in train(): running statistics and num_batches_tracked unchanged
    gm = G.build(M, _BN_CASE)
    G.perturb(gm, _BN_CASE["seed"])
    gm = gm.to(dev).train()
    bn0 = {k: v.clone() for k, v in gm.state_dict().items()}
    xg = {k: v.to(dev) for k, v in G.make_inputs(_BN_CASE).items()}
    integrated_gradients(gm, xg, 1, steps=2)
    assert gm.training and all(p.grad is None for p in gm.parameters())
    assert all(torch.equal(gm.state_dict()[k], v) for k, v in bn0.items())


def test_state_is_restored_when_a_pass_raises(cuda_device, monkeypatch):
    model, x, x0, tgt = _fast_setup(cuda_device, B=2, S=4)
    model.train()
    model.sequence_mixer.eval()  # a mixed pattern of training flags comes back as it was
    model.classifier.weight.requires_grad_(False)
    eng = model._get_engine()
    hooks = [lambda name: None]
    eng.bucket_hooks, eng.loss_scale = hooks, 1024.0
    calls = {"n": 0}
    real = torch.autograd.grad

    def failing(*a, **k):
        calls["n"] += 1
        if calls["n"] == 2:
            raise RuntimeError("injected failure")
        return real(*a, **k)
    monkeypatch.setattr(torch.autograd, "grad", failing)
    with pytest.raises(RuntimeError, match="injected"):
        integrated_gradients(model, x, tgt, steps=4, internal_batch_size=2)
    assert calls["n"] == 2
    assert model.training and not model.sequence_mixer.training
    assert all(not m.training for m in model.sequence_mixer.modules())
    assert all(p.requires_grad == (p is not model.classifier.weight) for p in model.parameters())
    assert eng.bucket_hooks is hooks and eng.loss_scale == 1024.0
    assert all(p.grad is None for p in model.parameters())


def test_fast_path_launches_no_weight_gradient_kernel(cuda_device):
    lib = _lib.load()
    model, x, x0, tgt = _fast_setup(cuda_device, B=2, S=4)
    model.train()
    labels = _profile_labels(lib, lambda: integrated_gradients(model, x, tgt, baseline=x0, steps=2))
    assert "ig_path_inputs" in labels and "ig_accumulate" in labels and "first_conv_dgrad" in labels
    for k in ("gemm_tn", "colsum", "first_conv_wgrad", "adamw"):
        assert not any(lab.startswith(k) for lab in labels), (k, sorted(set(labels)))


# ------------------------------------------------------------------------------------------------ SleepPPGNet input gradients
def _ppg_data(B=2, seed=5):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, T_PPG, generator=g), torch.randint(0, 4, (B, 1200), generator=g)


def test_ppgnet_input_gradients_match_fp64_oracle(cuda_device):
    model = _ppg_model(cuda_device)
    for p in model.parameters():
        p.requires_grad_(False)
    x, y = _ppg_data()
    xg = x.to(cuda_device).requires_grad_(True)
    logits = model(xg)
    assert logits.grad_fn is not None
    F.cross_entropy(logits.reshape(-1, 4), y.to(cuda_device).reshape(-1)).backward()
    assert all(p.grad is None for p in model.parameters())
    sd = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    xo = x.double().requires_grad_(True)
    F.cross_entropy(PO.ppgnet_forward(xo, sd, "silu").reshape(-1, 4), y.reshape(-1)).backward()
    err = _rel(xg.grad, xo.grad)
    print(f"MEASURED ppgnet eval input gradients vs fp64 oracle: {err:.3e}")
    assert xg.grad.dtype == torch.float32 and err <= PPG_EVAL
    wrong = _rel(xg.grad, xo.grad.roll(1, dims=1))  # gradients one sample off
    assert wrong >= 10 * PPG_EVAL


def test_ppgnet_eval_graph_logits_are_bitwise_inference(cuda_device):
    model = _ppg_model(cuda_device, act="leaky")
    x, _ = _ppg_data(seed=8)
    x = x.to(cuda_device)
    with torch.no_grad():
        ref = model(x)
    got = model(x.clone().requires_grad_(True))
    assert got.grad_fn is not None and torch.equal(got.detach(), ref)
    assert torch.equal(model(x), ref)  # nothing requires grad: inference, as before


def test_ppgnet_train_input_gradients_alongside_training(cuda_device):
    model = _ppg_model(cuda_device).train()
    x, y = _ppg_data(seed=6)
    sd0 = {k: v.detach().cpu().double().clone() for k, v in model.state_dict().items()}
    xg = x.to(cuda_device).requires_grad_(True)
    F.cross_entropy(model(xg).reshape(-1, 4), y.to(cuda_device).reshape(-1)).backward()
    names = {n for n, _ in model.named_parameters()}
    sd = {k: v.clone().requires_grad_(k in names) for k, v in sd0.items()}
    xo = x.double().requires_grad_(True)
    logits, _ = PO.ppgnet_forward(xo, sd, "silu", bn_train=True)
    F.cross_entropy(logits.reshape(-1, 4), y.reshape(-1)).backward()
    err = _rel(xg.grad, xo.grad)
    perr = max(_rel(p.grad, sd[n].grad) for n, p in model.named_parameters())
    print(f"MEASURED ppgnet train input gradients vs fp64 oracle: {err:.3e} (worst parameter {perr:.3e})")
    assert err <= PPG_TRAIN and perr <= 1e-3  # parameters: the general path's gate (measured 6.3e-4)
    assert int(model.conv_block.model[0].conv1.norm.num_batches_tracked) == 1
