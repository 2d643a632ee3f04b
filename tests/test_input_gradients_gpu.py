"""-m gpu: gradients of the logits with respect to the input signals (saliency, integrated gradients), on both CUDA paths.

Fast path: ``x[name].requires_grad_()`` makes ``Wav2Sleep.forward`` run the training forward and its backward continues
through block 0 into the raw signal (``w2s_first_conv_dgrad``), with the attribution loss scale of training.py.  The
reference is fp64 CPU autograd of the oracle with the signals on the graph; activations and activation gradients of the
fast path are fp16, so the comparison is per signal by relative L2 error and cosine similarity.  General path: fp32 on
both sides, at the general path's gate (rel <= 1e-3, cos >= 0.99999).

Bounds are 3x the error measured on an NVIDIA B200 (power limit 1000 W); the measured values are in DESIGN.md,
section "Input gradients"."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import gpu_utils as GU
from conftest import SPE, make_inputs
from oracle import general_oracle as GO
from oracle import make_golden_general as G
from oracle import wav2sleep_oracle as oracle
from test_general_training_gpu import CASES as GENERAL_CASES
from test_training_gpu import _dropout_masks, _no_dropout
from wav2sleep_b200 import _lib, build_default
from wav2sleep_b200 import model as M

pytestmark = pytest.mark.gpu
CARDIO = {"ABD": "ABD", "THX": "THX", "ECG": "ECG", "PPG": "PPG"}
EOG = {"EOG-L": "EOG-L", "EOG-R": "EOG-R"}
# measured: kernel 1.1e-7; cardio rel 2.3e-2 / cos 0.99974 (B = 2 and a full night alike); EOG rel 5.9e-2 / cos 0.99829;
# B = 16 vs B = 2 rel 5.0e-3; graph vs inference logits 7.2e-3; general path 1.9e-5
KERNEL_REL = 3e-7                  # w2s_first_conv_dgrad against fp64 (fp32 sums of 64 products)
FAST_REL, FAST_COS = 6e-2, 0.9992  # fast path input gradients against fp64 oracle autograd (cardio)
EOG_REL, EOG_COS = 0.15, 0.995     # the 30-conv EOG encoders
FAST_LOGITS = 2e-2                 # forward_train logits (un-fused mixers) against the fused inference kernels, max abs
BATCH_REL = 1.5e-2                 # B = 16 pass against a B = 2 pass of the same two nights (fp16, other sum orders)
GEN_REL, GEN_COS = 1e-3, 0.99999


def _rel_cos(g, r):
    g, r = g.detach().double().cpu().reshape(-1), r.detach().double().cpu().reshape(-1)
    rel = ((g - r).norm() / r.norm()).item()
    cos = F.cosine_similarity(g, r, dim=0).item()
    return rel, cos


def _assert_exact_zeros(x, grad):
    """Samples the forward reads as 0 (non-finite) and rows of missing signals get exactly zero gradient."""
    x, grad = x.detach().cpu(), grad.detach().cpu()
    bad = ~torch.isfinite(x)
    assert (grad[bad] == 0).all()
    rows = torch.isinf(x[:, 0])
    assert (grad[rows] == 0).all()


# ------------------------------------------------------------------------------------------------ kernel
def _dgrad_ref(x, dy1, dr, w1, wds, mask, scale):
    """fp64 autograd of conv1 (k=3, pad=1) + downsample (1x1, stride 2) with the reference's zero-fill of non-finite
    samples, driven by the same fp16 dy1 / dr."""
    xd = x.double().clone().requires_grad_(True)
    xz = torch.where(torch.isfinite(xd), xd, torch.zeros_like(xd))
    y1 = F.conv1d(xz.unsqueeze(1), w1.double(), padding=1)                 # [B, 16, T]
    r = F.conv1d(xz.unsqueeze(1), wds.double(), stride=2)                   # [B, 16, T/2]
    obj = (y1 * dy1.double().transpose(1, 2)).sum() + (r * dr.double().transpose(1, 2)).sum()
    obj.backward()
    g = xd.grad * scale
    g[mask.bool().cpu()] = 0.0
    return g


def _run_dgrad(lib, x, dy1, dr, w1, wds, mask, scale):
    dx = torch.full_like(x, float("nan"))
    B, T = x.shape
    _lib.check(lib.w2s_first_conv_dgrad(x.data_ptr(), dy1.data_ptr(), dr.data_ptr(), w1.data_ptr(), wds.data_ptr(),
                                        mask.data_ptr(), dx.data_ptr(), B, T, scale, GU.stream()))
    torch.cuda.synchronize()
    return dx


@pytest.mark.parametrize("T", [2, 4, 62, 64, 66, 4098, 1200 * 1024])
def test_first_conv_dgrad_matches_fp64(cuda_device, T):
    lib = _lib.load()
    g = torch.Generator().manual_seed(T)
    B = 3
    x = torch.randn(B, T, generator=g)
    x[1] = float("-inf")                      # missing signal
    x[0, T // 2] = float("inf")               # single non-finite samples of present rows
    if T > 2:                                 # (keep an odd finite sample at T = 2, for the wrong references below)
        x[2, T - 1] = float("-inf")
    mask = torch.isinf(x[:, 0]).to(torch.uint8)
    dy1 = torch.randn(B, T, 16, generator=g).half()
    dr = torch.randn(B, T // 2, 16, generator=g).half()
    w1, wds = torch.randn(16, 1, 3, generator=g), torch.randn(16, 1, 1, generator=g)
    scale = 0.25
    dev = cuda_device
    got = _run_dgrad(lib, x.to(dev), dy1.to(dev), dr.to(dev), w1.to(dev), wds.to(dev), mask.to(dev), scale).cpu()
    ref = _dgrad_ref(x, dy1, dr, w1, wds, mask, scale)
    assert torch.isfinite(got).all()
    _assert_exact_zeros(x, got)
    rel = ((got.double() - ref).norm() / ref.norm()).item()
    print(f"first_conv_dgrad T={T}: rel L2 {rel:.3e}")
    assert rel <= KERNEL_REL, rel
    # wrong references miss by >= 10x the bound: the test can tell these defects apart
    for what, w1_, wds_, odd in (("no downsample branch", w1, wds * 0, False), ("taps reversed", w1.flip(-1), wds, False),
                                 ("odd rows fed by dr", w1, wds, True)):
        bad = _dgrad_ref(x, dy1, dr, w1_, wds_, mask, scale)
        if odd:  # dr[t // 2] added at odd t as well
            extra = (dr.double() @ wds.double().view(16)).repeat_interleave(2, dim=1)[:, :T] * scale
            extra[:, 0::2] = 0
            bad = bad + torch.where(torch.isfinite(x), extra, torch.zeros_like(extra))
            bad[mask.bool()] = 0
        miss = ((bad - ref).norm() / ref.norm()).item()
        assert miss >= 10 * KERNEL_REL, (what, miss)


def test_first_conv_dgrad_refuses_bad_arguments(cuda_device):
    lib = _lib.load()
    dev = cuda_device
    B, T = 2, 8
    x, dx = torch.zeros(B, T, device=dev), torch.zeros(B, T, device=dev)
    dy1, dr = torch.zeros(B, T, 16, device=dev).half(), torch.zeros(B, T // 2, 16, device=dev).half()
    w1, wds, m = torch.zeros(16, 3, device=dev), torch.zeros(16, device=dev), torch.zeros(B, dtype=torch.uint8, device=dev)
    ops = [x, dy1, dr, w1, wds, m, dx]
    call = lambda o, b, t: lib.w2s_first_conv_dgrad(*[None if v is None else v.data_ptr() for v in o], b, t, 1.0, GU.stream())
    for b, t, text in ((0, T, b"B=0"), (-1, T, b"B=-1"), (B, 0, b"T=0"), (B, -4, b"T=-4"), (B, 7, b"T=7")):
        assert call(ops, b, t) != 0
        assert text in lib.w2s_last_error(), lib.w2s_last_error()
    for i in range(len(ops)):
        o = list(ops)
        o[i] = None
        assert call(o, B, T) != 0
        assert b"NULL operand" in lib.w2s_last_error()
    assert call(ops, B, T) == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ fast path
def _objective(kind, logits, labels=None):
    if kind == "ce":
        return F.cross_entropy(logits.reshape(-1, logits.shape[-1]), labels.reshape(-1), ignore_index=-1)
    if kind == "logit":
        return logits[0, logits.shape[1] // 2, 1]
    return logits[..., 2].sum()


def _oracle_logits(x, params, cfg, dropout=None):
    """oracle.forward_with_grad without its detach of the signals: the oracle's stages keep x on the autograd graph."""
    d = dropout or {}
    z = oracle.signal_encoders(x, params, cfg)
    mix = oracle.epoch_mixer(z, params, cfg, drop=d.get("mix"), p=d.get("p_mix", 0.0))
    s = oracle.sequence_mixer(mix, params, cfg, drop=d.get("seq"), p=d.get("p_seq", 0.0))
    return s @ params["classifier.weight"].t() + params["classifier.bias"]


def _oracle_input_grads(model, x, cfg, kind, labels, dropout=None):
    params = {k: v.detach().double().clone() for k, v in model.state_dict().items()}
    xs = {k: v.double().clone().requires_grad_(True) for k, v in x.items()}
    lo = _oracle_logits(xs, params, cfg, dropout=dropout)
    _objective(kind, lo, labels).backward()
    return {k: v.grad for k, v in xs.items()}, lo.detach()


def _fast_input_grads(model, x, kind, labels, dev):
    xs = {k: v.to(dev).requires_grad_(True) for k, v in x.items()}
    logits = model(xs)
    assert logits.grad_fn is not None
    _objective(kind, logits, None if labels is None else labels.to(dev)).backward()
    torch.cuda.synchronize()
    return {k: v.grad for k, v in xs.items()}, logits.detach()


def _compare_fast(got, ref, x, label, rel_max=FAST_REL, cos_min=FAST_COS):
    for n in ref:
        assert got[n] is not None and got[n].dtype == torch.float32 and got[n].shape == x[n].shape, n
        assert torch.isfinite(got[n]).all(), n
        _assert_exact_zeros(x[n], got[n])
        if ref[n].norm() == 0:
            assert (got[n] == 0).all(), n
            continue
        rel, cos = _rel_cos(got[n], ref[n])
        print(f"{label} {n}: rel L2 {rel:.3e} cos {cos:.6f}")
        assert rel <= rel_max and cos >= cos_min, (label, n, rel, cos)


@pytest.mark.parametrize("kind", ["ce", "logit", "sum"])
@pytest.mark.parametrize("mode", ["eval", "train_dropout"])
def test_fast_path_input_gradients_match_fp64_oracle(cuda_device, mode, kind):
    B, S = 2, 24
    model = build_default(CARDIO, 4, seed=0)
    x = make_inputs(CARDIO, B, S, masked=[("ABD", 0), ("PPG", 1)], seed=5)
    x["ECG"][0, 1000] = float("inf")
    x["THX"][1, 77] = float("-inf")
    labels = torch.randint(0, 4, (B, S), generator=torch.Generator().manual_seed(1))
    labels[0, ::5] = -1
    drop = None
    model = model.to(cuda_device)
    if mode == "train_dropout":
        eng = model._get_engine()
        eng.dropout_seed = 4321
        drop = _dropout_masks(model, eng, B, S, len(CARDIO) + 1, eng.dropout_seed, cuda_device)
        model.train()
    else:
        model.eval()
    for p in model.parameters():  # attribution on a frozen model: no weight gradient at all
        p.requires_grad_(False)
    got, logits = _fast_input_grads(model, x, kind, labels, cuda_device)
    ref, lo = _oracle_input_grads(model.cpu(), x, oracle.cardio_config(), kind, labels, dropout=drop)
    assert (logits.cpu().double() - lo).abs().max().item() < 2e-2
    _compare_fast(got, ref, x, f"{mode}/{kind}")


def test_fast_path_full_night_and_eog(cuda_device):
    """One 10-h cardio night (1.2 M ECG / PPG samples, 30 convs per encoder) and the 10-block EOG encoders."""
    for smap, cfg, n_cls, B, S, kind in ((CARDIO, oracle.cardio_config(), 4, 1, 1200, "sum"),
                                         (EOG, oracle.eog_config(), 5, 2, 4, "ce")):
        model = build_default(smap, n_cls, seed=0).to(cuda_device).eval()
        x = make_inputs(smap, B, S, seed=11)
        labels = torch.randint(0, n_cls, (B, S), generator=torch.Generator().manual_seed(2))
        got, _ = _fast_input_grads(model, x, kind, labels, cuda_device)
        ref, _ = _oracle_input_grads(model.cpu(), x, cfg, kind, labels)
        if B == 1:
            _compare_fast(got, ref, x, "cardio night")
        else:
            _compare_fast(got, ref, x, "EOG", EOG_REL, EOG_COS)


def test_fast_path_batch_scale(cuda_device):
    """B = 16 full cardio nights with a summed-logit objective: the attribution loss scale keeps every gradient finite,
    and nights 0-1 get what a B = 2 pass of those two nights gives them."""
    model = build_default(CARDIO, 4, seed=0).to(cuda_device).eval()
    for p in model.parameters():
        p.requires_grad_(False)
    x = make_inputs(CARDIO, 16, 1200, masked=[("THX", 3)], seed=21)
    big, _ = _fast_input_grads(model, x, "sum", None, cuda_device)
    eng = model._get_engine()
    assert eng.last_loss_scale == 4.0  # max |dlogits| = 1 -> [4, 8)
    small, _ = _fast_input_grads(model, {k: v[:2] for k, v in x.items()}, "sum", None, cuda_device)
    rels = {}
    for n in x:
        assert torch.isfinite(big[n]).all(), n
        rels[n], cos = _rel_cos(big[n][:2], small[n])
        print(f"B=16 vs B=2 {n}: rel {rels[n]:.3e} cos {cos:.7f}")
    assert max(rels.values()) <= BATCH_REL, rels
    del big, small


def test_attribution_loss_scale_policy():
    from wav2sleep_b200.training import TrainEngine
    for m, s in ((1.0, 4.0), (1.5, 4.0), (0.99, 8.0), (8.0, 0.5), (7.99, 1.0), (1e-30, 2.0 ** 24), (3.0, 2.0)):
        assert TrainEngine.attribution_loss_scale(m) == s, (m, s)
        assert 4 <= m * s < 8 or s == 2.0 ** 24


def test_zero_objective_gradient_launches_nothing(cuda_device):
    model = build_default({"ECG": "ECG"}, 4, seed=0).to(cuda_device).eval()
    x = {k: v.to(cuda_device).requires_grad_(True) for k, v in make_inputs({"ECG": "ECG"}, 2, 3, seed=1).items()}
    logits = model(x)
    lib = _lib.load()
    torch.cuda.synchronize()
    n0 = lib.w2s_launch_count()
    (logits * 0).sum().backward()
    torch.cuda.synchronize()
    assert lib.w2s_launch_count() == n0 + 1  # the max |dlogits| reduction that finds the zero, and nothing else
    assert (x["ECG"].grad == 0).all()
    assert all(p.grad is not None and (p.grad == 0).all() for p in model.parameters())


def test_nan_objective_gradient_propagates(cuda_device):
    """A NaN in d(objective)/d(logits) reaches the input and parameter gradients, as with torch autograd: the max |dlogits|
    that picks the loss scale must not drop the NaN and take the exact-zero shortcut above."""
    model = build_default({"ECG": "ECG"}, 4, seed=0).to(cuda_device).eval()
    x = {k: v.to(cuda_device).requires_grad_(True) for k, v in make_inputs({"ECG": "ECG"}, 2, 3, seed=1).items()}
    logits = model(x)
    w = torch.zeros_like(logits)
    w[0, 1, 2] = float("nan")
    (logits * w).sum().backward()
    torch.cuda.synchronize()
    assert torch.isnan(x["ECG"].grad).any()
    no_nan = [n for n, p in model.named_parameters() if not torch.isnan(p.grad).any()]
    assert not no_nan, no_nan


def _profile_labels(lib, fn):
    lib.w2s_profile_enable(1)
    try:
        fn()
        torch.cuda.synchronize()
        buf, ms = C.create_string_buffer(64), C.c_float()
        out = []
        for i in range(lib.w2s_profile_count()):
            _lib.check(lib.w2s_profile_get(i, buf, 64, C.byref(ms), None, None))
            out.append(buf.value.decode())
        return out
    finally:
        lib.w2s_profile_enable(0)


def test_frozen_parameters_get_no_gradient_and_no_weight_gradient_launch(cuda_device):
    lib = _lib.load()
    model = build_default(CARDIO, 4, seed=0).to(cuda_device).eval()
    for p in model.parameters():
        p.requires_grad_(False)
    x = {k: v.to(cuda_device).requires_grad_(True) for k, v in make_inputs(CARDIO, 2, 6, seed=2).items()}

    def run():
        model(x)[..., 0].sum().backward()
    labels = _profile_labels(lib, run)
    assert "first_conv_dgrad" in labels
    for k in ("gemm_tn", "colsum", "first_conv_wgrad"):
        assert not any(l.startswith(k) for l in labels), (k, sorted(set(labels)))
    assert all(p.grad is None for p in model.parameters())
    assert all(v.grad is not None for v in x.values())
    # general path (a BatchNorm model in eval(): differentiable with respect to its inputs)
    gm = _bn_model(cuda_device)
    for p in gm.parameters():
        p.requires_grad_(False)
    xg = {k: v.to(cuda_device).requires_grad_(True) for k, v in G.make_inputs(_BN_CASE).items()}
    labels = _profile_labels(lib, lambda: gm(xg).sum().backward())
    assert "gen_conv_dgrad" in labels and "gen_conv_wgrad" not in labels and "gen_bn_eval_bwd" not in labels
    assert all(p.grad is None for p in gm.parameters())


def test_frozen_encoders_leave_mixer_gradients_unchanged(cuda_device):
    """Skipping the encoders' backward (frozen, no input gradient) changes nothing upstream of them."""
    x = {k: v.to(cuda_device) for k, v in make_inputs(CARDIO, 2, 12, masked=[("PPG", 0)], seed=3).items()}
    labels = torch.randint(0, 4, (2, 12), generator=torch.Generator().manual_seed(3)).to(cuda_device)
    grads = []
    for freeze in (False, True):
        model = build_default(CARDIO, 4, seed=0)
        _no_dropout(model)
        model = model.to(cuda_device).train()
        for p in model.signal_encoders.parameters():
            p.requires_grad_(not freeze)
        F.cross_entropy(model(x).view(-1, 4), labels.view(-1)).backward()
        torch.cuda.synchronize()
        grads.append({n: p.grad for n, p in model.named_parameters()})
    for n, g in grads[0].items():
        if n.startswith("signal_encoders."):
            assert grads[1][n] is None, n
            continue
        d = (grads[1][n] - g).norm().item() / max(g.norm().item(), 1e-30)
        assert d < 2e-3, (n, d)  # atomics order of the fp32 accumulation


def test_fast_path_graph_logits_match_inference(cuda_device):
    model = build_default(CARDIO, 4, seed=0).to(cuda_device).eval()
    x = {k: v.to(cuda_device) for k, v in make_inputs(CARDIO, 2, 24, masked=[("ABD", 1)], seed=4).items()}
    with torch.no_grad():
        ref = model(x)
    got = model({k: v.clone().requires_grad_(True) for k, v in x.items()})
    assert got.grad_fn is not None
    diff = (got.detach() - ref).abs().max().item()
    print(f"forward_train (un-fused mixers) vs fused inference logits: max abs {diff:.3e}")
    assert diff <= FAST_LOGITS
    with torch.no_grad():  # with nothing requiring grad, the inference kernels run as before
        assert torch.equal(model(x), ref)


# ------------------------------------------------------------------------------------------------ general path
_BN_CASE = {**G.CASES["general_causal_batch_relu"],
            "enc": {**G.CASES["general_causal_batch_relu"]["enc"], "activation": "silu"},
            "seq": {**G.CASES["general_causal_batch_relu"]["seq"], "activation": "silu"}}


def _bn_model(dev):
    model = G.build(M, _BN_CASE)
    G.perturb(model, _BN_CASE["seed"])
    return model.to(dev).eval()


def _general_compare(model, case, dev, label, check_params=False):
    x = G.make_inputs(case)
    y = torch.randint(0, case["num_classes"], (case["B"], case["S"]), generator=torch.Generator().manual_seed(0))
    xs = {k: v.to(dev).requires_grad_(True) for k, v in x.items()}
    model.zero_grad(set_to_none=True)
    logits = model(xs)
    F.cross_entropy(logits.view(-1, logits.shape[-1]), y.to(dev).view(-1)).backward()
    names = dict(model.named_parameters())
    sd = {k: v.detach().cpu().float().clone().requires_grad_(check_params and k in names)
          for k, v in model.state_dict().items()}
    xo = {k: v.clone().requires_grad_(True) for k, v in x.items()}
    lo = GO.forward(xo, sd, GO.config(case))
    F.cross_entropy(lo.view(-1, lo.shape[-1]), y.view(-1)).backward()
    pairs = [(n, xs[n].grad, xo[n].grad) for n in x]
    if check_params:
        pairs += [(n, p.grad, sd[n].grad) for n, p in names.items()]
    worst = 0.0
    for n, g, r in pairs:
        assert g is not None, n
        if n in x:
            _assert_exact_zeros(x[n], g)
        if r.norm() == 0:
            assert g.abs().max().item() == 0.0, n
            continue
        rel, cos = _rel_cos(g, r)
        worst = max(worst, rel)
        assert rel <= GEN_REL and cos >= GEN_COS, (label, n, rel, cos)
    print(f"{label}: worst rel {worst:.3e} over {len(pairs)} tensors")


@pytest.mark.parametrize("name", list(GENERAL_CASES))
def test_general_path_input_gradients_match_oracle(cuda_device, name):
    case = GENERAL_CASES[name]
    model = G.build(M, case)
    G.perturb(model, case["seed"])
    model = model.to(cuda_device).eval()
    assert not model.fast_path
    _general_compare(model, case, cuda_device, name)


def test_general_path_batchnorm_eval_gradients(cuda_device):
    """A SiLU BatchNorm model in eval(): input gradients and every parameter gradient, BatchNorm weight / bias included
    (w2s_gen_bn_eval_bwd); train() with grad still raises."""
    model = _bn_model(cuda_device)
    _general_compare(model, _BN_CASE, cuda_device, "batchnorm eval", check_params=True)
    bn = [m for m in model.modules() if isinstance(m, torch.nn.BatchNorm1d)]
    assert bn and all(m.weight.grad is not None and m.weight.grad.abs().sum() > 0 for m in bn)
    x = {k: v.to(cuda_device).requires_grad_(True) for k, v in G.make_inputs(_BN_CASE).items()}
    with pytest.raises(NotImplementedError, match="BatchNorm"):
        model.train()(x)


def test_general_eval_graph_logits_are_bitwise_the_inference_logits(cuda_device):
    for case in (GENERAL_CASES["general_shared_embed_registers"], _BN_CASE):
        model = G.build(M, case)
        G.perturb(model, case["seed"])
        model = model.to(cuda_device).eval()
        x = {k: v.to(cuda_device) for k, v in G.make_inputs(case).items()}
        with torch.no_grad():
            ref = model(x)
        got = model({k: v.clone().requires_grad_(True) for k, v in x.items()})
        assert got.grad_fn is not None and torch.equal(got.detach(), ref)


@pytest.mark.parametrize("which", ["bn_chunk_causal", "general_causalconv_layer_silu"])
def test_causal_model_has_no_gradient_from_the_future(cuda_device, which):
    case = _BN_CASE if which == "bn_chunk_causal" else GENERAL_CASES[which]
    model = G.build(M, case)
    G.perturb(model, case["seed"])
    model = model.to(cuda_device).eval()
    x = {k: v.to(cuda_device).requires_grad_(True) for k, v in G.make_inputs(case).items()}
    s = case["S"] // 2
    model(x)[:, s, :].sum().backward()
    for n, v in x.items():
        after = v.grad[:, (s + 1) * SPE[n]:]
        before = v.grad[:, :(s + 1) * SPE[n]]
        assert (after == 0).all(), n
        present = ~torch.isinf(v.detach()[:, 0])
        assert (before[present].abs().sum(dim=-1) > 0).all(), n
