"""-m gpu: training path.  Gradients of every parameter against torch autograd over the CPU oracle (fp32), plus the
building blocks (cross entropy, clip + AdamW) against torch; the weight-gradient GEMM and the optimizer kernels are held
to fp64 one call at a time in test_train_kernels_gpu.py.

Tolerances: activations and activation gradients are stored in fp16 (the gradients loss-scaled by a power of two, see
training.py) and the whole-night InstanceNorm backward couples millions of positions, so parameter gradients are
compared per tensor by relative L2 error and cosine similarity against fp32 autograd:
  * small batches (B = 2, S = 24; few positions per weight, so fp16 rounding does not average out): rel <= REL_SMALL,
    cos >= COS_SMALL;
  * one full 10-h night with d(loss)/d(logits) scaled exactly as in the benchmarked batches (B = 16 cardio, B = 32
    ECG-only): rel <= REL_FULL, cos >= COS_FULL on all 183 tensors.
Where the tolerance comes from: rounding only the FORWARD activations / operands to fp16 inside the fp32 autograd graph
of the oracle (straight-through rounding, exact fp32 backward; tools/emulate_16bit.py --grad) already moves the block-0
and block-1 weight gradients by 2.0-2.9e-2 (median over all tensors 1.7e-3): they are sums over 1.2 M positions that
nearly cancel, so a 1e-3 perturbation of the deep activations shows up 20x larger there.  Measured on the GPU: median
2e-3 .. 1e-2, worst 2.9-3.8e-2 (cnn.0.conv1 / cnn.0.downsample, 48 and 16 elements), cosine >= 0.9993.  The floor of a
16-bit forward is therefore ~3e-2 on those two tensors; REL_FULL sits above it with margin, the cosine gate (0.999)
is the tight one.
Dropout is tested both off (p = 0 on both sides) and on: the CUDA path's counter-based keep masks are dumped through the
``w2s_dropout`` test hook and handed to the oracle, which applies exactly those masks in the reference's training graph."""
import ctypes as C

import pytest
import torch

import gpu_utils as G
from conftest import make_inputs
from oracle import wav2sleep_oracle as oracle
from wav2sleep_b200 import _lib, build_default

pytestmark = pytest.mark.gpu
CARDIO = {"ABD": "ABD", "THX": "THX", "ECG": "ECG", "PPG": "PPG"}
EOG = {"EOG-L": "EOG-L", "EOG-R": "EOG-R"}
REL_SMALL, COS_SMALL = 8e-2, 0.997
REL_FULL, COS_FULL = 5e-2, 0.999


def test_ce_and_adamw_match_torch(cuda_device):
    lib = _lib.load()
    torch.manual_seed(0)
    N, Cn = 5000, 4
    logits = torch.randn(N, Cn, device=cuda_device)
    labels = torch.randint(0, Cn, (N,), device=cuda_device)
    labels[::7] = -1
    scratch = torch.zeros(2, dtype=torch.float64, device=cuda_device)
    loss = torch.zeros(1, device=cuda_device)
    dlog = torch.empty_like(logits)
    _lib.check(lib.w2s_ce_fwd_bwd(logits.data_ptr(), labels.data_ptr(), N, Cn, -1, scratch.data_ptr(), loss.data_ptr(),
                                  dlog.data_ptr(), G.stream()))
    lt = logits.clone().requires_grad_(True)
    ref = torch.nn.functional.cross_entropy(lt, labels, ignore_index=-1)
    ref.backward()
    assert abs(loss.item() - ref.item()) < 1e-5
    assert (dlog - lt.grad).abs().max().item() < 1e-7
    # clip + AdamW, 3 steps
    n = 100_003
    p0 = torch.randn(n, device=cuda_device)
    p_ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([p_ref], lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4)
    p, mom, var = p0.clone(), torch.zeros(n, device=cuda_device), torch.zeros(n, device=cuda_device)
    nsq = torch.zeros(1, dtype=torch.float64, device=cuda_device)
    ema, ema_ref, decay = p0.clone(), p0.clone(), 0.99  # EMACallback: ema = decay * ema + (1 - decay) * p after each step
    for step in range(1, 4):
        g = torch.randn(n, device=cuda_device) * 0.05
        p_ref.grad = g.clone()
        torch.nn.utils.clip_grad_norm_([p_ref], 1.0)
        opt.step()
        ema_ref.mul_(decay).add_(p_ref.detach(), alpha=1 - decay)
        nsq.zero_()
        _lib.check(lib.w2s_sumsq(g.data_ptr(), n, nsq.data_ptr(), G.stream()))
        _lib.check(lib.w2s_adamw_step(p.data_ptr(), g.data_ptr(), mom.data_ptr(), var.data_ptr(), n, nsq.data_ptr(), 1e-3,
                                      0.9, 0.999, 1e-8, 1e-4, 1.0, 1.0, step, ema.data_ptr(), decay, G.stream()))
    torch.cuda.synchronize()
    assert (p - p_ref.detach()).abs().max().item() < 2e-6
    assert (ema - ema_ref).abs().max().item() < 2e-6


def test_fused_adamw_ema_swap(cuda_device):
    """FusedAdamW(ema_decay=...) mirrors EMACallback: update after every step from start_step on, swap for evaluation."""
    from wav2sleep_b200.optim import FusedAdamW
    torch.manual_seed(0)
    lin = torch.nn.Linear(8, 8).to(cuda_device)
    opt = FusedAdamW(lin.parameters(), lr=1e-2, weight_decay=0.0, ema_decay=0.5, ema_start_step=2)
    w0 = lin.weight.detach().clone()
    hist = []
    for _ in range(3):
        opt.zero_grad()
        lin(torch.randn(4, 8, device=cuda_device)).pow(2).sum().backward()
        opt.step()
        hist.append(lin.weight.detach().clone())
    # steps 2 and 3 update the average (start_step = 2): ema = 0.5 * (0.5 * w0 + 0.5 * w2) + 0.5 * w3
    expect = 0.5 * (0.5 * w0 + 0.5 * hist[1]) + 0.5 * hist[2]
    opt.swap_to_ema()
    assert (lin.weight.detach() - expect).abs().max().item() < 1e-6
    with pytest.raises(RuntimeError):
        opt.step()
    opt.swap_to_original()
    assert torch.equal(lin.weight.detach(), hist[2])
    with pytest.raises(ValueError):
        FusedAdamW(lin.parameters(), ema_decay=1.5)


def _grad_report(model, grads_ref):
    rows = []
    for name, p in model.named_parameters():
        g, r = p.grad.detach().float().cpu(), grads_ref[name]
        rn = r.norm().item()
        rel = (g - r).norm().item() / max(rn, 1e-12)
        cos = torch.nn.functional.cosine_similarity(g.flatten(), r.flatten(), dim=0).item() if rn > 0 else 1.0
        rows.append((name, rn, rel, cos))
    return rows


def _dropout_masks(model, eng, B, S, D, seed, device):
    """The keep masks the CUDA training path will use for this seed, in the oracle's layout."""
    N = B * S
    p_mix, out = float(model.epoch_mixer.dropout), {"p_mix": float(model.epoch_mixer.dropout), "mix": [], "seq": []}
    for l in range(model.epoch_mixer.num_layers):
        mk = lambda site, n: eng.dropout_mask(n, 8 * l + site, p_mix, seed, device).cpu()
        out["mix"].append({"attn": mk(0, (N * 8 * D * D + 7) // 8 * 8)[:N * 8 * D * D].view(N, 8, D, D),
                           "sa": mk(1, N * D * 128).view(N, D, 128), "ff": mk(2, N * D * 512).view(N, D, 512),
                           "out": mk(3, N * D * 128).view(N, D, 128)})
    blocks = model.sequence_mixer.dilated_convs
    out["p_seq"] = float(blocks[0].dropout.p)
    for bi in range(len(blocks)):
        out["seq"].append(eng.dropout_mask(N * 128, 64 + bi, out["p_seq"], seed, device).cpu().view(B, S, 128))
    return out


@pytest.mark.parametrize("masked,dropout", [(False, False), (True, False), (True, True)])
def test_parameter_gradients_match_oracle_autograd(cuda_device, masked, dropout):
    torch.manual_seed(0)
    B, S = 2, 24
    model = build_default(CARDIO, 4, seed=0)
    x = make_inputs(CARDIO, B, S, masked=[("ABD", 0), ("PPG", 1)] if masked else [], seed=5)
    labels = torch.randint(0, 4, (B, S))
    labels[0, ::5] = -1
    drop = None
    if dropout:  # default config: p = 0.1 in both mixers; fixed step seed so that the masks can be dumped up front
        eng = model._get_engine()
        eng.dropout_seed = 1234567
        drop = _dropout_masks(model, eng, B, S, len(CARDIO) + 1, eng.dropout_seed, cuda_device)
        kept = drop["mix"][0]["ff"].float().mean().item()
        assert abs(kept - 0.9) < 0.01, kept  # keep rate of the generator
    else:
        model.epoch_mixer.dropout = 0.0
        for blk in model.sequence_mixer.dilated_convs:
            blk.dropout.p = 0.0
    # oracle gradients (fp32 CPU autograd)
    params = {k: v.detach().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    lo = oracle.forward_with_grad(x, params, oracle.cardio_config(), dropout=drop)
    loss_ref = torch.nn.functional.cross_entropy(lo.view(-1, 4), labels.view(-1), ignore_index=-1)
    loss_ref.backward()
    grads_ref = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in params.items()}
    # CUDA path
    model = model.to(cuda_device).train()
    logits = model({k: v.to(cuda_device) for k, v in x.items()})
    assert logits.requires_grad
    loss = torch.nn.functional.cross_entropy(logits.view(-1, 4), labels.to(cuda_device).view(-1), ignore_index=-1)
    loss.backward()
    torch.cuda.synchronize()
    assert abs(loss.item() - loss_ref.item()) < 5e-3
    rows = _grad_report(model, grads_ref)
    worst = sorted(rows, key=lambda r: -r[2])
    for name, rn, rel, cos in worst[:12] + worst[-4:]:
        print(f"{name:70s} |g_ref| {rn:.3e} rel {rel:.3e} cos {cos:.5f}")
    import statistics
    print("median rel", statistics.median(r[2] for r in rows if r[1] > 0))
    _assert_grads(model, rows, REL_SMALL, COS_SMALL)


def test_fused_norm_backward_equals_separate_pass(cuda_device):
    """W2S_PRO_DNORM: the InstanceNorm backward of a layer's gradient computed inside the prologue of the data-gradient
    conv that consumes it (and written out for the weight gradient) must give the gradients of the separate
    enc_norm_bwd pass - same fp32 formula, same fp16 rounding of dy - for stride-1 and zero-stuffed stride-2 layers, with
    a masked night and ragged lengths (S = 13: tile tails and halos)."""
    torch.manual_seed(0)
    B, S = 3, 13
    x = {k: v.to(cuda_device) for k, v in make_inputs(CARDIO, B, S, masked=[("ABD", 0), ("ECG", 2)], seed=9).items()}
    labels = torch.randint(0, 4, (B, S), device=cuda_device)
    grads = {}
    for fuse in (True, False):
        model = build_default(CARDIO, 4, seed=0)
        _no_dropout(model)
        model = model.to(cuda_device).train()
        model._get_engine().fuse_norm_bwd = fuse
        loss = torch.nn.functional.cross_entropy(model(x).view(-1, 4), labels.view(-1))
        loss.backward()
        torch.cuda.synchronize()
        grads[fuse] = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
    worst = 0.0
    for n, g in grads[False].items():
        d = (grads[True][n] - g).norm().item()
        ref = g.norm().item()
        if ref == 0.0:
            assert d == 0.0, n
            continue
        worst = max(worst, d / ref)
        assert d / ref < 2e-3, (n, d / ref)  # atomics order in the fp32 weight-gradient accumulation is the only difference
    print(f"fused vs separate InstanceNorm backward: worst relative gradient difference {worst:.2e}")


def _assert_grads(model, rows, rel_max, cos_min):
    import statistics
    worst = sorted(rows, key=lambda r: -r[2])
    for name, rn, rel, cos in worst[:12] + worst[-4:]:
        print(f"{name:70s} |g_ref| {rn:.3e} rel {rel:.3e} cos {cos:.5f}")
    print("median rel", statistics.median(r[2] for r in rows if r[1] > 0), "worst rel", worst[0][2],
          "min cos", min(r[3] for r in rows))
    for name, rn, rel, cos in rows:
        if rn == 0.0:  # parameters of fully masked encoders get exact zero gradients
            assert model.get_parameter(name).grad.abs().max().item() == 0.0, name
            continue
        assert rel < rel_max and cos > cos_min, (name, rn, rel, cos)


def _no_dropout(model):
    model.epoch_mixer.dropout = 0.0
    for blk in model.sequence_mixer.dilated_convs:
        blk.dropout.p = 0.0


def _oracle_grads(model, x, labels, cfg, n_classes, loss_div=1.0):
    params = {k: v.detach().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    lo = oracle.forward_with_grad(x, params, cfg)
    loss = torch.nn.functional.cross_entropy(lo.view(-1, n_classes), labels.view(-1), ignore_index=-1) / loss_div
    loss.backward()
    return loss.item(), {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in params.items()}


@pytest.mark.parametrize("case,batch,masked", [("cardio_b16", 16, ()), ("ecg_only_b32", 32, ("ABD", "THX", "PPG"))])
def test_full_night_gradients_at_benchmark_scale(cuda_device, case, batch, masked):
    """BASELINE configs[3] / [4] numerics: one 10-h night whose d(loss)/d(logits) is 1/batch of its own mean-CE gradient,
    i.e. exactly what this night sees inside a batch of `batch` nights (mean over batch * 1200 epochs), with the loss scale
    the engine picks for that batch.  Unscaled, every encoder activation gradient would be an fp16 subnormal
    (median 1e-7); all 183 parameter gradients must match fp32 autograd of the reference graph."""
    torch.manual_seed(0)
    S = 1200
    model = build_default(CARDIO, 4, seed=0)
    _no_dropout(model)
    x = make_inputs(CARDIO, 1, S, masked=[(n, 0) for n in masked], seed=11)
    labels = torch.randint(0, 4, (1, S))
    labels[torch.rand(1, S) < 0.05] = -1
    loss_ref, grads_ref = _oracle_grads(model, x, labels, oracle.cardio_config(), 4, loss_div=float(batch))
    model = model.to(cuda_device).train()
    eng = model._get_engine()
    eng.loss_scale = eng.auto_loss_scale(batch * S)
    logits = model({k: v.to(cuda_device) for k, v in x.items()})
    loss = torch.nn.functional.cross_entropy(logits.view(-1, 4), labels.to(cuda_device).view(-1), ignore_index=-1) / batch
    loss.backward()
    torch.cuda.synchronize()
    assert eng.last_loss_scale == eng.auto_loss_scale(batch * S) and eng.last_loss_scale >= 2 ** 16
    assert abs(loss.item() - loss_ref) < 5e-3 / batch
    _assert_grads(model, _grad_report(model, grads_ref), REL_FULL, COS_FULL)


def test_unscaled_backward_underflows_at_benchmark_scale(cuda_device):
    """Why the loss scale exists: with loss_scale = 1 the same full-night backward loses the encoder gradients
    (fp16 subnormals), so the scaled run above is not passing by accident."""
    torch.manual_seed(0)
    S, batch = 1200, 16
    sig = {"ABD": "ABD"}
    model = build_default(sig, 4, seed=0)
    _no_dropout(model)
    x = make_inputs(sig, 1, S, seed=11)
    labels = torch.randint(0, 4, (1, S))
    _, grads_ref = _oracle_grads(model, x, labels, oracle.OracleConfig(signal_map=sig, num_classes=4), 4, float(batch))
    model = model.to(cuda_device).train()
    eng = model._get_engine()
    worst = {}
    for scale in (1.0, None):
        eng.loss_scale = scale if scale is not None else eng.auto_loss_scale(batch * S)
        model.zero_grad()
        logits = model({k: v.to(cuda_device) for k, v in x.items()})
        (torch.nn.functional.cross_entropy(logits.view(-1, 4), labels.to(cuda_device).view(-1)) / batch).backward()
        rows = [r for r in _grad_report(model, grads_ref) if "encoders" in r[0]]
        worst[scale] = max(r[2] for r in rows)
    print("worst encoder rel error: unscaled", worst[1.0], "scaled", worst[None])
    assert worst[None] < REL_FULL and worst[1.0] > 3 * worst[None]


def test_eog_model_gradients(cuda_device):
    """The 10-block EOG encoders (30 convs deep, 128-channel tail blocks) through the same backward."""
    torch.manual_seed(0)
    B, S = 2, 4
    model = build_default(EOG, 5, seed=0)
    _no_dropout(model)
    x = make_inputs(EOG, B, S, seed=3)
    labels = torch.randint(0, 5, (B, S))
    loss_ref, grads_ref = _oracle_grads(model, x, labels, oracle.eog_config(), 5)
    model = model.to(cuda_device).train()
    logits = model({k: v.to(cuda_device) for k, v in x.items()})
    loss = torch.nn.functional.cross_entropy(logits.view(-1, 5), labels.to(cuda_device).view(-1), ignore_index=-1)
    loss.backward()
    torch.cuda.synchronize()
    assert abs(loss.item() - loss_ref) < 5e-3
    _assert_grads(model, _grad_report(model, grads_ref), REL_SMALL, COS_SMALL)


def test_two_forwards_before_backward(cuda_device):
    """Saved activations live with the autograd graph (ctx), not in one engine slot: forward(a), forward(b),
    backward(a), backward(b) gives the gradients of a and of b, as with torch autograd."""
    sig = {"ABD": "ABD"}
    model = build_default(sig, 4, seed=0)
    _no_dropout(model)
    model = model.to(cuda_device).train()
    xa = {k: v.to(cuda_device) for k, v in make_inputs(sig, 2, 8, seed=1).items()}
    xb = {k: v.to(cuda_device) for k, v in make_inputs(sig, 2, 8, seed=2).items()}
    w = model.classifier.weight

    def grad_of(x):
        model.zero_grad()
        model(x).square().sum().backward()
        return {n: p.grad.detach().clone() for n, p in model.named_parameters()}

    ga, gb = grad_of(xa), grad_of(xb)
    model.zero_grad()
    la, lb = model(xa).square().sum(), model(xb).square().sum()
    la.backward()
    got_a = {n: p.grad.detach().clone() for n, p in model.named_parameters()}
    lb.backward()  # accumulates
    for n, p in model.named_parameters():
        # (weight gradients are sums over up to 1e5 positions accumulated with fp32 atomics: two runs of the same
        #  backward differ by the summation order; a backward through the WRONG forward's activations differs by O(1))
        scale = ga[n].abs().max().item() + 1e-6
        assert (got_a[n] - ga[n]).abs().max().item() <= 1e-3 * scale, n
        assert (p.grad - (ga[n] + gb[n])).abs().max().item() <= 2e-3 * scale, n
    with pytest.raises(RuntimeError):
        la.backward()  # a graph can be back-propagated once
    assert w.grad is not None


def test_fused_adamw_checkpoint_resume_and_realias(cuda_device):
    """state_dict()/load_state_dict() carry the Adam moments, the step count and the EMA; a foreign model.zero_grad()
    (p.grad = None -> fresh autograd tensors) does not make step() read a stale flat buffer."""
    from wav2sleep_b200.optim import FusedAdamW
    torch.manual_seed(0)

    def make():
        torch.manual_seed(1)
        return torch.nn.Sequential(torch.nn.Linear(8, 16), torch.nn.Linear(16, 4)).to(cuda_device)

    xs = [torch.randn(5, 8, device=cuda_device) for _ in range(6)]
    ref = make()
    opt_ref = FusedAdamW(ref.parameters(), lr=1e-2, weight_decay=1e-2, max_grad_norm=1.0, ema_decay=0.9)
    ckpt = None
    for i, x in enumerate(xs):
        if i == 3:
            ckpt = (ref.state_dict(), opt_ref.state_dict())
            ckpt = ({k: v.clone() for k, v in ckpt[0].items()}, ckpt[1])
        ref.zero_grad()  # set_to_none=True: breaks the alias on purpose; step() must gather the fresh gradients
        ref(x).square().sum().backward()
        opt_ref.step()
    assert "fused" in ckpt[1] and ckpt[1]["fused"]["step"] == 3
    resumed = make()
    resumed.load_state_dict(ckpt[0])
    opt = FusedAdamW(resumed.parameters(), lr=1e-2, weight_decay=1e-2, max_grad_norm=1.0, ema_decay=0.9)
    opt.load_state_dict(ckpt[1])
    for x in xs[3:]:
        opt.zero_grad()
        resumed(x).square().sum().backward()
        opt.step()
    for (n, a), (_, b) in zip(ref.named_parameters(), resumed.named_parameters()):
        assert torch.allclose(a, b, rtol=0, atol=1e-7), n
    assert torch.allclose(opt.ema, opt_ref.ema, rtol=0, atol=1e-7)
    # plain torch AdamW on the same gradients agrees as well (checks that zero_grad()'d gradients were really used)
    tref = make()
    topt = torch.optim.AdamW(tref.parameters(), lr=1e-2, weight_decay=1e-2)
    for x in xs:
        tref.zero_grad()
        tref(x).square().sum().backward()
        torch.nn.utils.clip_grad_norm_(tref.parameters(), 1.0)
        topt.step()
    for (n, a), (_, b) in zip(ref.named_parameters(), tref.named_parameters()):
        assert torch.allclose(a, b, rtol=0, atol=2e-6), n
    with pytest.raises(ValueError):
        FusedAdamW([{"params": list(ref[0].parameters())}, {"params": list(ref[1].parameters()), "lr": 1.0}])


def test_training_reduces_loss(cuda_device):
    """A few clip + AdamW steps on one fixed batch through the public training API lower the loss."""
    from wav2sleep_b200.optim import FusedAdamW
    torch.manual_seed(0)
    model = build_default({"ECG": "ECG", "ABD": "ABD"}, 4, seed=0).to(cuda_device).train()
    x = {k: v.to(cuda_device) for k, v in make_inputs({"ECG": "ECG", "ABD": "ABD"}, 2, 16, seed=9).items()}
    y = torch.randint(0, 4, (2, 16), device=cuda_device)
    opt = FusedAdamW(model.parameters(), lr=1e-3, weight_decay=1e-4, max_grad_norm=1.0)
    losses = []
    for _ in range(8):
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(model(x).view(-1, 4), y.view(-1))
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print(losses)
    assert losses[-1] < losses[0] - 0.05


def test_lightning_shaped_module_fit_with_masker(cuda_device):
    """SleepLightningModule-shaped harness: polarity flip + SignalMasker + CE + backward + fused clip/AdamW + scheduler."""
    from wav2sleep_b200.optim import ExpWarmUpScheduler, FusedAdamW
    from wav2sleep_b200.trainer import SignalMasker, SleepLightningModule
    torch.manual_seed(0)
    model = build_default(CARDIO, 4, seed=0).to(cuda_device)
    masker = SignalMasker({"ABD": 0.7, "THX": 0.7, "ECG": 0.5, "PPG": 0.1}, backups=["ECG", "PPG"])
    pl = SleepLightningModule(model, optimizer=lambda ps: FusedAdamW(ps, lr=1e-3, weight_decay=1e-4, max_grad_norm=1.0),
                              scheduler=lambda o: ExpWarmUpScheduler(o, lr_max=1e-3, warmup_steps=4, tau=1e4),
                              num_classes=4, masker=masker)
    y = torch.randint(0, 4, (4, 8), device=cuda_device)
    y[0, :2] = -1

    def batches():
        while True:
            x = {k: v.to(cuda_device) for k, v in make_inputs(CARDIO, 4, 8, seed=3).items()}
            yield x, y

    losses = pl.fit(batches(), max_steps=12)
    print(losses)
    assert all(l == l for l in losses) and min(losses[-4:]) < losses[0]
    assert int(pl.cmats["train"].sum()) == 12 * (4 * 8 - 2)
    # inference after training uses the updated weights (operand copies are re-packed)
    model.eval()
    with torch.no_grad():
        out = model({k: v.to(cuda_device) for k, v in make_inputs(CARDIO, 4, 8, seed=3).items()})
    assert torch.isfinite(out).all()


def test_masker_on_device_defers_data_errors(cuda_device):
    """On CUDA the masker never synchronises: a night with every signal unavailable is reported by the next call /
    check(); the dropout statistics are those of the reference masker."""
    from wav2sleep_b200.trainer import SignalMasker
    torch.manual_seed(0)
    masker = SignalMasker({"ABD": 0.7, "THX": 0.7, "ECG": 0.5, "PPG": 0.1}, backups=["ECG", "PPG"])
    n, drops = 0, torch.zeros(4, device=cuda_device)
    for _ in range(40):
        x = {k: torch.randn(32, 8, device=cuda_device) for k in ("ABD", "THX", "ECG", "PPG")}
        masker(x)
        miss = torch.stack([torch.isinf(v[:, 0]) for v in x.values()], -1)
        assert not miss.all(-1).any()
        drops += miss.sum(0)
        n += 32
    masker.check()
    frac = (drops / n).tolist()
    assert 0.6 < frac[0] < 0.8 and 0.6 < frac[1] < 0.8 and 0.4 < frac[2] < 0.6 and frac[3] < 0.25
    bad = {k: torch.full((2, 8), float("-inf"), device=cuda_device) for k in ("ECG", "PPG")}
    masker(bad)  # recorded, not raised
    with pytest.raises(ValueError):
        masker.check()
    masker({k: torch.randn(2, 8, device=cuda_device) for k in ("ECG", "PPG")})  # flag was consumed
    strict = SignalMasker({"ECG": 0.5}, deferred_errors=False)
    with pytest.raises(ValueError):
        strict({"ECG": torch.full((2, 8), float("-inf"), device=cuda_device)})
