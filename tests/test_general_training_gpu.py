"""Training of the non-default model options on the general CUDA path (general.py autograd Functions over the kernels
of csrc/general_bwd.cuh).

Gradient reference: oracle/general_oracle.py, an fp32 CPU functional restatement whose eval forward is pinned to the
real reference's logits (tests/test_general_oracle.py).  Both sides are fp32, so the gate is tight: relative L2 error
<= 1e-3 and cosine >= 0.99999 for the loss and every parameter gradient.
"""
import os
import socket
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

from oracle import general_oracle as GO
from oracle import make_golden_general as G
from wav2sleep_b200 import model as M

pytestmark = pytest.mark.gpu

REL, COS = 1e-3, 0.99999

CASES = {
    **{k: G.CASES[k] for k in ("general_causalconv_layer_silu", "general_shared_embed_registers", "general_group_nores_narrow")},
    # chunk-causal encoders (every epoch its own sample) with instance norm, causal sequence mixer with group norm.
    # SiLU, not ReLU: with a kinked activation this configuration's first-layer gradients are not a continuous function
    # of the parameters at fp32 resolution - scaling every parameter by (1 + 1e-7 noise) in an fp64 oracle moves the
    # ECG cnn.0 conv gradients by 2e-3 .. 8e-3 with ReLU and 2e-3 .. 5e-3 with leaky ReLU (pre-activations crossing
    # zero), but by <= 1.2e-5 with SiLU.  ReLU / leaky derivatives are checked on identical inputs by the kernel tests.
    "chunk_causal_instance": dict(
        seed=5, signal_map={"ECG": "ECG", "THX": "THX"}, num_classes=4,
        enc=dict(feature_dim=16, activation="silu", norm="instance", causal=True, chunk_causal=True),
        mix=dict(feature_dim=16, layers=1, nhead=2, dim_ff=32),
        seq=dict(feature_dim=16, norm="group", activation="silu", causal=True, num_layers=1, num_dilations=2,
                 kernel_size=3),
        B=2, S=4, masked=[("THX", 1)]),
    # post-LN mixer (norm_first=False) with GELU, RMS norm encoders, linear sequence-mixer activation
    "postln_mixer_rms": dict(
        seed=6, signal_map={"ABD": "ABD", "PPG": "PPG"}, num_classes=3,
        enc=dict(feature_dim=24, activation="gelu", norm="rms", initial_channels=8, max_channels=24),
        mix=dict(feature_dim=24, layers=2, nhead=3, dim_ff=40, activation="gelu", norm_first=False),
        seq=dict(feature_dim=24, norm="layer", activation="linear", num_layers=1, num_dilations=2, kernel_size=5),
        B=2, S=3, masked=[("PPG", 0)]),
}


def _no_dropout(case):
    return {**case, "mix": {**case["mix"], "dropout": 0.0}, "seq": {**case["seq"], "dropout": 0.0}}


def _build(case, dev):
    model = G.build(M, case)
    G.perturb(model, case["seed"])
    return model.to(dev).train()


def _labels(case, seed=0):
    y = torch.randint(0, case["num_classes"], (case["B"], case["S"]), generator=torch.Generator().manual_seed(seed))
    y[0, 0] = -100  # ignore_index, as the reference's padded epochs
    return y


def _cuda_loss_and_grads(model, x, y, dev):
    model.zero_grad(set_to_none=True)
    logits = model({k: v.to(dev) for k, v in x.items()})
    loss = F.cross_entropy(logits.view(-1, logits.shape[-1]), y.to(dev).view(-1), ignore_index=-100)
    loss.backward()
    return loss.detach().cpu(), {n: p.grad for n, p in model.named_parameters()}


def _oracle_loss_and_grads(model, case, x, y, dropout=None):
    names = dict(model.named_parameters())
    sd = {k: v.detach().cpu().to(torch.float32).clone().requires_grad_(k in names) for k, v in model.state_dict().items()}
    logits = GO.forward(x, sd, GO.config(case), dropout=dropout)
    loss = F.cross_entropy(logits.view(-1, logits.shape[-1]), y.view(-1), ignore_index=-100)
    loss.backward()
    return loss.detach(), {k: sd[k].grad for k in names}


def _compare(loss, grads, loss_o, grads_o, label):
    assert abs(loss.item() - loss_o.item()) <= REL * abs(loss_o.item()), (loss.item(), loss_o.item())
    worst = (0.0, 1.0, None)
    for n, go in grads_o.items():
        g = grads[n]
        assert go is not None, f"oracle has no gradient for {n}"
        assert g is not None, f"{n}: no gradient from the CUDA backward"
        g = g.detach().cpu().reshape(-1).double()
        go = go.reshape(-1).double()
        if go.norm() == 0:
            assert g.norm() <= 1e-12, n
            continue
        rel = ((g - go).norm() / go.norm()).item()
        cos = F.cosine_similarity(g, go, dim=0).item()
        if rel > worst[0]:
            worst = (rel, cos, n)
        assert rel <= REL and cos >= COS, f"{label}: {n} rel {rel:.3e} cos {cos:.7f}"
    print(f"{label}: loss {loss.item():.6f} (oracle {loss_o.item():.6f}); worst gradient {worst[2]} rel {worst[0]:.3e} "
          f"cos {worst[1]:.7f} over {len(grads_o)} tensors")


@pytest.mark.parametrize("name", list(CASES))
def test_gradients_match_oracle_autograd(cuda_device, name):
    case = _no_dropout(CASES[name])
    model = _build(case, cuda_device)
    for blk in model.sequence_mixer.dilated_convs:
        blk.dropout.p = 0.0
    model.epoch_mixer.dropout = 0.0
    for layer in model.epoch_mixer.transformer_encoder.layers:
        layer.self_attn.dropout = 0.0
        layer.dropout.p = layer.dropout1.p = layer.dropout2.p = 0.0
    assert not model.fast_path
    x, y = G.make_inputs(case), _labels(case)
    loss, grads = _cuda_loss_and_grads(model, x, y, cuda_device)
    loss_o, grads_o = _oracle_loss_and_grads(model, case, x, y)
    _compare(loss, grads, loss_o, grads_o, name)


def _site_masks(eng, model, case, seed, dev):
    """The keep masks of every dropout site of one training forward, shaped as the oracle takes them."""
    mix, cfg = model.epoch_mixer, GO.config(case)
    B, S, Fd, H = case["B"], case["S"], mix.feature_dim, mix.nhead
    D = 1 + mix.num_register_tokens + len(case["signal_map"])
    N = B * S
    p_mix, p_seq = cfg["mix"]["dropout"], cfg["seq"]["dropout"]
    get = lambda n, site, p, shape: eng.dropout_mask(n, site, p, seed, dev).cpu().view(*shape)
    out = {"mix": [], "seq": []}
    for li in range(mix.num_layers):
        out["mix"].append({"attn": get(N * H * D * D, 8 * li, p_mix, (N, H, D, D)),
                           "sa": get(N * D * Fd, 8 * li + 1, p_mix, (N, D, Fd)),
                           "ff": get(N * D * mix.dim_ff, 8 * li + 2, p_mix, (N, D, mix.dim_ff)),
                           "out": get(N * D * Fd, 8 * li + 3, p_mix, (N, D, Fd))})
    for bi in range(len(model.sequence_mixer.dilated_convs)):
        out["seq"].append(get(B * S * Fd, 64 + bi, p_seq, (B, S, Fd)))
    return out


def test_dropout_gradients_match_oracle_with_the_same_masks(cuda_device):
    base = G.CASES["general_shared_embed_registers"]
    case = {**base, "mix": {**base["mix"], "dropout": 0.25}, "seq": {**base["seq"], "dropout": 0.2}}
    model = _build(case, cuda_device)
    eng = model._get_general()
    eng.dropout_seed = 1234
    x, y = G.make_inputs(case), _labels(case, 1)
    loss, grads = _cuda_loss_and_grads(model, x, y, cuda_device)
    assert eng.last_dropout_seed == 1234
    masks = _site_masks(eng, model, case, 1234, cuda_device)
    kept = torch.cat([m.reshape(-1).float() for d in masks["mix"] for m in d.values()]).mean().item()
    assert 0.6 < kept < 0.9  # the masks really drop (p = 0.25)
    loss_o, grads_o = _oracle_loss_and_grads(model, case, x, y, dropout=masks)
    _compare(loss, grads, loss_o, grads_o, "dropout")
    # a different seed draws different masks, and train() under no_grad stays without dropout
    eng.dropout_seed = 99
    with torch.no_grad():
        a = model({k: v.to(cuda_device) for k, v in x.items()})
        b = model.eval()({k: v.to(cuda_device) for k, v in x.items()})
    assert torch.equal(a, b)
    assert not torch.equal(eng.dropout_mask(4096, 1, 0.25, 99, cuda_device), eng.dropout_mask(4096, 1, 0.25, 1234, cuda_device))


def test_full_night_gradients_match_oracle(cuda_device):
    """One 10-h night (S = 1200, 1.2 M ECG samples) of the causal-conv / layer-norm / SiLU architecture: the long
    weight-gradient and norm-parameter reductions against fp32 CPU autograd."""
    case = _no_dropout({**G.CASES["general_causalconv_layer_silu"], "B": 1, "S": 1200})
    model = _build(case, cuda_device)
    for blk in model.sequence_mixer.dilated_convs:
        blk.dropout.p = 0.0
    x, y = G.make_inputs(case, seed=7), _labels(case, 2)
    loss, grads = _cuda_loss_and_grads(model, x, y, cuda_device)
    loss_o, grads_o = _oracle_loss_and_grads(model, case, x, y)
    _compare(loss, grads, loss_o, grads_o, "full night")


def test_train_forward_logits_equal_eval_forward(cuda_device):
    case = _no_dropout(G.CASES["general_shared_embed_registers"])
    model = _build(case, cuda_device)
    for blk in model.sequence_mixer.dilated_convs:
        blk.dropout.p = 0.0
    x = {k: v.to(cuda_device) for k, v in G.make_inputs(case).items()}
    train_logits = model(x)
    assert train_logits.grad_fn is not None
    with torch.no_grad():
        eval_logits = model.eval()(x)
    assert torch.equal(train_logits.detach(), eval_logits)


def test_batchnorm_training_still_raises(cuda_device):
    enc = M.SignalEncoders(signal_map={"ECG": "ECG"}, feature_dim=16, activation="relu", norm="layer", causal=True)
    model = M.Wav2Sleep(enc, M.MultiModalAttentionEmbedder(feature_dim=16), M.SequenceCNN(feature_dim=16, norm="batch"), 4)
    model = model.to(cuda_device).train()
    x = {"ECG": torch.randn(1, 2048, device=cuda_device)}
    with pytest.raises(NotImplementedError, match="BatchNorm"):
        model(x)
    with torch.no_grad():
        assert model(x).shape == (1, 2, 4)  # train() under no_grad: inference kernels, eval-mode statistics


def test_fit_steps_lower_the_loss_with_masker(cuda_device):
    from wav2sleep_b200.optim import FusedAdamW
    from wav2sleep_b200.trainer import SignalMasker, SleepLightningModule
    torch.manual_seed(0)
    case = G.CASES["general_causalconv_layer_silu"]
    model = _build(case, cuda_device)
    masker = SignalMasker({"ABD": 0.5, "ECG": 0.5}, backups=["ECG"])
    pl = SleepLightningModule(model, optimizer=lambda ps: FusedAdamW(ps, lr=2e-3, weight_decay=1e-4, max_grad_norm=1.0),
                              num_classes=case["num_classes"], masker=masker)
    x = {k: v.to(cuda_device) for k, v in G.make_inputs({**case, "S": 8}).items()}
    y = _labels({**case, "S": 8})
    y[y == -100] = -1  # the module's criterion: CrossEntropyLoss(ignore_index=-1), as in the reference trainer
    y = y.to(cuda_device)
    losses = []
    for _ in range(12):
        losses.append(float(pl.fit_step(({k: v.clone() for k, v in x.items()}, y))))
        assert pl._opt.grads_aliased()  # autograd accumulated into the optimizer's flat gradient buffer
    print(losses)
    assert all(l == l for l in losses) and min(losses[-4:]) < losses[0]
    assert pl._opt.flat_grad.abs().sum() > 0


# ------------------------------------------------------------------ kernels against torch CPU autograd
def _eng():
    from wav2sleep_b200.general import GeneralEngine
    return GeneralEngine(None)


def _check(got, want, what, tol=1e-4):
    got, want = got.detach().cpu().double().reshape(-1), want.detach().cpu().double().reshape(-1)
    err = ((got - want).norm() / want.norm().clamp_min(1e-30)).item()
    assert err <= tol, f"{what}: rel L2 {err:.3e}"


@pytest.mark.parametrize("stride,dil,causal,taps,cin,cout,taps_major,raw,masked", [
    (1, 1, False, 3, 12, 20, 0, 0, False), (2, 1, True, 3, 1, 9, 0, 1, True), (1, 4, True, 5, 10, 10, 0, 0, True),
    (1, 32, False, 7, 9, 13, 0, 0, False), (2, 1, False, 1, 11, 7, 0, 0, True), (4, 1, False, 4, 12, 17, 1, 0, True),
    (1, 2, True, 7, 24, 24, 0, 0, False), (1, 1, False, 1, 5, 3, 0, 1, False),
])
def test_conv_dgrad_wgrad(cuda_device, stride, dil, causal, taps, cin, cout, taps_major, raw, masked):
    g = torch.Generator().manual_seed(taps * 100 + dil)
    B, L_in = 3, 301 if not taps_major else 64
    x = torch.randn(B, L_in, cin, generator=g)
    if raw:
        x[0, 5, 0] = float("inf")
        x[1, 17, 0] = float("-inf")
    w = torch.randn(cout, taps * cin, generator=g) if taps_major else torch.randn(cout, cin, taps, generator=g)
    bias = torch.randn(cout, generator=g)
    if taps_major:
        pad_left, L_out = 0, L_in // 4
    else:
        pad_left = (taps - 1) * dil if causal else (taps - 1) * dil // 2
        L_out = (L_in - 1) // stride + 1 if causal else (L_in + 2 * pad_left - dil * (taps - 1) - 1) // stride + 1
    mask = torch.tensor([0, 1, 0] if masked else [0, 0, 0], dtype=torch.uint8)
    gout = torch.randn(B, L_out, cout, generator=g)
    # reference: zero-pad, conv, keep L_out outputs; masked samples excluded
    xr = torch.where(torch.isinf(x), torch.zeros_like(x), x).requires_grad_(not raw)
    wr = (w.view(cout, taps, cin).permute(0, 2, 1) if taps_major else w).clone().requires_grad_()
    br = bias.clone().requires_grad_()
    right = max(0, (L_out - 1) * stride + (taps - 1) * dil + 1 - pad_left - L_in)
    ref = F.conv1d(F.pad(xr.transpose(1, 2), (pad_left, right)), wr, br, stride=stride, dilation=dil)[..., :L_out]
    keep = (1 - mask.float())[:, None, None]
    (ref.transpose(1, 2) * gout * keep).sum().backward()
    xd = x.to(cuda_device).requires_grad_(not raw)
    wd = w.to(cuda_device).requires_grad_()
    bd = bias.to(cuda_device).requires_grad_()
    out = _eng().conv(xd, wd, bd, L_out, stride=stride, dil=dil, pad_left=pad_left, mask=mask.to(cuda_device),
                      taps_major=taps_major, raw=raw)
    _check(out * keep.to(cuda_device), ref.transpose(1, 2) * keep, "conv forward")
    out.backward(gout.to(cuda_device))
    if not raw:
        _check(xd.grad, xr.grad, "dgrad")
    wgrad_ref = wr.grad.permute(0, 2, 1).reshape(cout, taps * cin) if taps_major else wr.grad
    _check(wd.grad, wgrad_ref, "wgrad")
    _check(bd.grad, br.grad, "bias grad")


REF_ACT = {"relu": torch.relu, "leaky": lambda t: F.leaky_relu(t, 0.01), "gelu": F.gelu, "silu": F.silu,
           "linear": lambda t: t}


@pytest.mark.parametrize("act", list(REF_ACT))
@pytest.mark.parametrize("mode", ["scale_shift_res", "per_channel", "plain"])
def test_affine_act_backward(cuda_device, act, mode):
    g = torch.Generator().manual_seed(3)
    B, L, Cc = 3, 257, 37
    x, res, gout = (torch.randn(B, L, Cc, generator=g) for _ in range(3))
    if mode == "per_channel":
        scale, shift, res = torch.randn(Cc, generator=g), torch.randn(Cc, generator=g), None
    elif mode == "plain":
        scale = shift = res = None
    else:
        scale, shift = torch.randn(B, Cc, generator=g), torch.randn(B, Cc, generator=g)
    mask = torch.tensor([0, 0, 1], dtype=torch.uint8)
    leaf = lambda t, d: None if t is None else t.clone().to(d).requires_grad_()
    cpu = [leaf(t, "cpu") for t in (x, scale, shift, res)]
    sc = cpu[1] if cpu[1] is None or mode == "per_channel" else cpu[1][:, None, :]
    sh = cpu[2] if cpu[2] is None or mode == "per_channel" else cpu[2][:, None, :]
    pre = cpu[0] * (1 if sc is None else sc) + (0 if sh is None else sh) + (0 if cpu[3] is None else cpu[3])
    keep = (1 - mask.float())[:, None, None]
    (REF_ACT[act](pre) * gout * keep).sum().backward()
    gpu = [leaf(t, cuda_device) for t in (x, scale, shift, res)]
    out = _eng().affine_act(gpu[0], act, gpu[1], gpu[2], gpu[3], mask=mask.to(cuda_device), per_channel=int(mode == "per_channel"))
    out.backward(gout.to(cuda_device))
    for a, b, n in zip(gpu, cpu, ("x", "scale", "shift", "res")):
        if a is not None:
            _check(a.grad, b.grad, f"{act} {mode} d{n}")


@pytest.mark.parametrize("kind,Cc", [("instance", 20), ("group", 24), ("group", 6)])
def test_instance_group_norm_backward(cuda_device, kind, Cc):
    g = torch.Generator().manual_seed(Cc)
    B, L = 3, 333
    y, gout = 2 + torch.randn(B, L, Cc, generator=g), torch.randn(B, L, Cc, generator=g)
    norm = torch.nn.InstanceNorm1d(Cc, eps=1e-2) if kind == "instance" else M.ConvGroupNorm(Cc)
    if kind == "group":
        with torch.no_grad():
            norm.norm.weight.copy_(1 + 0.3 * torch.randn(Cc, generator=g))
            norm.norm.bias.copy_(0.3 * torch.randn(Cc, generator=g))
    mask = torch.tensor([0, 1, 0], dtype=torch.uint8)
    keep = (1 - mask.float())[:, None, None]
    yc = y.clone().requires_grad_()
    sd = {k: v.detach().clone().requires_grad_() for k, v in norm.state_dict(prefix="n.").items()}
    ref = GO.act(GO.norm(yc.transpose(1, 2), kind, sd, "n", 1e-2), "silu").transpose(1, 2)
    (ref * gout * keep).sum().backward()
    normd = norm.to(cuda_device)
    yd = y.to(cuda_device).requires_grad_()
    out = _eng().norm_act(yd, SimpleNamespace(norm_name=kind, norm=normd), "silu", mask=mask.to(cuda_device))
    out.backward(gout.to(cuda_device))
    _check(yd.grad * keep.to(cuda_device), yc.grad * keep, f"{kind} dx")
    if kind == "group":
        _check(normd.norm.weight.grad, sd["n.norm.weight"].grad, "group dweight")
        _check(normd.norm.bias.grad, sd["n.norm.bias"].grad, "group dbias")


@pytest.mark.parametrize("rms,Cc,act", [(0, 40, "silu"), (1, 40, "gelu"), (0, 128, "linear"), (1, 7, "leaky")])
def test_rownorm_backward(cuda_device, rms, Cc, act):
    g = torch.Generator().manual_seed(Cc + rms)
    R = 1000
    x, gout = torch.randn(R, Cc, generator=g), torch.randn(R, Cc, generator=g)
    w, b = 1 + 0.3 * torch.randn(Cc, generator=g), 0.3 * torch.randn(Cc, generator=g)
    xc, wc, bc = (t.clone().requires_grad_() for t in (x, w, b))
    if rms:
        ref = wc * xc / torch.sqrt(xc.pow(2).mean(-1, keepdim=True) + 1e-5)
    else:
        ref = F.layer_norm(xc, (Cc,), wc, bc, 1e-5)
    (REF_ACT[act](ref) * gout).sum().backward()
    xd, wd, bd = (t.to(cuda_device).requires_grad_() for t in (x, w, b))
    out = _eng().rownorm(xd, wd, None if rms else bd, 1e-5, act, rms=rms)
    out.backward(gout.to(cuda_device))
    _check(xd.grad, xc.grad, "dx")
    _check(wd.grad, wc.grad, "dweight")
    if not rms:
        _check(bd.grad, bc.grad, "dbias")


@pytest.mark.parametrize("H,hd,D", [(1, 8, 2), (4, 8, 5), (3, 16, 4), (8, 4, 7)])
def test_attention_backward(cuda_device, H, hd, D):
    from wav2sleep_b200.general import _Attn
    g = torch.Generator().manual_seed(H * 10 + D)
    N, Fd = 37, H * hd
    qkv, gout = torch.randn(N * D, 3 * Fd, generator=g), torch.randn(N * D, Fd, generator=g)
    km = (torch.rand(N, D, generator=g) < 0.3).to(torch.uint8)
    km[:, 0] = 0
    km[:4, 1:] = 1  # epochs in which every key but the CLS token is masked
    qc = qkv.clone().requires_grad_()
    q, k, v = (t.reshape(N, D, H, hd).transpose(1, 2) for t in qc.split(Fd, -1))
    s = (q @ k.transpose(-1, -2)) / hd ** 0.5
    s = s.masked_fill(km.bool()[:, None, None, :], float("-inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(N * D, Fd)
    (ref * gout).sum().backward()
    qd = qkv.to(cuda_device).requires_grad_()
    out = _Attn.apply(qd, _eng(), km.reshape(-1).to(cuda_device), N, D, H, 0.0, 0, 0)
    _check(out, ref, "attention forward")
    out.backward(gout.to(cuda_device))
    _check(qd.grad, qc.grad, "dqkv")


# ------------------------------------------------------------------ two GPUs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _ddp_worker(rank, world, port, q):
    import sys
    from pathlib import Path
    import torch.distributed as dist
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    sys.path.insert(0, str(Path(__file__).resolve().parent))
    from oracle import make_golden_general as G
    from wav2sleep_b200 import model as M
    from wav2sleep_b200.optim import FusedAdamW
    from wav2sleep_b200.trainer import SleepLightningModule
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    case = {**G.CASES["general_causalconv_layer_silu"], "B": 2 * world, "S": 6}
    model = G.build(M, case).to(dev)
    for blk in model.sequence_mixer.dilated_convs:
        blk.dropout.p = 0.0
    pl = SleepLightningModule(model, optimizer=lambda ps: FusedAdamW(ps, lr=1e-3, weight_decay=0.0, max_grad_norm=None),
                              num_classes=case["num_classes"], masker=None, flip_polarity=False)
    pl.setup_training()
    x = G.make_inputs(case)
    y = torch.randint(0, case["num_classes"], (case["B"], case["S"]), generator=torch.Generator().manual_seed(3))
    sl = slice(rank * 2, rank * 2 + 2)
    # one fit_step's gradient path: this rank's slice, then the all-reduce of every bucket after the backward
    model.train()
    pl._opt.zero_grad()
    loss = pl.training_step(({k: v[sl].to(dev) for k, v in x.items()}, y[sl].to(dev)))
    loss.backward()
    for name in pl._reducer.segments:
        pl._reducer(name)
    pl._reducer.wait()
    torch.cuda.synchronize()
    g_dp = (pl._opt.flat_grad * pl._opt.grad_scale).clone()
    pl._opt.zero_grad()
    logits = model({k: v.to(dev) for k, v in x.items()})
    F.cross_entropy(logits.view(-1, case["num_classes"]), y.to(dev).view(-1)).backward()
    torch.cuda.synchronize()
    g_full = pl._opt.flat_grad.clone()
    rel = ((g_dp - g_full).norm() / g_full.norm()).item()
    cos = F.cosine_similarity(g_dp, g_full, dim=0).item()
    q.put((rank, rel, cos))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_rank_averaged_gradient_equals_full_batch():
    import torch.multiprocessing as mp
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_ddp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=600) for _ in range(world)), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, rel, cos in res:
        print(f"rank {rank}: rank-averaged vs full-batch gradient rel {rel:.3e} cos {cos:.7f}")
        assert rel < 1e-4 and cos > 0.99999
