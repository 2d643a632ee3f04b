"""Integrated gradients (Sundararajan et al., 2017) of ``Wav2Sleep`` and ``SleepPPGNet`` on the GPU.

For night b the objective is ``F_b = sum_s logit[b, s, target[b, s]]`` over the epochs with ``target >= 0``, and the
attribution of sample (b, t) is ``(x - x0) * integral_0^1 dF_b/dx (x0 + a (x - x0)) da``.  The integral is a
Gauss-Legendre rule on [0, 1] (nodes and weights from ``numpy.polynomial.legendre.leggauss``, on the host).  The
interpolated nights go through the model in passes of at most ``internal_batch_size`` nights; each pass takes the input
gradients of the existing attribution path (``Wav2Sleep.forward`` / ``SleepPPGNet.forward`` with inputs that require
grad, eval semantics).  Building the interpolated inputs and summing the weighted gradients are the library kernels
``w2s_ig_path_inputs`` and ``w2s_ig_accumulate``; torch only allocates, views and indexes.

A non-finite sample of x is left as it is at every step: a missing (``-inf``) row stays missing along the whole path,
and such samples get exactly 0 attribution.  The call freezes the parameters and switches the model to ``eval()`` for
its duration, so the fast path launches no weight-gradient kernel and no ``p.grad``, optimizer buffer or BatchNorm
buffer is touched; ``requires_grad`` and every module's ``training`` flag are restored on return, also when it raises.
"""
from __future__ import annotations

import numpy as np
import torch
from torch import Tensor

from . import _lib
from .engine import _f32, _stream, check_inputs

__all__ = ("integrated_gradients", "gauss_legendre")

DEFAULT_INTERNAL_BATCH = 16  # nights per pass: the training batch


def gauss_legendre(steps: int) -> tuple[np.ndarray, np.ndarray]:
    """Nodes and weights (fp64) of the ``steps``-point Gauss-Legendre rule on [0, 1]; the weights sum to 1."""
    if isinstance(steps, bool) or not isinstance(steps, (int, np.integer)) or steps < 1:
        raise ValueError(f"steps must be a positive integer, got {steps!r}")
    t, w = np.polynomial.legendre.leggauss(int(steps))
    return (t + 1.0) / 2.0, w / 2.0


def _model_kind(model) -> str:
    from .model import Wav2Sleep
    from .ppgnet import SleepPPGNet
    if isinstance(model, SleepPPGNet):
        return "ppgnet"
    if isinstance(model, Wav2Sleep):
        return "wav2sleep"
    raise TypeError(f"integrated_gradients takes a Wav2Sleep or a SleepPPGNet, got {type(model).__name__}")


def _signals(model, kind: str, x, what: str) -> tuple[dict[str, Tensor], int, int, torch.device]:
    """The input (or baseline) as {name: [B, T]}, with its B, S and device; SleepPPGNet's single tensor is named "x"."""
    if kind == "ppgnet":
        if not isinstance(x, Tensor):
            raise TypeError(f"{what}: SleepPPGNet takes a [B, {model.INPUT_LENGTH}] tensor, got {type(x).__name__}")
        if x.dim() != 2 or x.size(1) != model.INPUT_LENGTH:
            raise ValueError(f"{what}: expected [B, {model.INPUT_LENGTH}], got {tuple(x.shape)}")
        if not x.is_cuda:
            raise RuntimeError(f"{what}: wav2sleep_b200 runs on CUDA (sm_100a) only; there is no CPU fallback")
        if x.size(0) == 0:
            raise ValueError(f"{what}: empty batch")
        xs, B, S, dev = {"x": x}, x.size(0), 1200, x.device
    else:
        _, B, S, dev = check_inputs(model.signal_encoders, x, what)
        xs = dict(x)
    for n, t in xs.items():
        if not t.is_floating_point():
            raise TypeError(f"{what}[{n!r}]: expected a floating-point tensor, got {t.dtype}")
    return xs, B, S, dev


def parse_target(target, B: int, S: int, n_classes: int) -> Tensor:
    """int, [B] or [B, S] integer target -> int64 [B, S] on the host; -1 skips an epoch (a [B] entry of -1: the night)."""
    if isinstance(target, bool):
        raise TypeError("target must be an int or an integer tensor, got a bool")
    if isinstance(target, (int, np.integer)):
        if not 0 <= int(target) < n_classes:
            raise ValueError(f"target class {int(target)} is outside [0, {n_classes})")
        return torch.full((B, S), int(target), dtype=torch.int64)
    if not isinstance(target, Tensor) or target.is_floating_point() or target.is_complex() or target.dtype == torch.bool:
        raise TypeError(f"target must be an int or an integer tensor, got {type(target).__name__}"
                        + (f" of {target.dtype}" if isinstance(target, Tensor) else ""))
    t = target.detach().to("cpu", torch.int64)
    if t.shape == (B,):
        t = t.view(B, 1).expand(B, S)
    elif t.shape != (B, S):
        raise ValueError(f"target must be an int, [B] = [{B}] or [B, S] = [{B}, {S}], got {tuple(t.shape)}")
    if t.numel() and (t.min().item() < -1 or t.max().item() >= n_classes):
        raise ValueError(f"target values must lie in [-1, {n_classes}) (-1 skips an epoch), got "
                         f"[{t.min().item()}, {t.max().item()}]")
    return t.contiguous()


def passes(B: int, K: int, internal_batch_size: int) -> list[tuple[int, int, int, int]]:
    """(b0, b1, k0, k1) of every model pass: nights [b0, b1) at steps [k0, k1), at most ``internal_batch_size`` nights
    each, steps in order within a night range (the accumulation adds them in that order)."""
    bc = min(B, internal_batch_size)
    kc = max(1, internal_batch_size // bc)
    return [(b0, min(B, b0 + bc), k0, min(K, k0 + kc)) for b0 in range(0, B, bc) for k0 in range(0, K, kc)]


def _internal_batch(internal_batch_size) -> int:
    if internal_batch_size is None:
        return DEFAULT_INTERNAL_BATCH
    if isinstance(internal_batch_size, bool) or not isinstance(internal_batch_size, (int, np.integer)) \
            or internal_batch_size < 1:
        raise ValueError(f"internal_batch_size must be a positive integer or None, got {internal_batch_size!r}")
    return int(internal_batch_size)


def integrated_gradients(model, x, target, baseline=None, steps: int = 32, internal_batch_size: int | None = None):
    """Integrated gradients of the per-night objective ``F_b = sum_s logit[b, s, target_bs]`` (epochs with
    ``target_bs >= 0``) along the straight path from ``baseline`` to ``x``.

    ``model``: a ``Wav2Sleep`` (fast or general path) or a ``SleepPPGNet``.  ``x``: ``{signal: [B, T]}`` CUDA tensors
    (``-inf`` rows = missing signal), or a ``[B, 1228800]`` tensor for ``SleepPPGNet``; ``baseline``: the same
    structure, None = zeros.  ``target``: an int class, a ``[B]`` or a ``[B, S]`` integer tensor (-1 skips).
    ``steps``: Gauss-Legendre nodes on [0, 1].  ``internal_batch_size``: interpolated nights per model pass (default 16).

    Returns ``(attr, delta)``: ``attr`` has the structure of ``x`` (fp32 ``[B, T]`` per signal); ``delta`` is fp64 [B],
    ``F_b(x) - F_b(x0) - sum(attr[b])``, the completeness gap, with both endpoint values from the same graph forward
    the gradients use.  The call runs with eval semantics and leaves the model as it found it."""
    kind = _model_kind(model)
    steps_nodes, steps_weights = gauss_legendre(steps)
    ibs = _internal_batch(internal_batch_size)
    xs, B, S, dev = _signals(model, kind, x, "x")
    x0s = None
    if baseline is not None:
        x0s, _, _, dev0 = _signals(model, kind, baseline, "baseline")
        if set(x0s) != set(xs):
            raise ValueError(f"baseline signals {sorted(x0s)} differ from the input's {sorted(xs)}")
        for n in xs:
            if x0s[n].shape != xs[n].shape:
                raise ValueError(f"baseline[{n!r}] has shape {tuple(x0s[n].shape)}, the input {tuple(xs[n].shape)}")
        if dev0 != dev:
            raise ValueError("every input and baseline tensor must be on one device")
    n_classes = model.classifier.out_features
    tgt = parse_target(target, B, S, n_classes)
    if torch.is_inference_mode_enabled():
        raise RuntimeError("integrated_gradients needs autograd: call it outside torch.inference_mode()")
    if B > 65535:
        raise ValueError(f"B = {B} nights: at most 65535 per call")

    lib = _lib.load()
    names = sorted(xs)
    modes = [(m, m.training) for m in model.modules()]
    grads_on = [(p, p.requires_grad) for p in model.parameters()]
    eng = getattr(model, "_engine", None) if kind == "wav2sleep" else None
    eng_state = None if eng is None else (eng.bucket_hooks, eng.loss_scale)
    try:
        model.eval()
        for p, _ in grads_on:
            p.requires_grad_(False)
        if eng is not None:  # no data-parallel gradient exchange, and the attribution loss scale of every pass
            eng.bucket_hooks, eng.loss_scale = [], None
        with torch.cuda.device(dev), torch.enable_grad():
            return _run(lib, model, kind, names, xs, x0s, tgt, steps_nodes, steps_weights, ibs, B, S, n_classes, dev)
    finally:
        for p, r in grads_on:
            p.requires_grad_(r)
        for m, t in modes:
            m.training = t
        if eng is not None:
            eng.bucket_hooks, eng.loss_scale = eng_state


def _run(lib, model, kind, names, xs, x0s, tgt, nodes, weights, ibs, B, S, n_classes, dev):
    xs = {n: _f32(xs[n]) for n in names}
    x0s = None if x0s is None else {n: _f32(x0s[n]) for n in names}
    alphas = torch.tensor(nodes, dtype=torch.float32).to(dev)
    wts = torch.tensor(weights, dtype=torch.float32).to(dev)
    ends = torch.tensor([0.0, 1.0], dtype=torch.float32).to(dev)
    valid = (tgt >= 0).to(dev)
    cls = torch.where(tgt >= 0, tgt, torch.zeros_like(tgt)).to(dev).unsqueeze(-1)  # [B, S, 1]
    onehot = torch.zeros(B, S, n_classes, dtype=torch.float32, device=dev)
    onehot.scatter_(2, cls, valid.unsqueeze(-1).to(torch.float32))  # d F_b / d logits

    def path_batch(b0, b1, a, k0, k1):
        """The interpolated nights of steps [k0, k1) of a, nights [b0, b1): {name: [(k1 - k0) * (b1 - b0), T]}."""
        out = {}
        for n in names:
            T = xs[n].size(1)
            t = torch.empty((k1 - k0) * (b1 - b0), T, dtype=torch.float32, device=dev)
            x0p = None if x0s is None else x0s[n][b0:b1].data_ptr()
            _lib.check(lib.w2s_ig_path_inputs(xs[n][b0:b1].data_ptr(), x0p, a[k0:].data_ptr(), k1 - k0, b1 - b0, T,
                                              t.data_ptr(), _stream()), ValueError)
            out[n] = t.requires_grad_(True)
        return out

    def call(batch):
        return model(batch["x"]) if kind == "ppgnet" else model(batch)

    attr = {n: torch.empty_like(xs[n]) for n in names}
    for b0, b1, k0, k1 in passes(B, len(nodes), ibs):
        batch = path_batch(b0, b1, alphas, k0, k1)
        logits = call(batch)
        go = onehot[b0:b1].repeat(k1 - k0, 1, 1)
        grads = torch.autograd.grad(logits, [batch[n] for n in names], grad_outputs=go)
        del logits, batch
        for n, g in zip(names, grads):
            g = g.to(torch.float32).contiguous()
            x0p = None if x0s is None else x0s[n][b0:b1].data_ptr()
            _lib.check(lib.w2s_ig_accumulate(g.data_ptr(), wts[k0:].data_ptr(), k1 - k0, xs[n][b0:b1].data_ptr(), x0p,
                                             b1 - b0, xs[n].size(1), attr[n][b0:b1].data_ptr(), int(k0 == 0), _stream()))
        del grads

    # completeness: F_b at a = 0 and a = 1 from the graph forward of the gradient passes, sums in fp64 (w2s_gen_stats)
    def row_sums(t3):  # [R, L, 1] fp32 -> [R] fp64
        st = torch.empty(t3.size(0), 1, 2, dtype=torch.float64, device=dev)
        _lib.check(lib.w2s_gen_stats(t3.data_ptr(), st.data_ptr(), None, t3.size(0), t3.size(1), 1, _stream()))
        return st[:, 0, 0]

    F_end = torch.empty(2, B, dtype=torch.float64, device=dev)
    for b0, b1, k0, k1 in passes(B, 2, ibs):
        logits = call(path_batch(b0, b1, ends, k0, k1)).detach()
        picked = logits.gather(2, cls[b0:b1].repeat(k1 - k0, 1, 1))
        picked = torch.where(valid[b0:b1].repeat(k1 - k0, 1).unsqueeze(-1), picked, torch.zeros_like(picked)).contiguous()
        F_end[k0:k1, b0:b1] = row_sums(picked).view(k1 - k0, b1 - b0)
        del logits
    delta = F_end[1] - F_end[0]
    for n in names:
        delta = delta - row_sums(attr[n].view(B, -1, 1))
    return (attr["x"] if kind == "ppgnet" else attr), delta
