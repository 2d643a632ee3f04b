"""General inference engine: every model option of the reference that is outside the fused tcgen05 path
(SURVEY section 8f, row N3) on the dimension-generic fp32 kernels of ``csrc/general.cuh``.

What is restated, with the reference lines it follows (relative to /root/reference/src/wav2sleep/):
  SignalEncoders.forward          models/wav2sleep.py:146-161   (-inf rows, optional signal embedding :155-159)
  SignalEncoder.forward           models/wav2sleep.py:235-267   (chunk-causal per-epoch path :248-255, output_norm :266)
  ConvBlock1D / ConvLayer1D       models/blocks.py:57-71, 173-186 (causal padding + right-trim :150-152, :178-182)
  norms / activations             models/utils.py:9-96
  MultiModalAttentionEmbedder     models/wav2sleep.py:301-346   (register tokens :299, :330-335; norm_first either way)
  SequenceCNN / DilatedConvBlock  models/wav2sleep.py:379-390 ; models/blocks.py:115-126

Tensors are fp32, channels-last ``[B, L, C]``; weights stay in their PyTorch layouts (no packing).  torch is used for
allocation and pure data movement (views, stack, index) only - every FLOP is in ``libw2s_b200.so``, except that autograd
sums the gradients of a tensor that feeds two branches (residuals).

Inference (``forward``, under ``no_grad``): BatchNorm uses its running statistics, dropout is the identity.
``forward_graph`` is the same eval-semantics forward with autograd on: what ``Wav2Sleep.forward`` runs in ``eval()`` when
an input requires grad (attribution); the raw signal stays on the graph, its gradient is 0 at non-finite samples (the
reference replaces them by 0, wav2sleep.py:150-151) and on missing rows.  Training
(``forward_train``, what ``Wav2Sleep.forward`` calls under ``train()`` with grad): every primitive below is a
``torch.autograd.Function`` whose backward runs the kernels of ``csrc/general_bwd.cuh``, and dropout is applied where
the reference applies it (attention weights, the FF / dropout1 / dropout2 dropouts of each mixer layer,
DilatedConvBlock.dropout) with counter-based masks: ``dropout_seed`` (None: drawn from torch's CPU generator per step)
and the fixed site numbers of training.py; ``dropout_mask`` returns a site's keep decisions.  BatchNorm in a training
forward normalises with the batch statistics and updates the running statistics (``_BatchNormTrainAct``); SleepPPGNet
trains through it, while model.py still refuses to train Wav2Sleep models with BatchNorm layers (their masked samples
would need the reference's zero-filled semantics, which the row-masked kernels do not have).
"""
from __future__ import annotations

import contextlib

import torch
from torch import Tensor, nn

from . import _lib
from .engine import _argmax, _dropout_seed, _f32, _p, _stream, check_inputs

ACT = {"linear": 0, "relu": 1, "leaky": 2, "gelu": 3, "silu": 4, "swish": 4}
NORM_INSTANCE, NORM_GROUP, NORM_BATCH = 0, 1, 2


def _g(t: Tensor) -> Tensor:
    """An incoming gradient as the kernels read it (fp32, contiguous)."""
    return t.to(torch.float32).contiguous()


# Every primitive is a torch.autograd.Function: its forward runs the forward kernel, its backward the backward kernels of
# csrc/general_bwd.cuh.  Under no_grad the same forward runs and nothing is saved, so inference and training share one
# stage code (GeneralEngine.encode / epoch_mixer / dilated_blocks / _forward).  Parameters go in as they are (detached
# inside the forward), so their gradients reach p.grad.
class _Conv(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, bias, eng, L_out, stride, dil, pad_left, mask, taps_major, raw):
        B, L_in, cin = x.shape
        xd, wd = _f32(x), _f32(w)
        if taps_major:
            cout, taps = wd.shape[0], wd.shape[1] // cin
        else:
            cout, _, taps = wd.shape
        out = torch.zeros(B, L_out, cout, dtype=torch.float32, device=x.device)
        _lib.check(eng.lib.w2s_gen_conv(xd.data_ptr(), wd.data_ptr(), _p(_f32(bias)), out.data_ptr(), _p(mask), B, L_in,
                                        L_out, cin, cout, taps, stride, dil, pad_left, taps_major, raw, _stream()))
        ctx.save_for_backward(xd, wd, mask)
        ctx.eng, ctx.has_bias = eng, bias is not None
        ctx.geo = (B, L_in, L_out, cin, cout, taps, stride, dil, pad_left, taps_major, raw)
        return out

    @staticmethod
    def backward(ctx, g):
        xd, wd, mask = ctx.saved_tensors
        B, L_in, L_out, cin, cout, taps, stride, dil, pad_left, taps_major, raw = ctx.geo
        lib, g = ctx.eng.lib, _g(g)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.zeros_like(xd)
            _lib.check(lib.w2s_gen_conv_dgrad(g.data_ptr(), wd.data_ptr(), dx.data_ptr(), _p(mask), B, L_in, L_out, cin, cout,
                                              taps, stride, dil, pad_left, taps_major, _stream()))
            if raw:  # the forward read non-finite raw samples as 0: they have no gradient (data movement, no arithmetic)
                dx = torch.where(torch.isfinite(xd), dx, torch.zeros_like(dx))
        want_b = ctx.has_bias and ctx.needs_input_grad[2]
        if ctx.needs_input_grad[1] or want_b:
            ws = torch.empty(taps * cin * cout + cout, dtype=torch.float64, device=g.device)
            dw = torch.empty_like(wd) if ctx.needs_input_grad[1] else None
            db = torch.empty(cout, dtype=torch.float32, device=g.device) if want_b else None
            _lib.check(lib.w2s_gen_conv_wgrad(xd.data_ptr(), g.data_ptr(), _p(dw), _p(db), ws.data_ptr(), _p(mask), B, L_in,
                                              L_out, cin, cout, taps, stride, dil, pad_left, taps_major, raw, _stream()))
        return dx, dw, db, None, None, None, None, None, None, None, None


class _AffineAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, scale, shift, res, eng, act, mask, per_channel):
        B, L, Cc = x.shape
        xd, sc, sh, rs = _f32(x), _f32(scale), _f32(shift), _f32(res)
        out = torch.zeros_like(xd)
        _lib.check(eng.lib.w2s_gen_affine_act(xd.data_ptr(), _p(sc), _p(sh), _p(rs), out.data_ptr(), _p(mask), B, L, Cc,
                                              ACT[act], per_channel, _stream()))
        ctx.save_for_backward(xd, sc, sh, rs, mask)
        ctx.eng, ctx.act, ctx.per_channel = eng, act, per_channel
        return out

    @staticmethod
    def backward(ctx, g):
        xd, sc, sh, rs, mask = ctx.saved_tensors
        B, L, Cc = xd.shape
        need_x, need_sc, need_sh, need_res = ctx.needs_input_grad[:4]
        g = _g(g)
        din = torch.zeros_like(xd) if need_x else None
        dpre = torch.zeros_like(xd) if need_res else None
        sums = None
        if need_sc or need_sh:
            sums = torch.empty(1 if ctx.per_channel else B, Cc, 2, dtype=torch.float64, device=g.device)
        _lib.check(ctx.eng.lib.w2s_gen_affine_act_bwd(xd.data_ptr(), _p(sc), _p(sh), _p(rs), g.data_ptr(), _p(din), _p(dpre),
                                                      _p(sums), _p(mask), B, L, Cc, ACT[ctx.act], ctx.per_channel, _stream()))
        dsc = sums[..., 1].to(torch.float32).view(sc.shape) if need_sc else None
        dsh = sums[..., 0].to(torch.float32).view(sh.shape) if need_sh else None
        return din, dsc, dsh, dpre, None, None, None, None


class _BatchNormConsts(torch.autograd.Function):
    """Eval-mode BatchNorm1d as a per-channel affine: scale = w / sqrt(running_var + eps), shift = b - running_mean * scale
    ([1, C] each), differentiable in w and b (the running statistics are buffers)."""

    @staticmethod
    def forward(ctx, weight, bias, eng, running_mean, running_var, eps):
        Cc = running_mean.numel()
        dev = running_mean.device
        rm, rv = _f32(running_mean), _f32(running_var)
        scale = torch.empty(1, Cc, dtype=torch.float32, device=dev)
        shift = torch.empty(1, Cc, dtype=torch.float32, device=dev)
        _lib.check(eng.lib.w2s_gen_norm_consts(None, _p(_f32(weight)), _p(_f32(bias)), rm.data_ptr(), rv.data_ptr(),
                                               scale.data_ptr(), shift.data_ptr(), 1, Cc, 1, NORM_BATCH, 1, eps, _stream()))
        ctx.save_for_backward(rm, rv)
        ctx.eng, ctx.eps = eng, eps
        return scale, shift

    @staticmethod
    def backward(ctx, dscale, dshift):
        rm, rv = ctx.saved_tensors
        Cc, dev = rm.numel(), rm.device
        dscale = torch.zeros(Cc, dtype=torch.float32, device=dev) if dscale is None else _g(dscale)
        dshift = torch.zeros(Cc, dtype=torch.float32, device=dev) if dshift is None else _g(dshift)
        dw = torch.empty(Cc, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        db = torch.empty(Cc, dtype=torch.float32, device=dev) if ctx.needs_input_grad[1] else None
        if dw is not None or db is not None:
            _lib.check(ctx.eng.lib.w2s_gen_bn_eval_bwd(dscale.data_ptr(), dshift.data_ptr(), rm.data_ptr(), rv.data_ptr(), _p(dw),
                                                       _p(db), Cc, ctx.eps, _stream()))
        return dw, db, None, None, None, None


class _BatchNormTrainAct(torch.autograd.Function):
    """Train-mode BatchNorm1d + activation of a conv output y [B, L, C].  Viewed as [1, B * L, C], BatchNorm's statistics
    group is an InstanceNorm's: w2s_gen_bn_stats gives the per-channel sums over every row, norm_consts (instance mode,
    biased variance) scale = w * rstd and shift = b - mean * w * rstd, affine_act applies them, and the backward is
    the InstanceNorm backward of that view (affine_act_bwd -> norm_bwd with groups = C).  The module's running
    statistics are updated in place, once per forward, on the forward's stream (unbiased variance, as PyTorch)."""

    @staticmethod
    def forward(ctx, y, weight, bias, eng, norm, act):
        B, L, Cc = y.shape
        rows = B * L
        if rows >= 2 ** 31:
            raise ValueError(f"train-mode BatchNorm over {rows} rows: at most 2^31 - 1")
        lib, dev = eng.lib, y.device
        yd, w, b = _f32(y), _f32(weight), _f32(bias)
        stats = torch.empty(1, Cc, 2, dtype=torch.float64, device=dev)
        _lib.check(lib.w2s_gen_bn_stats(yd.data_ptr(), stats.data_ptr(), rows, Cc, _stream()))
        if norm.track_running_stats and norm.running_mean is not None:
            for buf in (norm.running_mean, norm.running_var):
                if buf.dtype != torch.float32 or not buf.is_contiguous():
                    raise ValueError("BatchNorm running statistics must be contiguous fp32")
            momentum = -1.0 if norm.momentum is None else float(norm.momentum)
            _lib.check(lib.w2s_gen_bn_update_running(stats.data_ptr(), rows, norm.running_mean.data_ptr(),
                                                     norm.running_var.data_ptr(), norm.num_batches_tracked.data_ptr(),
                                                     momentum, Cc, _stream()))
        scale = torch.empty(1, Cc, dtype=torch.float32, device=dev)
        shift = torch.empty(1, Cc, dtype=torch.float32, device=dev)
        _lib.check(lib.w2s_gen_norm_consts(stats.data_ptr(), _p(w), _p(b), None, None, scale.data_ptr(), shift.data_ptr(), 1,
                                           Cc, rows, NORM_INSTANCE, 1, norm.eps, _stream()))
        out = torch.empty_like(yd)
        _lib.check(lib.w2s_gen_affine_act(yd.data_ptr(), scale.data_ptr(), shift.data_ptr(), None, out.data_ptr(), None, 1,
                                          rows, Cc, ACT[act], 1, _stream()))
        ctx.save_for_backward(yd, w, stats, scale, shift)
        ctx.eng, ctx.eps, ctx.act = eng, norm.eps, act
        return out

    @staticmethod
    def backward(ctx, g):
        yd, w, stats, scale, shift = ctx.saved_tensors
        B, L, Cc = yd.shape
        rows = B * L
        lib, g, dev = ctx.eng.lib, _g(g), g.device
        dpre = torch.empty_like(yd)
        sums = torch.empty(1, Cc, 2, dtype=torch.float64, device=dev)
        _lib.check(lib.w2s_gen_affine_act_bwd(yd.data_ptr(), scale.data_ptr(), shift.data_ptr(), None, g.data_ptr(), None,
                                              dpre.data_ptr(), sums.data_ptr(), None, 1, rows, Cc, ACT[ctx.act], 1, _stream()))
        coef = torch.empty(1, Cc, 3, dtype=torch.float32, device=dev)
        dy = torch.empty_like(yd)
        dw = torch.empty(Cc, dtype=torch.float32, device=dev) if ctx.needs_input_grad[1] else None
        db = torch.empty(Cc, dtype=torch.float32, device=dev) if ctx.needs_input_grad[2] else None
        _lib.check(lib.w2s_gen_norm_bwd(yd.data_ptr(), dpre.data_ptr(), stats.data_ptr(), sums.data_ptr(), _p(w),
                                        coef.data_ptr(), dy.data_ptr(), _p(dw), _p(db), None, 1, rows, Cc, Cc, ctx.eps,
                                        _stream()))
        return dy, dw, db, None, None, None


class _NormAct(torch.autograd.Function):
    """InstanceNorm1d / GroupNorm (statistics over L, or L x channels of a group) + activation of a conv output."""

    @staticmethod
    def forward(ctx, y, weight, bias, eng, groups, mode, eps, act, mask):
        B, L, Cc = y.shape
        lib, dev = eng.lib, y.device
        yd, w, b = _f32(y), _f32(weight), _f32(bias)
        stats = torch.zeros(B, Cc, 2, dtype=torch.float64, device=dev)
        _lib.check(lib.w2s_gen_stats(yd.data_ptr(), stats.data_ptr(), _p(mask), B, L, Cc, _stream()))
        scale = torch.zeros(B, Cc, dtype=torch.float32, device=dev)
        shift = torch.zeros(B, Cc, dtype=torch.float32, device=dev)
        _lib.check(lib.w2s_gen_norm_consts(stats.data_ptr(), _p(w), _p(b), None, None, scale.data_ptr(), shift.data_ptr(), B,
                                           Cc, L, mode, groups, eps, _stream()))
        out = torch.zeros_like(yd)
        _lib.check(lib.w2s_gen_affine_act(yd.data_ptr(), scale.data_ptr(), shift.data_ptr(), None, out.data_ptr(), _p(mask),
                                          B, L, Cc, ACT[act], 0, _stream()))
        ctx.save_for_backward(yd, w, stats, scale, shift, mask)
        ctx.eng, ctx.groups, ctx.eps, ctx.act = eng, groups if mode == NORM_GROUP else Cc, eps, act
        return out

    @staticmethod
    def backward(ctx, g):
        yd, w, stats, scale, shift, mask = ctx.saved_tensors
        B, L, Cc = yd.shape
        lib, g, dev = ctx.eng.lib, _g(g), g.device
        dpre = torch.zeros_like(yd)
        sums = torch.empty(B, Cc, 2, dtype=torch.float64, device=dev)
        _lib.check(lib.w2s_gen_affine_act_bwd(yd.data_ptr(), scale.data_ptr(), shift.data_ptr(), None, g.data_ptr(), None,
                                              dpre.data_ptr(), sums.data_ptr(), _p(mask), B, L, Cc, ACT[ctx.act], 0, _stream()))
        coef = torch.empty(B, Cc, 3, dtype=torch.float32, device=dev)
        dy = torch.zeros_like(yd)
        dw = torch.empty(Cc, dtype=torch.float32, device=dev) if ctx.needs_input_grad[1] else None
        db = torch.empty(Cc, dtype=torch.float32, device=dev) if ctx.needs_input_grad[2] else None
        _lib.check(lib.w2s_gen_norm_bwd(yd.data_ptr(), dpre.data_ptr(), stats.data_ptr(), sums.data_ptr(), _p(w),
                                        coef.data_ptr(), dy.data_ptr(), _p(dw), _p(db), _p(mask), B, L, Cc, ctx.groups, ctx.eps,
                                        _stream()))
        return dy, dw, db, None, None, None, None, None, None


class _RowNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eng, eps, act, rms):
        Cc = x.shape[-1]
        rows = x.numel() // Cc
        xd, w, b = _f32(x), _f32(weight), _f32(bias)
        out = torch.empty_like(xd)
        _lib.check(eng.lib.w2s_gen_rownorm(xd.data_ptr(), _p(w), _p(b), out.data_ptr(), rows, Cc, rms, ACT[act], eps,
                                           _stream()))
        ctx.save_for_backward(xd, w, b)
        ctx.eng, ctx.eps, ctx.act, ctx.rms = eng, eps, act, rms
        return out

    @staticmethod
    def backward(ctx, g):
        xd, w, b = ctx.saved_tensors
        Cc = xd.shape[-1]
        rows, g, dev = xd.numel() // Cc, _g(g), g.device
        dx = torch.empty_like(xd)
        dw = torch.empty(Cc, dtype=torch.float32, device=dev) if (w is not None and ctx.needs_input_grad[1]) else None
        db = torch.empty(Cc, dtype=torch.float32, device=dev) if (b is not None and ctx.needs_input_grad[2]) else None
        ws = torch.empty(2 * Cc, dtype=torch.float64, device=dev) if (dw is not None or db is not None) else None
        _lib.check(ctx.eng.lib.w2s_gen_rownorm_bwd(xd.data_ptr(), _p(w), _p(b), g.data_ptr(), dx.data_ptr(), _p(dw), _p(db),
                                                   _p(ws), rows, Cc, ctx.rms, ACT[ctx.act], ctx.eps, _stream()))
        return dx, dw, db, None, None, None, None


class _Attn(torch.autograd.Function):
    """Attention of the fused in-projection output qkv [N * D, 3F] (q, k, v = column thirds) -> o [N * D, F]."""

    @staticmethod
    def forward(ctx, qkv, eng, km, N, D, H, p, seed, site):
        qkv = _f32(qkv)
        F3 = qkv.shape[1]
        Fd = F3 // 3
        o = torch.empty(qkv.shape[0], Fd, dtype=torch.float32, device=qkv.device)
        q = qkv.data_ptr()
        _lib.check(eng.lib.w2s_gen_attn(q, q + 4 * Fd, q + 8 * Fd, o.data_ptr(), km.data_ptr(), N, D, H, Fd // H, F3, p, seed,
                                        site, _stream()))
        ctx.save_for_backward(qkv, km)
        ctx.eng, ctx.cfg = eng, (N, D, H, p, seed, site)
        return o

    @staticmethod
    def backward(ctx, g):
        qkv, km = ctx.saved_tensors
        N, D, H, p, seed, site = ctx.cfg
        F3 = qkv.shape[1]
        Fd = F3 // 3
        g = _g(g)
        d = torch.empty_like(qkv)
        q, dq = qkv.data_ptr(), d.data_ptr()
        _lib.check(ctx.eng.lib.w2s_gen_attn_bwd(q, q + 4 * Fd, q + 8 * Fd, g.data_ptr(), dq, dq + 4 * Fd, dq + 8 * Fd,
                                                km.data_ptr(), N, D, H, Fd // H, F3, p, seed, site, _stream()))
        return d, None, None, None, None, None, None, None, None


class _Dropout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, eng, p, seed, site):
        xd = _f32(x)
        out = torch.empty_like(xd)
        _lib.check(eng.lib.w2s_gen_dropout(xd.data_ptr(), out.data_ptr(), None, xd.numel(), p, seed, site, _stream()))
        ctx.eng, ctx.cfg = eng, (p, seed, site)
        return out

    @staticmethod
    def backward(ctx, g):
        p, seed, site = ctx.cfg
        g = _g(g)
        dx = torch.empty_like(g)
        _lib.check(ctx.eng.lib.w2s_gen_dropout(g.data_ptr(), dx.data_ptr(), None, g.numel(), p, seed, site, _stream()))
        return dx, None, None, None, None


class _Broadcast(torch.autograd.Function):
    """A [F] parameter row repeated over n rows (register / CLS tokens); the backward is its column sum."""

    @staticmethod
    def forward(ctx, row, eng, n):
        rd = _f32(row)
        ctx.eng = eng
        return torch.empty(n, rd.shape[0], dtype=torch.float32, device=rd.device).copy_(rd)

    @staticmethod
    def backward(ctx, g):
        g = _g(g)
        n, Fd = g.shape
        sums = torch.empty(1, Fd, 2, dtype=torch.float64, device=g.device)
        # the per-channel sums of a linear affine_act backward: sums[c, 0] = sum over rows of g
        _lib.check(ctx.eng.lib.w2s_gen_affine_act_bwd(g.data_ptr(), None, None, None, g.data_ptr(), None, None,
                                                      sums.data_ptr(), None, 1, n, Fd, ACT["linear"], 1, _stream()))
        return sums[0, :, 0].to(torch.float32), None, None


class GeneralEngine:
    def __init__(self, model):
        self.model = model
        self.lib = _lib.load()
        self.dropout_seed = None  # int: fixed seed for every training step (tests); None: drawn from torch's CPU generator
        self.last_dropout_seed = 0
        self._seed = None         # the current training forward's seed; None = no dropout (eval, or no_grad)

    # ------------------------------------------------------------------ kernel wrappers
    def conv(self, x: Tensor, w: Tensor, bias, L_out: int, stride=1, dil=1, pad_left=0, mask=None, taps_major=0, raw=0):
        """x [B, L_in, cin] -> [B, L_out, cout]; w [cout, cin, taps] (taps_major: [cout, taps * cin] with taps given by
        the caller through w.shape[1] // cin)."""
        return _Conv.apply(x, w, bias, self, L_out, stride, dil, pad_left, mask, taps_major, raw)

    def linear(self, x: Tensor, lin: nn.Linear | None = None, weight=None, bias=None) -> Tensor:
        """rows [R, K] -> [R, N] = x W^T + b (a 1-tap conv over R positions)."""
        if lin is not None:
            weight, bias = lin.weight, lin.bias
        R, K = x.shape
        return self.conv(x.reshape(1, R, K), weight.unsqueeze(-1), bias, R).view(R, -1)

    def affine_act(self, x: Tensor, act: str, scale=None, shift=None, res=None, mask=None, per_channel=0) -> Tensor:
        return _AffineAct.apply(x, scale, shift, res, self, act, mask, per_channel)

    def rownorm(self, x: Tensor, weight, bias, eps: float, act: str = "linear", rms: int = 0) -> Tensor:
        return _RowNorm.apply(x, weight, bias, self, eps, act, rms)

    def dropout(self, x: Tensor, p: float, site: int) -> Tensor:
        """nn.Dropout(p) of a training forward (identity otherwise): the counter-based masks of w2s_gen_dropout."""
        if self._seed is None or p <= 0:
            return x
        return _Dropout.apply(x, self, float(p), self._seed, site)

    def dropout_mask(self, n: int, site: int, p: float, seed: int, device) -> Tensor:
        """The keep decisions (uint8 0/1) of the first n elements of a dropout site (test hook).  For the attention
        weights of a mixer layer the element index is ((epoch * H + head) * D + query) * D + key."""
        m = torch.empty(n, dtype=torch.uint8, device=device)
        with torch.cuda.device(device):
            _lib.check(self.lib.w2s_gen_dropout(None, None, m.data_ptr(), n, p, seed, site, _stream()))
        return m

    def norm_act(self, y: Tensor, layer, act: str, mask=None, res=None) -> Tensor:
        """norm (by the layer's kind) -> activation of a conv output y [B, L, C]   (ConvLayer1D.forward, blocks.py:183-185)."""
        kind, norm = layer.norm_name, layer.norm
        if kind is None:
            return self.affine_act(y, act, mask=mask)
        if kind in ("layer", "rms"):
            w = norm.weight.reshape(-1)
            b = norm.bias.reshape(-1) if kind == "layer" else None
            return self.rownorm(y, w, b, norm.eps, act, rms=int(kind == "rms"))
        if kind == "batch":
            if self._seed is not None:  # a training forward: batch statistics, running-statistics update
                if mask is not None:
                    raise NotImplementedError("train-mode BatchNorm of masked samples is not built")
                return _BatchNormTrainAct.apply(y, norm.weight, norm.bias, self, norm, act)
            # eval mode: running statistics
            scale, shift = _BatchNormConsts.apply(norm.weight, norm.bias, self, norm.running_mean, norm.running_var, norm.eps)
            return self.affine_act(y, act, scale, shift, mask=mask, per_channel=1)
        if kind == "instance":
            affine = getattr(norm, "affine", False)
            return _NormAct.apply(y, norm.weight if affine else None, norm.bias if affine else None, self, 1, NORM_INSTANCE,
                                  norm.eps, act, mask)
        if kind == "group":
            gn = norm.norm
            return _NormAct.apply(y, gn.weight, gn.bias, self, gn.num_groups, NORM_GROUP, gn.eps, act, mask)
        raise NotImplementedError(f"norm {kind!r}")

    def conv_layer(self, a: Tensor, layer, mask=None, raw=0) -> Tensor:
        """ConvLayer1D.forward (blocks.py:173-186) on a [B, L, Cin] input."""
        L_out = layer.output_length(a.shape[1])
        y = self.conv(a, layer.conv.weight, layer.conv.bias, L_out, stride=layer.stride, dil=layer.dilation,
                      pad_left=layer.padding, mask=mask, raw=raw)
        return self.norm_act(y, layer, layer.activation_name, mask=mask)

    def conv_block(self, a: Tensor, blk, mask=None, raw=0) -> Tensor:
        """ConvBlock1D.forward (blocks.py:57-71): act(conv3(conv2(conv1(x))) [+ downsample(x)])."""
        y = self.conv_layer(a, blk.conv1, mask, raw)
        y = self.conv_layer(y, blk.conv2, mask)
        y = self.conv_layer(y, blk.conv3, mask)
        if not blk.use_residual:
            return self.affine_act(y, blk.activation_name, mask=mask)
        r = self.conv(a, blk.downsample.weight, None, (a.shape[1] - 1) // 2 + 1, stride=2, mask=mask, raw=raw)
        if r.shape[1] != y.shape[1]:
            raise ValueError(f"residual length {r.shape[1]} != conv path length {y.shape[1]}")
        return self.affine_act(y, blk.activation_name, res=r, mask=mask)

    def dilated_blocks(self, x_BSF: Tensor, blocks) -> Tensor:
        """Sequential(DilatedConvBlock) (blocks.py:115-126): act(dropout(layers(x)) + x)."""
        cur = x_BSF
        for bi, blk in enumerate(blocks):
            blk_in = cur
            for layer in blk.conv_layers:
                cur = self.conv_layer(cur, layer)
            cur = self.affine_act(self.dropout(cur, blk.dropout.p, 64 + bi), blk.activation_name, res=blk_in)
        return cur

    # ------------------------------------------------------------------ stages
    def encode(self, enc, x_BT: Tensor):
        """SignalEncoder.forward (wav2sleep.py:235-267) -> (z [B, S, F], mask [B] uint8).  x_BT has passed
        ``check_inputs``."""
        B, T = x_BT.shape
        spe = enc.samples_per_epoch
        S = T // spe
        xs = x_BT.to(torch.float32).contiguous()  # stays on the autograd graph when the input requires grad
        mask = torch.isinf(xs.detach()[:, 0]).to(torch.uint8).contiguous()  # data-dependent control, no arithmetic
        if enc.causal and enc.chunk_causal:  # every epoch is its own sample (wav2sleep.py:248-255)
            a = xs.view(B * S, spe, 1)
            m = mask.repeat_interleave(S).contiguous()
        else:
            a = xs.view(B, T, 1)
            m = mask
        raw = 1
        for blk in enc.cnn:
            a = self.conv_block(a, blk, m, raw)
            raw = 0
        return self.epoch_features(enc, a, m, B, S), mask

    def epoch_features(self, enc, a: Tensor, m: Tensor, B: int, S: int) -> Tensor:
        """The encoder's Linear(4C -> F) + activation (+ output_norm) on the last block's output a -> z [B, S, F]."""
        Bp, L4, Cc = a.shape
        if L4 % 4 or (Bp * L4) // 4 != B * S:
            raise ValueError(f"encoder output length {L4} does not give 4 frames per epoch")
        z = self.conv(a, enc.linear.weight, enc.linear.bias, L4 // 4, stride=4, mask=m, taps_major=1)  # [Bp, L4/4, F]
        z = self.affine_act(z, enc.activation_name, mask=m)
        if isinstance(enc.output_norm, nn.LayerNorm):
            z = self.rownorm(z, enc.output_norm.weight, enc.output_norm.bias, enc.output_norm.eps)
        return z.view(B, S, -1)

    def epoch_mixer(self, zs: list[Tensor], masks: list[Tensor], B: int, S: int) -> Tensor:
        """MultiModalAttentionEmbedder.forward (wav2sleep.py:301-346) -> CLS features [B, S, F]."""
        mix = self.model.epoch_mixer
        Fd, R = mix.feature_dim, mix.num_register_tokens
        N, dev = B * S, zs[0].device
        if zs[0].shape[-1] != Fd:
            raise ValueError(f"Feature dimension {zs[0].shape[-1]} does not match self.feature_dim={Fd}.")
        reg = mix.register_tokens[0, 0].t()  # [R + 1, F]; token 0 is the CLS token
        toks = [_Broadcast.apply(reg[i], self, N).view(B, S, Fd) for i in range(R + 1)]
        toks += [torch.where(m.bool()[:, None, None], torch.zeros_like(z), z) for z, m in zip(zs, masks)]
        D = len(toks)
        x = torch.stack(toks, dim=2).reshape(N * D, Fd)
        km = torch.stack([torch.zeros_like(masks[0])] * (R + 1) + masks, dim=1)[:, None, :].expand(B, S, D)
        km = km.reshape(N * D).contiguous()
        H = mix.nhead
        act = mix.activation_name
        # dropout sites (as in training.py): 8 * layer + {0 attention weights, 1 dropout1, 2 FF dropout, 3 dropout2}
        for li, layer in enumerate(mix.transformer_encoder.layers):
            def sa(h):
                qkv = self.linear(h, weight=layer.self_attn.in_proj_weight, bias=layer.self_attn.in_proj_bias)  # [R, 3F]
                p = layer.self_attn.dropout if self._seed is not None else 0.0
                o = _Attn.apply(qkv, self, km, N, D, H, float(p), self._seed or 0, 8 * li)
                return self.dropout(self.linear(o, layer.self_attn.out_proj), layer.dropout1.p, 8 * li + 1)

            def ff(h):
                hid = self.affine_act(self.linear(h, layer.linear1).unsqueeze(0), act).squeeze(0)
                hid = self.dropout(hid, layer.dropout.p, 8 * li + 2)
                return self.dropout(self.linear(hid, layer.linear2), layer.dropout2.p, 8 * li + 3)

            add = lambda a, b: self.affine_act(a.unsqueeze(0), "linear", res=b.unsqueeze(0)).squeeze(0)
            ln = lambda t, nrm: self.rownorm(t, nrm.weight, nrm.bias, nrm.eps)
            if mix.norm_first:
                x = add(sa(ln(x, layer.norm1)), x)
                x = add(ff(ln(x, layer.norm2)), x)
            else:
                x = ln(add(sa(x), x), layer.norm1)
                x = ln(add(ff(x), x), layer.norm2)
        return x.view(N, D, Fd)[:, 0, :].contiguous().view(B, S, Fd)

    def sequence_mixer(self, x_BSF: Tensor) -> Tensor:
        """SequenceCNN.forward (wav2sleep.py:379-390) + DilatedConvBlock.forward (blocks.py:115-126)."""
        return self.dilated_blocks(x_BSF, self.model.sequence_mixer.dilated_convs)

    # ------------------------------------------------------------------ model
    @torch.no_grad()
    def forward(self, x: dict[str, Tensor]) -> Tensor:
        """Inference (eval semantics: running BatchNorm statistics, no dropout)."""
        self._seed = None
        return self._forward(x)

    def forward_graph(self, x: dict[str, Tensor]) -> Tensor:
        """The inference forward (eval semantics) with autograd on, for gradients with respect to the inputs."""
        self._seed = None
        return self._forward(x)

    @contextlib.contextmanager
    def training_forward(self):
        """The scope of one training forward: dropout at every site the reference applies it in training, with masks
        from ``dropout_seed`` (None: a seed drawn from torch's CPU generator, distinct per rank), and train-mode
        BatchNorm (batch statistics, running-statistics update)."""
        self.last_dropout_seed = self._seed = _dropout_seed(self.dropout_seed)
        try:
            yield
        finally:
            self._seed = None

    def forward_train(self, x: dict[str, Tensor]) -> Tensor:
        """Training forward: builds the autograd graph whose backward runs the kernels of csrc/general_bwd.cuh."""
        with self.training_forward():
            return self._forward(x)

    def _forward(self, x: dict[str, Tensor]) -> Tensor:
        m = self.model
        names, B, S, dev = check_inputs(m.signal_encoders, x)  # sorted: the token order, wav2sleep.py:311
        zs, masks = [], []
        with torch.cuda.device(dev):
            for n in names:
                z, mask = self.encode(m.signal_encoders.get_encoder(n), x[n])
                if m.signal_encoders.embed_signals:  # wav2sleep.py:155-159
                    e = m.signal_encoders.embedder.weight[m.signal_encoders.sig_to_embedding_idx[n]]
                    z = self.affine_act(z, "linear", shift=e, mask=mask, per_channel=1)
                zs.append(z)
                masks.append(mask)
            feat = self.sequence_mixer(self.epoch_mixer(zs, masks, B, S))
            logits = self.linear(feat.view(B * S, -1), m.classifier).view(B, S, m.num_classes)
        return logits

    @torch.no_grad()
    def predict(self, x: dict[str, Tensor]) -> Tensor:
        return _argmax(self.lib, self.forward(x))
