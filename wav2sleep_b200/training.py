"""Training path (SURVEY section 8 row a-11): forward with saved activations, backward, for ``Wav2Sleep``.

Replaces what the reference gets from autograd over ``Wav2Sleep.forward`` (trainer/main.py:161-163 ->
``loss.backward()``).  Every FLOP runs in ``libw2s_b200.so``; this file is the host-side schedule (which kernel on which
buffer), written in Python like the reference's training code is.  Encoders reuse the streaming tcgen05 kernels with
``keep_activations=1``; epoch mixer and sequence mixer run un-fused in training (tcgen05 implicit-GEMM kernel with a
plain epilogue + row-wise kernels) so that every intermediate needed by the backward is materialised once.  Data
gradients are tcgen05 convolutions with flipped/transposed weights, weight gradients are the streaming ``gemm_tn``
kernel, everything else is element-/row-wise.

Dropout (epoch mixer p, sequence mixer p; the encoder ConvLayer1D dropout is p = 0 in the reference config) uses a
counter-based generator: the keep decision of an element is a hash of (step seed, dropout site, element index), so the
backward regenerates the masks instead of storing them, and a test can dump them (``w2s_dropout`` mask_out) to feed the
oracle the very same masks.  The masks are therefore not the ones torch's Philox stream would draw - same distribution,
different realisation.  Storage: fp16 activations and activation gradients, fp32 parameter gradients.

Loss scaling: the reference trains in fp32 (scripts/config/training/main.yaml:16), where the ~1e-7 activation gradients
of a mean cross entropy over B*S = 19 200 epochs are harmless; in fp16 they would be subnormal.  The backward therefore
runs on gradients multiplied by a power of two (``TrainEngine.loss_scale``; default: 4 * 2^ceil(log2(B*S)), i.e. as if
the loss were 4x the *sum* over epochs, which centres the activation gradients in fp16's range for any batch size), and
every kernel that accumulates a parameter gradient multiplies by the inverse - fp32 parameter gradients are unscaled,
exactly (powers of two), and nothing outside this file sees the scale.

Input gradients (saliency, integrated gradients: ``x[name].requires_grad_()`` before the forward) come out of the same
backward: block 0's data gradient into the raw signal is ``w2s_first_conv_dgrad``.  Their objectives are not a mean cross
entropy - one logit or a class's summed logits give d(objective)/d(logits) of order 1, which the batch-size rule above
would push past fp16's 65 504 - so a backward that produces input gradients without an explicit ``loss_scale`` picks
the power of two that brings max|dlogits| into [4, 8) (one device reduction, one scalar read back).  Only the requested
work runs: parameters with ``requires_grad=False`` get no buffer and no weight-gradient launch, and an encoder whose
parameters are frozen and whose signal needs no gradient is not back-propagated at all.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import math

import torch
from torch import Tensor

from . import _lib
from ._lib import PRO_DNORM, ConvCall, EPI_ACT_BWD, EPI_PLAIN, PRO_NONE
from .engine import ForwardEngine, _dropout_seed, _f32, _p, _stream, check_inputs

F16 = torch.float16


class TrainEngine(ForwardEngine):
    """Adds forward_train / backward to the inference engine (shares the packed forward weights)."""

    def __init__(self, model):
        super().__init__(model)
        self._train_key = None
        self.saved = None
        self.bucket_hooks = []  # callables(name) fired as gradient buckets become final (data-parallel overlap)
        self.direct = set()
        self.dropout_seed = None  # int: fixed seed for every step (tests); None: drawn from torch's CPU generator
        self.last_dropout_seed = 0
        self._side_streams = {}   # device -> per-encoder CUDA streams (same overlap of kernel tails as in inference)
        # InstanceNorm backward of a layer's gradient inside the prologue of the data-gradient conv that consumes it
        # (W2S_PRO_DNORM) instead of a separate enc_norm_bwd pass; False keeps the separate kernels
        self.fuse_norm_bwd = True
        self._wg = None
        self._wg_streams = {}
        self.loss_scale = None    # power of two applied to the fp16 activation gradients; None = from B*S (see below)
        self._inv_scale = 1.0
        self.last_loss_scale = 1.0
        self.input_grads = {}     # signal -> fp32 [B, T] d(objective)/dx of the last backward that was asked for them

    @staticmethod
    def auto_loss_scale(n_epochs: int) -> float:
        """4 * 2^ceil(log2(B*S)): d(loss)/d(logits) of a mean cross entropy is (p - onehot) / n_valid, so this brings the
        logit gradients to O(1..8) and the encoder activation gradients (measured ~1e-2 of that) to ~1e-2..1e-1, the
        middle of fp16's normal range [6e-5, 65504], whatever the batch size."""
        k = max(int(n_epochs) - 1, 0).bit_length() + 2
        return float(2 ** min(k, 24))

    @staticmethod
    def attribution_loss_scale(max_abs_dlogits: float) -> float:
        """2^k with max|dlogits| * 2^k in [4, 8), k <= 24: the scale of a backward whose objective is not a mean cross
        entropy (a logit, a class's summed logits), where the batch-size rule would overflow fp16."""
        k = 3 - math.frexp(max_abs_dlogits)[1]
        return math.ldexp(1.0, min(k, 24))

    def _encoder_streams(self, device, n):
        """n side streams (one per signal encoder) that have been made to wait for the current stream, or None."""
        if not self.enc_streams or n < 2:
            return None
        pool = self._side_streams.setdefault(str(device), [])
        while len(pool) < n:
            pool.append(torch.cuda.Stream(device=device))
        fork = torch.cuda.Event()
        fork.record(torch.cuda.current_stream(device))
        for st in pool[:n]:
            st.wait_event(fork)
        return pool[:n]

    @staticmethod
    def _join(streams, device):
        if streams is not None:
            cur = torch.cuda.current_stream(device)
            for st in streams:
                cur.wait_stream(st)

    # dropout sites: 8 * layer + {0 attention weights, 1 after self-attention, 2 FF hidden, 3 after FF}; 64 + seq block
    def dropout(self, x: Tensor, site: int, p: float, seed: int, res: Tensor | None = None, out: Tensor | None = None):
        out = torch.empty_like(x) if out is None else out
        _lib.check(self.lib.w2s_dropout(x.data_ptr(), _p(res), out.data_ptr(), None, x.numel(), p, seed, site, _stream()))
        return out

    def dropout_mask(self, n: int, site: int, p: float, seed: int, device) -> Tensor:
        """The keep decisions (uint8 0/1) of the first n elements of a dropout site (test hook)."""
        m = torch.empty(n, dtype=torch.uint8, device=device)
        _lib.check(self.lib.w2s_dropout(None, None, None, m.data_ptr(), n, p, seed, site, _stream()))
        return m

    # ------------------------------------------------------------------ weight packing for the backward
    def _ensure_train_packed(self, device):
        """fp16 UMMA-layout weights of the training path (no hi/lo split): forward GEMM weights of the un-fused mixers and
        the flipped / transposed weights of every data-gradient conv, as jobs of a second PackPlan over views of the live
        parameters - re-packed with one launch after each optimizer step."""
        self._ensure_packed(device)
        skey, vkey = self._weights_key
        if self._train_key is not None and self._train_key[0] == skey:
            if self._train_key[1] != vkey:
                self.tplan.run()
                self._train_key = (skey, vkey)
            return
        from .engine import PackPlan
        m = self.model
        plan = self.tplan = PackPlan(self.lib, device)

        class _W:  # packed weight handle: the kernels only need the device pointer
            def __init__(self, ptr):
                self.ptr = ptr

            def data_ptr(self):
                return self.ptr

        P = lambda view, flip=False: _W(plan.conv(view, split=0, flip=flip))
        dgrad = lambda w: P(w.permute(1, 0, 2), flip=True)  # conv weight of the data gradient (transposed conv)
        self.tw = {"enc": {}, "mix": [], "seq": []}
        for name, enc in m.signal_encoders.encoders.items():
            e = {"conv": [], "ds": [], "lin_fwd": None, "lin_dgrad": []}
            for i, blk in enumerate(enc.cnn):
                e["conv"].append([dgrad(blk.conv1.conv.weight) if i > 0 else None, dgrad(blk.conv2.conv.weight),
                                  dgrad(blk.conv3.conv.weight)])
                e["ds"].append(P(blk.downsample.weight.permute(1, 0, 2)) if i > 0 else None)
            Cl = enc.channels[-1]
            Wl = enc.linear.weight
            e["lin_fwd"] = P(Wl.view(Wl.shape[0], 4, Cl).permute(0, 2, 1))
            e["lin_dgrad"] = [P(Wl[:, t * Cl:(t + 1) * Cl].t().unsqueeze(-1)) for t in range(4)]
            self.tw["enc"][name] = e
        for layer in m.epoch_mixer.transformer_encoder.layers:
            Win, W1, W2 = layer.self_attn.in_proj_weight, layer.linear1.weight, layer.linear2.weight
            Wo = layer.self_attn.out_proj.weight
            self.tw["mix"].append({
                "qkv": [P(Win[j * 128:(j + 1) * 128].unsqueeze(-1)) for j in range(3)],
                "qkv_T": [P(Win[j * 128:(j + 1) * 128].t().unsqueeze(-1)) for j in range(3)],
                "o": P(Wo.unsqueeze(-1)), "o_T": P(Wo.t().unsqueeze(-1)),
                "ff1": [P(W1[j * 128:(j + 1) * 128].unsqueeze(-1)) for j in range(4)],
                "ff1_T": P(W1.view(4, 128, 128).permute(2, 1, 0)),          # taps=4 conv for d(h2)
                "ff2": P(W2.view(W2.shape[0], 4, 128).permute(0, 2, 1)),
                "ff2_T": [P(W2[:, j * 128:(j + 1) * 128].t().unsqueeze(-1)) for j in range(4)],
            })
        for blk in m.sequence_mixer.dilated_convs:
            self.tw["seq"].append([{"fwd": P(l.conv.weight), "T": dgrad(l.conv.weight)} for l in blk.conv_layers])
        plan.run()
        self._train_key = (skey, vkey)

    # ------------------------------------------------------------------ kernel helpers
    def conv(self, inp, w, cin, cout, taps, B, L_in, L_out, out, stride=1, dil=1, pad=0, bias=None, res=None,
             out_stride=0, out_offset=0, out_rows=0, row_mask=None):
        c = ConvCall()
        c.cin, c.cout, c.taps, c.stride, c.dilation, c.pad = cin, cout, taps, stride, dil, pad
        c.prologue, c.epilogue, c.has_ds = PRO_NONE, EPI_PLAIN, 0
        c.B, c.L_in, c.L_out = B, L_in, L_out
        c.in_, c.w, c.out = inp.data_ptr(), w.data_ptr(), out.data_ptr()
        c.bias = bias.data_ptr() if bias is not None else None
        c.res = res.data_ptr() if res is not None else None
        c.row_mask = row_mask.data_ptr() if row_mask is not None else None
        c.out_stride, c.out_offset, c.out_rows = out_stride, out_offset, out_rows
        _lib.check(self.lib.w2s_conv1d_fwd(C.byref(c), _stream()))

    def conv_act_bwd(self, dy, w, cin, cout, B, L, y, stats, sums, dxh, a_out, eps, row_mask, res=None, r=None, dr=None,
                     dnorm=None):
        """Data gradient of a k=3 / pad=1 / stride-1 conv (flipped, transposed weights w) fused with the backward through
        the activation of the layer that produced the conv's input: writes d(x_hat) of that layer (dxh), its activated
        output (a_out, operand of this conv's weight gradient), d(residual branch) (dr, block outputs) and accumulates
        the two InstanceNorm-backward reductions into sums.

        dnorm = (dxh_in, y_in, stats_in, sums_in, upsample): the conv input dy is not given but computed in the kernel's
        prologue as the InstanceNorm backward of this layer's own d(x_hat) (W2S_PRO_DNORM) and written to `dy` for the
        weight gradient - one pass over the tensors instead of a separate enc_norm_bwd launch."""
        c = ConvCall()
        c.cin, c.cout, c.taps, c.stride, c.dilation, c.pad = cin, cout, 3, 1, 1, 1
        c.prologue, c.epilogue, c.has_ds = PRO_NONE, EPI_ACT_BWD, 0
        c.B, c.L_in, c.L_out = B, L, L
        c.in_, c.w, c.out = dy.data_ptr(), w.data_ptr(), dxh.data_ptr()
        if dnorm is not None:
            dxh_in, y_in, stats_in, sums_in, upsample = dnorm
            c.prologue = PRO_DNORM
            c.in_, c.in_res, c.in_stats = dxh_in.data_ptr(), y_in.data_ptr(), stats_in.data_ptr()
            c.dn_sums, c.dn_out, c.dn_upsample, c.in_eps = sums_in.data_ptr(), dy.data_ptr(), int(upsample), eps
        c.res = res.data_ptr() if res is not None else None
        c.row_mask = row_mask.data_ptr() if row_mask is not None else None
        c.out_stats = sums.data_ptr()
        c.act_y, c.act_stats, c.act_eps = y.data_ptr(), stats.data_ptr(), eps
        c.act_a = a_out.data_ptr() if a_out is not None else None
        c.act_r = r.data_ptr() if r is not None else None
        c.act_dr = dr.data_ptr() if dr is not None else None
        _lib.check(self.lib.w2s_conv1d_fwd(C.byref(c), _stream()))

    def _wgrad_stream(self, *tensors):
        """Stream for a parameter-gradient launch.  Inside the classifier / mixer part of the backward (`_wg` set) these
        launches leave the critical path: that part is a chain of ~150 small dependent kernels, of which only the data
        gradients (convs, LayerNorm / attention backward) depend on each other - the weight-gradient GEMMs and bias
        column sums (more than half of the launches) only have to be done before the optimizer / the gradient bucket
        hook.  They run on a side stream ordered after the current position of the main stream."""
        side = self._wg
        if side is None:
            return _stream()
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        side.wait_event(ev)
        for t in tensors:
            if t is not None:
                t.record_stream(side)
        return side.cuda_stream

    def gemm_tn(self, X, Y, Cbuf, M, N, B, LX, LY, ldc_m, ldc_n, y_stride=1, y_offset=0, row_mask=None, c_off=0, taps=1,
                ldc_t=0, tap_stride=1):
        if Cbuf is None:  # frozen parameter
            return
        _lib.check(self.lib.w2s_gemm_tn(X.data_ptr(), Y.data_ptr(), Cbuf.data_ptr() + 4 * c_off, M, N, taps, tap_stride, B,
                                        LX, LY, y_stride, y_offset, ldc_m, ldc_n, ldc_t, self._inv_scale, _p(row_mask),
                                        self._wgrad_stream(X, Y, Cbuf, row_mask)))

    def ln_fwd(self, x, g, b, rows, gelu, eps, res=None):
        out = torch.empty_like(x)
        _lib.check(self.lib.w2s_row_ln_fwd(x.data_ptr(), _p(res), g.data_ptr(), b.data_ptr(), out.data_ptr(), rows, gelu,
                                           eps, _stream()))
        return out

    def ln_bwd(self, x, g, b, dout, dg, db, rows, gelu, eps, res=None, dadd=None, want_ds=False):
        dx = torch.empty_like(x)
        ds = torch.empty_like(x) if want_ds else None
        if (dg is None) != (db is None):  # one of the two frozen: the kernel computes both or neither
            dg = torch.zeros_like(g) if dg is None else dg
            db = torch.zeros_like(b) if db is None else db
        _lib.check(self.lib.w2s_row_ln_bwd(x.data_ptr(), _p(res), g.data_ptr(), b.data_ptr(), dout.data_ptr(), _p(dadd),
                                           dx.data_ptr(), _p(ds), _p(dg), _p(db), rows, gelu, eps,
                                           self._inv_scale, _stream()))
        return dx, ds

    def colsum(self, x, out, rows, Cc, row_stride=1, row_offset=0, row_mask=None, rows_per_sample=0, out_off=0):
        if out is None:  # frozen parameter
            return
        _lib.check(self.lib.w2s_colsum(x.data_ptr(), out.data_ptr() + 4 * out_off, rows, Cc, row_stride, row_offset,
                                       _p(row_mask), rows_per_sample, self._inv_scale, self._wgrad_stream(x, out, row_mask)))

    # ------------------------------------------------------------------ gradients storage
    def _grad(self, p: Tensor) -> Tensor | None:
        """fp32 gradient buffer of a parameter, zeroed at the start of every backward, accumulated by the kernels; None for
        a parameter that does not require grad (its weight-gradient launches are skipped)."""
        if not p.requires_grad:
            return None
        g = self.grads.get(id(p))
        if g is None:
            if p.grad is not None and p.grad.dtype == torch.float32 and p.grad.is_contiguous():
                g = p.grad  # accumulate straight into the (flat-buffer) gradient: no copy, no autograd hand-over
                self.direct.add(id(p))
            else:
                g = torch.zeros_like(p, dtype=torch.float32, memory_format=torch.contiguous_format)
            self.grads[id(p)] = g
        return g

    def _encoder_forward_train(self, n, x_n, B, S, device, side_stream):
        """One signal encoder with every layer output kept (on the current stream); returns its saved-state dict."""
        lib, m = self.lib, self.model
        st = _stream()
        enc = m.signal_encoders.get_encoder(n)
        pe = self.enc[m.signal_encoders.signal_map[n]]
        xs = _f32(x_n)
        if side_stream is not None:
            xs.record_stream(side_stream)
        T = xs.size(1)
        ws_bytes = lib.w2s_encoder_workspace_bytes(C.byref(pe.desc), B, T, 1)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=device)
        mask = torch.zeros(B, dtype=torch.uint8, device=device)
        z_unused = torch.empty(B, S, 128, dtype=F16, device=device)
        _lib.check(lib.w2s_encoder_fwd(C.byref(pe.desc), xs.data_ptr(), B, T, ws.data_ptr(), ws_bytes, 1,
                                       z_unused.data_ptr(), mask.data_ptr(), st), ValueError)
        nb = len(enc.channels)
        offs = (C.c_int64 * (7 * nb))()
        _lib.check(lib.w2s_encoder_layout(C.byref(pe.desc), B, T, offs))
        e = {"x": xs, "ws": ws, "mask": mask, "T": T, "blocks": [], "enc": enc,
             "tw": self.tw["enc"][m.signal_encoders.signal_map[n]]}
        L = T
        for i, c in enumerate(enc.channels):
            o = offs[7 * i:7 * i + 7]
            view = lambda off, rows, ch: ws[off: off + B * rows * ch * 2].view(F16).view(B, rows, ch)
            stat = lambda off, ch: ws[off: off + B * ch * 16].view(torch.float64).view(B, ch, 2)
            e["blocks"].append({"C": c, "L": L, "s1": stat(o[0], c), "s2": stat(o[1], c), "s3": stat(o[2], c),
                                "y1": view(o[3], L, c), "r": view(o[4], L // 2, c), "y2": view(o[5], L, c),
                                "y3": view(o[6], L // 2, c)})
            L //= 2
        # time-distributed linear on the re-materialised activated block output
        last = e["blocks"][-1]
        Cl, L4 = last["C"], last["L"] // 2  # L4 = 4 * S
        a_last = torch.empty(B, L4, Cl, dtype=F16, device=device)
        _lib.check(lib.w2s_enc_act_fwd(last["y3"].data_ptr(), last["r"].data_ptr(), last["s3"].data_ptr(),
                                       a_last.data_ptr(), mask.data_ptr(), B, L4, Cl, enc.norm_eps, st))
        z_pre = torch.zeros(B, S, 128, dtype=F16, device=device)
        bl = _f32(enc.linear.bias)
        self.conv(a_last, e["tw"]["lin_fwd"], Cl, 128, 4, B, L4, S, z_pre, stride=4, bias=bl, row_mask=mask)
        z = torch.zeros(B, S, 128, dtype=F16, device=device)
        _lib.check(lib.w2s_gelu_fwd(z_pre.data_ptr(), z.data_ptr(), z.numel(), st))
        e.update(a_last=a_last, z_pre=z_pre, z=z)
        return e

    # ================================================================== forward (training)
    @torch.no_grad()
    def forward_train(self, x: dict[str, Tensor], return_saved: bool = False):
        """Training-mode forward.  The activations the backward needs are returned (``return_saved``: the autograd bridge
        keeps them on its ``ctx``, so several forwards may precede their backwards, like with torch autograd) and also
        remembered as ``self.saved`` for a direct ``backward(dlogits)`` call."""
        names, B, S, device = check_inputs(self.model.signal_encoders, x)
        lib, m = self.lib, self.model
        with torch.cuda.device(device):
            self._ensure_train_packed(device)
            st = _stream()
            N = B * S
            sv = {"B": B, "S": S, "names": names, "enc": {}, "device": device}
            seed = self.last_dropout_seed = _dropout_seed(self.dropout_seed)
            p_mix = float(m.epoch_mixer.dropout) if m.training else 0.0
            sv.update(seed=seed, p_mix=p_mix)
            # ---- encoders (streaming kernels, every layer output kept), one CUDA stream each, longest first ----
            order = sorted(names, key=lambda k: -x[k].size(1))
            streams = self._encoder_streams(device, len(order))
            for si, n in enumerate(order):
                with (torch.cuda.stream(streams[si]) if streams is not None else contextlib.nullcontext()):
                    sv["enc"][n] = self._encoder_forward_train(n, x[n], B, S, device,
                                                               streams[si] if streams is not None else None)
            self._join(streams, device)
            st = _stream()
            # ---- epoch mixer (un-fused) ----
            mix = m.epoch_mixer
            D = len(names) + 1
            T_tok = N * D
            zs = (C.c_void_p * len(names))(*[sv["enc"][n]["z"].data_ptr() for n in names])
            ms = (C.c_void_p * len(names))(*[sv["enc"][n]["mask"].data_ptr() for n in names])
            tokens = torch.empty(T_tok, 128, dtype=F16, device=device)
            key_mask = torch.empty(T_tok, dtype=torch.uint8, device=device)
            cls = _f32(mix.register_tokens[0, 0, :, 0])
            _lib.check(lib.w2s_tokens_fwd(zs, ms, cls.data_ptr(), tokens.data_ptr(), key_mask.data_ptr(), N, S, len(names), st))
            sv.update(D=D, key_mask=key_mask, layers=[])
            xcur = tokens
            for l, layer in enumerate(mix.transformer_encoder.layers):
                tw = self.tw["mix"][l]
                eps = layer.norm1.eps
                f = _f32
                h1 = self.ln_fwd(xcur, f(layer.norm1.weight), f(layer.norm1.bias), T_tok, 0, eps)
                qkv = []
                bin_ = f(layer.self_attn.in_proj_bias)
                for j in range(3):
                    o = torch.empty(T_tok, 128, dtype=F16, device=device)
                    self.conv(h1, tw["qkv"][j], 128, 128, 1, 1, T_tok, T_tok, o, bias=bin_[j * 128:(j + 1) * 128])
                    qkv.append(o)
                ao = torch.empty(T_tok, 128, dtype=F16, device=device)
                _lib.check(lib.w2s_attn_fwd(qkv[0].data_ptr(), qkv[1].data_ptr(), qkv[2].data_ptr(), ao.data_ptr(),
                                            key_mask.data_ptr(), N, D, p_mix, seed, 8 * l, st))
                x_mid = torch.empty(T_tok, 128, dtype=F16, device=device)
                if p_mix > 0:  # x + dropout1(out_proj(attention))
                    self.conv(ao, tw["o"], 128, 128, 1, 1, T_tok, T_tok, x_mid, bias=f(layer.self_attn.out_proj.bias))
                    self.dropout(x_mid, 8 * l + 1, p_mix, seed, res=xcur, out=x_mid)
                else:
                    self.conv(ao, tw["o"], 128, 128, 1, 1, T_tok, T_tok, x_mid, bias=f(layer.self_attn.out_proj.bias),
                              res=xcur)
                h2 = self.ln_fwd(x_mid, f(layer.norm2.weight), f(layer.norm2.bias), T_tok, 0, eps)
                hpre = torch.empty(4 * T_tok, 128, dtype=F16, device=device)  # [T, 512] row-major
                b1 = f(layer.linear1.bias)
                for j in range(4):
                    self.conv(h2, tw["ff1"][j], 128, 128, 1, 1, T_tok, T_tok, hpre, bias=b1[j * 128:(j + 1) * 128],
                              out_stride=4, out_offset=j, out_rows=4 * T_tok)
                hact = torch.empty_like(hpre)
                _lib.check(lib.w2s_gelu_fwd(hpre.data_ptr(), hact.data_ptr(), hpre.numel(), st))
                x_out = torch.empty(T_tok, 128, dtype=F16, device=device)
                if p_mix > 0:  # x + dropout2(linear2(dropout(gelu(linear1(.)))))
                    self.dropout(hact, 8 * l + 2, p_mix, seed, out=hact)
                    self.conv(hact, tw["ff2"], 128, 128, 4, 1, 4 * T_tok, T_tok, x_out, stride=4, bias=f(layer.linear2.bias))
                    self.dropout(x_out, 8 * l + 3, p_mix, seed, res=x_mid, out=x_out)
                else:
                    self.conv(hact, tw["ff2"], 128, 128, 4, 1, 4 * T_tok, T_tok, x_out, stride=4,
                              bias=f(layer.linear2.bias), res=x_mid)
                sv["layers"].append(dict(x=xcur, h1=h1, q=qkv[0], k=qkv[1], v=qkv[2], ao=ao, x_mid=x_mid, h2=h2, hpre=hpre,
                                         hact=hact))
                xcur = x_out
            mixed = torch.empty(N, 128, dtype=F16, device=device)
            _lib.check(lib.w2s_rows_gather(xcur.data_ptr(), mixed.data_ptr(), N, D, 0, 0, st))
            # ---- sequence mixer (un-fused) + classifier ----
            sv["seq"] = []
            blk_in = mixed
            for bi, blk in enumerate(m.sequence_mixer.dilated_convs):
                cur = blk_in
                rec = {"in": blk_in, "layers": []}
                nl = len(blk.conv_layers)
                for k, layer in enumerate(blk.conv_layers):
                    d = blk.dilations[k]
                    c = torch.empty(B, S, 128, dtype=F16, device=device)
                    self.conv(cur, self.tw["seq"][bi][k]["fwd"], 128, 128, 7, B, S, S, c, dil=d, pad=3 * d)
                    g_, b_ = _f32(layer.norm.weight.reshape(-1)), _f32(layer.norm.bias.reshape(-1))
                    p_seq = float(blk.dropout.p) if m.training else 0.0
                    lrec = {"in": cur, "c": c, "g": g_, "b": b_, "eps": layer.norm.eps, "d": d}
                    if k == nl - 1 and p_seq > 0:  # gelu(dropout(layers(x)) + x), models/blocks.py:123-125
                        y = self.ln_fwd(c.view(N, 128), g_, b_, N, 1, layer.norm.eps)
                        t = self.dropout(y, 64 + bi, p_seq, seed, res=blk_in.view(N, 128), out=y)
                        y = torch.empty(B, S, 128, dtype=F16, device=device)
                        _lib.check(lib.w2s_gelu_fwd(t.data_ptr(), y.data_ptr(), t.numel(), st))
                        lrec.update(t=t, p=p_seq)
                    else:
                        y = self.ln_fwd(c.view(N, 128), g_, b_, N, 1, layer.norm.eps,
                                        res=blk_in.view(N, 128) if k == nl - 1 else None).view(B, S, 128)
                    rec["layers"].append(lrec)
                    cur = y
                sv["seq"].append(rec)
                blk_in = cur
            feat = blk_in
            logits = torch.empty(B, S, m.num_classes, dtype=torch.float32, device=device)
            wc, bc = _f32(m.classifier.weight), _f32(m.classifier.bias)
            _lib.check(lib.w2s_head_fwd(feat.data_ptr(), wc.data_ptr(), bc.data_ptr(), logits.data_ptr(), N, m.num_classes, st))
            sv.update(feat=feat, wc=wc)
            self.saved = sv
        return (logits, sv) if return_saved else logits

    # ================================================================== backward
    @torch.no_grad()
    def backward(self, dlogits: Tensor, saved: dict | None = None, inputs=()) -> dict[int, Tensor]:
        """Back-propagates d(loss)/d(logits) through a saved forward (``saved``: what forward_train returned; default:
        the most recent forward); returns {id(param): fp32 grad} for the parameters that require grad.  ``inputs``:
        signals whose d(loss)/dx is wanted as well, left in ``self.input_grads`` (fp32 [B, T]).  A saved forward can be
        back-propagated once."""
        sv, lib, m = (self.saved if saved is None else saved), self.lib, self.model
        if sv is None:
            raise RuntimeError("backward called without a preceding forward_train")
        if sv.get("consumed"):
            raise RuntimeError("this forward has already been back-propagated (its activations were released)")
        B, S, device = sv["B"], sv["S"], sv["device"]
        N = B * S
        self.grads = {}
        self.direct = set()
        self._wg = None
        inputs = set(inputs)
        self.input_grads = {}
        with torch.cuda.device(device):
            dlogits = dlogits.detach().to(torch.float32).contiguous()
            if self.loss_scale is not None:
                scale = float(self.loss_scale)
            elif inputs:
                amax = torch.empty(1, dtype=torch.float32, device=device)
                _lib.check(lib.w2s_absmax(dlogits.data_ptr(), dlogits.numel(), amax.data_ptr(), _stream()))
                amax = amax.item()
                if amax == 0.0:  # every gradient is exactly zero: nothing to launch
                    return self._zero_backward(sv, inputs)
                scale = self.attribution_loss_scale(amax)
            else:
                scale = self.auto_loss_scale(N)
            if scale <= 0 or (scale != 2.0 ** round(math.log2(scale))):
                raise ValueError(f"loss_scale must be a positive power of two, got {scale}")
            self.last_loss_scale, self._inv_scale = scale, 1.0 / scale
            st = _stream()
            G = self._grad
            Gv = lambda p: None if G(p) is None else G(p).view(-1)
            self._wg = self._wg_streams.setdefault(str(device), torch.cuda.Stream(device=device))
            # ---- classifier ----
            dfeat = torch.empty(N, 128, dtype=F16, device=device)
            _lib.check(lib.w2s_head_bwd(sv["feat"].data_ptr(), sv["wc"].data_ptr(), dlogits.data_ptr(), dfeat.data_ptr(),
                                        _p(G(m.classifier.weight)), _p(G(m.classifier.bias)), N,
                                        m.num_classes, scale, st))
            # ---- sequence mixer ----
            dout = dfeat
            for bi in reversed(range(len(sv["seq"]))):
                rec, blk = sv["seq"][bi], m.sequence_mixer.dilated_convs[bi]
                nl = len(rec["layers"])
                ds = None
                for k in reversed(range(nl)):
                    lr, layer = rec["layers"][k], blk.conv_layers[k]
                    dg, db = Gv(layer.norm.weight), Gv(layer.norm.bias)
                    last = k == nl - 1
                    if last and "t" in lr:  # dropout between the layers and the residual add
                        ds = torch.empty(N, 128, dtype=F16, device=device)
                        _lib.check(lib.w2s_gelu_bwd(lr["t"].data_ptr(), dout.data_ptr(), ds.data_ptr(), ds.numel(), st))
                        dy = self.dropout(ds, 64 + bi, lr["p"], sv["seed"])
                        dc, _ = self.ln_bwd(lr["c"].view(N, 128), lr["g"], lr["b"], dy, dg, db, N, 1, lr["eps"])
                    else:
                        dc, ds_k = self.ln_bwd(lr["c"].view(N, 128), lr["g"], lr["b"], dout, dg, db, N, 1, lr["eps"],
                                               res=rec["in"].view(N, 128) if last else None, want_ds=last)
                        if last:
                            ds = ds_k
                    d = lr["d"]
                    dW = G(layer.conv.weight)
                    self.gemm_tn(dc, lr["in"], dW, 128, 128, B, S, S, 128 * 7, 7, y_offset=-3 * d, taps=7, tap_stride=d, ldc_t=1)
                    din = torch.empty(N, 128, dtype=F16, device=device)
                    self.conv(dc, self.tw["seq"][bi][k]["T"], 128, 128, 7, B, S, S, din, dil=d, pad=3 * d,
                              res=ds if k == 0 else None)
                    dout = din
            dmix = dout  # [N, 128]
            # ---- epoch mixer ----
            D, key_mask = sv["D"], sv["key_mask"]
            T_tok = N * D
            dx = torch.zeros(T_tok, 128, dtype=F16, device=device)
            _lib.check(lib.w2s_rows_gather(dmix.data_ptr(), dx.data_ptr(), N, D, 0, 1, st))
            mix = m.epoch_mixer
            for l in reversed(range(len(sv["layers"]))):
                L_, layer, tw = sv["layers"][l], mix.transformer_encoder.layers[l], self.tw["mix"][l]
                eps = layer.norm1.eps
                f = _f32
                # FFN
                dW2, dW1 = G(layer.linear2.weight), G(layer.linear1.weight)
                d_hact = torch.empty(4 * T_tok, 128, dtype=F16, device=device)
                p_mix, seed = sv["p_mix"], sv["seed"]
                g2 = self.dropout(dx, 8 * l + 3, p_mix, seed) if p_mix > 0 else dx  # gradient of the linear2 output
                for j in range(4):
                    self.conv(g2, tw["ff2_T"][j], 128, 128, 1, 1, T_tok, T_tok, d_hact, out_stride=4, out_offset=j,
                              out_rows=4 * T_tok)
                    self.gemm_tn(g2, L_["hact"], dW2, 128, 128, 1, T_tok, 4 * T_tok, 512, 1, y_stride=4, y_offset=j, c_off=j * 128)
                self.colsum(g2, G(layer.linear2.bias), T_tok, 128)
                if p_mix > 0:
                    self.dropout(d_hact, 8 * l + 2, p_mix, seed, out=d_hact)
                d_hpre = torch.empty_like(d_hact)
                _lib.check(lib.w2s_gelu_bwd(L_["hpre"].data_ptr(), d_hact.data_ptr(), d_hpre.data_ptr(), d_hact.numel(), st))
                for j in range(4):
                    # dW1[j*128 + n, m] += sum_o h2[o, m] * d_hpre[4o + j, n]   (transposed addressing of C)
                    self.gemm_tn(L_["h2"], d_hpre, dW1, 128, 128, 1, T_tok, 4 * T_tok, 1, 128, y_stride=4, y_offset=j,
                                 c_off=j * 128 * 128)
                    self.colsum(d_hpre, G(layer.linear1.bias), T_tok, 128, row_stride=4, row_offset=j, out_off=j * 128)
                d_h2 = torch.empty(T_tok, 128, dtype=F16, device=device)
                self.conv(d_hpre, tw["ff1_T"], 128, 128, 4, 1, 4 * T_tok, T_tok, d_h2, stride=4)
                dx_mid, _ = self.ln_bwd(L_["x_mid"], f(layer.norm2.weight), f(layer.norm2.bias), d_h2, G(layer.norm2.weight),
                                        G(layer.norm2.bias), T_tok, 0, eps, dadd=dx)
                # attention
                d_ao = torch.empty(T_tok, 128, dtype=F16, device=device)
                g1 = self.dropout(dx_mid, 8 * l + 1, p_mix, seed) if p_mix > 0 else dx_mid  # gradient of out_proj's output
                self.conv(g1, tw["o_T"], 128, 128, 1, 1, T_tok, T_tok, d_ao)
                self.gemm_tn(g1, L_["ao"], G(layer.self_attn.out_proj.weight), 128, 128, 1, T_tok, T_tok, 128, 1)
                self.colsum(g1, G(layer.self_attn.out_proj.bias), T_tok, 128)
                dq, dk, dv = (torch.empty(T_tok, 128, dtype=F16, device=device) for _ in range(3))
                _lib.check(lib.w2s_attn_bwd(L_["q"].data_ptr(), L_["k"].data_ptr(), L_["v"].data_ptr(), d_ao.data_ptr(),
                                            dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), key_mask.data_ptr(), N, D, p_mix,
                                            seed, 8 * l, st))
                dWin, dbin = G(layer.self_attn.in_proj_weight), G(layer.self_attn.in_proj_bias)
                d_h1 = None
                for j, dj in enumerate((dq, dk, dv)):
                    self.gemm_tn(dj, L_["h1"], dWin, 128, 128, 1, T_tok, T_tok, 128, 1, c_off=j * 128 * 128)
                    self.colsum(dj, dbin, T_tok, 128, out_off=j * 128)
                    nxt = torch.empty(T_tok, 128, dtype=F16, device=device)
                    self.conv(dj, tw["qkv_T"][j], 128, 128, 1, 1, T_tok, T_tok, nxt, res=d_h1)
                    d_h1 = nxt
                dx, _ = self.ln_bwd(L_["x"], f(layer.norm1.weight), f(layer.norm1.bias), d_h1, G(layer.norm1.weight),
                                    G(layer.norm1.bias), T_tok, 0, eps, dadd=dx_mid)
            names = sv["names"]
            dz = {n: torch.zeros(B, S, 128, dtype=F16, device=device) for n in names}
            dzs = (C.c_void_p * len(names))(*[dz[n].data_ptr() for n in names])
            ms = (C.c_void_p * len(names))(*[sv["enc"][n]["mask"].data_ptr() for n in names])
            # register_tokens is [1, 1, 128, 1]: with no extra register tokens its gradient is the 128 CLS sums
            _lib.check(lib.w2s_tokens_bwd(dx.data_ptr(), dzs, ms, _p(G(mix.register_tokens)), N, S, len(names),
                                          self._inv_scale, st))
            # ---- encoders ----
            if self._wg is not None:  # the side stream's weight gradients are part of the "tail" bucket
                torch.cuda.current_stream(device).wait_stream(self._wg)
                self._wg = None
            for hook in self.bucket_hooks:
                hook("tail")  # classifier + sequence mixer + epoch mixer gradients are final
            if self.bucket_hooks and len(self.direct) != len(self.grads):
                raise RuntimeError("gradient bucket hooks (data-parallel all-reduce) need every p.grad to be its view of "
                                   "the optimizer's flat buffer during the backward: clear gradients with "
                                   "FusedAdamW.zero_grad(), not model.zero_grad() / p.grad = None")
            # largest encoders first, so that the exposed tail of the data-parallel exchange is the smallest bucket
            order = sorted(names, key=lambda n: -sv["enc"][n]["T"])
            smap = m.signal_encoders.signal_map
            pending = {}  # encoder name -> signals still to back-propagate (encoders may be shared between signals)
            for n in order:
                pending[smap[n]] = pending.get(smap[n], 0) + 1
            shared = len(set(smap[n] for n in order)) < len(order)  # a shared encoder: its passes stay in stream order
            streams = None if shared else self._encoder_streams(device, len(order))
            main = torch.cuda.current_stream(device)
            for si, n in enumerate(order):
                with (torch.cuda.stream(streams[si]) if streams is not None else contextlib.nullcontext()):
                    if streams is not None:
                        dz[n].record_stream(streams[si])
                    enc = sv["enc"][n]["enc"]
                    if n in inputs or any(p.requires_grad for p in enc.parameters()):
                        dxn = self._encoder_backward(sv["enc"][n], dz[n], B, S, want_dx=n in inputs)
                        if dxn is not None:
                            if streams is not None:
                                dxn.record_stream(main)
                            self.input_grads[n] = dxn
                    sv["enc"][n] = None  # release this encoder's activations
                    pending[smap[n]] -= 1
                    if pending[smap[n]] == 0:
                        for hook in self.bucket_hooks:
                            hook("encoder:" + smap[n])  # this encoder's parameter gradients are final
            self._join(streams, device)
            for hook in self.bucket_hooks:
                hook("encoders")
            sv["consumed"] = True
            for k in ("layers", "seq", "feat", "key_mask"):
                sv.pop(k, None)
            if self.saved is sv:
                self.saved = None
        return self.grads

    def _zero_backward(self, sv, inputs):
        """d(objective)/d(logits) is exactly zero: so is every gradient.  No kernel runs; the bucket hooks still fire."""
        B, device = sv["B"], sv["device"]
        self.grads = {id(p): torch.zeros_like(p, dtype=torch.float32) for p in self.model.parameters() if p.requires_grad}
        self.input_grads = {n: torch.zeros(B, sv["enc"][n]["T"], dtype=torch.float32, device=device) for n in inputs}
        smap = self.model.signal_encoders.signal_map
        for bucket in ["tail"] + sorted({"encoder:" + smap[n] for n in sv["names"]}) + ["encoders"]:
            for hook in self.bucket_hooks:
                hook(bucket)
        sv["consumed"] = True
        for k in ("layers", "seq", "feat", "key_mask", "enc"):
            sv.pop(k, None)
        if self.saved is sv:
            self.saved = None
        self.last_loss_scale, self._inv_scale = 1.0, 1.0
        return self.grads

    def _encoder_backward(self, e, dz, B, S, want_dx=False):
        lib, st, G = self.lib, _stream(), self._grad
        enc, mask, tw, device = e["enc"], e["mask"], e["tw"], dz.device
        eps = enc.norm_eps
        blocks = e["blocks"]
        last = blocks[-1]
        Cl, L4 = last["C"], last["L"] // 2
        new = lambda *shape: torch.empty(*shape, dtype=F16, device=device)
        zeros64 = lambda c: torch.zeros(B, c, 2, dtype=torch.float64, device=device)
        # linear + GELU
        d_zpre = new(B, S, 128)
        _lib.check(lib.w2s_gelu_bwd(e["z_pre"].data_ptr(), dz.data_ptr(), d_zpre.data_ptr(), dz.numel(), st))
        dWl = G(enc.linear.weight)
        d_a = new(B, L4, Cl)
        for t in range(4):
            self.gemm_tn(d_zpre, e["a_last"], dWl, 128, Cl, B, S, L4, 4 * Cl, 1, y_stride=4, y_offset=t, row_mask=mask,
                         c_off=t * Cl)
            self.conv(d_zpre, tw["lin_dgrad"][t], 128, Cl, 1, B, S, S, d_a, out_stride=4, out_offset=t, out_rows=L4,
                      row_mask=mask)
        self.colsum(d_zpre, G(enc.linear.bias), B * S, 128, row_mask=mask, rows_per_sample=S)
        # The backward through a layer's activation (GELU', residual add, the two InstanceNorm reductions) runs in the
        # epilogue of the data-gradient conv that produces its input gradient (EPI_ACT_BWD), which also writes the
        # activated tensor that conv's own weight gradient needs - so each weight gradient runs right after its data
        # gradient.  Only the last block's output (fed by the Linear) goes through the stand-alone enc_act_bwd kernel.
        nb = len(blocks)
        last_bk = blocks[-1]
        Cc, Lh = last_bk["C"], last_bk["L"] // 2
        dxh, dr, sums = new(B, Lh, Cc), new(B, Lh, Cc), zeros64(Cc)
        _lib.check(lib.w2s_enc_act_bwd(d_a.data_ptr(), last_bk["y3"].data_ptr(), last_bk["r"].data_ptr(),
                                       last_bk["s3"].data_ptr(), dxh.data_ptr(), dr.data_ptr(), sums.data_ptr(), None,
                                       mask.data_ptr(), B, Lh, Cc, eps, st))
        for i in reversed(range(nb)):
            bk, blk = blocks[i], enc.cnn[i]
            Cc, L = bk["C"], bk["L"]
            Lh = L // 2
            # here: dxh / dr / sums = backward through this block's output activation GELU(GELU(IN(y3)) + r)
            dy_up = new(B, L, Cc)  # even rows = dy, odd rows = zeros (written by the kernel): transposed stride-2 conv
            fuse = self.fuse_norm_bwd
            if not fuse:
                _lib.check(lib.w2s_enc_norm_bwd(dxh.data_ptr(), bk["y3"].data_ptr(), bk["s3"].data_ptr(), sums.data_ptr(),
                                                dy_up.data_ptr(), mask.data_ptr(), B, Lh, Cc, 1, eps, st))
            # ---- conv3 (stride 2): data gradient + backward through GELU(IN(y2)) in one kernel ----
            dn = (dxh, bk["y3"], bk["s3"], sums, 1) if fuse else None
            dxh, a2, sums = new(B, L, Cc), new(B, L, Cc), zeros64(Cc)
            self.conv_act_bwd(dy_up, tw["conv"][i][2], Cc, Cc, B, L, bk["y2"], bk["s2"], sums, dxh, a2, eps, mask, dnorm=dn)
            self.gemm_tn(dy_up, a2, G(blk.conv3.conv.weight), Cc, Cc, B, L, L, Cc * 3, 3, y_offset=-1, row_mask=mask,
                         taps=3, ldc_t=1)
            del dy_up
            # ---- conv2 ----
            dy2 = a2  # a2 is consumed: reuse its storage
            if not fuse:
                _lib.check(lib.w2s_enc_norm_bwd(dxh.data_ptr(), bk["y2"].data_ptr(), bk["s2"].data_ptr(), sums.data_ptr(),
                                                dy2.data_ptr(), mask.data_ptr(), B, L, Cc, 0, eps, st))
                dn, dxh_next = None, dxh  # (the un-fused kernel may overwrite d(x_hat) in place)
            else:
                dn, dxh_next = (dxh, bk["y2"], bk["s2"], sums, 0), new(B, L, Cc)
            a1, sums = new(B, L, Cc), zeros64(Cc)
            self.conv_act_bwd(dy2, tw["conv"][i][1], Cc, Cc, B, L, bk["y1"], bk["s1"], sums, dxh_next, a1, eps, mask, dnorm=dn)
            dxh = dxh_next
            self.gemm_tn(dy2, a1, G(blk.conv2.conv.weight), Cc, Cc, B, L, L, Cc * 3, 3, y_offset=-1, row_mask=mask, taps=3,
                         ldc_t=1)
            del dy2, a2
            # ---- conv1 (+ 1x1 stride-2 residual branch) ----
            dy1 = a1
            fuse1 = fuse and i > 0  # block 0 has no data gradient to fuse into (its input is the raw signal)
            if not fuse1:
                _lib.check(lib.w2s_enc_norm_bwd(dxh.data_ptr(), bk["y1"].data_ptr(), bk["s1"].data_ptr(), sums.data_ptr(),
                                                dy1.data_ptr(), mask.data_ptr(), B, L, Cc, 0, eps, st))
            dn = (dxh, bk["y1"], bk["s1"], sums, 0) if fuse1 else None
            del dxh
            if i == 0:
                dw1, dwds = G(blk.conv1.conv.weight), G(blk.downsample.weight)
                if dw1 is not None or dwds is not None:  # the kernel computes both: a frozen one goes to scratch
                    dw1 = torch.zeros(16, 1, 3, device=device) if dw1 is None else dw1
                    dwds = torch.zeros(16, 1, 1, device=device) if dwds is None else dwds
                    _lib.check(lib.w2s_first_conv_wgrad(e["x"].data_ptr(), dy1.data_ptr(), dr.data_ptr(), dw1.data_ptr(),
                                                        dwds.data_ptr(), mask.data_ptr(), B, L, self._inv_scale, st))
                if want_dx:
                    dx = torch.empty(B, L, dtype=torch.float32, device=device)
                    _lib.check(lib.w2s_first_conv_dgrad(e["x"].data_ptr(), dy1.data_ptr(), dr.data_ptr(),
                                                        _f32(blk.conv1.conv.weight).data_ptr(),
                                                        _f32(blk.downsample.weight).data_ptr(), mask.data_ptr(),
                                                        dx.data_ptr(), B, L, self._inv_scale, st))
                    return dx
                return None
            pb = blocks[i - 1]
            Ci = pb["C"]
            tmp = torch.zeros(B, L, Ci, dtype=F16, device=device)
            self.conv(dr, tw["ds"][i], Cc, Ci, 1, B, Lh, Lh, tmp, out_stride=2, out_offset=0, out_rows=L, row_mask=mask)
            # data gradient of conv1 (+ the residual-branch gradient) fused with the backward through the previous
            # block's output activation; a_in is this block's input, needed by the two weight gradients below
            dxh_p, dr_p, a_in, sums = new(B, L, Ci), new(B, L, Ci), new(B, L, Ci), zeros64(Ci)
            self.conv_act_bwd(dy1, tw["conv"][i][0], Cc, Ci, B, L, pb["y3"], pb["s3"], sums, dxh_p, a_in, eps, mask,
                              res=tmp, r=pb["r"], dr=dr_p, dnorm=dn)
            dn = None
            del tmp
            self.gemm_tn(dy1, a_in, G(blk.conv1.conv.weight), Cc, Ci, B, L, L, Ci * 3, 3, y_offset=-1, row_mask=mask,
                         taps=3, ldc_t=1)
            self.gemm_tn(dr, a_in, G(blk.downsample.weight), Cc, Ci, B, Lh, L, Ci, 1, y_stride=2, y_offset=0,
                         row_mask=mask)
            del dy1, dr, a_in, a1
            dxh, dr = dxh_p, dr_p


class _TrainFn(torch.autograd.Function):
    """autograd bridge: ``logits = model(x)`` gets a grad_fn whose backward runs the CUDA backward.  The signals are
    inputs of the graph (in ``names`` order, then the parameters), so ``x[name].grad`` receives d(objective)/dx where
    ``x[name].requires_grad``."""

    @staticmethod
    def forward(ctx, engine, names, *tensors):
        n = len(names)
        ctx.engine, ctx.names = engine, names
        ctx.dtypes, ctx.params = [t.dtype for t in tensors[:n]], tensors[n:]
        # per-graph state, like autograd's saved tensors
        logits, ctx.saved = engine.forward_train(dict(zip(names, tensors[:n])), return_saved=True)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        wanted = [name for i, name in enumerate(ctx.names) if ctx.needs_input_grad[2 + i]]
        grads = ctx.engine.backward(dlogits, ctx.saved, inputs=wanted)
        dx = ctx.engine.input_grads
        ctx.saved = None
        out = [dx[name].to(dt) if name in dx else None for name, dt in zip(ctx.names, ctx.dtypes)]
        for p in ctx.params:
            g = grads.get(id(p))
            direct = id(p) in ctx.engine.direct  # already accumulated into p.grad by the kernels
            out.append(None if (g is None or direct) else g.to(p.dtype).view_as(p))
        return (None, None, *out)


def forward_with_grad(model, x: dict[str, Tensor]) -> Tensor:
    eng = model._get_train_engine()
    params = tuple(p for p in model.parameters() if p.requires_grad)
    names = tuple(check_inputs(model.signal_encoders, x)[0])  # before x is unpacked
    return _TrainFn.apply(eng, names, *(x[n] for n in names), *params)
