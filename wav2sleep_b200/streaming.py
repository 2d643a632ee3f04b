"""Epoch-by-epoch inference of causal models with carried state (real-time use: one stream per bed).

A causal ``Wav2Sleep`` gives the logits of epoch t from the epochs up to t only, so a new epoch needs just a bounded
piece of the past: nothing for a chunk-causal encoder (each epoch is its own sample), the last (k-1)*d = 2 input rows of
every causal conv layer of a causal-conv encoder, and the last (k-1)*d input rows of every dilated layer of the causal
sequence mixer.  ``StreamingSession`` keeps that state on the device for N streams, so each call costs O(R) work for R
new epochs instead of a forward over the whole prefix of the night.

    sess = StreamingSession(model, n_streams=N)
    logits = sess.step({"ECG": x_ecg, "PPG": x_ppg})   # [N, R * samples_per_epoch] fp32 -> [N, R, num_classes]
    preds = sess.predict_step({...})                   # int64 [N, R]
    sess.reset([2])                                    # stream 2 starts a new night

The logits of epoch t of a stream equal ``model(x)[:, t]`` of the full-night forward over that stream's data since its
last ``reset``.  Semantics per call:
  * a stream's chunk of a signal is missing when its first sample is -inf (the reference's row rule); an absent key
    means that signal is missing for every stream.  Missing chunks are key-masked in the epoch mixer, and a causal-conv
    encoder restarts after one: that signal's context rows of the stream are zeroed.
  * non-finite samples inside a present chunk of the raw signal read as 0 (``w2s_gen_conv``'s raw_inf_to_zero).
  * eval semantics whatever ``model.training`` says: running BatchNorm statistics, no dropout, no autograd.

Compute: encoders and epoch mixer are the general path's kernels (``GeneralEngine.encode`` / ``epoch_mixer``; a
causal-conv encoder runs each conv on [context, chunk] without padding); the sequence mixer and classifier are one launch
of ``w2s_gen_seq_stream_step`` (csrc/stream.cuh) with its ring buffers.
"""
from __future__ import annotations

import ctypes as C

import torch
from torch import Tensor

from . import _lib
from .engine import _argmax, _f32, _p, _stream, check_inputs
from .general import ACT, GeneralEngine
from .model import Wav2Sleep

_PER_POSITION_NORMS = ("batch", "layer", "rms", None)
_SEQ_NORM = {None: 0, "batch": 1, "layer": 2, "rms": 3}


def _check_streamable(model) -> None:
    """ValueError naming the first component that is not causal (prefix-invariant), or that the kernel cannot take."""
    if not isinstance(model, Wav2Sleep):
        raise ValueError(f"{type(model).__name__} is not a causal Wav2Sleep model; only those stream")
    encs = model.signal_encoders
    if not encs.causal:
        raise ValueError("signal_encoders is not causal (causal=False): its features depend on later epochs")
    for name, enc in encs.encoders.items():
        if not enc.chunk_causal:
            bad = [(i, n) for i, n in enumerate(enc.block_norms) if n not in _PER_POSITION_NORMS]
            if bad:
                i, n = bad[0]
                raise ValueError(f"signal_encoders.encoders[{name!r}]: causal-conv block {i} has norm {n!r}, whose statistics "
                                 "span the whole night; streaming needs a per-position norm (batch, layer, rms or none)")
    seq = model.sequence_mixer
    blk = seq.dilated_convs[0]
    norm = blk.conv_layers[0].norm_name
    if not seq.causal:
        raise ValueError("sequence_mixer is not causal (causal=False): its output depends on later epochs")
    if norm not in _PER_POSITION_NORMS:
        raise ValueError(f"sequence_mixer has norm {norm!r}, whose statistics span the whole night; streaming needs batch, "
                         "layer, rms or none")
    n_blocks, n_dil, k = len(seq.dilated_convs), len(blk.dilations), blk.kernel_size
    if seq.feature_dim > _lib.STREAM_MAX_FEATURES:
        raise ValueError(f"sequence_mixer feature_dim {seq.feature_dim} > {_lib.STREAM_MAX_FEATURES} (streaming kernel limit)")
    if not 1 <= k <= _lib.STREAM_MAX_KERNEL:
        raise ValueError(f"sequence_mixer kernel_size {k} outside [1, {_lib.STREAM_MAX_KERNEL}] (streaming kernel limit)")
    if not 1 <= n_dil <= _lib.STREAM_MAX_DILATIONS:
        raise ValueError(f"sequence_mixer num_dilations {n_dil} outside [1, {_lib.STREAM_MAX_DILATIONS}] (streaming kernel limit)")
    if not 1 <= n_blocks * n_dil <= _lib.STREAM_MAX_LAYERS:
        raise ValueError(f"sequence_mixer num_layers x num_dilations = {n_blocks * n_dil} > {_lib.STREAM_MAX_LAYERS} "
                         "(streaming kernel limit)")


class StreamingSession:
    """N streams of a causal ``Wav2Sleep`` on its CUDA device, fed R >= 1 new epochs per call (see the module doc)."""

    def __init__(self, model: Wav2Sleep, n_streams: int):
        _check_streamable(model)
        if isinstance(n_streams, bool) or not isinstance(n_streams, int) or n_streams < 1:
            raise ValueError(f"n_streams must be a positive int, got {n_streams!r}")
        dev = model.classifier.weight.device
        if dev.type != "cuda":
            raise RuntimeError("wav2sleep_b200 runs on CUDA (sm_100a) only: move the model with .to('cuda'); there is no "
                               "CPU fallback")
        self.model, self.n_streams, self.device = model, n_streams, dev
        self.eng: GeneralEngine = model._get_general()
        self.lib = self.eng.lib
        seq = model.sequence_mixer
        blk = seq.dilated_convs[0]
        self._k, self._n_dil, self._n_blocks = blk.kernel_size, len(blk.dilations), len(seq.dilated_convs)
        rows = self._n_blocks * (self._k - 1) * (2 ** self._n_dil - 1)
        self.pos = 0  # epochs stepped since the session was built: the ring slot of epoch e is e mod M
        self.ring = torch.zeros(n_streams, rows, seq.feature_dim, dtype=torch.float32, device=dev)
        # per signal name (not per encoder: a shared encoder serves two signals): the last (k-1)*d = 2 input rows of
        # every causal conv layer, [block][conv1, conv2, conv3] of [N, 2, C_in]
        self.context: dict[str, list[list[Tensor]]] = {}
        for name in model.signal_encoders.signal_map:
            enc = model.signal_encoders.get_encoder(name)
            if enc.chunk_causal:
                continue
            ctx, cin = [], 1
            for blk_e in enc.cnn:
                ctx.append([torch.zeros(n_streams, blk_e.conv1.padding, cin, device=dev)]
                           + [torch.zeros(n_streams, layer.padding, layer.conv.in_channels, device=dev)
                              for layer in (blk_e.conv2, blk_e.conv3)])
                cin = blk_e.conv1.conv.out_channels
            self.context[name] = ctx

    # ------------------------------------------------------------------ public
    def step(self, x: dict[str, Tensor]) -> Tensor:
        """{signal: [N, R * samples_per_epoch]} -> logits fp32 [N, R, num_classes] of the R new epochs of every stream.

        A call that raises leaves the session as it was before the call (an error the CUDA device reports asynchronously
        leaves the whole CUDA context unusable, the session with it)."""
        R = self._check(x)
        m = self.model
        N = self.n_streams
        # encode() replaces (never modifies) the context tensors, so this snapshot restores them if a later stage raises
        saved = {name: [list(layers) for layers in ctx] for name, ctx in self.context.items()}
        try:
            with torch.no_grad(), torch.cuda.device(self.device):
                zs, masks = [], []
                for name in sorted(x):  # token order of the mixer, wav2sleep.py:311
                    z, mask = self.encode(name, x[name])
                    if m.signal_encoders.embed_signals:  # wav2sleep.py:155-159
                        e = m.signal_encoders.embedder.weight[m.signal_encoders.sig_to_embedding_idx[name]]
                        z = self.eng.affine_act(z, "linear", shift=e, mask=mask, per_channel=1)
                    zs.append(z)
                    masks.append(mask)
                feat = self.eng.epoch_mixer(zs, masks, N, R)
                logits = self.sequence_step(feat)
        except BaseException:
            self.context = saved
            raise
        for name, ctx in self.context.items():
            if name not in x:  # missing for every stream: that encoder restarts
                for layers in ctx:
                    layers[:] = [torch.zeros_like(t) for t in layers]
        return logits

    def predict_step(self, x: dict[str, Tensor]) -> Tensor:
        """Most likely class of each new epoch, int64 [N, R] (the argmax kernel of ``Wav2Sleep.predict``)."""
        return _argmax(self.lib, self.step(x))

    def reset(self, streams=None) -> None:
        """Zero every carried state of the given stream indices (all streams if None): they start a new night."""
        if streams is None:
            idx = slice(None)
        else:
            idx = torch.as_tensor(streams, dtype=torch.long).reshape(-1)
            if idx.numel() and (idx.min() < 0 or idx.max() >= self.n_streams):
                raise ValueError(f"stream indices {idx.tolist()} outside [0, {self.n_streams})")
            idx = idx.to(self.device)
        with torch.no_grad():
            self.ring[idx] = 0.0
            for ctx in self.context.values():
                for t in (t for layers in ctx for t in layers):
                    t[idx] = 0.0

    # ------------------------------------------------------------------ stages (callable on their own, e.g. by tests)
    def encode(self, name: str, x_NT: Tensor) -> tuple[Tensor, Tensor]:
        """The encoder features of signal ``name`` for R new epochs -> (z [N, R, F], mask [N] uint8), advancing its
        carried context.  Chunk-causal encoders have none and are exactly ``GeneralEngine.encode``."""
        enc = self.model.signal_encoders.get_encoder(name)
        if enc.chunk_causal:
            return self.eng.encode(enc, x_NT)
        N, T = x_NT.shape
        R = T // enc.samples_per_epoch
        xs = _f32(x_NT)
        mask = torch.isinf(xs[:, 0]).to(torch.uint8).contiguous()  # data-dependent control, no arithmetic
        ctx = self.context[name]
        a, raw = xs.view(N, T, 1), 1
        for blk, c in zip(enc.cnn, ctx):  # ConvBlock1D.forward (blocks.py:57-71) with carried context
            y, c[0] = self._conv_layer(a, blk.conv1, c[0], mask, raw)
            y, c[1] = self._conv_layer(y, blk.conv2, c[1], mask, 0)
            y, c[2] = self._conv_layer(y, blk.conv3, c[2], mask, 0)
            if blk.use_residual:  # the 1x1 stride-2 branch needs no context; chunk starts are even at every level
                r = self.eng.conv(a, blk.downsample.weight, None, (a.shape[1] - 1) // 2 + 1, stride=2, mask=mask, raw=raw)
                a = self.eng.affine_act(y, blk.activation_name, res=r, mask=mask)
            else:
                a = self.eng.affine_act(y, blk.activation_name, mask=mask)
            raw = 0
        return self.eng.epoch_features(enc, a, mask, N, R), mask

    def _conv_layer(self, a: Tensor, layer, ctx: Tensor, mask: Tensor, raw: int) -> tuple[Tensor, Tensor]:
        """A causal ConvLayer1D on a chunk a [N, L, C]: the conv runs on [context, chunk] without padding, so output j
        reads chunk rows j*stride - 2 .. j*stride as the full forward does.  Returns (output, next context); the context
        of a missing chunk is zero, so that stream's signal restarts at its next present chunk."""
        full = torch.cat([ctx, a], dim=1)
        y = self.eng.conv(full, layer.conv.weight, layer.conv.bias, a.shape[1] // layer.stride, stride=layer.stride,
                          dil=layer.dilation, mask=mask, raw=raw)
        nxt = full[:, full.shape[1] - layer.padding:].masked_fill(mask.bool()[:, None, None], 0.0).contiguous()
        return self.eng.norm_act(y, layer, layer.activation_name, mask=mask), nxt

    def sequence_step(self, feat: Tensor) -> Tensor:
        """Causal SequenceCNN + classifier for epoch-mixer features [N, R, F] of the next R epochs -> logits [N, R, C]:
        one launch of w2s_gen_seq_stream_step, which reads and advances the ring buffers."""
        m = self.model
        N, R, Fd = feat.shape
        if N != self.n_streams or Fd != m.sequence_mixer.feature_dim:
            raise ValueError(f"features {tuple(feat.shape)} do not match [{self.n_streams}, R, {m.sequence_mixer.feature_dim}]")
        x = _f32(feat)
        keep = [x]  # every fp32 tensor the descriptor points to stays referenced until the launch is enqueued

        def ptr(t):
            t = _f32(t)
            keep.append(t)
            return _p(t)

        seq = m.sequence_mixer
        first = seq.dilated_convs[0].conv_layers[0]
        d = _lib.SeqStreamDesc()
        d.n_blocks, d.n_dilations, d.kernel_size = self._n_blocks, self._n_dil, self._k
        d.feature_dim, d.n_classes = Fd, m.num_classes
        d.norm, d.act = _SEQ_NORM[first.norm_name], ACT[first.activation_name]
        d.eps = float(getattr(first.norm, "eps", 0.0))
        for bi, blk in enumerate(seq.dilated_convs):
            for j, layer in enumerate(blk.conv_layers):
                L = d.layer[bi * self._n_dil + j]
                L.w, L.bias = ptr(layer.conv.weight), ptr(layer.conv.bias)
                if layer.norm_name is not None:
                    norm = layer.norm
                    L.norm_w = ptr(norm.weight.reshape(-1)) if norm.weight is not None else None
                    L.norm_b = ptr(norm.bias.reshape(-1)) if getattr(norm, "bias", None) is not None else None
                    if layer.norm_name == "batch":
                        L.running_mean, L.running_var = ptr(norm.running_mean), ptr(norm.running_var)
        d.head_w, d.head_b = ptr(m.classifier.weight), ptr(m.classifier.bias)
        d.ring = self.ring.data_ptr()
        logits = torch.empty(N, R, m.num_classes, dtype=torch.float32, device=feat.device)
        with torch.cuda.device(feat.device):
            _lib.check(self.lib.w2s_gen_seq_stream_step(C.byref(d), x.data_ptr(), logits.data_ptr(), N, R, self.pos,
                                                        _stream()))
        self.pos += R
        return logits

    # ------------------------------------------------------------------ input checks (host side, before any launch)
    def _check(self, x) -> int:
        _, N, R, device = check_inputs(self.model.signal_encoders, x)
        if device != self.device:
            raise RuntimeError(f"input on {device}, session on {self.device}")
        if N != self.n_streams:
            raise ValueError(f"{N} rows, the session has {self.n_streams} streams")
        if N * R > 65535:
            raise ValueError(f"{self.n_streams} streams x {R} epochs exceed the 65535 epoch rows the encoder kernels take per "
                             "call; send fewer epochs per call")
        return R
