"""Host-side driver of the CUDA forward: packs weights, carves workspaces, calls the C ABI stage by stage.

PyTorch is plumbing here (device memory, current stream); every FLOP of the forward runs in
``libw2s_b200.so``.  Mirrors the call ``model(x)`` of the reference (api.py:181-183, trainer/main.py:114).
"""
from __future__ import annotations

import ctypes as C

import torch
from torch import Tensor

from . import _lib
from ._lib import EncoderDesc, MixerDesc, SeqDesc


def _p(t: Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _f32(t: Tensor | None) -> Tensor | None:
    """A tensor as the kernels read it: detached, fp32, contiguous (no copy when it already is)."""
    return None if t is None else t.detach().to(torch.float32).contiguous()


def _stream() -> int:
    """Raw handle of the current CUDA stream of the current device (the fast C accessor: this is called per launch)."""
    try:
        return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())
    except AttributeError:  # older / newer torch without the private accessors
        return torch.cuda.current_stream().cuda_stream


def _argmax(lib, logits: Tensor) -> Tensor:
    """Most likely class of every epoch of logits [B, S, C] -> int64 [B, S] (first maximum wins), on the current
    stream of the logits' device."""
    B, S, Cn = logits.shape
    out = torch.empty(B, S, dtype=torch.int64, device=logits.device)
    with torch.cuda.device(logits.device):
        _lib.check(lib.w2s_argmax(logits.data_ptr(), B * S, Cn, out.data_ptr(), _stream()))
    return out


def _rank() -> int:
    import torch.distributed as dist
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


def _dropout_seed(fixed: int | None) -> int:
    """The dropout seed of one training forward: ``fixed``, or (None) one drawn from torch's CPU generator and made
    distinct per data-parallel rank."""
    if fixed is not None:
        return int(fixed)
    return int(torch.randint(0, 2 ** 62, (1,)).item()) ^ (0x5851F42D4C957F2D * (1 + _rank()) & (2 ** 62 - 1))


class UnknownSignal(KeyError, ValueError):
    """A signal the model has no encoder for (a KeyError like a dict lookup, and a ValueError like any bad input)."""


class NotASignalDict(ValueError, TypeError):
    """An input that is not a non-empty ``{signal: [B, T]}`` dict."""


def check_inputs(encoders, x, what: str = "", joint: bool = True):
    """The host-side check of a ``Wav2Sleep`` input ``{signal: [B, T]}`` against ``encoders`` (the model's
    ``SignalEncoders``), before any launch and without a device synchronisation -> (sorted names, B, S, device).
    ``what`` prefixes the messages.  ``joint=False`` checks every signal on its own, for callers that encode each one
    separately: an empty dict passes, and B, S and the device may differ between signals (those of the last one are
    returned)."""
    p = f"{what}: " if what else ""
    if not isinstance(x, dict) or (joint and not x):
        raise NotASignalDict(f"{p}No signals provided to MultiModalAttentionEmbedder: expected a non-empty "
                             "{signal: [B, T]} dict")  # wav2sleep.py:312-313
    smap = encoders.signal_map
    B = S = device = None
    for name, t in x.items():
        if name not in smap:
            raise UnknownSignal(f"{p}Signal {name!r} has no encoder (valid: {list(smap)})")
        if not isinstance(t, Tensor) or t.dim() != 2:
            raise ValueError(f"{p}{name}: expected a [B, T] tensor")
        if not t.is_cuda:
            raise RuntimeError(f"{p}wav2sleep_b200 runs on CUDA (sm_100a) only: move inputs with .to('cuda'); there is "
                               "no CPU fallback")
        spe = encoders.get_encoder(name).samples_per_epoch
        if t.size(1) % spe:
            raise ValueError(f"{p}{name}: Input length {t.size(1)} must be divisible by self.samples_per_epoch={spe}.")
        b, s = t.size(0), t.size(1) // spe
        if b == 0 or s == 0:
            raise ValueError(f"{p}{name}: empty batch (B={b}, S={s})")
        if joint and device is not None and t.device != device:
            raise ValueError(f"{p}{name}: on {t.device}, other signals on {device}")
        if joint and B is not None and (b, s) != (B, S):
            raise ValueError(f"{p}{name}: batch/epoch count {(b, s)} differs from {(B, S)}")
        B, S, device = b, s, t.device
    return sorted(x), B, S, device


class PackPlan:
    """Weight re-packing as data: every job reads a (possibly flipped / transposed / sliced) *view* of an fp32 master
    parameter through explicit strides and writes a persistent fp16 buffer, and all jobs of a model run in ONE launch
    (``w2s_pack_batch``).  After an optimizer step only ``run()`` is needed: no torch copies, no re-allocation, the
    descriptors keep pointing at the same buffers."""

    def __init__(self, lib, device):
        self.lib, self.device = lib, device
        self.jobs: list[_lib.PackJob] = []
        self.keep: list[Tensor] = []          # destinations (+ fp32 copies of non-fp32 sources)
        self.refresh: list[tuple[Tensor, Tensor]] = []  # (source parameter, fp32 copy) pairs to re-copy before a run
        self.max_elems = 0
        self._dev_jobs = None

    def _source(self, view: Tensor) -> Tensor:
        v = view.detach()
        if v.dtype == torch.float32 and v.device == self.device:
            return v  # alias of the live parameter: in-place updates are seen by the next run
        c = v.to(device=self.device, dtype=torch.float32)
        self.keep.append(c)
        self.refresh.append((v, c))
        return c

    def f32(self, t: Tensor) -> Tensor:
        """A small tensor the kernels read as fp32 (bias, LayerNorm weight ...): the live parameter itself when it is
        contiguous fp32 on the device, else a copy that is refreshed before every run."""
        v = t.detach()
        if v.dtype == torch.float32 and v.device == self.device and v.is_contiguous():
            return v
        c = v.to(device=self.device, dtype=torch.float32).contiguous()
        self.keep.append(c)
        self.refresh.append((v, c))
        return c

    def conv(self, view: Tensor, split: int = 0, flip: bool = False) -> int:
        """view: [cout, cin, taps] (any strides).  flip: reverse the taps (data-gradient weights).  -> device pointer."""
        v = self._source(view)
        cout, cin, taps = v.shape
        sn, sc, st = v.stride()
        ptr = v.data_ptr()
        if flip:
            ptr += (taps - 1) * st * 4
            st = -st
        n = cout * cin * taps
        out = torch.empty(n * (2 if split else 1), dtype=torch.float16, device=self.device)
        self.keep.append(out)
        self.jobs.append(_lib.PackJob(ptr, out.data_ptr(), 0, cout, cin, taps, sn, sc, st, int(split), 0))
        self.max_elems = max(self.max_elems, n)
        self._dev_jobs = None
        return out.data_ptr()

    def frag(self, view: Tensor) -> int:
        """view: nn.Linear weight [n, k] -> mma.sync fragment order."""
        v = self._source(view)
        n, k = v.shape
        sn, sc = v.stride()
        out = torch.empty(n * k, dtype=torch.float16, device=self.device)
        self.keep.append(out)
        self.jobs.append(_lib.PackJob(v.data_ptr(), out.data_ptr(), 1, n, k, 1, sn, sc, 0, 0, 0))
        self.max_elems = max(self.max_elems, n * k)
        self._dev_jobs = None
        return out.data_ptr()

    def run(self) -> None:
        if not self.jobs:
            return
        for src, dst in self.refresh:
            dst.copy_(src)
        if self._dev_jobs is None:
            arr = (_lib.PackJob * len(self.jobs))(*self.jobs)
            host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
            self._dev_jobs = host.to(self.device)
        _lib.check(self.lib.w2s_pack_batch(self._dev_jobs.data_ptr(), len(self.jobs), self.max_elems, _stream()))


class _PackedEncoder:
    """The C descriptor of one SignalEncoder, pointing at the plan's packed fp16 weights and at the live fp32 tensors."""

    def __init__(self, lib, enc, device, plan: PackPlan):
        d = EncoderDesc()
        d.n_blocks = len(enc.channels)
        for i, c in enumerate(enc.channels):
            d.channels[i] = c
        d.feature_dim = enc.feature_dim
        d.norm_eps = enc.norm_eps
        d.wide_blocks = int(getattr(enc, "wide_blocks", 0))
        f32 = plan.f32

        def pack(w, block):
            cout, cin, _ = w.shape
            return plan.conv(w, split=lib.w2s_encoder_conv_split(d.wide_blocks, block, cin, cout))

        blk0 = enc.cnn[0]
        d.w_first = f32(blk0.conv1.conv.weight[:, 0, :]).data_ptr()
        d.w_first_ds = f32(blk0.downsample.weight[:, 0, 0]).data_ptr()
        for i, blk in enumerate(enc.cnn):
            if i > 0:
                d.w_conv[i][0] = pack(blk.conv1.conv.weight, i)
                d.w_ds[i] = pack(blk.downsample.weight, i)
            d.w_conv[i][1] = pack(blk.conv2.conv.weight, i)
            d.w_conv[i][2] = pack(blk.conv3.conv.weight, i)
        F, K = enc.linear.weight.shape  # Linear(4C -> F) as a 4-tap conv: input index = tap * C + c
        d.w_lin = plan.conv(enc.linear.weight.view(F, 4, K // 4).permute(0, 2, 1))
        d.b_lin = f32(enc.linear.bias).data_ptr()
        self.desc = d
        self.samples_per_epoch = enc.samples_per_epoch


class Pending:
    """Result of an asynchronous forward: ``wait()`` makes the *current stream* wait for it (no host synchronisation) and
    returns the tensor."""

    def __init__(self, tensor: Tensor, done: "torch.cuda.Event"):
        self.tensor, self.done = tensor, done

    def wait(self) -> Tensor:
        cur = torch.cuda.current_stream(self.tensor.device)
        cur.wait_event(self.done)
        self.tensor.record_stream(cur)
        return self.tensor


class ForwardEngine:
    """Inference forward of ``Wav2Sleep`` on one CUDA device."""

    def __init__(self, model):
        self.model = model
        self.lib = _lib.load()
        self._weights_key = None
        self._ws: dict = {}
        self.use_graph = True          # CUDA-graph replay of small-batch forwards (see forward)
        self.replayed_launches = 0     # kernels launched through graph replays (not seen by w2s_launch_count)
        # One CUDA stream per signal encoder: the encoders are independent chains of ~25 persistent kernels, each of
        # which ends with a tail (CTAs finish 3-20 % apart) and starts with a ~5 us pipeline fill.  On separate
        # streams the next chain's CTAs take over the SMs the moment a kernel's early finishers release them, so
        # fill and tail of one encoder are covered by the other encoders' work.  False serialises them.
        self.enc_streams = True
        # encoders of identical architecture on inputs of equal length (ECG + PPG, ABD + THX) share their conv launches
        # (w2s_encoder_fwd_pair).  0: one launch chain per signal; 1 (default): only while at least two launch chains
        # remain to overlap each other's kernel tails - the two-signal EOG model keeps one chain per signal (paired: 44.4
        # vs 42.3 ms per 16 x 14-h nights); 2: always
        self.enc_pairs = 1
        # measurement mode: the encoder streams run one after the other (isolated per-kernel durations of exactly the
        # launches of a normal step, paired launches included)
        self.serial_groups = False
        # Asynchronous forwards (forward_async / predict_async) run on the engine's own streams and workspaces (the
        # current stream only records the fork event); a batch starts once the previous one has finished with them.
        # One set: two alternating sets, which would let consecutive batches overlap, buy nothing on B200 (6.91 vs 6.89
        # ms per step) - every kernel of the forward claims 150-230 KB of shared memory, so the mixer tail of one batch
        # and the encoder kernels of the next cannot be co-resident on an SM - and double the workspaces.

    # ------------------------------------------------------------------ weights
    def _params_key(self, device):
        """(structure, values): the structure (device, storage policy, parameter addresses) decides whether the pack plan
        and the descriptors are still valid; the values (tensor versions + the fused optimizer's epoch, whose in-place
        updates do not bump versions) decide whether the plan has to run again."""
        from . import optim
        params = list(self.model.parameters())
        wide = tuple(int(getattr(e, "wide_blocks", 0)) for e in self.model.signal_encoders.encoders.values())
        return ((str(device), wide) + tuple(p.data_ptr() for p in params),
                (optim.WEIGHTS_EPOCH,) + tuple(p._version for p in params))

    def _ensure_packed(self, device):
        skey, vkey = self._params_key(device)
        if self._weights_key is not None and self._weights_key[0] == skey:
            if self._weights_key[1] != vkey:
                self.plan.run()  # same tensors, new values: one launch
                self._weights_key = (skey, vkey)
            return
        m, lib = self.model, self.lib
        plan = self.plan = PackPlan(lib, device)
        f32 = plan.f32
        self.enc = {name: _PackedEncoder(lib, enc, device, plan) for name, enc in m.signal_encoders.encoders.items()}

        mix = m.epoch_mixer
        md = MixerDesc()
        md.n_layers = mix.num_layers
        md.feature_dim, md.n_heads, md.dim_ff = mix.feature_dim, mix.nhead, mix.dim_ff
        md.ln_eps = mix.transformer_encoder.layers[0].norm1.eps
        md.cls = f32(mix.register_tokens[0, 0, :, 0]).data_ptr()
        for l, layer in enumerate(mix.transformer_encoder.layers):
            L = md.layer[l]
            L.in_w = plan.frag(layer.self_attn.in_proj_weight)
            L.out_w = plan.frag(layer.self_attn.out_proj.weight)
            L.ff1_w = plan.frag(layer.linear1.weight)
            L.ff2_w = plan.frag(layer.linear2.weight)
            L.in_b = f32(layer.self_attn.in_proj_bias).data_ptr()
            L.out_b = f32(layer.self_attn.out_proj.bias).data_ptr()
            L.ff1_b = f32(layer.linear1.bias).data_ptr()
            L.ff2_b = f32(layer.linear2.bias).data_ptr()
            L.ln1_w, L.ln1_b = f32(layer.norm1.weight).data_ptr(), f32(layer.norm1.bias).data_ptr()
            L.ln2_w, L.ln2_b = f32(layer.norm2.weight).data_ptr(), f32(layer.norm2.bias).data_ptr()
        self.mixer_desc = md

        seq = m.sequence_mixer
        sd = SeqDesc()
        sd.n_blocks = len(seq.dilated_convs)
        sd.n_dilations = len(seq.dilated_convs[0].conv_layers)
        sd.kernel_size = seq.dilated_convs[0].kernel_size
        sd.feature_dim = seq.feature_dim
        sd.n_classes = m.num_classes
        sd.ln_eps = seq.dilated_convs[0].conv_layers[0].norm.eps
        for b, blk in enumerate(seq.dilated_convs):
            for k, layer in enumerate(blk.conv_layers):
                sd.w[b][k] = plan.conv(layer.conv.weight)
                sd.ln_w[b][k] = f32(layer.norm.weight.reshape(-1)).data_ptr()
                sd.ln_b[b][k] = f32(layer.norm.bias.reshape(-1)).data_ptr()
        sd.head_w = f32(m.classifier.weight).data_ptr()
        sd.head_b = f32(m.classifier.bias).data_ptr()
        self.seq_desc = sd
        plan.run()
        self._weights_key = (skey, vkey)
        self._release_buffers()  # workspace sizes depend on the encoders' storage policy

    # ------------------------------------------------------------------ buffers
    def _release_buffers(self) -> None:
        """Drop every workspace.  Batches still in flight on the engine's own streams must finish before their memory
        goes back to the allocator of the current stream."""
        for old in self._ws.values():
            if old.get("tail_done") is not None:
                torch.cuda.current_stream(old["mix"].device).wait_event(old["tail_done"])
        self._ws.clear()

    def _buffers(self, device, names, B, S, detached: bool = False):
        """Workspaces of one shape; detached: the set of the asynchronous forwards, with their own tail stream."""
        key = (str(device), tuple(names), B, S, self.enc_streams, detached)
        buf = self._ws.get(key)
        if buf is not None:
            return buf
        if any(k[:5] != key[:5] for k in self._ws):
            self._release_buffers()  # one live shape at a time keeps the footprint bounded
        lib = self.lib
        sizes = {}
        for n in names:
            pe = self.enc[self.model.signal_encoders.signal_map[n]]
            sizes[n] = lib.w2s_encoder_workspace_bytes(C.byref(pe.desc), B, S * pe.samples_per_epoch, 0)
        seq_ws = lib.w2s_seqmixer_workspace_bytes(C.byref(self.seq_desc), B, S, 0)
        concurrent = (self.enc_streams and len(names) > 1) or detached
        if concurrent:  # encoders run side by side: one workspace each
            enc_ws = {n: torch.empty(sizes[n], dtype=torch.uint8, device=device) for n in names}
        else:           # encoders run back to back: one workspace of the largest size
            shared = torch.empty(max(sizes.values()), dtype=torch.uint8, device=device)
            enc_ws = {n: shared for n in names}
        buf = {
            "enc_ws": enc_ws,
            "streams": [torch.cuda.Stream(device=device) for _ in names] if concurrent else None,
            "tail": torch.cuda.Stream(device=device) if detached else None,   # mixer + sequence mixer + head
            "tail_done": None,
            "seq_ws": torch.empty(seq_ws, dtype=torch.uint8, device=device),
            "z": {n: torch.empty(B, S, 128, dtype=torch.float16, device=device) for n in names},
            "mask": {n: torch.zeros(B, dtype=torch.uint8, device=device) for n in names},
            "mix": torch.empty(B, S, 128, dtype=torch.float16, device=device),
        }
        self._ws[key] = buf
        return buf

    # ------------------------------------------------------------------ forward
    def _seq_head(self, buf, B: int, S: int, logits: Tensor, stream: "torch.cuda.Stream") -> None:
        """Sequence mixer + classifier on `stream`."""
        ws = buf["seq_ws"]
        _lib.check(self.lib.w2s_seqmixer_head_fwd(C.byref(self.seq_desc), buf["mix"].data_ptr(), B, S, ws.data_ptr(),
                                                  ws.numel(), 0, None, logits.data_ptr(), stream.cuda_stream))

    def _enc_groups(self, names, xs, paired: bool):
        """Signals in launch order (longest chains first - they set the critical path when the encoders overlap), grouped
        in pairs where two encoders have the same architecture and input length."""
        order = sorted(names, key=lambda k: -xs[k].size(1))
        if not (paired and self.enc_pairs):
            return [(n,) for n in order]
        smap = self.model.signal_encoders.signal_map

        def arch(n):
            d = self.enc[smap[n]].desc
            return (d.n_blocks, tuple(d.channels[:d.n_blocks]), d.feature_dim, d.wide_blocks, d.norm_eps, xs[n].size(1))

        groups, used = [], set()
        for i, n in enumerate(order):
            if n in used:
                continue
            used.add(n)
            mate = next((m for m in order[i + 1:] if m not in used and arch(m) == arch(n)), None)
            if mate is None:
                groups.append((n,))
            else:
                used.add(mate)
                groups.append((n, mate))
        if len(groups) < 2 and self.enc_pairs < 2:
            return [(n,) for n in order]
        return groups

    def _encode(self, buf, xs, grp, B: int, stream_ptr) -> None:
        """One signal encoder, or two of the same architecture in shared launches, on the given stream."""
        lib, smap = self.lib, self.model.signal_encoders.signal_map
        n = grp[0]
        pe, ws = self.enc[smap[n]], buf["enc_ws"][n]
        if len(grp) == 1:
            _lib.check(lib.w2s_encoder_fwd(C.byref(pe.desc), xs[n].data_ptr(), B, xs[n].size(1), ws.data_ptr(), ws.numel(), 0,
                                           buf["z"][n].data_ptr(), buf["mask"][n].data_ptr(), stream_ptr), ValueError)
            return
        m = grp[1]
        pm, wm = self.enc[smap[m]], buf["enc_ws"][m]
        assert ws.numel() == wm.numel() and ws.data_ptr() != wm.data_ptr()
        _lib.check(lib.w2s_encoder_fwd_pair(C.byref(pe.desc), xs[n].data_ptr(), ws.data_ptr(), buf["z"][n].data_ptr(),
                                            buf["mask"][n].data_ptr(), C.byref(pm.desc), xs[m].data_ptr(), wm.data_ptr(),
                                            buf["z"][m].data_ptr(), buf["mask"][m].data_ptr(), B, xs[n].size(1), ws.numel(),
                                            0, stream_ptr), ValueError)

    def _launch(self, buf, xs: dict[str, Tensor], names, B: int, S: int, logits: Tensor) -> None:
        """Enqueue the three stage calls on the current stream (also what gets captured into a CUDA graph)."""
        lib, st = self.lib, _stream()
        streams = buf["streams"]
        if streams is not None:
            cur = torch.cuda.current_stream()
            fork = torch.cuda.Event()
            fork.record(cur)
        # (pairs need one workspace per encoder: only when the encoders have their own streams / workspaces)
        prev = None
        for i, grp in enumerate(self._enc_groups(names, xs, paired=streams is not None)):
            if streams is not None:
                streams[i].wait_event(fork)
                if self.serial_groups and prev is not None:
                    streams[i].wait_event(prev)
                est = streams[i].cuda_stream
            else:
                est = st
            self._encode(buf, xs, grp, B, est)
            if streams is not None:
                join = torch.cuda.Event()
                join.record(streams[i])
                cur.wait_event(join)
                prev = join
        zs = (C.c_void_p * len(names))(*[buf["z"][n].data_ptr() for n in names])
        ms = (C.c_void_p * len(names))(*[buf["mask"][n].data_ptr() for n in names])
        _lib.check(lib.w2s_epoch_mixer_fwd(C.byref(self.mixer_desc), zs, ms, len(names), B, S, buf["mix"].data_ptr(), st))
        self._seq_head(buf, B, S, logits, torch.cuda.current_stream())

    def _launch_async(self, buf, xs: dict[str, Tensor], names, B: int, S: int, argmax: bool, ready=None) -> Pending:
        """The whole forward on the engine's own streams: nothing is enqueued on the current stream except the fork event.
        ready: optional {signal: event} - the signal's encoder additionally waits for its event (e.g. the end of that
        signal's host -> device copy on another stream), so the first encoders start while the other signals still
        arrive."""
        lib = self.lib
        cur = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(cur)
        tail, streams = buf["tail"], buf["streams"]
        tail.wait_event(fork)
        for i, grp in enumerate(self._enc_groups(names, xs, paired=True)):
            st = streams[i]
            st.wait_event(fork)
            for n in grp:
                if ready is not None and ready.get(n) is not None:
                    st.wait_event(ready[n])
                xs[n].record_stream(st)
            if buf["tail_done"] is not None:
                st.wait_event(buf["tail_done"])  # the previous batch has finished reading z / masks
            self._encode(buf, xs, grp, B, st.cuda_stream)
            ev = torch.cuda.Event()
            ev.record(st)
            tail.wait_event(ev)
        with torch.cuda.stream(tail):
            logits = torch.empty(B, S, self.model.num_classes, dtype=torch.float32, device=buf["mix"].device)
            zs = (C.c_void_p * len(names))(*[buf["z"][n].data_ptr() for n in names])
            ms = (C.c_void_p * len(names))(*[buf["mask"][n].data_ptr() for n in names])
            _lib.check(lib.w2s_epoch_mixer_fwd(C.byref(self.mixer_desc), zs, ms, len(names), B, S, buf["mix"].data_ptr(),
                                               tail.cuda_stream))
            self._seq_head(buf, B, S, logits, tail)
            out = _argmax(lib, logits) if argmax else logits  # on the tail stream: it is the current one here
            done = torch.cuda.Event()
            done.record(tail)
        buf["tail_done"] = done
        return Pending(out, done)

    @torch.no_grad()
    def forward_async(self, x: dict[str, Tensor], argmax: bool = False, ready=None) -> Pending:
        """Enqueue a forward on the engine's own streams and return at once; ``.wait()`` on the result orders the current
        stream after it.  Inputs must stay untouched until then."""
        names, B, S, device = check_inputs(self.model.signal_encoders, x)
        with torch.cuda.device(device):
            self._ensure_packed(device)
            buf = self._buffers(device, names, B, S, detached=True)
            xs = {n: _f32(x[n]) for n in names}
            return self._launch_async(buf, xs, names, B, S, argmax, ready)

    def predict_async(self, x: dict[str, Tensor], ready=None) -> Pending:
        return self.forward_async(x, argmax=True, ready=ready)

    # Small batches are launch-latency bound (~100 launches for ~2 ms of GPU work at B = 1): from the second call with
    # the same shape on, the whole forward is replayed from one CUDA graph over static input / output buffers.
    GRAPH_MAX_INPUT_BYTES = 32 << 20

    @torch.no_grad()
    def forward(self, x: dict[str, Tensor]) -> Tensor:
        names, B, S, device = check_inputs(self.model.signal_encoders, x)  # sorted: the token order, wav2sleep.py:311
        with torch.cuda.device(device):
            self._ensure_packed(device)
            buf = self._buffers(device, names, B, S)
            xs = {n: _f32(x[n]) for n in names}
            in_bytes = sum(t.numel() * 4 for t in xs.values())
            if (self.use_graph and in_bytes <= self.GRAPH_MAX_INPUT_BYTES and buf.get("calls", 0) >= 1
                    and not torch.cuda.is_current_stream_capturing()):
                if buf.get("graph") is None or buf.get("graph_wkey") != self._weights_key[0]:
                    # static graph buffers must be ordinary tensors: created under inference_mode they could not be
                    # written by a later call that runs under plain no_grad
                    with torch.inference_mode(False):
                        buf["xin"] = {n: torch.empty(xs[n].shape, dtype=torch.float32, device=device) for n in names}
                        buf["logits"] = torch.empty(B, S, self.model.num_classes, dtype=torch.float32, device=device)
                    l0 = self.lib.w2s_launch_count()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._launch(buf, buf["xin"], names, B, S, buf["logits"])
                    buf.update(graph=g, graph_wkey=self._weights_key[0], graph_launches=self.lib.w2s_launch_count() - l0)
                for n in names:
                    buf["xin"][n].copy_(xs[n], non_blocking=True)
                buf["graph"].replay()
                self.replayed_launches += buf["graph_launches"]
                return buf["logits"].clone()
            buf["calls"] = buf.get("calls", 0) + 1
            logits = torch.empty(B, S, self.model.num_classes, dtype=torch.float32, device=device)
            self._launch(buf, xs, names, B, S, logits)
        return logits

    @torch.no_grad()
    def predict(self, x: dict[str, Tensor]) -> Tensor:
        return _argmax(self.lib, self.forward(x))
