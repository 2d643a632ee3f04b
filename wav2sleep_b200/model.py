"""Drop-in mirror of ``wav2sleep.models.wav2sleep`` whose forward runs on hand-written sm_100a kernels.

Same class names, constructor keywords, attribute names and ``state_dict`` keys as the reference
(/root/reference/src/wav2sleep/models/wav2sleep.py:16-390, blocks.py, utils.py), so that
``hydra.utils.instantiate`` configs, ``load_state_dict(torch.load('state_dict.pth'))`` and the Lightning module
of the reference keep working when ``_target_`` is pointed at this module.

The ``torch.nn`` leaf modules below (``nn.Conv1d``, ``nn.Linear``, ``nn.TransformerEncoderLayer`` ...) are
*parameter containers only*: they give identical parameter names, shapes and default initialisation (same RNG
consumption order as the reference, so ``torch.manual_seed(s)`` reproduces the reference's random init
bit-for-bit), but their ``forward`` is never called.  All compute goes through ``engine.ForwardEngine`` ->
``libw2s_b200.so``.  There is no CPU or eager fallback: a CPU tensor or a missing library raises.

Two CUDA paths sit behind the same classes.  The default model family of the reference's configs (non-causal,
instance-norm encoders with 16..128 channels, GELU, feature_dim 128, nhead 8, dim_ff 512, layer-norm sequence mixer with
kernel 7) runs on the fused tcgen05 kernels (engine.py / training.py).  Every other option the reference constructors
accept (SURVEY.md section 8f, row N3: causal / chunk-causal mode, norms batch / layer / rms / group / auto / none,
activations relu / leaky / silu / linear, ``embed_signals``, ``register_tokens > 0``, ``output_norm``,
``use_residual=False``, other widths and feature dims) runs on the dimension-generic fp32 kernels of csrc/general.cuh
(general.py): inference and training (an autograd graph over fp32 forward / backward kernels, dropout included), same
results as the reference to fp32 accuracy, not tuned.  ``norm='weight'`` (a parametrisation with different state_dict
keys) is the one option that raises ``NotImplementedError``; a Wav2Sleep model with BatchNorm layers (norm='batch')
runs inference but raises ``NotImplementedError`` under ``train()`` with grad (train-mode BatchNorm is built, see
general.py, but the reference's batch statistics include the zero-filled rows of missing signals, which the general
path skips); in ``eval()`` it is differentiable, in its inputs and its parameters.  SleepPPGNet (ppgnet.py) trains.
"""
from __future__ import annotations

import math

import torch
from torch import Tensor, nn

# settings.py:16-26 of the reference: samples per 30-s epoch after resampling.
COLS_TO_SAMPLES_PER_EPOCH = {"ABD": 256, "THX": 256, "ECG": 1024, "PPG": 1024, "EOG-L": 4096, "EOG-R": 4096}


def _require(cond: bool, what: str) -> None:
    if not cond:
        raise NotImplementedError(f"wav2sleep_b200: {what} is not built on the CUDA path")


class ConvLayerNorm(nn.Module):
    """Parameters of the channel-first LayerNorm (reference models/utils.py:9-23); applied inside the conv epilogue."""

    def __init__(self, num_features: int, eps: float = 1e-5):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(1, num_features, 1))
        self.bias = nn.Parameter(torch.zeros(1, num_features, 1))
        self.eps = eps


class ConvRMSNorm(nn.Module):
    """Parameters of the channel-first RMS norm (reference models/utils.py:26-36)."""

    def __init__(self, num_features: int, eps: float = 1e-5):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(1, num_features, 1))
        self.eps = eps


class ConvGroupNorm(nn.Module):
    """Parameters of the group norm wrapper (reference models/utils.py:38-58): keys ``norm.weight`` / ``norm.bias``."""

    def __init__(self, num_features: int, num_groups: int = 8, channels_per_group: int | None = None, eps: float = 1e-5):
        super().__init__()
        if channels_per_group is not None:
            num_groups = num_features // channels_per_group
        if num_features < num_groups:
            num_groups = num_features
        if num_features % num_groups != 0:
            raise ValueError(f"{num_features=} must be divisible by {num_groups=}.")
        self.norm = nn.GroupNorm(num_groups=num_groups, num_channels=num_features, eps=eps)


ACTIVATIONS = ("relu", "leaky", "gelu", "silu", "swish", "linear")


def get_activation(name: str) -> nn.Module:
    """reference models/utils.py:61-74 (parameter-free modules; kept for attribute / repr compatibility)."""
    if name not in ACTIVATIONS:
        raise ValueError(f"{name=} is unsupported.")
    return {"relu": nn.ReLU, "leaky": nn.LeakyReLU, "gelu": nn.GELU, "silu": nn.SiLU, "swish": nn.SiLU,
            "linear": nn.Identity}[name]()


def get_norm(name: str | None, num_features: int, norm_eps: float | None = None) -> nn.Module:
    """reference models/utils.py:77-96: the parameter / buffer containers of each normalisation."""
    if name == "batch":
        return nn.BatchNorm1d(num_features)
    if name == "layer":
        return ConvLayerNorm(num_features)
    if name == "rms":
        return ConvRMSNorm(num_features)
    if name is None:
        return nn.Identity()
    if name == "instance":
        return nn.InstanceNorm1d(num_features, **({"eps": norm_eps} if norm_eps is not None else {}))
    if name == "group":
        return ConvGroupNorm(num_features)
    if name == "weight":
        _require(False, "norm='weight' (weight-norm parametrisation)")
    raise ValueError(f"Normalisation with {name=} unknown.")


class ConvLayer1D(nn.Module):
    """conv -> norm -> activation; holds ``conv.weight`` (+ ``norm.*``).  reference models/blocks.py:129-186."""

    def __init__(self, input_dim: int, output_dim: int, kernel_size: int = 3, stride: int = 1, padding: int = 1,
                 dilation: int = 1, dropout: float = 0.0, causal: bool = False, groups: int = 1, activation: str = "relu",
                 bias: bool = False, norm: str | None = "batch", norm_eps: float | None = None):
        super().__init__()
        _require(groups == 1, f"groups={groups}")
        self.causal = causal
        self.padding = (kernel_size - 1) * dilation if causal else padding  # blocks.py:150-153
        self.kernel_size, self.stride, self.dilation = kernel_size, stride, dilation
        self.norm_name, self.activation_name = norm, activation
        self.conv = nn.Conv1d(input_dim, output_dim, kernel_size=kernel_size, stride=stride, padding=self.padding,
                              dilation=dilation, bias=bias or norm is None)
        self.norm = get_norm(norm, output_dim, norm_eps)
        self.activation = get_activation(activation)
        self.dropout = nn.Dropout(p=dropout)

    def output_length(self, L: int) -> int:
        """Length after the conv and, in causal mode, the right-trim of blocks.py:178-182."""
        full = (L + 2 * self.padding - self.dilation * (self.kernel_size - 1) - 1) // self.stride + 1
        if self.causal and self.padding > 0:
            full -= max(self.padding - (self.stride - 1), 0)
        return full


class ConvBlock1D(nn.Module):
    """Three conv layers + 1x1 stride-2 residual; out = act(conv3(conv2(conv1(x))) + downsample(x)).  blocks.py:8-71."""

    def __init__(self, input_dim: int, output_dim: int, dropout: float = 0.0, activation: str = "leaky",
                 norm: str | None = "batch", causal: bool = False, norm_eps: float | None = None,
                 use_residual: bool = True):
        super().__init__()
        self.use_residual = use_residual
        kw = dict(kernel_size=3, padding=1, activation=activation, norm=norm, dropout=dropout, causal=causal,
                  norm_eps=norm_eps)
        self.conv1 = ConvLayer1D(input_dim, output_dim, **kw)
        self.conv2 = ConvLayer1D(output_dim, output_dim, **kw)
        self.conv3 = ConvLayer1D(output_dim, output_dim, stride=2, **kw)
        self.activation = get_activation(activation)
        self.activation_name = activation
        if use_residual:
            self.downsample = nn.Conv1d(input_dim, output_dim, kernel_size=1, stride=2, padding=0, bias=False)
        else:
            self.register_parameter("downsample", None)


class SignalEncoder(nn.Module):
    """Per-signal CNN: log2(samples_per_epoch)-2 ConvBlock1D + Linear(4C -> F).  models/wav2sleep.py:164-267."""

    def __init__(self, input_dim: int = 1, feature_dim: int = 256, activation: str = "gelu",
                 samples_per_epoch: int = 1024, norm: str = "instance", initial_channels: int = 16,
                 max_channels: int = 128, causal: bool = False, chunk_causal: bool = True, output_norm: bool = False,
                 use_residual: bool = True) -> None:
        super().__init__()
        if samples_per_epoch & (samples_per_epoch - 1) != 0:
            raise ValueError(f"samples_per_epoch must be a power of 2, got {samples_per_epoch}")
        _require(input_dim == 1, f"input_dim={input_dim}")
        self.feature_dim = feature_dim
        self.samples_per_epoch = samples_per_epoch
        self.causal = causal
        self.chunk_causal = chunk_causal
        self.norm_name, self.activation_name, self.use_residual = norm, activation, use_residual
        num_blocks = int(math.log2(samples_per_epoch)) - 2
        _require(1 <= num_blocks <= 12, f"samples_per_epoch={samples_per_epoch}")
        self.channels = [min(initial_channels * 2 ** (i // 2), max_channels) for i in range(num_blocks)]
        self.norm_eps = 1e-2  # models/wav2sleep.py:213-215 (instance norm only)
        causal_conv = causal and not chunk_causal  # wav2sleep.py:201
        self.block_norms = []
        blocks, cin = [], input_dim
        for i, cout in enumerate(self.channels):
            norm_i = ("instance" if i < 2 else "layer") if norm == "auto" else norm  # wav2sleep.py:204-212
            self.block_norms.append(norm_i)
            blocks.append(ConvBlock1D(cin, cout, activation=activation, norm=norm_i,
                                      norm_eps=self.norm_eps if norm_i == "instance" else None, causal=causal_conv,
                                      use_residual=use_residual))
            cin = cout
        self.cnn = nn.Sequential(*blocks)
        self.epoch_dim = self.channels[-1] * 4
        self.linear = nn.Linear(self.epoch_dim, feature_dim)
        self.activation = get_activation(activation)
        self.output_norm = nn.LayerNorm(feature_dim) if output_norm else nn.Identity()
        # True when this encoder is in the model family the fused tcgen05 kernels are built for
        self.fast_path = (activation == "gelu" and norm == "instance" and not causal and not output_norm and use_residual
                          and initial_channels == 16 and max_channels == 128 and feature_dim == 128)
        # Inference storage policy of the fast path (not a reference argument): number of leading blocks whose conv
        # outputs are kept as fp32 instead of fp16 and whose convs carry split (hi + lo) operands (0, 2, 4 or 6).
        # Stacks of >= 10 blocks (EOG: 30 convs, 6.9 M samples) default to 6 = every block up to 64 channels: with
        # all-fp16 storage the logits sit on the 2e-2 gate, and the argmax gate needs the 64-channel blocks as well
        # (DESIGN.md "Numerics", tools/emulate_16bit.py).
        self.wide_blocks = 6 if num_blocks >= 10 else 0


class SignalEncoders(nn.Module):
    """Container of the per-signal encoders.  models/wav2sleep.py:83-161."""

    def __init__(self, signal_map: dict[str, str], feature_dim: int, activation: str, norm: str = "instance",
                 causal: bool = False, chunk_causal: bool = True, embed_signals: bool = False,
                 initial_channels: int = 16, max_channels: int = 128, output_norm: bool = False,
                 use_residual: bool = True) -> None:
        super().__init__()
        self.feature_dim = feature_dim
        self.signal_map = dict(signal_map)
        self.causal = causal
        encoders = {}
        for signal_name, encoder_name in self.signal_map.items():
            if encoder_name in encoders:
                continue
            if signal_name not in COLS_TO_SAMPLES_PER_EPOCH:
                raise ValueError(f"Column {signal_name} unrecognised. Doesn't have a sampling rate.")
            encoders[encoder_name] = SignalEncoder(
                input_dim=1, feature_dim=feature_dim, samples_per_epoch=COLS_TO_SAMPLES_PER_EPOCH[signal_name],
                activation=activation, norm=norm, causal=causal, chunk_causal=chunk_causal,
                initial_channels=initial_channels, max_channels=max_channels, output_norm=output_norm,
                use_residual=use_residual)
        self.encoders = nn.ModuleDict(encoders)
        self.embed_signals = embed_signals
        self.sig_to_embedding_idx = {sig: i for i, sig in enumerate(sorted(self.signal_map.keys()))}
        if embed_signals:
            self.embedder = nn.Embedding(num_embeddings=len(self.signal_map), embedding_dim=feature_dim)
        else:
            self.register_parameter("embedder", None)
        self.fast_path = not embed_signals and all(e.fast_path for e in self.encoders.values())

    def __len__(self) -> int:
        return len(self.encoders)

    def get_encoder(self, signal_name: str) -> SignalEncoder:
        return self.encoders[self.signal_map[signal_name]]  # type: ignore[return-value]

    def compile(self, *args, **kwargs) -> None:
        """``nn.Module.compile`` of the reference (tests/model/test_compile.py:27, api.py:96-97) has nothing to trace here:
        the forward is pre-compiled CUDA behind a C ABI.  Accepted and ignored, so that callers need no change."""

    def forward(self, x: dict[str, Tensor]) -> dict[str, Tensor]:
        """Stand-alone call of the encoders (reference models/wav2sleep.py:146-161): {signal: [B, T]} ->
        {signal: fp32 [B, S, feature_dim]}, rows of samples whose signal is missing (-inf input) filled with -inf,
        plus the optional signal-source embedding.  ``Wav2Sleep.forward`` does not come through here (its fused path
        keeps the features in fp16 and hands masks over separately); this entry runs the dimension-generic fp32 CUDA
        kernels for every configuration."""
        from .engine import check_inputs
        from .general import GeneralEngine  # deferred: loads the CUDA library
        check_inputs(self, x, joint=False)  # each signal is encoded on its own
        if getattr(self, "_general", None) is None:
            object.__setattr__(self, "_general", GeneralEngine(None))
        eng, out = self._general, {}
        for name, x_BT in x.items():
            with torch.no_grad(), torch.cuda.device(x_BT.device):
                z, mask = eng.encode(self.get_encoder(name), x_BT)
                if self.embed_signals:  # wav2sleep.py:155-159 (the reference adds it to the -inf rows as well)
                    e = self.embedder.weight[self.sig_to_embedding_idx[name]].detach().float().contiguous()
                    z = eng.affine_act(z, "linear", shift=e, mask=mask, per_channel=1)
                z = z.masked_fill(mask.bool()[:, None, None], float("-inf"))  # data movement, no arithmetic
            out[name] = z
        return out


class MultiModalAttentionEmbedder(nn.Module):
    """CLS-token set transformer over the modality tokens of one epoch.  models/wav2sleep.py:270-346."""

    def __init__(self, feature_dim: int, layers: int = 4, dropout: float = 0.0, dim_ff: int = 512,
                 activation: str = "gelu", norm_first: bool = True, nhead: int = 4, register_tokens: int = 0):
        super().__init__()
        if feature_dim % nhead:
            raise ValueError(f"feature_dim={feature_dim} must be divisible by nhead={nhead}")
        self.feature_dim = feature_dim
        self.dropout = dropout
        self.nhead = nhead
        self.dim_ff = dim_ff
        self.norm_first = norm_first
        self.activation_name = activation
        encoder_layer = nn.TransformerEncoderLayer(d_model=feature_dim, dim_feedforward=dim_ff,
                                                   activation=get_activation(activation), nhead=nhead, batch_first=True,
                                                   dropout=dropout, norm_first=norm_first)
        self.num_layers = layers
        self.transformer_encoder = nn.TransformerEncoder(encoder_layer, num_layers=layers, enable_nested_tensor=False)
        self.num_register_tokens = register_tokens
        self.register_tokens = nn.Parameter(torch.randn(1, 1, feature_dim, register_tokens + 1))
        self.fast_path = (feature_dim == 128 and nhead == 8 and dim_ff == 512 and activation == "gelu" and norm_first
                          and register_tokens == 0 and 1 <= layers <= 8)

    def compile(self, *args, **kwargs) -> None:
        """Accepted and ignored (see SignalEncoders.compile): the CUDA path needs no tracing compiler."""


class DilatedConvBlock(nn.Module):
    """num_dilations x (dilated conv k -> norm -> act), dropout, + input, act.  models/blocks.py:74-126."""

    def __init__(self, feature_dim: int = 128, dropout: float = 0.2, activation: str = "leaky", norm: str = "batch",
                 kernel_size: int = 7, causal: bool = False, num_dilations: int = 6):
        super().__init__()
        self.kernel_size = kernel_size
        self.dilations = [2 ** i for i in range(num_dilations)]
        layers = []
        for d in self.dilations:
            k_eff = kernel_size + (kernel_size - 1) * (d - 1)
            layers.append(ConvLayer1D(feature_dim, feature_dim, kernel_size=kernel_size, stride=1, dilation=d,
                                      padding=k_eff // 2, activation=activation, norm=norm, causal=causal))
        self.dropout = nn.Dropout(p=dropout)
        self.conv_layers = nn.Sequential(*layers)
        self.activation = get_activation(activation)
        self.activation_name = activation


class SequenceCNN(nn.Module):
    """Dilated-CNN sequence mixer.  models/wav2sleep.py:349-390."""

    def __init__(self, feature_dim: int = 128, dropout: float = 0.2, num_layers: int = 2, activation: str = "gelu",
                 norm: str = "batch", causal: bool = False, num_dilations: int = 6, kernel_size: int = 7) -> None:
        super().__init__()
        self.feature_dim = feature_dim
        self.causal = causal
        self.dilated_convs = nn.Sequential(*[
            DilatedConvBlock(feature_dim=feature_dim, dropout=dropout, activation=activation, norm=norm, causal=causal,
                             kernel_size=kernel_size, num_dilations=num_dilations) for _ in range(num_layers)])
        # num_dilations <= 6: the training forward / backward and long nights run every layer as its own tile-per-CTA
        # conv, which stages (kernel_size - 1) * dilation rows beyond each tile in shared memory; dilation 64 (7 layers)
        # needs 269,328 B, over the 232,448 B a block can have, so deeper stacks go to the general path
        self.fast_path = (feature_dim == 128 and kernel_size == 7 and activation == "gelu" and norm == "layer"
                          and not causal and 1 <= num_layers <= 4 and 1 <= num_dilations <= 6)

    def compile(self, *args, **kwargs) -> None:
        """Accepted and ignored (see SignalEncoders.compile): the CUDA path needs no tracing compiler."""


class Wav2Sleep(nn.Module):
    """Sleep-staging model: encoders -> epoch mixer -> sequence mixer -> classifier.  models/wav2sleep.py:16-80."""

    def __init__(self, signal_encoders: SignalEncoders, epoch_mixer: MultiModalAttentionEmbedder,
                 sequence_mixer: SequenceCNN, num_classes: int):
        super().__init__()
        self.signal_encoders = signal_encoders
        self.epoch_mixer = epoch_mixer
        self.sequence_mixer = sequence_mixer
        self.feature_dim = self.epoch_mixer.feature_dim
        self.num_classes = num_classes
        self.classifier = nn.Linear(in_features=self.feature_dim, out_features=num_classes)
        self._engine = None
        self._general = None
        # the fused tcgen05 path serves the default model family; everything else goes to the general fp32 kernels
        self.fast_path = (signal_encoders.fast_path and epoch_mixer.fast_path and sequence_mixer.fast_path
                          and 1 <= num_classes <= 8 and signal_encoders.feature_dim == epoch_mixer.feature_dim
                          == sequence_mixer.feature_dim)

    @property
    def valid_signals(self) -> list[str]:
        return list(self.signal_encoders.signal_map.keys())

    def compile(self, *args, **kwargs) -> None:
        """``model.compile(mode='max-autotune')`` of the reference (api.py:96-97, tests/model/test_compile.py:35): accepted
        and ignored - the forward is hand-written CUDA behind a C ABI, there is nothing for a tracing compiler to do (and
        tracing it with ``fullgraph=True`` would stop at the first library call)."""

    def _get_engine(self):
        from .training import TrainEngine  # deferred: loads the CUDA library
        if self._engine is None:
            object.__setattr__(self, "_engine", TrainEngine(self))
        return self._engine

    _get_train_engine = _get_engine

    def _get_general(self):
        from .general import GeneralEngine  # deferred: loads the CUDA library
        if self._general is None:
            object.__setattr__(self, "_general", GeneralEngine(self))
        return self._general

    def forward(self, x: dict[str, Tensor]) -> Tensor:
        """dict of [B, S * samples_per_epoch] fp32 (rows of -inf = missing signal) -> logits [B, S, num_classes].

        Under ``train()`` with grad enabled the logits carry a grad_fn whose backward runs the CUDA backward pass
        (dropout with counter-based masks, see training.py; for the non-default options the general path's autograd
        Functions, general.py).  So do they, in ``train()`` or ``eval()``, when an input tensor requires grad: then
        ``x[name].grad`` receives d(objective)/dx (0 at non-finite samples and on missing rows), as with the reference,
        and an ``eval()`` graph has eval semantics (no dropout, BatchNorm on its running statistics).  Otherwise the
        inference kernels run."""
        grad_on = torch.is_grad_enabled()
        input_grad = grad_on and isinstance(x, dict) and any(isinstance(t, Tensor) and t.requires_grad for t in x.values())
        train_grad = self.training and grad_on and any(p.requires_grad for p in self.parameters())
        if not self.fast_path:
            if train_grad or (input_grad and self.training):
                if any(isinstance(mod, nn.BatchNorm1d) for mod in self.modules()):
                    raise NotImplementedError("wav2sleep_b200: training a model with BatchNorm layers (train-mode batch "
                                              "statistics and running-statistics updates) is not built on the CUDA path; "
                                              "eval-mode inference is")
                return self._get_general().forward_train(x)
            if input_grad:
                return self._get_general().forward_graph(x)
            return self._get_general().forward(x)
        if train_grad or input_grad:
            from .training import forward_with_grad
            return forward_with_grad(self, x)
        if self.training and (self.epoch_mixer.dropout > 0 or any(b.dropout.p > 0 for b in
                                                                   self.sequence_mixer.dilated_convs)):
            # train() under no_grad: dropout stays active, as in the reference (nn.Dropout follows .training, not grad mode)
            eng = self._get_engine()
            logits = eng.forward_train(x)
            eng.saved = None
            return logits
        return self._get_engine().forward(x)

    def predict(self, x: dict[str, Tensor]) -> Tensor:
        """Most likely class per epoch, int64 [B, S]  (argmax kernel on the logits)."""
        if not self.fast_path:
            return self._get_general().predict(x)
        return self._get_engine().predict(x)

    def predict_async(self, x: dict[str, Tensor], ready=None):
        """``predict`` without ordering the current stream after it: returns a handle whose ``wait()`` does (and hands
        back the int64 [B, S] tensor).  The host can enqueue the next batches while the GPU works (throughput mode for
        loops over batches); each batch runs on the engine's own streams and starts once the previous one is done.
        ``ready``: optional ``{signal: torch.cuda.Event}``; a signal's encoder starts once its event has completed (e.g.
        that signal's host -> device copy on a copy stream), so a batch need not be fully uploaded before work begins."""
        if not self.fast_path:
            from .engine import Pending
            for ev in (ready or {}).values():
                if ev is not None:
                    torch.cuda.current_stream().wait_event(ev)
            out = self._get_general().predict(x)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(out.device))
            return Pending(out, ev)
        return self._get_engine().predict_async(x, ready=ready)

    def forward_fp32_check(self, x: dict[str, Tensor]) -> Tensor:
        """The same forward through the general path's un-fused fp32 CUDA-core kernels (general.py: fp32 storage, exact
        erf GELU, fp64 statistics), with eval semantics whatever the mode (no dropout, BatchNorm on its running
        statistics) and under ``no_grad``: slow, <= 1e-4 from the reference's fp32 logits.  A validation aid that
        separates the algorithm from the fast path's 16-bit storage, not an inference path."""
        return self._get_general().forward(x)


def build_default(signal_map: dict[str, str], num_classes: int, seed: int | None = None) -> Wav2Sleep:
    """The model of scripts/config/model/wav2sleep.yaml + main.yaml (feature_dim 128, non-causal)."""
    if seed is not None:
        torch.manual_seed(seed)
    enc = SignalEncoders(signal_map=signal_map, feature_dim=128, activation="gelu", norm="instance", causal=False,
                         chunk_causal=False, initial_channels=16, max_channels=128, output_norm=False,
                         use_residual=True)
    mix = MultiModalAttentionEmbedder(feature_dim=128, dropout=0.1, activation="gelu", layers=2, dim_ff=512, nhead=8)
    seq = SequenceCNN(feature_dim=128, dropout=0.1, activation="gelu", norm="layer", causal=False, num_layers=2,
                      kernel_size=7, num_dilations=6)
    return Wav2Sleep(enc, mix, seq, num_classes)
