"""CPU oracle for the NON-DEFAULT model options (the general path, wav2sleep_b200/general.py).  TEST INFRASTRUCTURE ONLY.

A functional fp32 restatement of the reference in plain torch CPU ops, with autograd: the configuration comes from the
constructor keywords of a case (``oracle/make_golden_general.CASES`` format, reference defaults written out below), the
parameters from a reference-keyed state_dict.  No code is shared with the CUDA path.  The eval forward (eval-mode
BatchNorm, no dropout) is pinned to the real reference's logits in ``tests/golden/general_*.npz``
(tests/test_general_oracle.py); the same graph with autograd is the gradient reference of the general path's training
(tests/test_general_training_gpu.py).  Training-mode dropout takes explicit keep masks instead of torch's random draws.

Reference lines followed (relative to the reference's src/wav2sleep/):
  SignalEncoders / SignalEncoder   models/wav2sleep.py:83-267 (chunk-causal :248-255, output norm :266, embedding :155-159)
  ConvBlock1D / ConvLayer1D        models/blocks.py:8-71, 129-186 (causal padding + right trim :150-152, :178-182)
  norms / activations              models/utils.py:9-96
  MultiModalAttentionEmbedder      models/wav2sleep.py:270-346 (+ torch nn.TransformerEncoderLayer, either norm order)
  SequenceCNN / DilatedConvBlock   models/wav2sleep.py:349-390 ; models/blocks.py:74-126
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

SAMPLES_PER_EPOCH = {"ABD": 256, "THX": 256, "ECG": 1024, "PPG": 1024, "EOG-L": 4096, "EOG-R": 4096}

# constructor defaults of the reference (models/wav2sleep.py)
ENC_DEFAULTS = dict(norm="instance", causal=False, chunk_causal=True, embed_signals=False, initial_channels=16,
                    max_channels=128, output_norm=False, use_residual=True)
MIX_DEFAULTS = dict(layers=4, dropout=0.0, dim_ff=512, activation="gelu", norm_first=True, nhead=4, register_tokens=0)
SEQ_DEFAULTS = dict(dropout=0.2, num_layers=2, activation="gelu", norm="batch", causal=False, num_dilations=6,
                    kernel_size=7)


def config(case: dict) -> dict:
    """A case's constructor keywords with the reference defaults filled in."""
    return dict(signal_map=dict(case["signal_map"]), num_classes=case["num_classes"],
                enc={**ENC_DEFAULTS, **case["enc"]}, mix={**MIX_DEFAULTS, **case["mix"]}, seq={**SEQ_DEFAULTS, **case["seq"]})


def act(x, name):
    """get_activation (models/utils.py:61-74)."""
    if name == "relu":
        return torch.relu(x)
    if name == "leaky":
        return torch.where(x > 0, x, 0.01 * x)
    if name == "gelu":
        return 0.5 * x * (1.0 + torch.erf(x * (1.0 / math.sqrt(2.0))))
    if name in ("silu", "swish"):
        return x * torch.sigmoid(x)
    if name == "linear":
        return x
    raise ValueError(name)


def norm(x_BCL, kind, sd, pre, eps=None):
    """get_norm (models/utils.py:9-96) on a [B, C, L] tensor; BatchNorm in eval mode (running statistics)."""
    C = x_BCL.shape[1]
    if kind is None:
        return x_BCL
    if kind == "instance":  # affine=False, biased variance over L
        mu = x_BCL.mean(2, keepdim=True)
        var = (x_BCL - mu).pow(2).mean(2, keepdim=True)
        return (x_BCL - mu) / torch.sqrt(var + eps)
    if kind == "layer":  # ConvLayerNorm: statistics over channels
        mu = x_BCL.mean(1, keepdim=True)
        var = (x_BCL - mu).pow(2).mean(1, keepdim=True)
        return sd[f"{pre}.weight"] * ((x_BCL - mu) / torch.sqrt(var + 1e-5)) + sd[f"{pre}.bias"]
    if kind == "rms":  # ConvRMSNorm
        return sd[f"{pre}.weight"] * (x_BCL / torch.sqrt(x_BCL.pow(2).mean(1, keepdim=True) + 1e-5))
    if kind == "group":  # ConvGroupNorm(num_features): 8 groups, fewer when C < 8
        G = min(8, C)
        xg = x_BCL.reshape(x_BCL.shape[0], G, -1)
        mu = xg.mean(2, keepdim=True)
        var = (xg - mu).pow(2).mean(2, keepdim=True)
        y = ((xg - mu) / torch.sqrt(var + 1e-5)).reshape_as(x_BCL)
        return y * sd[f"{pre}.norm.weight"][None, :, None] + sd[f"{pre}.norm.bias"][None, :, None]
    if kind == "batch":
        rm, rv = sd[f"{pre}.running_mean"][None, :, None], sd[f"{pre}.running_var"][None, :, None]
        return (x_BCL - rm) / torch.sqrt(rv + 1e-5) * sd[f"{pre}.weight"][None, :, None] + sd[f"{pre}.bias"][None, :, None]
    raise ValueError(kind)


def conv_layer(x, sd, pre, k, stride, dil, padding, causal, norm_kind, activation, eps=None):
    """ConvLayer1D.forward (blocks.py:173-186): conv (bias only without a norm), causal right trim, norm, activation."""
    pad = (k - 1) * dil if causal else padding
    y = F.conv1d(x, sd[f"{pre}.conv.weight"], sd.get(f"{pre}.conv.bias") if norm_kind is None else None, stride=stride,
                 padding=pad, dilation=dil)
    if causal and pad > 0:
        trim = max(pad - (stride - 1), 0)
        if trim:
            y = y[..., :-trim]
    return act(norm(y, norm_kind, sd, f"{pre}.norm", eps), activation)


def signal_encoder(x_BT, sd, pre, spe, e):
    """SignalEncoder.forward (models/wav2sleep.py:235-267) -> [B, S, F] (before output masking)."""
    B, T = x_BT.shape
    S = T // spe
    chunked = e["causal"] and e["chunk_causal"]
    causal_conv = e["causal"] and not e["chunk_causal"]
    y = x_BT.reshape(B * S, 1, spe) if chunked else x_BT.unsqueeze(1)
    n_blocks = int(math.log2(spe)) - 2
    for i in range(n_blocks):
        nk = ("instance" if i < 2 else "layer") if e["norm"] == "auto" else e["norm"]
        eps = 1e-2 if nk == "instance" else None
        bp = f"{pre}.cnn.{i}"
        a = e["activation"]
        out = conv_layer(y, sd, f"{bp}.conv1", 3, 1, 1, 1, causal_conv, nk, a, eps)
        out = conv_layer(out, sd, f"{bp}.conv2", 3, 1, 1, 1, causal_conv, nk, a, eps)
        out = conv_layer(out, sd, f"{bp}.conv3", 3, 2, 1, 1, causal_conv, nk, a, eps)
        if e["use_residual"]:
            out = out + F.conv1d(y, sd[f"{bp}.downsample.weight"], None, stride=2)
        y = act(out, a)
    C = y.shape[1]
    z = y.transpose(1, 2).reshape(B, S, 4 * C) @ sd[f"{pre}.linear.weight"].t() + sd[f"{pre}.linear.bias"]
    z = act(z, e["activation"])
    if e["output_norm"]:
        z = F.layer_norm(z, (z.shape[-1],), sd[f"{pre}.output_norm.weight"], sd[f"{pre}.output_norm.bias"], 1e-5)
    return z


def _drop(x, mask, p):
    """nn.Dropout in training with an explicit keep mask (1 = keep); identity without a mask."""
    return x if mask is None else x * mask.to(x.dtype).reshape(x.shape) / (1.0 - p)


def transformer_layer(x, key_mask, sd, pre, m, drop=None):
    """nn.TransformerEncoderLayer (batch_first, either norm order) with nn.MultiheadAttention written out.  ``drop``:
    training keep masks {"attn": [N, H, D, D], "sa": [N, D, F], "ff": [N, D, dim_ff], "out": [N, D, F]}."""
    drop = drop or {}
    p = m["dropout"]
    N, D, Fd = x.shape
    H = m["nhead"]
    hd = Fd // H
    ln = lambda t, k: F.layer_norm(t, (Fd,), sd[f"{pre}.{k}.weight"], sd[f"{pre}.{k}.bias"], 1e-5)

    def sa(h):
        q, k, v = (h @ sd[f"{pre}.self_attn.in_proj_weight"].t() + sd[f"{pre}.self_attn.in_proj_bias"]).split(Fd, -1)
        q, k, v = (t.reshape(N, D, H, hd).transpose(1, 2) for t in (q, k, v))
        s = (q @ k.transpose(-1, -2)) / math.sqrt(hd)
        s = s.masked_fill(key_mask[:, None, None, :], float("-inf"))
        o = (_drop(torch.softmax(s, -1), drop.get("attn"), p) @ v).transpose(1, 2).reshape(N, D, Fd)
        return _drop(o @ sd[f"{pre}.self_attn.out_proj.weight"].t() + sd[f"{pre}.self_attn.out_proj.bias"], drop.get("sa"), p)

    def ff(h):
        h = _drop(act(h @ sd[f"{pre}.linear1.weight"].t() + sd[f"{pre}.linear1.bias"], m["activation"]), drop.get("ff"), p)
        return _drop(h @ sd[f"{pre}.linear2.weight"].t() + sd[f"{pre}.linear2.bias"], drop.get("out"), p)

    if m["norm_first"]:
        x = x + sa(ln(x, "norm1"))
        return x + ff(ln(x, "norm2"))
    x = ln(x + sa(x), "norm1")
    return ln(x + ff(x), "norm2")


def forward(x: dict, sd: dict, cfg: dict, dropout: dict | None = None) -> torch.Tensor:
    """Wav2Sleep.forward (models/wav2sleep.py:48-67) -> logits [B, S, num_classes].  Autograd flows into whichever
    ``sd`` tensors require grad.  ``dropout``: None (eval) or {"mix": [per-layer mask dicts], "seq": [[B, S, F] per
    sequence-mixer block]} with the sites' keep masks; p is the configuration's."""
    e, m, s = cfg["enc"], cfg["mix"], cfg["seq"]
    d = dropout or {}
    names = sorted(x.keys())
    toks, masks = [], []
    emb_idx = {sig: i for i, sig in enumerate(sorted(cfg["signal_map"]))}
    dtype = sd["classifier.weight"].dtype  # fp32; fp64 parameters give an fp64 graph (a rounding-free reference)
    for n in names:
        x_BT = x[n].to(dtype)
        mask = torch.isinf(x_BT[:, 0])
        x_BT = torch.where(torch.isinf(x_BT), torch.zeros_like(x_BT), x_BT)
        z = signal_encoder(x_BT, sd, f"signal_encoders.encoders.{cfg['signal_map'][n]}", SAMPLES_PER_EPOCH[n], e)
        if e["embed_signals"]:
            z = z + sd["signal_encoders.embedder.weight"][emb_idx[n]]
        # the reference writes -inf into missing rows and the mixer turns them into zeroed, key-masked tokens
        toks.append(torch.where(mask[:, None, None], torch.zeros_like(z), z))
        masks.append(mask)
    B, S, Fd = toks[0].shape
    reg = sd["epoch_mixer.register_tokens"][0, 0]  # [F, R + 1]; column 0 is the CLS token
    R1 = reg.shape[1]
    xt = torch.stack([reg[:, i].expand(B, S, Fd) for i in range(R1)] + toks, dim=2).reshape(B * S, R1 + len(names), Fd)
    km = torch.stack([torch.zeros(B, dtype=torch.bool)] * R1 + masks, dim=1)[:, None, :].expand(B, S, -1).reshape(B * S, -1)
    for li in range(m["layers"]):
        xt = transformer_layer(xt, km, sd, f"epoch_mixer.transformer_encoder.layers.{li}", m,
                               None if "mix" not in d else d["mix"][li])
    h = xt[:, 0, :].reshape(B, S, Fd).transpose(1, 2)
    k = s["kernel_size"]
    for bi in range(s["num_layers"]):
        out = h
        for j in range(s["num_dilations"]):
            dil = 2 ** j
            k_eff = k + (k - 1) * (dil - 1)
            out = conv_layer(out, sd, f"sequence_mixer.dilated_convs.{bi}.conv_layers.{j}", k, 1, dil, k_eff // 2, s["causal"],
                             s["norm"], s["activation"])
        if "seq" in d:
            out = _drop(out, d["seq"][bi].transpose(1, 2), s["dropout"])
        h = act(out + h, s["activation"])
    return h.transpose(1, 2) @ sd["classifier.weight"].t() + sd["classifier.bias"]
