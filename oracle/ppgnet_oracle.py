"""CPU oracle for SleepPPGNet training (wav2sleep_b200/ppgnet.py on the general path).  TEST INFRASTRUCTURE ONLY.

A functional fp32 restatement of the reference in plain torch CPU ops, with autograd, built on the helpers of
``oracle/general_oracle.py`` (``act``, ``_drop``): train-mode BatchNorm as ``nn.BatchNorm1d`` computes it, and the
SleepPPGNet forward (models/ppgnet.py:42-74).  No code is shared with the CUDA path.  ``ppgnet_forward`` in eval mode is
pinned to the real reference's logits in ``tests/golden/general_ppgnet.npz`` and ``batch_norm_train`` to
``nn.BatchNorm1d`` (tests/test_ppgnet_oracle.py); the same graph with autograd is the gradient reference of
tests/test_ppgnet_training_gpu.py.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle.general_oracle import _drop, act

PPG_CHANNELS = [16, 16, 32, 32, 64, 64, 128, 256]
EPS = 1e-5


def batch_norm_train(x_BCL, sd, pre, upd, momentum=0.1):
    """nn.BatchNorm1d in train mode (torch.nn.functional.batch_norm, training=True) on a [B, C, L] tensor: mean and biased
    variance over (B, L) normalise.  The updated buffers - num_batches_tracked + 1, then running statistics
    (1 - f) old + f new with the unbiased variance, f = momentum or 1 / num_batches_tracked for momentum None - are
    written to ``upd`` under the state_dict keys ``{pre}.running_mean`` / ``.running_var`` / ``.num_batches_tracked``
    (detached)."""
    C = x_BCL.shape[1]
    mu = x_BCL.mean((0, 2), keepdim=True)
    var = (x_BCL - mu).pow(2).mean((0, 2), keepdim=True)
    n = x_BCL.shape[0] * x_BCL.shape[2]
    nbt = sd[f"{pre}.num_batches_tracked"] + 1
    f = 1.0 / float(nbt) if momentum is None else momentum
    with torch.no_grad():
        upd[f"{pre}.num_batches_tracked"] = nbt
        upd[f"{pre}.running_mean"] = (1 - f) * sd[f"{pre}.running_mean"] + f * mu.reshape(C)
        upd[f"{pre}.running_var"] = (1 - f) * sd[f"{pre}.running_var"] + f * var.reshape(C) * (n / (n - 1))
    y = (x_BCL - mu) / torch.sqrt(var + EPS)
    return y * sd[f"{pre}.weight"][None, :, None] + sd[f"{pre}.bias"][None, :, None]


def batch_norm_eval(x_BCL, sd, pre):
    """nn.BatchNorm1d in eval mode (running statistics)."""
    rm, rv = sd[f"{pre}.running_mean"][None, :, None], sd[f"{pre}.running_var"][None, :, None]
    return (x_BCL - rm) / torch.sqrt(rv + EPS) * sd[f"{pre}.weight"][None, :, None] + sd[f"{pre}.bias"][None, :, None]


def conv_bn_act(x, sd, pre, k, stride, dil, padding, activation, upd):
    """ConvLayer1D.forward (blocks.py:173-186) with BatchNorm: conv (no bias), norm (train mode when ``upd`` is a dict),
    activation."""
    y = F.conv1d(x, sd[f"{pre}.conv.weight"], None, stride=stride, padding=padding, dilation=dil)
    y = batch_norm_eval(y, sd, f"{pre}.norm") if upd is None else batch_norm_train(y, sd, f"{pre}.norm", upd)
    return act(y, activation)


def ppgnet_forward(x, sd, activation="leaky", dropout=None, bn_train=False):
    """SleepPPGNet.forward (models/ppgnet.py:42-74): x [B, 1228800] -> logits [B, 1200, n_classes].  Eight ConvBlock1D
    (batch norm, ``activation``) -> time-distributed Linear(1024 -> F) + leaky ReLU (DenseBlock keeps its default
    activation, ppgnet.py:35) -> two DilatedConvBlock (k = 7, dilations 1 .. 32) -> classifier.  ``dropout``: None or
    {"p": p, "seq": the two DilatedConvBlock keep masks [B, 1200, F]}.  ``bn_train``: train-mode BatchNorm; then
    (logits, updated buffers as a state_dict-keyed dict) is returned."""
    upd = {} if bn_train else None
    dtype = sd["classifier.weight"].dtype
    B = x.shape[0]
    y = x.to(dtype).unsqueeze(1)
    for i in range(len(PPG_CHANNELS)):
        bp = f"conv_block.model.{i}"
        out = conv_bn_act(y, sd, f"{bp}.conv1", 3, 1, 1, 1, activation, upd)
        out = conv_bn_act(out, sd, f"{bp}.conv2", 3, 1, 1, 1, activation, upd)
        out = conv_bn_act(out, sd, f"{bp}.conv3", 3, 2, 1, 1, activation, upd)
        y = act(out + F.conv1d(y, sd[f"{bp}.downsample.weight"], None, stride=2), activation)
    z = y.transpose(-1, -2).reshape(B, 1200, 1024) @ sd["dense.linear.weight"].t() + sd["dense.linear.bias"]
    h = act(z, "leaky").transpose(1, 2)
    for bi in range(2):
        out = h
        for j in range(6):
            dil = 2 ** j
            out = conv_bn_act(out, sd, f"dilated_convs.{bi}.conv_layers.{j}", 7, 1, dil, (7 + 6 * (dil - 1)) // 2,
                              activation, upd)
        if dropout is not None:
            out = _drop(out, dropout["seq"][bi].transpose(1, 2), dropout["p"])
        h = act(out + h, activation)
    logits = h.transpose(1, 2) @ sd["classifier.weight"].t() + sd["classifier.bias"]
    return (logits, upd) if bn_train else logits
