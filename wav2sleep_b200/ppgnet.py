"""``SleepPPGNet`` baseline (SURVEY section 8f, row N4): drop-in mirror of ``wav2sleep.models.ppgnet.SleepPPGNet``
(/root/reference/src/wav2sleep/models/ppgnet.py:19-126) whose forward runs on the general fp32 CUDA kernels
(csrc/general.cuh through general.py): eight ``ConvBlock1D`` (batch norm, leaky ReLU) -> time-distributed
``Linear(1024 -> F)`` -> two ``DilatedConvBlock`` -> classifier.  Same constructor keywords, parameter names and default
initialisation as the reference, not tuned.  In ``eval()``, and in ``train()`` under ``no_grad``, BatchNorm uses its
running statistics; under ``train()`` with grad the forward builds the general path's autograd graph with train-mode
BatchNorm (batch statistics over B x length, running-statistics update) and dropout at ``DilatedConvBlock.dropout``.
In ``eval()`` an input that requires grad gets an eval-semantics graph (input gradients, attribution.py).
"""
from __future__ import annotations

import torch
from torch import Tensor, nn

from .model import ConvBlock1D, DilatedConvBlock, get_activation

__all__ = ("SleepPPGNet",)


class WindowEncoder(nn.Module):
    """ppgnet.py:77-101"""

    CHANNELS = [16, 16, 32, 32, 64, 64, 128, 256]

    def __init__(self, activation: str = "leaky", norm: str = "batch") -> None:
        super().__init__()
        blocks, cin = [], 1
        for cout in self.CHANNELS:
            blocks.append(ConvBlock1D(cin, cout, activation=activation, norm=norm))
            cin = cout
        self.model = nn.Sequential(*blocks)


class DenseBlock(nn.Module):
    """ppgnet.py:104-126"""

    def __init__(self, in_dim: int = 1024, out_dim: int = 128, activation: str = "leaky") -> None:
        super().__init__()
        self.linear = nn.Linear(in_dim, out_dim)
        self.activation = get_activation(activation)
        self.activation_name = activation


class SleepPPGNet(nn.Module):
    INPUT_LENGTH: int = 1228800  # ppgnet.py:20

    def __init__(self, n_classes: int = 4, feature_dim: int = 128, dropout: float = 0.2, activation: str = "leaky",
                 norm: str = "batch") -> None:
        super().__init__()
        self.feature_dim = feature_dim
        self.conv_block = WindowEncoder(activation=activation, norm=norm)
        self.dense = DenseBlock(in_dim=1024, out_dim=feature_dim)
        self.dilated_convs = nn.Sequential(*[
            DilatedConvBlock(feature_dim=feature_dim, dropout=dropout, activation=activation, norm=norm) for _ in range(2)])
        self.classifier = nn.Linear(in_features=feature_dim, out_features=n_classes)
        self._general = None

    def _engine(self):
        from .general import GeneralEngine  # deferred: loads the CUDA library
        if self._general is None:
            object.__setattr__(self, "_general", GeneralEngine(self))
        return self._general

    @torch.no_grad()
    def encode(self, x_BT: Tensor) -> Tensor:
        """[N, 1228800] -> features [N, 1200, F]   (ppgnet.py:42-59), inference kernels."""
        return self._features(x_BT)

    def _features(self, x_BT: Tensor) -> Tensor:
        if x_BT.dim() != 2 or x_BT.size(1) != self.INPUT_LENGTH:
            raise ValueError(f"Input tensor had unexpected shape: {x_BT.size()}")
        if not x_BT.is_cuda:
            raise RuntimeError("wav2sleep_b200 runs on CUDA (sm_100a) only: move inputs with .to('cuda'); "
                               "there is no CPU fallback")
        eng = self._engine()
        B = x_BT.size(0)
        with torch.cuda.device(x_BT.device):
            # stays on the autograd graph when the input requires grad; block 0 reads the signal as it is (no
            # missing-sample rule, as in the reference), so its convs run with raw = 0 in every mode
            a = x_BT.to(torch.float32).contiguous().view(B, self.INPUT_LENGTH, 1)
            for blk in self.conv_block.model:
                a = eng.conv_block(a, blk)
            # [B, 4800, 256] channels-last == transpose(-1, -2) of the reference tensor; reshape(-1, 1200, 1024)
            rows = a.reshape(B * 1200, 1024)
            z = eng.affine_act(eng.linear(rows, self.dense.linear).view(B, 1200, -1), self.dense.activation_name)
            return eng.dilated_blocks(z, self.dilated_convs)

    def _logits(self, feat: Tensor) -> Tensor:
        B, S, Fd = feat.shape
        with torch.cuda.device(feat.device):
            return self._engine().linear(feat.reshape(B * S, Fd), self.classifier).view(B, S, -1)

    def forward(self, x_BT: Tensor) -> Tensor:
        """[N, 1228800] -> logits [N, 1200, n_classes]   (ppgnet.py:61-74).

        Under ``train()`` with grad enabled (and a parameter or the input that requires grad) the logits carry a grad_fn
        whose backward runs the general path's backward kernels; BatchNorm normalises with the batch statistics and
        updates its running statistics, and ``DilatedConvBlock.dropout`` draws its masks as
        ``GeneralEngine.training_forward`` describes.  In ``eval()``, an input that requires grad gets an eval-semantics
        graph (BatchNorm on its running statistics, no dropout) whose logits are bitwise those of inference, and
        ``x_BT.grad`` receives d(objective)/dx.  Otherwise the inference kernels run with the running statistics and no
        dropout."""
        grad_on = torch.is_grad_enabled()
        input_grad = grad_on and isinstance(x_BT, Tensor) and x_BT.requires_grad
        if self.training and grad_on and (input_grad or any(p.requires_grad for p in self.parameters())):
            with self._engine().training_forward():
                return self._logits(self._features(x_BT))
        if input_grad:
            return self._logits(self._features(x_BT))
        return self._logits(self.encode(x_BT))
