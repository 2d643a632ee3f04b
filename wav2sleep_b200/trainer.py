"""Training harness with the shape of the reference's ``SleepLightningModule`` (trainer/main.py:62-297), without
Lightning (not installed here): same constructor keywords and the same ``forward`` / ``reshape_for_loss`` /
``on_after_batch_transfer`` / ``_step`` / ``training_step`` / ``configure_optimizers`` methods, so a Lightning
``Trainer`` (or the small ``fit`` loop below) can drive it.  The forward/backward it drives is the CUDA path
(model.py -> training.py); the optimizer is the fused clip + AdamW (optim.py).

Data parallelism (SURVEY section 8e): one process per GPU, replicated parameters, ONE exchange per step - the SUM
all-reduce of the flat gradient buffer over NCCL/NVLink.  It is issued in buckets from hooks inside the backward
(``tail`` = classifier + sequence mixer + epoch mixer as soon as they are final, then one bucket per signal encoder as
its backward finishes, largest encoders first) on a side stream, so every bucket but the last, smallest one overlaps
the encoder backward, which is >90 % of the step.
"""
from __future__ import annotations

from typing import Callable, Iterable, Optional

import torch
import torch.distributed as dist
from torch import Tensor, nn

from .optim import ExpWarmUpScheduler, FusedAdamW

TRAIN, VAL, TEST = "train", "val", "test"
# signal / dataset names of the reference (settings.py:2-5, 35-39)
ECG, PPG, THX = "ECG", "PPG", "THX"
SHHS, MESA, CFS, CHAT, CCSHS = "shhs", "mesa", "cfs", "chat", "ccshs"


class SignalMasker:
    """Stochastic modality dropout (reference trainer/masker.py:5-51): per sample keep signal i with prob 1 - p_i; if
    nothing is left, draw one of the available backup signals; dropped signals become rows of -inf, in place.

    On CUDA tensors nothing here synchronises the host with the device (no boolean-mask indexing, no ``if tensor``): the
    two data errors of the reference (a night with every signal unavailable, no backup channel available) are written to
    a device flag, copied to pinned memory asynchronously and raised by the *next* call or by ``check()`` - one step
    late, so that the host can keep enqueueing the training step ahead of the GPU.  ``deferred_errors=False`` restores
    the immediate (synchronising) raise; CPU tensors always raise immediately."""

    def __init__(self, dropouts: dict[str, float], backups: list[str] | None = None, deferred_errors: bool = True):
        self.channel_dropouts = dropouts
        self.backup_channels = backups
        self.deferred_errors = deferred_errors
        self._pending = None  # (pinned flags [2], event)
        self._p_cache = {}    # (device, names) -> probabilities on the device (torch.tensor from a list synchronises)
        for v in dropouts.values():  # host-side checks: the probabilities are Python floats
            if v < 0 or v > 1:
                raise ValueError("dropout probabilities must be in [0, 1]")

    def check(self) -> None:
        """Raise the data error recorded by the previous call, if any."""
        if self._pending is None:
            return
        flags, ev = self._pending
        self._pending = None
        ev.synchronize()
        self._raise(bool(flags[0]), bool(flags[1]))

    @staticmethod
    def _raise(all_missing: bool, no_backup: bool) -> None:
        if all_missing:
            raise ValueError("Found batch element with all signals unavailable.")
        if no_backup:
            raise ValueError("No backup channels for stochastic sampling were available")

    def __call__(self, signals: dict[str, Tensor]) -> dict[str, Tensor]:
        self.check()
        names = list(signals.keys())
        dev = signals[names[0]].device
        ps = [float(self.channel_dropouts.get(n, 0.0)) for n in names]
        if all(v == 1 for v in ps):
            raise ValueError("Dropout probability equal to 1 for all channels.")
        missing = torch.stack([torch.isinf(signals[n][:, 0]) for n in names], dim=-1)  # [B, C] True = unavailable
        key = (str(dev), tuple(names))
        p = self._p_cache.get(key)
        if p is None:
            p = self._p_cache[key] = torch.tensor(ps, device=dev)
        B = missing.size(0)
        keep = torch.rand(B, len(names), device=dev) >= p  # Bernoulli(1 - p)
        if self.backup_channels is not None:
            w = torch.stack([(~missing[:, i]).float() if n in self.backup_channels else torch.zeros(B, device=dev)
                             for i, n in enumerate(names)], dim=-1)
        else:
            w = (~missing).float() * (1 - p)
        flags = torch.stack([missing.all(dim=-1).any(), (w == 0).all(dim=-1).any()])
        if dev.type == "cuda" and self.deferred_errors:
            host = torch.empty(2, dtype=torch.bool).pin_memory()
            host.copy_(flags, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            self._pending = (host, ev)
            w = w + (w == 0).all(dim=-1, keepdim=True).float()  # keep multinomial well defined on a bad row
        else:
            f = flags.tolist()
            self._raise(f[0], f[1])
        backup = torch.nn.functional.one_hot(torch.multinomial(w, 1).squeeze(-1), len(names)).bool()
        none_left = (missing | ~keep).all(dim=-1, keepdim=True)
        keep = torch.where(none_left, backup, keep)
        for i, n in enumerate(names):
            signals[n].masked_fill_(~keep[:, i:i + 1], float("-inf"))
        return signals


def invert_signals(signals: dict[str, Tensor]) -> dict[str, Tensor]:
    """Random polarity flip per (sample, signal), p = 0.5 (reference trainer/main.py:342-353)."""
    for name, x in signals.items():
        flip = 2 * torch.randint(0, 2, (x.size(0), 1), dtype=x.dtype, device=x.device) - 1
        signals[name] = x.mul_(flip)
    return signals


def confusion_matrix(logits_NC: Tensor, y_N: Tensor, num_classes: int, ignore_index: int = -1) -> Tensor:
    """[true, predicted] counts; scatter-add instead of boolean indexing + bincount, so nothing synchronises the host."""
    pred = logits_NC.argmax(-1)
    nn_ = num_classes * num_classes
    idx = torch.where(y_N != ignore_index, y_N.long() * num_classes + pred, torch.full_like(pred, nn_))
    cm = torch.zeros(nn_ + 1, dtype=torch.int64, device=pred.device).scatter_add_(0, idx, torch.ones_like(idx))
    return cm[:nn_].view(num_classes, num_classes)


def sum_if_distributed(t: Tensor) -> Tensor:
    """reference trainer/main.py:41-46 (kept in torch: off the performance path)."""
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


class GradReducer:
    """Bucketed SUM all-reduce of a flat gradient buffer, fired from the backward's bucket hooks."""

    def __init__(self, flat_grad: Tensor, segments: dict[str, tuple[int, int]], process_group=None, use_stream=True):
        """Each bucket is reduced on a side stream as soon as the backward has finished it.  Measured on 2 x B200, one
        all-reduce of the whole flat gradient after the backward takes the same step time (55.5 ms): the exchange is
        only 11.8 MB; the multi-GPU step is longer than the single-GPU one because each rank draws its own modality
        masks and the slowest rank sets the pace."""
        self.flat_grad, self.segments, self.group = flat_grad, segments, process_group
        self.use_stream = use_stream and flat_grad.is_cuda
        self.comm = torch.cuda.Stream(device=flat_grad.device) if self.use_stream else None
        self.done = []
        self.fired = []

    @property
    def world_size(self) -> int:
        return dist.get_world_size(self.group) if (dist.is_available() and dist.is_initialized()) else 1

    def __call__(self, bucket: str) -> None:
        self.fired.append(bucket)
        if self.world_size == 1 or bucket not in self.segments:
            return
        a, b = self.segments[bucket]
        seg = self.flat_grad[a:b]
        if self.use_stream:
            ready = torch.cuda.Event()
            ready.record(torch.cuda.current_stream(seg.device))
            with torch.cuda.stream(self.comm):
                self.comm.wait_event(ready)
                dist.all_reduce(seg, op=dist.ReduceOp.SUM, group=self.group)
                ev = torch.cuda.Event()
                ev.record(self.comm)
            self.done.append(ev)
        else:
            dist.all_reduce(seg, op=dist.ReduceOp.SUM, group=self.group)

    def wait(self) -> None:
        """Make the current stream wait for every bucket issued since the last call (before the optimizer step)."""
        for ev in self.done:
            torch.cuda.current_stream().wait_event(ev)
        self.done.clear()
        self.fired.clear()


class SleepLightningModule(nn.Module):
    def __init__(self, model, criterion=None, optimizer: Optional[Callable] = None, aux_metrics=None,
                 scheduler: Optional[Callable] = None, debug_level=2, on_step: bool = False, on_epoch: bool = True,
                 num_classes: int = 4, masker: SignalMasker | None = None, flip_polarity: bool = True,
                 causal: bool = False):
        super().__init__()
        self.model = model
        self.num_classes = num_classes
        self.criterion = criterion if criterion is not None else nn.CrossEntropyLoss(ignore_index=-1)
        self.optimizer = optimizer if optimizer is not None else (
            lambda params: FusedAdamW(params, lr=1e-3, weight_decay=1e-4, max_grad_norm=1.0))
        self.scheduler = scheduler
        self.masker = masker
        self.flip_polarity = flip_polarity
        self.causal = causal
        # is the model unified, i.e. does it work on multiple modalities (reference trainer/main.py:103-106)
        self.unified = hasattr(model, "signal_encoders") and len(model.signal_encoders) > 1
        if not hasattr(model, "signal_encoders"):
            self.masker = None  # trainer/main.py:97-100: the masker applies to Wav2Sleep models only
        self.cmats = {m: torch.zeros(num_classes, num_classes, dtype=torch.long) for m in (TRAIN, VAL, TEST)}
        # per (signal prefix, dataset) confusion matrices, as the reference's aux_outputs (trainer/main.py:91)
        self.aux_outputs = {m: {} for m in (TRAIN, VAL, TEST)}
        self.val_dataset_map: dict[int, str] = {}
        self.test_dataset_map: dict[int, str] = {}
        self._opt = self._sched = self._reducer = None
        self._bn_buffers, self._process_group = [], None

    def forward(self, x: dict[str, Tensor], y: Tensor | None = None) -> Tensor:
        if not hasattr(self.model, "signal_encoders"):  # SleepPPGNet: one tensor (reference trainer/main.py:108-114)
            if len(x) != 1:
                raise ValueError(f"x.keys()={x.keys()} but expected unimodal input!")
            x = x[list(x.keys())[0]]
        return self.model(x)

    def reshape_for_loss(self, outputs: Tensor, labels: Tensor):
        return outputs.view(-1, outputs.size(-1)), labels.view(-1)

    def on_after_batch_transfer(self, batch, dataloader_idx: int = 0, training: bool = True):
        x, y = batch
        if training:
            if self.flip_polarity:
                invert_signals(x)
            if self.unified and self.masker is not None:
                self.masker(x)
        return x, y

    def get_ds_name(self, dataloader_idx: int, mode: str) -> str:
        """Dataset behind a dataloader index (reference trainer/main.py:118-126; the maps come from the datamodule there,
        here they are plain attributes ``val_dataset_map`` / ``test_dataset_map`` a caller may set)."""
        if mode == TRAIN:
            return "all"
        ds_map = self.val_dataset_map if mode == VAL else self.test_dataset_map
        return ds_map.get(dataloader_idx, "all") if isinstance(ds_map, dict) else ds_map[dataloader_idx]

    def _step(self, batch, mode: str, dataloader_idx: int = 0, signals=None) -> Tensor:
        """Generic step (reference trainer/main.py:140-186): optionally on a subset of the signals; the confusion matrix
        is accumulated per (mode, signal prefix, dataset) as the reference's ``aux_outputs`` are."""
        x, y = batch
        if signals is not None:
            x = {s: x[s] for s in signals}
            sig_prefix = "_".join(signals)
        else:
            sig_prefix = None if self.unified else "_".join(x.keys())
        logits = self(x, y)
        logits_NC, y_N = self.reshape_for_loss(logits, y)
        loss = self.criterion(logits_NC, y_N.long())
        with torch.no_grad():
            cm = sum_if_distributed(confusion_matrix(logits_NC.detach(), y_N, self.num_classes))
            if signals is None:
                self.cmats[mode] = self.cmats[mode].to(cm.device) + cm
            key = (sig_prefix, self.get_ds_name(dataloader_idx, mode))
            prev = self.aux_outputs[mode].get(key)
            self.aux_outputs[mode][key] = cm if prev is None else prev.to(cm.device) + cm
        return loss

    def training_step(self, batch, batch_idx: int = 0) -> Tensor:
        return self._step(batch, TRAIN)

    def _subset_steps(self, batch, mode: str, dataloader_idx: int, ecg_thx_on, ppg_on, ppg_thx_on) -> None:
        """Re-evaluation on the modality subsets a deployment may see (reference trainer/main.py:188-226)."""
        x = batch[0]
        valid = self.model.valid_signals
        ds_name = self.get_ds_name(dataloader_idx, mode)
        if ECG in x and ECG in valid:
            self._step(batch, mode, dataloader_idx, signals=(ECG,))
            if THX in x and THX in valid and (ecg_thx_on is None or ds_name in ecg_thx_on):
                self._step(batch, mode, dataloader_idx, signals=(ECG, THX))
        if PPG in x and PPG in valid and ds_name in ppg_on:
            self._step(batch, mode, dataloader_idx, signals=(PPG,))
            if THX in x and THX in valid and ds_name in ppg_thx_on:
                self._step(batch, mode, dataloader_idx, signals=(PPG, THX))

    def validation_step(self, batch, batch_idx: int = 0, dataloader_idx: int = 0) -> Tensor:
        with torch.no_grad():
            loss = self._step(batch, VAL, dataloader_idx)
            if dataloader_idx == 0 or not self.unified:  # the combined loader / single-modality models: no subsets
                return loss
            self._subset_steps(batch, VAL, dataloader_idx, ecg_thx_on=(SHHS, MESA), ppg_on=(MESA, CFS, CCSHS, CHAT),
                               ppg_thx_on=(MESA,))
            return loss

    def test_step(self, batch, batch_idx: int = 0, dataloader_idx: int = 0) -> Tensor:
        with torch.no_grad():
            loss = self._step(batch, TEST, dataloader_idx)
            if self.unified:
                self._subset_steps(batch, TEST, dataloader_idx, ecg_thx_on=None, ppg_on=(MESA, CFS, CCSHS, CHAT),
                                   ppg_thx_on=(MESA,))
            return loss

    def predict_step(self, batch) -> dict:
        """Predictions from ECG only, ECG + THX and all modalities (reference trainer/main.py:228-243)."""
        x, y = batch
        out = {"labels": y}
        with torch.no_grad():
            if ECG in x:
                out[f"preds_{ECG}"] = self.model.predict({ECG: x[ECG]})
            if ECG in x and THX in x:
                out[f"preds_{ECG}_{THX}"] = self.model.predict({ECG: x[ECG], THX: x[THX]})
            out["preds"] = self.model.predict(x)
        return out

    # EMACallback hooks (reference trainer/callbacks.py:88-110): evaluate with the averaged weights kept by the optimizer
    def on_validation_epoch_start(self) -> None:
        if isinstance(self._opt, FusedAdamW):
            self._opt.swap_to_ema()

    def on_validation_epoch_end(self) -> None:
        if isinstance(self._opt, FusedAdamW):
            self._opt.swap_to_original()

    on_test_epoch_start, on_test_epoch_end = on_validation_epoch_start, on_validation_epoch_end

    def configure_optimizers(self) -> dict:
        optimizer = self.optimizer(self.model.parameters())
        out = {"optimizer": optimizer}
        if self.scheduler is not None:
            out["lr_scheduler"] = {"scheduler": self.scheduler(optimizer), "interval": "step", "frequency": 1,
                                   "strict": True}
        return out

    # ---- Lightning-free driver (what Lightning's loop + DDP strategy would do) ----
    def setup_training(self, process_group=None) -> None:
        cfg = self.configure_optimizers()
        self._opt = cfg["optimizer"]
        self._sched = cfg.get("lr_scheduler", {}).get("scheduler")
        if isinstance(self._opt, FusedAdamW):
            if hasattr(self.model, "signal_encoders"):
                enc = list(self.model.signal_encoders.parameters())
                enc_ids = {id(p) for p in enc}
                tail = [p for p in self.model.parameters() if id(p) not in enc_ids]
                segs = {"tail": self._opt.segment(tail)}
                for name, e in self.model.signal_encoders.encoders.items():
                    segs["encoder:" + name] = self._opt.segment(list(e.parameters()))
                covered = sum(b - a for a, b in segs.values())
                if covered != self._opt.flat_grad.numel():  # e.g. a parameter outside encoders / tail: one late bucket
                    segs = {"tail": segs["tail"], "encoders": self._opt.segment(enc)}
            else:  # SleepPPGNet: one bucket covering every parameter
                segs = {"all": self._opt.segment(list(self.model.parameters()))}
            self._reducer = GradReducer(self._opt.flat_grad, segs, process_group)
            self._opt.grad_scale = 1.0 / self._reducer.world_size
            if self._reducer.world_size > 1:
                # what Lightning's DDP strategy does at start-up: every replica begins from rank 0's parameters
                dist.broadcast(self._opt.flat_param, src=0, group=process_group)
                if self._opt.ema is not None:
                    dist.broadcast(self._opt.ema, src=0, group=process_group)
                self._opt._bump()
            if getattr(self.model, "fast_path", False):
                self.model._get_train_engine().bucket_hooks = [self._reducer]
        # BatchNorm buffers (running mean / var, num_batches_tracked) for the rank-0 broadcast of fit_step
        self._bn_buffers = [b for m in self.model.modules() if isinstance(m, nn.modules.batchnorm._BatchNorm)
                            for b in (m.running_mean, m.running_var, m.num_batches_tracked) if b is not None]
        self._process_group = process_group

    def _broadcast_buffers(self) -> None:
        """What DDP does with broadcast_buffers=True (Lightning's default) before each forward: every rank starts the step
        from rank 0's BatchNorm running statistics and counters, in one flat collective.  Each rank still normalises
        with its own batch statistics.  A model without BatchNorm buffers (or one process) issues nothing."""
        if not self._bn_buffers or not (dist.is_available() and dist.is_initialized()):
            return
        if dist.get_world_size(self._process_group) == 1:
            return
        bufs = self._bn_buffers
        f32 = [b for b in bufs if b.dtype == torch.float32]
        i64 = [b for b in bufs if b.dtype == torch.int64]
        # the int64 counters travel bit-exactly as pairs of fp32 words, so one fp32 buffer carries everything
        flat = torch.cat([b.reshape(-1) for b in f32] + [b.reshape(-1).view(torch.float32) for b in i64])
        dist.broadcast(flat, src=dist.get_global_rank(self._process_group, 0) if self._process_group is not None else 0,
                       group=self._process_group)
        off = 0
        for b in f32:
            b.copy_(flat[off:off + b.numel()].view_as(b))
            off += b.numel()
        for b in i64:
            b.copy_(flat[off:off + 2 * b.numel()].view(torch.int64).view_as(b))
            off += 2 * b.numel()

    def fit_step(self, batch) -> Tensor:
        """One optimisation step: transforms -> forward -> loss -> backward (+ overlapped all-reduce) -> clip + AdamW."""
        if self._opt is None:
            self.setup_training()
        self.model.train()
        self._broadcast_buffers()
        batch = self.on_after_batch_transfer(batch, training=True)
        self._opt.zero_grad()
        loss = self.training_step(batch)
        loss.backward()
        if self._reducer is not None:
            if not getattr(self.model, "fast_path", False):
                # the general path's backward is plain autograd and fires no bucket hooks: every gradient is final now
                for name in self._reducer.segments:
                    self._reducer(name)
            self._reducer.wait()
        self._opt.step()
        if self._sched is not None:
            self._sched.step()
        return loss.detach()

    def fit(self, batches: Iterable, max_steps: int | None = None) -> list[float]:
        losses = []
        for i, batch in enumerate(batches):
            if max_steps is not None and i >= max_steps:
                break
            losses.append(float(self.fit_step(batch)))
        return losses
