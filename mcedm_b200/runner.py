"""Lightning-free runner with the hook order the reference relies on.

The reference is orchestrated by `pytorch_lightning.Trainer` (run.py:74-112, configs/trainer/
trainer_ddim.yaml); Lightning is not part of this image and orchestration is outside the hot path, so
this module provides the minimum that keeps the reference's module code shape intact:

  * `LightningModule` — base class with `log`, `save_hyperparameters`, `current_epoch`, `trainer`,
    `optimizer_step` (if pytorch_lightning is importable its class is used instead, so the same
    `PlMcedm` also runs under a real Lightning Trainer);
  * `Trainer.fit / validate / test` — one process per GPU (torchrun), NCCL gradient all-reduce on one
    flat buffer per step, gradient-norm clipping as `gradient_clip_val` (trainer_ddim.yaml:8-9),
    hooks called in Lightning's order: setup('fit') -> training_step -> backward -> [all-reduce] ->
    clip -> optimizer_step (module hook, which also updates the EMA) -> validation_step / test_step;
  * `ModelCheckpoint` — `checkpoints/last.ckpt` with Lightning's top-level key layout (`state_dict`,
    `optimizer_states`, `epoch`, `global_step`, `hyper_parameters`, ...); `fit(ckpt_path=...)` resumes like
    `trainer.fit(ckpt_path=...)` of run.py:99: weights, Adam moments + step counter, global step, next epoch;
  * `precision=16` / "16" / "16-mixed" — dynamic loss scaling (loss_scale.py) of a network training on the fp16 plan,
    checkpointed as Lightning's `native_amp_scaling_state` (torch.amp.GradScaler.state_dict() layout).

Data parallelism is THIS trainer's flat all-reduce; the kernels' autograd nodes bind `p.grad` to slices of the engine's
flat gradient buffer directly, so the per-parameter reducer hooks of `torch.nn.parallel.DistributedDataParallel`
(Lightning's `strategy: ddp`) never fire: under a real Lightning Trainer the module runs on one device only.
"""
from __future__ import annotations

import os
from typing import Any, Dict, Optional

import torch
import torch.distributed as dist

try:  # pragma: no cover - not installed in this image
    import pytorch_lightning as _pl

    _PlBase = _pl.LightningModule
    HAVE_LIGHTNING = True
except Exception:  # noqa: BLE001
    _pl = None
    _PlBase = None
    HAVE_LIGHTNING = False


class _ShimLightningModule(torch.nn.Module):
    """The subset of pytorch_lightning.LightningModule the m-cedm modules use."""

    def __init__(self, *args, **kwargs):
        super().__init__()
        self.trainer = None
        self.current_epoch = 0
        self.global_step = 0
        self.logged: Dict[str, Any] = {}
        self._hparams_saved = None

    def save_hyperparameters(self, *args, **kwargs):
        self._hparams_saved = True

    def log(self, name, value, **kwargs):
        self.logged[name] = value.detach() if torch.is_tensor(value) else value
        if self.trainer is not None:
            self.trainer._record(name, value, kwargs)

    def setup(self, stage: Optional[str] = None):
        return None

    def optimizer_step(self, epoch=None, batch_idx=None, optimizer=None, optimizer_closure=None, **kwargs):
        if optimizer_closure is not None:
            optimizer_closure()
        if optimizer is not None:
            optimizer.step()

    @property
    def device(self):
        for p in self.parameters():
            return p.device
        return torch.device("cpu")


LightningModule = _PlBase if HAVE_LIGHTNING else _ShimLightningModule


class ModelCheckpoint:
    def __init__(self, dirpath="checkpoints/", filename="epoch", save_last=True, **_unused):
        self.dirpath, self.filename, self.save_last = dirpath, filename, save_last

    def format_name(self, epoch: int, step: int) -> str:
        """Lightning's naming: `{epoch}` / `{step}` fields are substituted as `epoch=3`; a filename without fields gets
        the default `epoch=E-step=S` suffix-free form only when it is None."""
        name = self.filename if self.filename is not None else "{epoch}-{step}"
        return name.replace("{epoch}", f"epoch={epoch}").replace("{step}", f"step={step}")

    def save(self, trainer, module, epoch):
        if trainer.global_rank != 0:
            return
        os.makedirs(self.dirpath, exist_ok=True)
        hp = getattr(module, "hparams", None)
        ckpt = {
            "epoch": epoch, "global_step": module.global_step,
            # Lightning reads these when a checkpoint is handed to `trainer.fit/test(ckpt_path=...)` (eval_model.py:77)
            "pytorch-lightning_version": getattr(_pl, "__version__", "1.9.0") if _pl is not None else "1.9.0",
            "state_dict": module.state_dict(),
            "loops": None, "callbacks": {}, "lr_schedulers": [],
            "hyper_parameters": hp if isinstance(hp, dict) else ({} if hp is None else dict(hp)),
        }
        if trainer.optimizer is not None:
            ckpt["optimizer_states"] = [trainer.optimizer.state_dict()]
        scaler = trainer.loss_scaler(module)
        if scaler is not None:
            ckpt["native_amp_scaling_state"] = scaler.state_dict()
        torch.save(ckpt, os.path.join(self.dirpath, f"{self.format_name(epoch, module.global_step)}.ckpt"))
        if self.save_last:
            torch.save(ckpt, os.path.join(self.dirpath, "last.ckpt"))


class Trainer:
    """Single-node data-parallel trainer: one process per GPU, launched by torchrun."""

    def __init__(self, max_epochs=500, accelerator="gpu", devices=1, num_nodes=1, precision=32, strategy="ddp",
                 gradient_clip_algorithm="norm", gradient_clip_val=1.0, check_val_every_n_epoch=1, callbacks=None,
                 max_steps=None, **_unused):
        if gradient_clip_algorithm != "norm":
            raise NotImplementedError("only gradient_clip_algorithm='norm' is supported")
        self.max_epochs, self.max_steps = max_epochs, max_steps
        self.gradient_clip_val = gradient_clip_val
        self.precision = precision
        self.check_val_every_n_epoch = check_val_every_n_epoch
        self.callbacks = list(callbacks or [])
        self.datamodule = None
        self.optimizer = None
        self.optimizers = []
        self.metrics: Dict[str, list] = {}
        self.world_size = dist.get_world_size() if dist.is_initialized() else 1
        self.global_rank = dist.get_rank() if dist.is_initialized() else 0
        self._flat_grad = None

    # ---- logging -------------------------------------------------------------------------------
    def _record(self, name, value, kwargs):
        v = value.detach().float() if torch.is_tensor(value) else torch.tensor(float(value))
        self.metrics.setdefault(name, []).append((v, bool(kwargs.get("sync_dist", False))))

    def epoch_metrics(self) -> Dict[str, float]:
        """Mean over the epoch's logged values; `sync_dist=True` entries are mean-reduced over ranks."""
        out = {}
        for name, vals in self.metrics.items():
            m = torch.stack([v.reshape(()).to("cpu") if not v.is_cuda else v.reshape(()) for v, _ in vals]).mean()
            if vals[0][1] and self.world_size > 1:
                m = m.to(self._device) if m.device.type == "cpu" and dist.get_backend() == "nccl" else m
                dist.all_reduce(m)
                m = m / self.world_size
            out[name] = float(m)
        self.metrics.clear()
        return out

    # ---- dynamic loss scaling --------------------------------------------------------------------
    def loss_scaler(self, module):
        """The LossScaler of the module's network when it trains on the fp16 plan with dynamic scaling, else None."""
        from .loss_scale import active_scaler

        net = getattr(module, "model", None)
        return active_scaler(net) if net is not None else None

    def _enable_loss_scaling(self, module):
        """precision 16 / "16" / "16-mixed": a LossScaler on the network's engine when its backward runs on the fp16
        plan (other precision values and the fp32-stream plan keep the static path)."""
        from .loss_scale import LossScaler, dynamic_precision

        net = getattr(module, "model", None)
        if not dynamic_precision(self.precision) or net is None or not hasattr(net, "engine"):
            return
        eng = net.engine()
        if getattr(eng, "train_plan", None) == "fused16" and getattr(eng, "loss_scaler", None) is None:
            from .optim import FusedAdam

            if not isinstance(self.optimizer, FusedAdam):
                raise NotImplementedError("dynamic loss scaling skips steps inside the fused Adam kernel: precision=16 "
                                          "needs optimizer 'Adam'")
            eng.loss_scaler = LossScaler()

    # ---- data-parallel gradient exchange -------------------------------------------------------
    def _allreduce_grads(self, params):
        """One all-reduce over a single flat buffer (SURVEY §2c: 196 tensors, 6.35 MB fp32)."""
        if self.world_size == 1:
            return
        grads = [p.grad for p in params if p.grad is not None]
        if not grads:
            return
        n = sum(g.numel() for g in grads)
        if self._flat_grad is None or self._flat_grad.numel() != n or self._flat_grad.device != grads[0].device:
            self._flat_grad = torch.empty(n, device=grads[0].device, dtype=grads[0].dtype)
        flat = self._flat_grad
        views, off = [], 0
        for g in grads:
            views.append(flat[off:off + g.numel()].view_as(g))
            off += g.numel()
        torch._foreach_copy_(views, grads)
        dist.all_reduce(flat)
        flat.div_(self.world_size)
        torch._foreach_copy_(grads, views)

    # ---- loops ---------------------------------------------------------------------------------
    def _attach(self, module, datamodule):
        module.trainer = self
        self.datamodule = datamodule
        self._device = next(module.parameters()).device

    def _to_device(self, batch):
        if torch.is_tensor(batch):
            return batch.to(self._device, non_blocking=True)
        if isinstance(batch, dict):
            return {k: self._to_device(v) for k, v in batch.items()}
        if isinstance(batch, (list, tuple)):
            return type(batch)(self._to_device(v) for v in batch)
        return batch

    def fit(self, module, datamodule, ckpt_path=None):
        self._attach(module, datamodule)
        datamodule.setup("fit")
        module.setup("fit")
        self.optimizer = module.configure_optimizers()["optimizer"]
        self.optimizers = [self.optimizer]
        self._enable_loss_scaling(module)
        params = [p for g in self.optimizer.param_groups for p in g["params"]]
        from .optim import FusedAdam

        fused = isinstance(self.optimizer, FusedAdam)
        if fused:
            self.optimizer.max_grad_norm = self.gradient_clip_val or None
            self.optimizer.grad_scale = 1.0 / self.world_size
        step = 0
        first_epoch = module.current_epoch
        if ckpt_path:
            # resume as `trainer.fit(model, datamodule, ckpt_path=...)` (run.py:99): weights, optimizer moments and
            # step counter (bias correction continues), global step; the saved epoch is complete -> start at the next
            ckpt = torch.load(ckpt_path, map_location=self._device, weights_only=False)
            module.load_state_dict(ckpt["state_dict"])
            if ckpt.get("optimizer_states"):
                self.optimizer.load_state_dict(ckpt["optimizer_states"][0])
            scaler = self.loss_scaler(module)
            if scaler is not None and ckpt.get("native_amp_scaling_state"):
                scaler.load_state_dict(ckpt["native_amp_scaling_state"])
            module.global_step = step = int(ckpt.get("global_step", 0))
            first_epoch = int(ckpt.get("epoch", -1)) + 1
            net = getattr(module, "model", None)
            if getattr(net, "dropout", 0.0):
                # dropout masks are keyed by the step counter: a resumed run continues it instead of repeating masks
                net.engine().dropout_step = step
        history = []
        for epoch in range(first_epoch, self.max_epochs):
            module.current_epoch = epoch
            module.train()
            for batch_idx, batch in enumerate(datamodule.train_dataloader()):
                batch = self._to_device(batch)
                self.optimizer.zero_grad(set_to_none=True)
                loss = module.training_step(batch, batch_idx)
                loss.backward()
                if fused:
                    # gradients already live in one flat buffer: all-reduce it in place (sum; the 1/world factor and
                    # the clip coefficient are folded into the Adam kernel).  flat_grads() is idempotent within a step,
                    # so the optimizer.step() inside the module's optimizer_step hook consumes this reduced tensor.
                    if self.world_size > 1:
                        dist.all_reduce(self.optimizer.flat_grads())
                else:
                    self._allreduce_grads(params)
                    if self.gradient_clip_val:
                        torch.nn.utils.clip_grad_norm_(params, self.gradient_clip_val)
                module.optimizer_step(epoch, batch_idx, self.optimizer)
                module.global_step = step = step + 1
                if self.max_steps and step >= self.max_steps:
                    break
            if (epoch + 1) % self.check_val_every_n_epoch == 0:
                self.validate(module, datamodule, _attached=True)
            history.append(self.epoch_metrics())
            for cb in self.callbacks:
                if isinstance(cb, ModelCheckpoint):
                    cb.save(self, module, epoch)
            if self.max_steps and step >= self.max_steps:
                break
        return history

    @torch.no_grad()
    def validate(self, module, datamodule, _attached=False):
        if not _attached:
            self._attach(module, datamodule)
            datamodule.setup("validate")
        module.eval()
        outs = [module.validation_step(self._to_device(b), i) for i, b in enumerate(datamodule.val_dataloader())]
        return outs

    @torch.no_grad()
    def test(self, module, datamodule, ckpt_path=None):
        self._attach(module, datamodule)
        datamodule.setup("test")
        if ckpt_path:
            module.load_state_dict(torch.load(ckpt_path, map_location=self._device, weights_only=False)["state_dict"])
        module.eval()
        outs = [module.test_step(self._to_device(b), i) for i, b in enumerate(datamodule.test_dataloader())]
        return outs, self.epoch_metrics()
