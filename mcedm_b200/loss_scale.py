"""Dynamic loss scaling of the fp16 training plan ("fused16", train16_engine.py): torch.amp.GradScaler's policy with its
state in device memory.

The backward seeds S * dL/dF and stores every data gradient in fp16.  With a `LossScaler` on the engine
(`UNetEngine.loss_scaler`, or `runner.Trainer(precision=16)`), those stores convert WITHOUT saturation (op_fmt
MCEDM_FMT_F16_INF): a gradient beyond fp16's range becomes inf and reaches the fp32 flat gradient as inf / NaN.  The
fused Adam step (optim.FusedAdam) then reads found-inf from its sum-of-squares partials, writes nothing on a skipped
step, and runs `torch._amp_update_scale_`'s rule on the device words below.  No step synchronises with the host, and a
CUDA graph replay reads the current scale.

Without a LossScaler the plan runs its static scale (Train16Mixin.LOSS_SCALE = 1024) as before.
"""
from __future__ import annotations

import math
from typing import Optional

import torch

DYNAMIC_PRECISIONS = (16, "16", "16-mixed")


def dynamic_precision(precision) -> bool:
    """True for the `Trainer(precision=...)` values that turn dynamic loss scaling on (Lightning's fp16 settings)."""
    return any(precision == p and type(precision) is type(p) for p in DYNAMIC_PRECISIONS)


def active_scaler(net) -> Optional["LossScaler"]:
    """The LossScaler of network `net`'s engine when its backward runs on the fused16 plan, else None (the fp32-stream
    plan keeps fp32 gradients and has no loss scale)."""
    eng = net.engine() if hasattr(net, "engine") else None
    sc = getattr(eng, "loss_scaler", None)
    return sc if sc is not None and getattr(eng, "train_plan", None) == "fused16" else None


def _power_of_two(x: float) -> bool:
    if not (isinstance(x, (int, float)) and math.isfinite(x) and x > 0):
        return False
    m, _ = math.frexp(x)
    return m == 0.5


def update_rule(scale: float, tracker: int, found_inf: bool, growth_factor: float, backoff_factor: float,
                growth_interval: int):
    """torch._amp_update_scale_ on host values, in fp32: what mcedm_loss_scale_update does on the device."""
    import numpy as np

    scale = np.float32(scale)
    if found_inf:
        return float(np.float32(scale * np.float32(backoff_factor))), 0
    successful = tracker + 1
    if successful == growth_interval:
        with np.errstate(over="ignore"):
            grown = np.float32(scale * np.float32(growth_factor))
        return float(grown if np.isfinite(grown) else scale), 0
    return float(scale), successful


class LossScaler:
    """Scale, growth tracker and found-inf word of dynamic loss scaling, in device memory.

    Defaults are torch.amp.GradScaler's except `init_scale`: 1024, the static plan's scale, so a run without overflow
    and before the first growth computes the static plan's bits.  The factors must be powers of two (unscaling stays
    exact)."""

    def __init__(self, init_scale: float = 1024.0, growth_factor: float = 2.0, backoff_factor: float = 0.5,
                 growth_interval: int = 2000):
        if not (isinstance(init_scale, (int, float)) and math.isfinite(init_scale) and init_scale > 0):
            raise ValueError(f"LossScaler: init_scale must be positive and finite, got {init_scale!r}")
        if not _power_of_two(growth_factor) or growth_factor <= 1.0:
            raise ValueError(f"LossScaler: growth_factor must be a power of two above 1, got {growth_factor!r}")
        if not _power_of_two(backoff_factor) or backoff_factor >= 1.0:
            raise ValueError(f"LossScaler: backoff_factor must be a power of two below 1, got {backoff_factor!r}")
        if not isinstance(growth_interval, int) or growth_interval < 1:
            raise ValueError(f"LossScaler: growth_interval must be a positive int, got {growth_interval!r}")
        self.growth_factor = float(growth_factor)
        self.backoff_factor = float(backoff_factor)
        self.growth_interval = growth_interval
        self._init_scale = float(init_scale)
        self._init_tracker = 0
        self.scale_t: Optional[torch.Tensor] = None         # fp32 [1]
        self.tracker_t: Optional[torch.Tensor] = None       # int32 [1]
        self.found_inf_t: Optional[torch.Tensor] = None     # fp32 [1]: 1.0 when the last step skipped

    def state(self, dev) -> "LossScaler":
        """Allocates the device words on `dev` on first use (graphs capture their addresses: never reallocated on the
        same device)."""
        if self.scale_t is None or self.scale_t.device != dev:
            scale = self._init_scale if self.scale_t is None else float(self.scale_t.item())
            tracker = self._init_tracker if self.tracker_t is None else int(self.tracker_t.item())
            self.scale_t = torch.full((1,), scale, dtype=torch.float32, device=dev)
            self.tracker_t = torch.full((1,), tracker, dtype=torch.int32, device=dev)
            self.found_inf_t = torch.zeros(1, dtype=torch.float32, device=dev)
        return self

    def update(self, step_count: Optional[torch.Tensor], stream) -> None:
        """One torch._amp_update_scale_ on the device words after an optimizer step; `step_count` (int32 [1], may be
        None) gains one when the step applied."""
        from . import _lib as L

        L.check(L.lib().mcedm_loss_scale_update(L.ptr(self.scale_t), L.ptr(self.tracker_t), L.ptr(self.found_inf_t),
                                                L.ptr(step_count), self.growth_factor, self.backoff_factor,
                                                self.growth_interval, stream), "loss_scale_update")

    # ---- GradScaler-compatible state (synchronises) -----------------------------------------------------------
    def get_scale(self) -> float:
        return float(self.scale_t.item()) if self.scale_t is not None else self._init_scale

    def get_growth_tracker(self) -> int:
        return int(self.tracker_t.item()) if self.tracker_t is not None else self._init_tracker

    def state_dict(self) -> dict:
        """torch.amp.GradScaler.state_dict()'s layout (Lightning stores it as `native_amp_scaling_state`)."""
        return {"scale": self.get_scale(), "growth_factor": self.growth_factor, "backoff_factor": self.backoff_factor,
                "growth_interval": self.growth_interval, "_growth_tracker": self.get_growth_tracker()}

    def load_state_dict(self, sd: dict) -> None:
        fresh = LossScaler(float(sd["scale"]), float(sd["growth_factor"]), float(sd["backoff_factor"]),
                           int(sd["growth_interval"]))
        self.growth_factor, self.backoff_factor = fresh.growth_factor, fresh.backoff_factor
        self.growth_interval = fresh.growth_interval
        self._init_scale, self._init_tracker = fresh._init_scale, int(sd["_growth_tracker"])
        if self.scale_t is not None:                      # in place: captured graphs keep reading these words
            self.scale_t.fill_(self._init_scale)
            self.tracker_t.fill_(self._init_tracker)
            self.found_inf_t.zero_()
