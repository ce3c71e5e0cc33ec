"""Fused optimizer step of the training path: gradient-norm clipping + Adam on ONE flat fp32 buffer, and the EMA
update (models/mcedm.py:139-168 configure_optimizers / optimizer_step, models/ddim_blocks.py:38-59 EmaModel,
configs/trainer/trainer_ddim.yaml:8-9 gradient_clip_val).

`FusedAdam` keeps torch.optim.Adam's constructor arguments, `param_groups` and `state_dict()` layout
(`step`, `exp_avg`, `exp_avg_sq` per parameter) so checkpoints interchange; the parameters are re-bound as views
of one contiguous buffer, which is also what the data-parallel gradient all-reduce runs on.

Under dynamic loss scaling (loss_scale.py; `loss_scaler_provider` returns the engine's LossScaler) a step is
sum-of-squares partials -> Adam that writes nothing when they are not finite (found-inf) -> the scale update.  The
applied-step count then lives in device memory (no host synchronisation per step); `state_dict()` reads it back.
"""
from __future__ import annotations

import weakref
from typing import Optional

import torch

from . import _lib as L


# data_ptr of the first parameter -> the flat buffer its parameter list lives in.  Weak values: the buffer is owned by
# the optimizer / EMA state that created it (and by the parameter views into it); a re-bind or a dead owner drops the
# entry instead of pinning ~6 MB of device memory per stale binding for the life of the process.
_FLAT = weakref.WeakValueDictionary()


def _flatten_(params):
    """Re-binds every parameter's storage to a slice of one flat fp32 buffer (values preserved)."""
    n = sum(p.numel() for p in params)
    flat = torch.empty(n, device=params[0].device, dtype=torch.float32)
    off = 0
    for p in params:
        v = flat[off:off + p.numel()].view(p.shape)
        v.copy_(p.data)
        p.data = v
        off += p.numel()
    _FLAT[flat.data_ptr()] = flat
    return flat


def _is_flat(params, flat) -> bool:
    if flat is None or not params or flat.device != params[0].device:
        return False
    off = 0
    for p in (params[0], params[-1]):
        if p is params[-1]:
            off = flat.numel() - p.numel()
        if p.data_ptr() != flat.data_ptr() + 4 * off:
            return False
    return True


class FusedAdam(torch.optim.Adam):
    """torch.optim.Adam whose `step()` is one CUDA kernel over flat buffers (binding happens on first use, once the
    module has been moved to its device; stepping CPU parameters raises — there is no CPU path)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False,
                 max_grad_norm: Optional[float] = None):
        if amsgrad:
            raise NotImplementedError("FusedAdam: amsgrad has no kernel")
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False)
        if len(self.param_groups) != 1:
            raise NotImplementedError("FusedAdam: one parameter group")
        self.max_grad_norm = max_grad_norm      # set by the trainer from gradient_clip_val
        self.grad_scale = 1.0                   # 1/world_size when the all-reduce sums
        self.grad_provider = None               # callable -> the engine's flat gradient buffer (zero-copy path)
        self.loss_scaler_provider = None        # callable -> the engine's LossScaler or None (dynamic loss scaling)
        self._step_dev = None                   # int32 [1]: applied steps, while dynamic loss scaling steps
        self._params = list(self.param_groups[0]["params"])
        self._flat_p = None
        self._flat_g = None
        self._pending_g = None                  # the flat gradient of the current step, once fetched (see flat_grads)
        self._steps = 0
        self._n_partial = 128
        if self._params[0].is_cuda:             # normally true: optimizers are configured after the module moved
            self._bind()

    def _bind(self):
        self._sync_steps()
        if not self._params[0].is_cuda:
            raise L.McedmError("FusedAdam needs CUDA parameters: the optimizer kernels have no CPU path")
        dev = self._params[0].device
        if self._flat_p is None or self._partial.device != dev:      # first bind, or the module moved to another device
            self.last_grad_norm = torch.zeros(1, device=dev)
            self._partial = torch.empty(self._n_partial, device=dev, dtype=torch.float64)
        old_m = old_v = None
        if self._flat_p is not None:            # parameters were moved (Module.to): keep the moments
            old_m, old_v = self._m, self._v
            _FLAT.pop(self._flat_p.data_ptr(), None)
        self._pending_g = None
        self._flat_p = _flatten_(self._params)
        dev = self._flat_p.device
        self._m = torch.zeros_like(self._flat_p) if old_m is None else old_m.to(dev)
        self._v = torch.zeros_like(self._flat_p) if old_v is None else old_v.to(dev)
        off = 0
        self._step_t = torch.tensor(float(self._steps))       # one shared host tensor, updated in place
        for p in self._params:
            n = p.numel()
            self.state[p] = {"step": self._step_t,
                             "exp_avg": self._m[off:off + n].view(p.shape),
                             "exp_avg_sq": self._v[off:off + n].view(p.shape)}
            off += n

    def flat_params(self) -> torch.Tensor:
        if not _is_flat(self._params, self._flat_p):
            self._bind()
        return self._flat_p

    def flat_grads(self) -> torch.Tensor:
        """All gradients as one contiguous tensor: the engine's own flat buffer when `.grad` already aliases it
        (the normal case after UNetFunction.backward), otherwise a gathered copy.  Idempotent within a step: the
        tensor fetched first is the one `step()` consumes, so `dist.all_reduce(opt.flat_grads())` followed by
        `opt.step()` steps on the REDUCED gradient on either path (a second gather used to overwrite it with the
        local gradients).  Cleared by step() and zero_grad()."""
        if self._pending_g is not None:
            return self._pending_g
        g = self._fetch_flat_grads()
        self._pending_g = g
        return g

    def zero_grad(self, set_to_none: bool = True):
        self._pending_g = None
        return super().zero_grad(set_to_none=set_to_none)

    def _fetch_flat_grads(self) -> torch.Tensor:
        ps = self._params
        g0 = ps[0].grad
        if g0 is None:
            raise L.McedmError("FusedAdam.step() before backward()")
        base = self.grad_provider() if self.grad_provider is not None else None
        if base is not None and base.dim() == 1 and base.numel() == self._flat_p.numel() and \
                base.dtype == torch.float32 and all(p.grad is not None for p in ps):
            off, ok = 0, True
            for p in ps:
                if p.grad.data_ptr() != base.data_ptr() + 4 * off or not p.grad.is_contiguous():
                    ok = False
                    break
                off += p.numel()
            if ok:
                return base
        if self._flat_g is None or self._flat_g.device != self._flat_p.device:
            self._flat_g = torch.zeros_like(self._flat_p)
        views, srcs, off = [], [], 0
        for p in ps:
            if p.grad is not None:
                views.append(self._flat_g[off:off + p.numel()].view(p.shape))
                srcs.append(p.grad)
            else:
                self._flat_g[off:off + p.numel()].zero_()
            off += p.numel()
        torch._foreach_copy_(views, srcs)
        return self._flat_g

    def _sync_steps(self):
        """Host step counter <- the device one (synchronises; only while dynamic loss scaling has stepped)."""
        if self._step_dev is not None:
            self._steps = int(self._step_dev.item())
            self._step_t.fill_(float(self._steps))

    def state_dict(self):
        self._sync_steps()
        return super().state_dict()

    def _step_dynamic(self, scaler, p, g, grp, st):
        lib = L.lib()
        dev = p.device
        scaler.state(dev)
        if self._step_dev is None or self._step_dev.device != dev:
            self._sync_steps()
            self._step_dev = torch.full((1,), self._steps, dtype=torch.int32, device=dev)
        n = p.numel()
        clip = self.max_grad_norm is not None and self.max_grad_norm > 0
        L.check(lib.mcedm_sumsq_partial(L.ptr(g), n, L.ptr(self._partial), self._n_partial, st), "sumsq_partial")
        L.check(lib.mcedm_adam_step_dyn(L.ptr(p), L.ptr(g), L.ptr(self._m), L.ptr(self._v), n, float(grp["lr"]),
                                        float(grp["betas"][0]), float(grp["betas"][1]), float(grp["eps"]),
                                        float(grp["weight_decay"]), L.ptr(self._step_dev), L.ptr(self._partial),
                                        self._n_partial, float(self.max_grad_norm) if clip else 0.0,
                                        float(self.grad_scale), L.ptr(self.last_grad_norm), L.ptr(scaler.found_inf_t),
                                        st), "adam_step_dyn")
        scaler.update(self._step_dev, st)

    @torch.no_grad()
    def step(self, closure=None, flat_grads: Optional[torch.Tensor] = None):
        loss = closure() if closure is not None else None
        from .engine import WEIGHT_EPOCH

        lib = L.lib()
        grp = self.param_groups[0]
        p = self.flat_params()
        g = flat_grads if flat_grads is not None else self.flat_grads()
        st = L.stream_ptr()
        scaler = self.loss_scaler_provider() if self.loss_scaler_provider is not None else None
        if scaler is not None:
            self._step_dynamic(scaler, p, g, grp, st)
            self._pending_g = None
            WEIGHT_EPOCH[0] += 1
            return loss
        if self._step_dev is not None:          # dynamic loss scaling was switched off: the host counter continues
            self._sync_steps()
            self._step_dev = None
        n = p.numel()
        self._steps += 1
        clip = self.max_grad_norm is not None and self.max_grad_norm > 0
        if clip:
            L.check(lib.mcedm_sumsq_partial(L.ptr(g), n, L.ptr(self._partial), self._n_partial, st), "sumsq_partial")
        L.check(lib.mcedm_adam_step(L.ptr(p), L.ptr(g), L.ptr(self._m), L.ptr(self._v), n, float(grp["lr"]),
                                    float(grp["betas"][0]), float(grp["betas"][1]), float(grp["eps"]),
                                    float(grp["weight_decay"]), self._steps, L.ptr(self._partial) if clip else None,
                                    self._n_partial, float(self.max_grad_norm or 0.0), float(self.grad_scale),
                                    L.ptr(self.last_grad_norm), st), "adam_step")
        self._step_t.fill_(float(self._steps))
        self._pending_g = None
        WEIGHT_EPOCH[0] += 1                    # packed bf16 weights of every engine are stale now
        return loss

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        off = 0
        for p in self._params:                  # re-home the loaded moments into the flat buffers
            s = self.state[p]
            n = p.numel()
            self._m[off:off + n].view(p.shape).copy_(s["exp_avg"])
            self._v[off:off + n].view(p.shape).copy_(s["exp_avg_sq"])
            s["exp_avg"], s["exp_avg_sq"] = self._m[off:off + n].view(p.shape), self._v[off:off + n].view(p.shape)
            self._steps = int(float(s["step"]))
            s["step"] = self._step_t
            off += n
        self._step_t.fill_(float(self._steps))
        if self._step_dev is not None:
            self._step_dev.fill_(self._steps)


def ema_update_(ema_params, cur_params, beta: float, state: dict):
    """ema <- ema*beta + (1-beta)*p over all tensors with ONE launch (flat buffers are built on first use and
    re-validated every call; `state` is a dict owned by the caller)."""
    from .engine import WEIGHT_EPOCH

    lib = L.lib()
    if not _is_flat(ema_params, state.get("ema")):
        state["ema"] = _flatten_(ema_params)
    if not _is_flat(cur_params, state.get("cur")):
        # the optimizer normally flattened these already: reuse its buffer
        base = _FLAT.get(cur_params[0].data_ptr())
        ok = base is not None and base.numel() == sum(p.numel() for p in cur_params) and _is_flat(cur_params, base)
        state["cur"] = base if ok else _flatten_(cur_params)
    L.check(lib.mcedm_ema_update(L.ptr(state["ema"]), L.ptr(state["cur"]), state["ema"].numel(), float(beta),
                                 L.stream_ptr()), "ema_update")
    WEIGHT_EPOCH[0] += 1
