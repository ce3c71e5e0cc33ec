"""torch.autograd bridges of the kernel path, so `loss.backward()` in the reference's training loop
(models/mcedm.py:254-281 under a Lightning Trainer) drives the hand-written backward kernels.

  * UNetFunction     — F_x = DhariwalUNet(x_in, c_noise, cond); backward = UNetEngine.backward (train_engine.py).
                       Parameter gradients are slices of the engine's flat gradient buffer.
  * EdmLossFunction  — masked, weighted EDM loss on top of the preconditioning (mcedm.py:199-211, :237-239, :278;
                       losses.py:48-53) as ONE kernel that also emits dL/dF (K6).

Neither has a CPU path.
"""
from __future__ import annotations

import torch

from . import _lib as L


class UNetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, unet, x, noise_labels, cond, *params):
        eng = unet.engine()
        ctx.eng = eng
        ctx.n_params = len(params)
        return eng.forward_train(x, noise_labels, cond)

    @staticmethod
    def backward(ctx, dF):
        eng = ctx.eng
        eng.backward(dF)
        if eng.accumulate_grads:
            # `.grad` is bound to the window buffer directly: returned gradients would be added onto it a second time
            eng.fold_grads()
            return (None,) * (4 + ctx.n_params)
        grads = [eng.grad_of(p) if p.requires_grad else None for p in eng.unet.parameters()]
        assert len(grads) == ctx.n_params
        return (None, None, None, None, *grads)


class EdmLossFunction(torch.autograd.Function):
    """loss = mean_b sum_{chw} w_b (m*(c_skip_b x_noise + c_out_b F) - m*x)^2 ; returns (loss, D_x)."""

    @staticmethod
    def forward(ctx, F_x, x_noise, x, mask, c_skip, c_out, weight):
        lib = L.lib()
        B = F_x.shape[0]
        chw = F_x[0].numel()
        n_cta = 16
        dF = torch.empty_like(F_x)
        part = torch.empty(B, n_cta, device=F_x.device, dtype=torch.float32)
        F_x = F_x.contiguous()                       # a named tensor: L.ptr() only carries the address
        L.check(lib.mcedm_edm_loss(L.ptr(F_x), L.ptr(x_noise), L.ptr(x), L.ptr(mask), L.ptr(c_skip),
                                   L.ptr(c_out), L.ptr(weight), B, chw, L.ptr(dF), None, 0, L.ptr(part), n_cta,
                                   L.stream_ptr()), "edm_loss")
        loss = torch.empty((), device=F_x.device, dtype=torch.float32)
        L.check(lib.mcedm_reduce_rows(L.ptr(part), B * n_cta, 1, 1, 1, L.ptr(loss), 0, 1.0 / B, L.stream_ptr()),
                "reduce_rows")
        ctx.save_for_backward(dF)
        return loss

    @staticmethod
    def backward(ctx, g):
        (dF,) = ctx.saved_tensors
        return dF * g, None, None, None, None, None, None
