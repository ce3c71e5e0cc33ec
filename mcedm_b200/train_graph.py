"""CUDA-graph replay of one training step's device work (forward + loss, backward) for PlMcedm.training_step.

A training step issues ~500 kernel launches (weight re-packing, 30 convolutions and their two gradients, 35
GroupNorm passes forward and backward, attention, reductions); launched one by one from Python the step is
host-bound.  `TrainStepGraph` captures them once per batch shape into two graphs on static buffers:

    fwd graph : re-pack bf16 weights from the (in-place updated) fp32 parameters -> noise injection + c_in ->
                U-Net forward (saving the backward's operands) -> preconditioning + masked weighted loss + dL/dF
    bwd graph : UNetEngine.backward -> every parameter gradient in the engine's flat gradient buffer

`GraphedLossFunction` replays them from `loss = ...` / `loss.backward()`, so the reference's training loop
(models/mcedm.py:254-281 under a Lightning-style trainer) is unchanged.  Parameter `.grad`s are bound to slices of
the flat buffer (written, not accumulated: one backward per optimizer step, as in the reference).
"""
from __future__ import annotations

import torch

from . import _lib as L


class TrainStepGraph:
    def __init__(self, pl, B, C, H, W, cond_channels, dev):
        self.pl, self.dev = pl, dev
        f32 = dict(device=dev, dtype=torch.float32)
        self.x = torch.zeros(B, C, H, W, **f32)
        self.noise = torch.zeros(B, C, H, W, **f32)
        self.mask = torch.ones(B, C, H, W, **f32)
        self.cond = torch.zeros(B, cond_channels, H, W, **f32) if cond_channels else None
        self.sigma = torch.ones(B, **f32)
        self.weight = torch.ones(B, **f32)
        self.x_noise = torch.empty(B, C, H, W, **f32)
        self.x_in = torch.empty(B, C, H, W, **f32)
        self.dF = torch.empty(B, C, H, W, **f32)
        self.n_cta = 16
        self.part = torch.empty(B, self.n_cta, **f32)
        self.loss = torch.zeros((), **f32)
        self.coef = torch.empty(4, B, **f32)          # c_skip | c_out | c_in | c_noise
        self.g_fwd = self.g_bwd = None
        self.launches = (0, 0)

    # -- the device work of one step (no allocation after the first call, no host sync) ------------------------
    def _fwd(self):
        pl, lib, st = self.pl, L.lib(), L.stream_ptr()
        eng = pl.model.engine()
        eng.pack_fused()                   # every operand copy of the parameters: one gather launch (pack_plan.py)
        B = self.x.shape[0]
        chw = self.x[0].numel()
        s = self.sigma
        den = s * s + pl.sigma_data ** 2
        torch.div(pl.sigma_data ** 2, den, out=self.coef[0])
        torch.div(s * pl.sigma_data, den.sqrt(), out=self.coef[1])
        torch.div(1.0, den.sqrt(), out=self.coef[2])
        torch.div(s.log(), 4.0, out=self.coef[3])
        L.check(lib.mcedm_edm_noise_in(L.ptr(self.x), L.ptr(self.noise), L.ptr(self.mask), L.ptr(s), L.ptr(self.coef[2]),
                                       B, chw, L.ptr(self.x_noise), L.ptr(self.x_in), st), "edm_noise_in")
        F_x = eng.forward_train(self.x_in, self.coef[3], self.cond)
        L.check(lib.mcedm_edm_loss(L.ptr(F_x), L.ptr(self.x_noise), L.ptr(self.x), L.ptr(self.mask), L.ptr(self.coef[0]),
                                   L.ptr(self.coef[1]), L.ptr(self.weight), B, chw, L.ptr(self.dF), None, 0,
                                   L.ptr(self.part), self.n_cta, st), "edm_loss")
        L.check(lib.mcedm_reduce_rows(L.ptr(self.part), B * self.n_cta, 1, 1, 1, L.ptr(self.loss), 0, 1.0 / B, st),
                "reduce_rows")

    def _bwd(self):
        self.pl.model.engine().backward(self.dF)

    def capture(self):
        eng = self.pl.model.engine()
        step = eng.dropout_step
        with torch.no_grad():
            self._fwd()                      # eager warm-up: allocates workspaces, sets kernel attributes
            self._bwd()
            eng.dropout_step = step          # the warm-up is not a training step: it draws no dropout masks of its own
            torch.cuda.current_stream().synchronize()
            n0 = L.LAUNCHES[0]
            self.g_fwd = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.g_fwd):
                self._fwd()
            n1 = L.LAUNCHES[0]
            self.g_bwd = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.g_bwd, pool=self.g_fwd.pool()):
                self._bwd()
            self.launches = (n1 - n0, L.LAUNCHES[0] - n1)

    def load(self, x, sigma, noise, cond, mask, weight):
        self.x.copy_(x)
        self.noise.copy_(noise)
        if mask is None:
            self.mask.fill_(1.0)
        else:
            self.mask.copy_(mask)
        if self.cond is not None:
            if cond is None:
                self.cond.zero_()
            else:
                self.cond.copy_(cond)
        self.sigma.copy_(sigma.reshape(-1))
        self.weight.copy_(weight.reshape(-1))
        eng = self.pl.model.engine()
        if eng.dropout_p() > 0:
            eng.dropout_fill(self.dev)       # {seed, step} of the next replay (GraphedLossFunction advances the step)


class GraphedLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tg, trigger):
        tg.g_fwd.replay()
        L.LAUNCHES[0] += tg.launches[0]
        eng = tg.pl.model.engine()
        if eng.dropout_p() > 0:
            eng.dropout_step += 1
        ctx.tg = tg
        return tg.loss.clone()

    @staticmethod
    def backward(ctx, g):
        tg = ctx.tg
        tg.g_bwd.replay()
        L.LAUNCHES[0] += tg.launches[1]
        eng = tg.pl.model.engine()
        flat = eng.flat_grad()
        flat.mul_(g)                          # dL/dloss (1 under a plain loss.backward())
        for p in eng.unet.parameters():
            if p.requires_grad:
                p.grad = eng.grad_of(p)
        return None, None
