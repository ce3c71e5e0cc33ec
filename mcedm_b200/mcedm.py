"""Drop-in host mirror of the reference Lightning module `models.mcedm.PlMcedm`.

Same constructor (`PlMcedm(hparams)`), same public methods with the same argument meaning and the
same return layouts as the reference (all file:line citations are models/mcedm.py):

    model_precond(x_noise, sigma, cond, ...)                       :199-211
    forward(x, sigma, noise, cond=None, mask=None)                 :213-235
    get_loss_weight / get_cond_in                                  :237-252
    training_step / validation_step / test_step                    :254-441
    get_denoised(model, xt, t, cond, ..., w) -> (D_x, F_x)          :443-461
    sample_edm(hu, cond, hu_mask, sparams, return_last, guide_dx)   :570-638   -> xs[b,t,h,w,c] float64
    configure_optimizers / optimizer_step (EMA) / setup            :128-168

and the same state_dict keys (`model.*`, `ema_model.ma_model.*`, `normalizer_{input,target}.*`).
The arithmetic of the hot path runs in hand-written sm_100a kernels (include/mcedm_b200.h):

  * network evaluation           -> DhariwalUNet.forward (engine.py; K1 conv, K2 GroupNorm, K3 attention)
  * preconditioning              -> mcedm_edm_precond_in / _out (K4)
  * Heun / churn / mask blending -> mcedm_edm_init / _churn / _euler / _correct (K5), fp64 state
  * classifier-free guidance     -> `sparams.w` / get_denoised's `w` with |w| >= 1e-3 and a condition (the gate of
    :453-458): one network evaluation of 2B rows, rows [B, 2B) with the all-zero condition (what the training step's
    condition drop feeds), combined as F_w = (1+w)*F_c - w*F_u in fp32 by mcedm_edm_*_cfg (K4/K5); the sampler
    updates use D_w = c_skip*x + c_out*F_w, while mask blending and the known values still come from `cond`

What is not mirrored: `dx_cond` (rejected in __init__), self-conditioning, the PDE guidance of this module's sampler
(`guide_dx` raises, as :501-517 does in the reference), and guided get_denoised under autograd in train mode (raises
NotImplementedError; the reference only calls it from no_grad sampling).

Host-side differences that do not change results: the sigma schedule, gamma and the per-step fp32
preconditioning scalars are computed on the host (the reference computes them on the device and
synchronises once per step at :606); the disabled guidance branches (:611, :615) are not evaluated.
Random numbers are drawn with the same torch calls, dtypes, shapes and order as the reference
(:576 one fp32 randn_like, :608 one fp64 randn_like per step), so a given seed and device yields the
same noise in both code bases.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch
from einops import rearrange

from . import _lib as L
from .adm_blocks import DhariwalUNet
from .config import AttrDict
from .loss_scale import active_scaler
from .nn_misc import EmaModel, MaskedLoss, NoiseEstimationLoss, Normalizer, fused_masked_mae
from .pde_loss import DarcyLoss, get_pde_loss_function
from .runner import LightningModule


def _f32(x) -> np.float32:
    return np.float32(x)


def guidance_weight(w, cond) -> Optional[float]:
    """The classifier-free-guidance weight to sample with, or None when guidance is off.  Guidance is on under the gate
    of get_denoised (:453-458): w is not None, |w| >= 1e-3 and there is a condition to drop.  A non-finite w raises
    ValueError.  Guided, the network output is F_w = (1+w)*F_c - w*F_u (F_c with cond, F_u with the all-zero
    condition), evaluated in fp32 by the mcedm_edm_*_cfg kernels on one network batch of 2B rows."""
    if w is None:
        return None
    w = float(w)
    if not math.isfinite(w):
        raise ValueError(f"the guidance weight w must be finite, got {w}")
    return w if abs(w) >= 1e-3 and cond is not None else None


def _dropout_active(unet) -> bool:
    """True for a network in training mode with dropout > 0: only its training forward applies the masks."""
    return bool(unet.training and getattr(unet, "dropout", 0.0))


def precond_scalars(sigma: float):
    """fp32 (c_skip, c_out, c_in, c_noise) of one sigma with sigma_data = 1, evaluated with the same
    sequence of fp32 operations as :203-206 / :448-451 (IEEE mul, add, sqrt, div; log)."""
    s = _f32(sigma)
    den = _f32(_f32(s * s) + _f32(1.0))
    root = np.sqrt(den, dtype=np.float32)
    c_skip = _f32(_f32(1.0) / den)
    c_out = _f32(s / root)
    c_in = _f32(_f32(1.0) / root)
    c_noise = _f32(np.log(s, dtype=np.float32) / _f32(4.0))
    return float(c_skip), float(c_out), float(c_in), float(c_noise)


class PlMcedm(LightningModule):
    def __init__(self, hparams):
        super().__init__()
        self.save_hyperparameters()
        self.cond_p = 1.0
        m = hparams.model
        self.dx_norm = m.dx_norm if hasattr(m, "dx_norm") else "l2"
        self.dx_detach = m.dx_detach if hasattr(m, "dx_detach") else False
        self.dx_cond = m.dx_cond if hasattr(m, "dx_cond") else False
        self.add_cond_mask = m.add_cond_mask if hasattr(m, "add_cond_mask") else False
        self.add_xt = m.add_xt if hasattr(m, "add_xt") else False
        if self.add_cond_mask:
            m.cond_channels = m.cond_channels + m.in_channels      # :28-30
        if self.add_xt:
            m.cond_channels = m.cond_channels + 2                  # :32-34
        if self.dx_cond:
            raise NotImplementedError("dx_cond (PDE-gradient conditioning) has no sm_100a kernel yet (SURVEY §8f)")
        if hparams.name.startswith("adm"):                            # :36-39
            self.model = DhariwalUNet(hparams)
        else:
            from .ddpm_blocks import Model

            self.model = Model(hparams)
        self.ema_model = EmaModel(self.model, beta=m.ema_rate) if m.ema else None

        # EDM constants (:45-50)
        self.P_mean, self.P_std, self.sigma_data = -1.2, 1.2, 1.0
        self.sigma_min, self.sigma_max = 0.002, 80

        d = hparams.data
        self.normalization = d.normalization
        self.uniform_dequantization = d.uniform_dequantization
        self.gaussian_dequantization = d.gaussian_dequantization
        self.rescaled = d.rescaled
        self.normalizer_input = Normalizer(stats_shape=self.get_inp_stats_shape(hparams))
        self.normalizer_target = Normalizer(stats_shape=self.get_tar_stats_shape(hparams))

        o = hparams.optimization
        self.optimizer, self.lr, self.weight_decay = o.optimizer, o.lr, o.weight_decay
        self.beta1, self.amsgrad, self.eps = o.beta1, o.amsgrad, o.eps
        self.factor, self.step_size, self.loss = o.factor, o.step_size, o.loss
        self.pde_loss_lambda = o.pde_loss_lambda if hasattr(o, "pde_loss_lambda") else 0.0
        self.pde_loss_prop_t = o.pde_loss_prop_t if hasattr(o, "pde_loss_prop_t") else False
        self.use_gt_pde = o.use_gt_pde if hasattr(o, "use_gt_pde") else False

        self.criteria = NoiseEstimationLoss()
        self.mae_criterion = MaskedLoss()
        # PDE residual metric / guidance term on the K6 kernels (overridden by set_pde_loss_function, :82-84)
        self.pde_loss, self.pde_loss_simulator = get_pde_loss_function(system="swe", flip_xy=False)

        self.sparams = self.get_sampler_params(hparams)
        self.test_sparams = self.sparams
        self.h_ch = self.u_ch = m.out_ch // 2 if m.out_ch > 1 else 1
        self.use_cuda_graph = True   # replay the captured U-Net launch sequence inside sample_edm
        self.fused_prep = True       # training_step: normalise + cond_in + rearranges in one kernel (mcedm_mcedm_prep)
        self._noise_hook = None      # tests inject pre-drawn noise here: fn(kind, like) -> tensor
        self._trace = None           # tests: list receiving (step, which, sigma, D_x, x_t)

    # ---------------------------------------------------------------- configuration helpers
    def get_inp_stats_shape(self, hparams):
        ch = hparams.model.out_ch // 2
        return (ch,) if ch > 1 else ()

    def get_tar_stats_shape(self, hparams):
        ch = hparams.model.out_ch // 2
        return (ch,) if ch > 1 else ()

    def set_pde_loss_function(self, system, flip_xy):                 # :100-104
        self.pde_loss, self.pde_loss_simulator = get_pde_loss_function(system, flip_xy)

    @staticmethod
    def get_sampler_params(params):
        if params.get("sampler", None) is None:
            return AttrDict(type="ddim", timesteps=50, skip_type="uniform", eta=0.0, n_samples=1, n_repeat=5,
                            n_time_h=128, n_time_u=0)
        return params.sampler

    def set_test_sampler_params(self, params):
        self.test_sparams = params

    def setup(self, stage: Optional[str] = None) -> None:
        if stage == "fit":
            stats = self.trainer.datamodule.get_norm_stats()
            if self.normalization == "min_max":
                self.normalizer_input.set_stats(stats["input_min"], stats["input_min_max"])
                self.normalizer_target.set_stats(stats["target_min"], stats["target_min_max"])
            else:
                self.normalizer_input.set_stats(stats["input_mean"], stats["input_std"])
                self.normalizer_target.set_stats(stats["target_mean"], stats["target_std"])

    def configure_optimizers(self):
        params = self.model.parameters()
        if self.optimizer == "Adam":
            from .optim import FusedAdam

            # torch.optim.Adam's arguments and state_dict layout, one fused clip+Adam kernel over a flat buffer
            opt = FusedAdam(params, lr=self.lr, weight_decay=self.weight_decay, betas=(self.beta1, 0.999),
                            amsgrad=self.amsgrad, eps=self.eps)
            opt.grad_provider = lambda: self.model.engine().flat_grad()
            opt.loss_scaler_provider = lambda: active_scaler(self.model)
        elif self.optimizer == "RMSProp":
            opt = torch.optim.RMSprop(params, lr=self.lr, weight_decay=self.weight_decay)
        elif self.optimizer == "SGD":
            opt = torch.optim.SGD(params, lr=self.lr, momentum=0.9)
        else:
            raise NotImplementedError("Optimizer {} not understood.".format(self.optimizer))
        return {"optimizer": opt}

    def optimizer_step(self, *args, **kwargs):
        super().optimizer_step(*args, **kwargs)
        if self.ema_model is not None:                              # :166-168
            self.ema_model.update(self.model)

    # ---------------------------------------------------------------- data transforms (host glue)
    def data_transform(self, h, u):
        x = torch.cat([self.normalizer_input(h), self.normalizer_target(u)], dim=-1)
        if self.uniform_dequantization:
            x = x / 256.0 * 255.0 + torch.rand_like(x) / 256.0
        if self.gaussian_dequantization:
            x = x + torch.randn_like(x) * 0.01
        if self.rescaled:
            x = 2 * x - 1.0
        return x

    def inverse_data_transform(self, h, u):
        if self.rescaled:
            h, u = (h + 1.0) / 2.0, (u + 1.0) / 2.0
        if self.normalization == "min_max":
            h, u = torch.clamp(h, 0.0, 1.0), torch.clamp(u, 0.0, 1.0)
        return self.normalizer_input(h, inverse=True), self.normalizer_target(u, inverse=True)

    def get_loss_weight(self, sigma):
        return (sigma ** 2 + self.sigma_data ** 2) / (sigma * self.sigma_data) ** 2

    def get_cond_in(self, x, mask, dx, dt):
        if self.add_cond_mask:
            cond_in = torch.cat([x * (1 - mask), (1.0 - mask)], dim=-1)
        else:
            cond_in = x * (1 - mask) + self._randn_like("cond", x) * mask
        if self.add_xt:
            cond_in = torch.cat([cond_in, dx, dt], dim=-1)
        return cond_in

    def _randn_like(self, kind, like):
        if self._noise_hook is not None:
            return self._noise_hook(kind, like)
        return torch.randn_like(like)

    # ---------------------------------------------------------------- network + preconditioning
    @staticmethod
    def _unet_of(model):
        return model.ma_model if isinstance(model, EmaModel) else model

    def _precond_apply(self, model, x, sigma, cond, w=None):
        """(D_x, F_x) for per-sample or scalar sigma; x fp32 NCHW on the GPU.  With a guidance weight w (see
        guidance_weight; cond not None) the network runs once on 2B rows, [x_in | x_in] with [cond | 0], and the pair
        returned is (D_w, F_w)."""
        lib = L.lib()
        unet = self._unet_of(model)
        B = x.shape[0]
        chw = x[0].numel()
        sigma = sigma.to(torch.float32).reshape(-1)
        den = sigma ** 2 + self.sigma_data ** 2
        c_skip = (self.sigma_data ** 2 / den).contiguous()
        c_out = (sigma * self.sigma_data / den.sqrt()).contiguous()
        c_in = (1 / den.sqrt()).contiguous()
        c_noise = (sigma.log() / 4).contiguous()
        stride = 1 if sigma.numel() == B and B > 1 else 0
        if sigma.numel() not in (1, B):
            raise ValueError(f"sigma must have 1 or {B} entries")
        st = L.stream_ptr()
        x = x.contiguous()
        x_in = torch.empty_like(x) if w is None else x.new_empty((2 * B,) + tuple(x.shape[1:]))
        L.check(lib.mcedm_edm_precond_in(L.ptr(x), L.ptr(c_in), stride, B, chw, L.ptr(x_in), st), "precond_in")
        if w is not None:
            x_in[B:].copy_(x_in[:B])
            cond = cond.to(torch.float32)
            F2 = unet(x_in, c_noise.repeat(2) if stride else c_noise, torch.cat([cond, torch.zeros_like(cond)]))
            if F2.shape[1:] != x.shape[1:]:
                raise ValueError("classifier-free guidance needs a network output shaped like its input")
            D_x, F_x = torch.empty_like(x), torch.empty_like(x)
            L.check(lib.mcedm_edm_precond_out_cfg(L.ptr(x), L.ptr(F2), L.ptr(c_skip), L.ptr(c_out), stride, w, B, chw,
                                                  L.ptr(D_x), L.ptr(F_x), st), "precond_out_cfg")
            return D_x, F_x
        F_x = unet(x_in, c_noise, cond)
        D_x = torch.empty_like(x)
        L.check(lib.mcedm_edm_precond_out(L.ptr(x), L.ptr(F_x), L.ptr(c_skip), L.ptr(c_out), stride, B, chw,
                                          L.ptr(D_x), st), "precond_out")
        return D_x, F_x

    def model_precond(self, x_noise, sigma, cond=None, x_self_cond=None, dx=None):
        if x_self_cond is not None or dx is not None:
            raise NotImplementedError("self-conditioning / dx conditioning are not supported")
        return self._precond_apply(self.model, x_noise, sigma, cond)[0]

    def forward(self, x, sigma, noise, cond=None, mask=None):
        x_noise = x + mask * noise * sigma if mask is not None else x + noise * sigma
        if torch.rand(1) >= self.cond_p:                            # :231, host RNG draw kept for RNG parity
            cond = None
        return self.model_precond(x_noise, sigma.float(), cond, x_self_cond=None, dx=None)

    def forward_loss(self, x, sigma, noise, cond, mask, weight):
        """Fused equivalent of `criteria(forward(x, sigma, noise, cond, mask) * mask, x * mask, weight)`
        (mcedm.py:213-235, :278; losses.py:48-53), differentiable w.r.t. the U-Net parameters."""
        from .autograd import EdmLossFunction

        lib = L.lib()
        if torch.rand(1) >= self.cond_p:                            # :231, host RNG draw kept for RNG parity
            cond = None
        B = x.shape[0]
        chw = x[0].numel()
        s = sigma.to(torch.float32).reshape(-1)
        if s.numel() != B:
            raise ValueError(f"sigma must have {B} entries")
        if self.use_cuda_graph and self.model.training and torch.is_grad_enabled():
            return self._graphed_loss(x, s, noise, cond, mask, weight)
        den = s ** 2 + self.sigma_data ** 2
        c_skip = (self.sigma_data ** 2 / den).contiguous()
        c_out = (s * self.sigma_data / den.sqrt()).contiguous()
        c_in = (1 / den.sqrt()).contiguous()
        c_noise = (s.log() / 4).contiguous()
        w = weight.to(torch.float32).reshape(-1).contiguous()
        x = x.contiguous()
        x_noise, x_in = torch.empty_like(x), torch.empty_like(x)
        noise, s = noise.contiguous(), s.contiguous()   # named tensors: L.ptr() only carries the address
        L.check(lib.mcedm_edm_noise_in(L.ptr(x), L.ptr(noise), L.ptr(mask), L.ptr(s),
                                       L.ptr(c_in), B, chw, L.ptr(x_noise), L.ptr(x_in), L.stream_ptr()), "edm_noise_in")
        F_x = self.model(x_in, c_noise, cond)
        return EdmLossFunction.apply(F_x, x_noise, x, mask, c_skip, c_out, w)

    def _graphed_loss(self, x, s, noise, cond, mask, weight):
        """The same three nodes replayed from two CUDA graphs on static buffers (train_graph.py)."""
        from .train_graph import GraphedLossFunction, TrainStepGraph

        unet = self.model
        params = list(unet.parameters())
        # the backward graph captures the loss-scaling mode and the scaler's device words
        key = (tuple(x.shape), x.device.index, params[0].data_ptr(), params[-1].data_ptr(), active_scaler(unet))
        graphs = self.__dict__.setdefault("_train_graphs", {})
        tg = graphs.get(key)
        if tg is None:
            if len(graphs) > 4:
                graphs.clear()
            tg = TrainStepGraph(self, x.shape[0], x.shape[1], x.shape[2], x.shape[3], unet.cat_channels, x.device)
            tg.load(x, s, noise, cond, mask, weight)
            tg.capture()
            graphs[key] = tg
            self.__dict__["_train_trigger"] = torch.zeros((), device=x.device, requires_grad=True)
        tg.load(x, s, noise, cond, mask, weight)
        return GraphedLossFunction.apply(tg, self.__dict__["_train_trigger"])

    def get_denoised(self, model, xt, t, cond=None, x_self_cond=None, dx=None, w=None):
        if x_self_cond is not None or dx is not None:
            raise NotImplementedError("self-conditioning / dx conditioning are not supported")
        w = guidance_weight(w, cond)
        if w is not None and torch.is_grad_enabled() and self._unet_of(model).training:
            # the reference only calls get_denoised from no_grad sampling; the guided pair has no backward here
            raise NotImplementedError("classifier-free guidance (w != 0) runs on the inference path only (no_grad or "
                                      "eval mode)")
        if w is not None and _dropout_active(self._unet_of(model)):
            raise NotImplementedError("classifier-free guidance runs on the inference path, which has no dropout: put "
                                      "the module in eval mode")
        t = torch.as_tensor(t, device=xt.device)
        return self._precond_apply(model, xt.to(torch.float32), t, cond, w)

    def round_sigma(self, sigma, return_index=False):
        return 0 if return_index else torch.as_tensor(sigma)

    # ---------------------------------------------------------------- training / evaluation steps
    def _prep_batch(self, h_unnorm, u_unnorm, mask):
        """(x, cond_in, mask) as `b c h w` fp32 from the datamodule's `b h w c` tensors: data_transform (:257), get_cond_in
        (:259, incl. its randn_like draw) and the three rearranges (:263-265) in one kernel (mcedm_mcedm_prep,
        bit-identical to the torch expressions).  Returns None when an option the kernel does not cover is on."""
        if not (self.fused_prep and h_unnorm.is_cuda and h_unnorm.shape[-1] == 1 and u_unnorm.shape[-1] == 1
                and self.normalization != "min_max" and not (self.uniform_dequantization or self.gaussian_dequantization
                                                             or self.rescaled or self.add_cond_mask or self.add_xt)
                and h_unnorm.dtype == torch.float32 and (mask.dtype == torch.float32 or mask.dim() == 2)):
            if mask.dim() == 2:
                raise NotImplementedError("observation-row masks (device_masks datamodule) need the fused batch "
                                          "preparation: fp32 CUDA inputs, gauss normalisation, no dequantisation")
            return None
        from .pde_loss import _norm_args

        h_div, h_sub, u_div, u_sub = _norm_args(self.normalizer_input, self.normalizer_target)
        B, H, W, _ = h_unnorm.shape
        h, u = h_unnorm.contiguous(), u_unnorm.contiguous()
        x = torch.empty(B, 2, H, W, device=h.device, dtype=torch.float32)
        cond, mask_c = torch.empty_like(x), torch.empty_like(x)
        if mask.dim() == 2:
            # [B, 2] int32 observation rows from a `device_masks` datamodule: the mask is expanded inside the kernel
            rows = mask.to(device=h.device, dtype=torch.int32).contiguous()
            r = self._randn_like("cond", torch.empty(B, H, W, 2, device=h.device, dtype=torch.float32)).contiguous()
            L.check(L.lib().mcedm_mcedm_prep_rows(L.ptr(h), L.ptr(u), L.ptr(rows), L.ptr(r), h_sub, h_div, u_sub, u_div,
                                                  B, H, W, L.ptr(x), L.ptr(cond), L.ptr(mask_c), None, L.stream_ptr()),
                    "mcedm_prep_rows")
            return x, cond, mask_c
        m = mask.contiguous()
        r = self._randn_like("cond", m).contiguous()                 # the draw of get_cond_in (:247): b h w c, fp32
        L.check(L.lib().mcedm_mcedm_prep(L.ptr(h), L.ptr(u), L.ptr(m), L.ptr(r), h_sub, h_div, u_sub, u_div, B, H * W,
                                         L.ptr(x), L.ptr(cond), L.ptr(mask_c), L.stream_ptr()), "mcedm_prep")
        return x, cond, mask_c

    def training_step(self, train_batch, batch_idx):
        h_unnorm, dx, dt, u_unnorm, mask = train_batch
        self.h_ch, self.u_ch = h_unnorm.shape[-1], u_unnorm.shape[-1]
        prep = self._prep_batch(h_unnorm, u_unnorm, mask)
        if prep is not None:
            x, cond_in, mask_pre = prep
        else:
            x = self.data_transform(h_unnorm, u_unnorm)                 # b h w c
            cond_in = rearrange(self.get_cond_in(x, mask, dx, dt), "b h w c -> b c h w").contiguous()
            x = rearrange(x, "b h w c -> b c h w").contiguous()
            mask_pre = None
        noise = self._randn_like("noise", x)
        rnd_normal = torch.randn([x.shape[0], 1, 1, 1]).type_as(x)  # CPU RNG, as :269-270
        sigma = (rnd_normal * self.P_std + self.P_mean).exp()
        weight = self.get_loss_weight(sigma)
        mask_c = mask_pre if mask_pre is not None else rearrange(mask, "b h w c -> b c h w").contiguous()
        # reference: D_x = self.forward(...); loss = self.criteria(D_x * mask, x * mask, weight)  (:277-278).
        # Here noise injection + c_in scaling, the U-Net, and preconditioning + masked weighted loss (+ dL/dF) are
        # three fused launches/nodes; `loss.backward()` runs the backward kernels.
        loss = self.forward_loss(x, sigma, noise, cond_in, mask_c, weight)
        self.log("train_loss", loss, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        return loss

    def validation_step(self, val_batch, batch_idx):
        if (self.current_epoch + 1) % 100 != 0 and self.current_epoch != 0:
            return {"epoch": self.current_epoch}
        h_unnorm, dx, dt, u_unnorm, masks = val_batch
        self.h_ch = h_ch = h_unnorm.shape[-1]
        self.u_ch = u_ch = u_unnorm.shape[-1]
        state_gt = self.data_transform(h_unnorm, u_unnorm)
        state_gt_c = rearrange(state_gt, "b h w c -> b c h w")
        noise = self._randn_like("val_noise", state_gt_c)
        result_dict = {"epoch": self.current_epoch}
        for name, mask in masks.items():
            cond_in = rearrange(self.get_cond_in(state_gt, mask, dx, dt), "b h w c -> b c h w").contiguous()
            mask_c = rearrange(mask, "b h w c -> b c h w").contiguous()
            if self.sparams.type != "edm":
                raise TypeError("Non EDM sampler is not supported for the model")
            xs = self.sample_edm(noise, cond_in, mask_c, self.sparams, return_last=True,
                                 guide_dx=self.sparams.guide_dx)
            fm = self._fused_mae(xs[:, -1], 1, state_gt, h_unnorm, u_unnorm, mask, 0, h_ch + u_ch)
            if fm is not None:                                        # one kernel pass (csrc/metrics.cu), :309-320
                loss_hu, loss_hu_un = fm
            else:
                hu_last = xs[:, -1]
                loss_hu = self.mae_criterion(hu_last, state_gt, mask)
                h_last, u_last = xs[:, -1, :, :, 0:h_ch], xs[:, -1, :, :, h_ch:u_ch + h_ch]
                h_un, u_un = self.inverse_data_transform(h_last, u_last)
                loss_hu_un = self.mae_criterion(torch.cat([h_un, u_un], dim=-1),
                                                torch.cat([h_unnorm, u_unnorm], dim=-1), mask)
            self.log(f"val_mae_{name}", loss_hu, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
            self.log(f"val_mae_{name}_un", loss_hu_un, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
            pde_loss = self.get_pde_loss(xs[:, -1], clamp_loss=False, do_rearrange=False) / len(h_unnorm)   # :325-328
            self.log(f"val_pde_loss_{name}", pde_loss, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
            result_dict[f"loss_{name}"] = loss_hu
            result_dict[f"loss_{name}_un"] = loss_hu_un
            result_dict[f"traj_{name}"] = xs[:, -1].unsqueeze(dim=1)
            result_dict[f"gt_{name}"] = state_gt
        return result_dict

    def test_step(self, test_batch, test_idx):
        h_unnorm, dx, dt, u_unnorm, masks = test_batch
        self.h_ch = h_ch = h_unnorm.shape[-1]
        self.u_ch = u_ch = u_unnorm.shape[-1]
        dm = getattr(self.trainer, "datamodule", None) if self.trainer is not None else None
        down_factor = dm.down_factor if dm is not None and getattr(dm, "down_interp", False) else 1
        state_gt = self.data_transform(h_unnorm, u_unnorm)
        state_gt_c = rearrange(state_gt, "b h w c -> b c h w")
        n_samples = self.test_sparams.n_samples
        return_last = self.test_sparams.return_last
        guide_dx = self.test_sparams.guide_dx
        state_gt_rep = state_gt_c.repeat(n_samples, 1, 1, 1)
        result_dict = {}
        for name, mask in masks.items():
            start = 0 if name.startswith("h") else h_ch
            end = h_ch if name.startswith("h") else h_ch + u_ch
            loss_dim = torch.arange(start, end, 1).long()
            cond_in = rearrange(self.get_cond_in(state_gt, mask, dx, dt), "b h w c -> b c h w")
            cond_in_rep = cond_in.repeat(n_samples, 1, 1, 1).contiguous()
            noise = self._randn_like("test_noise", state_gt_rep)    # unused draw kept for RNG parity (:373)
            mask_c_rep = rearrange(mask, "b h w c -> b c h w").repeat(n_samples, 1, 1, 1).contiguous()
            if self.test_sparams.type != "edm":
                raise TypeError("Non EDM sampler is not supported for the model")
            xs = self.sample_edm(noise, cond_in_rep, mask_c_rep, self.test_sparams, return_last=return_last,
                                 guide_dx=guide_dx)
            if down_factor > 1:
                each_x = 2 ** (down_factor - 1)
                mask_down = torch.zeros_like(mask)
                mask_down[:, ::each_x, ::each_x] = 1.0
                mask_loss = mask * mask_down
            else:
                mask_loss = mask
            # mean over n_samples (:385-386) + both masked errors (:398-408) in one kernel pass over the fp64 fields
            fm = self._fused_mae(xs[:, -1], n_samples, state_gt, h_unnorm, u_unnorm, mask_loss, start, end)
            if fm is not None:
                loss_hu, loss_hu_un = fm
            else:
                xs_mean = torch.mean(rearrange(xs, "(n b) t h w c -> n b t h w c", n=n_samples), dim=0)
                hu_last = xs_mean[:, -1]
                loss_hu = self.mae_criterion(hu_last, state_gt, mask_loss, loss_dim)
                h_un, u_un = self.inverse_data_transform(xs_mean[:, -1, :, :, 0:h_ch],
                                                         xs_mean[:, -1, :, :, h_ch:u_ch + h_ch])
                loss_hu_un = self.mae_criterion(torch.cat([h_un, u_un], dim=-1),
                                                torch.cat([h_unnorm, u_unnorm], dim=-1), mask_loss, loss_dim)
            self.log(f"test_mae_{name}", loss_hu, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
            self.log(f"test_mae_{name}_un", loss_hu_un, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
            # PDE residual of every prediction, then of the ground truth (:416-428)
            n_batch = len(h_unnorm)
            pde_loss = self.get_pde_loss(xs[:, -1], clamp_loss=False, do_rearrange=False) / n_samples / n_batch
            self.log(f"test_pde_loss_{name}", pde_loss, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
            pde_loss_gt = self.get_pde_loss(state_gt, clamp_loss=False, do_rearrange=False) / n_batch
            self.log("test_pde_loss_gt", pde_loss_gt, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
            result_dict[f"loss_{name}"] = loss_hu
            result_dict[f"loss_{name}_un"] = loss_hu_un
            if n_samples < 15:
                result_dict[f"traj_{name}"] = rearrange(xs[:, -1], "(n b) h w c -> b h w n c",
                                                        n=n_samples).unsqueeze(dim=1)
                result_dict[f"gt_{name}"] = state_gt
        return result_dict

    def _fused_mae(self, xs_last, n_samples, state_gt, h_unnorm, u_unnorm, mask, c0, c1):
        """(masked MAE, masked MAE un-normalised) of the sample mean through csrc/metrics.cu, or None when an option the
        kernel does not cover is on (`rescaled`: the inverse transform is not the plain x*divide + subtract)."""
        if self.rescaled or not getattr(self, "fused_metrics", True):
            return None
        return fused_masked_mae(xs_last, n_samples, state_gt, h_unnorm, u_unnorm, mask, c0, c1, self.normalizer_input,
                                self.normalizer_target, clamp01=self.normalization == "min_max")

    # ---------------------------------------------------------------- PDE residual (K6) and guidance
    def _pde_planes(self, h, u):
        """The two [B,T,X] channel planes for the fused kernel: normalised planes + apply_norm=True when the inverse
        transform is the plain `x*divide + subtract` (normalization 'gauss', not rescaled), otherwise the host-side
        inverse transform (clamp / rescale, :186-197) and apply_norm=False."""
        if self.rescaled or self.normalization == "min_max":
            h, u = self.inverse_data_transform(h.to(torch.float32), u.to(torch.float32))
            return h, u, False
        return h, u, True

    def _pde_residual(self, h, u, x_gt_unnorm, noise_level, clamp_loss, reduce, sum_channels=False):
        h, u, apply_norm = self._pde_planes(h, u)
        fast = reduce and not clamp_loss and noise_level is None
        if isinstance(self.pde_loss, DarcyLoss):
            m, total = self.pde_loss.residual(h, u, self.normalizer_input, self.normalizer_target,
                                              apply_norm=apply_norm, want_matrix=not fast)
        else:
            m, total = self.pde_loss.residual(h, u, self.normalizer_input, self.normalizer_target, gt=x_gt_unnorm,
                                              apply_norm=apply_norm, want_matrix=not fast)
        if fast:
            return total.to(torch.float32)
        if clamp_loss:
            m = torch.clamp(m, max=1.0)
        if sum_channels and m.dim() > 3:
            m = torch.sum(m, dim=-1)                                 # ddim.py:1408-1411
        if noise_level is not None:
            m = m / (noise_level.reshape(-1, 1, 1, 1) + 1.0)
        return torch.sum(m) if reduce else m

    def get_pde_loss(self, x_denoised, x_gt_unnorm=None, noise_level=None, clamp_loss=True, do_rearrange=True,
                     reduce=True):
        """:468-499. x_denoised: normalised (h, u) sample, `b c h w` (do_rearrange) or `b h w c`, any float dtype."""
        if do_rearrange:
            x_denoised = rearrange(x_denoised, "b c h w -> b h w c")
        if self.h_ch != 1 or self.u_ch != 1:
            raise NotImplementedError("the PDE residual kernels take one h and one u channel")
        return self._pde_residual(x_denoised[..., 0], x_denoised[..., 1], x_gt_unnorm, noise_level, clamp_loss, reduce)

    def get_dx_pde(self, cond, x_denoised, calc_prob=False):
        # :501-517 slices the LAST axis of a `b c h w` tensor into "h" and "u" and then fails inside
        # SweFvLoss.calculate_loss (torch.cat of 4- and 2-channel tensors): the reference raises RuntimeError here.
        raise NotImplementedError("PlMcedm.get_dx_pde is not runnable in the reference either (models/mcedm.py:504: "
                                  "channel slices taken on the width axis); PDE guidance is implemented for PlCondEdm")

    def get_dx_input(self, cond, x_denoised):                         # :519-557 (dx_cond is rejected in __init__)
        return None

    def get_dx_log_prob(self, cond, x_denoised, guide_dx):            # :559-568
        if guide_dx:
            return self.get_dx_pde(cond, x_denoised, calc_prob=True)
        return torch.zeros_like(x_denoised)

    # ---------------------------------------------------------------- sampler
    def edm_time_steps(self, sparams):
        """fp64 rho-schedule with t_N = 0 (:579-588), evaluated once on the host with torch."""
        sigma_min = max(sparams.sigma_min, self.sigma_min)
        sigma_max = min(sparams.sigma_max, self.sigma_max)
        n = sparams.timesteps
        i = torch.arange(n, dtype=torch.float64)
        t = (sigma_max ** (1 / sparams.rho) + i / (n - 1) * (sigma_min ** (1 / sparams.rho)
                                                            - sigma_max ** (1 / sparams.rho))) ** sparams.rho
        return torch.cat([t, torch.zeros_like(t[:1])]).tolist()

    @torch.no_grad()
    def sample_edm(self, hu, cond, hu_mask, sparams, return_last=True, guide_dx=False):
        if guide_dx:
            self.get_dx_pde(cond, hu)                                 # raises: see get_dx_pde
        w = guidance_weight(sparams.w, cond)
        if not hu.is_cuda:
            raise L.McedmError("sample_edm needs CUDA tensors: the sm_100a kernels have no CPU fallback")
        hu_noise = self._randn_like("init", hu)                     # :576
        return self._sample_core(hu_noise, cond, hu_mask, sparams, return_last, w=w)

    @torch.no_grad()
    def _sample_core(self, hu_noise, cond, hu_mask, sparams, return_last=True, guide_fn=None, w=0.0):
        """Stochastic Heun with mask blending on the kernels, given the initial N(0,1) draw `hu_noise` [B,C,H,W]
        (shared with PlCondEdm, whose sampler takes the draw from its caller and uses an all-ones mask).
        guide_fn(cond, D fp32 [B,C,H,W]) -> fp32 [B,C,H,W]: the PDE-guidance gradient of PlCondDdim.sample_edm
        (ddim.py:1569-1571, :1588-1590); the updates then subtract (5*dx)/t_hat from both slopes.
        w: classifier-free guidance weight (see guidance_weight).  Guided, every evaluation is one network batch of 2B
        rows (rows [B, 2B) see the all-zero condition) and the updates use D_w = c_skip*x + c_out*F_w; the mask blending
        and the known values still come from `cond`, and no extra noise is drawn."""
        hu = hu_noise
        lib = L.lib()
        model = self.ema_model if self.ema_model is not None else self.model
        unet = self._unet_of(model)
        if _dropout_active(unet):
            raise NotImplementedError("the sampler runs the inference plan, which has no dropout, on a network in "
                                      "training mode with dropout > 0: put the module in eval mode")
        t_steps = self.edm_time_steps(sparams)
        num_steps = sparams.timesteps
        B, C, H, W = hu.shape
        total = hu.numel()
        dev = hu.device
        w = guidance_weight(w, cond)
        cfg = w is not None
        if cfg and unet.out_channels != C:
            raise ValueError("classifier-free guidance needs a network output shaped like the sampler state")
        bufs = self._sampler_buffers(B, C, H, W, cond.shape[1], unet.out_channels, dev, cfg)
        cond_s, mask_s = bufs["cond"], bufs["mask"]
        cond_s[:B].copy_(cond)                                      # static addresses -> the captured graph is reused
        mask_s.copy_(hu_mask)
        cond, mask = cond_s[:B], mask_s
        hu_noise = hu_noise.to(torch.float32).contiguous()
        x_cur, x_hat, x_e, d_cur = bufs["x_cur"], bufs["x_hat"], bufs["x_e"], bufs["d_cur"]
        x_in, F_buf, nl = bufs["x_in"], bufs["F"], bufs["nl"]
        c_noise_all = []
        D_buf = (torch.empty(B, C, H, W, device=dev, dtype=torch.float32)
                 if (self._trace is not None or guide_fn is not None) else None)
        st = L.stream_ptr()
        L.check(lib.mcedm_edm_init(L.ptr(hu_noise), L.ptr(cond), cond.shape[1], L.ptr(mask), t_steps[0], B, C, H, W,
                                   L.ptr(x_cur), st), "edm_init")
        xs = [x_cur.clone()] if not return_last else None
        S_min, S_max = sparams.S_min, float(sparams.S_max)
        gamma_on = min(sparams.S_churn / num_steps, math.sqrt(2) - 1)
        t_hats = []
        for i in range(num_steps):
            gamma = gamma_on if S_min <= t_steps[i] <= S_max else 0
            t_hats.append(t_steps[i] + gamma * t_steps[i])
            c_noise_all.append(precond_scalars(t_hats[i])[3])
            c_noise_all.append(precond_scalars(t_steps[i + 1])[3] if i < num_steps - 1 else 0.0)
        c_noise_dev = torch.tensor(c_noise_all, dtype=torch.float32).to(dev)
        engine = unet.engine()
        x_in_c, cond_c = engine._check_inputs(x_in, nl, cond_s)[0::2]
        assert x_in_c.data_ptr() == x_in.data_ptr()

        # all (scale | shift) rows of the trajectory's noise levels from one embedding-MLP launch; an evaluation then
        # only copies its row (engine.embedding_table); plans that do not take rows evaluate the MLP per evaluation
        table = engine.embedding_table(c_noise_dev) if getattr(engine, "supports_ss_rows", False) else None

        def net_eval(k):
            if table is not None:
                return engine.forward_static(x_in, nl, cond_c, F_buf, use_graph=self.use_cuda_graph, ss_rows=table[:, k])
            nl.copy_(c_noise_dev[k:k + 1])
            return engine.forward_static(x_in, nl, cond_c, F_buf, use_graph=self.use_cuda_graph)

        # guided: the *_cfg kernels, which take w after the fp32 coefficients and read F = [F_c | F_u]
        wa = (w,) if cfg else ()
        churn = lib.mcedm_edm_churn_cfg if cfg else lib.mcedm_edm_churn
        euler = lib.mcedm_edm_euler_cfg if cfg else lib.mcedm_edm_euler
        correct = lib.mcedm_edm_correct_cfg if cfg else lib.mcedm_edm_correct
        denoised = lib.mcedm_edm_denoised_cfg if cfg else lib.mcedm_edm_denoised

        for i in range(num_steps):
            t_cur, t_next = t_steps[i], t_steps[i + 1]
            t_hat = t_hats[i]
            coef = math.sqrt(t_hat ** 2 - t_cur ** 2) * sparams.S_noise
            eps = self._randn_like("step", x_cur)                   # fp64, :608
            c_skip, c_out, c_in, c_noise = precond_scalars(t_hat)
            L.check(churn(L.ptr(x_cur), L.ptr(eps), L.ptr(mask), coef, c_in, total, L.ptr(x_hat), L.ptr(x_in), st),
                    "edm_churn")
            F1 = net_eval(2 * i)
            last = i == num_steps - 1
            c_skip2, c_out2, c_in2, c_noise2 = precond_scalars(t_next) if not last else (0.0, 0.0, 0.0, 0.0)
            # Euler step; on the last step x_e already is the result (t_next = 0, no correction)
            out_e = x_cur if last else x_e
            if guide_fn is None:
                L.check(euler(L.ptr(x_hat), L.ptr(F1), L.ptr(mask), t_hat, t_next, c_skip, c_out, c_in2, *wa, total,
                              L.ptr(d_cur), L.ptr(out_e), None if last else L.ptr(x_in), L.ptr(D_buf), st), "edm_euler")
            else:
                L.check(denoised(L.ptr(x_hat), L.ptr(F1), c_skip, c_out, *wa, total, L.ptr(D_buf), st), "edm_denoised")
                gdx = guide_fn(cond, D_buf)
                L.check(lib.mcedm_edm_euler_guided(L.ptr(x_hat), L.ptr(D_buf), L.ptr(gdx), L.ptr(mask), t_hat, t_next,
                                                   c_in2, total, L.ptr(d_cur), L.ptr(out_e),
                                                   None if last else L.ptr(x_in), st), "edm_euler_guided")
                if cfg and not last:
                    x_in[B:].copy_(x_in[:B])                        # the unconditional half sees the same input
            if self._trace is not None:
                self._trace.append((i, 0, t_hat, D_buf.clone(), x_hat.clone()))
            if not last:
                F2 = net_eval(2 * i + 1)
                if guide_fn is None:
                    L.check(correct(L.ptr(x_hat), L.ptr(x_e), L.ptr(F2), L.ptr(d_cur), L.ptr(mask), t_hat, t_next,
                                    c_skip2, c_out2, *wa, total, L.ptr(x_cur), L.ptr(D_buf), st), "edm_correct")
                else:
                    L.check(denoised(L.ptr(x_e), L.ptr(F2), c_skip2, c_out2, *wa, total, L.ptr(D_buf), st),
                            "edm_denoised")
                    gdx = guide_fn(cond, D_buf)
                    L.check(lib.mcedm_edm_correct_guided(L.ptr(x_hat), L.ptr(x_e), L.ptr(D_buf), L.ptr(gdx),
                                                         L.ptr(d_cur), L.ptr(mask), t_hat, t_next, total,
                                                         L.ptr(x_cur), st), "edm_correct_guided")
                if self._trace is not None:
                    self._trace.append((i, 1, t_next, D_buf.clone(), x_e.clone()))
            if xs is not None:
                xs.append(x_cur.clone())
        xs = torch.stack(xs, dim=0) if xs is not None else x_cur.clone().unsqueeze(0)
        return rearrange(xs, "t b c h w -> b t h w c")

    def _sampler_buffers(self, B, C, H, W, Cc, Cout, dev, cfg=False):
        """Persistent device buffers of one sampling batch shape (state fp64, network I/O fp32).  cfg: the network input,
        output and condition hold the 2B rows of a guided evaluation; condition rows [B, 2B) are zeroed here, once."""
        cache = self.__dict__.setdefault("_sampler_buf_cache", {})
        key = (B, C, H, W, Cc, Cout, str(dev), cfg)
        bufs = cache.get(key)
        if bufs is None:
            if len(cache) > 4:
                cache.clear()
            f64 = dict(device=dev, dtype=torch.float64)
            f32 = dict(device=dev, dtype=torch.float32)
            rows = 2 * B if cfg else B
            bufs = dict(x_cur=torch.empty(B, C, H, W, **f64), x_hat=torch.empty(B, C, H, W, **f64),
                        x_e=torch.empty(B, C, H, W, **f64), d_cur=torch.empty(B, C, H, W, **f64),
                        x_in=torch.empty(rows, C, H, W, **f32), F=torch.empty(rows, Cout, H, W, **f32),
                        cond=torch.empty(rows, Cc, H, W, **f32), mask=torch.empty(B, C, H, W, **f32),
                        nl=torch.empty(1, **f32))
            bufs["cond"][B:].zero_()
            cache[key] = bufs
        return bufs
