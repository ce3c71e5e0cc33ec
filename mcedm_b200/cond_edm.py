"""Drop-in host mirror of the reference's single-task EDM module `PlCondEdm` (models/ddim.py:1608-1773, on top of
`PlCondDdim` :1054-1606): the baseline of BASELINE config 5 (`config_adm_edm_res32_cond_h`) — `u` is denoised, `h`
(or the Darcy permeability `a`) is the condition, there is no mask.

Same EDM mathematics as `PlMcedm`, so the class reuses its kernel path unchanged:
  * the network + preconditioning (`model_precond`, `get_denoised`) are `PlMcedm._precond_apply`;
  * the sampler `sample_edm(h, u_noise, sparams)` (ddim.py:1532-1601: plain stochastic Heun) is the masked sampler core
    with an all-ones mask — `x*1`, `+ known*0` and `*mask` are exact in floating point, so it is the same arithmetic
    (checked against the reference fixture by tests/test_gpu_parity.py::test_cond_edm_sampler_and_training_step);
  * `training_step` is the fused noise-injection / U-Net / loss(+dL/dF) path with `mask=None` (loss over every pixel,
    ddim.py:1723).
  * the PDE residual metric (`get_pde_loss`, ddim.py:1388-1422) and the PDE guidance of the sampler (`guide_dx`:
    `get_dx_pde` / `get_dx_log_prob`, ddim.py:1424-1450, :641-650) run on the K6 kernels (csrc/pde.cu); with guidance
    the denoised field is materialised after each network evaluation, the residual gradient is one stencil launch, and
    the Euler / correction kernels subtract `(5*dx)/t_hat` (ddim.py:1571, :1590).  No host synchronisation: the
    reference's `has_nan ... .item()` test is dead code (SweFvLoss.forward already zeroes NaNs, pde_loss.py:241).
  * classifier-free guidance (`sparams.w`, |w| >= 1e-3): each evaluation is one network batch of 2B rows, the second
    half with the all-zero condition that the training step's condition drop (`cond_p`) feeds, and the sampler uses
    D_w = c_skip*x + c_out*((1+w)*F_c - w*F_u) (mcedm.guidance_weight); with `guide_dx` the PDE-guidance gradient is
    taken of D_w.
What is NOT mirrored: `dx_cond`, self-conditioning, `node_type`, `select_by_pde`, the Darcy residual *gradient*, the
training-time PDE loss term, and the DDIM sampler (`sample`, `sample_with_repeat` raise, as in the reference).
"""
from __future__ import annotations

import torch
from einops import rearrange

from .mcedm import PlMcedm, guidance_weight
from .nn_misc import CorrelationLoss


class PlCondEdm(PlMcedm):
    def __init__(self, hparams):
        super().__init__(hparams)
        m = hparams.model
        # probability of keeping the conditioning during training (PlCondDdim.__init__, ddim.py:1058-1059)
        self.cond_p = m.cond_p if hasattr(m, "cond_p") else 0.8
        self.node_type = m.node_type if hasattr(m, "node_type") else False
        if self.node_type:
            raise NotImplementedError("node_type conditioning is not on the hot path")
        if getattr(m, "self_cond", False):
            raise NotImplementedError("self-conditioning is not supported")
        self.mae_criterion = torch.nn.L1Loss()                       # PlDdim.__init__, ddim.py:75
        self.correlation = CorrelationLoss()                          # ddim.py:77
        self.h_ch = m.cond_channels if m.cond_channels else 1
        self.u_ch = m.out_ch
        self.log_lr = False

    # ---------------------------------------------------------------- configuration helpers
    def get_inp_stats_shape(self, hparams):                           # ddim.py:1061-1064
        ch = hparams.model.in_channels
        return (ch,) if ch > 1 else ()

    def get_tar_stats_shape(self, hparams):                           # ddim.py:1066-1069
        ch = hparams.model.out_ch
        return (ch,) if ch > 1 else ()

    @staticmethod
    def get_edm_sampler_params():                                     # ddim.py:1620-1645
        from .config import AttrDict

        return AttrDict(name="edm", type="edm", timesteps=50, sigma_min=0.002, sigma_max=80, rho=7, S_churn=15.0, S_min=0,
                        S_max="inf", S_noise=1, n_samples=5, n_repeat=2, n_time_h=128, n_time_u=0, return_last=True,
                        select_by_pde=False, use_gt_pde_select=True, guide_dx=False, w=0.0, plot_scaled=False)

    def set_test_sampler_params(self, params):                        # ddim.py:1647-1652
        if params.type != "edm":
            print("Model with EDM preconditioning supports only EDM sampler ")
            params = self.get_edm_sampler_params()
        self.test_sparams = params

    def inverse_data_transform_u(self, u):                            # ddim.py:1071-1079
        if self.rescaled:
            u = (u + 1.0) / 2.0
        if self.normalization == "min_max":
            u = torch.clamp(u, 0.0, 1.0)
        return self.normalizer_target(u, inverse=True)

    def get_cond_in(self, h, u, dx, dt):                              # ddim.py:1081-1116 (node_type False)
        cond_ch = self.model.cond_channels
        if cond_ch == self.h_ch:
            return h
        if cond_ch == self.h_ch + self.u_ch:
            return torch.cat([h, u[:, 0:1].repeat(1, u.shape[1], 1, 1)], dim=-1)
        if cond_ch == self.h_ch + 2:
            return torch.cat([h, dt, dx], dim=-1)
        if cond_ch == self.h_ch + self.u_ch + 2:
            return torch.cat([h, u[:, 0:1].repeat(1, u.shape[1], 1, 1), dt, dx], dim=-1)
        raise TypeError(f"Number of conditional channels {cond_ch} should be changed to match the known states "
                        f"channels {self.h_ch}")                      # the reference raises a str here (a TypeError)

    # ---------------------------------------------------------------- training
    def forward(self, x, sigma, noise, cond=None):                    # ddim.py:1668-1694 -> (D_x, x0_t)
        x_noise = x + noise * sigma
        if torch.rand(1) >= self.cond_p:                              # host RNG draw kept for RNG parity (:1684)
            cond = None
        d = self.model_precond(x_noise, sigma.float(), cond)
        return d, d

    def training_step(self, train_batch, batch_idx):                  # ddim.py:1700-1737
        h_unnorm, dx, dt, u_unnorm = train_batch
        self.h_ch = h_ch = h_unnorm.shape[-1]
        self.u_ch = u_ch = u_unnorm.shape[-1]
        x = self.data_transform(h_unnorm, u_unnorm)
        h, u = x[..., 0:h_ch], x[..., h_ch:h_ch + u_ch]
        cond_in = rearrange(self.get_cond_in(h, u, dx, dt), "b h w c -> b c h w").contiguous()
        u = rearrange(u, "b h w c -> b c h w").contiguous()
        noise = self._randn_like("noise", u)
        rnd_normal = torch.randn([u.shape[0], 1, 1, 1]).type_as(u)    # CPU RNG, as :1714-1715
        sigma = (rnd_normal * self.P_std + self.P_mean).exp()
        weight = self.get_loss_weight(sigma)
        # reference: D_x, _ = self.forward(u, sigma, noise, cond=cond_in); loss = self.criteria(D_x, u, weight).
        # Fused here exactly as in PlMcedm.training_step, with no mask (the cond_p coin is drawn inside forward_loss).
        loss = self.forward_loss(u, sigma, noise, cond_in, None, weight)
        self.log("train_loss", loss, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        if self.pde_loss_lambda > 0.0:
            raise NotImplementedError("the PDE residual loss term is outside the hot path (SURVEY §8f)")
        return loss

    # ---------------------------------------------------------------- sampling
    def sample(self, h, u_noise, sparams, return_last=True, guide_dx=False):
        raise NotImplementedError("Only EDM sampler is supported for the model with EDM pre-conditioning")

    def sample_with_repeat(self, h, u, sparams, return_last=True, guide_dx=False):
        raise NotImplementedError("Only EDM sampler is supported for the model with EDM pre-conditioning")

    # ---------------------------------------------------------------- PDE residual and guidance (K6)
    def get_pde_loss(self, cond, x_denoised, x_gt_unnorm=None, noise_level=None, clamp_loss=True, do_rearrange=True,
                     reduce=True):                                    # ddim.py:1388-1422
        """cond: the (normalised) condition `b h w c` whose first channel is h; x_denoised: the normalised u sample
        `b h w c`; any float dtype.  Every caller in the reference passes do_rearrange=False except the training-time
        PDE term, where :1390 slices the channel range off the *width* axis of a `b c h w` tensor."""
        if do_rearrange:
            raise NotImplementedError("get_pde_loss(do_rearrange=True) is only reached by the training-time PDE term")
        h, u = cond[..., :self.h_ch], x_denoised
        if h.shape[-1] != 1 or u.shape[-1] != 1:
            raise NotImplementedError("the PDE residual kernels take one h and one u channel")
        return self._pde_residual(h[..., 0], u[..., 0], x_gt_unnorm, noise_level, clamp_loss, reduce,
                                  sum_channels=True)

    def get_dx_pde(self, cond, x_denoised, calc_prob=False):          # ddim.py:1424-1450; cond, x_denoised `b c h w`
        if self.h_ch != 1 or x_denoised.shape[1] != 1:
            raise NotImplementedError("the PDE residual kernels take one h and one u channel")
        h, u, apply_norm = self._pde_planes(cond[:, 0], x_denoised[:, 0])
        g = self.pde_loss.gradient(h, u, self.normalizer_input, self.normalizer_target, apply_norm=apply_norm,
                                   mode=1 if calc_prob else 2)
        return g.unsqueeze(1) if calc_prob else g                     # mean(dim=1, keepdim) | sum(dim=1)

    def get_dx_log_prob(self, cond, x_denoised, guide_dx):            # ddim.py:641-650
        if guide_dx:
            return self.get_dx_pde(cond, x_denoised, calc_prob=True)
        return torch.zeros_like(x_denoised)

    @staticmethod
    def scale_each_min_max(state, return_min_max=False):              # ddim.py:689-698
        flat = rearrange(state, "b h w c -> b c (h w)")
        if state.is_cuda and state.dtype == torch.float64:
            # the two range reductions as one kernel over the channel-last fields (csrc/metrics.cu mcedm_corr_minmax)
            from . import _lib as L

            b, H, W, C = state.shape
            sc = state.contiguous()
            lo = torch.empty(b, C, 1, device=state.device, dtype=torch.float64)
            hi = torch.empty(b, C, 1, device=state.device, dtype=torch.float64)
            L.check(L.lib().mcedm_corr_minmax(L.ptr(sc), None, b, H * W, C, None, L.ptr(lo), L.ptr(hi), L.stream_ptr()),
                    "corr_minmax")
        else:
            lo = torch.min(flat, dim=2, keepdim=True)[0]
            hi = torch.max(flat, dim=2, keepdim=True)[0]
        scaled = rearrange((flat - lo) / (hi - lo), "b c (h w) -> b h w c", h=state.size(1), w=state.size(2))
        return (scaled, lo, hi) if return_min_max else scaled

    @torch.no_grad()
    def sample_edm(self, h, u_noise, sparams, return_last=True, guide_dx=False):   # ddim.py:1532-1601
        """h: condition b h w c; u_noise: the caller's N(0,1) draw b h w c. Returns xs [b, t, h, w, c] float64."""
        w = guidance_weight(sparams.w, h)
        if not u_noise.is_cuda:
            from . import _lib as L

            raise L.McedmError("sample_edm needs CUDA tensors: the sm_100a kernels have no CPU fallback")
        cond = rearrange(h, "b h w c -> b c h w").contiguous().float()
        noise = rearrange(u_noise, "b h w c -> b c h w").contiguous()
        guide_fn = (lambda c, D: self.get_dx_pde(c, D, calc_prob=True)) if guide_dx else None
        return self._sample_core(noise, cond, torch.ones_like(noise, dtype=torch.float32), sparams, return_last,
                                 guide_fn=guide_fn, w=w)

    # ---------------------------------------------------------------- evaluation steps
    def validation_step(self, val_batch, batch_idx):                  # ddim.py:1154-1217
        if (self.current_epoch + 1) % 100 != 0 and self.current_epoch != 0:
            return {"epoch": self.current_epoch}
        h_unnorm, dx, dt, u_unnorm = val_batch
        self.h_ch = h_ch = h_unnorm.shape[-1]
        self.u_ch = u_ch = u_unnorm.shape[-1]
        state_gt = self.data_transform(h_unnorm, u_unnorm)
        h, u = state_gt[..., :h_ch], state_gt[..., h_ch:u_ch + h_ch]
        u_noise = self._randn_like("val_noise", u)
        if self.sparams.type != "edm":
            raise TypeError("Non EDM sampler is not supported for the model")
        xs = self.sample_edm(self.get_cond_in(h, u, dx, dt), u_noise, self.sparams, return_last=True,
                             guide_dx=self.sparams.guide_dx)
        u_last = xs[:, -1, :, :, :u_ch]
        loss_u = self.mae_criterion(u_last, u)
        loss_u_un = self.mae_criterion(self.inverse_data_transform_u(u_last), u_unnorm)
        gt_scaled = self.scale_each_min_max(state_gt)
        xs_scaled = self.scale_each_min_max(xs[:, -1])
        loss_u_scaled = self.mae_criterion(xs_scaled, gt_scaled[:, :, :, h_ch:u_ch + h_ch])
        self.log("val_mae_u", loss_u, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        self.log("val_mae_u_un", loss_u_un, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        self.log("val_mae_u_scaled", loss_u_scaled, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        corr_u = torch.mean(self.correlation(xs[:, -1], state_gt[..., h_ch:u_ch + h_ch]))
        self.log("val_corr_u", corr_u, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        pde_loss = self.get_pde_loss(state_gt[..., 0:h_ch], xs[:, -1], clamp_loss=False,
                                     do_rearrange=False) / len(h_unnorm)
        self.log("val_pde_loss", pde_loss, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        if getattr(self.sparams, "plot_scaled", False):
            xs_traj, gt_plot = xs_scaled.unsqueeze(dim=1), gt_scaled[..., h_ch:u_ch + h_ch]
        else:
            xs_traj, gt_plot = xs[:, -1].unsqueeze(dim=1), state_gt[..., h_ch:u_ch + h_ch]
        return {"epoch": self.current_epoch, "loss": loss_u, "loss_u_un": loss_u_un, "val_loss_u_scaled": loss_u_scaled,
                "traj": xs_traj, "gt": gt_plot}

    def test_step(self, test_batch, test_idx):                        # ddim.py:1219-1319
        h_unnorm, dx, dt, u_unnorm = test_batch
        self.h_ch = h_ch = h_unnorm.shape[-1]
        self.u_ch = u_ch = u_unnorm.shape[-1]
        state_gt = self.data_transform(h_unnorm, u_unnorm)
        h, u = state_gt[..., :h_ch], state_gt[..., h_ch:u_ch + h_ch]
        n_samples = self.test_sparams.n_samples
        state_gt_rep = state_gt.repeat(n_samples, 1, 1, 1)
        cond_in_rep = self.get_cond_in(h, u, dx, dt).repeat(n_samples, 1, 1, 1)
        u_noise = self._randn_like("test_noise", u.repeat(n_samples, 1, 1, 1))
        if self.test_sparams.type != "edm":
            raise TypeError("Non EDM sampler is not supported for the model")
        if getattr(self.test_sparams, "select_by_pde", False):
            raise NotImplementedError("select_by_pde (best-of-n by PDE error) is not supported")
        xs = self.sample_edm(cond_in_rep, u_noise, self.test_sparams, return_last=self.test_sparams.return_last,
                             guide_dx=self.test_sparams.guide_dx)
        xs_mean = torch.mean(rearrange(xs, "(n b) t h w c -> n b t h w c", n=n_samples), dim=0)
        u_last = xs_mean[:, -1, :, :, :u_ch]
        loss_u = self.mae_criterion(u_last, u)
        loss_u_un = self.mae_criterion(self.inverse_data_transform_u(u_last), u_unnorm)
        gt_scaled = self.scale_each_min_max(state_gt)
        xs_scaled = self.scale_each_min_max(xs[:, -1])
        xs_scaled_mean = torch.mean(rearrange(xs_scaled, "(n b) h w c -> n b h w c", n=n_samples), dim=0)
        loss_u_scaled = self.mae_criterion(xs_scaled_mean, gt_scaled[:, :, :, h_ch:u_ch + h_ch])
        corr_u = torch.mean(self.correlation(xs_mean[:, -1], state_gt[..., h_ch:u_ch + h_ch]))
        self.log("test_corr_u", corr_u, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        self.log("test_mae_u", loss_u, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        self.log("test_mae_u_un", loss_u_un, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        self.log("test_mae_u_scaled", loss_u_scaled, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        n_batch = len(h_unnorm)
        pde_loss = self.get_pde_loss(state_gt_rep[..., 0:h_ch], xs[:, -1], clamp_loss=False,
                                     do_rearrange=False) / n_samples / n_batch
        self.log("test_pde_loss", pde_loss, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        pde_loss_gt = self.get_pde_loss(state_gt[..., 0:h_ch], state_gt[..., h_ch:u_ch + h_ch], clamp_loss=False,
                                        do_rearrange=False) / n_batch
        self.log("test_pde_loss_gt", pde_loss_gt, prog_bar=True, on_epoch=True, on_step=False, sync_dist=True)
        if getattr(self.test_sparams, "plot_scaled", False):
            traj = rearrange(xs_scaled, "(n b) h w c -> b h w n c", n=n_samples).unsqueeze(dim=1)
            gt_plot = gt_scaled[..., h_ch:u_ch + h_ch]
        else:
            traj = rearrange(xs[:, -1], "(n b) h w c -> b h w n c", n=n_samples).unsqueeze(dim=1)
            gt_plot = state_gt[..., h_ch:u_ch + h_ch]
        return {"loss": loss_u, "loss_u_un": loss_u_un, "test_mae_u_scaled": loss_u_scaled, "traj": traj, "gt": gt_plot}
