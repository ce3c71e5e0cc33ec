"""CPU oracle of classifier-free guidance (CFG) in the EDM samplers: test infrastructure on top of oracle/edm_oracle.py,
in plain fp32 / fp64 torch ops.

The reference has a CFG branch in `get_denoised` (models/mcedm.py:453-458) but no fixture for w != 0, so these functions
state the definition the kernels implement (DESIGN.md §3):

    F_c = F(c_in*x, c_noise, cond)      F_u = F(c_in*x, c_noise, 0)      (the all-zero condition, as cond=None)
    F_w = (1+w)*F_c - w*F_u             fp32, (1+w) and w rounded to fp32, each product and the difference rounded
    D_w = c_skip*x + c_out*F_w

Combining F rather than D makes w = 0 give the bits of F_c and w = -1 the bits of F_u.  The samplers are
oracle.edm_oracle.sample_edm / cond_sample_edm with `denoise` replaced by `denoise_cfg`; with w = 0 they reproduce them
bit for bit.
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np
import torch

from oracle import edm_oracle as O

Tensor = torch.Tensor


def cfg_weights(w: float):
    """(1+w, w) as fp32 scalar tensors: the rounding the kernels apply to the host's double w."""
    return torch.tensor(1.0 + w, dtype=torch.float32), torch.tensor(w, dtype=torch.float32)


def combine(f_c: Tensor, f_u: Tensor, w: float) -> Tensor:
    w_c, w_u = cfg_weights(w)
    return w_c * f_c - w_u * f_u


def denoise_cfg(sd, model_cfg, xt: Tensor, sigma: Tensor, cond: Tensor, w: float):
    """Guided get_denoised: (D_w, F_w) in fp32."""
    xt = xt.to(torch.float32)
    c_skip, c_out, c_in, c_noise = O.precond_coeffs(sigma)
    x_in = c_in * xt
    f_c = O.unet_forward(sd, model_cfg, x_in, c_noise.flatten(), cond)
    f_u = O.unet_forward(sd, model_cfg, x_in, c_noise.flatten(), None)
    f_w = combine(f_c, f_u, w)
    return c_skip * xt + c_out * f_w, f_w


def sample_edm_cfg(sd, model_cfg, hu_noise: Tensor, cond: Tensor, hu_mask: Tensor, sparams,
                   step_noise: Callable[[int, Tensor], Tensor], w: float, n_state_ch: Optional[int] = None,
                   return_last: bool = True, record: Optional[list] = None) -> Tensor:
    """oracle.edm_oracle.sample_edm with every evaluation guided: the mask blending and the known values come from
    `cond`, only the unconditional evaluation sees zeros; no extra noise is drawn."""
    num_steps = int(sparams["timesteps"])
    t_steps = O.edm_schedule(num_steps, sparams["sigma_min"], sparams["sigma_max"], sparams["rho"])
    c = n_state_ch if n_state_ch is not None else hu_noise.shape[1]
    known = cond[:, 0:c]
    x_next = hu_noise.to(torch.float64) * t_steps[0]
    x_next = known * (1 - hu_mask) + x_next * hu_mask
    xs = [x_next]
    s_min, s_max = sparams["S_min"], float(sparams["S_max"])
    for i, (t_cur, t_next) in enumerate(zip(t_steps[:-1], t_steps[1:])):
        x_cur = x_next
        gamma = min(sparams["S_churn"] / num_steps, np.sqrt(2) - 1) if s_min <= t_cur <= s_max else 0
        t_hat = t_cur + gamma * t_cur
        x_hat = x_cur + (t_hat ** 2 - t_cur ** 2).sqrt() * sparams["S_noise"] * step_noise(i, x_cur) * hu_mask
        d1, _ = denoise_cfg(sd, model_cfg, x_hat, t_hat, cond, w)
        if record is not None:
            record.append((i, 0, float(t_hat), d1))
        d_cur = (x_hat - d1.to(torch.float64)) / t_hat
        x_next = x_hat + (t_next - t_hat) * d_cur * hu_mask
        if i < num_steps - 1:
            d2, _ = denoise_cfg(sd, model_cfg, x_next, t_next, cond, w)
            if record is not None:
                record.append((i, 1, float(t_next), d2))
            d_prime = (x_next - d2.to(torch.float64)) / t_next
            x_next = x_hat + (t_next - t_hat) * (0.5 * d_cur + 0.5 * d_prime) * hu_mask
        xs = [x_next] if return_last else xs + [x_next]
    return torch.stack(xs, dim=0).permute(1, 0, 3, 4, 2)


def cond_sample_edm_cfg(sd, model_cfg, u_noise: Tensor, h_cond: Tensor, sparams,
                        step_noise: Callable[[int, Tensor], Tensor], w: float, return_last: bool = True,
                        record: Optional[list] = None,
                        guide: Optional[Callable[[Tensor, Tensor], Tensor]] = None) -> Tensor:
    """oracle.edm_oracle.cond_sample_edm with every evaluation guided; the PDE guidance, when given, is taken of D_w."""
    num_steps = int(sparams["timesteps"])
    t_steps = O.edm_schedule(num_steps, sparams["sigma_min"], sparams["sigma_max"], sparams["rho"])
    x_next = u_noise.to(torch.float64) * t_steps[0]
    xs = [x_next]
    s_min, s_max = sparams["S_min"], float(sparams["S_max"])
    for i, (t_cur, t_next) in enumerate(zip(t_steps[:-1], t_steps[1:])):
        x_cur = x_next
        gamma = min(sparams["S_churn"] / num_steps, np.sqrt(2) - 1) if s_min <= t_cur <= s_max else 0
        t_hat = t_cur + gamma * t_cur
        x_hat = x_cur + (t_hat ** 2 - t_cur ** 2).sqrt() * sparams["S_noise"] * step_noise(i, x_cur)
        d1, _ = denoise_cfg(sd, model_cfg, x_hat, t_hat, h_cond, w)
        if record is not None:
            record.append((i, 0, float(t_hat), d1))
        d1 = d1.to(torch.float64)
        d_cur = (x_hat - d1) / t_hat
        if guide is not None:
            d_cur = d_cur - 5. * guide(h_cond, d1) / t_hat
        x_next = x_hat + (t_next - t_hat) * d_cur
        if i < num_steps - 1:
            d2, _ = denoise_cfg(sd, model_cfg, x_next, t_next, h_cond, w)
            if record is not None:
                record.append((i, 1, float(t_next), d2))
            d2 = d2.to(torch.float64)
            d_prime = (x_next - d2) / t_next
            if guide is not None:
                d_prime = d_prime - 5. * guide(h_cond, d2) / t_hat
            x_next = x_hat + (t_next - t_hat) * (0.5 * d_cur + 0.5 * d_prime)
        xs = [x_next] if return_last else xs + [x_next]
    return torch.stack(xs, dim=0).permute(1, 0, 3, 4, 2)
