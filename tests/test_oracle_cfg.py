"""CPU: the classifier-free-guidance oracle (tests/cfg_oracle.py) against the unguided oracle, and the guidance gate.

Combining the network outputs as F_w = (1+w)*F_c - w*F_u makes w = 0 and w = -1 exact: the guided denoiser then
returns the bits of the conditional and of the unconditional one, and the guided samplers at w = 0 the bits of the
existing ones."""
import copy
import math

import pytest
import torch

from cfg_oracle import cond_sample_edm_cfg, denoise_cfg, sample_edm_cfg
from common import NoiseFeed, golden, stress_unet
from mcedm_b200.mcedm import guidance_weight
from oracle import edm_oracle as O


def _sd_cfg(config="config_adm_edm_mcedm_res32"):
    net, cfg, _ = stress_unet(config)
    return {k: v.detach() for k, v in net.state_dict().items()}, dict(cfg.model.hparams.model), cfg


def test_denoise_cfg_identities():
    sd, mcfg, _ = _sd_cfg()
    case = golden("denoise.pt")["cases"][1]
    xt, sigma, cond = case["xt"], torch.tensor(case["sigma"], dtype=torch.float64), case["cond"]
    with torch.no_grad():
        d_c, f_c = O.denoise(sd, mcfg, xt, sigma, cond)
        d_u, f_u = O.denoise(sd, mcfg, xt, sigma, None)
        d0, f0 = denoise_cfg(sd, mcfg, xt, sigma, cond, 0.0)
        dm1, fm1 = denoise_cfg(sd, mcfg, xt, sigma, cond, -1.0)
        d2, f2 = denoise_cfg(sd, mcfg, xt, sigma, cond, 2.0)
    assert torch.equal(d0, d_c) and torch.equal(f0, f_c)
    assert torch.equal(dm1, d_u) and torch.equal(fm1, f_u)
    # the two halves differ on this input, so the identities above are not vacuous, and w = 2 extrapolates
    assert float((f_c - f_u).abs().max()) > 1e-2
    assert torch.equal(f2, torch.tensor(3.0) * f_c - torch.tensor(2.0) * f_u)


def test_guided_oracle_samplers_at_w0_are_the_unguided_ones():
    sd, mcfg, cfg = _sd_cfg()
    sp = dict(copy.deepcopy(cfg.diff_sampler))
    sp["timesteps"] = 2
    g = torch.Generator().manual_seed(4)
    cond = torch.randn(1, 2, 128, 128, generator=g)
    mask = torch.zeros(1, 2, 128, 128)
    mask[:, 1] = 1.0
    hu = torch.randn(1, 2, 128, 128, generator=g)
    outs = []
    for fn in (lambda **k: O.sample_edm(**k), lambda **k: sample_edm_cfg(w=0.0, **k)):
        feed = NoiseFeed(11)
        with torch.no_grad():
            outs.append(fn(sd=sd, model_cfg=mcfg, hu_noise=hu, cond=cond, hu_mask=mask, sparams=sp,
                           step_noise=lambda i, x: feed.draw(x)))
    assert torch.equal(outs[0], outs[1])

    sd, mcfg, cfg = _sd_cfg("config_adm_edm_res32_cond_h")
    sp = dict(copy.deepcopy(cfg.diff_sampler))
    sp["timesteps"] = 2
    h = torch.randn(1, 1, 128, 128, generator=g)
    u = torch.randn(1, 1, 128, 128, generator=g)
    outs = []
    for fn in (lambda **k: O.cond_sample_edm(**k), lambda **k: cond_sample_edm_cfg(w=0.0, **k)):
        feed = NoiseFeed(12)
        with torch.no_grad():
            outs.append(fn(sd=sd, model_cfg=mcfg, u_noise=u, h_cond=h, sparams=sp,
                           step_noise=lambda i, x: feed.draw(x)))
    assert torch.equal(outs[0], outs[1])


def test_guidance_gate():
    c = torch.zeros(1)
    assert guidance_weight(None, c) is None
    assert guidance_weight(0.0, c) is None and guidance_weight(-9.99e-4, c) is None
    assert guidance_weight(1.5, None) is None
    assert guidance_weight(1e-3, c) == 1e-3 and guidance_weight(-1, c) == -1.0
    for bad in (math.nan, math.inf, -math.inf):
        with pytest.raises(ValueError):
            guidance_weight(bad, c)
        with pytest.raises(ValueError):
            guidance_weight(bad, None)
