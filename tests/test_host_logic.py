"""CPU: host-side logic — config composition, module surface / checkpoint keys, schedule and scalars,
synthetic data contract, and the multi-process sharding paths on gloo (world_size 2)."""
import copy
import os
import subprocess
import sys

import numpy as np
import torch

from common import golden, hparams, stress_module
from mcedm_b200 import data as D
from mcedm_b200.config import AttrDict, compose
from mcedm_b200.utils import state_hash
from oracle import edm_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# state_hash of the reference's modules right after torch.manual_seed(1) and construction from the shipped configs: the
# whole PlDdim (config_adm_ddim_res32, after set_test_sampler_params) and the DDPM U-Net `Model` (config_ddim_res32).
# Recorded from the mirrors while they were checked bit for bit against the unmodified reference.
REF_DDIM_MODULE_INIT_HASH = "f254c85ee38659d84dc7db0d3c93a108c4cc33506dc1dea30dcad06c261e3982"
REF_DDPM_MODEL_INIT_HASH = "244dadc6bfc09af46ff5dda22bfaf258657f2c2c6c001bf4a3cd2c0e452c27cf"


def test_compose_applies_reference_style_overrides():
    cfg = compose("config_adm_edm_mcedm_res32", ["datamodule.batch_size=16", "diff_sampler.n_samples=1",
                                                 "system=swe_per"])
    assert cfg.datamodule.batch_size == 16 and cfg.diff_sampler.n_samples == 1 and cfg.system == "swe_per"
    m = cfg.model.hparams.model
    assert (m.ch, list(m.ch_mult), m.resolution, list(m.attn_resolutions)) == (64, [1, 1, 1], 128, [32])
    assert not hasattr(m, "node_type") and m.get("node_type", 7) == 7     # OmegaConf-like missing-key semantics
    assert float(cfg.model.hparams.sampler.S_max) == float("inf")


def test_module_surface_and_checkpoint_keys():
    pl, cfg = stress_module()
    sd = pl.state_dict()
    assert len(sd) == 412
    for k in ("model.map_layer0.weight", "model.enc.128x128_conv.weight", "model.dec.32x32_block0.qkv.weight",
              "model.dec.128x128_block1.skip.weight", "model.out_conv.weight", "ema_model.ma_model.out_conv.weight",
              "normalizer_input.subtract", "normalizer_target.divide", "model.enc.64x64_down.conv0.resample_filter"):
        assert k in sd, k
    assert tuple(sd["model.dec.32x32_block0.qkv.weight"].shape) == (192, 64, 1, 1)
    assert tuple(sd["model.out_conv.weight"].shape) == (2, 64, 3, 3)
    opt = pl.configure_optimizers()["optimizer"]
    assert isinstance(opt, torch.optim.Adam) and sum(p.numel() for g in opt.param_groups for p in g["params"]) == 1587010
    for name in ("model_precond", "forward", "get_denoised", "sample_edm", "training_step", "validation_step",
                 "test_step", "get_cond_in", "get_loss_weight", "round_sigma", "set_test_sampler_params"):
        assert callable(getattr(pl, name))


def test_ema_update_matches_reference_rule():
    pl, _ = stress_module()
    before = copy.deepcopy(pl.ema_model.ma_model.state_dict())
    with torch.no_grad():
        for p in pl.model.parameters():
            p.add_(0.01)
    pl.ema_model.update(pl.model)
    for (k, v), p in zip(pl.ema_model.ma_model.named_parameters(), pl.model.parameters()):
        assert torch.allclose(v, before[k] * 0.999 + 0.001 * p, rtol=0, atol=1e-7)


def test_schedule_and_precond_scalars_match_oracle():
    from mcedm_b200.mcedm import precond_scalars

    pl, cfg = stress_module()
    t = pl.edm_time_steps(cfg.diff_sampler)
    ref = O.edm_schedule(50, 0.002, 80, 7)
    assert len(t) == 51 and t[-1] == 0.0 and t == ref.tolist()
    assert abs(t[0] - 80.0) < 1e-9 and abs(t[1] - 71.5010) < 1e-3 and abs(t[49] - 0.002) < 1e-12
    for sigma in (80.0, 104.0, 1.3, 0.0026, 0.002):
        cs, co, ci, cn = precond_scalars(sigma)
        r = [float(v.reshape(())) for v in O.precond_coeffs(torch.tensor(sigma, dtype=torch.float64))]
        assert (cs, co, ci) == (r[0], r[1], r[2])
        assert abs(cn - r[3]) <= 2e-7 * max(1.0, abs(r[3]))


def test_synthetic_batches_have_the_reference_contract():
    h, tg, xg, u, m = D.make_batch("swe_per", 3, "train", seed=1)
    assert h.shape == u.shape == (3, 128, 128, 1) and m.shape == (3, 128, 128, 2) and tg.shape == (3, 128, 128, 1)
    assert 0.99 <= float(h.min()) and float(h.max()) <= 2.01 and float(u.abs().max()) < 1.0
    assert set(m.unique().tolist()) <= {0.0, 1.0}
    # each item misses exactly one whole variable
    assert all(float(m[i, ..., 0].mean()) + float(m[i, ..., 1].mean()) == 1.0 for i in range(3))
    _, _, _, _, md = D.make_batch("swe", 2, "eval")
    assert set(md) == {"u", "h"} and float(md["u"][..., 1].min()) == 1.0 and float(md["u"][..., 0].max()) == 0.0
    a, ud = D.darcy_fields(2)
    assert set(np.unique(a).tolist()) <= {np.float32(0.1), np.float32(1.0)} and ud.min() >= 0
    dm = D.SyntheticMaskDatamodule(system="swe_per", n_train=8, n_test=4, batch_size=4)
    dm.setup("fit")
    st = dm.get_norm_stats()
    assert tuple(st["input_mean"].shape) == (1,)
    b = next(iter(dm.train_dataloader()))
    assert len(b) == 5 and b[4].shape == (4, 128, 128, 2)
    bt = next(iter(dm.test_dataloader()))
    assert isinstance(bt[4], dict) and bt[4]["h"].shape == (4, 128, 128, 2)


def test_unsupported_reference_options_raise():
    from mcedm_b200.mcedm import PlMcedm

    hp = copy.deepcopy(hparams().model.hparams)
    hp.model.dx_cond = True
    try:
        PlMcedm(hp)
        raise AssertionError("dx_cond must raise")
    except NotImplementedError:
        pass
    hp = copy.deepcopy(hparams().model.hparams)
    hp.optimization.optimizer = "Lion"
    pl = PlMcedm(hp)
    try:
        pl.configure_optimizers()
        raise AssertionError("unknown optimizer must raise")
    except NotImplementedError:
        pass


def test_two_rank_gloo_sharding_and_gradient_allreduce():
    """world_size 2 on CPU: row sharding + gather reproduces the single-process order; flat all-reduce averages."""
    script = os.path.join(ROOT, "tests", "dist_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29611")
    procs = [subprocess.Popen([sys.executable, script, str(r), "2"], env=env, stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
    assert "OK" in outs[0]


def test_cond_edm_module_surface():
    """PlCondEdm (config 5) keeps the reference constructor / method surface and the PlCondDdim conditioning variants."""
    import copy

    from mcedm_b200.cond_edm import PlCondEdm
    from mcedm_b200.config import compose

    cfg = compose("config_adm_edm_res32_cond_h")
    pl = PlCondEdm(copy.deepcopy(cfg.model.hparams))
    for name in ("training_step", "validation_step", "test_step", "sample_edm", "get_denoised", "model_precond", "forward",
                 "get_cond_in", "set_test_sampler_params", "get_edm_sampler_params", "inverse_data_transform_u",
                 "configure_optimizers", "optimizer_step", "round_sigma"):
        assert callable(getattr(pl, name))
    assert pl.model.x_channels == 1 and pl.model.cond_channels == 1 and pl.model.out_channels == 1
    assert pl.normalizer_input.subtract.shape == () and pl.normalizer_target.divide.shape == ()   # scalar stats
    h, u = torch.randn(2, 8, 8, 1), torch.randn(2, 8, 8, 1)
    pl.h_ch = pl.u_ch = 1
    assert torch.equal(pl.get_cond_in(h, u, None, None), h)
    sp = pl.get_edm_sampler_params()
    assert sp.type == "edm" and sp.n_samples == 5 and float(sp.S_max) == float("inf")
    pl.set_test_sampler_params(compose("config_adm_edm_res32_cond_h").diff_sampler)
    assert pl.test_sparams.type == "edm"
    for fn in (pl.sample, pl.sample_with_repeat):
        try:
            fn(None, None, None)
            raise AssertionError("DDIM samplers must raise")
        except NotImplementedError:
            pass


def test_ddim_module_surface_and_vp_grid_scalars():
    """PlDdim host mirror (config 4): state_dict surface, VP sigma grid, sigma snapping, alpha-bar look-ups and the fp32
    preconditioning scalars against the oracle's restatement (which the reference fixture pins); the seeded init and the
    sigma range against the reference's."""
    from mcedm_b200.ddim import PlDdim, get_beta_schedule

    cfg = compose("config_adm_ddim_res32")
    torch.manual_seed(1)
    pl = PlDdim(copy.deepcopy(cfg.model.hparams))
    sd = pl.state_dict()
    assert "betas" in sd and "logvar" in sd and tuple(sd["betas"].shape) == (1000,)
    assert tuple(sd["model.enc.128x128_conv.weight"].shape) == (64, 4, 3, 3)        # [x_self_cond | x]: 2 + 2 channels
    assert pl.model.cat_channels == 2 and pl.model.cond_channels == 0 and pl.model.x_channels == 2
    pl.set_test_sampler_params(cfg.diff_sampler)
    grid = O.VpGrid()
    assert torch.equal(pl.edm_steps, grid.edm_steps)
    assert pl.sigma_min == grid.sigma_min and pl.sigma_max == grid.sigma_max
    assert torch.equal(get_beta_schedule("linear", beta_start=1e-4, beta_end=0.02, num_diffusion_timesteps=1000), grid.betas)
    t = pl._edm_grid(cfg.diff_sampler)
    assert t.dtype == torch.float64 and t.shape == (51,) and float(t[-1]) == 0.0
    for s in (80.0, 3.3, 0.011, 0.0):
        sig = torch.tensor(s, dtype=torch.float64)
        assert torch.equal(pl.round_sigma(sig), grid.round_sigma(sig))
        assert torch.equal(pl.round_sigma(sig, return_index=True), grid.round_sigma(sig, return_index=True))
        assert torch.equal(pl.compute_alpha(sig.long()), grid.compute_alpha(sig.long()))
    for s in t[:5].tolist() + t[-4:-1].tolist():
        c_out, c_in, c_noise = pl._vp_scalars(s)
        sigma = torch.tensor(s, dtype=torch.float64).to(torch.float32).reshape(-1, 1, 1, 1)
        assert c_out == float(-sigma) and c_in == float(1 / (sigma ** 2 + 1).sqrt())
        assert c_noise == float(999 - grid.round_sigma(sigma, return_index=True).to(torch.float32))
    hp = copy.deepcopy(cfg.model.hparams)
    hp.name = "ddim"                                                   # any other name builds the DDPM U-Net (ddim.py:40-43)
    from mcedm_b200.ddpm_blocks import Model

    assert isinstance(PlDdim(hp).model, Model)
    g = golden("ddim_path.pt")
    assert len(sd) == 414 and state_hash(pl.state_dict()) == REF_DDIM_MODULE_INIT_HASH   # seeded init is bit-identical
    assert state_hash(pl.model.state_dict()) == g["init_hash"]
    assert abs(pl.sigma_min - g["sigma_min"]) < 1e-12 and abs(pl.sigma_max - g["sigma_max"]) < 1e-9


def test_pde_loss_selection_and_cpu_inputs_raise():
    from mcedm_b200 import _lib as L
    from mcedm_b200.nn_misc import Normalizer
    from mcedm_b200.pde_loss import DarcyLoss, SweFvLoss, get_pde_loss_function

    f, fs = get_pde_loss_function("swe_per", False)
    assert isinstance(f, SweFvLoss) and (f.Tn, f.x_min, f.x_max) == (0.128, -0.5, 0.5) and isinstance(fs, SweFvLoss)
    f, _ = get_pde_loss_function("swe", False)
    assert (f.Tn, f.x_min, f.x_max) == (1.28, -2.5, 2.5)
    f, _ = get_pde_loss_function("anything-else", False)                # loss_helper.py:35-39 default branch
    assert f.Tn == 1.28
    d, _ = get_pde_loss_function("darcy", False)
    assert isinstance(d, DarcyLoss)
    half_dt, dx = get_pde_loss_function("swe_per", False)[0]._grid(128, 128)
    assert dx == 2.0 ** -7 and half_dt == 0.5 * 0.128 / 128
    n = Normalizer(torch.tensor(0.0), torch.tensor(1.0))
    x = torch.zeros(1, 8, 8, 2)
    for fn in (lambda: f(x, x, n, n), lambda: f(x, x, n, n, return_d=True), lambda: d(x, x, n, n)):
        try:
            fn()
            raise AssertionError("CPU tensors were accepted")
        except L.McedmError:
            pass


def test_ddpm_model_mirror_state_dict():
    """Parameter mirror of the DDPM U-Net: names / shapes / order fixed by the reference fixture (tests/golden/ddpm_path.pt
    holds the reference's shapes); seeded init bit-identical to the reference's; without a CUDA device the forward fails
    loudly (no CPU path); the shipped config builds it through PlDdim."""
    from mcedm_b200.ddpm_blocks import Model

    cfg = compose("config_ddim_res32")
    hp = copy.deepcopy(cfg.model.hparams)
    assert hp.name == "ddim"
    torch.manual_seed(1)
    net = Model(hp)
    assert (net.x_channels, net.cat_channels, net.out_channels) == (2, 2, 2)
    sd = net.state_dict()
    shapes = golden("ddpm_path.pt")["shapes"]
    assert list(sd) == list(shapes) and all(tuple(sd[k].shape) == tuple(v) for k, v in shapes.items())
    assert sum(v.numel() for v in sd.values()) == 1568514
    assert state_hash(sd) == REF_DDPM_MODEL_INIT_HASH                  # seeded init is bit-identical
    if not torch.cuda.is_available():
        import pytest

        with pytest.raises(Exception):                 # McedmError: parameters / inputs must live on a CUDA device
            with torch.no_grad():
                net.eval()(torch.zeros(1, 2, 128, 128), torch.zeros(1))
    from mcedm_b200.ddim import PlDdim

    torch.manual_seed(1)
    pl = PlDdim(copy.deepcopy(cfg.model.hparams))
    assert isinstance(pl.model, Model) and list(pl.model.state_dict()) == list(shapes)


def test_reference_arm_contract_under_torchrun_env():
    """`bench.py --impl reference`: rank 0 prints exactly one JSON object on stdout (banners go to stderr), every other
    rank exits 0 without output."""
    import json

    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == ""
    env["RANK"] = "0"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--timesteps", "3", "--gpus", "2"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    d = json.loads(r.stdout)                                   # the whole of stdout is one JSON object
    assert d["impl"] == "reference" and d["unit"] == "fields/s" and d["n_gpus"] == 2 and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["cpu_baseline"]["kind"] == "port"


def test_trainer_resume_matches_uninterrupted_run(tmp_path):
    """`Trainer.fit(ckpt_path=last.ckpt)` continues like the reference's `trainer.fit(ckpt_path=...)` (run.py:99):
    weights, Adam moments + step counter, global step and the NEXT epoch — 2 epochs + resume for 1 == 3 epochs."""
    from mcedm_b200.runner import ModelCheckpoint, Trainer, _ShimLightningModule

    class Tiny(_ShimLightningModule):
        def __init__(self):
            super().__init__()
            torch.manual_seed(0)
            self.lin = torch.nn.Linear(4, 3)

        def configure_optimizers(self):
            return {"optimizer": torch.optim.Adam(self.parameters(), lr=1e-2)}

        def training_step(self, batch, idx):
            x, y = batch
            loss = ((self.lin(x) - y) ** 2).mean()
            self.log("train_loss", loss)
            return loss

        def validation_step(self, batch, idx):
            return {}

    class DM:
        def setup(self, stage):
            g = torch.Generator().manual_seed(3)
            self.batches = [(torch.randn(8, 4, generator=g), torch.randn(8, 3, generator=g)) for _ in range(3)]

        def train_dataloader(self):
            return self.batches

        def val_dataloader(self):
            return []

    full = Tiny()
    Trainer(max_epochs=3, gradient_clip_val=1.0).fit(full, DM())
    part = Tiny()
    cb = ModelCheckpoint(dirpath=str(tmp_path), filename="{epoch}")
    Trainer(max_epochs=2, gradient_clip_val=1.0, callbacks=[cb]).fit(part, DM())
    assert os.path.exists(tmp_path / "epoch=0.ckpt") and os.path.exists(tmp_path / "epoch=1.ckpt")
    ckpt = torch.load(tmp_path / "last.ckpt", weights_only=False)
    for key in ("epoch", "global_step", "pytorch-lightning_version", "state_dict", "optimizer_states", "lr_schedulers",
                "hyper_parameters", "loops", "callbacks"):
        assert key in ckpt, key
    assert ckpt["epoch"] == 1 and ckpt["global_step"] == 6
    resumed = Tiny()
    with torch.no_grad():
        for p in resumed.parameters():
            p.add_(1.0)                                         # must be overwritten by the checkpoint
    tr = Trainer(max_epochs=3, gradient_clip_val=1.0)
    hist = tr.fit(resumed, DM(), ckpt_path=str(tmp_path / "last.ckpt"))
    assert len(hist) == 1 and resumed.current_epoch == 2 and resumed.global_step == 9
    assert int(tr.optimizer.state_dict()["state"][0]["step"]) == 9
    for a, b in zip(full.parameters(), resumed.parameters()):
        assert torch.equal(a, b)
