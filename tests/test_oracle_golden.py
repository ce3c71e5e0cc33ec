"""CPU: the oracle (oracle/edm_oracle.py) against fixtures produced by the unmodified reference."""
import pytest
import torch

from common import NoiseFeed, fixture_state, golden, hparams, stress_unet
from mcedm_b200 import data as D
from mcedm_b200.utils import rel_l2, state_hash
from oracle import edm_oracle as O


@pytest.fixture(autouse=True)
def fixture_thread_count():
    """torch's CPU reductions split their work by thread count, so the fp32 result depends on it: the fixtures were
    written with 8 threads, and the same count reproduces them bit for bit on any host (16 threads move a 4-step
    trajectory by 1.3e-6)."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def _sd_cfg(config="config_adm_edm_mcedm_res32"):
    net, cfg, init_hash = stress_unet(config)
    return {k: v.detach() for k, v in net.state_dict().items()}, dict(cfg.model.hparams.model), cfg, init_hash


def test_init_and_stress_weights_match_reference():
    g = golden("unet_forward.pt")
    sd, _, _, init_hash = _sd_cfg()
    assert init_hash == g["init_hash"], "seeded initialisation differs from the reference's"
    assert state_hash(sd) == g["stress_hash"]
    assert sum(v.numel() for k, v in sd.items() if "resample_filter" not in k) == g["n_params"] == 1587010


def test_oracle_unet_forward_matches_reference():
    g = golden("unet_forward.pt")
    sd, mcfg, _, _ = _sd_cfg()
    for case in g["cases"]:
        with torch.no_grad():
            y = O.unet_forward(sd, mcfg, case["x"], case["noise_labels"], case["cond"])
        assert rel_l2(y, case["out"]) < 1e-6
        assert case["out"].abs().max() > 0.5, "fixture must not be the vacuous zero-output network"


def test_oracle_cond_edm_network_matches_reference():
    g = golden("cond_edm_forward.pt")
    sd, mcfg, _, init_hash = _sd_cfg("config_adm_edm_res32_cond_h")
    assert init_hash == g["init_hash"] and state_hash(sd) == g["stress_hash"]
    with torch.no_grad():
        y = O.unet_forward(sd, mcfg, g["x"], g["noise_labels"], g["cond"])
    assert y.shape == (2, 1, 128, 128) and rel_l2(y, g["out"]) < 1e-6


def test_oracle_denoise_matches_reference():
    g = golden("denoise.pt")
    sd, mcfg, _, _ = _sd_cfg()
    for case in g["cases"]:
        with torch.no_grad():
            d, f = O.denoise(sd, mcfg, case["xt"], torch.tensor(case["sigma"], dtype=torch.float64), case["cond"])
        assert rel_l2(d, case["D"]) < 1e-6 and rel_l2(f, case["F"]) < 1e-6


def test_oracle_trajectory_matches_reference():
    g = golden("trajectory.pt")
    sd, mcfg, cfg, _ = _sd_cfg()
    state, _, _, _ = fixture_state()
    for tr in g["trajs"]:
        assert torch.equal(tr["state"], state), "synthetic field generator drifted from the fixture"
        feed = NoiseFeed(tr["seed"])
        mask = tr["mask"]
        cond_in = O.get_cond_in(state, mask, feed.draw(state)).permute(0, 3, 1, 2).contiguous()
        mask_c = mask.permute(0, 3, 1, 2).contiguous()
        hu_arg = feed.draw(mask_c)          # the caller's draw passed as `hu` (mcedm.py:373); only its shape is used
        hu_noise = feed.draw(hu_arg)        # the sampler's own initial noise (mcedm.py:576)
        sp = dict(cfg.diff_sampler)
        sp["timesteps"] = tr["steps"]
        rec = []
        with torch.no_grad():
            xs = O.sample_edm(sd, mcfg, hu_noise, cond_in, mask_c, sp, lambda i, x: feed.draw(x), record=rec)
        assert feed.calls == tr["calls"], "RNG call sequence (shapes/dtypes/order) differs from the reference"
        assert len(rec) == len(tr["denoised"])
        for (i, which, sigma, d), ref in zip(rec, tr["denoised"]):
            assert abs(sigma - ref["sigma"]) <= 1e-6 * max(1.0, abs(ref["sigma"]))
            assert rel_l2(d, ref["D"]) < 1e-5
        assert xs.dtype == torch.float64 and xs.shape == tr["xs"].shape
        assert rel_l2(xs, tr["xs"]) < 1e-6
        # observed entries (mask == 0) keep their clean value bit-exactly through the trajectory
        known = mask == 0
        assert torch.equal(xs[:, -1][known], state.double()[known])


def test_oracle_training_loss_matches_reference():
    g = golden("train_step.pt")
    sd, mcfg, _, _ = _sd_cfg()
    B = g["mask"].shape[0]
    state, _, _, _ = fixture_state(n=B, seed=g["seed_fields"])
    feed = NoiseFeed(g["noise_seed"])
    mask = g["mask"]
    cond = O.get_cond_in(state, mask, feed.draw(state)).permute(0, 3, 1, 2).contiguous()
    x = state.permute(0, 3, 1, 2).contiguous()
    noise = feed.draw(x)
    torch.manual_seed(g["cpu_seed"])
    sigma = (torch.randn([B, 1, 1, 1]) * 1.2 - 1.2).exp()
    with torch.no_grad():
        loss, _ = O.training_loss(sd, mcfg, x, sigma, noise, cond, mask.permute(0, 3, 1, 2).contiguous())
    assert abs(float(loss) - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))


def test_mask_generators_bit_identical():
    g = golden("masks.pt")
    _, h, u, _ = fixture_state()
    torch.manual_seed(g["train_seed"])
    mine = torch.stack([D.sample_mask(h[0], u[0], True) for _ in range(8)])
    assert torch.equal(mine.to(torch.uint8), g["train_masks"])
    torch.manual_seed(g["train_seed"])
    coins = [float(torch.rand(1)) for _ in range(8)]
    orc = torch.stack([O.train_mask(h[0], u[0], c) for c in coins])
    assert torch.equal(orc.to(torch.uint8), g["train_masks"])
    torch.manual_seed(g["time_seed"])
    mine_t = torch.stack([D.sample_time_mask(h[0], u[0], True) for _ in range(8)])
    assert torch.equal(mine_t.to(torch.uint8), g["time_train"])
    # the same masks as two observation rows per item (device-side generation, data.sample_*_rows): same RNG calls, and
    # their expansion is the reference-generated mask bit for bit
    torch.manual_seed(g["train_seed"])
    rows = torch.stack([D.sample_mask_rows(128) for _ in range(8)])
    assert torch.equal(D.expand_mask_rows(rows, 128, 128).to(torch.uint8), g["train_masks"])
    torch.manual_seed(g["train_seed"])
    [D.sample_mask(h[0], u[0], True) for _ in range(8)]
    after_ref = torch.rand(1)
    torch.manual_seed(g["train_seed"])
    [D.sample_mask_rows(128) for _ in range(8)]
    assert torch.equal(torch.rand(1), after_ref)                      # generator left in the same state
    torch.manual_seed(g["time_seed"])
    rows_t = torch.stack([D.sample_time_mask_rows(128) for _ in range(8)])
    assert torch.equal(D.expand_mask_rows(rows_t, 128, 128).to(torch.uint8), g["time_train"])
    ev = D.sample_mask(h[0], u[0], False)
    assert torch.equal(ev["u"].to(torch.uint8), g["eval_u"]) and torch.equal(ev["h"].to(torch.uint8), g["eval_h"])
    oe = O.eval_masks(h[0], u[0])
    assert torch.equal(oe["u"].to(torch.uint8), g["eval_u"]) and torch.equal(oe["h"].to(torch.uint8), g["eval_h"])
    te = D.sample_time_mask(h[0], u[0], False, add_time_masks=True)
    ot = O.time_eval_masks(h[0], u[0])
    for k in ("hu", "u", "h"):
        assert torch.equal(te[k].to(torch.uint8), g["time_eval"][k])
        assert torch.equal(ot[k].to(torch.uint8), g["time_eval"][k])


def test_oracle_cond_edm_path_matches_reference():
    """Config 5 (PlCondEdm: u denoised, h as condition, no mask): the oracle's unmasked sampler and loss against the
    fixture produced by the unmodified reference (tests/golden/make_golden_cond.py)."""
    import copy

    from mcedm_b200 import data as D
    from oracle import edm_oracle as O

    g = golden("cond_edm_path.pt")
    net, cfg, _ = stress_unet("config_adm_edm_res32_cond_h")
    sd = {k: v.detach() for k, v in net.state_dict().items()}
    mcfg = dict(cfg.model.hparams.model)
    a, u = D._FIELDS["darcy"](2, 128, first_seed=g["field_seed"])
    a, u = torch.from_numpy(a), torch.from_numpy(u)
    st = g["stats"]
    h_n = ((a - st["input_mean"]) / st["input_std"]).permute(0, 3, 1, 2).contiguous()
    u_n = ((u - st["target_mean"]) / st["target_std"]).permute(0, 3, 1, 2).contiguous()
    # ---- sampler: same draws in the same order (u_noise fp32 b h w c, then one fp64 draw per step)
    feed = NoiseFeed(g["sample"]["seed"])
    u_noise = feed.draw(torch.empty(1, 128, 128, 1)).permute(0, 3, 1, 2).contiguous()
    sp = dict(copy.deepcopy(cfg.diff_sampler))
    sp["timesteps"] = g["sample"]["steps"]
    rec = []
    with torch.no_grad():
        xs = O.cond_sample_edm(sd, mcfg, u_noise, h_n[:1], sp, lambda i, x: feed.draw(x), record=rec)
    assert [tuple(c) for c in feed.calls] == [tuple(c) for c in g["sample"]["calls"]]
    assert len(rec) == len(g["sample"]["denoised"])
    for (i, which, sigma, d), ref in zip(rec, g["sample"]["denoised"]):
        assert abs(sigma - ref["sigma"]) <= 1e-9 * max(1.0, ref["sigma"])
        assert rel_l2(d, ref["D"]) < 1e-5
    assert rel_l2(xs, g["sample"]["xs"]) < 1e-5
    # ---- training loss: noise = randn_like(u) (NoiseFeed), sigma from the CPU RNG, one cond_p coin (cond_p = 1: kept)
    nf = NoiseFeed(g["train"]["noise_seed"])
    noise = nf.draw(u_n)
    torch.manual_seed(g["train"]["cpu_seed"])
    sigma = (torch.randn([2, 1, 1, 1]) * 1.2 - 1.2).exp()
    with torch.no_grad():
        loss, _ = O.cond_training_loss(sd, mcfg, u_n, sigma, noise, h_n)
    assert abs(float(loss) - float(g["train"]["loss"])) < 2e-5 * abs(float(g["train"]["loss"]))


def test_oracle_ddim_repaint_sampler_matches_reference():
    """BASELINE config 4 (PlDdim.sample_edm, n_time_h=0, n_time_u=64, n_repeat=2, ADM network with self_cond): the
    oracle's VP-grid sampler against the fixture produced by the unmodified reference (tests/golden/make_golden_ddim.py)."""
    import copy

    g = golden("ddim_path.pt")
    net, cfg, init_hash = stress_unet("config_adm_ddim_res32")
    assert init_hash == g["init_hash"]
    sd = {k: v.detach() for k, v in net.state_dict().items()}
    mcfg = dict(cfg.model.hparams.model)
    grid = O.VpGrid()
    assert abs(grid.sigma_min - g["sigma_min"]) < 1e-12 and abs(grid.sigma_max - g["sigma_max"]) < 1e-9
    h, u = D._FIELDS["swe"](1, 128, first_seed=g["field_seed"])
    st = g["stats"]
    hu = torch.cat([(torch.from_numpy(h) - st["input_mean"]) / st["input_std"],
                    (torch.from_numpy(u) - st["target_mean"]) / st["target_std"]], dim=-1).permute(0, 3, 1, 2).contiguous()
    s = g["sample"]
    sp = dict(copy.deepcopy(cfg.diff_sampler))
    sp.update(timesteps=s["steps"], n_time_h=s["n_time_h"], n_time_u=s["n_time_u"], n_repeat=s["n_repeat"])
    feed = NoiseFeed(s["seed"])
    hu_noise = feed.draw(hu)
    rec = []
    with torch.no_grad():
        xs = O.ddim_sample_edm(sd, mcfg, grid, hu, hu_noise, sp, feed.draw, record=rec)
    assert [tuple(c) for c in feed.calls] == [tuple(c) for c in s["calls"]]
    assert len(rec) == len(s["denoised"])
    for (i, k, which, sigma, d), ref in zip(rec, s["denoised"]):
        assert abs(sigma - ref["sigma"]) <= 1e-9 * max(1.0, ref["sigma"])
        assert rel_l2(d, ref["D"]) < 1e-5
    assert rel_l2(xs, s["xs"]) < 1e-5
    # the observed region (u for t < 64) is re-imposed exactly; the rest is generated
    assert torch.equal(xs[0, 0, :64, :, 1], hu[0, 1, :64].double())


def test_oracle_ddpm_unet_and_repaint_sampler_match_reference():
    """SURVEY §8f rank 2, oracle first: the DDPM U-Net (`ddim_blocks.Model`, what the shipped ddim_res32.yaml builds) and
    BASELINE config 4 through it — one network evaluation and a 3-step RePaint-conditioned PlDdim.sample_edm trajectory
    against the unmodified reference (tests/golden/make_golden_ddpm.py).  No CUDA path for this network yet."""
    from common import seeded_weights
    from mcedm_b200.utils import state_hash
    from oracle import ddpm_oracle as DO

    g = golden("ddpm_path.pt")
    sd = seeded_weights(g["shapes"], seed=3)
    assert state_hash(sd) == g["weights_hash"]
    mcfg = g["model_cfg"]
    gen = torch.Generator().manual_seed(g["forward"]["seed"])
    x = torch.randn(2, 2, 128, 128, generator=gen)
    with torch.no_grad():
        y = DO.ddpm_unet_forward(sd, mcfg, x, g["forward"]["t"])
    assert rel_l2(y, g["forward"]["y"]) < 1e-6
    grid = O.VpGrid()
    h, u = D._FIELDS["swe"](1, 128, first_seed=g["field_seed"])
    st = g["stats"]
    hu = torch.cat([(torch.from_numpy(h) - st["input_mean"]) / st["input_std"],
                    (torch.from_numpy(u) - st["target_mean"]) / st["target_std"]], dim=-1).permute(0, 3, 1, 2).contiguous()
    s = g["sample"]
    sp = dict(hparams("config_adm_ddim_res32").diff_sampler)
    sp.update(timesteps=s["steps"], n_time_h=s["n_time_h"], n_time_u=s["n_time_u"], n_repeat=s["n_repeat"])
    feed = NoiseFeed(s["seed"])
    hu_noise = feed.draw(hu)
    rec = []
    with torch.no_grad():
        xs = O.ddim_sample_edm(sd, mcfg, grid, hu, hu_noise, sp, feed.draw, record=rec, net=DO.ddpm_net)
    assert [tuple(c) for c in feed.calls] == [tuple(c) for c in s["calls"]]
    assert len(rec) == len(s["denoised"])
    for (i, k, which, sigma, d), ref in zip(rec, s["denoised"]):
        assert abs(sigma - ref["sigma"]) <= 1e-9 * max(1.0, ref["sigma"])
        assert rel_l2(d, ref["D"]) < 1e-5
    assert rel_l2(xs, s["xs"]) < 1e-5
    assert torch.equal(xs[0, 0, :64, :, 1], hu[0, 1, :64].double())


def test_oracle_ddim_sample_with_repeat_matches_reference():
    """PlDdim.sample_with_repeat (models/ddim.py:808-913) through the DDPM U-Net: the oracle against the unmodified
    reference (tests/golden/make_golden_ddim_repeat.py): per-evaluation network outputs, every x_t and x0 prediction."""
    from common import seeded_weights
    from oracle import ddpm_oracle as DO

    g = golden("ddim_repeat.pt")
    gd = golden("ddpm_path.pt")
    sd = seeded_weights(gd["shapes"], seed=3)
    mcfg = gd["model_cfg"]
    grid = O.VpGrid()
    h, u = D._FIELDS["swe"](1, 128, first_seed=g["field_seed"])
    st = g["stats"]
    hu = torch.cat([(torch.from_numpy(h) - st["input_mean"]) / st["input_std"],
                    (torch.from_numpy(u) - st["target_mean"]) / st["target_std"]], dim=-1).permute(0, 3, 1, 2).contiguous()
    sp = dict(hparams("config_ddim_res32").diff_sampler)
    sp.update(type="ddim", skip_type="uniform", eta=0.0, timesteps=g["steps"], n_time_h=g["n_time_h"],
              n_time_u=g["n_time_u"], n_repeat=g["n_repeat"])
    feed = NoiseFeed(g["seed"])
    hu_noise = feed.draw(hu)
    rec = []
    with torch.no_grad():
        xs, x0 = O.ddim_sample_with_repeat(sd, mcfg, grid, hu, hu_noise, sp, DO.ddpm_net, return_last=False, record=rec)
    assert [tuple(c) for c in feed.calls] == [tuple(c) for c in g["calls"]]
    assert len(rec) == len(g["evals"]) == 8
    for mine, ref in zip(rec, g["evals"]):
        assert mine["t"] == ref["t"] and (mine["x_self_cond"] is not None) == ref["self_cond"]
        assert rel_l2(mine["et"], ref["et"]) < 2e-5
    assert xs.shape == g["xs"].shape and x0.shape == g["x0_preds"].shape
    assert rel_l2(xs, g["xs"]) < 1e-4 and rel_l2(x0, g["x0_preds"]) < 1e-4
    assert torch.equal(xs[0, -1, :64, :, 1], hu[0, 1, :64])            # known region of the final state: exactly the data
