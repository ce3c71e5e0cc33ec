"""GPU: dynamic loss scaling on the fp16 training plan (mcedm_b200/loss_scale.py) at B = 32, eager and graph-replayed.

Gradients that apply are held to the bars of test_gpu_train_batch.py against its float64 reference (imported)."""
import ctypes as C
import math
import os
import subprocess
import sys

import pytest
import torch

from test_gpu_train_batch import TOL, _compare, _inputs, _module, _named_params, _step, _with_env, reference_step

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B = 32


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda")


def _setup(dev, graph, scaler=None):
    pl, mcfg = _module(dev)
    pl.use_cuda_graph = graph
    opt = pl.configure_optimizers()["optimizer"]
    opt.max_grad_norm = 1.0                           # the Trainer's gradient_clip_val
    pl.model.engine().loss_scaler = scaler
    return pl, mcfg, opt


def _state(pl, opt):
    """(p, m, v, ema) flat copies"""
    ema = torch.cat([p.detach().flatten() for p in pl.ema_model.ma_model.parameters()])
    return opt.flat_params().clone(), opt._m.clone(), opt._v.clone(), ema.clone()


def _train_step(pl, opt, inp):
    loss, grads = _step(pl, inp)
    flat = pl.model.engine().flat_grad().clone()
    pl.optimizer_step(0, 0, opt)
    return loss, grads, flat


@gpu
@pytest.mark.parametrize("graph", [False, True])
def test_dynamic_without_overflow_is_the_static_path_bit_for_bit(dev, graph):
    """(a) init_scale 1024 (the static scale), no overflow, no growth: flat gradient and p, m, v after each of 3 clipped
    Adam steps are bit-identical to the static path."""
    from mcedm_b200.loss_scale import LossScaler

    pl_s, _, opt_s = _setup(dev, graph)
    sc = LossScaler()
    pl_d, _, opt_d = _setup(dev, graph, sc)
    assert torch.equal(opt_s.flat_params(), opt_d.flat_params())
    for it in range(3):
        inp = _inputs(pl_s, dev, B, seed=300 + it)
        _, _, g_s = _train_step(pl_s, opt_s, inp)
        inp = _inputs(pl_d, dev, B, seed=300 + it)
        _, _, g_d = _train_step(pl_d, opt_d, inp)
        assert torch.isfinite(g_s).all()
        assert torch.equal(g_s, g_d), it
        for a, b, name in zip(_state(pl_s, opt_s), _state(pl_d, opt_d), ("p", "m", "v", "ema")):
            assert torch.equal(a, b), (it, name)
    assert sc.get_scale() == 1024.0 and sc.get_growth_tracker() == 3 and float(sc.found_inf_t) == 0.0
    assert opt_d.state_dict()["state"][0]["step"] == opt_s.state_dict()["state"][0]["step"] == 3


@gpu
@pytest.mark.parametrize("graph", [False, True])
def test_head_overflow_skips_then_backs_off_until_a_step_applies(dev, graph):
    """(b) S = 2^40 overflows S * dL/dF at the head: the step is skipped (p, m, v and the applied-step count unchanged
    bit for bit, EMA as the torch expression, scale halved); later steps back off until one applies, and that step's
    unscaled gradients meet the float64 reference's bars."""
    from mcedm_b200.loss_scale import LossScaler

    sc = LossScaler(init_scale=2.0 ** 40)
    pl, mcfg, opt = _setup(dev, graph, sc)
    inp = _inputs(pl, dev, B, seed=400)
    beta = pl.ema_model.beta
    p0, m0, v0, e0 = _state(pl, opt)
    _, _, g = _train_step(pl, opt, inp)
    assert not torch.isfinite(g).all()
    p1, m1, v1, e1 = _state(pl, opt)
    assert torch.equal(p0, p1) and torch.equal(m0, m1) and torch.equal(v0, v1)
    torch.testing.assert_close(e1, e0 * beta + (1 - beta) * p0, rtol=1e-6, atol=1e-7)
    assert float(sc.found_inf_t) == 1.0 and sc.get_scale() == 2.0 ** 39 and sc.get_growth_tracker() == 0
    assert int(opt._step_dev) == 0
    scale = 2.0 ** 39
    ref = reference_step(_named_params(pl), mcfg, *inp)      # the parameters do not move until a step applies
    for it in range(40):
        p0 = opt.flat_params().clone()
        loss, grads, g = _train_step(pl, opt, inp)
        if float(sc.found_inf_t) == 0.0:
            break
        scale /= 2
        assert sc.get_scale() == scale and torch.equal(p0, opt.flat_params()) and int(opt._step_dev) == 0
    else:
        pytest.fail("no step applied")
    print(f"first applied step at S = 2^{int(math.log2(scale))} after {it + 1} skips")
    _compare(pl, loss, grads, ref, f"first applied step, S = 2^{int(math.log2(scale))}")
    assert int(opt._step_dev) == 1 and opt.state_dict()["state"][0]["step"] == 1
    assert sc.get_scale() == scale and sc.get_growth_tracker() == 1
    assert not torch.equal(p0, opt.flat_params())


def _max_dF(pl, inp):
    eng = pl.model.engine()
    seen = []
    orig = eng.backward

    def spy(dF):
        seen.append(float(dF.abs().max()))
        return orig(dF)

    eng.backward = spy
    try:
        _step(pl, inp)
    finally:
        eng.backward = orig
    return seen[0]


@gpu
def test_interior_overflow_skips(dev):
    """(c) S keeps S * max|dL/dF| below 65504 (the head stores stay finite), but the static path at that S saturates
    inside the backward (MCEDM_DBG=4 audit > 0): the dynamic step at that S is skipped."""
    from mcedm_b200 import _lib as L
    from mcedm_b200.loss_scale import LossScaler

    pl, _, opt = _setup(dev, False)
    inp = _inputs(pl, dev, B, seed=500)
    m = _max_dF(pl, inp)
    k = math.floor(math.log2(65504.0 / m))
    S = 2.0 ** k
    assert S * m < 65504.0 <= 2 * S * m
    eng = pl.model.engine()
    eng.LOSS_SCALE = S                                # the static path at S
    lib, cnt = L.lib(), C.c_longlong(0)

    def audited():
        L.check(lib.mcedm_saturation_count(C.byref(cnt), 1, L.stream_ptr()))
        _step(pl, inp)
        torch.cuda.synchronize()
        L.check(lib.mcedm_saturation_count(C.byref(cnt), 1, L.stream_ptr()))
        return cnt.value

    n_sat = _with_env("MCEDM_DBG", "4", audited)
    print(f"max|dL/dF| = {m:.4g}, S = 2^{k}, saturated interior gradient values at S: {n_sat}")
    assert n_sat > 0
    del eng.LOSS_SCALE
    sc = LossScaler(init_scale=S)
    eng.loss_scaler = sc
    p0 = opt.flat_params().clone()
    _, _, g = _train_step(pl, opt, inp)
    assert not torch.isfinite(g).all()
    assert float(sc.found_inf_t) == 1.0 and sc.get_scale() == S / 2
    assert torch.equal(p0, opt.flat_params()) and int(opt._step_dev) == 0


@gpu
def test_growth_keeps_gradients_within_the_bars(dev):
    """(d) growth_interval = 2: the scale doubles after two applied steps, and the step at the doubled scale meets the
    float64 reference's bars."""
    from mcedm_b200.loss_scale import LossScaler

    sc = LossScaler(growth_interval=2)
    pl, mcfg, opt = _setup(dev, True, sc)
    for it in range(3):
        inp = _inputs(pl, dev, B, seed=600 + it)
        ref = reference_step(_named_params(pl), mcfg, *inp)
        loss, grads, _ = _train_step(pl, opt, inp)
        _compare(pl, loss, grads, ref, f"step {it}")
        assert float(sc.found_inf_t) == 0.0
        assert sc.get_scale() == (1024.0 if it == 0 else 2048.0), (it, sc.get_scale())
    assert int(opt._step_dev) == 3


def _sequence(dev, graph, n):
    from mcedm_b200.loss_scale import LossScaler

    sc = LossScaler(init_scale=2.0 ** 40, growth_interval=2)
    pl, _, opt = _setup(dev, graph, sc)
    inps = [_inputs(pl, dev, B, seed=700 + i) for i in range(2)]
    skips = []
    for it in range(n):
        _train_step(pl, opt, inps[it % 2])
        skips.append(float(sc.found_inf_t))
    return pl, opt, sc, skips


@gpu
def test_skip_and_growth_sequence_is_identical_eager_and_replayed(dev):
    """(e) a sequence with skips, applied steps and a growth gives bit-identical p, m, v, EMA, scale, tracker and
    applied-step count eagerly and as CUDA-graph replays."""
    pl_e, opt_e, sc_e, skips_e = _sequence(dev, False, 40)
    n_applied = skips_e.count(0.0)
    print(f"skips {skips_e.count(1.0)}, applied {n_applied}, final scale {sc_e.get_scale()}")
    assert skips_e[0] == 1.0 and n_applied >= 3          # a skip, then applied steps including a growth
    pl_g, opt_g, sc_g, skips_g = _sequence(dev, True, 40)
    assert skips_g == skips_e
    for a, b, name in zip(_state(pl_e, opt_e), _state(pl_g, opt_g), ("p", "m", "v", "ema")):
        assert torch.equal(a, b), name
    assert sc_e.state_dict() == sc_g.state_dict()
    assert int(opt_e._step_dev) == int(opt_g._step_dev) == n_applied


@gpu
def test_steady_state_step_does_not_synchronise(dev):
    """(f) a graph-replayed training step with its dynamic Adam step and scale update runs under
    torch.cuda.set_sync_debug_mode("error")."""
    from mcedm_b200.loss_scale import LossScaler

    pl, _, opt = _setup(dev, True, LossScaler())
    inp = _inputs(pl, dev, B, seed=800)
    for _ in range(2):
        _train_step(pl, opt, inp)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        x, sigma, noise, cond, mask = inp
        pl.zero_grad(set_to_none=True)
        loss = pl.forward_loss(x, sigma, noise, cond, mask, pl.get_loss_weight(sigma))
        loss.backward()
        pl.optimizer_step(0, 0, opt)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert int(opt._step_dev) == 3


@gpu
@pytest.mark.parametrize("dropout", [0.0, 0.1])
def test_trainer_precision16_skips_checkpoints_and_resumes(dev, tmp_path, dropout):
    """(g) Trainer(precision=16) trains with a forced initial skip (init_scale 2^40), checkpoints
    `native_amp_scaling_state`, and fit(ckpt_path=...) restores scale, tracker and the applied-step count."""
    from test_gpu_dropout import _pl

    from mcedm_b200 import _lib as L
    from mcedm_b200.data import SyntheticMaskDatamodule
    from mcedm_b200.loss_scale import LossScaler
    from mcedm_b200.runner import ModelCheckpoint, Trainer

    def dm():
        return SyntheticMaskDatamodule(system="swe_per", n_train=8, n_test=2, batch_size=4)

    pl, _, _ = _pl(dev, dropout)
    pl.sparams.timesteps = 3
    sc = LossScaler(init_scale=2.0 ** 40)
    pl.model.engine().loss_scaler = sc
    tr = Trainer(max_epochs=16, precision=16, check_val_every_n_epoch=16,
                 callbacks=[ModelCheckpoint(dirpath=str(tmp_path))])
    tr.fit(pl, dm())
    assert pl.model.engine().loss_scaler is sc and tr.loss_scaler(pl) is sc
    applied = tr.optimizer.state_dict()["state"][0]["step"]
    print(f"dropout {dropout}: {pl.global_step} steps, {int(applied)} applied, scale {sc.get_scale()}")
    assert pl.global_step == 32 and 0 < applied < 32
    state = torch.load(os.path.join(tmp_path, "last.ckpt"), map_location="cpu", weights_only=False)
    assert state["native_amp_scaling_state"] == sc.state_dict()
    assert state["optimizer_states"][0]["state"][0]["step"] == applied
    assert all(torch.isfinite(v).all() for v in state["state_dict"].values() if v.is_floating_point())
    resumed, _, _ = _pl(dev, dropout)
    resumed.sparams.timesteps = 3
    tr2 = Trainer(max_epochs=16, precision="16-mixed")
    tr2.fit(resumed, dm(), ckpt_path=os.path.join(tmp_path, "last.ckpt"))      # the saved epoch was the last one
    sc2 = resumed.model.engine().loss_scaler
    assert sc2 is not sc and sc2.state_dict() == state["native_amp_scaling_state"]
    assert tr2.optimizer.state_dict()["state"][0]["step"] == applied
    assert torch.equal(tr2.optimizer.flat_params(), tr.optimizer.flat_params())
    tr3 = Trainer(max_epochs=17, precision=16, check_val_every_n_epoch=100)
    tr3.fit(resumed, dm(), ckpt_path=os.path.join(tmp_path, "last.ckpt"))
    assert resumed.global_step == 34
    assert applied <= tr3.optimizer.state_dict()["state"][0]["step"] <= applied + 2
    L.check_watchdog()


@gpu
def test_data_parallel_ranks_skip_together(tmp_path):
    """(h) two ranks (gloo, one device): inf injected into rank 1's gradient before the flat all-reduce makes both
    ranks skip and halve their scales; the next step applies on both with identical parameters and scales."""
    script = os.path.join(ROOT, "tests", "dist_loss_scale_worker.py")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533", PYTHONPATH=ROOT)
    procs = [subprocess.Popen([sys.executable, script, str(r), "2", str(tmp_path)], env=env) for r in range(2)]
    codes = [p.wait(timeout=600) for p in procs]
    assert codes == [0, 0]
    res = [torch.load(os.path.join(tmp_path, f"rank{r}.pt")) for r in range(2)]
    assert res[0]["scales"] == res[1]["scales"] == [512.0, 512.0]
    assert res[0]["found_inf"] == res[1]["found_inf"] == [1.0, 0.0]
    assert torch.equal(res[0]["p"], res[1]["p"])
