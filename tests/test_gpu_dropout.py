"""Dropout in the fp16 training plan: the two kernels against the Philox oracle (tests/dropout_oracle.py), one training
step of the whole network against the float64 reference built with the same masks, and the module surface (eval mode
unchanged, sampling refuses a training-mode network, graph replay, resume)."""
import copy
import ctypes as C
import os

import pytest
import torch
import torch.nn.functional as F

import dropout_oracle as DO

gpu = pytest.mark.gpu
SEED = 0x0123_4567_89AB_CDEF


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def L():
    from mcedm_b200 import _lib

    _lib.lib()
    return _lib


def _geom(L, H, W):
    p, b = C.c_int(0), C.c_int(0)
    L.check(L.lib().mcedm_flat_geometry(H, W, C.byref(p), C.byref(b)))
    L.LAUNCHES[0] -= 1
    return p.value, b.value


def _flat_index(B, H, W, pitch, blk, dev):
    """storage position of every (b, y, x) of the padded-flat layout, [B, H, W]"""
    b = torch.arange(B, device=dev).view(B, 1, 1)
    y = torch.arange(H, device=dev).view(1, H, 1)
    x = torch.arange(W, device=dev).view(1, 1, W)
    return b * blk + (y + 1) * pitch + x


def _to_flat(t, pitch, blk):
    B, H, W, _ = t.shape
    out = torch.zeros(B * blk, 64, device=t.device, dtype=t.dtype)
    out[_flat_index(B, H, W, pitch, blk, t.device).flatten()] = t.reshape(-1, 64)
    return out


def _from_flat(f, B, H, W, pitch, blk):
    return f[_flat_index(B, H, W, pitch, blk, f.device).flatten()].reshape(B, H, W, 64)


def _padding_of(f, B, H, W, pitch, blk):
    keep = torch.ones(f.shape[0], dtype=torch.bool, device=f.device)
    keep[_flat_index(B, H, W, pitch, blk, f.device).flatten()] = False
    return f[keep]


def _rng(dev, seed, step):
    s = seed & (2 ** 64 - 1)
    v = [s & 0xFFFFFFFF, s >> 32, step & 0xFFFFFFFF]
    return torch.tensor([x - 2 ** 32 if x >= 2 ** 31 else x for x in v], dtype=torch.int32, device=dev)


def _apply(L, x, coef, p, layer, rng, flat=None):
    """mcedm_gn_apply16_dropout of fp16 x [B, H, W, 64] (dense, or converted to padded-flat) -> dense fp16 output"""
    B, H, W, _ = x.shape
    if flat is None:
        src, out, lay = x, torch.zeros_like(x), (0, 0)
    else:
        src, lay = _to_flat(x, *flat), flat
        out = torch.zeros_like(src)
    L.check(L.lib().mcedm_gn_apply16_dropout(L.ptr(src), lay[0], lay[1], L.ptr(coef), B, H, W, lay[0], lay[1], L.ptr(out),
                                             DO.threshold(p), DO.scale(p), layer, L.ptr(rng), 1, L.stream_ptr()))
    if flat is None:
        return out, None
    return _from_flat(out, B, H, W, *flat), _padding_of(out, B, H, W, *flat)


def _ulp16(v):
    """one fp16 ulp at |v| (subnormal spacing below 2^-14)"""
    e = torch.floor(torch.log2(v.abs().clamp_min(2.0 ** -14)))
    return torch.exp2(e - 10)


# ------------------------------------------------------------------------------------------------ 1./2. the kernels
LAYOUTS = [(128, False), (64, False), (64, True), (32, False), (32, True)]


@gpu
@pytest.mark.parametrize("H,flat", LAYOUTS)
def test_gn_apply16_dropout_against_the_oracle(L, dev, H, flat):
    """Zero pattern = keep_mask exactly wherever silu != 0, values within 1 fp16 ulp of fp32 silu(a x + b) * s, dense and
    padded-flat masks of the same field identical, padding positions still 0."""
    W = H
    geom = _geom(L, H, W) if H <= 64 else None
    for B in (1, 5, 32):
        for p in (0.1, 0.5):
            g = torch.Generator().manual_seed(B * 1000 + H + int(p * 10))
            x = (torch.randn(B, H, W, 64, generator=g) * 2).to(dev).half()
            coef = torch.cat([torch.rand(B, 64, generator=g) + 0.5, torch.rand(B, 64, generator=g) * 2 - 1], 1).to(dev)
            layer, step = (B + H) % 15, 1000 + B
            rng = _rng(dev, SEED, step)
            y, pad = _apply(L, x, coef, p, layer, rng, geom if flat else None)
            keep = DO.keep_mask(SEED, step, layer, B, H, W, p, device=dev).permute(0, 2, 3, 1)
            u = x.float() * coef[:, None, None, :64] + coef[:, None, None, 64:]
            want = F.silu(u) * DO.scale(p)
            nz = want.half() != 0
            assert torch.equal((y != 0) & nz, keep & nz), (B, p)
            err = (y.float() - want).abs()
            assert bool((err[keep] <= _ulp16(want[keep])).all()), (B, p, float(err[keep].max()))
            assert bool((y[~keep] == 0).all())
            if flat:
                assert bool((pad == 0).all())
                y_dense, _ = _apply(L, x, coef, p, layer, rng, None)
                assert torch.equal(y.view(torch.int16), y_dense.view(torch.int16))
    L.check_watchdog()


def _kernel_mask(L, dev, B, H, p, layer, seed, step):
    """the kernel's keep pattern on a field whose operand is nonzero everywhere (a = 0, b = 1: silu(1) * s)"""
    x = torch.zeros(B, H, H, 64, device=dev, dtype=torch.float16)
    coef = torch.cat([torch.zeros(B, 64), torch.ones(B, 64)], 1).to(dev)
    y, _ = _apply(L, x, coef, p, layer, _rng(dev, seed, step))
    return y != 0


@gpu
def test_dropout_keep_rate_and_independence(L, dev):
    """Keep fraction over 33.5 M elements within 5 sigma of 1 - p; masks of another layer, step or seed uncorrelated
    (|corr| within 5 sigma of 0)."""
    for p in (0.1, 0.5):
        m = _kernel_mask(L, dev, 32, 128, p, 3, SEED, 7)
        n = m.numel()
        sd = (p * (1 - p) / n) ** 0.5
        frac = float(m.float().mean())
        print(f"p={p}: keep fraction {frac:.6f} over {n} elements (1-p = {1 - p}, sigma {sd:.2e})")
        assert n >= 30_000_000 and abs(frac - (1 - p)) < 5 * sd
        a = m.float().flatten()
        for tag, other in (("layer", _kernel_mask(L, dev, 32, 128, p, 4, SEED, 7)),
                           ("step", _kernel_mask(L, dev, 32, 128, p, 3, SEED, 8)),
                           ("seed", _kernel_mask(L, dev, 32, 128, p, 3, SEED ^ 1, 7))):
            b = other.float().flatten()
            corr = float(((a - a.mean()) * (b - b.mean())).mean() / (a.std() * b.std()))
            print(f"p={p}: correlation with another {tag}: {corr:.2e}")
            assert abs(corr) < 5 / n ** 0.5, (tag, corr)


@gpu
@pytest.mark.parametrize("H,flat", LAYOUTS)
def test_dropout_bwd16_against_the_oracle(L, dev, H, flat):
    """In place g <- fp16(g * s) where kept, 0 elsewhere: exact, in both layouts, padding untouched."""
    W = H
    geom = _geom(L, H, W) if flat else None
    for B, p in ((1, 0.1), (5, 0.5), (32, 0.1)):
        g = (torch.randn(B, H, W, 64, generator=torch.Generator().manual_seed(B + H)) * 100).to(dev).half()
        layer, step = 14 - (B % 15), 3 + B
        buf = _to_flat(g, *geom) if flat else g.clone()
        L.check(L.lib().mcedm_dropout_bwd16(L.ptr(buf), geom[0] if flat else 0, geom[1] if flat else 0, B, H, W,
                                            DO.threshold(p), DO.scale(p), layer, L.ptr(_rng(dev, SEED, step)), 1,
                                            L.stream_ptr()))
        keep = DO.keep_mask(SEED, step, layer, B, H, W, p, device=dev).permute(0, 2, 3, 1)
        want = torch.where(keep, (g.float() * DO.scale(p)).half(), torch.zeros_like(g))
        got = _from_flat(buf, B, H, W, *geom) if flat else buf
        assert torch.equal(got.view(torch.int16), want.view(torch.int16)), (B, p)
        if flat:
            assert bool((_padding_of(buf, B, H, W, *geom) == 0).all())
    L.check_watchdog()


# ------------------------------------------------------------------------------------------------ 3.-8. the network
P = 0.1


def _pl(dev, p, config="config_adm_edm_mcedm_res32", cls=None):
    """The stress module of tests/common.py (seed-1 init, zero-init tensors randomised) with `dropout: p`."""
    from common import hparams
    from mcedm_b200 import data as D
    from mcedm_b200.mcedm import PlMcedm
    from mcedm_b200.utils import randomize_zero_init

    cfg = hparams(config)
    h = copy.deepcopy(cfg.model.hparams)
    h.model.dropout = p
    torch.manual_seed(1)
    pl = (cls or PlMcedm)(h)
    randomize_zero_init(pl.model, 2)
    pl.ema_model.ma_model.load_state_dict(pl.model.state_dict())
    pl = pl.to(dev).train()
    if config == "config_adm_edm_mcedm_res32":
        st = D.field_stats("swe_per", 16)
        pl.normalizer_input.set_stats(st["input_mean"].to(dev), st["input_std"].to(dev))
        pl.normalizer_target.set_stats(st["target_mean"].to(dev), st["target_std"].to(dev))
    return pl, dict(h.model), cfg


def _named(pl):
    return {k: p.detach().clone() for k, p in pl.model.named_parameters()}


def _set(eng, seed, step):
    eng.dropout_seed, eng.dropout_step = seed, step


def _same(a, b):
    return torch.equal(a[0], b[0]) and all(torch.equal(x, y) for x, y in zip(a[1], b[1]))


@gpu
@pytest.mark.parametrize("B", [2, 16, 32])
def test_training_step_with_dropout_matches_fp64_reference(dev, L, B):
    """p = 0.1: one step against the float64 reference built with the masks the kernels drew (keep_mask of the
    engine's seed and step, which the kernel tests above pin), at the bars of test_gpu_train_batch.  Eager with the
    weight-gradient side stream, eager without it, and graph-replayed: bit-identical for the same {seed, step}; then
    one eager step under MCEDM_DBG=4 leaves the fp16 saturation counter at 0."""
    from test_gpu_train_batch import _compare, _inputs, _step, _with_env

    pl, mcfg, _ = _pl(dev, P)
    eng = pl.model.engine()
    inp = _inputs(pl, dev, B, seed=300 + B)
    step = 5 + B
    masks = DO.network_masks(SEED, step, mcfg, B, P, device=dev)
    ref = DO.reference_step_dropout(_named(pl), mcfg, *inp, masks, DO.scale(P))
    pl.use_cuda_graph = False
    _set(eng, SEED, step)
    a = _step(pl, inp)
    assert eng.dropout_step == step + 1
    _compare(pl, a[0], a[1], ref, f"B={B} p={P} eager, side stream")
    _set(eng, SEED, step)
    b = _with_env("MCEDM_WGRAD_SIDE", "0", lambda: _step(pl, inp))
    pl.use_cuda_graph = True
    _set(eng, SEED, step)
    c = _step(pl, inp)
    assert eng.dropout_step == step + 1
    L.check_watchdog()
    assert _same(b, a), "side stream off"
    assert _same(c, a), "graph"
    pl.use_cuda_graph = False
    lib = L.lib()
    cnt = C.c_longlong(0)

    def audited():
        L.check(lib.mcedm_saturation_count(C.byref(cnt), 1, L.stream_ptr()))
        _set(eng, SEED, step)
        _step(pl, inp)
        torch.cuda.synchronize()
        L.check(lib.mcedm_saturation_count(C.byref(cnt), 1, L.stream_ptr()))
        return cnt.value

    assert _with_env("MCEDM_DBG", "4", audited) == 0
    L.check_watchdog()


@gpu
def test_graph_steps_draw_new_masks_and_replay_reproduces(dev, L):
    """Two consecutive graph-replayed steps on the same inputs draw different masks (different gradients); resetting
    the step and replaying reproduces the first step's gradients bit for bit."""
    from test_gpu_train_batch import _inputs, _step

    pl, _, _ = _pl(dev, P)
    eng = pl.model.engine()
    pl.use_cuda_graph = True
    inp = _inputs(pl, dev, 16, seed=401)
    _set(eng, SEED, 0)
    first = _step(pl, inp)
    second = _step(pl, inp)
    assert eng.dropout_step == 2
    assert not torch.equal(first[0], second[0])
    assert sum(not torch.equal(x, y) for x, y in zip(first[1], second[1])) > 100
    eng.dropout_step = 0
    again = _step(pl, inp)
    assert _same(again, first)
    L.check_watchdog()


@gpu
def test_eval_mode_ignores_dropout_and_sampling_refuses_training_mode(dev, L):
    """Eval mode: p = 0.1 gives the bits of the same weights at p = 0, for get_denoised and a 3-step sample_edm.  In
    training mode sample_edm and guided get_denoised raise instead of sampling without dropout."""
    from common import NoiseFeed

    pls = [_pl(dev, p) for p in (0.0, P)]
    cfg = pls[0][2]
    g = torch.Generator().manual_seed(9)
    xt = torch.randn(2, 2, 128, 128, generator=g).to(dev)
    cond = torch.randn(2, 2, 128, 128, generator=g).to(dev)
    mask = (torch.rand(2, 2, 128, 128, generator=g) > 0.5).float().to(dev)
    sp = copy.deepcopy(cfg.diff_sampler)
    sp.timesteps = 3
    outs = []
    for pl, _, _ in pls:
        pl.eval()
        with torch.no_grad():
            d, f = pl.get_denoised(pl.model, xt, torch.tensor([0.5, 7.0], device=dev), cond)
        pl._noise_hook = NoiseFeed(5).hook
        xs = pl.sample_edm(torch.zeros_like(xt), cond, mask, sp, return_last=False)
        outs.append((d, f, xs))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    pl = pls[1][0]
    pl.train()
    with pytest.raises(NotImplementedError, match="eval mode"):
        pl.sample_edm(torch.zeros_like(xt), cond, mask, sp)
    with pytest.raises(NotImplementedError, match="eval mode"), torch.no_grad():
        pl.get_denoised(pl.model, xt, torch.tensor([0.5, 7.0], device=dev), cond, w=1.5)
    # a training-mode evaluation without autograd still applies dropout (and advances the step)
    eng = pl.model.engine()
    _set(eng, SEED, 0)
    with torch.no_grad():
        d_train, _ = pl.get_denoised(pl.model, xt, torch.tensor([0.5, 7.0], device=dev), cond)
    assert eng.dropout_step == 1 and eng._tape is None
    assert not torch.equal(d_train, outs[1][0])


@gpu
def test_dropout_zero_runs_the_plain_launch_sequence(dev, L):
    """p = 0 draws nothing: no rng words, no operand kept, and the step issues exactly 15 + 15 fewer launches than at
    p = 0.1 (one gn_apply16_dropout and one dropout_bwd16 per UNetBlock); its gradients match the float64 reference
    without masks, and p = 0.1 with every element kept (threshold 0, scale 1) is not what p = 0 runs."""
    from test_gpu_train_batch import _compare, _inputs, _step, reference_step

    counts = {}
    for p in (0.0, P):
        pl, mcfg, _ = _pl(dev, p)
        pl.use_cuda_graph = False
        eng = pl.model.engine()
        inp = _inputs(pl, dev, 16, seed=500)
        n0 = L.LAUNCHES[0]
        loss, grads = _step(pl, inp)
        counts[p] = L.LAUNCHES[0] - n0
        recs = eng._tape["blocks"] if eng._tape else []
        if p == 0.0:
            assert getattr(eng, "_rng_words", None) is None and eng.dropout_step == 0
            assert not any("op1" in r for r in recs)
            _compare(pl, loss, grads, reference_step(_named(pl), mcfg, *inp), "p=0")
        else:
            assert sum("op1" in r for r in recs) == 15
    assert counts[P] - counts[0.0] == 30, counts


@gpu
def test_cond_edm_training_step_with_dropout(dev, L):
    """PlCondEdm (no mask, condition h) at p = 0.1, B = 4: one eager step against the float64 reference."""
    from mcedm_b200.cond_edm import PlCondEdm
    from test_gpu_train_batch import _compare, _step

    pl, mcfg, _ = _pl(dev, P, "config_adm_edm_res32_cond_h", PlCondEdm)
    pl.cond_p = 1.0
    pl.use_cuda_graph = False
    eng = pl.model.engine()
    B = 4
    g = torch.Generator().manual_seed(44)
    u = torch.randn(B, 1, 128, 128, generator=g).to(dev)
    cond = torch.randn(B, pl.model.cond_channels, 128, 128, generator=g).to(dev)
    noise = torch.randn(B, 1, 128, 128, generator=g).to(dev)
    sigma = torch.tensor([0.01, 0.3, 2.0, 40.0]).view(B, 1, 1, 1).to(dev)
    ones = torch.ones_like(u)
    masks = DO.network_masks(SEED, 2, mcfg, B, P, device=dev)
    ref = DO.reference_step_dropout(_named(pl), mcfg, u, sigma, noise, cond, ones, masks, DO.scale(P))
    _set(eng, SEED, 2)
    pl.zero_grad(set_to_none=True)
    loss = pl.forward_loss(u, sigma, noise, cond, None, pl.get_loss_weight(sigma))
    loss.backward()
    _compare(pl, loss.detach(), [p.grad.detach().clone() for p in pl.model.parameters()], ref, "PlCondEdm p=0.1")


@gpu
def test_trainer_trains_validates_samples_and_resumes_with_dropout(dev, L, tmp_path):
    """A `dropout: 0.1` module through runner.Trainer: trains (graph-replayed steps), validates (eval mode, sampling),
    saves a checkpoint; fit(ckpt_path=...) resumes with the dropout step at the checkpoint's global_step, and the
    checkpoint loads with strict=True into a dropout 0 module."""
    from mcedm_b200.data import SyntheticMaskDatamodule
    from mcedm_b200.runner import ModelCheckpoint, Trainer

    pl, _, _ = _pl(dev, P)
    pl.sparams.timesteps = 3
    dm = SyntheticMaskDatamodule(system="swe_per", n_train=8, n_test=2, batch_size=4)
    Trainer(max_epochs=1, callbacks=[ModelCheckpoint(dirpath=str(tmp_path))]).fit(pl, dm)
    eng = pl.model.engine()
    assert pl.global_step == 2 and eng.dropout_step == 2
    assert any(k.startswith("val_mae") for k in pl.logged), list(pl.logged)
    ckpt = os.path.join(tmp_path, "last.ckpt")
    state = torch.load(ckpt, map_location="cpu", weights_only=False)
    assert state["global_step"] == 2 and len(state["state_dict"]) == 412
    pl0, _, _ = _pl(dev, 0.0)
    pl0.load_state_dict(state["state_dict"], strict=True)
    resumed, _, _ = _pl(dev, P)
    resumed.sparams.timesteps = 3
    tr = Trainer(max_epochs=2, max_steps=3)
    tr.fit(resumed, SyntheticMaskDatamodule(system="swe_per", n_train=8, n_test=2, batch_size=4), ckpt_path=ckpt)
    assert resumed.global_step == 3 and resumed.model.engine().dropout_step == 3
    L.check_watchdog()
