"""GPU tests of classifier-free guidance (CFG) in the EDM samplers (run with -m gpu on a B200).

Guided, every network evaluation is one batch of 2B rows: rows [0, B) with the condition, rows [B, 2B) with the all-zero
condition, both on the same input; the mcedm_edm_*_cfg kernels read F_w = (1+w)*F_c - w*F_u where their siblings read F.
Most of the path is checked bit for bit: the kernels against their torch expressions, w = -1 against unconditional
sampling, get_denoised against two separate evaluations, and the doubled batch against smaller ones (rows are
independent, DESIGN §6).  The network itself is checked per evaluation against the CPU oracle (tests/cfg_oracle.py) on
the input this path fed it: rel-L2 < 1e-2 on the fp16 inference plan, < 1e-4 on the fp32-accuracy plan."""
import copy
import math

import pytest
import torch

from cfg_oracle import combine, cond_sample_edm_cfg, denoise_cfg
from common import NoiseFeed, fixture_state, golden, hparams, stress_module
from mcedm_b200 import data as D
from mcedm_b200.utils import rel_l2
from oracle import edm_oracle as O
from oracle import pde_oracle as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def L():
    from mcedm_b200 import _lib

    _lib.lib()
    return _lib


def _cond_module(dev, stats=None):
    """PlCondEdm (config 5) with the stress weights, in eval mode; `stats` sets the normalisers and the SWE residual."""
    from mcedm_b200.cond_edm import PlCondEdm
    from mcedm_b200.utils import randomize_zero_init

    cfg = hparams("config_adm_edm_res32_cond_h")
    torch.manual_seed(1)
    pl = PlCondEdm(copy.deepcopy(cfg.model.hparams))
    randomize_zero_init(pl.model, 2)
    pl.ema_model.ma_model.load_state_dict(pl.model.state_dict())
    sd = {k: v.detach().clone() for k, v in pl.model.state_dict().items()}
    pl = pl.to(dev).eval()
    if stats is not None:
        pl.normalizer_input.set_stats(stats["input_mean"].to(dev), stats["input_std"].to(dev))
        pl.normalizer_target.set_stats(stats["target_mean"].to(dev), stats["target_std"].to(dev))
        pl.set_pde_loss_function("swe_per", False)
    return pl, cfg, sd


def _masked_inputs(B, seed, dev):
    """cond / mask of PlMcedm's eval masks: even rows have u missing, odd rows h missing."""
    g = torch.Generator().manual_seed(seed)
    state = torch.randn(B, 2, 128, 128, generator=g)
    mask = torch.zeros(B, 2, 128, 128)
    mask[0::2, 1] = 1.0
    mask[1::2, 0] = 1.0
    cond = state * (1 - mask) + torch.randn(B, 2, 128, 128, generator=g) * mask
    return cond.to(dev), mask.to(dev)


def _sparams(cfg, steps, w):
    sp = copy.deepcopy(cfg.diff_sampler)
    sp.timesteps, sp.w = steps, w
    return sp


# ----------------------------------------------------------------------------------------------- 1. kernels
@pytest.mark.parametrize("w", [0.0, -1.0, 0.5, 3.0])
def test_cfg_kernels_match_torch_expressions(L, dev, w):
    from mcedm_b200.mcedm import precond_scalars

    lib = L.lib()
    g = torch.Generator().manual_seed(21)
    B, C, H, W = 2, 2, 64, 128
    n = B * C * H * W
    x_cur = torch.randn(B, C, H, W, generator=g, dtype=torch.float64) * 40
    eps = torch.randn(B, C, H, W, generator=g, dtype=torch.float64)
    mask = (torch.rand(B, C, H, W, generator=g) > 0.3).float()
    F1 = torch.randn(2 * B, C, H, W, generator=g)              # [F_c | F_u]
    F2 = torch.randn(2 * B, C, H, W, generator=g)
    t_cur, t_next = 63.788, 56.7995
    t_hat = t_cur + 0.3 * t_cur
    cs, co, ci, _ = precond_scalars(t_hat)
    cs2, co2, ci2, _ = precond_scalars(t_next)
    coef = math.sqrt(t_hat ** 2 - t_cur ** 2)
    f32 = lambda v: torch.tensor(v, dtype=torch.float32)  # noqa: E731
    # torch (CPU) restatement
    x_hat = x_cur + coef * eps * mask
    x_in = f32(ci) * x_hat.float()
    Fw1, Fw2 = combine(F1[:B], F1[B:], w), combine(F2[:B], F2[B:], w)
    d1 = f32(cs) * x_hat.float() + f32(co) * Fw1
    d_cur = (x_hat - d1.double()) / t_hat
    x_e = x_hat + (t_next - t_hat) * d_cur * mask
    x_in2 = f32(ci2) * x_e.float()
    d2 = f32(cs2) * x_e.float() + f32(co2) * Fw2
    x_new = x_hat + (t_next - t_hat) * (0.5 * d_cur + 0.5 * (x_e - d2.double()) / t_next) * mask
    # kernels (device copies kept alive: L.ptr() only carries the address)
    x_cur_d, eps_d, mask_d, F1_d, F2_d = [t.to(dev).contiguous() for t in (x_cur, eps, mask, F1, F2)]
    s = L.stream_ptr()
    xh = torch.empty_like(x_cur_d)
    xin = torch.full((2 * B, C, H, W), float("nan"), device=dev)
    L.check(lib.mcedm_edm_churn_cfg(L.ptr(x_cur_d), L.ptr(eps_d), L.ptr(mask_d), coef, ci, n, L.ptr(xh), L.ptr(xin), s))
    assert torch.equal(xh.cpu(), x_hat)
    assert torch.equal(xin[:B].cpu(), x_in) and torch.equal(xin[B:].cpu(), x_in)
    dc, xe, Db = torch.empty_like(xh), torch.empty_like(xh), torch.empty(B, C, H, W, device=dev)
    xin.fill_(float("nan"))
    L.check(lib.mcedm_edm_euler_cfg(L.ptr(xh), L.ptr(F1_d), L.ptr(mask_d), t_hat, t_next, cs, co, ci2, w, n, L.ptr(dc),
                                    L.ptr(xe), L.ptr(xin), L.ptr(Db), s))
    assert torch.equal(Db.cpu(), d1) and torch.equal(dc.cpu(), d_cur) and torch.equal(xe.cpu(), x_e)
    assert torch.equal(xin[:B].cpu(), x_in2) and torch.equal(xin[B:].cpu(), x_in2)
    xn, D2b = torch.empty_like(xh), torch.empty_like(Db)
    L.check(lib.mcedm_edm_correct_cfg(L.ptr(xh), L.ptr(xe), L.ptr(F2_d), L.ptr(dc), L.ptr(mask_d), t_hat, t_next, cs2,
                                      co2, w, n, L.ptr(xn), L.ptr(D2b), s))
    assert torch.equal(D2b.cpu(), d2) and torch.equal(xn.cpu(), x_new)
    Dd = torch.empty_like(Db)
    L.check(lib.mcedm_edm_denoised_cfg(L.ptr(xh), L.ptr(F1_d), cs, co, w, n, L.ptr(Dd), s))
    assert torch.equal(Dd.cpu(), d1)
    # get_denoised's preconditioning: per-sample (stride 1) and shared (stride 0) coefficients
    x32 = x_hat.float().to(dev)
    csv, cov = torch.tensor([cs, cs2], device=dev), torch.tensor([co, co2], device=dev)
    for stride in (1, 0):
        Dp, Fp = torch.empty_like(Db), torch.empty_like(Db)
        L.check(lib.mcedm_edm_precond_out_cfg(L.ptr(x32), L.ptr(F1_d), L.ptr(csv), L.ptr(cov), stride, w, B, C * H * W,
                                              L.ptr(Dp), L.ptr(Fp), s))
        c_s = csv.cpu().reshape(B, 1, 1, 1) if stride else csv.cpu()[0]
        c_o = cov.cpu().reshape(B, 1, 1, 1) if stride else cov.cpu()[0]
        assert torch.equal(Fp.cpu(), Fw1) and torch.equal(Dp.cpu(), c_s * x32.cpu() + c_o * Fw1)
    # w = 0 gives the bits of the unguided sibling fed F_c, w = -1 those of the sibling fed F_u
    if w in (0.0, -1.0):
        half = F1_d[:B] if w == 0.0 else F1_d[B:]
        half2 = F2_d[:B] if w == 0.0 else F2_d[B:]
        half, half2 = half.contiguous(), half2.contiguous()
        dc0, xe0, Db0, xin0 = torch.empty_like(dc), torch.empty_like(xe), torch.empty_like(Db), torch.empty_like(Db)
        L.check(lib.mcedm_edm_euler(L.ptr(xh), L.ptr(half), L.ptr(mask_d), t_hat, t_next, cs, co, ci2, n, L.ptr(dc0),
                                    L.ptr(xe0), L.ptr(xin0), L.ptr(Db0), s))
        assert torch.equal(Db0, Db) and torch.equal(dc0, dc) and torch.equal(xe0, xe) and torch.equal(xin0, xin[:B])
        xn0, D20 = torch.empty_like(xn), torch.empty_like(Db)
        L.check(lib.mcedm_edm_correct(L.ptr(xh), L.ptr(xe), L.ptr(half2), L.ptr(dc), L.ptr(mask_d), t_hat, t_next, cs2,
                                      co2, n, L.ptr(xn0), L.ptr(D20), s))
        assert torch.equal(xn0, xn) and torch.equal(D20, D2b)
        Dd0 = torch.empty_like(Db)
        L.check(lib.mcedm_edm_denoised(L.ptr(xh), L.ptr(half), cs, co, n, L.ptr(Dd0), s))
        assert torch.equal(Dd0, Dd)
    torch.cuda.synchronize()


def test_cfg_kernels_reject_non_finite_w(L, dev):
    lib = L.lib()
    x = torch.zeros(4, device=dev, dtype=torch.float64)
    F = torch.zeros(8, device=dev)
    D = torch.empty(4, device=dev)
    with pytest.raises(L.McedmError, match="not finite"):
        L.check(lib.mcedm_edm_denoised_cfg(L.ptr(x), L.ptr(F), 0.5, 0.5, math.nan, 4, L.ptr(D), L.stream_ptr()))


# ----------------------------------------------------------------------------------------------- 2. w = -1
def test_cond_edm_w_minus_one_is_unconditional_sampling(dev):
    """PlCondEdm (all-ones mask: the known values never enter) at w = -1 returns the bits of the unguided sampler run
    on the all-zero condition."""
    pl, cfg, _ = _cond_module(dev)
    g = torch.Generator().manual_seed(8)
    h = torch.randn(2, 128, 128, 1, generator=g).to(dev)
    u_noise = torch.randn(2, 128, 128, 1, generator=g).to(dev)
    outs = []
    for cond, w in ((h, -1.0), (torch.zeros_like(h), 0.0)):
        pl._noise_hook = NoiseFeed(5).hook
        outs.append(pl.sample_edm(cond, u_noise, _sparams(cfg, 3, w), return_last=False))
    pl._noise_hook = None
    assert torch.isfinite(outs[0]).all()
    assert torch.equal(outs[0], outs[1])
    # and the condition does matter to this network: guidance off on `h` gives another trajectory
    pl._noise_hook = NoiseFeed(5).hook
    plain = pl.sample_edm(h, u_noise, _sparams(cfg, 3, 0.0), return_last=False)
    pl._noise_hook = None
    assert not torch.equal(plain, outs[0])


# ----------------------------------------------------------------------------------------------- 3. get_denoised
def test_get_denoised_cfg_matches_two_evaluations(dev):
    pl, _ = stress_module()
    pl = pl.to(dev).eval()
    cond, _ = _masked_inputs(2, 31, dev)
    g = torch.Generator().manual_seed(32)
    xt = (torch.randn(2, 2, 128, 128, generator=g) * 2).to(dev)
    w = 1.5
    for sigma in (torch.tensor(1.5, dtype=torch.float64), torch.tensor([0.3, 12.0], dtype=torch.float64)):
        with torch.no_grad():
            d_w, f_w = pl.get_denoised(pl.ema_model, xt, sigma, cond=cond, w=w)
            _, f_c = pl.get_denoised(pl.ema_model, xt, sigma, cond=cond, w=0.0)
            _, f_u = pl.get_denoised(pl.ema_model, xt, sigma, cond=None, w=0.0)
        # the preconditioning coefficients exactly as PlMcedm._precond_apply forms them (fp32 torch ops)
        s = sigma.to(dev).to(torch.float32).reshape(-1)
        den = s ** 2 + 1.0
        c_skip = (1.0 / den).reshape(-1, 1, 1, 1)
        c_out = (s * 1.0 / den.sqrt()).reshape(-1, 1, 1, 1)
        f_ref = combine(f_c.cpu(), f_u.cpu(), w)
        d_ref = c_skip.cpu() * xt.cpu() + c_out.cpu() * f_ref
        assert torch.equal(f_w.cpu(), f_ref) and torch.equal(d_w.cpu(), d_ref)
        assert not torch.equal(f_c, f_u)


# ----------------------------------------------------------------------------------------------- 4. RNG
def test_guidance_draws_no_extra_noise(dev):
    pl, cfg = stress_module()
    pl = pl.to(dev).eval()
    cond, mask = _masked_inputs(1, 41, dev)
    calls = []
    for w in (1.5, 0.0):
        feed = NoiseFeed(3)
        pl._noise_hook = feed.hook
        pl.sample_edm(torch.zeros(1, 2, 128, 128, device=dev), cond, mask, _sparams(cfg, 3, w))
        calls.append(feed.calls)
    pl._noise_hook = None
    assert calls[0] == calls[1] and len(calls[0]) == 4


# ----------------------------------------------------------------------------------------------- 5. row independence
def test_doubled_batch_keeps_rows_independent(dev):
    """128 rows at w = 1.5 (a network batch of 256): a sub-batch sampled alone with the same draws gives bit-identical
    fields, observed entries equal the condition bit for bit, everything is finite."""
    pl, cfg = stress_module()
    pl = pl.to(dev).eval()
    B, lo, hi = 128, 40, 48
    cond, mask = _masked_inputs(B, 51, dev)
    sp = _sparams(cfg, 2, 1.5)
    g = torch.Generator().manual_seed(52)
    draws = []

    def record(kind, like):
        t = torch.randn(like.shape, dtype=like.dtype, generator=g).to(like.device)
        draws.append(t)
        return t

    pl._noise_hook = record
    xs = pl.sample_edm(torch.zeros(B, 2, 128, 128, device=dev), cond, mask, sp, return_last=True)
    assert xs.shape == (B, 1, 128, 128, 2) and torch.isfinite(xs).all()
    keep = (mask == 0).permute(0, 2, 3, 1)
    assert torch.equal(xs[:, 0][keep], cond.permute(0, 2, 3, 1).double()[keep])
    replay = iter(draws)
    pl._noise_hook = lambda kind, like: next(replay)[lo:hi].contiguous()
    xs_sub = pl.sample_edm(torch.zeros(hi - lo, 2, 128, 128, device=dev), cond[lo:hi].contiguous(),
                           mask[lo:hi].contiguous(), sp, return_last=True)
    pl._noise_hook = None
    assert torch.equal(xs_sub, xs[lo:hi])


# ----------------------------------------------------------------------------------------------- 6. replay modes
def test_guided_replay_modes_agree(dev):
    """Graph replay with precomputed embedding rows, graph replay with the embedding MLP per evaluation, and eager
    evaluation give bit-identical guided fields."""
    pl, cfg = stress_module()
    pl = pl.to(dev).eval()
    cond, mask = _masked_inputs(2, 61, dev)
    hu = torch.zeros(2, 2, 128, 128, device=dev)
    eng = pl.ema_model.ma_model.engine()
    outs = []
    for rows, graph in ((True, True), (False, True), (True, False)):
        eng.supports_ss_rows = rows
        pl.use_cuda_graph = graph
        pl._noise_hook = NoiseFeed(17).hook
        outs.append(pl.sample_edm(hu, cond, mask, _sparams(cfg, 3, 1.5)))
    del eng.supports_ss_rows
    pl.use_cuda_graph, pl._noise_hook = True, None
    assert torch.isfinite(outs[0]).all()
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


# ----------------------------------------------------------------------------------------------- 7. sharding
def test_sharded_sampling_passes_w_through(dev):
    from mcedm_b200 import dist as MD

    pl, cfg = stress_module()
    pl = pl.to(dev).eval()
    B, chunk = 4, 2
    cond, mask = _masked_inputs(B, 71, dev)
    hu = torch.empty(B, 2, 128, 128, device=dev)
    g = torch.Generator().manual_seed(72)
    draws = []

    def record(kind, like):
        t = torch.randn(like.shape, dtype=like.dtype, generator=g).to(like.device)
        draws.append(t)
        return t

    pl._noise_hook = record
    whole = MD.sample_edm_sharded(pl, hu, cond, mask, _sparams(cfg, 2, 1.5), return_last=True, chunk=None)
    pos = {"k": 0, "lo": 0}

    def replay(kind, like):                              # the same draws, served row block by row block
        t = draws[pos["k"]][pos["lo"]:pos["lo"] + like.shape[0]].contiguous()
        pos["k"] += 1
        if pos["k"] == len(draws):
            pos["k"], pos["lo"] = 0, pos["lo"] + like.shape[0]
        return t

    pl._noise_hook = replay
    chunked = MD.sample_edm_sharded(pl, hu, cond, mask, _sparams(cfg, 2, 1.5), return_last=True, chunk=chunk)
    pos.update(k=0, lo=0)
    unguided = MD.sample_edm_sharded(pl, hu, cond, mask, _sparams(cfg, 2, 0.0), return_last=True, chunk=chunk)
    pl._noise_hook = None
    assert torch.equal(chunked, whole)
    assert not torch.equal(unguided, whole)


# ----------------------------------------------------------------------------------------------- 8-9. oracle parity
@pytest.mark.parametrize("precision,tol", [("fp16", 1e-2), ("fp32", 1e-4)])
def test_guided_sampler_parity_with_oracle(dev, precision, tol):
    """PlMcedm, 3 Heun steps: every recorded D_w against denoise_cfg on the input this path fed the network."""
    pl, cfg = stress_module()
    pl = pl.to(dev).eval()
    if precision == "fp32":
        pl.ema_model.ma_model.engine().precision = "fp32"
    state, _, _, _ = fixture_state()
    mask = torch.zeros(1, 128, 128, 2)
    mask[..., 1] = 1.0
    cond_in = pl.get_cond_in(state.to(dev), mask.to(dev), None, None).permute(0, 3, 1, 2).contiguous()
    mask_c = mask.permute(0, 3, 1, 2).contiguous().to(dev)
    sd = {k: v.detach().cpu() for k, v in pl.ema_model.ma_model.state_dict().items()}
    mcfg = dict(cfg.model.hparams.model)
    for w in (0.5, 2.0):
        feed = NoiseFeed(9)
        pl._noise_hook = feed.hook
        pl._trace = []
        xs = pl.sample_edm(feed.draw(mask_c), cond_in, mask_c, _sparams(cfg, 3, w), return_last=True)
        assert torch.isfinite(xs).all() and len(pl._trace) == 5
        for i, which, sigma, d, xt in pl._trace:
            with torch.no_grad():
                d_or, _ = denoise_cfg(sd, mcfg, xt.cpu(), torch.tensor(sigma, dtype=torch.float64), cond_in.cpu(), w)
            err = rel_l2(d, d_or)
            print(f"{precision} w={w} step {i}.{which} sigma {sigma:9.4f}: rel-L2 vs oracle {err:.3e}")
            assert err < tol, f"w={w} step {i}.{which} sigma {sigma}"
    pl._noise_hook = pl._trace = None


# ----------------------------------------------------------------------------------------------- 10. PDE guidance
def test_guided_cond_sampler_with_pde_guidance(dev):
    """PlCondEdm with guide_dx=True and w = 1: the PDE-guidance gradient is taken of D_w.  Every recorded D_w against
    denoise_cfg on the fed input, and the sample against the oracle sampler with the oracle gradient."""
    gc = golden("pde.pt")["cond"]
    pl, cfg, sd = _cond_module(dev, gc["stats"])
    mcfg = dict(cfg.model.hparams.model)
    s = {k: float(v) for k, v in gc["stats"].items() if torch.is_tensor(v)}
    h, u = D._FIELDS["swe_per"](1, 128, first_seed=gc["field_seed"])
    state = pl.data_transform(torch.from_numpy(h).to(dev), torch.from_numpy(u).to(dev))
    h_n, u_n = state[..., :1], state[..., 1:2]
    sp = _sparams(cfg, 3, 1.0)
    feed = NoiseFeed(gc["sample"]["seed"])
    pl._noise_hook = feed.hook
    pl._trace = []
    u_noise = feed.draw(u_n)
    xs = pl.sample_edm(pl.get_cond_in(h_n, u_n, None, None), u_noise, sp, return_last=True, guide_dx=True)
    cond_c = h_n.permute(0, 3, 1, 2).contiguous().cpu()
    assert len(pl._trace) == 5 and torch.isfinite(xs).all()
    for i, which, sigma, d, xt in pl._trace:
        with torch.no_grad():
            d_or, _ = denoise_cfg(sd, mcfg, xt.cpu(), torch.tensor(sigma, dtype=torch.float64), cond_c, 1.0)
        err = rel_l2(d, d_or)
        print(f"guide_dx w=1 step {i}.{which} sigma {sigma:9.4f}: rel-L2 vs oracle {err:.3e}")
        assert err < 1e-2
    pl._noise_hook = pl._trace = None

    def guide(hc, den):
        return torch.from_numpy(P.get_dx_pde_cond(hc[:, 0].numpy(), den[:, 0].numpy(), s, "swe_per", calc_prob=True))

    feed = NoiseFeed(gc["sample"]["seed"])
    un = feed.draw(torch.empty(1, 128, 128, 1)).permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        xs_or = cond_sample_edm_cfg(sd, mcfg, un, cond_c, dict(sp), lambda i, x: feed.draw(x), 1.0, guide=guide)
    err = rel_l2(xs, xs_or)
    print(f"guide_dx w=1 sample: rel-L2 vs oracle {err:.3e}")
    assert err < 5e-2


# ----------------------------------------------------------------------------------------------- 11. rejections
def test_guidance_rejections(dev):
    pl, cfg = stress_module()
    pl = pl.to(dev).eval()
    cond, mask = _masked_inputs(1, 81, dev)
    hu = torch.zeros(1, 2, 128, 128, device=dev)
    for bad in (math.nan, math.inf):
        with pytest.raises(ValueError):
            pl.sample_edm(hu, cond, mask, _sparams(cfg, 2, bad))
        with torch.no_grad(), pytest.raises(ValueError):
            pl.get_denoised(pl.ema_model, hu, torch.tensor(1.0), cond=cond, w=bad)
    plc, cfgc, _ = _cond_module(dev)
    with pytest.raises(ValueError):
        plc.sample_edm(torch.zeros(1, 128, 128, 1, device=dev), torch.zeros(1, 128, 128, 1, device=dev),
                       _sparams(cfgc, 2, -math.inf))
    # guided get_denoised has no backward: autograd on in train mode raises
    pl.train()
    with pytest.raises(NotImplementedError):
        pl.get_denoised(pl.ema_model, hu, torch.tensor(1.0), cond=cond, w=1.5)
    pl.eval()
    # PlDdim keeps rejecting guidance
    from mcedm_b200.ddim import PlDdim
    from mcedm_b200.utils import randomize_zero_init

    cfgd = hparams("config_adm_ddim_res32")
    torch.manual_seed(1)
    pld = PlDdim(copy.deepcopy(cfgd.model.hparams))
    randomize_zero_init(pld.model, 2)
    pld = pld.to(dev).eval()
    sp = copy.deepcopy(cfgd.diff_sampler)
    sp.w = 1.5
    x = torch.zeros(1, 128, 128, 1, device=dev)
    with pytest.raises(NotImplementedError):
        pld.sample_edm(x, x, sp)
    with pytest.raises(NotImplementedError):
        pld.get_denoised(pld.model, torch.zeros(1, 2, 128, 128, device=dev), torch.tensor(1.0),
                         cond=torch.zeros(1, 2, 128, 128, device=dev), w=1.5)
