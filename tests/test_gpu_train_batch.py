"""The fp16 training backward ("fused16", mcedm_b200/train16_engine.py) at the batch sizes it trains at.

The batch decides how the backward kernels split their work: pixels per CTA and one-kernel vs two-kernel GroupNorm
backward (gn_bwd.cu pick_pix_per_cta16), which CTAs of the weight-gradient GEMM span two images (conv_wgrad.cu), and
the magnitude of the loss-scaled dL/dF (1024 * 2/B * ...).  The whole-network comparisons elsewhere run at B = 2;
here every kernel case asserts the regime it was written for, the whole network runs at B = 16 and 32 (the per-GPU
batch of the shipped configs) against a float64 reference of the step, and one module takes a 32 -> 5 -> 32 -> 16
sequence of batch shapes with optimizer steps in between.
"""
import ctypes as C
import math
import os

import pytest
import torch
import torch.nn.functional as F

from test_gpu_train16 import check_gn_bwd16, to_flat

gpu = pytest.mark.gpu


def rel(a, b):
    """||a - b|| / ||b|| in float64, on the tensors' device"""
    a, b = a.detach().double(), b.detach().double().to(a.device)
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def L():
    from mcedm_b200 import _lib

    _lib.lib()
    return _lib


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------ 1. fp64 reference
def reference_step(named, model_cfg, x, sigma, noise, cond, mask, chunk=8):
    """Loss and every parameter gradient of one training step in float64, on the device of `x`.

    oracle.edm_oracle.training_loss restated in float64: the preconditioning coefficients and the loss weight are
    computed in float64 (precond_coeffs / denoise cast to float32), and unet_forward runs on float64 inputs with float64
    leaf copies of `named` (parameter name -> tensor).  The loss is a mean over samples and GroupNorm works per sample,
    so the step is evaluated in chunks of `chunk` samples whose gradients are added with weight chunk / B.  TF32 is off
    for the duration (the oracle's attention logits are an fp32 einsum)."""
    from oracle import edm_oracle as O

    dev = x.device
    B = x.shape[0]
    flags = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        leaves = {k: v.detach().to(dev, torch.float64).requires_grad_(True) for k, v in named.items()}
        grads = {k: torch.zeros_like(v) for k, v in leaves.items()}
        loss = 0.0
        for i in range(0, B, chunk):
            j = min(B, i + chunk)
            xs, ns, cs, ms = (t[i:j].to(dev, torch.float64) for t in (x, noise, cond, mask))
            s = sigma.reshape(-1)[i:j].to(dev, torch.float64).reshape(-1, 1, 1, 1)
            den = s ** 2 + 1.0                                                 # sigma_data = 1
            c_skip, c_out, c_in, c_noise = 1.0 / den, s / den.sqrt(), 1.0 / den.sqrt(), s.log() / 4
            x_noise = xs + ms * ns * s
            f_x = O.unet_forward(leaves, model_cfg, c_in * x_noise, c_noise.flatten(), cs)
            d_x = c_skip * x_noise + c_out * f_x
            per = (O.loss_weight(s) * (d_x * ms - xs * ms) ** 2).sum(dim=(1, 2, 3))
            part = per.mean() * ((j - i) / B)
            gs = torch.autograd.grad(part, list(leaves.values()))
            for k, g in zip(leaves, gs):
                grads[k] += g
            loss += float(part.detach())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = flags
    return loss, grads


def _named_params(pl):
    return {k: p.detach().clone() for k, p in pl.model.named_parameters()}


def test_reference_step_matches_fp32_oracle_autograd():
    """CPU, B = 2: the float64 step reference against fp32 autograd through oracle.edm_oracle.training_loss, which the
    oracle tests pin to fixtures of the unmodified reference.  8 threads, the count those fixtures were written with."""
    from common import fixture_state, golden, stress_module
    from oracle import edm_oracle as O

    n = torch.get_num_threads()
    torch.set_num_threads(8)
    try:
        g = golden("train_step.pt")
        pl, cfg = stress_module()
        mcfg = dict(cfg.model.hparams.model)
        named = _named_params(pl)
        assert len(named) == 196
        state, _, _, _ = fixture_state(n=2, seed=g["seed_fields"])
        x = state.permute(0, 3, 1, 2).contiguous()
        mask = g["mask"].permute(0, 3, 1, 2).contiguous()
        gen = torch.Generator().manual_seed(1)
        noise = torch.randn(x.shape, generator=gen)
        cond = (x * (1 - mask) + torch.randn(x.shape, generator=gen) * mask).contiguous()
        sigma = torch.tensor([0.7, 3.0]).view(2, 1, 1, 1)
        sd = {k: v.clone().requires_grad_(True) for k, v in named.items()}
        ref, _ = O.training_loss(sd, mcfg, x, sigma, noise, cond, mask)
        ref.backward()
        loss, grads = reference_step(named, mcfg, x, sigma, noise, cond, mask)
    finally:
        torch.set_num_threads(n)
    ref = float(ref.detach())
    assert abs(loss - ref) < 1e-5 * abs(ref)
    errs = sorted(((rel(sd[k].grad, grads[k]), k) for k in named), reverse=True)
    print(f"loss {loss:.9g} vs fp32 oracle {ref:.9g}; worst gradients {errs[:3]}")
    assert errs[0][0] < 1e-5, errs[:5]


# ------------------------------------------------------------------------------------------------ 2. gn_bwd16 regimes
def gn_bwd16_regime(L, H, W, B):
    """(one-kernel?, pixels per CTA) of mcedm_gn_bwd16 at this shape, as its launcher decides (gn_bwd.cu)"""
    n_cta = L.lib().mcedm_gn_bwd16_ctas_per_img(H, W, B)
    per = H * W // n_cta
    split = bool(os.environ.get("MCEDM_GNBWD_SPLIT") and int(os.environ["MCEDM_GNBWD_SPLIT"]))
    return (not split and n_cta * B <= 2 * n_sms() and per % 64 == 0), per


# (B, H, rs, act, use_ss, add0_mode, use_add1, x_flat, dy_flat, one-kernel, pixels per CTA); W = H.  Layouts follow
# the network: 128 wide dense, 64 and narrower padded-flat.  rs 1 (up block norm0: dy, add0 at 2H), 2 (down block
# norm0: dy, add0 at H/2).  Regimes are those of a 148-SM B200.
GN_CASES = [
    (3, 128, 0, 1, True, None, False, False, False, False, 128),    # norm1 at the widest level
    (5, 128, 2, 1, False, 2, False, False, True, False, 256),       # down block norm0, dy / add0 at 64x64
    (16, 128, 0, 1, True, 0, True, False, False, True, 1024),
    (32, 128, 0, 1, True, None, False, False, False, True, 2048),
    (32, 128, 2, 1, False, 2, False, False, True, True, 2048),
    (40, 128, 0, 0, False, 0, True, False, False, False, 2048),
    (3, 64, 1, 1, False, 1, True, True, False, True, 128),          # up block norm0, dy / add0 at 128x128
    (5, 64, 0, 1, True, 0, False, True, True, True, 128),
    (16, 64, 2, 1, False, 2, False, True, True, True, 256),
    (32, 64, 0, 1, True, 0, True, True, True, True, 512),
    (40, 64, 1, 1, False, 1, False, True, False, False, 512),
    (3, 32, 1, 1, False, 1, True, True, True, True, 128),
    (5, 32, 0, 0, False, 0, False, True, False, True, 128),         # norm2 in front of qkv: dense dy
    (16, 32, 0, 1, True, None, False, True, True, True, 128),
    (32, 32, 1, 1, False, 1, False, True, True, True, 128),
    (40, 32, 0, 1, True, 0, True, True, True, False, 128),
]


def test_gn_bwd16_cases_cover_every_regime():
    """The cases below together run the one-kernel and the two-kernel path, with 128 and with more pixels per CTA,
    and every resample mode: a change of the table cannot drop a regime unnoticed (each case asserts its own)."""
    regimes = {(c[-2], c[-1] == 128) for c in GN_CASES}
    assert {(True, True), (True, False), (False, True), (False, False)} <= regimes
    assert {c[2] for c in GN_CASES} == {0, 1, 2}
    assert {c[0] for c in GN_CASES} == {3, 5, 16, 32, 40} and {c[1] for c in GN_CASES} == {32, 64, 128}


@gpu
@pytest.mark.parametrize("add16", [0, 1])
@pytest.mark.parametrize("B,H,rs,act,use_ss,add0_mode,use_add1,x_flat,dy_flat,one_kernel,per", GN_CASES)
def test_gn_bwd16_at_training_batches(L, dev, add16, B, H, rs, act, use_ss, add0_mode, use_add1, x_flat, dy_flat,
                                      one_kernel, per):
    """Inputs with per-sample statistics far apart: a pass that used a neighbouring sample's coefficients misses the
    bar (fp64 autograd, the bars of test_gpu_train16)."""
    assert gn_bwd16_regime(L, H, H, B) == (one_kernel, per), "the launcher no longer runs this case's regime"
    check_gn_bwd16(L, dev, 1, add16, B, H, H, rs, act, use_ss, add0_mode, use_add1, x_flat, dy_flat, spread=True)


# ------------------------------------------------------------------------------------------------ 3. weight gradients
def wgrad_segments(L, B, H, W):
    """Per CTA of conv_wgrad_kernel: its (image, rows) segments - the contiguous row range B*H*i/g .. B*H*(i+1)/g cut
    at image boundaries (conv_wgrad.cu), g = mcedm_wgrad_ctas."""
    g = L.lib().mcedm_wgrad_ctas(B, H, W)
    total, out = B * H, []
    for i in range(g):
        r, r_end, segs = total * i // g, total * (i + 1) // g, []
        while r < r_end:
            b = r // H
            n = min(r_end - r, H - (r - b * H))
            segs.append((b, n))
            r += n
        out.append(segs)
    return out


def wgrad_reference(dy, a, k):
    """dW of y = conv2d(a, W, padding=k//2) for upstream gradient dy (NHWC, float64): one GEMM per tap, the contraction
    over every pixel of every image (a zero outside the image)."""
    B, H, W, _ = a.shape
    p = k // 2
    ap = F.pad(a, (0, 0, p, p, p, p))
    dyf = dy.reshape(-1, dy.shape[-1])
    dw = torch.empty(dy.shape[-1], a.shape[-1], k, k, dtype=torch.float64, device=a.device)
    for ky in range(k):
        for kx in range(k):
            dw[:, :, ky, kx] = dyf.t() @ ap[:, ky:ky + H, kx:kx + W].reshape(-1, a.shape[-1])
    return dw


def test_wgrad_reference_is_conv2d_weight_gradient():
    g = torch.Generator().manual_seed(4)
    for k in (3, 1):
        dy, a = torch.randn(3, 8, 16, 64, generator=g, dtype=torch.float64), torch.randn(3, 8, 16, 64, generator=g, dtype=torch.float64)
        w = torch.zeros(64, 64, k, k, dtype=torch.float64, requires_grad=True)
        F.conv2d(a.permute(0, 3, 1, 2), w, padding=k // 2).backward(dy.permute(0, 3, 1, 2))
        assert rel(wgrad_reference(dy, a, k), w.grad) < 1e-12


# (B, H, taps, single-row segment intended); 128 wide: dense layout, 64 and 32 wide: padded-flat (both operands)
WG_CASES = [
    (16, 128, 9, False), (32, 128, 9, False), (33, 128, 1, True), (40, 128, 1, False),
    (16, 64, 1, True), (32, 64, 9, True), (33, 64, 9, True), (40, 64, 1, True),
    (40, 32, 9, True), (40, 32, 1, True),
]


def _wgrad_segments_as_intended(L, B, H, single_row):
    segs = wgrad_segments(L, B, H, H)
    spanning = [s for s in segs if len(s) > 1]
    assert spanning, "no CTA spans two images at this shape any more"
    if single_row:
        assert any(n == 1 for s in spanning for _, n in s), "no single-row segment at this shape any more"
    return segs


def _wgrad_fold(L, dev, partial, n, taps):
    k = 3 if taps == 9 else 1
    dw = torch.zeros(64, 64, k, k, device=dev)
    L.check(L.lib().mcedm_wgrad_reduce(L.ptr(partial), n, taps, L.ptr(dw), 64, 0, 1, 0, 64, 64, 0, L.stream_ptr()))
    return dw, k


@gpu
@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("B,H,taps,single_row", WG_CASES)
def test_conv_wgrad16_with_ctas_spanning_images(L, dev, fused, B, H, taps, single_row):
    """conv_wgrad16 / conv_wgrad16_fused where CTAs' row ranges cross image boundaries (and, where intended, end or
    begin with a single row of an image).  The fused variant forms silu(a*x + b) with per-SAMPLE coefficients drawn
    with a wide spread, so a segment transformed with a neighbouring sample's coefficients misses the bar."""
    lib = L.lib()
    segs = _wgrad_segments_as_intended(L, B, H, single_row)
    flat = H <= 64
    g = torch.Generator().manual_seed(B * 100 + H + taps)
    dy =torch.randn(B, H, H, 64, generator=g).to(dev).half()
    x = (torch.randn(B, H, H, 64, generator=g) * 1.5 + 0.3).to(dev).half()
    dy_buf, x_buf = (to_flat(L, dy), to_flat(L, x)) if flat else (dy, x)
    lay = int(flat)
    n = len(segs)
    partial = torch.full((n, taps, 64, 64), float("nan"), device=dev)
    if fused:
        coef = torch.cat([torch.rand(B, 64, generator=g) + 0.5, torch.rand(B, 64, generator=g) * 2 - 1], 1).to(dev)
        L.check(lib.mcedm_conv_wgrad16_fused(L.ptr(dy_buf), lay, 64, 0, L.ptr(x_buf), lay, 64, 0, L.ptr(coef), 1, B, H, H,
                                             taps, L.ptr(partial), 1, L.stream_ptr()), "conv_wgrad16_fused")
        u = x.double() * coef[:, None, None, :64].double() + coef[:, None, None, 64:].double()
        a = F.silu(u).half()                  # the kernel rounds the operand to fp16
    else:
        L.check(lib.mcedm_conv_wgrad16(L.ptr(dy_buf), lay, 64, 0, L.ptr(x_buf), lay, 64, 0, B, H, H, taps, L.ptr(partial),
                                       1, L.stream_ptr()), "conv_wgrad16")
        a = x
    L.check_watchdog()
    dw, k = _wgrad_fold(L, dev, partial, n, taps)
    err = rel(dw, wgrad_reference(dy.double(), a.double(), k))
    assert err < (5e-4 if fused else 1e-4), err       # tanh.approx (2^-11) in the fused SiLU
    if fused and flat:      # the raw activation itself is untouched
        assert torch.equal(x_buf, to_flat(L, x))


@gpu
def test_conv_wgrad_bf16_padded_flat_with_ctas_spanning_images(L, dev):
    """The bf16 weight-gradient kernel (fp32-stream training plan) at 64x64 padded-flat with single-row segments."""
    B, H, taps = 32, 64, 9
    segs = _wgrad_segments_as_intended(L, B, H, True)
    g = torch.Generator().manual_seed(7)
    dy =torch.randn(B, H, H, 64, generator=g).to(dev).bfloat16()
    a = torch.randn(B, H, H, 64, generator=g).to(dev).bfloat16()
    dy_buf, a_buf = to_flat(L, dy), to_flat(L, a)
    partial = torch.full((len(segs), taps, 64, 64), float("nan"), device=dev)
    L.check(L.lib().mcedm_conv_wgrad(L.ptr(dy_buf), 1, 64, 0, L.ptr(a_buf), 1, 64, 0, B, H, H, taps, L.ptr(partial),
                                     L.stream_ptr()), "conv_wgrad")
    L.check_watchdog()
    dw, k = _wgrad_fold(L, dev, partial, len(segs), taps)
    assert rel(dw, wgrad_reference(dy.double(), a.double(), k)) < 1e-4


# ------------------------------------------------------------------------------------------------ 4./5. whole network
TOL = dict(loss=2e-3, glob=4e-3, worst=6e-3)          # the bars of the B = 2 whole-network test (test_gpu_train.py)


def _module(dev):
    from common import stress_module
    from mcedm_b200 import data as D

    pl, cfg = stress_module()
    pl = pl.to(dev).train()
    st = D.field_stats("swe_per", 16)
    pl.normalizer_input.set_stats(st["input_mean"].to(dev), st["input_std"].to(dev))
    pl.normalizer_target.set_stats(st["target_mean"].to(dev), st["target_std"].to(dev))
    assert pl.model.engine().train_plan == "fused16"
    return pl, dict(cfg.model.hparams.model)


def _inputs(pl, dev, B, seed):
    """swe_per fields and train masks (data.make_batch) through pl._prep_batch, seeded noise, and sigma log-spaced
    over the sampler's range [0.002, 80] - both tails of EDM's log-normal - shuffled so that neighbouring samples (and
    the CTAs that span them) see very different noise levels."""
    from common import NoiseFeed
    from mcedm_b200 import data as D

    torch.manual_seed(seed)                            # the mask coins
    h, _, _, u, mask = (t.to(dev) for t in D.make_batch("swe_per", B, "train", seed=seed))
    pl._noise_hook = NoiseFeed(seed).hook
    x, cond, mask_c = pl._prep_batch(h, u, mask)
    gen = torch.Generator().manual_seed(seed + 1)
    noise = torch.randn(x.shape, generator=gen).to(dev)
    sigma = torch.logspace(math.log10(0.002), math.log10(80.0), B)[torch.randperm(B, generator=gen)]
    return x, sigma.view(B, 1, 1, 1).to(dev), noise, cond, mask_c


def _step(pl, inp):
    """(loss, [gradient of every parameter]) of one pl.forward_loss step"""
    x, sigma, noise, cond, mask = inp
    pl.zero_grad(set_to_none=True)
    loss = pl.forward_loss(x, sigma, noise, cond, mask, pl.get_loss_weight(sigma))
    loss.backward()
    return loss.detach().clone(), [p.grad.detach().clone() for p in pl.model.parameters()]


def _compare(pl, loss, grads, ref, tag):
    ref_loss, ref_g = ref
    names = [k for k, _ in pl.model.named_parameters()]
    worst = sorted(((rel(g, ref_g[k]), k) for k, g in zip(names, grads)), reverse=True)
    glob = rel(torch.cat([g.flatten() for g in grads]), torch.cat([ref_g[k].flatten() for k in names]))
    lerr = abs(float(loss) - ref_loss) / abs(ref_loss)
    print(f"{tag}: loss {float(loss):.6g} (ref {ref_loss:.6g}, err {lerr:.2e}), global gradient error {glob:.2e}, "
          f"worst tensors {[(f'{e:.2e}', k) for e, k in worst[:8]]}")
    assert all(torch.isfinite(g).all() for g in grads)
    assert lerr < TOL["loss"], (tag, lerr)
    assert glob < TOL["glob"], (tag, glob)
    assert worst[0][0] < TOL["worst"], (tag, worst[:5])


def _with_env(name, value, fn):
    old = os.environ.get(name)
    os.environ[name] = value
    try:
        return fn()
    finally:
        if old is None:
            os.environ.pop(name, None)
        else:
            os.environ[name] = old


@gpu
@pytest.mark.parametrize("B", [16, 32])
def test_training_step_at_training_batch_matches_fp64_reference(dev, B):
    """All 196 parameter gradients of one step at B = 16 / 32 against the float64 reference, through the eager
    autograd bridge with the weight gradients on the side stream and without it (MCEDM_WGRAD_SIDE=0), and through the
    CUDA-graph replay (replayed, then replayed on other inputs, then replayed again on these).  Every fold of the
    backward has a fixed order, so the four gradient sets are bit-identical.  Then one eager step under MCEDM_DBG=4
    must leave the fp16 saturation counter at 0: it audits the epilogues of the fused forward and data-gradient
    convolutions, not gn_bwd16's outputs."""
    from mcedm_b200 import _lib as L

    pl, mcfg = _module(dev)
    inp = _inputs(pl, dev, B, seed=100 + B)
    ref = reference_step(_named_params(pl), mcfg, *inp)
    pl.use_cuda_graph = False
    loss_a, g_a = _step(pl, inp)
    _compare(pl, loss_a, g_a, ref, f"B={B} eager, side stream")
    loss_b, g_b = _with_env("MCEDM_WGRAD_SIDE", "0", lambda: _step(pl, inp))
    pl.use_cuda_graph = True
    loss_c, g_c = _step(pl, inp)
    other = tuple(t.flip(0).contiguous() for t in inp)
    _step(pl, other)
    loss_d, g_d = _step(pl, inp)
    L.check_watchdog()
    for tag, (lo, gr) in (("side stream off", (loss_b, g_b)), ("graph", (loss_c, g_c)), ("graph again", (loss_d, g_d))):
        assert torch.equal(lo, loss_a), tag
        diff = [k for (k, _), x, y in zip(pl.model.named_parameters(), gr, g_a) if not torch.equal(x, y)]
        assert not diff, (tag, diff)
    pl.use_cuda_graph = False
    lib = L.lib()
    cnt = C.c_longlong(0)

    def audited():
        L.check(lib.mcedm_saturation_count(C.byref(cnt), 1, L.stream_ptr()))
        _step(pl, inp)
        torch.cuda.synchronize()
        L.check(lib.mcedm_saturation_count(C.byref(cnt), 1, L.stream_ptr()))
        return cnt.value

    assert _with_env("MCEDM_DBG", "4", audited) == 0
    L.check_watchdog()


@gpu
def test_batch_shape_changes_with_optimizer_steps_on_one_module(dev):
    """Graph mode, one PlMcedm, batches of 32 -> 5 -> 32 -> 16 with an optimizer step (lr 2e-3) after each: every
    step against the float64 reference of the module's CURRENT parameters.  B = 5 runs the two-kernel gn_bwd16 at
    128x128; each shape has its own workspaces and graphs, and the packed fp16 weights must follow every update.  The
    two B = 32 steps take the same inputs and their losses must differ far beyond the bar, so stale weights or a
    stale graph could not pass."""
    from mcedm_b200 import _lib as L

    pl, mcfg = _module(dev)
    pl.use_cuda_graph = True
    opt = pl.configure_optimizers()["optimizer"]
    opt.param_groups[0]["lr"] = 2e-3
    assert not gn_bwd16_regime(L, 128, 128, 5)[0]
    inputs = {B: _inputs(pl, dev, B, seed=200 + B) for B in (32, 5, 16)}
    losses = []
    for it, B in enumerate((32, 5, 32, 16)):
        ref = reference_step(_named_params(pl), mcfg, *inputs[B])
        loss, grads = _step(pl, inputs[B])
        L.check_watchdog()
        _compare(pl, loss, grads, ref, f"step {it} B={B}")
        losses.append(float(loss))
        pl.optimizer_step(0, it, opt)
    moved = abs(losses[2] - losses[0]) / abs(losses[0])
    print(f"B=32 loss before / after two optimizer steps: {losses[0]:.6g} / {losses[2]:.6g} ({moved:.2e})")
    assert moved > 10 * TOL["loss"], moved
