"""GPU parity tests of the kernels behind the "fused16" training plan (mcedm_b200/train16_engine.py): GroupNorm backward
on raw 16-bit activations / 16-bit gradients in either layout, fp16 weight-gradient and attention-backward GEMMs, the
16-bit helpers.  References: fp64 autograd of the same torch expressions (models/adm_blocks.py:86-97, :103-118, :65-81).
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def L():
    from mcedm_b200 import _lib
    _lib.lib()
    return _lib


def flat_geom(L, H, W):
    pitch, blk = C.c_int(0), C.c_int(0)
    L.check(L.lib().mcedm_flat_geometry(H, W, C.byref(pitch), C.byref(blk)))
    return pitch.value, blk.value


def to_flat(L, x):
    B, H, W, Cc = x.shape
    P, blk = flat_geom(L, H, W)
    f = torch.zeros(B, blk, Cc, device=x.device, dtype=x.dtype)
    f[:, P:P + H * P].view(B, H, P, Cc)[:, :, :W] = x
    return f.reshape(B * blk, Cc).contiguous()


def from_flat(L, f, B, H, W):
    P, blk = flat_geom(L, H, W)
    return f.view(B, blk, -1)[:, P:P + H * P].reshape(B, H, P, -1)[:, :, :W]


@pytest.mark.parametrize("fmt,add16", [(0, 0), (1, 0), (1, 1)])
@pytest.mark.parametrize("B,H,W,rs,act,use_ss,add0_mode,use_add1,x_flat,dy_flat", [
    (2, 128, 128, 0, 1, True, None, False, False, False),      # norm1 at the widest level
    (3, 32, 32, 1, 1, False, 1, True, True, True),             # norm0 of an up block (dy / add0 at 64x64, padded-flat)
    (2, 128, 128, 2, 1, False, 2, False, False, True),         # norm0 of a down block (dy / add0 at 64x64)
    (2, 32, 32, 0, 0, False, 0, False, True, False),           # norm2 in front of qkv: dense dy, flat x
    (2, 64, 64, 0, 1, True, 0, True, True, True),
    (33, 16, 16, 0, 1, False, None, False, True, True)])       # 16 pixels per CTA
def test_gn_bwd16_matches_autograd(L, dev, fmt, add16, B, H, W, rs, act, use_ss, add0_mode, use_add1, x_flat, dy_flat):
    check_gn_bwd16(L, dev, fmt, add16, B, H, W, rs, act, use_ss, add0_mode, use_add1, x_flat, dy_flat)


def check_gn_bwd16(L, dev, fmt, add16, B, H, W, rs, act, use_ss, add0_mode, use_add1, x_flat, dy_flat, spread=False):
    """mcedm_gn_bwd16 on seeded inputs, launched twice, against fp64 autograd of the same GroupNorm(+scale/shift, +SiLU,
    +resample) expression.  After each launch the watchdog word is clear (a timed-out wait for the sample's coefficients
    records 0xdead7000 and then carries on with stale ones) and every ticket word is back at zero.  `spread`: x and dy
    get a per-sample scale and x a per-sample offset, so that one sample's coefficients are far from its neighbours'."""
    lib = L.lib()
    dt = torch.float16 if fmt else torch.bfloat16
    g = torch.Generator().manual_seed(H * 7 + rs + fmt)
    x = torch.randn(B, H, W, 64, generator=g) * 2 + 0.5
    if spread:
        x = x * (torch.rand(B, 1, 1, 1, generator=g) * 1.5 + 0.25) + (torch.rand(B, 1, 1, 1, generator=g) * 4 - 2)
    x = x.to(dev).to(dt)                                  # the RAW stored activation
    gamma, beta = torch.randn(64, generator=g).to(dev), torch.randn(64, generator=g).to(dev)
    ss = (torch.randn(B, 128, generator=g) * 0.3).to(dev)
    xf = x.float().contiguous()
    st = torch.empty(B * H * W // 128, 16, 2, device=dev)
    L.check(lib.mcedm_gn_stats(L.ptr(xf), B * H * W, L.ptr(st), L.stream_ptr()))
    mr = torch.empty(B, 16, 2, device=dev)
    coef = torch.empty(B, 128, device=dev)
    L.check(lib.mcedm_gn_coef(L.ptr(st), H * W // 128, L.ptr(gamma), L.ptr(beta), L.ptr(ss) if use_ss else None, 128, 64,
                              1e-5, B, H, W, L.ptr(coef), L.ptr(mr), L.stream_ptr()))
    Ho, Wo = (2 * H, 2 * W) if rs == 1 else (H // 2, W // 2) if rs == 2 else (H, W)
    dy = torch.randn(B, Ho, Wo, 64, generator=g)
    if spread:
        dy = dy * (torch.rand(B, 1, 1, 1, generator=g) * 3.75 + 0.25)
    dy = dy.to(dev).to(dt)
    xl = flat_geom(L, H, W) if x_flat else (0, 0)
    dyl = flat_geom(L, Ho, Wo) if dy_flat else (0, 0)
    x_buf = to_flat(L, x) if x_flat else x.contiguous()
    dy_buf = to_flat(L, dy) if dy_flat else dy.contiguous()
    add0 = add0_buf = None
    a0l = (0, 0)
    if add0_mode is not None:
        Ha, Wa = {0: (H, W), 1: (2 * H, 2 * W), 2: (H // 2, W // 2)}[add0_mode]
        add0 = torch.randn(B, Ha, Wa, 64, generator=g).to(dev)
        if add16:
            add0 = add0.to(dt)
        a0_flat = Wa <= 64
        a0l = flat_geom(L, Ha, Wa) if a0_flat else (0, 0)
        add0_buf = to_flat(L, add0) if a0_flat else add0
    add1 = torch.randn(B, H, W, 64, generator=g).to(dev) if use_add1 else None
    if use_add1 and add16:
        add1 = add1.to(dt)
    add1_buf = (to_flat(L, add1) if x_flat else add1) if use_add1 else None
    n_cta = lib.mcedm_gn_bwd16_ctas_per_img(H, W, B)
    red = torch.empty(B, n_cta, 64, 2, device=dev)
    dgb = torch.empty(B, 64, 2, device=dev)
    dss = torch.zeros(B, 128, device=dev)
    n_pos = B * xl[1] if x_flat else B * H * W
    dx = torch.zeros(n_pos, 64, device=dev)
    dx16 = torch.zeros(n_pos, 64, device=dev, dtype=dt)
    dxd = torch.empty(B, H, W, 64, device=dev, dtype=dt)
    cs = torch.empty(B * n_cta, 64, device=dev)
    kcoef = torch.empty(B, 192, device=dev)
    ticket = torch.zeros(3 * B, device=dev, dtype=torch.int32)
    for _ in range(2):      # twice: the ticket counters must be back at zero after a launch
        L.check(lib.mcedm_gn_bwd16(L.ptr(dy_buf), dyl[0], dyl[1], L.ptr(x_buf), xl[0], xl[1], fmt, L.ptr(mr),
                                   L.ptr(coef), L.ptr(gamma), L.ptr(beta), L.ptr(ss) if use_ss else None, 128, 64, act, rs, B, H, W,
                                   L.ptr(red), L.ptr(kcoef), L.ptr(ticket), L.ptr(dgb), L.ptr(dss) if use_ss else None,
                                   128, L.ptr(add0_buf), add0_mode or 0, a0l[0], a0l[1], L.ptr(add1_buf), add16,
                                   L.ptr(dx), L.ptr(dx16), L.ptr(dxd), L.ptr(cs), L.stream_ptr()), "gn_bwd16")
        L.check_watchdog()
        assert int(ticket.abs().sum()) == 0
    xd = x.double().permute(0, 3, 1, 2).requires_grad_(True)
    gd, bd, sd = gamma.double().requires_grad_(True), beta.double().requires_grad_(True), ss.double().requires_grad_(True)
    y = F.group_norm(xd, 16, gd, bd, 1e-5)
    if use_ss:
        y = torch.addcmul(sd[:, 64:, None, None], y, sd[:, :64, None, None] + 1)
    y = F.silu(y) if act else y
    y = y.repeat_interleave(2, 2).repeat_interleave(2, 3) if rs == 1 else F.avg_pool2d(y, 2) if rs == 2 else y
    y.backward(dy.double().permute(0, 3, 1, 2))
    ref = xd.grad.permute(0, 2, 3, 1)
    if add0 is not None:
        a0 = add0.double().permute(0, 3, 1, 2)
        a0 = F.avg_pool2d(a0, 2) * 4 if add0_mode == 1 else \
            0.25 * a0.repeat_interleave(2, 2).repeat_interleave(2, 3) if add0_mode == 2 else a0
        ref = ref + a0.permute(0, 2, 3, 1)
    if add1 is not None:
        ref = ref + add1.double()
    got = from_flat(L, dx, B, H, W) if x_flat else dx.view(B, H, W, 64)
    got16 = from_flat(L, dx16, B, H, W) if x_flat else dx16.view(B, H, W, 64)
    # silu' goes through tanh.approx (2^-11): 1e-3-class agreement with fp64 autograd
    assert rel_l2(got, ref) < 1e-3
    assert rel_l2(got16.float(), ref) < (1e-3 if fmt else 4e-3) and torch.equal(got16, dxd)
    if x_flat:   # the padding of the flat layout stays zero
        assert dx16.float().abs().sum().item() == pytest.approx(got16.float().abs().sum().item(), rel=1e-6)
    assert rel_l2(dgb[:, :, 0].sum(0), gd.grad) < 1e-3 and rel_l2(dgb[:, :, 1].sum(0), bd.grad) < 1e-3
    if use_ss:
        assert rel_l2(dss, sd.grad) < 1e-3
    assert rel_l2(cs.view(B, n_cta, 64).sum((0, 1)), ref.sum((0, 1, 2))) < 1e-3


@pytest.mark.parametrize("B,H,W,taps,dy_layout,a_layout", [
    (2, 128, 128, 9, 0, 0), (3, 64, 64, 9, 1, 1), (5, 32, 32, 1, 1, 1), (2, 128, 128, 1, 0, 0)])
def test_conv_wgrad_fp16_matches_autograd(L, dev, B, H, W, taps, dy_layout, a_layout):
    lib = L.lib()
    g = torch.Generator().manual_seed(B * 100 + H + taps)
    dy = torch.randn(B, H, W, 64, generator=g).to(dev).to(torch.float16).contiguous()
    a = torch.randn(B, H, W, 64, generator=g).to(dev).to(torch.float16).contiguous()
    dy_buf = to_flat(L, dy) if dy_layout else dy
    a_buf = to_flat(L, a) if a_layout else a
    n = lib.mcedm_wgrad_ctas(B, H, W)
    partial = torch.full((n, taps, 64, 64), float("nan"), device=dev)
    L.check(lib.mcedm_conv_wgrad16(L.ptr(dy_buf), dy_layout, 64, 0, L.ptr(a_buf), a_layout, 64, 0, B, H, W, taps,
                                   L.ptr(partial), 1, L.stream_ptr()), "conv_wgrad16")
    L.check_watchdog()
    k = 3 if taps == 9 else 1
    dw = torch.zeros(64, 64, k, k, device=dev)
    L.check(lib.mcedm_wgrad_reduce(L.ptr(partial), n, taps, L.ptr(dw), 64, 0, 1, 0, 64, 64, 0, L.stream_ptr()))
    w = torch.zeros(64, 64, k, k, device=dev, dtype=torch.float64, requires_grad=True)
    F.conv2d(a.double().permute(0, 3, 1, 2), w, padding=k // 2).backward(dy.double().permute(0, 3, 1, 2))
    assert rel_l2(dw, w.grad) < 1e-4


@pytest.mark.parametrize("B,H,W,taps,dy_layout,a_layout,act", [
    (2, 128, 128, 9, 0, 0, 1), (3, 64, 64, 9, 1, 1, 1), (5, 32, 32, 1, 0, 1, 0), (37, 32, 32, 9, 1, 1, 1)])
def test_conv_wgrad_fused_transform_matches_autograd(L, dev, B, H, W, taps, dy_layout, a_layout, act):
    """mcedm_conv_wgrad16_fused: the operand silu(a*x + b) is formed from the RAW activation inside the kernel."""
    lib = L.lib()
    g = torch.Generator().manual_seed(B * 100 + H + taps)
    dy = torch.randn(B, H, W, 64, generator=g).to(dev).to(torch.float16).contiguous()
    x = (torch.randn(B, H, W, 64, generator=g) * 1.5 + 0.3).to(dev).to(torch.float16).contiguous()
    coef = torch.cat([torch.rand(B, 64, generator=g) + 0.5, torch.randn(B, 64, generator=g) * 0.5], 1).to(dev).contiguous()
    dy_buf = to_flat(L, dy) if dy_layout else dy
    x_buf = to_flat(L, x) if a_layout else x
    n = lib.mcedm_wgrad_ctas(B, H, W)
    partial = torch.full((n, taps, 64, 64), float("nan"), device=dev)
    L.check(lib.mcedm_conv_wgrad16_fused(L.ptr(dy_buf), dy_layout, 64, 0, L.ptr(x_buf), a_layout, 64, 0, L.ptr(coef), act,
                                         B, H, W, taps, L.ptr(partial), 1, L.stream_ptr()), "conv_wgrad16_fused")
    L.check_watchdog()
    k = 3 if taps == 9 else 1
    dw = torch.zeros(64, 64, k, k, device=dev)
    L.check(lib.mcedm_wgrad_reduce(L.ptr(partial), n, taps, L.ptr(dw), 64, 0, 1, 0, 64, 64, 0, L.stream_ptr()))
    u = x.double() * coef[:, None, None, :64].double() + coef[:, None, None, 64:].double()
    a = (F.silu(u) if act else u).to(torch.float16)        # the kernel rounds the operand to fp16
    w = torch.zeros(64, 64, k, k, device=dev, dtype=torch.float64, requires_grad=True)
    F.conv2d(a.double().permute(0, 3, 1, 2), w, padding=k // 2).backward(dy.double().permute(0, 3, 1, 2))
    assert rel_l2(dw, w.grad) < 5e-4            # tanh.approx (2^-11) in the SiLU
    if a_layout:    # the raw activation itself is untouched
        assert torch.equal(x_buf, to_flat(L, x))


def test_attention_bwd_fp16_matches_autograd(L, dev):
    lib = L.lib()
    B, Lq = 2, 1024
    g = torch.Generator().manual_seed(5)
    qkv = torch.randn(B, Lq, 192, generator=g).to(dev).to(torch.float16)
    d_out = torch.randn(B, Lq, 64, generator=g).to(dev).to(torch.float16)
    out = torch.empty(B, Lq, 64, device=dev, dtype=torch.float16)
    lse = torch.empty(B, Lq, device=dev)
    L.check(lib.mcedm_attention(L.ptr(qkv), B, Lq, L.ptr(out), L.ptr(lse), 1, L.stream_ptr()), "attention")
    dvec = torch.empty(B, Lq, device=dev)
    dq, dk, dv = (torch.full((B, Lq, 64), float("nan"), device=dev, dtype=torch.float16) for _ in range(3))
    L.check(lib.mcedm_attention_bwd16(L.ptr(qkv), L.ptr(out), L.ptr(d_out), L.ptr(lse), B, Lq, L.ptr(dvec), L.ptr(dq),
                                      L.ptr(dk), L.ptr(dv), 1, L.stream_ptr()), "attention_bwd16")
    L.check_watchdog()
    x = qkv.double().requires_grad_(True)
    q, k, v = x.split(64, dim=2)
    s = q @ k.transpose(1, 2) / 8.0
    ref = torch.softmax(s, dim=2) @ v
    assert rel_l2(out.float(), ref) < 2e-3
    ref.backward(d_out.double())
    rq, rk, rv = x.grad.split(64, dim=2)
    assert rel_l2(dv.float(), rv) < 1.5e-3        # fp16 P, fp16 output: 8x tighter than the bf16 kernel's bars
    assert rel_l2(dq.float(), rq) < 3e-3
    assert rel_l2(dk.float(), rk) < 3e-3


def test_pad16_and_colsum16(L, dev):
    lib = L.lib()
    B, H, W = 3, 32, 64
    g = torch.Generator().manual_seed(3)
    x, y = torch.randn(B, 2, H, W, generator=g).to(dev), torch.randn(B, 2, H, W, generator=g).to(dev)
    for fmt, dt in ((0, torch.bfloat16), (1, torch.float16)):
        pad = torch.zeros(B, H, W, 64, device=dev, dtype=dt)
        L.check(lib.mcedm_nchw_to_nhwc_pad16(L.ptr(x), 2, L.ptr(y), 2, B, H, W, L.ptr(pad), 0, 8.0, fmt, L.stream_ptr()))
        ref = (torch.cat([x, y], 1) * 8.0).permute(0, 2, 3, 1).to(dt)
        assert torch.equal(pad[..., :4], ref) and pad[..., 4:].abs().max() == 0
        part = torch.empty(7, 64, device=dev)
        L.check(lib.mcedm_colsum16(L.ptr(pad), B * H * W, 64, 0, L.ptr(part), 7, fmt, L.stream_ptr()))
        assert rel_l2(part.sum(0)[:4], ref.float().sum((0, 1, 2))) < 1e-5


@pytest.mark.parametrize("H,W,taps", [(128, 128, 9), (32, 32, 9), (64, 64, 1)])
def test_wgrad_kx_stacked_operand_is_bit_identical_to_one_mma_per_tap(dev, H, W, taps):
    """conv_wgrad16_fused issues one N = 192 MMA per K block whose B operand is three 64-channel blocks ONE PIXEL apart
    (leading-dimension offset 128 B: the kx taps); MCEDM_WG_DBG=4 issues the three N = 64 MMAs separately.  Same products
    in the same order per accumulator column: the per-CTA partial sums must be bit-identical."""
    import os

    from mcedm_b200 import _lib as L
    lib = L.lib()
    B = 3
    g = torch.Generator(device="cpu").manual_seed(5)
    dy = (torch.randn(B, H, W, 64, generator=g) * 0.1).to(dev).half()
    a = torch.randn(B, H, W, 64, generator=g).to(dev).half()
    coef = torch.cat([torch.rand(B, 64, generator=g) + 0.5, torch.randn(B, 64, generator=g) * 0.3], 1).to(dev).contiguous()
    nc = lib.mcedm_wgrad_ctas(B, H, W)

    def run():
        part = torch.zeros(nc * taps * 4096, device=dev)
        L.check(lib.mcedm_conv_wgrad16_fused(L.ptr(dy), 0, 64, 0, L.ptr(a), 0, 64, 0, L.ptr(coef), 1, B, H, W, taps, L.ptr(part),
                                             1, L.stream_ptr()), "conv_wgrad")
        torch.cuda.synchronize()
        L.check_watchdog()
        return part

    p_stacked = run()
    old = os.environ.get("MCEDM_WG_DBG")
    os.environ["MCEDM_WG_DBG"] = "4"
    try:
        p_single = run()
    finally:
        if old is None:
            os.environ.pop("MCEDM_WG_DBG", None)
        else:
            os.environ["MCEDM_WG_DBG"] = old
    assert torch.equal(p_stacked, p_single)
    assert float(p_stacked.abs().sum()) > 0
