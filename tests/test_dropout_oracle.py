"""CPU: the dropout oracle (tests/dropout_oracle.py) and the module surface of `dropout`."""
import copy

import numpy as np
import pytest
import torch

import dropout_oracle as DO


def test_philox_known_answer_vectors():
    """The Random123 known-answer vectors of Philox4x32-10."""
    cases = [
        ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
        ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
        ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
         (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
    ]
    for ctr, key, want in cases:
        got = DO.philox4x32_10(*[np.array([c], dtype=np.uint64) for c in ctr], *key)
        assert tuple(int(w[0]) for w in got) == want
        got_t = DO._philox_torch(*[torch.tensor([c], dtype=torch.int64) for c in ctr], *key)
        assert tuple(int(w[0]) for w in got_t) == want


def test_torch_mask_words_equal_the_numpy_philox():
    seed = 0x1234_5678_9ABC_DEF0
    a = DO.mask_words(seed, 7, 3, 2, 16, 8)
    b = DO.mask_words(seed, 7, 3, 2, 16, 8, device="cpu")
    assert torch.equal(a, b)
    # the logical index: element (b, c, y, x) uses quad ((b*H + y)*W + x)*16 + c // 4, word c % 4
    q = ((1 * 16 + 5) * 8 + 2) * 16 + 37 // 4
    w = DO.philox4x32_10(np.array([q], np.uint64), np.array([0], np.uint64), np.array([3], np.uint64),
                         np.array([7], np.uint64), seed & 0xFFFFFFFF, seed >> 32)
    assert int(a[1, 37, 5, 2]) == int(w[37 % 4][0])


def test_keep_mask_threshold_and_rate():
    assert DO.threshold(0.0) == 0 and DO.threshold(0.5) == 2 ** 31 and DO.threshold(1 - 1e-12) == 2 ** 32 - 1
    assert DO.scale(0.1) == float(np.float32(1 / 0.9))
    m = DO.keep_mask(5, 0, 0, 4, 32, 32, 0.25)
    assert m.dtype == torch.bool and m.shape == (4, 64, 32, 32)
    n = m.numel()
    assert abs(float(m.float().mean()) - 0.75) < 5 * (0.75 * 0.25 / n) ** 0.5
    assert bool(DO.keep_mask(5, 0, 0, 1, 16, 16, 0.0).all())


def test_layer_shapes_follow_the_network():
    from common import hparams

    mcfg = dict(hparams().model.hparams.model)
    shapes = DO.layer_shapes(mcfg)
    assert len(shapes) == 15
    assert shapes[0] == (128, 128) and shapes[1] == (64, 64) and shapes[4] == (32, 32) and shapes[-1] == (128, 128)


def test_unet_forward_dropout_with_all_true_masks_is_the_oracle():
    """All-true masks and s = 1 on the unet_forward.pt inputs: the bits of oracle.edm_oracle.unet_forward."""
    from common import golden, stress_unet
    from oracle import edm_oracle as O

    g = golden("unet_forward.pt")
    net, cfg, _ = stress_unet()
    mcfg = dict(cfg.model.hparams.model)
    sd = {k: v.detach() for k, v in net.state_dict().items()}
    for case in g["cases"]:
        x, nl, cond = case["x"], case["noise_labels"], case["cond"]
        B = x.shape[0]
        masks = {i: torch.ones(B, 64, h, w, dtype=torch.bool) for i, (h, w) in enumerate(DO.layer_shapes(mcfg))}
        with torch.no_grad():
            ref = O.unet_forward(sd, mcfg, x, nl, cond)
            got = DO.unet_forward_dropout(sd, mcfg, x, nl, cond, masks, 1.0)
        assert torch.equal(got, ref)


def test_dropout_reference_step_matches_fp32_autograd():
    """B = 2, p = 0.1: the float64 step reference with masks against fp32 autograd through the dropout oracle."""
    from common import fixture_state, golden, stress_module

    n = torch.get_num_threads()
    torch.set_num_threads(8)
    try:
        g = golden("train_step.pt")
        pl, cfg = stress_module()
        mcfg = dict(cfg.model.hparams.model)
        named = {k: p.detach().clone() for k, p in pl.model.named_parameters()}
        state, _, _, _ = fixture_state(n=2, seed=g["seed_fields"])
        x = state.permute(0, 3, 1, 2).contiguous()
        mask = g["mask"].permute(0, 3, 1, 2).contiguous()
        gen = torch.Generator().manual_seed(1)
        noise = torch.randn(x.shape, generator=gen)
        cond = (x * (1 - mask) + torch.randn(x.shape, generator=gen) * mask).contiguous()
        sigma = torch.tensor([0.7, 3.0]).view(2, 1, 1, 1)
        p = 0.1
        masks = DO.network_masks(11, 3, mcfg, 2, p)
        s = DO.scale(p)
        sd = {k: v.clone().requires_grad_(True) for k, v in named.items()}
        from oracle import edm_oracle as O

        c_skip, c_out, c_in, c_noise = O.precond_coeffs(sigma)
        x_noise = x + mask * noise * sigma
        f_x = DO.unet_forward_dropout(sd, mcfg, c_in * x_noise, c_noise.flatten(), cond, masks, s)
        d_x = c_skip * x_noise + c_out * f_x
        ref = (O.loss_weight(sigma) * (d_x * mask - x * mask) ** 2).sum(dim=(1, 2, 3)).mean()
        ref.backward()
        loss, grads = DO.reference_step_dropout(named, mcfg, x, sigma, noise, cond, mask, masks, s)
        # the masks do change the step
        loss0, _ = DO.reference_step_dropout(named, mcfg, x, sigma, noise, cond, mask, None, 1.0)
    finally:
        torch.set_num_threads(n)
    ref = float(ref.detach())
    assert abs(loss - ref) < 1e-5 * abs(ref)
    assert abs(loss - loss0) > 1e-3 * abs(loss0)
    errs = sorted((float((sd[k].grad.double() - grads[k]).norm() / grads[k].norm().clamp_min(1e-300)), k)
                  for k in named)[::-1]
    print(f"loss {loss:.9g} vs fp32 {ref:.9g} (no dropout {loss0:.9g}); worst gradients {errs[:3]}")
    assert errs[0][0] < 1e-5, errs[:5]


def _module_with_dropout(p, config="config_adm_edm_mcedm_res32"):
    from common import hparams
    from mcedm_b200.mcedm import PlMcedm

    cfg = hparams(config)
    h = copy.deepcopy(cfg.model.hparams)
    h.model.dropout = p
    torch.manual_seed(1)
    return PlMcedm(h)


def test_module_with_dropout_has_the_same_state_and_seeded_init():
    from mcedm_b200.utils import state_hash

    pl0, pl1 = _module_with_dropout(0.0), _module_with_dropout(0.1)
    sd0, sd1 = pl0.state_dict(), pl1.state_dict()
    assert len(sd1) == 412 and list(sd0) == list(sd1)
    assert state_hash(sd0) == state_hash(sd1)
    assert pl1.model.dropout == 0.1 and pl1.ema_model.ma_model.dropout == 0.1
    assert all(b.dropout == 0.1 for b in list(pl1.model.enc.values())[1:] + list(pl1.model.dec.values()))
    pl1.load_state_dict(sd0, strict=True)


@pytest.mark.parametrize("p", [1.0, -0.1, 1.5, float("nan")])
def test_dropout_outside_unit_interval_raises(p):
    with pytest.raises(ValueError):
        _module_with_dropout(p)
