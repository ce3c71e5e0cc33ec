"""CPU oracle of dropout in the training forward: test infrastructure on top of oracle/edm_oracle.py.

The reference applies dropout to conv1's operand of every UNetBlock (models/adm_blocks.py:167,
`conv1(F.dropout(silu(...), p, training))`); its masks come from torch's generator, whose bits no kernel can reproduce.
The kernels draw them from a counter-based Philox4x32-10 stream instead (DESIGN.md §3, csrc/philox.cuh):

    element (b, y, x, c) of the block with layer id `layer` (its aff_index) at H x W: n = ((b*H + y)*W + x)*64 + c
    word  = philox4x32_10(ctr = (n >> 2, n >> 34, layer, step), key = (seed_lo, seed_hi))[n & 3]
    keep  = word >= T,  T = min(2^32 - 1, floor(p * 2^32))          operand = silu(...) * keep * s,  s = fp32(1/(1-p))

`philox4x32_10` is the numpy statement of the generator (uint64 arrays holding 32-bit words); `keep_mask` evaluates the
masks with it, or with the same arithmetic in torch int64 on a device when one is given.  `unet_forward_dropout` is
oracle.edm_oracle.unet_forward with `x * keep * s` before conv1, and `reference_step_dropout` the float64 training step
of tests/test_gpu_train_batch.py through it.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F

from oracle import edm_oracle as O

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
_MASK = 0xFFFFFFFF


def philox4x32_10(c0, c1, c2, c3, k0: int, k1: int):
    """Philox4x32-10 (Random123 constants and round function) on uint64 arrays holding 32-bit counter words."""
    m = np.uint64(_MASK)
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & m for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0 & _MASK), np.uint64(k1 & _MASK)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c0, np.uint64(M1) * c2          # 32 x 32 -> 64 bits: exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & m
        k0, k1 = (k0 + np.uint64(W0)) & m, (k1 + np.uint64(W1)) & m
    return c0, c1, c2, c3


def _philox_torch(c0, c1, c2, c3, k0: int, k1: int):
    """The same rounds in torch int64 (products wrap modulo 2^64; every result is masked to 32 bits)."""
    m = _MASK
    k0, k1 = k0 & m, k1 & m
    for _ in range(10):
        p0, p1 = c0 * M0, c2 * M1
        c0, c1, c2, c3 = ((p1 >> 32) & m) ^ c1 ^ k0, p1 & m, ((p0 >> 32) & m) ^ c3 ^ k1, p0 & m
        k0, k1 = (k0 + W0) & m, (k1 + W1) & m
    return c0, c1, c2, c3


def threshold(p: float) -> int:
    return min(2 ** 32 - 1, math.floor(float(p) * 2.0 ** 32))


def scale(p: float) -> float:
    return float(np.float32(1.0 / (1.0 - float(p))))


def mask_words(seed: int, step: int, layer: int, B: int, H: int, W: int, device=None):
    """The mask word of every element, [B, 64, H, W] (int64 torch tensor; numpy Philox on the CPU when device is None)."""
    s = int(seed) & (2 ** 64 - 1)
    k0, k1 = s & _MASK, s >> 32
    nq = B * H * W * 16                                            # quads of 4 consecutive channels
    if device is None:
        q = np.arange(nq, dtype=np.uint64)
        out = philox4x32_10(q, q >> np.uint64(32), np.full_like(q, layer), np.full_like(q, step & _MASK), k0, k1)
        words = torch.from_numpy(np.stack(out, axis=1).astype(np.int64))
    else:
        q = torch.arange(nq, dtype=torch.int64, device=device)
        out = _philox_torch(q & _MASK, q >> 32, torch.full_like(q, layer), torch.full_like(q, step & _MASK), k0, k1)
        words = torch.stack(out, dim=1)
    return words.reshape(B, H, W, 64).permute(0, 3, 1, 2)


def keep_mask(seed: int, step: int, layer: int, B: int, H: int, W: int, p: float, device=None) -> torch.Tensor:
    """bool [B, 64, H, W]: True where the element is kept."""
    return mask_words(seed, step, layer, B, H, W, device) >= threshold(p)


def layer_shapes(model_cfg):
    """(H, W) of every UNetBlock's conv1 operand, in layer-id order (encoder then decoder)."""
    plan = O.unet_plan(model_cfg)
    res = model_cfg["resolution"]
    out = []
    for spec in plan["enc"] + plan["dec"]:
        if spec["kind"] == "conv":
            continue
        if spec["down"]:
            res //= 2
        if spec["up"]:
            res *= 2
        out.append((res, res))
    return out


def network_masks(seed: int, step: int, model_cfg, B: int, p: float, device=None) -> Dict[int, torch.Tensor]:
    return {i: keep_mask(seed, step, i, B, h, w, p, device) for i, (h, w) in enumerate(layer_shapes(model_cfg))}


def _block_dropout(sd, pfx: str, spec: dict, x, emb, keep: Optional[torch.Tensor], s: float):
    """oracle.edm_oracle._block with `x * keep * s` in front of conv1 (adm_blocks.py:167)."""
    g = lambda n: sd.get(pfx + n)  # noqa: E731
    orig = x
    x = O._conv(F.silu(O._gn(x, g("norm0.weight"), g("norm0.bias"))), g("conv0.weight"), g("conv0.bias"),
                up=spec["up"], down=spec["down"])
    params = O._linear(emb, g("affine.weight"), g("affine.bias")).unsqueeze(2).unsqueeze(3)
    sc, shift = params.chunk(2, dim=1)
    x = F.silu(torch.addcmul(shift, O._gn(x, g("norm1.weight"), g("norm1.bias")), sc + 1))
    if keep is not None:
        x = x * keep.to(x.dtype) * s
    x = O._conv(x, g("conv1.weight"), g("conv1.bias"))
    if spec["cin"] != spec["cout"] or spec["up"] or spec["down"]:
        x = x + O._conv(orig, g("skip.weight"), g("skip.bias"), up=spec["up"], down=spec["down"])
    else:
        x = x + orig
    if spec["attn"]:
        n, c, h, w = x.shape
        heads = c // 64
        qkv = O._conv(O._gn(x, g("norm2.weight"), g("norm2.bias")), g("qkv.weight"), g("qkv.bias"))
        q, k, v = qkv.reshape(n * heads, c // heads, 3, -1).unbind(2)
        wts = torch.einsum("ncq,nck->nqk", q.float(), (k / math.sqrt(k.shape[1])).float()).softmax(dim=2).to(q.dtype)
        a = torch.einsum("nqk,nck->ncq", wts, v)
        x = O._conv(a.reshape(n, c, h, w), g("proj.weight"), g("proj.bias")) + x
    return x


def unet_forward_dropout(sd, model_cfg, x, noise_labels, cond=None, masks: Optional[Dict[int, torch.Tensor]] = None,
                         s: float = 1.0):
    """oracle.edm_oracle.unet_forward with masks[layer] (bool / 0-1 [B, 64, H, W]) applied before conv1 of every block;
    masks None: no dropout."""
    ch = model_cfg["ch"]
    half = ch // 2
    freqs = torch.arange(half, device=noise_labels.device).to(noise_labels.dtype) / half
    freqs = (1 / 10000) ** freqs
    e = noise_labels.ger(freqs)
    emb = torch.cat([e.cos(), e.sin()], dim=1)
    emb = F.silu(O._linear(emb, sd["map_layer0.weight"], sd["map_layer0.bias"]))
    emb = F.silu(O._linear(emb, sd["map_layer1.weight"], sd["map_layer1.bias"]))
    if model_cfg.get("self_cond", False):
        x = torch.cat([torch.zeros_like(x), x], dim=1)
    cc = model_cfg.get("cond_channels", 0) if model_cfg.get("cat_cond", False) else 0
    if cc > 0:
        if cond is None:
            cond = torch.zeros(x.shape[0], cc, x.shape[2], x.shape[3], dtype=x.dtype, device=x.device)
        x = torch.cat([cond, x], dim=1)
    plan = O.unet_plan(model_cfg)
    skips = []
    layer = 0

    def keep_of(i):
        return None if masks is None else masks[i]

    for spec in plan["enc"]:
        pfx = f"enc.{spec['name']}."
        if spec["kind"] == "conv":
            x = O._conv(x, sd[pfx + "weight"], sd[pfx + "bias"])
        else:
            x = _block_dropout(sd, pfx, spec, x, emb, keep_of(layer), s)
            layer += 1
        skips.append(x)
    for spec in plan["dec"]:
        if x.shape[1] != spec["cin"]:
            x = torch.cat([x, skips.pop()], dim=1)
        x = _block_dropout(sd, f"dec.{spec['name']}.", spec, x, emb, keep_of(layer), s)
        layer += 1
    return O._conv(F.silu(O._gn(x, sd["out_norm.weight"], sd["out_norm.bias"])), sd["out_conv.weight"], sd["out_conv.bias"])


def reference_step_dropout(named, model_cfg, x, sigma, noise, cond, mask, masks, s, chunk=8):
    """reference_step of tests/test_gpu_train_batch.py (float64 loss and gradients of one step, evaluated in chunks of
    samples) through unet_forward_dropout with masks[layer] [B, 64, H, W] (sliced per chunk) and scale s."""
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
            sg = sigma.reshape(-1)[i:j].to(dev, torch.float64).reshape(-1, 1, 1, 1)
            den = sg ** 2 + 1.0                                                 # sigma_data = 1
            c_skip, c_out, c_in, c_noise = 1.0 / den, sg / den.sqrt(), 1.0 / den.sqrt(), sg.log() / 4
            x_noise = xs + ms * ns * sg
            mk = None if masks is None else {k: v[i:j].to(dev) for k, v in masks.items()}
            f_x = unet_forward_dropout(leaves, model_cfg, c_in * x_noise, c_noise.flatten(), cs, mk, s)
            d_x = c_skip * x_noise + c_out * f_x
            per = (O.loss_weight(sg) * (d_x * ms - xs * ms) ** 2).sum(dim=(1, 2, 3))
            part = per.mean() * ((j - i) / B)
            gs = torch.autograd.grad(part, list(leaves.values()))
            for k, g in zip(leaves, gs):
                grads[k] += g
            loss += float(part.detach())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = flags
    return loss, grads
