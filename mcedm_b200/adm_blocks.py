"""Drop-in host mirror of the reference ADM/EDM U-Net (`models/adm_blocks.py`).

`DhariwalUNet(hparams)` has the reference constructor, the reference `forward(x, noise_labels, cond,
...)` signature (models/adm_blocks.py:364), and registers parameters and buffers under the same names,
shapes and order (so reference checkpoints / `state_dict`s load with `strict=True`, `deepcopy` for the
EMA works, and Adam sees the same parameter list).  Initialisation consumes the torch RNG in the same
order with the same formulas (models/adm_blocks.py:10-15), so `torch.manual_seed(s)` gives bit-identical
weights in both code bases.

What differs is everything below the Python surface: the sub-modules here are parameter containers
only; the arithmetic runs in hand-written sm_100a kernels through `mcedm_b200.engine.UNetEngine`
(C ABI in include/mcedm_b200.h).  There is no PyTorch/CPU fallback: calling forward on a non-CUDA tensor,
or without the built library, raises.

`dropout` (p in [0, 1)) applies where the reference applies it, to conv1's operand in every UNetBlock, and only in
training mode: there every forward runs the fp16 training plan (train16_engine.py), whose kernels draw the masks from a
counter-based Philox stream keyed by the engine's `dropout_seed` and `dropout_step` (DESIGN.md §3).  The masks are
i.i.d. Bernoulli(1 - p) with scale 1 / (1 - p), as in the reference, but not torch's bits; dropout draws nothing from
torch's generators.  In eval mode p plays no part, so a checkpoint trained with dropout samples on the inference plans.
"""
from __future__ import annotations

import numpy as np
import torch


def _init_tensor(shape, mode: str, fan_in: int, fan_out: int) -> torch.Tensor:
    # same draws and the same float arithmetic as the reference initialiser (adm_blocks.py:10-15)
    if mode == "kaiming_uniform":
        return np.sqrt(3 / fan_in) * (torch.rand(*shape) * 2 - 1)
    if mode == "kaiming_normal":
        return np.sqrt(1 / fan_in) * torch.randn(*shape)
    if mode == "xavier_uniform":
        return np.sqrt(6 / (fan_in + fan_out)) * (torch.rand(*shape) * 2 - 1)
    if mode == "xavier_normal":
        return np.sqrt(2 / (fan_in + fan_out)) * torch.randn(*shape)
    raise ValueError(f'Invalid init mode "{mode}"')


class _Container(torch.nn.Module):
    def forward(self, *a, **k):  # noqa: D401
        raise RuntimeError(
            f"{type(self).__name__} is a parameter container in mcedm_b200; the arithmetic runs inside "
            "DhariwalUNet.forward (fused sm_100a kernels), not per sub-module")


class Linear(_Container):
    """Parameters of models/adm_blocks.py:19-32."""

    def __init__(self, in_features, out_features, bias=True, init_mode="kaiming_normal", init_weight=1, init_bias=0):
        super().__init__()
        self.in_features, self.out_features = in_features, out_features
        kw = dict(mode=init_mode, fan_in=in_features, fan_out=out_features)
        self.weight = torch.nn.Parameter(_init_tensor([out_features, in_features], **kw) * init_weight)
        self.bias = torch.nn.Parameter(_init_tensor([out_features], **kw) * init_bias) if bias else None


class Conv2d(_Container):
    """Parameters (and the resample_filter buffer) of models/adm_blocks.py:36-56."""

    def __init__(self, in_channels, out_channels, kernel, bias=True, up=False, down=False, resample_filter=(1, 1),
                 fused_resample=False, init_mode="kaiming_normal", init_weight=1, init_bias=0):
        assert not (up and down)
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.up, self.down, self.fused_resample = up, down, fused_resample
        kw = dict(mode=init_mode, fan_in=in_channels * kernel * kernel, fan_out=out_channels * kernel * kernel)
        self.weight = torch.nn.Parameter(
            _init_tensor([out_channels, in_channels, kernel, kernel], **kw) * init_weight) if kernel else None
        self.bias = torch.nn.Parameter(_init_tensor([out_channels], **kw) * init_bias) if kernel and bias else None
        f = torch.as_tensor(list(resample_filter), dtype=torch.float32)
        f = f.ger(f).unsqueeze(0).unsqueeze(1) / f.sum().square()
        self.register_buffer("resample_filter", f if up or down else None)
        if (up or down) and list(resample_filter) != [1, 1]:
            raise NotImplementedError("only the [1,1] resample filter (2x2 mean / nearest x2) has a kernel")


class GroupNorm(_Container):
    """Parameters of models/adm_blocks.py:86-92."""

    def __init__(self, num_channels, num_groups=32, min_channels_per_group=4, eps=1e-5):
        super().__init__()
        self.num_groups = min(num_groups, num_channels // min_channels_per_group)
        self.eps = eps
        self.weight = torch.nn.Parameter(torch.ones(num_channels))
        self.bias = torch.nn.Parameter(torch.zeros(num_channels))


class UNetBlock(_Container):
    """Parameters of models/adm_blocks.py:124-157, registered in the same order."""

    def __init__(self, in_channels, out_channels, emb_channels, up=False, down=False, attention=False,
                 num_heads=None, channels_per_head=64, dropout=0, skip_scale=1, eps=1e-5, resample_filter=(1, 1),
                 resample_proj=False, adaptive_scale=True, init=None, init_zero=None, init_attn=None):
        super().__init__()
        init = dict(init or {})
        init_zero = dict(init_zero if init_zero is not None else dict(init_weight=0))
        self.in_channels, self.out_channels, self.emb_channels = in_channels, out_channels, emb_channels
        self.num_heads = 0 if not attention else (num_heads if num_heads is not None
                                                  else out_channels // channels_per_head)
        self.dropout, self.skip_scale, self.adaptive_scale = dropout, skip_scale, adaptive_scale
        self.up, self.down = up, down
        self.norm0 = GroupNorm(num_channels=in_channels, eps=eps)
        self.conv0 = Conv2d(in_channels, out_channels, kernel=3, up=up, down=down, resample_filter=resample_filter,
                            **init)
        self.affine = Linear(emb_channels, out_channels * (2 if adaptive_scale else 1), **init)
        self.norm1 = GroupNorm(num_channels=out_channels, eps=eps)
        self.conv1 = Conv2d(out_channels, out_channels, kernel=3, **init_zero)
        self.skip = None
        if out_channels != in_channels or up or down:
            kernel = 1 if resample_proj or out_channels != in_channels else 0
            self.skip = Conv2d(in_channels, out_channels, kernel=kernel, up=up, down=down,
                               resample_filter=resample_filter, **init)
        if self.num_heads:
            self.norm2 = GroupNorm(num_channels=out_channels, eps=eps)
            self.qkv = Conv2d(out_channels, out_channels * 3, kernel=1, **(init_attn if init_attn is not None else init))
            self.proj = Conv2d(out_channels, out_channels, kernel=1, **init_zero)


class PositionalEmbedding(_Container):
    def __init__(self, num_channels, max_positions=10000, endpoint=False):
        super().__init__()
        self.num_channels, self.max_positions, self.endpoint = num_channels, max_positions, endpoint

    def frequencies(self, dtype=torch.float32) -> torch.Tensor:
        # models/adm_blocks.py:192-196, evaluated with torch so the table matches the reference bit for bit
        freqs = torch.arange(start=0, end=self.num_channels // 2).to(dtype)
        freqs = freqs / (self.num_channels // 2 - (1 if self.endpoint else 0))
        return (1 / self.max_positions) ** freqs


def _has(node, key) -> bool:
    return hasattr(node, key)


class DhariwalUNet(torch.nn.Module):
    """B200-native ADM U-Net with the reference's constructor and call signature."""

    def __init__(self, hparams):
        super().__init__()
        m = hparams.model
        ch, out_channels = m.ch, m.out_ch
        channel_mult = tuple(m.ch_mult)
        cond_channels = m.cond_channels if _has(m, "cond_channels") else 0
        attn_resolutions = list(m.attn_resolutions)
        resolution, num_res_blocks = m.resolution, m.num_res_blocks
        self.resolution = resolution
        augment_dim, label_dim = m.augment_dim, m.label_dim
        dropout, self.label_dropout = m.dropout, m.label_dropout
        if not 0.0 <= float(dropout) < 1.0:
            raise ValueError(f"dropout must lie in [0, 1), got {dropout}")
        self.dropout = float(dropout)                  # one p for every UNetBlock, as in the reference
        emb_channels = ch
        init = dict(init_mode="kaiming_uniform", init_weight=np.sqrt(1 / 3), init_bias=np.sqrt(1 / 3))
        init_zero = dict(init_mode="kaiming_uniform", init_weight=0, init_bias=0)
        block_kwargs = dict(emb_channels=emb_channels, channels_per_head=64, dropout=dropout, init=init,
                            init_zero=init_zero)
        self.self_condition = m.self_cond if _has(m, "self_cond") else False
        self.cat_condition = m.cat_cond if _has(m, "cat_cond") else False
        self.dx_cond = m.dx_cond if _has(m, "dx_cond") else False
        self.cat_dx = m.cat_dx if _has(m, "cat_dx") else False
        # features of the reference network that have no sm_100a kernel (off in every shipped m-cedm config)
        unsupported = []
        if self.dx_cond:
            unsupported.append("dx_cond")
        if augment_dim:
            unsupported.append("augment_dim")
        if label_dim:
            unsupported.append("label_dim")
        if cond_channels > 0 and not self.cat_condition:
            unsupported.append("cat_cond=False (separate conditioning encoder)")
        if ch != 64 or any(int(c) != 1 for c in channel_mult):
            unsupported.append("ch*ch_mult != 64 (kernels are specialised for 64-channel tensors)")
        if unsupported:
            raise NotImplementedError("mcedm_b200.DhariwalUNet: unsupported options: " + ", ".join(unsupported))

        in_channels = m.in_channels
        # self-conditioning stacks a second copy of the state in front of it (adm_blocks.py:235, :321-324); the first
        # conv sees [cond | x_self_cond | x], so the kernels treat the self-conditioning block as extra cond channels
        self.sc_channels = in_channels if self.self_condition else 0
        self.in_channels = in_channels + self.sc_channels + (cond_channels if self.cat_condition else 0)
        self.cond_channels = cond_channels
        self.cat_channels = self.in_channels - in_channels            # channels concatenated in front of x
        self.x_channels = in_channels
        self.out_channels = out_channels
        self.ch = ch * channel_mult[0]

        # ---- parameters, in the reference's registration order (models/adm_blocks.py:239-317) ----
        self.map_noise = PositionalEmbedding(num_channels=ch)
        self.map_augment = None
        self.map_layer0 = Linear(ch, emb_channels, **init)
        self.map_layer1 = Linear(emb_channels, emb_channels, **init)
        self.map_label = None
        self.cond_enc = None
        self.dx_enc = None
        self.combine_enc = None
        self.enc = torch.nn.ModuleDict()
        cout = self.in_channels
        for level, mult in enumerate(channel_mult):
            res = resolution >> level
            if level == 0:
                cin, cout = cout, ch * mult
                self.enc[f"{res}x{res}_conv"] = Conv2d(cin, cout, kernel=3, **init)
            else:
                self.enc[f"{res}x{res}_down"] = UNetBlock(cout, cout, down=True, **block_kwargs)
            for idx in range(num_res_blocks):
                cin, cout = cout, ch * mult
                self.enc[f"{res}x{res}_block{idx}"] = UNetBlock(cin, cout, attention=(res in attn_resolutions),
                                                                **block_kwargs)
        skips = [block.out_channels for block in self.enc.values()]
        self.dec = torch.nn.ModuleDict()
        for level, mult in reversed(list(enumerate(channel_mult))):
            res = resolution >> level
            if level == len(channel_mult) - 1:
                self.dec[f"{res}x{res}_in0"] = UNetBlock(cout, cout, attention=True, **block_kwargs)
                self.dec[f"{res}x{res}_in1"] = UNetBlock(cout, cout, **block_kwargs)
            else:
                self.dec[f"{res}x{res}_up"] = UNetBlock(cout, cout, up=True, **block_kwargs)
            for idx in range(num_res_blocks + 1):
                cin = cout + skips.pop()
                cout = ch * mult
                self.dec[f"{res}x{res}_block{idx}"] = UNetBlock(cin, cout, attention=(res in attn_resolutions),
                                                                **block_kwargs)
        self.out_norm = GroupNorm(num_channels=cout)
        self.out_conv = Conv2d(cout, out_channels, kernel=3, **init_zero)
        self._engine = None

    # the engine holds packed bf16 weights and workspaces; it is not part of the module state
    def engine(self):
        if self._engine is None:
            from .engine import UNetEngine

            self._engine = UNetEngine(self)
        return self._engine

    def __deepcopy__(self, memo):
        import copy

        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            new.__dict__[k] = None if k == "_engine" else copy.deepcopy(v, memo)
        return new

    def __getstate__(self):
        d = dict(self.__dict__)
        d["_engine"] = None
        return d

    def forward(self, x, noise_labels, cond=None, x_self_cond=None, dx=None, class_labels=None, augment_labels=None):
        """F_x = U-Net(x, c_noise, cond): x [B,Cx,H,W] fp32 CUDA (already scaled by c_in), noise_labels [B] or [1],
        cond [B,Cc,H,W] fp32 or None (zeros, as in models/adm_blocks.py:327-331). Returns [B,out_ch,H,W] fp32."""
        if dx is not None or class_labels is not None or augment_labels is not None:
            raise NotImplementedError("dx conditioning, class and augment labels are not supported")
        if x_self_cond is not None and not self.self_condition:
            raise ValueError("x_self_cond given to a network built without self_cond")
        if self.self_condition:                                       # cat_conditioning, adm_blocks.py:319-333
            sc = torch.zeros_like(x) if x_self_cond is None else x_self_cond
            if self.cond_channels > 0:
                if cond is None:
                    cond = torch.zeros(x.shape[0], self.cond_channels, x.shape[2], x.shape[3], device=x.device,
                                       dtype=x.dtype)
                cond = torch.cat([cond, sc], dim=1)
            else:
                cond = sc
        if self.training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # training: the autograd node's backward runs the hand-written backward kernels (train_engine.py)
            from .autograd import UNetFunction

            return UNetFunction.apply(self, x, noise_labels, cond, *self.parameters())
        if self.training and self.dropout > 0:
            # only the training forward has dropout kernels: a training-mode call without autograd runs it as well
            # (its saved tape is dropped), so no training-mode evaluation silently skips the masks
            eng = self.engine()
            out = eng.forward_train(x, noise_labels, cond)
            eng._tape = None
            return out
        return self.engine().forward(x, noise_labels, cond)
