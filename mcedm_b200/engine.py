"""Launch plan of the B200-native ADM U-Net forward pass.

`UNetEngine` turns a `DhariwalUNet` parameter container into (a) packed device weights in the layouts
the sm_100a kernels want and (b) a fixed sequence of C-ABI launches per forward call
(include/mcedm_b200.h).  It follows DhariwalUNet.forward / UNetBlock.forward of the reference
(models/adm_blocks.py:364-404, :159-181) with these fusions:

  * every tensor in the trunk is a 64-channel NHWC tensor; the decoder's channel concat
    (adm_blocks.py:401) never materialises — conv0 of those blocks reads two sources;
  * GroupNorm statistics come out of the producing conv's epilogue (per-tile partial sums);
  * GroupNorm-apply + (1+scale)/shift + SiLU + the 2x up/down resampling of conv0 is ONE pass that
    writes the bf16 tensor-core operand;
  * bias, residual add (identity / 2x2-mean / nearest-x2 skip) and the 1x1 skip projection of the
    128->64 blocks are folded into conv1's implicit GEMM (extra K segments on the raw input);
  * q/k/v de-interleave is a one-time weight-row permutation; softmax(QK^T)V never leaves the SM.

HBM layout: fp32 NHWC for the residual stream and conv0 outputs, bf16 NHWC for every tensor-core
operand.  Workspaces are torch tensors owned by this object, keyed by batch size.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional

import torch

from . import _lib as L
from .fused_engine import FusedMixin
from .pack_plan import PackMixin
from .precise_engine import PreciseMixin
from .train_engine import TrainMixin
from .train16_engine import Train16Mixin

WEIGHT_EPOCH = [0]
_SEG9 = [(ky - 1, kx - 1) for ky in range(3) for kx in range(3)]


def pack_conv3x3(weight: torch.Tensor, n_out_pad: Optional[int] = None, dtype=torch.bfloat16) -> torch.Tensor:
    """[Cout, 64*n_src, k, k] fp32 -> 16-bit [n_src*k*k][Cout(_pad)][64], segment order (source, ky, kx)."""
    cout, cin, k, _ = weight.shape
    n_src = cin // 64
    w = weight.detach().reshape(cout, n_src, 64, k, k).permute(1, 3, 4, 0, 2).reshape(n_src * k * k, cout, 64)
    if n_out_pad is not None and n_out_pad > cout:
        w = torch.cat([w, w.new_zeros(w.shape[0], n_out_pad - cout, 64)], dim=1)
    return w.to(dtype).contiguous()


class _Block:
    """Packed weights + static description of one UNetBlock."""

    def __init__(self, name: str, mod, aff_index: int):
        self.name = name
        self.mod = mod
        self.n_src = mod.in_channels // 64
        self.up, self.down = mod.up, mod.down
        self.attn = bool(mod.num_heads)
        self.aff_index = aff_index
        self.skip_conv = mod.skip is not None and mod.skip.weight is not None
        if mod.num_heads not in (0, 1):
            raise NotImplementedError("attention kernel handles one 64-channel head")
        if not mod.adaptive_scale:
            raise NotImplementedError("adaptive_scale=False has no kernel")

    def pack(self, dtype=torch.bfloat16):
        m = self.mod
        self.w0 = pack_conv3x3(m.conv0.weight, dtype=dtype)
        self.b0 = m.conv0.bias.detach().float().contiguous()
        w1 = pack_conv3x3(m.conv1.weight, dtype=dtype)
        b1 = m.conv1.bias.detach().float()
        if self.skip_conv:
            w1 = torch.cat([w1, pack_conv3x3(m.skip.weight, dtype=dtype)], dim=0).contiguous()
            b1 = b1 + m.skip.bias.detach().float()
        self.w1, self.b1 = w1, b1.contiguous()
        self.g0, self.be0 = m.norm0.weight.detach().float().contiguous(), m.norm0.bias.detach().float().contiguous()
        self.g1, self.be1 = m.norm1.weight.detach().float().contiguous(), m.norm1.bias.detach().float().contiguous()
        if self.attn:
            # reference channel order is (c*3 + {q,k,v}) (adm_blocks.py:175-176) -> blocked (q | k | v)
            perm = torch.arange(192, device=m.qkv.weight.device).reshape(64, 3).t().reshape(-1)
            self.wqkv = m.qkv.weight.detach()[perm].reshape(1, 192, 64).to(dtype).contiguous()
            self.bqkv = m.qkv.bias.detach().float()[perm].contiguous()
            self.wproj = m.proj.weight.detach().reshape(1, 64, 64).to(dtype).contiguous()
            self.bproj = m.proj.bias.detach().float().contiguous()
            self.g2 = m.norm2.weight.detach().float().contiguous()
            self.be2 = m.norm2.bias.detach().float().contiguous()


class UNetEngine(TrainMixin, Train16Mixin, FusedMixin, PreciseMixin, PackMixin):
    supports_ss_rows = True      # forward_static can take precomputed (scale | shift) rows (embedding_table)

    def __init__(self, unet):
        self.unet = unet
        self.lib = L.lib()
        self.blocks_enc: List[_Block] = []
        self.blocks_dec: List[_Block] = []
        aff = 0
        self.conv_in_name = None
        self._attn_levels = set()
        level = 0
        for name, mod in unet.enc.items():
            if name.endswith("_conv"):
                self.conv_in_name = name
            else:
                if mod.down:
                    level += 1
                self.blocks_enc.append(_Block("enc." + name, mod, aff))
                if mod.num_heads:
                    self._attn_levels.add(level)
                aff += 1
        for name, mod in unet.dec.items():
            if mod.up:
                level -= 1
            self.blocks_dec.append(_Block("dec." + name, mod, aff))
            if mod.num_heads:
                self._attn_levels.add(level)
            aff += 1
        self.n_aff = aff
        self._packed_key = None
        self.use_rows = True     # row-resident conv kernel (conv_rows.cu) for the 128-pixel-wide level
        self.use_flat = True     # padded-flat conv kernel (conv_flat.cu) for the narrower levels
        self._ws: Dict[tuple, dict] = {}
        self._graphs: Dict[tuple, tuple] = {}
        self._tape = None
        # format of the 16-bit tensor-core operands (include/mcedm_b200.h `op_fmt`): inference defaults to fp16
        # (11 significand bits: ~8x smaller operand-rounding error than bf16, same throughput; activations are
        # normalised and weights O(1), so the narrower range is safe); training always runs bf16.
        self.infer_fmt = 1
        self._fmt = 1
        # training plan: "fused16" = 16-bit activations end to end, fp16 operands, loss-scaled fp16 gradients
        # (train16_engine.py); "fp32" = the fp32-stream plan with bf16 operands (train_engine.py; any field width)
        self.train_plan = os.environ.get("MCEDM_TRAIN_PLAN", "fused16")
        # dropout masks of the training forward (train16_engine.py): Philox key = seed (torch.initial_seed() when the
        # engine first trains, unless set), counter word = step (one per training-mode forward)
        self.dropout_seed: Optional[int] = None
        self.dropout_step = 0
        # dynamic loss scaling of the fused16 plan's backward (loss_scale.LossScaler; None = the static scale)
        self.loss_scaler = None
        # inference plan: True = GroupNorm fused into the convs + 16-bit activations (fused_engine.py);
        # False = the unfused fp32-stream plan below (what training's forward uses)
        self.fused = os.environ.get("MCEDM_FUSED", "1") != "0"
        # "fp16": the plans above (bar 1e-2);  "fp32": split-operand fp32-accuracy plan (bar 1e-4, precise_engine.py)
        self.precision = "fp16"
        self._gn_coef: Dict[tuple, torch.Tensor] = {}

    @property
    def train_fmt(self) -> int:
        """16-bit operand format of the training plan (include/mcedm_b200.h `op_fmt`)."""
        return 1 if self.train_plan == "fused16" else 0

    # ------------------------------------------------------------------ weights
    def _param_key(self):
        # WEIGHT_EPOCH counts in-place parameter updates made by the fused optimizer kernels (no autograd version bump)
        return (WEIGHT_EPOCH[0], self._fmt) + tuple((p.data_ptr(), p._version) for p in self.unet.parameters())

    def pack(self, force: bool = False):
        key = self._param_key()
        if not force and key == self._packed_key:
            return
        u = self.unet
        dev = u.out_conv.weight.device
        if dev.type != "cuda":
            raise L.McedmError("mcedm_b200.DhariwalUNet parameters must live on a CUDA (sm_100) device; "
                               "there is no CPU path")
        dt = torch.float16 if self._fmt else torch.bfloat16
        if getattr(self, "_pack_dtype_override", None) is not None:
            dt = self._pack_dtype_override
        with torch.no_grad():
            for b in self.blocks_enc + self.blocks_dec:
                b.pack(dt)
            cin = u.enc[self.conv_in_name]
            self.w_in = cin.weight.detach().float().contiguous()
            self.b_in = cin.bias.detach().float().contiguous()
            # the same weights for the tensor-core first conv (conv_in_tc.cu): [ky][co][k = kx*Cin + c], zero-padded to 64
            c_tot = cin.weight.shape[1]
            if 3 * c_tot <= 15 and cin.weight.shape[0] == 64:
                wk = cin.weight.detach().float().permute(2, 0, 3, 1).reshape(3, 64, 3 * c_tot)      # ky, co, (kx, c)
                self.w_in_tc = torch.cat([wk, wk.new_zeros(3, 64, 64 - 3 * c_tot)], 2).to(dt).contiguous()
            else:
                self.w_in_tc = None
            self.w_out = pack_conv3x3(u.out_conv.weight, n_out_pad=16, dtype=dt)
            self.b_out = torch.cat([u.out_conv.bias.detach().float(),
                                    torch.zeros(16 - u.out_channels, device=dev)]).contiguous()
            self.g_out = u.out_norm.weight.detach().float().contiguous()
            self.be_out = u.out_norm.bias.detach().float().contiguous()
            if getattr(self, "freqs", None) is None or self.freqs.device != dev:   # constants: one H2D copy ever
                self.freqs = u.map_noise.frequencies(torch.float32).to(dev).contiguous()
            self.w_m0, self.b_m0 = u.map_layer0.weight.detach().float().contiguous(), \
                u.map_layer0.bias.detach().float().contiguous()
            self.w_m1, self.b_m1 = u.map_layer1.weight.detach().float().contiguous(), \
                u.map_layer1.bias.detach().float().contiguous()
            blocks = self.blocks_enc + self.blocks_dec
            self.aff_w = torch.stack([b.mod.affine.weight.detach().float() for b in blocks]).contiguous()
            self.aff_b = torch.stack([b.mod.affine.bias.detach().float() for b in blocks]).contiguous()
        self._packed_key = key

    # ------------------------------------------------------------------ workspaces
    def _workspace(self, B: int, H: int, W: int, dev) -> dict:
        key = (B, H, W, dev.index)
        ws = self._ws.get(key)
        if ws is not None:
            return ws
        f32 = dict(device=dev, dtype=torch.float32)
        bf = dict(device=dev, dtype=torch.bfloat16)
        ws = {}
        # residual-stream tensors are allocated per block output on first use (see _tensor)
        ws["pool"] = {}
        ws["h"] = torch.empty(B * H * W * 64, **f32)            # conv0 output (largest resolution)
        ws["h_st"] = torch.empty(B * (H * W // 128 + H // 4 + 8) * 4 * 32, **f32)
        ws["a"] = [torch.empty(B * H * W * 64, **bf) for _ in range(2)]   # normalised operands (2 sources)
        ws["raw"] = [torch.empty(B * H * W * 64, **bf) for _ in range(2)]  # raw bf16 copies for 1x1 skips
        ws["a1"] = torch.empty(B * H * W * 64, **bf)
        att_pix = max([B * (H >> lv) * (W >> lv) for lv in self._attn_levels] or [128])
        ws["qkv"] = torch.empty(att_pix * 192, **bf)
        ws["att"] = torch.empty(att_pix * 64, **bf)
        ws["o16"] = torch.empty(B * H * W * 16, **f32)
        ws["ss"] = torch.empty(self.n_aff * B * 128, **f32)
        ws["F"] = torch.empty(B, self.unet.out_channels, H, W, **f32)
        self._ws[key] = ws
        return ws

    @staticmethod
    def _tensor(ws, name: str, B: int, H: int, W: int, dev):
        """(fp32 NHWC tensor, GroupNorm partial-sum records) of a named activation; the record buffer holds
        up to 4 records per 128-pixel tile (the conv_rows format)."""
        t = ws["pool"].get(name)
        if t is None:
            t = (torch.empty(B, H, W, 64, device=dev, dtype=torch.float32),
                 torch.empty(B * (H * W // 128 + H // 4 + 8) * 4, 16, 2, device=dev, dtype=torch.float32))
            ws["pool"][name] = t
        return t

    # ------------------------------------------------------------------ launches
    def _conv(self, srcs, segs, w, bias, B, H, W, N, out, out_bf16, res, res_mode, stats, st, fmt=None):
        L.check(self.lib.mcedm_conv_igemm(
            L.ptr_array(srcs), len(srcs), L.int_array([s[0] for s in segs]), L.int_array([s[1] for s in segs]),
            L.int_array([s[2] for s in segs]), len(segs), L.ptr(w), L.ptr(bias), B, H, W, N, L.ptr(out), out_bf16,
            L.ptr(res), res_mode, L.ptr(stats), self._fmt if fmt is None else fmt, st), "conv_igemm")

    def _flat_geom(self, H, W):
        pitch, blk = C.c_int(0), C.c_int(0)
        L.check(self.lib.mcedm_flat_geometry(H, W, C.byref(pitch), C.byref(blk)), "flat_geometry")
        L.LAUNCHES[0] -= 1
        return pitch.value, blk.value

    def _flat_buffers(self, ws, B, H, W, dev):
        """Zero-padded flat bf16 operand buffers of one level: (two conv0 sources, conv1 source, pitch, blk).
        Allocated zeroed once; the kernels only ever write data positions, so the padding stays zero."""
        key = ("flat", H, W)
        fb = ws["pool"].get(key)
        if fb is None:
            pitch, blk = self._flat_geom(H, W)
            mk = lambda: torch.zeros(B * blk * 64, device=dev, dtype=torch.bfloat16)  # noqa: E731
            fb = ([mk(), mk()], mk(), pitch, blk)
            ws["pool"][key] = fb
        return fb

    def _conv_flat(self, src, w, bias, B, H, W, out, res, res_mode, stats, st):
        L.check(self.lib.mcedm_conv_flat(L.ptr(src), L.ptr(w), L.ptr(bias), B, H, W, 64, L.ptr(out), L.ptr(res),
                                         res_mode, L.ptr(stats), self._fmt, st), "conv_flat")

    def _conv3x3(self, halo, ctr, w, bias, B, H, W, N, out, res, res_mode, stats, st, flat=None):
        if flat is not None:
            pitch, blk = flat
            parts = 4 * (blk // 128)
            if len(halo) == 2:
                # split K over the two sources, second pass accumulates in place (see the W == 128 case)
                self._conv_flat(halo[0], w[:9], None, B, H, W, out, None, 0, None, st)
                self._conv_flat(halo[1], w[9:18], bias, B, H, W, out, out, 1, stats, st)
                return parts
            if ctr:
                # 1x1 skip projection of the raw (dense) block input first, then the 3x3 part accumulates onto
                # it in place (conv_flat prefetches its residual; conv_igemm's residual path is the slow one)
                self._conv(list(ctr), [(i, 0, 0) for i in range(len(ctr))], w[9:], None, B, H, W, N, out, 0, None, 0,
                           None, st)
                self._conv_flat(halo[0], w[:9], bias, B, H, W, out, out, 1, stats, st)
                return parts
            self._conv_flat(halo[0], w, bias, B, H, W, out, res, res_mode, stats, st)
            return parts
        """3x3 conv of the concatenated `halo` sources (+ 1x1 of the `ctr` sources) -> fp32 out (+ stats).
        Returns the number of statistics records per image written to `stats`."""
        if W == 128 and self.use_rows and res_mode in (0, 1, 2) and N in (16, 64):
            if len(halo) == 1:
                L.check(self.lib.mcedm_conv_rows(L.ptr_array(halo), 1, L.ptr_array(ctr) if ctr else None, len(ctr),
                                                 L.ptr(w), L.ptr(bias), B, H, N, L.ptr(out), 0, L.ptr(res), res_mode,
                                                 L.ptr(stats), self._fmt, st), "conv_rows")
                return 4 * H
            if len(halo) == 2 and not ctr and res_mode == 0:
                # K = 1152 weights (144 KB) cannot stay resident next to the row ring: split K over the two
                # sources; the second pass accumulates onto the first pass's fp32 result in place.
                L.check(self.lib.mcedm_conv_rows(L.ptr_array(halo[:1]), 1, None, 0, L.ptr(w[:9]), None, B, H, N,
                                                 L.ptr(out), 0, None, 0, None, self._fmt, st), "conv_rows")
                L.check(self.lib.mcedm_conv_rows(L.ptr_array(halo[1:]), 1, None, 0, L.ptr(w[9:]), L.ptr(bias), B, H, N,
                                                 L.ptr(out), 0, L.ptr(out), 1, L.ptr(stats), self._fmt, st), "conv_rows")
                return 4 * H
        segs = [(i, dy, dx) for i in range(len(halo)) for (dy, dx) in _SEG9]
        segs += [(len(halo) + i, 0, 0) for i in range(len(ctr))]
        self._conv(list(halo) + list(ctr), segs, w, bias, B, H, W, N, out, 0, res, res_mode, stats, st)
        return H * W // 128

    def _gn_apply(self, x, stats, parts, gamma, beta, ss, ss_stride, act, resample, B, Hin, Win, out, raw, st,
                  eps=1e-5, flat=None, meanrstd=None):
        pitch, blk = flat if flat is not None else (0, 0)
        coef = self._gn_coef.get((B, x.device.index))
        if coef is None:
            coef = self._gn_coef[(B, x.device.index)] = torch.empty(B, 128, device=x.device, dtype=torch.float32)
        L.check(self.lib.mcedm_gn_apply(L.ptr(x), L.ptr(stats), L.ptr(gamma), L.ptr(beta), L.ptr(ss), ss_stride, 64,
                                        eps, act, resample, B, Hin, Win, parts, pitch, blk, L.ptr(out), L.ptr(raw),
                                        L.ptr(meanrstd), L.ptr(coef), self._fmt, st), "gn_apply")
        L.LAUNCHES[0] += 1      # finalize + streaming pass

    def _run_block(self, blk: _Block, inputs, B, H_in, W_in, ws, emb_stride, st, dev):
        """inputs: list of (fp32 NHWC tensor, stats, parts) at H_in x W_in. Returns ((out, stats, parts), H, W)."""
        if blk.up:
            H, W, rs, res_mode = H_in * 2, W_in * 2, 1, 2
        elif blk.down:
            H, W, rs, res_mode = H_in // 2, W_in // 2, 2, 3
        else:
            H, W, rs, res_mode = H_in, W_in, 0, 1
        eps = blk.mod.norm0.eps
        flat = None
        a_bufs, a1_buf = ws["a"], ws["a1"]
        if self.use_flat and W <= 64:
            a_bufs, a1_buf, pitch, fblk = self._flat_buffers(ws, B, H, W, dev)
            flat = (pitch, fblk)
        a_srcs, raw_srcs = [], []
        for i, (x, x_st, x_parts) in enumerate(inputs):
            raw = ws["raw"][i] if blk.skip_conv else None
            self._gn_apply(x, x_st, x_parts, blk.g0[64 * i:64 * (i + 1)], blk.be0[64 * i:64 * (i + 1)], None, 0, 1, rs,
                           B, H_in, W_in, a_bufs[i], raw, st, eps, flat=flat)
            a_srcs.append(a_bufs[i])
            if blk.skip_conv:
                raw_srcs.append(raw)
        h_parts = self._conv3x3(a_srcs, [], blk.w0, blk.b0, B, H, W, 64, ws["h"], None, 0, ws["h_st"], st, flat=flat)
        ss = ws["ss"][blk.aff_index * self._ss_rows * 128:]
        self._gn_apply(ws["h"], ws["h_st"], h_parts, blk.g1, blk.be1, ss, emb_stride, 1, 0, B, H, W, a1_buf, None, st,
                       eps, flat=flat)
        out, out_st = self._tensor(ws, blk.name, B, H, W, dev)
        if blk.skip_conv:
            parts = self._conv3x3([a1_buf], raw_srcs, blk.w1, blk.b1, B, H, W, 64, out, None, 0, out_st, st, flat=flat)
        else:
            parts = self._conv3x3([a1_buf], [], blk.w1, blk.b1, B, H, W, 64, out, inputs[0][0], res_mode, out_st, st,
                                  flat=flat)
        if blk.attn:
            self._gn_apply(out, out_st, parts, blk.g2, blk.be2, None, 0, 0, 0, B, H, W, ws["a1"], None, st, eps)
            self._conv([ws["a1"]], [(0, 0, 0)], blk.wqkv, blk.bqkv, B, H, W, 192, ws["qkv"], 1, None, 0, None, st)
            L.check(self.lib.mcedm_attention(L.ptr(ws["qkv"]), B, H * W, L.ptr(ws["att"]), None, self._fmt, st), "attention")
            out2, out2_st = self._tensor(ws, blk.name + ".attn", B, H, W, dev)
            self._conv([ws["att"]], [(0, 0, 0)], blk.wproj, blk.bproj, B, H, W, 64, out2, 0, out, 1, out2_st, st)
            out, out_st, parts = out2, out2_st, H * W // 128
        return (out, out_st, parts), H, W

    # ------------------------------------------------------------------ forward
    def _check_inputs(self, x, noise_labels, cond):
        u = self.unet
        if not x.is_cuda:
            raise L.McedmError("DhariwalUNet.forward needs CUDA tensors: the sm_100a kernels have no CPU fallback")
        if x.dtype != torch.float32 or x.dim() != 4 or x.shape[1] != u.x_channels:
            raise ValueError(f"x must be fp32 [B,{u.x_channels},H,W], got {x.dtype} {tuple(x.shape)}")
        B, _, H, W = x.shape
        if H * W % 128 != 0 or W > 128 or 128 % W != 0:
            raise ValueError(f"unsupported field size {H}x{W} (needs W | 128 and 128 | H*W)")
        dev = x.device
        x = x.contiguous()
        if u.cat_channels > 0:
            if cond is None:
                cond = torch.zeros(B, u.cat_channels, H, W, device=dev, dtype=torch.float32)
            if cond.shape != (B, u.cat_channels, H, W) or cond.dtype != torch.float32:
                raise ValueError(f"cond must be fp32 [B,{u.cat_channels},H,W], got {cond.dtype} {tuple(cond.shape)}")
            cond = cond.contiguous()
        else:
            cond = None
        nl = noise_labels.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
        if nl.numel() not in (1, B):
            raise ValueError(f"noise_labels must have 1 or B={B} entries, got {nl.numel()}")
        return x, nl, cond

    def _launch_all(self, x, nl, cond, out):
        """The launch sequence of one forward pass; no allocation, no host sync (CUDA-graph capturable
        once the workspace for this batch size exists)."""
        if self.precision == "fp32":
            if self._fmt != 1:
                raise ValueError("the fp32-accuracy plan splits operands into fp16 pairs: infer_fmt must be 1")
            return self._launch_all_precise(x, nl, cond, out)
        if self.fused and self._fmt == 1 and x.shape[-1] == 128:      # bf16 storage would miss the 1e-2 bar
            return self._launch_all_fused(x, nl, cond, out)
        u = self.unet
        B, _, H, W = x.shape
        dev = x.device
        ws = self._workspace(B, H, W, dev)
        st = L.stream_ptr()
        lib = self.lib
        Bemb = nl.numel()
        self._ss_rows = Bemb
        emb_stride = 128 if Bemb == B and B > 1 else 0
        L.check(lib.mcedm_emb_mlp(L.ptr(nl), L.ptr(self.freqs), L.ptr(self.w_m0), L.ptr(self.b_m0), L.ptr(self.w_m1),
                                  L.ptr(self.b_m1), L.ptr(self.aff_w), L.ptr(self.aff_b), self.n_aff, Bemb, None,
                                  L.ptr(ws["ss"]), st), "emb_mlp")
        t0, t0_st = self._tensor(ws, "conv_in", B, H, W, dev)
        L.check(lib.mcedm_conv_in(L.ptr(x), u.x_channels, L.ptr(cond), u.cat_channels, L.ptr(self.w_in),
                                  L.ptr(self.b_in), B, H, W, L.ptr(t0), L.ptr(t0_st), st), "conv_in")
        cur, ch, cw = (t0, t0_st, H * W // 128), H, W
        skips = [cur]
        for blk in self.blocks_enc:
            cur, ch, cw = self._run_block(blk, [cur], B, ch, cw, ws, emb_stride, st, dev)
            skips.append(cur)
        for blk in self.blocks_dec:
            inputs = [cur]
            if blk.n_src == 2:
                inputs.append(skips.pop())
            cur, ch, cw = self._run_block(blk, inputs, B, ch, cw, ws, emb_stride, st, dev)
        # out_conv(silu(out_norm(x)))  (adm_blocks.py:403), N padded to 16 for the tensor cores
        self._gn_apply(cur[0], cur[1], cur[2], self.g_out, self.be_out, None, 0, 1, 0, B, H, W, ws["a1"], None, st,
                       u.out_norm.eps)
        self._conv3x3([ws["a1"]], [], self.w_out, self.b_out, B, H, W, 16, ws["o16"], None, 0, None, st)
        L.check(lib.mcedm_head_to_nchw(L.ptr(ws["o16"]), 16, u.out_channels, B, H, W, L.ptr(out), st), "head_to_nchw")
        return out

    @torch.no_grad()
    def forward(self, x: torch.Tensor, noise_labels: torch.Tensor, cond: Optional[torch.Tensor]) -> torch.Tensor:
        x, nl, cond = self._check_inputs(x, noise_labels, cond)
        self._fmt = self.infer_fmt
        self.pack()
        B, _, H, W = x.shape
        out = torch.empty(B, self.unet.out_channels, H, W, device=x.device, dtype=torch.float32)
        return self._launch_all(x, nl, cond, out)

    # ------------------------------------------------------------------ CUDA-graph replay
    @torch.no_grad()
    def embedding_table(self, c_noise: torch.Tensor) -> Optional[torch.Tensor]:
        """Every block's (scale | shift) for K noise levels at once: fp32 [n_aff][K][128] from ONE mcedm_emb_mlp launch.
        The sampler knows its 99 noise levels up front, so the embedding MLP (a 40 us latency chain at the head of every
        evaluation: 3 dependent mat-vecs on one CTA per block) leaves the per-evaluation launch sequence; an evaluation
        then receives its row through `forward_static(..., ss_rows=table[:, k])`.  None when the current plan does not take
        external rows (unfused / fp32-accuracy plans)."""
        self._fmt = self.infer_fmt
        self.pack()
        if not (self.fused and self._fmt == 1 and self.precision != "fp32"):
            return None
        c = c_noise.to(dtype=torch.float32).reshape(-1).contiguous()
        K = c.numel()
        table = torch.empty(self.n_aff, K, 128, device=c.device, dtype=torch.float32)
        L.check(self.lib.mcedm_emb_mlp(L.ptr(c), L.ptr(self.freqs), L.ptr(self.w_m0), L.ptr(self.b_m0), L.ptr(self.w_m1),
                                       L.ptr(self.b_m1), L.ptr(self.aff_w), L.ptr(self.aff_b), self.n_aff, K, None,
                                       L.ptr(table), L.stream_ptr()), "emb_mlp")
        return table

    @torch.no_grad()
    def forward_static(self, x: torch.Tensor, nl: torch.Tensor, cond: Optional[torch.Tensor], out: torch.Tensor,
                       use_graph: bool = True, ss_rows: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Forward pass on caller-owned STATIC buffers (same addresses every call): the ~125 launches are
        captured once into a CUDA graph and replayed, which removes the per-launch host cost from the
        99-evaluations-per-field sampling loop.  `nl` is a device tensor whose VALUE may change between calls.
        ss_rows: fp32 [n_aff][128] from `embedding_table` (one noise level for the whole batch): copied into the plan's
        static (scale | shift) buffer, and the embedding MLP is left out of the launch sequence (`nl` is then unused)."""
        # the training entry points leave `_fmt = 0` (bf16 operands) on the engine: inference always runs its own format,
        # whatever ran before on this engine (sampling with `ema: False` after a training step used to fall back to the
        # unfused bf16 plan)
        self._fmt = self.infer_fmt
        self.pack()
        ext = (ss_rows is not None and getattr(self, "supports_ss_rows", False) and self.fused and self._fmt == 1
               and self.precision != "fp32" and x.shape[-1] == 128)
        self._ss_external = ext
        if ext:
            B = x.shape[0]
            ws = self._fws(B, x.shape[2], x.shape[3], x.device)
            ss = self._fbuf(ws, "ss_buf", (self.n_aff * B * 128,), torch.float32, x.device)
            ss[: self.n_aff * 128].view(self.n_aff, 128).copy_(ss_rows)
        try:
            return self._forward_static(x, nl, cond, out, use_graph, ext)
        finally:
            self._ss_external = False

    def _forward_static(self, x, nl, cond, out, use_graph, ext):
        if not use_graph:
            return self._launch_all(x, nl, cond, out)
        key = (x.data_ptr(), nl.data_ptr(), 0 if cond is None else cond.data_ptr(), out.data_ptr(), tuple(x.shape),
               self._packed_key, self.fused, self.precision, ext)
        entry = self._graphs.get(key)
        if entry is None:
            if len(self._graphs) > 8:
                self._graphs.clear()
            # eager warm-up: allocates workspaces, sets function attributes, creates the watchdog word
            self._launch_all(x, nl, cond, out)
            torch.cuda.current_stream().synchronize()
            n0 = L.LAUNCHES[0]
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._launch_all(x, nl, cond, out)
            entry = (g, L.LAUNCHES[0] - n0)
            self._graphs[key] = entry
        entry[0].replay()
        L.LAUNCHES[0] += entry[1]
        return out

    # ------------------------------------------------------------------ per-kernel timing (bench roofline)
    @torch.no_grad()
    def profile_kernels(self, x, noise_labels, cond, repeats: int = 3):
        """CUDA-event time of every C-ABI launch of one forward pass (current plan), on the launching stream.
        Returns a list of dicts {name, ms, flops, bytes} in launch order; ms = mean over `repeats`.  flops / bytes are
        the ALGORITHMIC figures of the launch (what DESIGN.md section 4 states per kernel), derived from its arguments."""
        x, nl, cond = self._check_inputs(x, noise_labels, cond)
        self._fmt = self.infer_fmt
        self.pack()
        out = torch.empty(x.shape[0], self.unet.out_channels, x.shape[2], x.shape[3], device=x.device)
        self._launch_all(x, nl, cond, out)
        real = self.lib
        runs = []

        def v(a):
            return a.value if hasattr(a, "value") else a

        def work(name, a):
            """(flops, bytes) of a launch from its C-ABI arguments (positions per include/mcedm_b200.h)."""
            if name == "mcedm_conv_rows_fused":
                n_halo, n_ctr, B, H, N, n_total, res_mode = v(a[2]), v(a[4]), v(a[7]), v(a[8]), v(a[9]), v(a[11]), v(a[15])
                px = B * H * 128
                out_b = 2 if v(a[13]) else 4
                return (2.0 * px * N * 64 * (9 * n_halo + n_ctr),
                        px * 64 * 2.0 * (n_halo + n_ctr) + px * N * out_b + (px * N * 2.0 * (1 if res_mode == 1 else 0.25)
                                                                             if res_mode else 0.0))
            if name == "mcedm_conv_head_fused":
                B, H, c_out = v(a[4]), v(a[5]), v(a[6])
                px = B * H * 128
                return 2.0 * px * 16 * 64 * 9, px * 64 * 2.0 + px * c_out * 4.0
            if name == "mcedm_conv_in_tc16":
                cin, B, H = v(a[1]) + v(a[3]), v(a[6]), v(a[7])
                px = B * H * 128
                return 2.0 * px * 64 * 9 * cin, px * (cin * 4.0 + 64 * 2.0)
            if name == "mcedm_conv_flat_fused":
                B, H, W, res_mode = v(a[4]), v(a[5]), v(a[6]), v(a[11])
                px = B * H * W
                return 2.0 * px * 64 * 576, px * 64 * 2.0 * (2 + {0: 0, 1: 1, 2: 0.25, 3: 4}[res_mode])
            if name == "mcedm_conv_rows":
                n_halo, n_ctr, B, H, N, res_mode = v(a[1]), v(a[3]), v(a[6]), v(a[7]), v(a[8]), v(a[12])
                px = B * H * 128
                return (2.0 * px * N * 64 * (9 * n_halo + n_ctr),
                        px * 64 * 2.0 * (n_halo + n_ctr) + px * N * 4.0 * (1 + (1 if res_mode == 1 else 0.25 if res_mode else 0)))
            if name == "mcedm_conv_flat":
                B, H, W, res_mode = v(a[3]), v(a[4]), v(a[5]), v(a[9])
                px = B * H * W
                return 2.0 * px * 64 * 576, px * 64 * (2.0 + 4.0 * (1 + {0: 0, 1: 1, 2: 0.25, 3: 4}[res_mode]))
            if name in ("mcedm_conv_igemm", "mcedm_conv_igemm16"):
                n_src, n_seg, B, H, W, N = v(a[1]), v(a[5]), v(a[8]), v(a[9]), v(a[10]), v(a[11])
                px = B * H * W
                return 2.0 * px * N * 64 * n_seg, px * 64 * 2.0 * n_src + px * N * 2.0
            if name == "mcedm_attention":
                B, Lq = v(a[1]), v(a[2])
                return 4.0 * B * Lq * Lq * 64, B * Lq * (192 + 64) * 2.0
            if name == "mcedm_gn_apply16":
                rs, B, H, W = v(a[5]), v(a[6]), v(a[7]), v(a[8])
                n_in = B * H * W * 64
                return 0.0, 2.0 * n_in + 2.0 * (n_in * 4 if rs == 1 else n_in // 4 if rs == 2 else n_in)
            if name == "mcedm_gn_apply":
                rs, B, H, W = v(a[9]), v(a[10]), v(a[11]), v(a[12])
                n_in = B * H * W * 64
                return 0.0, 4.0 * n_in + 2.0 * (n_in * 4 if rs == 1 else n_in // 4 if rs == 2 else n_in)
            if name in ("mcedm_conv_in", "mcedm_conv_in16"):
                cin, B, H, W = v(a[1]) + v(a[3]), v(a[6]), v(a[7]), v(a[8])
                px = B * H * W
                return 2.0 * px * 64 * 9 * cin, px * (cin * 4.0 + 64 * (2.0 if name.endswith("16") else 4.0))
            return 0.0, 0.0

        class _Proxy:
            def __init__(self, rec):
                self.rec = rec

            def __getattr__(self, name):
                fn = getattr(real, name)
                if not name.startswith("mcedm_") or name in ("mcedm_flat_geometry", "mcedm_last_error"):
                    return fn

                def call(*a):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    rc = fn(*a)
                    e1.record()
                    fl, by = work(name, a)
                    self.rec.append(dict(name=name[6:], flops=fl, bytes=by, ev=(e0, e1)))
                    return rc
                return call

        try:
            for _ in range(repeats):
                rec = []
                self.lib = _Proxy(rec)
                self._launch_all(x, nl, cond, out)
                torch.cuda.synchronize()
                runs.append(rec)
        finally:
            self.lib = real
        res = []
        for i, r in enumerate(runs[0]):
            ms = sum(rr[i]["ev"][0].elapsed_time(rr[i]["ev"][1]) for rr in runs) / len(runs)
            res.append(dict(name=r["name"], flops=r["flops"], bytes=r["bytes"], ms=ms))
        return res

    # (legacy per-conv timing of the unfused plan)
    @torch.no_grad()
    def profile_convs(self, x, noise_labels, cond, repeats: int = 3, with_gn: bool = False):
        """CUDA-event time of every 3x3-conv launch (and, with_gn, every GroupNorm pass) of one forward pass, on the
        launching stream.  Returns a list of dicts (kind 'conv': N, n_seg, pixels, H, flops, ms; kind 'gn': bytes, ms),
        ms = mean over `repeats`."""
        x, nl, cond = self._check_inputs(x, noise_labels, cond)
        self._fmt = self.infer_fmt
        self.pack()
        out = torch.empty(x.shape[0], self.unet.out_channels, x.shape[2], x.shape[3], device=x.device)
        self._launch_all(x, nl, cond, out)
        rec_all = []
        orig, orig_gn = self._conv3x3, self._gn_apply

        for _ in range(repeats):
            rec = []

            def timed(halo, ctr, w, bias, B, H, W, N, o, res, res_mode, stats, st, flat=None):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n_seg = 9 * len(halo) + len(ctr)
                e0.record()
                parts = orig(halo, ctr, w, bias, B, H, W, N, o, res, res_mode, stats, st, flat=flat)
                e1.record()
                rec.append(dict(kind="conv", N=N, n_seg=n_seg, pixels=B * H * W, H=H, res_mode=res_mode,
                                flops=2.0 * B * H * W * N * 64 * n_seg, ev=(e0, e1)))
                return parts

            def timed_gn(x_, stats, parts, gamma, beta, ss, ss_stride, act, resample, B, Hin, Win, out_, raw, st,
                         eps=1e-5, flat=None, meanrstd=None):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                orig_gn(x_, stats, parts, gamma, beta, ss, ss_stride, act, resample, B, Hin, Win, out_, raw, st, eps,
                        flat=flat, meanrstd=meanrstd)
                e1.record()
                n_in = B * Hin * Win * 64
                n_out = n_in * 4 if resample == 1 else n_in // 4 if resample == 2 else n_in
                rec.append(dict(kind="gn", H=Hin, resample=resample,
                                bytes=4.0 * n_in + 2.0 * n_out + (2.0 * n_in if raw is not None else 0.0), ev=(e0, e1)))

            self._conv3x3 = timed
            if with_gn:
                self._gn_apply = timed_gn
            try:
                self._launch_all(x, nl, cond, out)
            finally:
                del self._conv3x3
                if with_gn:
                    del self._gn_apply
            torch.cuda.synchronize()
            rec_all.append(rec)
        res = []
        for i, r in enumerate(rec_all[0]):
            ms = sum(rr[i]["ev"][0].elapsed_time(rr[i]["ev"][1]) for rr in rec_all) / len(rec_all)
            d = {k: v for k, v in r.items() if k != "ev"}
            d["ms"] = ms
            res.append(d)
        return res
