"""Inference launch plan with GroupNorm fused into the convolutions and 16-bit activations in HBM.

Same network as `UNetEngine._launch_all` (DhariwalUNet.forward, models/adm_blocks.py:364-404; UNetBlock.forward
:159-181), different data flow.  The unfused plan moves 28 B per activation element per block through HBM
(GroupNorm-apply passes read fp32 / write the 16-bit operand, convs read it back and write fp32); every kernel of it
measured at 65-80 % of the HBM roofline, so the only way to go faster was to move fewer bytes:

  * every activation of the trunk lives in HBM ONCE, as a raw 16-bit tensor (fp16 by default) plus the GroupNorm
    partial sums its producer's epilogue emitted;
  * `mcedm_gn_coef` (one tiny launch per GroupNorm) folds the partial sums into per-(sample, channel) coefficients;
  * the consuming conv applies silu(a*x + b) to its input rows in shared memory (transform warps of
    `mcedm_conv_rows_fused` / `mcedm_conv_flat_fused`), so the normalised operand never reaches HBM;
  * residuals and the raw inputs of the 1x1 skip projections are those same 16-bit tensors (no extra "raw" copies);
  * levels with W <= 64 keep every activation in the padded-flat layout of conv_flat.cu end to end;
  * a stand-alone apply pass (`mcedm_gn_apply16`) remains only where the operand must be materialised: in front of
    the four resampling conv0s and in front of the qkv projections (4 blocks at 32x32).

Per block this is ~10 B per activation element instead of 28.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import torch

from . import _lib as L


class Act:
    """A raw 16-bit activation: tensor, GroupNorm partial sums, records per image, geometry."""
    __slots__ = ("t", "st", "parts", "H", "W", "flat", "__weakref__")

    def __init__(self, t, st, parts, H, W, flat):
        self.t, self.st, self.parts, self.H, self.W, self.flat = t, st, parts, H, W, flat


class FusedMixin:
    # ------------------------------------------------------------------ buffers
    def _fws(self, B, H, W, dev, tag="fused") -> dict:
        key = (tag, B, H, W, dev.index, self._fmt)
        ws = self._ws.get(key)
        if ws is None:
            ws = self._ws[key] = {"geom": {}, "pool": {}, "dev": dev}
        return ws

    def _fgeom(self, ws, H, W):
        g = ws["geom"].get((H, W))
        if g is None:
            g = ws["geom"][(H, W)] = self._flat_geom(H, W) if W <= 64 else None
        return g

    def _dt16(self):
        return torch.float16 if self._fmt else torch.bfloat16

    def _fact(self, ws, name, B, H, W, dev, stats=True) -> Act:
        a = ws.get(name)
        if a is None:
            flat = self._fgeom(ws, H, W)
            if flat is None:
                t = torch.empty(B, H, W, 64, device=dev, dtype=self._dt16())
                n_rec = B * 4 * H                                    # conv_rows: 4 records per image row
            else:
                t = torch.zeros(B * flat[1], 64, device=dev, dtype=self._dt16())   # padding zeroed once, never written
                n_rec = B * (flat[1] // 128) * 4                     # conv_flat: 4 records per 128-position tile
            st = torch.empty(max(n_rec, B * (H * W // 128)), 16, 2, device=dev, dtype=torch.float32) if stats else None
            a = ws[name] = Act(t, st, 0, H, W, flat)
        return a

    def _fbuf(self, ws, name, shape, dtype, dev, zero=False):
        t = ws.get(name)
        if t is None:
            t = ws[name] = (torch.zeros if zero else torch.empty)(*shape, device=dev, dtype=dtype)
        return t

    # ------------------------------------------------------------------ launches
    def _fcoef(self, ws, name, act: Act, gamma, beta, ss, ss_stride, eps, B, st, save_mr=False):
        """Per-(sample, channel) coefficients of one GroupNorm; save_mr (training forward): also the (mean, rstd) per
        group that the backward needs -> returns (coef, meanrstd)."""
        coef = self._fbuf(ws, "coef." + name, (B, 128), torch.float32, act.t.device)
        mr = self._fbuf(ws, "mr." + name, (B, 16, 2), torch.float32, act.t.device) if save_mr else None
        L.check(self.lib.mcedm_gn_coef(L.ptr(act.st), act.parts, L.ptr(gamma), L.ptr(beta), L.ptr(ss), ss_stride, 64, eps,
                                       B, act.H, act.W, L.ptr(coef), L.ptr(mr), st), "gn_coef")
        return (coef, mr) if save_mr else coef

    def _fapply16(self, x: Act, coef, act_fn, resample, B, out: Act, st, dense_out=None, pooled: Optional[Act] = None):
        ip, ib = x.flat if x.flat is not None else (0, 0)
        if dense_out is not None:
            op, ob, o = 0, 0, dense_out
        else:
            op, ob = out.flat if out.flat is not None else (0, 0)
            o = out.t
        L.check(self.lib.mcedm_gn_apply16(L.ptr(x.t), ip, ib, L.ptr(coef), act_fn, resample, B, x.H, x.W, op, ob, L.ptr(o),
                                          L.ptr(pooled.t) if pooled is not None else None, self._fmt, st), "gn_apply16")

    def _fconv(self, srcs: List[Act], coefs, w, bias, B, out: Act, res, res_mode, st, ctr: Optional[List[Act]] = None,
                stats=True, ws=None, name=""):
        """3x3 conv of the (transformed) sources -> raw 16-bit `out` (+ statistics).  `coefs` None = the sources are
        already-normalised operands.  res: Act (16-bit) or None; res_mode as in the C ABI."""
        H, W = out.H, out.W
        rp, rb = (res.flat if (res is not None and res.flat is not None) else (0, 0))
        if out.flat is None:
            # ---------------- W == 128: row-resident kernel
            cptr = None if coefs is None else (C.c_void_p * len(coefs))(*[c.data_ptr() for c in coefs])
            hal = L.ptr_array([s.t for s in srcs])
            if len(srcs) == 2:
                # 128-channel conv0 (K = 1152: 144 KB of weights do not fit next to the row ring): K-split over the two
                # sources.  Pass 1 leaves its partial sum in `out` (16-bit), pass 2 adds it as an in-place residual.
                # (Two N = 32 output-channel passes with both sources resident were measured 40 % slower: the ring
                # shrinks to 4 two-source slots and every row is transformed twice.)
                assert not ctr and res is None
                for i in (0, 1):
                    L.check(self.lib.mcedm_conv_rows_fused(
                        L.ptr_array([srcs[i].t]), (C.c_void_p * 1)(coefs[i].data_ptr()), 1, None, 0, L.ptr(w[9 * i:9 * i + 9]),
                        L.ptr(bias) if i else None, B, H, 64, 0, 64, L.ptr(out.t), 1, L.ptr(out.t) if i else None, i, 0, 0,
                        L.ptr(out.st) if (stats and i) else None, self._fmt, st), "conv_rows_fused")
            else:
                cs = L.ptr_array([c.t for c in ctr]) if ctr else None
                L.check(self.lib.mcedm_conv_rows_fused(hal, cptr, 1, cs, len(ctr) if ctr else 0, L.ptr(w), L.ptr(bias), B, H,
                                                       64, 0, 64, L.ptr(out.t), 1, L.ptr(res.t) if res is not None else None,
                                                       res_mode, rp, rb, L.ptr(out.st) if stats else None, self._fmt, st),
                        "conv_rows_fused")
            out.parts = H        # one record per (4-row block, TMEM lane quarter): H / 4 * 4 per image
            return
        # ---------------- W <= 64: padded-flat kernel
        pitch, blk = out.flat
        lib = self.lib
        if len(srcs) == 2:
            # 128-channel conv0: K-split as above (16-bit partial in `out`, added in place by pass 2)
            assert not ctr and res is None
            for i in (0, 1):
                L.check(lib.mcedm_conv_flat_fused(L.ptr(srcs[i].t), L.ptr(coefs[i]), L.ptr(w[9 * i:9 * i + 9]),
                                                  L.ptr(bias) if i else None, B, H, W, 64, L.ptr(out.t), 0,
                                                  L.ptr(out.t) if i else None, i, 0, 0, 0,
                                                  L.ptr(out.st) if (stats and i) else None, self._fmt, st), "conv_flat_fused")
        else:
            res_t = res.t if res is not None else None
            if ctr:
                # 1x1 skip projection of the raw 128-channel input as a plain GEMM over the flat position sequence
                # (padding positions give 0 and are never read back), then consumed as conv1's residual
                assert res is None
                skip = self._fbuf(ws, f"skip.{H}", (B * blk, 64), self._dt16(), out.t.device)
                n = len(ctr)
                L.check(lib.mcedm_conv_igemm16(L.ptr_array([c.t for c in ctr]), n, L.int_array(list(range(n))),
                                               L.int_array([0] * n), L.int_array([0] * n), n, L.ptr(w[9:]), None, 1,
                                               B * blk // 128, 128, 64, L.ptr(skip), None, 0, 0, 0, None, self._fmt, st),
                        "conv_igemm16")
                res_t, res_mode, rp, rb = skip, 1, 0, 0
                w = w[:9]
            L.check(lib.mcedm_conv_flat_fused(L.ptr(srcs[0].t), L.ptr(coefs[0]) if coefs is not None else None, L.ptr(w),
                                              L.ptr(bias), B, H, W, 64, L.ptr(out.t), 0, L.ptr(res_t), res_mode, 0, rp, rb,
                                              L.ptr(out.st) if stats else None, self._fmt, st), "conv_flat_fused")
        out.parts = 4 * (blk // 128)

    # ------------------------------------------------------------------ one UNetBlock
    def _run_block_fused(self, blk, inputs: List[Act], B, ws, emb_stride, st, dev, tape=None) -> Act:
        """tape (training forward, train16_engine.py): a list receiving one record per block; every tensor the backward
        reads (conv0 output, qkv, attention output, log-sum-exp, coefficients, mean / rstd) then gets a per-block buffer
        instead of the per-level ones inference reuses."""
        x = inputs[0]
        train = tape is not None
        uq = (lambda s_: f"{s_}@{blk.name}") if train else (lambda s_: s_)
        if blk.up:
            H, W, rs, res_mode = x.H * 2, x.W * 2, 1, 2
        elif blk.down:
            H, W, rs, res_mode = x.H // 2, x.W // 2, 2, 3
        else:
            H, W, rs, res_mode = x.H, x.W, 0, 1
        eps = blk.mod.norm0.eps
        n = blk.name
        x_res = x                                                     # residual source of conv1 (identity skip)
        coef0 = [self._fcoef(ws, f"{n}.0.{i}", a, blk.g0[64 * i:64 * (i + 1)], blk.be0[64 * i:64 * (i + 1)], None, 0, eps,
                            B, st, save_mr=train) for i, a in enumerate(inputs)]
        mr0 = None
        if train:
            mr0 = [c[1] for c in coef0]
            coef0 = [c[0] for c in coef0]
        h = self._fact(ws, uq(f"h.{H}"), B, H, W, dev)
        if rs:
            # resampling conv0 (adm_blocks.py:73-77): materialise silu(norm0(x)) at the new resolution, conv it as is
            op = self._fact(ws, f"op.{H}", B, H, W, dev, stats=False)
            pooled = None
            if rs == 2 and not blk.skip_conv:
                # the skip path of a down block is the 2x2 mean of the raw input: emitted by the same pass (one more
                # 16-bit store per output pixel) and read by conv1 as a same-resolution residual; gathering the four
                # source pixels in conv1's epilogue instead cost 240 us per launch at 64x64 (B = 128).  (The same trick
                # for the nearest-x2 skip of the up blocks — the kernel can emit that copy too — measured neutral:
                # the gather reads an L2-resident quarter-size tensor, the copy costs a full-size store.)
                pooled = self._fact(ws, f"pool.{H}", B, H, W, dev, stats=False)
                x_res, res_mode = pooled, 1
            self._fapply16(x, coef0[0], 1, rs, B, op, st, pooled=pooled)
            self._fconv([op], None, blk.w0, blk.b0, B, h, None, 0, st, ws=ws)
        else:
            self._fconv(inputs, coef0, blk.w0, blk.b0, B, h, None, 0, st, ws=ws)
        ss = ws["ss"][blk.aff_index * self._ss_rows * 128:]
        coef1 = self._fcoef(ws, f"{n}.1", h, blk.g1, blk.be1, ss, emb_stride, eps, B, st, save_mr=train)
        mr1 = None
        if train:
            coef1, mr1 = coef1
        out = self._fact(ws, n, B, H, W, dev)
        rec = dict(blk=blk, inputs=list(inputs), coef0=coef0, mr0=mr0, h=h, coef1=coef1, mr1=mr1, out=out, final=out,
                   H=H, W=W, rs=rs) if train else None
        src1, coefs1 = [h], [coef1]
        drop = self._drop if train else None
        if drop is not None:
            # dropout (adm_blocks.py:167, training forward only): conv1's operand is materialised with the mask applied
            # and kept for the backward (the weight gradient contracts it, the data gradient takes the same mask)
            op1 = self._fact(ws, uq(f"op1.{H}"), B, H, W, dev, stats=False)
            thr, scale, rng = drop
            ip, ib = h.flat if h.flat is not None else (0, 0)
            L.check(self.lib.mcedm_gn_apply16_dropout(L.ptr(h.t), ip, ib, L.ptr(coef1), B, H, W, ip, ib, L.ptr(op1.t), thr,
                                                      scale, blk.aff_index, L.ptr(rng), self._fmt, st), "gn_apply16_dropout")
            src1, coefs1 = [op1], None
            rec["op1"] = op1
        if blk.skip_conv:
            self._fconv(src1, coefs1, blk.w1, blk.b1, B, out, None, 0, st, ctr=inputs, ws=ws)
        else:
            self._fconv(src1, coefs1, blk.w1, blk.b1, B, out, x_res, res_mode, st, ws=ws)
        if blk.attn:
            coef2 = self._fcoef(ws, f"{n}.2", out, blk.g2, blk.be2, None, 0, eps, B, st, save_mr=train)
            mr2 = None
            if train:
                coef2, mr2 = coef2
            a2 = self._fbuf(ws, "att.in", (B, H, W, 64), self._dt16(), dev)
            self._fapply16(out, coef2, 0, 0, B, None, st, dense_out=a2)
            qkv = self._fbuf(ws, uq("att.qkv"), (B, H * W, 192), self._dt16(), dev)
            att = self._fbuf(ws, uq("att.out"), (B, H * W, 64), self._dt16(), dev)
            lse = self._fbuf(ws, uq("att.lse"), (B, H * W), torch.float32, dev) if train else None
            self._conv([a2], [(0, 0, 0)], blk.wqkv, blk.bqkv, B, H, W, 192, qkv, 1, None, 0, None, st)
            L.check(self.lib.mcedm_attention(L.ptr(qkv), B, H * W, L.ptr(att), L.ptr(lse), self._fmt, st), "attention")
            if not train:
                L.LAUNCHES[0] += 1               # single-pass kernel + the flagged-tile two-pass launch
            out2 = self._fact(ws, n + ".attn", B, H, W, dev)
            pitch, fblk = out2.flat if out2.flat is not None else (0, 0)
            L.check(self.lib.mcedm_conv_igemm16(L.ptr_array([att]), 1, L.int_array([0]), L.int_array([0]), L.int_array([0]), 1,
                                                L.ptr(blk.wproj), L.ptr(blk.bproj), B, H, W, 64, L.ptr(out2.t), L.ptr(out.t),
                                                1, pitch, fblk, L.ptr(out2.st), self._fmt, st), "conv_igemm16")
            out2.parts = H * W // 128
            if train:
                rec.update(coef2=coef2, mr2=mr2, qkv=qkv, att=att, lse=lse, final=out2)
            out = out2
        if train:
            tape.append(rec)
        return out

    # ------------------------------------------------------------------ whole network
    def _launch_all_fused(self, x, nl, cond, out):
        u = self.unet
        B, _, H, W = x.shape
        if W != 128:
            raise ValueError("the fused inference plan is laid out for 128-pixel-wide fields")
        dev = x.device
        ws = self._fws(B, H, W, dev)
        st = L.stream_ptr()
        lib = self.lib
        Bemb = nl.numel()
        self._ss_rows = Bemb
        emb_stride = 128 if Bemb == B and B > 1 else 0
        ss = ws["ss"] = self._fbuf(ws, "ss_buf", (self.n_aff * B * 128,), torch.float32, dev)
        if getattr(self, "_ss_external", False):
            # the caller placed this evaluation's (scale | shift) rows in `ss` (UNetEngine.embedding_table): one noise
            # level for the whole batch, laid out as [n_aff][1][128]
            Bemb, emb_stride = 1, 0
            self._ss_rows = 1
        else:
            self._launch_emb(nl, Bemb, ss, st)
        self._launch_rest_fused(x, cond, out, ws, B, H, dev, emb_stride, st)
        return out

    def _launch_emb(self, nl, Bemb, ss, st):
        lib = self.lib
        L.check(lib.mcedm_emb_mlp(L.ptr(nl), L.ptr(self.freqs), L.ptr(self.w_m0), L.ptr(self.b_m0), L.ptr(self.w_m1),
                                  L.ptr(self.b_m1), L.ptr(self.aff_w), L.ptr(self.aff_b), self.n_aff, Bemb, None,
                                  L.ptr(ss), st), "emb_mlp")

    def _launch_rest_fused(self, x, cond, out, ws, B, H, dev, emb_stride, st, tape=None):
        u = self.unet
        train = tape is not None
        blocks_tape = [] if train else None
        lib = self.lib
        W = 128
        t0 = self._fact(ws, "conv_in", B, H, W, dev)
        if self.w_in_tc is not None:
            # first conv on the tensor cores: horizontal taps folded into K by builder warps, vertical taps stacked into N
            L.check(lib.mcedm_conv_in_tc16(L.ptr(x), u.x_channels, L.ptr(cond), u.cat_channels, L.ptr(self.w_in_tc),
                                           L.ptr(self.b_in), B, H, L.ptr(t0.t), L.ptr(t0.st), self._fmt, st), "conv_in_tc16")
            t0.parts = 4 * H
        else:
            L.check(lib.mcedm_conv_in16(L.ptr(x), u.x_channels, L.ptr(cond), u.cat_channels, L.ptr(self.w_in),
                                        L.ptr(self.b_in), B, H, W, L.ptr(t0.t), L.ptr(t0.st), self._fmt, st), "conv_in16")
            t0.parts = H * W // 128
        cur = t0
        skips = [cur]
        for blk in self.blocks_enc:
            cur = self._run_block_fused(blk, [cur], B, ws, emb_stride, st, dev, tape=blocks_tape)
            skips.append(cur)
        for blk in self.blocks_dec:
            inputs = [cur]
            if blk.n_src == 2:
                inputs.append(skips.pop())
            cur = self._run_block_fused(blk, inputs, B, ws, emb_stride, st, dev, tape=blocks_tape)
        # out_conv(silu(out_norm(x)))  (adm_blocks.py:403): the normalisation rides in the conv like everywhere else
        coef = self._fcoef(ws, "out", cur, self.g_out, self.be_out, None, 0, u.out_norm.eps, B, st, save_mr=train)
        if train:
            coef, mr_out = coef
            tape.update(blocks=blocks_tape, t0=t0, last=cur, coef_out=coef, mr_out=mr_out)
        L.check(lib.mcedm_conv_head_fused(L.ptr(cur.t), L.ptr(coef), L.ptr(self.w_out), L.ptr(self.b_out), B, H,
                                          u.out_channels, L.ptr(out), self._fmt, st), "conv_head_fused")
        return out
