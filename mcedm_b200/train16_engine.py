"""Training plan "fused16" of the B200-native ADM U-Net (mixin of `engine.UNetEngine`): 16-bit activations end to end.

The fp32-stream plan (train_engine.py) moves 28 B per activation element per block through HBM in the forward and 44 B
in the GroupNorm backward passes; its bf16 operands put the training-mode forward AT the 1e-2 bar.  This plan reuses the
inference data flow (fused_engine.py) for the forward and mirrors it in the backward:

  forward   = the fused inference launch sequence in fp16 (11 significand bits: the denoiser error of the training
              forward drops from 1e-2 to the 1.4e-3 class of inference).  Every activation exists ONCE in HBM as a raw
              fp16 tensor + the GroupNorm partial sums of its producer; the normalised operands never reach HBM.  What the
              backward needs is kept per block: the raw activations (they ARE the GroupNorm inputs), the per-(sample,
              channel) coefficients, (mean, rstd), qkv / attention output / log-sum-exp.
  backward  = fp16 as well, LOSS-SCALED: dL/dF enters as S * dL/dF (S = 1024; with EDM preconditioning
              dL/dF = (2/B) m (F - F_target), O(1/B) for every noise level, so a static scale is enough; conversions
              saturate instead of overflowing) and the flat gradient buffer is multiplied by 1/S at the end.
              With a LossScaler on the engine (loss_scale.py) S is read from device memory and the gradient stores
              do not saturate (op_fmt MCEDM_FMT_F16_INF): an overflow reaches the flat gradient as inf / NaN and
              the optimizer step skips.
              * data gradients of the 3x3 convs = the fused forward kernels on 16-bit gradients (no transform),
                writing 16-bit;
              * GroupNorm(+SiLU, scale/shift, resample) backward = mcedm_gn_bwd16: raw fp16 x, 16-bit dy, 16-bit
                residual-path gradients (GRAD_MASTER_FP32 keeps an fp32 master copy of the residual-stream gradient:
                measured no accuracy difference, 8 more bytes per element);
              * weight gradients need the normalised operand: formed from the raw activation inside the weight-gradient
                kernel (mcedm_conv_wgrad16_fused: the warps that otherwise only run its epilogue transform each row in
                shared memory), so it is neither stored by the forward nor recomputed through HBM; only the resampled
                operands of the four up / down blocks are materialised by an mcedm_gn_apply16 pass;
              * 1x1 convolutions on the narrow levels run on the padded-flat position sequence as is.
  Per block: forward 10 B, backward ~40 B per activation element (fp32-stream plan: 28 + ~75).

Reference: autograd of DhariwalUNet.forward / UNetBlock.forward (models/adm_blocks.py:364-404, :159-181) inside
PlMcedm.training_step (models/mcedm.py:254-281).
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib as L
from .fused_engine import Act


class Train16Mixin:
    LOSS_SCALE = 1024.0
    # True: the gradient of the residual stream keeps an fp32 master copy next to its 16-bit operand copy (8 more bytes
    # per element in every norm0 backward); False: fp16 only (one 2^-12 rounding per residual hop)
    GRAD_MASTER_FP32 = False
    # weight-gradient launches on a side stream / parallel graph branch (backward16); MCEDM_WGRAD_SIDE=0 disables
    WGRAD_SIDE_STREAM = True

    # ------------------------------------------------------------------ dropout state
    def dropout_p(self) -> float:
        return float(getattr(self.unet, "dropout", 0.0) or 0.0)

    def dropout_args(self):
        """(threshold, scale) of the dropout kernels: keep iff mask word >= threshold = min(2^32 - 1, floor(p 2^32)),
        both computed in double; scale = 1 / (1 - p) rounded to fp32."""
        p = self.dropout_p()
        return min(2 ** 32 - 1, math.floor(p * 2.0 ** 32)), float(np.float32(1.0 / (1.0 - p)))

    def dropout_rng(self, dev) -> torch.Tensor:
        """The device words {seed_lo, seed_hi, step} the kernels read (one buffer per engine: graphs capture its address)."""
        buf = getattr(self, "_rng_words", None)
        if buf is None or buf.device != dev:
            buf = self._rng_words = torch.zeros(3, dtype=torch.int32, device=dev)
        return buf

    def dropout_fill(self, dev):
        """Writes {seed, step} to the device words: three stream-ordered fills, no host synchronisation."""
        if self.dropout_seed is None:
            self.dropout_seed = torch.initial_seed()          # reads the seed, draws nothing
        s = int(self.dropout_seed) & (2 ** 64 - 1)
        buf = self.dropout_rng(dev)
        for i, v in enumerate((s & 0xFFFFFFFF, s >> 32, int(self.dropout_step) & 0xFFFFFFFF)):
            buf[i].fill_(v - 2 ** 32 if v >= 2 ** 31 else v)

    # ------------------------------------------------------------------ forward
    def forward_train16(self, x: torch.Tensor, nl: torch.Tensor, cond: Optional[torch.Tensor]) -> torch.Tensor:
        u = self.unet
        B, _, H, W = x.shape
        self.pack_train()
        self._grad_layout()
        dev = x.device
        st = L.stream_ptr()
        ws = self._fws(B, H, W, dev, tag="train16")
        self._drop = None
        if self.dropout_p() > 0:
            # eager: this forward's {seed, step} go to the device words now; under graph capture the kernels only
            # capture the words' address and TrainStepGraph.load writes them before every replay
            if not torch.cuda.is_current_stream_capturing():
                self.dropout_fill(dev)
                self.dropout_step += 1
            self._drop = self.dropout_args() + (self.dropout_rng(dev),)
        self._ss_external = False
        self._ss_rows = B
        ss = ws["ss"] = self._fbuf(ws, "ss_buf", (self.n_aff * B * 128,), torch.float32, dev)
        nl_saved = self._fbuf(ws, "nl", (B,), torch.float32, dev)
        nl_saved.copy_(nl)
        self._launch_emb(nl_saved, B, ss, st)
        # [cond, x] as a 64-channel 16-bit NHWC tensor: operand of the first conv's weight gradient
        xin_pad = self._fbuf(ws, "xin_pad", (B, H, W, 64), self._dt16(), dev, zero=True)
        L.check(self.lib.mcedm_nchw_to_nhwc_pad16(L.ptr(cond), u.cat_channels if cond is not None else 0, L.ptr(x),
                                                  u.x_channels, B, H, W, L.ptr(xin_pad), 0, 1.0, self._fmt, st),
                "nchw_to_nhwc_pad16")
        out = torch.empty(B, u.out_channels, H, W, device=dev, dtype=torch.float32)
        tape: dict = {}
        self._launch_rest_fused(x, cond, out, ws, B, H, dev, 128, st, tape=tape)
        tape.update(plan="fused16", ws=ws, B=B, H=H, W=W, drop=self._drop)
        self._tape = tape
        return out

    # ------------------------------------------------------------------ backward helpers
    def _lay(self, ws, H, W):
        g = self._fgeom(ws, H, W)
        return g if g is not None else (0, 0)

    def _buf16(self, ws, name, B, H, W, dev, dtype=None):
        """A 16-bit (or fp32) tensor in the layout of level H x W; padded-flat buffers are zeroed once and only ever
        written at data positions."""
        flat = self._fgeom(ws, H, W)
        dtype = dtype or self._dt16()
        if flat is None:
            return self._fbuf(ws, name, (B, H, W, 64), dtype, dev)
        return self._fbuf(ws, name, (B * flat[1], 64), dtype, dev, zero=True)

    def _gset16(self, ws, B, H, W, parity, need_dense, dev):
        key = ("g16", H, W, parity)
        gs = ws.get(key)
        if gs is None:
            f32 = self._buf16(ws, ("g16.f32", H, W, parity), B, H, W, dev, torch.float32) if self.GRAD_MASTER_FP32 \
                else None
            gs = ws[key] = dict(f32=f32, bf=self._buf16(ws, ("g16.h", H, W, parity), B, H, W, dev), dense=None,
                                n_cta=self.lib.mcedm_gn_bwd16_ctas_per_img(H, W, B), H=H, W=W, cs=None)
        if need_dense and gs["dense"] is None:
            gs["dense"] = self._fbuf(ws, ("g16.dense", H, W, parity), (B, H, W, 64), self._dt16(), dev)
        return gs

    def _dgrad16(self, ws, src, wd, B, H, W, out, st):
        """Data gradient of a 3x3 conv: the fused forward kernel on the 16-bit gradient (no transform, no bias)."""
        import ctypes as C
        flat = self._fgeom(ws, H, W)
        if flat is None:
            L.check(self.lib.mcedm_conv_rows_fused(L.ptr_array([src]), None, 1, None, 0, L.ptr(wd), None, B, H, 64, 0, 64,
                                                   L.ptr(out), 1, None, 0, 0, 0, None, self._gfmt, st), "conv_rows_fused")
        else:
            L.check(self.lib.mcedm_conv_flat_fused(L.ptr(src), None, L.ptr(wd), None, B, H, W, 64, L.ptr(out), 0, None, 0,
                                                   0, 0, 0, None, self._gfmt, st), "conv_flat_fused")

    def _gn_bwd16(self, ws, dy, dy_lay, x: Act, mr, coef, gamma, beta, ss, act, rs, B, dgamma, dbeta, dss, add0, add0_mode,
                  add0_lay, add1, pend, gs, want_dense, st):
        """One GroupNorm(+SiLU, +scale/shift, +resample) backward on raw 16-bit x / 16-bit dy.  `gs` (a _gset16 dict)
        receives dx, or `pend` (a bare tensor in x's layout: fp32 with the master copy, else 16-bit)."""
        lib = self.lib
        Hin, Win = x.H, x.W
        n_cta = lib.mcedm_gn_bwd16_ctas_per_img(Hin, Win, B)
        red = self._t(ws, ("gnred", B * n_cta), (B, n_cta, 64, 2), torch.float32)
        kcoef = self._t(ws, "gnkcoef", (B, 192), torch.float32)
        ticket = self._t(ws, "gnticket", (3 * B,), torch.int32, zero=True)
        jid = self._job_id()
        dgb = self._t(ws, ("gndgb", jid), (B, 64, 2), torch.float32)
        out_f32 = dx16 = dense = cs = None
        if gs is not None:
            gs["cs"] = self._t(ws, ("cs", jid), (B * n_cta, 64), torch.float32)
            out_f32, dx16, cs = gs["f32"], gs["bf"], gs["cs"]
            dense = gs["dense"] if want_dense else None
        elif self.GRAD_MASTER_FP32:
            out_f32 = pend
        else:
            dx16 = pend
        xl = x.flat if x.flat is not None else (0, 0)
        L.check(lib.mcedm_gn_bwd16(L.ptr(dy), dy_lay[0], dy_lay[1], L.ptr(x.t), xl[0], xl[1], self._gfmt, L.ptr(mr),
                                   L.ptr(coef), L.ptr(gamma), L.ptr(beta), L.ptr(ss), 128, 64, act, rs, B, Hin, Win, L.ptr(red),
                                   L.ptr(kcoef), L.ptr(ticket), L.ptr(dgb), L.ptr(dss), 128, L.ptr(add0), add0_mode,
                                   add0_lay[0], add0_lay[1], L.ptr(add1), 0 if self.GRAD_MASTER_FP32 else 1,
                                   L.ptr(out_f32), L.ptr(dx16), L.ptr(dense), L.ptr(cs), st), "gn_bwd16")
        L.LAUNCHES[0] += 1
        flat_dgb = dgb.view(-1)
        self._reduce_rows(flat_dgb, B, 128, 64, 2, dgamma, st)
        self._reduce_rows(flat_dgb[1:], B, 128, 64, 2, dbeta, st)

    def _igemm1x1(self, srcs, w, B, H, W, N, out, out16, st):
        self._conv(srcs, [(i, 0, 0) for i in range(len(srcs))], w, None, B, H, W, N, out, out16, None, 0, None, st,
                   fmt=self._gfmt if out16 else None)

    # ------------------------------------------------------------------ backward
    @torch.no_grad()
    def backward16(self, dF: torch.Tensor) -> torch.Tensor:
        T = self._tape
        u, lib = self.unet, self.lib
        B, H, W, ws, tape = T["B"], T["H"], T["W"], T["ws"], T["blocks"]
        self._fmt = self.train_fmt
        dev = ws["dev"]
        st = L.stream_ptr()
        G = self.grad_of
        fmt = self._fmt
        scaler = self.loss_scaler.state(dev) if self.loss_scaler is not None else None
        # format of the 16-bit gradient stores: fp16 without saturation under dynamic loss scaling
        self._gfmt = L.FMT_F16_INF if scaler is not None else fmt
        S = float(self.LOSS_SCALE)
        dF = dF.contiguous()
        self._jid, self._rjobs, self._wjobs, self._job_refs, self._post_copies = 0, [], [], [], []

        # Weight gradients leave the critical path: the data-gradient chain (dgrad conv -> GroupNorm backward -> next
        # block) never reads them, so the 3x3 / skip weight-gradient launches go to a SIDE stream (a parallel branch of
        # the captured graph).  Both branches are grids of persistent one-CTA-per-SM kernels, so nothing runs truly
        # side by side, but a branch's CTAs start on an SM the moment the other branch's CTA leaves it: launch gaps,
        # prologues and tails of the short launches at B = 32 (20 - 50 us each) are filled with the other branch's work.
        # Hazards: a weight-gradient launch only READS (a 16-bit gradient of this block, saved activations) and writes
        # its own partial buffer; the gradient buffers are rewritten by later blocks, hence join() at every block start
        # (joining later, just before the first rewrite, measured slower: 5.63 vs 5.48 ms - the lagging branch then
        # competes with the critical data-gradient chain instead of filling its gaps).
        main = torch.cuda.current_stream(dev)
        side_on = self.WGRAD_SIDE_STREAM and os.environ.get("MCEDM_WGRAD_SIDE", "1") != "0"
        if side_on:
            s2 = getattr(self, "_side_stream", None)
            if s2 is None or s2.device != dev:
                s2 = self._side_stream = torch.cuda.Stream(dev)
            st2 = s2.cuda_stream

        def wgrad_side(*a, **k):
            """_wgrad(..., st) on the side stream, ordered after everything enqueued on the main stream so far"""
            if not side_on:
                return self._wgrad(*a, **k)
            s2.wait_stream(main)
            return self._wgrad(*a[:-1], st2, **k)

        def join():
            if side_on:
                main.wait_stream(s2)

        consumers: Dict[int, list] = {}
        for rec in tape:
            for i, a in enumerate(rec["inputs"]):
                consumers.setdefault(id(a), []).append((rec["blk"].name, i))
        attn_out = {id(rec["final"]) for rec in tape if rec["blk"].attn}

        def need_dense(a: Act):
            return id(a) in attn_out and a.flat is not None

        def recompute(x: Act, coef, act_fn, rs, Ho, Wo):
            """silu(norm(x)) (resampled) as a materialised operand at Ho x Wo: what the weight-gradient GEMM contracts."""
            op = Act(self._buf16(ws, ("op16", Ho, Wo), B, Ho, Wo, dev), None, 0, Ho, Wo, self._fgeom(ws, Ho, Wo))
            self._fapply16(x, coef, act_fn, rs, B, op, st)
            return op

        master = self.GRAD_MASTER_FP32
        gdt, o16 = (torch.float32, 0) if master else (self._dt16(), 1)     # residual-path gradient tensors
        dss = self._t(ws, "dss", (self.n_aff, B, 128), torch.float32)
        ss_all = ws["ss"].view(self.n_aff, B, 128)
        parity = 0
        csn = 64

        # ---- head: out_conv(silu(out_norm(x)))
        dFp = self._fbuf(ws, "dFp", (B, H, W, 64), self._dt16(), dev, zero=True)
        if scaler is None:
            L.check(lib.mcedm_nchw_to_nhwc_pad16(L.ptr(dF), u.out_channels, None, 0, B, H, W, L.ptr(dFp), 0, S, fmt, st),
                    "pad dF")
        else:
            L.check(lib.mcedm_nchw_to_nhwc_pad16_scaled(L.ptr(dF), u.out_channels, None, 0, B, H, W, L.ptr(dFp), 0,
                                                        L.ptr(scaler.scale_t), self._gfmt, st), "pad dF")
        last: Act = T["last"]
        wgrad_side(ws, dFp, False, 64, 0, last.t, False, B, H, W, 9, G(u.out_conv.weight), 64, 0, st,
                   co_count=u.out_channels, a_coef=T["coef_out"])
        cs_tmp = self._t(ws, ("cs_tmp", self._job_id()), (csn, 64), torch.float32)
        L.check(lib.mcedm_colsum16(L.ptr(dFp), B * H * W, 64, 0, L.ptr(cs_tmp), csn, fmt, st), "colsum")
        self._reduce_rows(cs_tmp, csn, 64, u.out_channels, 1, G(u.out_conv.bias), st)
        d_a = self._buf16(ws, ("d16", H, W), B, H, W, dev)
        self._dgrad16(ws, dFp, self.wd_out, B, H, W, d_a, st)
        gs = self._gset16(ws, B, H, W, parity, need_dense(last), dev)
        self._gn_bwd16(ws, d_a, self._lay(ws, H, W), last, T["mr_out"], T["coef_out"], self.g_out, self.be_out, None, 1, 0, B,
                       G(u.out_norm.weight), G(u.out_norm.bias), None, None, 0, (0, 0), None, None, gs,
                       need_dense(last), st)
        grads = {id(last): gs}
        pending: Dict[int, torch.Tensor] = {}

        # ---- blocks, last to first
        for rec in reversed(tape):
            blk, m = rec["blk"], rec["blk"].mod
            Hb, Wb, rs = rec["H"], rec["W"], rec["rs"]
            lay = self._lay(ws, Hb, Wb)
            is_flat = lay[0] > 0
            gs = grads.pop(id(rec["final"]))
            out: Act = rec["out"]
            join()
            if blk.attn:
                # out2 = proj(att) + bproj + out
                Lq = Hb * Wb
                gd = gs["dense"] if is_flat else gs["bf"]
                self._bias_grad(gs, B, G(m.proj.bias), st)
                att, qkv = rec["att"], rec["qkv"]
                self._wgrad(ws, gd, False, 64, 0, att, False, B, Hb, Wb, 1, G(m.proj.weight), 64, 0, st)
                d_att = self._fbuf(ws, "d_att", (B * Lq, 64), self._dt16(), dev)
                self._igemm1x1([gd], blk.wdproj, B, Hb, Wb, 64, d_att, 1, st)
                dq, dk, dv = (self._fbuf(ws, n_, (B * Lq, 64), self._dt16(), dev) for n_ in ("dq", "dk", "dv"))
                dvec = self._fbuf(ws, "dvec", (B, Lq), torch.float32, dev)
                L.check(lib.mcedm_attention_bwd16(L.ptr(qkv), L.ptr(att), L.ptr(d_att), L.ptr(rec["lse"]), B, Lq,
                                                  L.ptr(dvec), L.ptr(dq), L.ptr(dk), L.ptr(dv), self._gfmt, st),
                        "attention_bwd")
                L.LAUNCHES[0] += 2
                qb = self._t(ws, ("qkv_bias_tmp", blk.name), (3, 64), torch.float32)
                for j, dj in enumerate((dq, dk, dv)):
                    self._wgrad(ws, dj, False, 64, 0, out.t, is_flat, B, Hb, Wb, 1, G(m.qkv.weight), 64, 0, st, co_mul=3,
                                co_add=j, a_coef=rec["coef2"], a_act=0)
                    cs_tmp = self._t(ws, ("cs_tmp", self._job_id()), (csn, 64), torch.float32)
                    L.check(lib.mcedm_colsum16(L.ptr(dj), B * Lq, 64, 0, L.ptr(cs_tmp), csn, fmt, st), "colsum")
                    self._reduce_rows(cs_tmp, csn, 64, 64, 1, qb[j], st)
                self._post_copies.append((G(m.qkv.bias).view(64, 3), qb))    # channel order (c*3 + {q,k,v})
                d_a2 = self._fbuf(ws, "d_a2", (B, Hb, Wb, 64), self._dt16(), dev)
                self._igemm1x1([dq, dk, dv], blk.wdqkv, B, Hb, Wb, 64, d_a2, 1, st)
                parity ^= 1
                gs_out = self._gset16(ws, B, Hb, Wb, parity, False, dev)
                self._gn_bwd16(ws, d_a2, (0, 0), out, rec["mr2"], rec["coef2"], blk.g2, blk.be2, None, 0, 0, B, G(m.norm2.weight),
                               G(m.norm2.bias), None, gs["f32"] if master else gs["bf"], 0, lay, None, None, gs_out,
                               False, st)
                gs = gs_out
            # out = conv1(a1) + b1 + skip(x)
            self._bias_grad(gs, B, G(m.conv1.bias), st)
            h: Act = rec["h"]
            op1: Optional[Act] = rec.get("op1")
            if op1 is None:
                wgrad_side(ws, gs["bf"], is_flat, 64, 0, h.t, is_flat, B, Hb, Wb, 9, G(m.conv1.weight), 64, 0, st,
                           a_coef=rec["coef1"])
            else:      # dropout: conv1 contracted the materialised, masked operand the forward kept
                wgrad_side(ws, gs["bf"], is_flat, 64, 0, op1.t, is_flat, B, Hb, Wb, 9, G(m.conv1.weight), 64, 0, st)
            if blk.skip_conv:
                self._bias_grad(gs, B, G(m.skip.bias), st)
                for i, xi in enumerate(rec["inputs"]):
                    wgrad_side(ws, gs["bf"], is_flat, 64, 0, xi.t, is_flat, B, Hb, Wb, 1, G(m.skip.weight),
                               64 * blk.n_src, 64 * i, st)
            d_a1 = self._buf16(ws, ("d16", Hb, Wb), B, Hb, Wb, dev)
            self._dgrad16(ws, gs["bf"], blk.wd1, B, Hb, Wb, d_a1, st)
            if op1 is not None:
                thr, scale, rng = T["drop"]
                L.check(lib.mcedm_dropout_bwd16(L.ptr(d_a1), lay[0], lay[1], B, Hb, Wb, thr, scale, blk.aff_index,
                                                L.ptr(rng), self._gfmt, st), "dropout_bwd16")
            d_hb = self._buf16(ws, ("d_h16", Hb, Wb), B, Hb, Wb, dev)
            hset = dict(f32=None, bf=d_hb, dense=None, cs=None, n_cta=lib.mcedm_gn_bwd16_ctas_per_img(Hb, Wb, B))
            self._gn_bwd16(ws, d_a1, lay, h, rec["mr1"], rec["coef1"], blk.g1, blk.be1, ss_all[blk.aff_index], 1, 0, B,
                           G(m.norm1.weight), G(m.norm1.bias), dss[blk.aff_index], None, 0, (0, 0), None, None, hset,
                           False, st)
            self._bias_grad(hset, B, G(m.conv0.bias), st)
            parity ^= 1
            for i in reversed(range(blk.n_src)):
                xi: Act = rec["inputs"][i]
                if rs:     # resampled operand: materialised (the in-kernel transform works on same-resolution rows)
                    a_i = recompute(xi, rec["coef0"][i], 1, rs, Hb, Wb)
                    self._wgrad(ws, d_hb, is_flat, 64, 0, a_i.t, is_flat, B, Hb, Wb, 9, G(m.conv0.weight),
                                64 * blk.n_src, 64 * i, st)
                else:
                    wgrad_side(ws, d_hb, is_flat, 64, 0, xi.t, is_flat, B, Hb, Wb, 9, G(m.conv0.weight),
                               64 * blk.n_src, 64 * i, st, a_coef=rec["coef0"][i])
                d_ai = self._buf16(ws, ("d16", Hb, Wb), B, Hb, Wb, dev)
                self._dgrad16(ws, d_hb, blk.wd0[i], B, Hb, Wb, d_ai, st)
                if blk.skip_conv:
                    # 1x1 data gradient on the level's position sequence as it is stored (padding positions produce
                    # values nobody reads)
                    add0 = self._buf16(ws, ("d_s", Hb, Wb), B, Hb, Wb, dev, gdt)
                    if is_flat:
                        self._igemm1x1([gs["bf"]], blk.wdskip[i], 1, B * lay[1] // 128, 128, 64, add0, o16, st)
                    else:
                        self._igemm1x1([gs["bf"]], blk.wdskip[i], B, Hb, Wb, 64, add0, o16, st)
                    add0_mode = 0
                else:
                    add0, add0_mode = gs["f32"] if master else gs["bf"], (1 if blk.up else 2 if blk.down else 0)
                g0, be0 = blk.g0[64 * i:64 * (i + 1)], blk.be0[64 * i:64 * (i + 1)]
                dg0 = G(m.norm0.weight)[64 * i:64 * (i + 1)]
                db0 = G(m.norm0.bias)[64 * i:64 * (i + 1)]
                first_consumer = consumers[id(xi)][0] == (blk.name, i)
                if not first_consumer:
                    # a later consumer (decoder skip connection): keep the partial gradient until the first one runs
                    pend = self._buf16(ws, ("pending", id(xi)), B, xi.H, xi.W, dev, gdt)
                    self._gn_bwd16(ws, d_ai, lay, xi, rec["mr0"][i], rec["coef0"][i], g0, be0, None, 1, rs, B, dg0, db0, None, add0,
                                   add0_mode, lay, None, pend, None, False, st)
                    pending[id(xi)] = pend
                else:
                    nd = need_dense(xi)
                    gnext = self._gset16(ws, B, xi.H, xi.W, parity, nd, dev)
                    self._gn_bwd16(ws, d_ai, lay, xi, rec["mr0"][i], rec["coef0"][i], g0, be0, None, 1, rs, B, dg0, db0, None, add0,
                                   add0_mode, lay, pending.pop(id(xi), None), None, gnext, nd, st)
                    grads[id(xi)] = gnext

        # ---- first conv (weights only; the network input carries no gradient)
        gs = grads.pop(id(T["t0"]))
        cin = u.enc[self.conv_in_name]
        self._bias_grad(gs, B, G(cin.bias), st)
        join()
        wgrad_side(ws, gs["bf"], False, 64, 0, ws["xin_pad"], False, B, H, W, 9, G(cin.weight), cin.weight.shape[1], 0,
                   st, ci_count=cin.weight.shape[1])

        # ---- embedding MLP and the per-block affine projections
        vec = self._t(ws, "embvec", (B, 320), torch.float32)
        d_aff_w = self._t(ws, "d_aff_w", (self.n_aff, 128, 64), torch.float32)
        d_aff_b = self._t(ws, "d_aff_b", (self.n_aff, 128), torch.float32)
        L.check(lib.mcedm_emb_mlp_bwd(L.ptr(ws["nl"]), L.ptr(self.freqs), L.ptr(self.w_m0), L.ptr(self.b_m0),
                                      L.ptr(self.w_m1), L.ptr(self.b_m1), L.ptr(self.aff_w), L.ptr(dss), self.n_aff, B,
                                      L.ptr(vec), L.ptr(d_aff_w), L.ptr(d_aff_b), L.ptr(G(u.map_layer1.weight)),
                                      L.ptr(G(u.map_layer1.bias)), L.ptr(G(u.map_layer0.weight)),
                                      L.ptr(G(u.map_layer0.bias)), st), "emb_mlp_bwd")
        blocks = self.blocks_enc + self.blocks_dec
        torch._foreach_copy_([G(b.mod.affine.weight) for b in blocks], list(d_aff_w.unbind(0)))
        torch._foreach_copy_([G(b.mod.affine.bias) for b in blocks], list(d_aff_b.unbind(0)))
        assert not grads and not pending, (list(grads), list(pending))
        join()
        self._flush_deferred(ws, st)
        for dst, src in self._post_copies:
            dst.copy_(src.t())
        if scaler is None:
            self._gflat.mul_(1.0 / S)             # loss scale off (a power of two: exact)
        else:
            L.check(lib.mcedm_grad_unscale(L.ptr(self._gflat), self._gflat.numel(), L.ptr(scaler.scale_t), st),
                    "grad_unscale")
        return self._gflat
