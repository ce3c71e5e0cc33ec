"""Training forward / backward launch plan of the B200-native ADM U-Net (mixin of `engine.UNetEngine`).

Backward of DhariwalUNet.forward / UNetBlock.forward (models/adm_blocks.py:364-404, :159-181) as autograd would
differentiate it inside PlMcedm.training_step (models/mcedm.py:254-281), built only from C-ABI launches:

  * data gradient of a 3x3 / 1x1 convolution  = the FORWARD implicit-GEMM kernels run on the bf16 output
    gradient with flipped + transposed packed weights (conv_rows / conv_flat / conv_igemm);
  * weight gradient                            = conv_wgrad (pixel-contraction GEMM on tcgen05) + ordered reduce;
  * GroupNorm + (1+scale)/shift + SiLU + resample backward = gn_bwd, which also folds in the residual-path
    gradients, emits the bf16 copy the previous convolution's gradient kernels consume and the per-CTA column
    sums that are that convolution's bias gradient;
  * attention backward                         = attn_bwd (recomputes P / dS tiles on the tensor cores);
  * embedding MLP backward                     = emb_mlp_bwd.

Activations saved by the training forward: every GroupNorm input (fp32; these are the residual-stream tensors and
conv0 outputs the forward writes anyway), its (mean, rstd), and every bf16 tensor-core operand.  Gradients are
written (never accumulated across calls) into one flat fp32 buffer whose slices are returned as the parameters'
`.grad`, so the data-parallel all-reduce and the fused Adam step work on a single contiguous tensor.  Gradient
accumulation (`accumulate_grads`) leaves the backward as it is and folds that buffer into a second one per call.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import _lib as L


DGRAD_DTYPE = [None]       # pack_plan.PackPlan probes the layouts with fp32 "index" weights (override of `dtype`)


def pack_dgrad3x3(weight: torch.Tensor, dtype=torch.bfloat16) -> torch.Tensor:
    """[Cout, 64, 3, 3] (one 64-channel input slice) -> 16-bit [9][ci][co(_pad 64)]: taps flipped, channels swapped."""
    cout = weight.shape[0]
    w = weight.detach().flip(2, 3).permute(2, 3, 1, 0).reshape(9, 64, cout)
    if cout < 64:
        w = torch.cat([w, w.new_zeros(9, 64, 64 - cout)], dim=2)
    return w.to(DGRAD_DTYPE[0] or dtype).contiguous()


def pack_dgrad1x1(weight2d: torch.Tensor, dtype=torch.bfloat16) -> torch.Tensor:
    """[co, ci] -> 16-bit [1][ci][co]"""
    return weight2d.detach().t().reshape(1, weight2d.shape[1], weight2d.shape[0]).to(DGRAD_DTYPE[0] or dtype).contiguous()


def _flat_views(flat, params) -> dict:
    views, off = {}, 0
    for p in params:
        views[id(p)] = flat[off:off + p.numel()].view(p.shape)
        off += p.numel()
    return views


class TrainMixin:
    # ------------------------------------------------------------------ gradient storage
    # Every backward writes its micro-batch gradient into `_gflat` (`_step_grad` views).  With `accumulate_grads = N`
    # (gradient accumulation over windows of N micro-batches) one fold launch after each backward adds _gflat / N into
    # `_gacc`, a second buffer of the same layout, and `.grad` / `grad_of` / `flat_grad` hand out `_gacc` instead.
    def _grad_layout(self):
        params = list(self.unet.parameters())
        key = tuple((id(p), p.numel()) for p in params)
        if getattr(self, "_glayout_key", None) != key or self._gflat.device != params[0].device:
            n = sum(p.numel() for p in params)
            self._gflat = torch.zeros(n, device=params[0].device, dtype=torch.float32)
            self._gview = _flat_views(self._gflat, params)
            self._gacc = None
            self._glayout_key = key
        if self.accumulate_grads and self._gacc is None:
            self._gacc = torch.zeros_like(self._gflat)
            self._aview = _flat_views(self._gacc, params)
        return self._gflat

    def _step_grad(self, p) -> torch.Tensor:
        """The slice of the micro-batch gradient buffer the backward writes p's gradient to."""
        return self._gview[id(p)]

    def grad_of(self, p) -> torch.Tensor:
        """p's gradient as `.grad` aliases it: the last backward's, or the accumulation window's."""
        return (self._aview if self.accumulate_grads else self._gview)[id(p)]

    def flat_grad(self) -> torch.Tensor:
        g = self._grad_layout()
        return self._gacc if self.accumulate_grads else g

    def fold_grads(self):
        """Accumulation mode: adds the micro-batch gradient / N into the window buffer (one launch), overwriting it on
        a window's first backward (the parameters' `.grad` is None after zero_grad(set_to_none=True)), and binds every
        parameter's `.grad` to its window slice.  The 1/N is applied here, never to dL/dF: the fp16 backward keeps the
        range of a plain step, which its loss scale is sized for."""
        params = [p for p in self.unet.parameters() if p.requires_grad]
        first = params[0].grad is None
        self._grad_layout()
        L.check(self.lib.mcedm_grad_accumulate(L.ptr(self._gacc), L.ptr(self._gflat), self._gflat.numel(),
                                               1.0 / self.accumulate_grads, int(first), L.stream_ptr()),
                "grad_accumulate")
        for p in params:
            p.grad = self._aview[id(p)]

    # ------------------------------------------------------------------ packed weights of the data-gradient convs
    def pack_train(self, force: bool = False):
        # operand format of the training plan: fp16 for the fused 16-bit plan (loss-scaled gradients), bf16 for the
        # fp32-stream plan
        self._fmt = self.train_fmt
        self.pack()
        if not force and getattr(self, "_packed_train_key", None) == self._packed_key:
            return
        dt = torch.float16 if self._fmt else torch.bfloat16
        with torch.no_grad():
            for b in self.blocks_enc + self.blocks_dec:
                m = b.mod
                b.wd0 = [pack_dgrad3x3(m.conv0.weight[:, 64 * i:64 * (i + 1)], dt) for i in range(b.n_src)]
                b.wd1 = pack_dgrad3x3(m.conv1.weight, dt)
                if b.skip_conv:
                    b.wdskip = [pack_dgrad1x1(m.skip.weight[:, 64 * i:64 * (i + 1), 0, 0], dt) for i in range(b.n_src)]
                if b.attn:
                    perm = torch.arange(192, device=m.qkv.weight.device).reshape(64, 3).t().reshape(-1)
                    wq = m.qkv.weight.detach()[perm][:, :, 0, 0]                      # [(q|k|v) x 64, ci]
                    b.wdqkv = torch.cat([pack_dgrad1x1(wq[64 * j:64 * (j + 1)], dt) for j in range(3)], 0).contiguous()
                    b.wdproj = pack_dgrad1x1(m.proj.weight[:, :, 0, 0], dt)
            self.wd_out = pack_dgrad3x3(self.unet.out_conv.weight, dt)
        self._packed_train_key = self._packed_key

    # ------------------------------------------------------------------ training workspace
    def _train_ws(self, B, H, W, dev) -> dict:
        key = ("train", B, H, W, dev.index)
        tw = self._ws.get(key)
        if tw is None:
            tw = {"pool": {}, "B": B, "H": H, "W": W, "dev": dev}
            self._ws[key] = tw
        return tw

    @staticmethod
    def _t(tw, name, shape, dtype, zero=False):
        t = tw["pool"].get(name)
        if t is None:
            t = (torch.zeros if zero else torch.empty)(shape, device=tw["dev"], dtype=dtype)
            tw["pool"][name] = t
        return t

    def _act(self, tw, name, B, H, W):
        """(fp32 NHWC tensor, GroupNorm partial records) of a named residual-stream activation."""
        return (self._t(tw, ("act", name), (B, H, W, 64), torch.float32),
                self._t(tw, ("act_st", name), (B * (H * W // 128 + H // 4 + 8) * 4, 16, 2), torch.float32))

    def _operand(self, tw, name, B, H, W):
        """bf16 tensor-core operand buffer in the layout of its level: dense for W == 128, padded-flat below."""
        if W <= 64 and self.use_flat:
            pitch, blk = self._flat_geom(H, W)
            return self._t(tw, ("op", name), (B * blk, 64), torch.bfloat16, zero=True), (pitch, blk)
        return self._t(tw, ("op", name), (B, H, W, 64), torch.bfloat16), None

    # ------------------------------------------------------------------ training forward
    def _block_fwd_train(self, blk, inputs, B, H_in, W_in, tw, ss_all, st):
        """inputs: list of (name, fp32 tensor, stats, parts). Mirrors UNetEngine._run_block with per-block buffers."""
        if blk.up:
            H, W, rs, res_mode = H_in * 2, W_in * 2, 1, 2
        elif blk.down:
            H, W, rs, res_mode = H_in // 2, W_in // 2, 2, 3
        else:
            H, W, rs, res_mode = H_in, W_in, 0, 1
        eps = blk.mod.norm0.eps
        rec = dict(blk=blk, inputs=[i[0] for i in inputs], H_in=H_in, W_in=W_in, H=H, W=W, rs=rs)
        a_srcs, raw_srcs, flat = [], [], None
        for i, (name, x, x_st, x_parts) in enumerate(inputs):
            a, flat = self._operand(tw, (blk.name, "a", i), B, H, W)
            raw = self._t(tw, (blk.name, "raw", i), (B, H, W, 64), torch.bfloat16) if blk.skip_conv else None
            mr = self._t(tw, (blk.name, "mr0", i), (B, 16, 2), torch.float32)
            self._gn_apply(x, x_st, x_parts, blk.g0[64 * i:64 * (i + 1)], blk.be0[64 * i:64 * (i + 1)], None, 0, 1, rs,
                           B, H_in, W_in, a, raw, st, eps, flat=flat, meanrstd=mr)
            a_srcs.append(a)
            if raw is not None:
                raw_srcs.append(raw)
        h = self._t(tw, (blk.name, "h"), (B, H, W, 64), torch.float32)
        h_st = self._t(tw, (blk.name, "h_st"), (B * (H * W // 128 + H // 4 + 8) * 4, 16, 2), torch.float32)
        h_parts = self._conv3x3(a_srcs, [], blk.w0, blk.b0, B, H, W, 64, h, None, 0, h_st, st, flat=flat)
        ss = ss_all[blk.aff_index]
        a1, _ = self._operand(tw, (blk.name, "a1"), B, H, W)
        mr1 = self._t(tw, (blk.name, "mr1"), (B, 16, 2), torch.float32)
        self._gn_apply(h, h_st, h_parts, blk.g1, blk.be1, ss, 128, 1, 0, B, H, W, a1, None, st, eps, flat=flat,
                       meanrstd=mr1)
        out, out_st = self._act(tw, blk.name, B, H, W)
        if blk.skip_conv:
            parts = self._conv3x3([a1], raw_srcs, blk.w1, blk.b1, B, H, W, 64, out, None, 0, out_st, st, flat=flat)
        else:
            parts = self._conv3x3([a1], [], blk.w1, blk.b1, B, H, W, 64, out, inputs[0][1], res_mode, out_st, st,
                                  flat=flat)
        rec.update(flat=flat, out_name=blk.name, final_name=blk.name)
        final = (blk.name, out, out_st, parts)
        if blk.attn:
            a2 = self._t(tw, (blk.name, "a2"), (B, H, W, 64), torch.bfloat16)
            mr2 = self._t(tw, (blk.name, "mr2"), (B, 16, 2), torch.float32)
            qkv = self._t(tw, (blk.name, "qkv"), (B * H * W, 192), torch.bfloat16)
            att = self._t(tw, (blk.name, "att"), (B * H * W, 64), torch.bfloat16)
            lse = self._t(tw, (blk.name, "lse"), (B, H * W), torch.float32)
            self._gn_apply(out, out_st, parts, blk.g2, blk.be2, None, 0, 0, 0, B, H, W, a2, None, st, eps, meanrstd=mr2)
            self._conv([a2], [(0, 0, 0)], blk.wqkv, blk.bqkv, B, H, W, 192, qkv, 1, None, 0, None, st)
            L.check(self.lib.mcedm_attention(L.ptr(qkv), B, H * W, L.ptr(att), L.ptr(lse), 0, st), "attention")
            out2, out2_st = self._act(tw, blk.name + ".attn", B, H, W)
            self._conv([att], [(0, 0, 0)], blk.wproj, blk.bproj, B, H, W, 64, out2, 0, out, 1, out2_st, st)
            rec["final_name"] = blk.name + ".attn"
            final = (blk.name + ".attn", out2, out2_st, H * W // 128)
        return rec, final, H, W

    def forward_train(self, x: torch.Tensor, noise_labels: torch.Tensor, cond: Optional[torch.Tensor]) -> torch.Tensor:
        """Forward pass that keeps what `backward` needs. Returns F_x [B,out_ch,H,W] fp32 (a fresh tensor)."""
        x, nl, cond = self._check_inputs(x, noise_labels, cond)
        B, _, H, W = x.shape
        if nl.numel() == 1:
            nl = nl.expand(B).contiguous()
        if self.dropout_p() > 0 and (self.train_plan != "fused16" or W != 128):
            raise NotImplementedError("dropout > 0 has kernels in the fp16 training plan only (MCEDM_TRAIN_PLAN=fused16, "
                                      "128-pixel-wide fields)")
        if self.train_plan == "fused16" and W != 128:
            self.train_plan = "fp32"          # the 16-bit plan is laid out for 128-pixel-wide fields
        if self.train_plan == "fused16":
            return self.forward_train16(x, nl, cond)
        self._fmt = 0
        u = self.unet
        if (W >> 2) % 16 != 0:
            raise ValueError(f"training needs the coarsest level to be a multiple of 16 pixels wide (W={W})")
        self.pack_train()
        self._grad_layout()
        dev = x.device
        tw = self._train_ws(B, H, W, dev)
        st = L.stream_ptr()
        lib = self.lib
        ss_all = self._t(tw, "ss", (self.n_aff, B, 128), torch.float32)
        nl_saved = self._t(tw, "nl", (B,), torch.float32)
        nl_saved.copy_(nl)
        L.check(lib.mcedm_emb_mlp(L.ptr(nl_saved), L.ptr(self.freqs), L.ptr(self.w_m0), L.ptr(self.b_m0),
                                  L.ptr(self.w_m1), L.ptr(self.b_m1), L.ptr(self.aff_w), L.ptr(self.aff_b), self.n_aff,
                                  B, None, L.ptr(ss_all), st), "emb_mlp")
        xin_pad = self._t(tw, "xin_pad", (B, H, W, 64), torch.bfloat16, zero=True)
        L.check(lib.mcedm_nchw_to_nhwc_pad(L.ptr(cond), u.cat_channels if cond is not None else 0, L.ptr(x),
                                           u.x_channels, B, H, W, L.ptr(xin_pad), 0, st), "nchw_to_nhwc_pad")
        t0, t0_st = self._act(tw, "conv_in", B, H, W)
        L.check(lib.mcedm_conv_in(L.ptr(x), u.x_channels, L.ptr(cond), u.cat_channels, L.ptr(self.w_in),
                                  L.ptr(self.b_in), B, H, W, L.ptr(t0), L.ptr(t0_st), st), "conv_in")
        cur, ch, cw = ("conv_in", t0, t0_st, H * W // 128), H, W
        skips = [cur]
        tape: List[dict] = []
        for blk in self.blocks_enc:
            rec, cur, ch, cw = self._block_fwd_train(blk, [cur], B, ch, cw, tw, ss_all, st)
            tape.append(rec)
            skips.append(cur)
        for blk in self.blocks_dec:
            inputs = [cur]
            if blk.n_src == 2:
                inputs.append(skips.pop())
            rec, cur, ch, cw = self._block_fwd_train(blk, inputs, B, ch, cw, tw, ss_all, st)
            tape.append(rec)
        a_out, _ = self._operand(tw, "a_out", B, H, W) if W == 128 else \
            (self._t(tw, ("op", "a_out"), (B, H, W, 64), torch.bfloat16), None)
        mr_out = self._t(tw, "mr_out", (B, 16, 2), torch.float32)
        self._gn_apply(cur[1], cur[2], cur[3], self.g_out, self.be_out, None, 0, 1, 0, B, H, W, a_out, None, st,
                       u.out_norm.eps, meanrstd=mr_out)
        o16 = self._t(tw, "o16", (B, H, W, 16), torch.float32)
        # the head always reads the dense operand (conv_rows for W == 128, conv_igemm otherwise)
        self._conv3x3([a_out], [], self.w_out, self.b_out, B, H, W, 16, o16, None, 0, None, st)
        out = torch.empty(B, u.out_channels, H, W, device=dev, dtype=torch.float32)
        L.check(lib.mcedm_head_to_nchw(L.ptr(o16), 16, u.out_channels, B, H, W, L.ptr(out), st), "head_to_nchw")
        self._tape = dict(tape=tape, last=cur[0], B=B, H=H, W=W, tw=tw)
        return out

    # ------------------------------------------------------------------ backward helpers
    def _gset(self, tw, B, H, W, parity, need_dense):
        """Buffers receiving the gradient of one residual-stream activation at H x W."""
        key = ("g", H, W, parity)
        gs = tw["pool"].get(key)
        if gs is None:
            n_cta = self.lib.mcedm_gn_bwd_ctas_per_img(H, W, B)
            bf, flat = self._operand(tw, ("g", H, W, parity), B, H, W)
            gs = dict(f32=torch.empty(B, H, W, 64, device=tw["dev"], dtype=torch.float32), bf=bf, flat=flat,
                      dense=None, cs=torch.empty(B * n_cta, 64, device=tw["dev"], dtype=torch.float32), n_cta=n_cta,
                      H=H, W=W)
            tw["pool"][key] = gs
        if gs["flat"] is not None and need_dense and gs["dense"] is None:
            gs["dense"] = torch.empty(B, H, W, 64, device=tw["dev"], dtype=torch.bfloat16)
        return gs

    @staticmethod
    def _dense_of(gs):
        return gs["bf"] if gs["flat"] is None else gs["dense"]

    # ---- deferred folds: every bias / gamma / beta / weight-gradient fold only feeds the flat gradient buffer, so the
    # backward queues them (each with its own partial buffer) and runs them in two batched launches at its end
    # instead of ~95 latency-bound launches spread through it (mcedm_reduce_rows_batched / mcedm_wgrad_reduce_batched)
    def _job_id(self):
        self._jid += 1
        return self._jid

    def _reduce_rows(self, src, n_rows, stride_r, n_cols, stride_j, out, st, accumulate=0):
        assert accumulate == 0
        self._rjobs.append((src.data_ptr(), out.data_ptr(), int(stride_r), int(stride_j), int(n_rows), int(n_cols), 0,
                            1.0))
        self._job_refs += [src, out]

    def _flush_deferred(self, tw, st):
        import struct

        key = (tuple(self._rjobs), tuple(self._wjobs))
        cache = tw.setdefault("fold_tables", {})
        tab = cache.get(key)
        if tab is None:
            if torch.cuda.is_current_stream_capturing():
                raise L.McedmError("deferred-fold tables must be built by an eager backward before graph capture")
            if len(cache) > 4:
                cache.clear()
            rb = b"".join(struct.pack("<QQqqiiif", *j) for j in self._rjobs)
            wb = b"".join(struct.pack("<QQiiiiiiii", *j) for j in self._wjobs)
            dev = tw["dev"]
            tab = cache[key] = (torch.frombuffer(bytearray(rb), dtype=torch.uint8).to(dev),
                                torch.frombuffer(bytearray(wb), dtype=torch.uint8).to(dev),
                                max(j[5] for j in self._rjobs))
        rt, wt, max_cols = tab
        L.check(self.lib.mcedm_wgrad_reduce_batched(L.ptr(wt), len(self._wjobs), st), "wgrad_reduce_batched")
        L.check(self.lib.mcedm_reduce_rows_batched(L.ptr(rt), len(self._rjobs), max_cols, st), "reduce_rows_batched")

    def _bias_grad(self, gs, B, out, st):
        self._reduce_rows(gs["cs"], B * gs["n_cta"], 64, 64, 1, out, st)

    def _gn_bwd(self, tw, dy, x, mr, gamma, beta, ss, act, rs, B, Hin, Win, dgamma, dbeta, dss, add0, add0_mode, add1,
                out_f32, gs, want_dense, eps, st):
        """One GroupNorm(+SiLU, +scale/shift, +resample) backward. `gs` (a _gset dict) or `out_f32` receives dx."""
        lib = self.lib
        n_cta = lib.mcedm_gn_bwd_ctas_per_img(Hin, Win, B)
        red = self._t(tw, ("gnred", B * n_cta), (B, n_cta, 64, 2), torch.float32)
        coef = self._t(tw, "gncoef", (B, 64, 4), torch.float32)
        jid = self._job_id()
        dgb = self._t(tw, ("gndgb", jid), (B, 64, 2), torch.float32)   # per call: folded at the end of the backward
        bf = dense = cs = None
        pitch = blk = 0
        if gs is not None:
            gs["cs"] = self._t(tw, ("cs", jid), (B * gs["n_cta"], 64), torch.float32)
            out_f32, bf, cs = gs["f32"], gs["bf"], gs["cs"]
            if gs["flat"] is not None:
                pitch, blk = gs["flat"]
                dense = gs["dense"] if want_dense else None
        L.check(lib.mcedm_gn_bwd(L.ptr(dy), L.ptr(x), L.ptr(mr), L.ptr(gamma), L.ptr(beta), L.ptr(ss), 128, 64, eps, act,
                                 rs, B, Hin, Win, L.ptr(red), L.ptr(coef), L.ptr(dgb), L.ptr(dss), 128, L.ptr(add0),
                                 add0_mode, L.ptr(add1), L.ptr(out_f32), L.ptr(bf), pitch, blk, L.ptr(dense), L.ptr(cs),
                                 st), "gn_bwd")
        flat_dgb = dgb.view(-1)
        self._reduce_rows(flat_dgb, B, 128, 64, 2, dgamma, st)
        self._reduce_rows(flat_dgb[1:], B, 128, 64, 2, dbeta, st)

    def _dgrad3x3(self, src, flat, wd, B, H, W, out, st):
        self._conv3x3([src], [], wd, None, B, H, W, 64, out, None, 0, None, st, flat=flat)

    def _wgrad(self, tw, dy, dy_flat, dy_ctot, dy_coff, a, a_flat, B, H, W, taps, dw, cin_total, ci_off, st, co_mul=1,
               co_add=0, co_count=64, ci_count=64, a_coef=None, a_act=1):
        """a_coef (fp32 [B][128]): `a` is a raw activation, the kernel forms act(coef.a * a + coef.b) in shared memory."""
        lib = self.lib
        n = lib.mcedm_wgrad_ctas(B, H, W)
        partial = self._t(tw, ("wgpart", self._job_id()), (n * taps * 4096,), torch.float32)
        L.check(lib.mcedm_conv_wgrad16_fused(L.ptr(dy), 1 if dy_flat else 0, dy_ctot, dy_coff, L.ptr(a),
                                             1 if a_flat else 0, 64, 0, L.ptr(a_coef), a_act, B, H, W, taps,
                                             L.ptr(partial), self._fmt, st), "conv_wgrad")
        self._wjobs.append((partial.data_ptr(), dw.data_ptr(), n, taps, cin_total, ci_off, co_mul, co_add, co_count,
                            ci_count))
        self._job_refs += [partial, dw]

    # ------------------------------------------------------------------ backward
    @torch.no_grad()
    def backward(self, dF: torch.Tensor) -> torch.Tensor:
        """dF: dL/dF_x [B,out_ch,H,W] fp32. Writes every parameter gradient into the flat buffer and returns it."""
        T = self._tape
        if T is None:
            raise L.McedmError("backward() without a preceding forward_train()")
        if T.get("plan") == "fused16":
            return self.backward16(dF)
        self._fmt = 0
        u, lib = self.unet, self.lib
        B, H, W, tw, tape = T["B"], T["H"], T["W"], T["tw"], T["tape"]
        dev = tw["dev"]
        st = L.stream_ptr()
        G = self._step_grad
        dF = dF.contiguous()
        pool = tw["pool"]
        self._jid, self._rjobs, self._wjobs, self._job_refs, self._post_copies = 0, [], [], [], []

        # which (block, source) consumes each activation, in forward order
        consumers: Dict[str, list] = {}
        for rec in tape:
            for i, name in enumerate(rec["inputs"]):
                consumers.setdefault(name, []).append((rec["blk"].name, i))
        producer = {"conv_in": None}
        for rec in tape:
            producer[rec["out_name"]] = rec
            producer[rec["final_name"]] = rec

        def need_dense(name):
            rec = producer[name]
            return rec is not None and (rec["blk"].attn or rec["blk"].skip_conv)

        d_a = self._t(tw, "d_a", (B, H, W, 64), torch.float32)       # conv data gradients (largest level)
        d_s = self._t(tw, "d_s", (B, H, W, 64), torch.float32)       # skip-projection data gradients
        dss = self._t(tw, "dss", (self.n_aff, B, 128), torch.float32)
        parity = 0

        # ---- head: out_conv(silu(out_norm(x)))
        dFp = self._t(tw, "dFp", (B, H, W, 64), torch.bfloat16, zero=True)
        L.check(lib.mcedm_nchw_to_nhwc_pad(L.ptr(dF), u.out_channels, None, 0, B, H, W, L.ptr(dFp), 0, st), "pad dF")
        a_out = pool[("op", "a_out")]
        self._wgrad(tw, dFp, False, 64, 0, a_out, False, B, H, W, 9, G(u.out_conv.weight), 64, 0, st,
                    co_count=u.out_channels)
        csn = 64
        cs_tmp = self._t(tw, ("cs_tmp", self._job_id()), (csn, 64), torch.float32)
        L.check(lib.mcedm_colsum_bf16(L.ptr(dFp), B * H * W, 64, 0, L.ptr(cs_tmp), csn, st), "colsum")
        self._reduce_rows(cs_tmp, csn, 64, u.out_channels, 1, G(u.out_conv.bias), st)
        self._conv3x3([dFp], [], self.wd_out, None, B, H, W, 64, d_a, None, 0, None, st)
        last = T["last"]
        x_last = pool[("act", last)]
        gs = self._gset(tw, B, H, W, parity, need_dense(last))
        self._gn_bwd(tw, d_a, x_last, pool["mr_out"], self.g_out, self.be_out, None, 1, 0, B, H, W,
                     G(u.out_norm.weight), G(u.out_norm.bias), None, None, 0, None, None, gs, need_dense(last),
                     u.out_norm.eps, st)
        grads = {last: gs}
        pending: Dict[str, torch.Tensor] = {}

        # ---- blocks, last to first
        for rec in reversed(tape):
            blk, m = rec["blk"], rec["blk"].mod
            Hb, Wb, Hi, Wi, rs, flat = rec["H"], rec["W"], rec["H_in"], rec["W_in"], rec["rs"], rec["flat"]
            eps = m.norm0.eps
            gs = grads.pop(rec["final_name"])
            if blk.attn:
                # out2 = proj(att) + bproj + out
                Lq = Hb * Wb
                gd = self._dense_of(gs)
                self._bias_grad(gs, B, G(m.proj.bias), st)
                att, qkv = pool[(blk.name, "att")], pool[(blk.name, "qkv")]
                self._wgrad(tw, gd, False, 64, 0, att, False, B, Hb, Wb, 1, G(m.proj.weight), 64, 0, st)
                d_att = self._t(tw, "d_att", (B * Lq, 64), torch.bfloat16)
                self._conv([gd], [(0, 0, 0)], blk.wdproj, None, B, Hb, Wb, 64, d_att, 1, None, 0, None, st)
                dq, dk, dv = (self._t(tw, n, (B * Lq, 64), torch.bfloat16) for n in ("dq", "dk", "dv"))
                dvec = self._t(tw, "dvec", (B, Lq), torch.float32)
                L.check(lib.mcedm_attention_bwd(L.ptr(qkv), L.ptr(att), L.ptr(d_att), L.ptr(pool[(blk.name, "lse")]), B,
                                                Lq, L.ptr(dvec), L.ptr(dq), L.ptr(dk), L.ptr(dv), st), "attention_bwd")
                a2 = pool[(blk.name, "a2")]
                qb = self._t(tw, ("qkv_bias_tmp", blk.name), (3, 64), torch.float32)   # folded at the end of the backward
                for j, dj in enumerate((dq, dk, dv)):
                    self._wgrad(tw, dj, False, 64, 0, a2, False, B, Hb, Wb, 1, G(m.qkv.weight), 64, 0, st, co_mul=3,
                                co_add=j)
                    cs_tmp = self._t(tw, ("cs_tmp", self._job_id()), (csn, 64), torch.float32)
                    L.check(lib.mcedm_colsum_bf16(L.ptr(dj), B * Lq, 64, 0, L.ptr(cs_tmp), csn, st), "colsum")
                    self._reduce_rows(cs_tmp, csn, 64, 64, 1, qb[j], st)
                self._post_copies.append((G(m.qkv.bias).view(64, 3), qb))    # channel order (c*3 + {q,k,v})
                d_a2 = d_a.view(-1)[:B * Lq * 64].view(B, Hb, Wb, 64)
                self._conv([dq, dk, dv], [(0, 0, 0), (1, 0, 0), (2, 0, 0)], blk.wdqkv, None, B, Hb, Wb, 64, d_a2, 0, None,
                           0, None, st)
                parity ^= 1
                gs_out = self._gset(tw, B, Hb, Wb, parity, blk.skip_conv)
                self._gn_bwd(tw, d_a2, pool[("act", blk.name)], pool[(blk.name, "mr2")], blk.g2, blk.be2, None, 0, 0, B,
                             Hb, Wb, G(m.norm2.weight), G(m.norm2.bias), None, gs["f32"], 0, None, None, gs_out,
                             blk.skip_conv, eps, st)
                gs = gs_out
            # out = conv1(a1) + b1 + skip(x)
            self._bias_grad(gs, B, G(m.conv1.bias), st)
            a1 = pool[("op", (blk.name, "a1"))]
            self._wgrad(tw, gs["bf"], flat is not None, 64, 0, a1, flat is not None, B, Hb, Wb, 9, G(m.conv1.weight), 64,
                        0, st)
            if blk.skip_conv:
                self._bias_grad(gs, B, G(m.skip.bias), st)
                gd = self._dense_of(gs)
                for i in range(blk.n_src):
                    self._wgrad(tw, gd, False, 64, 0, pool[(blk.name, "raw", i)], False, B, Hb, Wb, 1, G(m.skip.weight),
                                64 * blk.n_src, 64 * i, st)
            d_a1 = d_a.view(-1)[:B * Hb * Wb * 64].view(B, Hb, Wb, 64)
            self._dgrad3x3(gs["bf"], flat, blk.wd1, B, Hb, Wb, d_a1, st)
            d_hb, _ = self._operand(tw, ("d_h", Hb, Wb), B, Hb, Wb)
            hcs_n = lib.mcedm_gn_bwd_ctas_per_img(Hb, Wb, B)
            hcs = self._t(tw, ("hcs", Hb, Wb), (B * hcs_n, 64), torch.float32)
            hset = dict(f32=None, bf=d_hb, flat=flat, dense=None, cs=hcs, n_cta=hcs_n)
            self._gn_bwd(tw, d_a1, pool[(blk.name, "h")], pool[(blk.name, "mr1")], blk.g1, blk.be1,
                         pool["ss"][blk.aff_index], 1, 0, B, Hb, Wb, G(m.norm1.weight), G(m.norm1.bias),
                         dss[blk.aff_index], None, 0, None, None, hset, False, eps, st)
            self._bias_grad(hset, B, G(m.conv0.bias), st)
            parity ^= 1
            for i in reversed(range(blk.n_src)):
                name = rec["inputs"][i]
                a_i = pool[("op", (blk.name, "a", i))]
                self._wgrad(tw, d_hb, flat is not None, 64, 0, a_i, flat is not None, B, Hb, Wb, 9, G(m.conv0.weight),
                            64 * blk.n_src, 64 * i, st)
                d_ai = d_a.view(-1)[:B * Hb * Wb * 64].view(B, Hb, Wb, 64)
                self._dgrad3x3(d_hb, flat, blk.wd0[i], B, Hb, Wb, d_ai, st)
                if blk.skip_conv:
                    add0 = d_s.view(-1)[:B * Hb * Wb * 64].view(B, Hb, Wb, 64)
                    self._conv([self._dense_of(gs)], [(0, 0, 0)], blk.wdskip[i], None, B, Hb, Wb, 64, add0, 0, None, 0,
                               None, st)
                    add0_mode = 0
                else:
                    add0, add0_mode = gs["f32"], (1 if blk.up else 2 if blk.down else 0)
                x_i = pool[("act", name)]
                mr0 = pool[(blk.name, "mr0", i)]
                g0, be0 = blk.g0[64 * i:64 * (i + 1)], blk.be0[64 * i:64 * (i + 1)]
                dg0 = G(m.norm0.weight)[64 * i:64 * (i + 1)]
                db0 = G(m.norm0.bias)[64 * i:64 * (i + 1)]
                first_consumer = consumers[name][0] == (blk.name, i)
                if not first_consumer:
                    # a later consumer (decoder skip connection): keep the partial gradient until the first one runs
                    pend = self._t(tw, ("pending", name), (B, Hi, Wi, 64), torch.float32)
                    self._gn_bwd(tw, d_ai, x_i, mr0, g0, be0, None, 1, rs, B, Hi, Wi, dg0, db0, None, add0, add0_mode,
                                 None, pend, None, False, eps, st)
                    pending[name] = pend
                else:
                    nd = need_dense(name)
                    gnext = self._gset(tw, B, Hi, Wi, parity, nd)
                    self._gn_bwd(tw, d_ai, x_i, mr0, g0, be0, None, 1, rs, B, Hi, Wi, dg0, db0, None, add0, add0_mode,
                                 pending.pop(name, None), None, gnext, nd, eps, st)
                    grads[name] = gnext

        # ---- first conv (weights only; the network input carries no gradient)
        gs = grads.pop("conv_in")
        cin = u.enc[self.conv_in_name]
        self._bias_grad(gs, B, G(cin.bias), st)
        self._wgrad(tw, gs["bf"], gs["flat"] is not None, 64, 0, pool["xin_pad"], False, B, H, W, 9, G(cin.weight),
                    cin.weight.shape[1], 0, st, ci_count=cin.weight.shape[1])

        # ---- embedding MLP and the per-block affine projections
        vec = self._t(tw, "embvec", (B, 320), torch.float32)
        d_aff_w = self._t(tw, "d_aff_w", (self.n_aff, 128, 64), torch.float32)
        d_aff_b = self._t(tw, "d_aff_b", (self.n_aff, 128), torch.float32)
        L.check(lib.mcedm_emb_mlp_bwd(L.ptr(pool["nl"]), L.ptr(self.freqs), L.ptr(self.w_m0), L.ptr(self.b_m0),
                                      L.ptr(self.w_m1), L.ptr(self.b_m1), L.ptr(self.aff_w), L.ptr(dss), self.n_aff, B,
                                      L.ptr(vec), L.ptr(d_aff_w), L.ptr(d_aff_b), L.ptr(G(u.map_layer1.weight)),
                                      L.ptr(G(u.map_layer1.bias)), L.ptr(G(u.map_layer0.weight)),
                                      L.ptr(G(u.map_layer0.bias)), st), "emb_mlp_bwd")
        blocks = self.blocks_enc + self.blocks_dec
        torch._foreach_copy_([G(b.mod.affine.weight) for b in blocks], list(d_aff_w.unbind(0)))
        torch._foreach_copy_([G(b.mod.affine.bias) for b in blocks], list(d_aff_b.unbind(0)))
        assert not grads and not pending, (list(grads), list(pending))
        self._flush_deferred(tw, st)
        for dst, src in self._post_copies:
            dst.copy_(src.t())
        return self._gflat
