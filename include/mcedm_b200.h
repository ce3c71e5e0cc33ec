/*
 * mcedm_b200 — C ABI of the B200-native m-cedm hot path (libmcedm_b200.so).
 *
 * The reference (katehai/m-cedm) is pure Python/PyTorch: it has no FFI, and every numerical step of
 * its hot path is a library call made from models/adm_blocks.py, models/mcedm.py and
 * models/losses.py.  Each entry point below replaces one such call site (cited as file:line,
 * relative to the reference root) and is what a maintainer binds with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless named host_*;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that stream;
 *   - return 0 on success; non-zero on failure with a message in mcedm_last_error();
 *   - activations inside the U-Net are NHWC ("channels last"), 64 channels per tensor:
 *       fp32 NHWC  = residual stream / conv outputs,
 *       bf16 NHWC  = tensor-core operands (normalised + activated tensors);
 *   - the public tensors of the reference API (x, cond, mask, D_x, sampler state) stay NCHW,
 *     fp32 (sampler state fp64), exactly as models/mcedm.py passes them.
 *   - op_fmt selects the format of every 16-bit tensor-core operand of a call (activations, packed weights and a
 *     16-bit output): 0 = bf16, 1 = fp16 (same layouts, same tensor throughput; names keep the `_bf16` suffix).
 *     Training uses bf16 throughout (gradients need its range); inference may use fp16, whose 11 significand bits
 *     cut the operand-rounding error of the network output ~8x (activations are normalised, weights are O(1)).
 *     MCEDM_FMT_F16_INF (3) = fp16 whose stores round a value beyond +-65504 to +-inf instead of clamping it: the
 *     16-bit gradient stores of dynamic loss scaling, so that an overflow reaches the fp32 flat gradient as inf / NaN
 *     and the optimizer step skips.  Accepted only by the gradient-writing entries whose comment names it.
 *   - there is NO CPU implementation behind any of these: without an sm_100 device they fail.
 */
#ifndef MCEDM_B200_H
#define MCEDM_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define MCEDM_ABI_VERSION 1
#define MCEDM_FMT_F16_INF 3
#if defined(__GNUC__)
#define MCEDM_API __attribute__((visibility("default")))
#else
#define MCEDM_API
#endif

/* -------------------------------------------------------------------------------------------- */
/* runtime                                                                                      */
/* -------------------------------------------------------------------------------------------- */
MCEDM_API int mcedm_abi_version(void);
MCEDM_API const char* mcedm_last_error(void);
/* Synchronises `stream`, returns non-zero if any kernel's bounded mbarrier wait timed out. */
MCEDM_API int mcedm_check_watchdog(void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K1  convolution as implicit GEMM on tcgen05  (models/adm_blocks.py:65-81 Conv2d.forward;       */
/*     fused residual add :171,:179; fused decoder concat :401; fused 1x1 skip conv :150-151)     */
/* -------------------------------------------------------------------------------------------- */
/*
 * out[b,y,x,:N] = bias + sum_s  src[seg_src[s]][b, y+seg_dy[s], x+seg_dx[s], 0:64] . w_packed[s][:N][0:64]
 *                 (+ residual)
 *   src[i]      : n_src (1..4) bf16 NHWC tensors [B,H,W,64]; reads outside the image are zero (padding)
 *   seg_*       : HOST int arrays of length n_seg (<= 20); dy,dx in {-1,0,1}
 *   w_packed    : bf16 [n_seg][N][64]   (see mcedm_b200.packing for the reference-weight permutation)
 *   bias        : fp32 [N] or NULL
 *   N           : 16, 64, 128 or 192 output channels
 *   out         : [B,H,W,N] fp32 (out_bf16 = 0) or bf16 (out_bf16 = 1)
 *   res,res_mode: 0 none | 1 res is fp32 [B,H,W,N] | 2 res is [B,H/2,W/2,N], nearest x2 upsampled
 *                 (Conv2d up, adm_blocks.py:73-74) | 3 res is [B,2H,2W,N], 2x2 mean (down, :75-77)
 *   stats_partial: NULL, or fp32 [B*H*W/128][N/4][2] receiving per-128-pixel-tile (sum, sum of squares)
 *                 of the stored values per 4-channel GroupNorm group (feeds mcedm_gn_apply).
 * Requires W | 128, 128 | H*W.
 * op_fmt MCEDM_FMT_F16_INF (N = 64, out_bf16 = 1): fp16 output without saturation (the 1x1 data gradients of dynamic
 * loss scaling).
 */
MCEDM_API int mcedm_conv_igemm(const void* const* src, int n_src, const int* seg_src, const int* seg_dy, const int* seg_dx,
                     int n_seg, const void* w_packed, const float* bias, int B, int H, int W, int N, void* out,
                     int out_bf16, const float* res, int res_mode, float* stats_partial, int op_fmt, void* stream);

/*
 * Row-resident variant of mcedm_conv_igemm for W == 128 (one tile = one image row): every input row is
 * fetched once (TMA box with a 1-pixel zero halo) and reused by its 9 taps through row-shifted UMMA
 * descriptors.  Same weight packing: w_packed = bf16 [9*n_halo + n_ctr][N][64], segment order
 * (halo source, ky, kx) then the centre sources.
 *   halo_src[i] : n_halo (1..2) bf16 NHWC [B,H,128,64] tensors convolved 3x3
 *   ctr_src[i]  : n_ctr (0..2) bf16 NHWC tensors entering with the centre tap only (1x1 skip projection)
 *   N           : 16 or 64; res_mode 0 | 1 | 2 as in mcedm_conv_igemm; out may alias res when res_mode == 1.
 *   stats_partial: NULL or fp32 [B*H][4][N/4][2]: one (sum, sum of squares) record per image row and
 *                 32-pixel quarter of it (no cross-warp reduction in the epilogue).
 */
MCEDM_API int mcedm_conv_rows(const void* const* halo_src, int n_halo, const void* const* ctr_src, int n_ctr,
                              const void* w_packed, const float* bias, int B, int H, int N, void* out, int out_bf16,
                              const float* res, int res_mode, float* stats_partial, int op_fmt, void* stream);

/*
 * Narrow-level (W <= 64) variant: the bf16 operand is a zero-padded flat pixel sequence (written by
 * mcedm_gn_apply with out_pitch/out_blk), position(b,y,x) = b*blk + (y+1)*pitch + x, so every filter tap
 * is a constant row offset and each 16 KB chunk of the input is fetched once.
 *   mcedm_flat_geometry: pitch = W + 1 (16 <= W <= 64), block_positions = roundup((H+2)*pitch, 128)
 *   src_flat  bf16 [B*block_positions, 64]; w_packed bf16 [9][64][64]; out fp32 NHWC [B,H,W,64] (dense)
 *   res_mode  0 | 1 | 2 | 3 as in mcedm_conv_igemm; out may alias res when res_mode == 1
 *   stats_partial NULL or fp32 [B*block_positions/128][4][16][2]
 */
MCEDM_API int mcedm_flat_geometry(int H, int W, int* pitch, int* block_positions);
MCEDM_API int mcedm_conv_flat(const void* src_flat, const void* w_packed, const float* bias, int B, int H, int W, int N,
                              float* out, const float* res, int res_mode, float* stats_partial, int op_fmt,
                              void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K1f  GroupNorm-fused convolutions with 16-bit activations (inference path)                     */
/*      (adm_blocks.py:161 / :166 / :403 silu(norm(x)[*(1+scale)+shift]) folded into Conv2d.forward :65-81)  */
/* -------------------------------------------------------------------------------------------- */
/*
 * Inference keeps every activation of the trunk in HBM as a RAW 16-bit tensor (op_fmt: fp16 by default) plus the
 * GroupNorm partial sums its producer emitted.  The consumer conv normalises on the fly: mcedm_gn_coef folds the
 * partial sums of a tensor into per-(sample, channel) coefficients (a | b), and the *_fused convs apply
 * y = silu(a*x + b) to each input row / chunk in shared memory right after its TMA load (transform warps), so the
 * normalised operand never exists in HBM.  Zero padding is preserved (padding pixels are not transformed).
 *
 * mcedm_conv_rows_fused (W == 128):
 *   halo_src[i], halo_coef[i]  n_halo (1..2) raw 16-bit NHWC [B,H,128,64] tensors and their fp32 [B][128] coefficients
 *   ctr_src[i]                 n_ctr (0..2) raw 16-bit tensors entering with the centre tap only, NOT transformed
 *                              (1x1 skip projection of the raw block input, adm_blocks.py:150-151)
 *   w_packed                   16-bit [9*n_halo + n_ctr][n_total][64]; this launch computes output channels
 *                              [n_off, n_off + N) of n_total (N = 16 | 32 | 64): a 128-channel conv0 runs as two N = 32
 *                              launches whose 72 KB of weights stay resident
 *   bias fp32 [n_total] | NULL; out [B,H,128,n_total] 16-bit (out_16 = 1) or fp32 (0)
 *   res16, res_mode            0 none | 1 16-bit [B,H,128,n_total] | 2 16-bit half-resolution tensor, nearest-x2:
 *                              dense [B,H/2,64,n_total] (res_pitch = 0) or padded-flat (res_pitch, res_blk)
 *   halo_coef == NULL (or all entries NULL): the halo sources are already-normalised operands (no transform);
 *   likewise coef == NULL in mcedm_conv_flat_fused (the conv0 of an up/down block reads mcedm_gn_apply16 output)
 *   stats_partial              NULL or fp32 [B*H][4][n_total/4][2] (this launch fills groups n_off/4 ...)
 *   op_fmt                     1, or MCEDM_FMT_F16_INF for the data gradient of a 3x3 conv under dynamic loss
 *                              scaling (N = 64, no coefficients, no residual, 16-bit out without saturation); the
 *                              same holds for mcedm_conv_flat_fused
 * mcedm_conv_flat_fused (W <= 64): src/out/res in the padded-flat layout of mcedm_flat_geometry
 *   out_flat   16-bit [B*blk][64] (out_f32 = 0) or fp32 [B*blk][64] (out_f32 = 1, K-split partial); only data
 *              positions are written (padding must have been zeroed once by the owner)
 *   res        res_mode 1: same-resolution padded-flat, 16-bit or fp32 (res_f32 = 1);
 *              2: 16-bit at half resolution, 3: 16-bit at double resolution (2x2 mean); for 2/3 the residual tensor's
 *              own layout is given by res_pitch/res_blk (0,0 = dense NHWC, e.g. the 128-wide level)
 *   stats_partial  NULL or fp32 [B*blk/128][4][16][2]
 * mcedm_conv_igemm16: mcedm_conv_igemm with a 16-bit output and a prefetched 16-bit residual (res_mode 0 | 1);
 *   io_pitch/io_blk > 0 place out and res in the padded-flat layout (sources stay dense).
 * mcedm_gn_apply16: stand-alone apply for the places that still need a materialised operand (2x resampling in front
 *   of conv0, norm2 in front of the qkv projection): x16 raw 16-bit, dense (in_pitch = 0) or padded-flat; coef from
 *   mcedm_gn_coef; act / resample / out_pitch / out_blk as in mcedm_gn_apply.  out_pooled16 (resample != 0 only, may
 *   be NULL): the RAW input resampled the same way (2x2 mean / nearest x2) in out16's layout — the skip path of a down /
 *   up block (adm_blocks.py:149-151), consumed by conv1 as a same-resolution residual instead of a gather in its epilogue.
 * mcedm_conv_in16: mcedm_conv_in writing a 16-bit NHWC tensor.
 */
MCEDM_API int mcedm_gn_coef(const float* partial, int parts_per_img, const float* gamma, const float* beta,
                            const float* scale_shift, int emb_batch_stride, int emb_shift_offset, float eps, int B,
                            int Hin, int Win, float* coef_out, float* meanrstd_out, void* stream);
MCEDM_API int mcedm_gn_apply16(const void* x16, int in_pitch, int in_blk, const float* coef, int act, int resample,
                               int B, int Hin, int Win, int out_pitch, int out_blk, void* out16, void* out_pooled16,
                               int op_fmt, void* stream);
/* Dropout of the training forward (UNetBlock.forward, adm_blocks.py:167: conv1's operand).
 * mcedm_gn_apply16_dropout: mcedm_gn_apply16 with act = 1, resample = 0, then out = 16-bit(silu(a*x + b) * scale) where
 *   the element is kept and 0 elsewhere (one rounding, exact SiLU).  Layouts in / out as in mcedm_gn_apply16 (padding
 *   positions of a padded-flat output are not written).
 * mcedm_dropout_bwd16: g16 (dense: pitch = 0, or padded-flat) <- 16-bit(g16 * scale) where kept, 0 elsewhere, in place.
 * Mask of element (b, y, x, c) at H x W: logical index n = ((b*H + y)*W + x)*64 + c in either layout; Philox4x32-10 with
 *   counter (n >> 2, n >> 34, layer, step) and key (seed_lo, seed_hi), word n & 3; kept iff word >= threshold
 *   (= min(2^32 - 1, floor(p * 2^32))).  rng: device uint32 {seed_lo, seed_hi, step}, read at run time.
 *   mcedm_dropout_bwd16 also takes op_fmt MCEDM_FMT_F16_INF (fp16 without saturation, dynamic loss scaling). */
MCEDM_API int mcedm_gn_apply16_dropout(const void* x16, int in_pitch, int in_blk, const float* coef, int B, int H, int W,
                                       int out_pitch, int out_blk, void* out16, unsigned int threshold, float scale,
                                       int layer, const unsigned int* rng, int op_fmt, void* stream);
MCEDM_API int mcedm_dropout_bwd16(void* g16, int pitch, int blk, int B, int H, int W, unsigned int threshold, float scale,
                                  int layer, const unsigned int* rng, int op_fmt, void* stream);
MCEDM_API int mcedm_conv_rows_fused(const void* const* halo_src, const float* const* halo_coef, int n_halo,
                                    const void* const* ctr_src, int n_ctr, const void* w_packed, const float* bias,
                                    int B, int H, int N, int n_off, int n_total, void* out, int out_16,
                                    const void* res16, int res_mode, int res_pitch, int res_blk,
                                    float* stats_partial, int op_fmt, void* stream);
/* Output head: out_conv(silu(out_norm(x))) (adm_blocks.py:403) as one launch writing F_x fp32 NCHW [B, c_out, H, 128]
 * straight from the accumulators (w_packed 16-bit [9][16][64], rows >= c_out zero; bias fp32 [>= c_out]). */
MCEDM_API int mcedm_conv_head_fused(const void* src16, const float* coef, const void* w_packed, const float* bias, int B,
                                    int H, int c_out, float* F_nchw, int op_fmt, void* stream);
MCEDM_API int mcedm_conv_flat_fused(const void* src_flat16, const float* coef, const void* w_packed, const float* bias,
                                    int B, int H, int W, int N, void* out_flat, int out_f32, const void* res,
                                    int res_mode, int res_f32, int res_pitch, int res_blk, float* stats_partial,
                                    int op_fmt, void* stream);
MCEDM_API int mcedm_conv_igemm16(const void* const* src, int n_src, const int* seg_src, const int* seg_dy,
                                 const int* seg_dx, int n_seg, const void* w_packed, const float* bias, int B, int H,
                                 int W, int N, void* out16, const void* res16, int res_mode, int io_pitch, int io_blk,
                                 float* stats_partial, int op_fmt, void* stream);
/* The same first conv on the tensor cores (W == 128, Cc + Cx <= 5): builder warps fold the three horizontal taps into
 * K (k = kx*Cin + c, one K = 16 step per input row), the vertical taps are stacked into N as in mcedm_conv_rows_fused.
 * w16_packed: 16-bit [3 ky][64 co][64 k], zero beyond k = 3*Cin (engine.pack). Inputs are rounded to 16 bits once. */
MCEDM_API int mcedm_conv_in_tc16(const float* x, int Cx, const float* cond, int Cc, const void* w16_packed,
                                 const float* bias, int B, int H, void* out16, float* stats_partial, int op_fmt,
                                 void* stream);
MCEDM_API int mcedm_conv_in16(const float* x, int Cx, const float* cond, int Cc, const float* w, const float* bias,
                              int B, int H, int W, void* out16, float* stats_partial, int op_fmt, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* fp32-accuracy inference mode (per-step denoiser output within 1e-4 of the fp32 reference)      */
/* -------------------------------------------------------------------------------------------- */
/*
 * Every tensor-core operand is split into two fp16 terms (x = hi + lo) and every GEMM is issued three times
 * (hi*W_hi, lo*W_hi, hi*W_lo) through the regular entry points with in-place fp32 accumulation (res_mode 1, res == out).
 *   mcedm_gn_apply_split: mcedm_gn_apply writing the operand as a (hi, lo) fp16 pair (and the raw copy likewise);
 *   mcedm_split16:        fp32 [n] -> (hi, lo) fp16;
 *   mcedm_attention_f32:  softmax(q k^T / 8) v in fp32 (CUDA cores) on fp32 qkv [B,L,192] -> fp32 [B,L,64]
 *                         (adm_blocks.py:103-109 computes the softmax in fp32).
 */
MCEDM_API int mcedm_gn_apply_split(const float* x, const float* partial, const float* gamma, const float* beta,
                                   const float* scale_shift, int emb_batch_stride, int emb_shift_offset, float eps,
                                   int act, int resample, int B, int Hin, int Win, int parts_per_img, int out_pitch,
                                   int out_blk, void* out_hi, void* out_lo, void* raw_hi, void* raw_lo,
                                   float* coef_scratch, void* stream);
MCEDM_API int mcedm_split16(const float* x, long long n, void* hi16, void* lo16, void* stream);
MCEDM_API int mcedm_attention_f32(const float* qkv_f32, int B, int L, float* out_f32, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K2  GroupNorm statistics / fused GroupNorm + scale-shift + SiLU + resample                     */
/*     (models/adm_blocks.py:86-97 GroupNorm; :161, :163-166, :175, :403 call sites)              */
/* -------------------------------------------------------------------------------------------- */
/* partial[t][g][0..1] = (sum, sum of squares) over pixel tile t (128 pixels) and group g (4 channels)
 * of an fp32 [n_pixels, 64] tensor.  Same format conv_igemm/conv_in emit from their epilogues. */
MCEDM_API int mcedm_gn_stats(const float* x, long long n_pixels, float* partial, void* stream);
/*
 * out = act( GroupNorm(x) * (1 + scale) + shift ), optionally resampled, written as bf16 NHWC.
 *   x            fp32 NHWC [B,Hin,Win,64]; partial = its statistics records [B*parts_per_img][16][2]
 *                (parts_per_img = 0 means Hin*Win/128, the mcedm_conv_igemm / mcedm_gn_stats format;
 *                mcedm_conv_rows emits 4 records per image row: parts_per_img = 4*Hin)
 *   gamma, beta  fp32 [64] (slice of the GroupNorm affine for these 64 channels)
 *   scale_shift  NULL, or fp32 with scale[c] at [b*emb_batch_stride + c] and shift[c] at
 *                [b*emb_batch_stride + emb_shift_offset + c]  (affine(emb).chunk(2), adm_blocks.py:163-165;
 *                emb_batch_stride = 0 broadcasts one embedding over the batch, as in sampling)
 *   act          0 identity (norm2), 1 SiLU
 *   resample     0 none | 1 nearest x2 (out is [B,2Hin,2Win,64]) | 2 2x2 mean (out is [B,Hin/2,Win/2,64]);
 *                this is the resampling Conv2d applies before its 3x3 filter (adm_blocks.py:73-77)
 *   out_pitch, out_blk  0, 0: out is dense NHWC; otherwise out is the zero-padded flat layout consumed by
 *                mcedm_conv_flat (values from mcedm_flat_geometry at the OUTPUT resolution); only data
 *                positions are written, the padding must have been zeroed once by the owner of the buffer
 *   out_raw_bf16 NULL, or receives bf16(x) in dense NHWC (operand of the block's 1x1 skip projection)
 *   meanrstd_out NULL, or fp32 [B][16][2] receiving (mean, rstd) per group, saved for mcedm_gn_bwd
 *   coef_scratch fp32 [B][128] scratch: per-channel (a | b) of y = act(a*x + b), written by the finalize launch
 *                and read by the streaming launch (two launches per call)
 */
MCEDM_API int mcedm_gn_apply(const float* x, const float* partial, const float* gamma, const float* beta,
                             const float* scale_shift, int emb_batch_stride, int emb_shift_offset, float eps, int act,
                             int resample, int B, int Hin, int Win, int parts_per_img, int out_pitch, int out_blk,
                             void* out_bf16, void* out_raw_bf16, float* meanrstd_out, float* coef_scratch,
                             int op_fmt, void* stream);

/*
 * Backward of mcedm_gn_apply (training; autograd of adm_blocks.py:95, :161, :166).  Two launches: per-CTA partial
 * sums of (du, du*xh) per channel, and the element pass, whose CTAs first fold the partials of their sample in a fixed
 * order (CTA 0 of each sample also writes dgb_partial / d_scale_shift).
 *   dy            fp32 NHWC gradient w.r.t. the operand gn_apply wrote (at the conv resolution)
 *   x, meanrstd   saved forward input and its (mean, rstd) records
 *   red_partial   scratch fp32 [B][mcedm_gn_bwd_ctas_per_img(Hin,Win,B)][64][2];  coef: unused (NULL allowed)
 *   dgb_partial   out fp32 [B][64][2]: per-sample (d gamma, d beta) contributions (sum over b = the gradient)
 *   d_scale_shift NULL or out: d scale at [b*dss_batch_stride + c], d shift at [... + emb_shift_offset + c]
 *   add0/add1     NULL or fp32 tensors added to dx (residual-path gradients); add0_mode 0 same resolution,
 *                 1 add0 is at 2x resolution (adjoint of a nearest-x2 skip: sum of 4), 2 add0 is at 1/2 resolution
 *                 (adjoint of a 2x2-mean skip: 0.25 * nearest)
 *   dx            NULL or out fp32 NHWC [B,Hin,Win,64]; dx_bf16 NULL or bf16 copy (dense, or padded-flat with
 *                 out_pitch/out_blk); dx_bf16_dense NULL or a second, always dense bf16 copy (operand of the 1x1
 *                 convolutions); colsum_partial NULL or out fp32 [B*ctas_per_img][64] column sums of dx
 */
MCEDM_API int mcedm_gn_bwd_ctas_per_img(int Hin, int Win, int B);
MCEDM_API int mcedm_gn_bwd(const float* dy, const float* x, const float* meanrstd, const float* gamma,
                           const float* beta, const float* scale_shift, int emb_batch_stride, int emb_shift_offset,
                           float eps, int act, int resample, int B, int Hin, int Win, float* red_partial, float* coef,
                           float* dgb_partial, float* d_scale_shift, int dss_batch_stride, const float* add0,
                           int add0_mode, const float* add1, float* dx, void* dx_bf16, int out_pitch, int out_blk,
                           void* dx_bf16_dense, float* colsum_partial, void* stream);
/*
 * The same backward for the 16-bit training plan ("fused16", train_engine.py): x16 is the RAW 16-bit activation the
 * fused forward stored, dy16 the 16-bit output of a data-gradient conv, both in op_fmt (0 bf16, 1 fp16); residual-path
 * gradients (add0 / add1) and dx stay fp32.  Every tensor carries its own layout: (pitch, blk) = (0, 0) dense NHWC, else
 * the padded-flat layout of mcedm_flat_geometry AT THAT TENSOR'S RESOLUTION (dy: the conv resolution; add0: per
 * add0_mode; x, add1, dx, dx16: Hin x Win).  dx16: 16-bit copy in x's layout; dx16_dense: a second, dense copy.
 * add16 != 0: add0 / add1 are 16-bit (op_fmt) too — the gradient of the residual stream without an fp32 master copy.
 * meanrstd / coef_ab: what the forward's mcedm_gn_coef wrote for this GroupNorm ([B][16][2], [B][128]).
 * kcoef: scratch fp32 [B][192]; ticket: uint32 [3][B], ZERO before the first launch (each launch leaves it zero): the
 * last CTA of a sample to finish pass 1 folds that sample's partials once (fixed order: deterministic).  When the whole
 * grid is resident at once (ctas_per_img * B <= 2 x SM count) both passes run as ONE kernel: the sample's other CTAs
 * wait for that fold in the kernel and re-read their slice from L2 (words [B..3B) are the flag and the departure count).
 * Win must be a power of two.  red_partial / dgb_partial / colsum_partial as in mcedm_gn_bwd, sized with
 * mcedm_gn_bwd16_ctas_per_img.  op_fmt MCEDM_FMT_F16_INF: fp16 whose dx16 / dx16_dense stores do not saturate (dynamic
 * loss scaling).
 */
MCEDM_API int mcedm_gn_bwd16_ctas_per_img(int Hin, int Win, int B);
MCEDM_API int mcedm_gn_bwd16(const void* dy16, int dy_pitch, int dy_blk, const void* x16, int x_pitch, int x_blk,
                             int op_fmt, const float* meanrstd, const float* coef_ab, const float* gamma,
                             const float* beta, const float* scale_shift, int emb_batch_stride, int emb_shift_offset,
                             int act, int resample, int B, int Hin, int Win, float* red_partial, float* kcoef,
                             unsigned int* ticket, float* dgb_partial, float* d_scale_shift, int dss_batch_stride,
                             const void* add0, int add0_mode, int add0_pitch, int add0_blk, const void* add1,
                             int add16, float* dx, void* dx16, void* dx16_dense, float* colsum_partial, void* stream);
/* out[j] (+)= scale * sum_r in[r*stride_r + j*stride_j]  (ordered fp64 sum; folds per-CTA / per-sample partials) */
MCEDM_API int mcedm_reduce_rows(const float* in, int n_rows, long long stride_r, int n_cols, long long stride_j,
                                float* out, int accumulate, float scale, void* stream);
/* The same fold for a device-resident table of jobs in one launch (grid.y = job). The backward of a training step
 * queues its ~60 bias / gamma / beta folds and runs them together; outputs of different jobs must not overlap. */
typedef struct mcedm_reduce_job {
  const float* in;
  float* out;
  long long stride_r, stride_j;
  int n_rows, n_cols, accumulate;
  float scale;
} mcedm_reduce_job;
MCEDM_API int mcedm_reduce_rows_batched(const mcedm_reduce_job* jobs_dev, int n_jobs, int max_cols, void* stream);
/* K6: masked weighted EDM loss and dL/dF (mcedm.py:213-239, :278; losses.py:48-53). NCHW fp32, chw elements per
 * sample; loss = (1/B) * sum(loss_partial[B][ctas_per_sample]); dF may be NULL (forward value only).
 * dF_pad_bf16 NULL, or bf16 NHWC [B, hw, 64] whose first chw/hw channels receive dL/dF (the other channels must
 * have been zeroed by the owner): the tensor-core operand of out_conv's weight / data gradient. */
MCEDM_API int mcedm_edm_loss(const float* F, const float* x_noise, const float* x, const float* mask,
                             const float* c_skip, const float* c_out, const float* weight, int B, long long chw,
                             float* dF, void* dF_pad_bf16, long long hw, float* loss_partial, int ctas_per_sample,
                             void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K1w  convolution weight gradient on tcgen05 (autograd of models/adm_blocks.py:65-81)           */
/* -------------------------------------------------------------------------------------------- */
/*
 * partial[cta][tap][co][ci] = sum over the CTA's image rows of dy[b,y,x,co] * a[b,y+ky-1,x+kx-1,ci]
 *   dy, a      bf16 pixel tensors, each a 64-channel block (c_off) of a tensor with c_total channels, in
 *              layout 0 (dense NHWC [B,H,W,c_total]) or 1 (padded-flat of mcedm_flat_geometry, W <= 64)
 *   taps       9 (3x3, tap = ky*3+kx) or 1 (1x1 convolutions: qkv, proj, skip)
 *   partial    fp32 [mcedm_wgrad_ctas(B,H,W)][taps][64][64]
 * mcedm_wgrad_reduce folds the partials in a fixed order (fp64) into the reference weight layout:
 *   dw[(co*co_mul + co_add)][ci_off + ci][tap] (+)= sum_cta partial[cta][tap][co][ci],  dw = [Cout][cin_total][k][k]
 *   for co < co_count, ci < ci_count (out_conv has 2 real output channels, the first conv 4 real inputs)
 * W % 16 == 0, 16 <= W <= 128.
 */
MCEDM_API int mcedm_wgrad_ctas(int B, int H, int W);
MCEDM_API int mcedm_conv_wgrad(const void* dy, int dy_layout, int dy_ctotal, int dy_coff, const void* a, int a_layout,
                               int a_ctotal, int a_coff, int B, int H, int W, int taps, float* partial, void* stream);
/* mcedm_conv_wgrad with both operands in op_fmt (0 bf16, 1 fp16; kind::f16 MMAs need one format for A and B). */
MCEDM_API int mcedm_conv_wgrad16(const void* dy, int dy_layout, int dy_ctotal, int dy_coff, const void* a, int a_layout,
                                 int a_ctotal, int a_coff, int B, int H, int W, int taps, float* partial, int op_fmt,
                                 void* stream);
/* The same with `a` a RAW 64-channel activation: the operand act(a_coef.a * x + a_coef.b) (a_coef fp32 [B][128] from
 * mcedm_gn_coef; a_act 1 SiLU, 0 identity) is formed row by row in shared memory by the warps that otherwise only run
 * the epilogue, so the normalised operand of a weight gradient never exists in HBM (adm_blocks.py:161 / :166).
 * a_coef NULL = mcedm_conv_wgrad16. */
MCEDM_API int mcedm_conv_wgrad16_fused(const void* dy, int dy_layout, int dy_ctotal, int dy_coff, const void* a,
                                       int a_layout, int a_ctotal, int a_coff, const float* a_coef, int a_act, int B,
                                       int H, int W, int taps, float* partial, int op_fmt, void* stream);
MCEDM_API int mcedm_wgrad_reduce(const float* partial, int n_ctas, int taps, float* dw, int cin_total, int ci_off,
                                 int co_mul, int co_add, int co_count, int ci_count, int accumulate, void* stream);
/* Every weight-gradient fold of a step in one launch (same arithmetic and order as mcedm_wgrad_reduce, accumulate = 0);
 * each job needs its own partial buffer. */
typedef struct mcedm_wgrad_job {
  const float* partial;
  float* dw;
  int n_ctas, taps, cin_total, ci_off, co_mul, co_add, co_count, ci_count;
} mcedm_wgrad_job;
MCEDM_API int mcedm_wgrad_reduce_batched(const mcedm_wgrad_job* jobs_dev, int n_jobs, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K3  fused self-attention (models/adm_blocks.py:103-109 AttentionOp.forward, :176-178)          */
/* -------------------------------------------------------------------------------------------- */
/* qkv bf16 [B,L,192] = (q|k|v) x 64 channels; out bf16 [B,L,64]; softmax(q.k/8) in fp32. L % 128 == 0.
 * lse_out NULL, or fp32 [B,L] receiving the base-2 log-sum-exp of each row (saved for mcedm_attention_bwd). */
MCEDM_API int mcedm_attention(const void* qkv_bf16, int B, int L, void* out_bf16, float* lse_out, int op_fmt,
                              void* stream);
/*
 * Backward of mcedm_attention (autograd of adm_blocks.py:103-118 AttentionOp + the einsum at :178):
 *   given d_out bf16 [B,L,64] (gradient w.r.t. out), the saved qkv / out / lse, writes dq, dk, dv bf16 [B,L,64].
 *   dvec  scratch fp32 [B,L]  (D_i = sum_c d_out[i,c] * out[i,c])
 * Two tcgen05 kernels (one CTA per 128 queries for dq, one CTA per 128 keys for dk/dv) recompute
 * P = exp2(S*log2e/8 - lse) tile by tile; the L x L matrices never reach HBM.
 */
MCEDM_API int mcedm_attention_bwd(const void* qkv_bf16, const void* out_bf16, const void* d_out_bf16, const float* lse,
                                  int B, int L, float* dvec, void* dq_bf16, void* dk_bf16, void* dv_bf16, void* stream);
/* The same with every 16-bit tensor (inputs, P / dS operand tiles, outputs) in op_fmt (0 bf16, 1 fp16;
 * MCEDM_FMT_F16_INF: fp16 whose dS tiles and outputs do not saturate, dynamic loss scaling). */
MCEDM_API int mcedm_attention_bwd16(const void* qkv16, const void* out16, const void* d_out16, const float* lse, int B,
                                    int L, float* dvec, void* dq16, void* dk16, void* dv16, int op_fmt, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* embedding MLP, first conv, output head                                                        */
/* -------------------------------------------------------------------------------------------- */
/* emb = silu(L1(silu(L0([cos|sin](c_noise x freqs)))))  (adm_blocks.py:185-199, :367-379), then
 * out[a][b][0:128] = aff_w[a] @ emb[b] + aff_b[a] for the n_aff blocks (adm_blocks.py:163).
 * freqs fp32 [32]; w0,w1 fp32 [64,64]; aff_w fp32 [n_aff,128,64]; emb_out NULL or [Bemb,64]. */
MCEDM_API int mcedm_emb_mlp(const float* c_noise, const float* freqs, const float* w0, const float* b0,
                            const float* w1, const float* b1, const float* aff_w, const float* aff_b, int n_aff,
                            int Bemb, float* emb_out, float* out, void* stream);
/* 3x3 conv of cat([cond, x]) (NCHW fp32, Cc + Cx <= 8 channels) -> fp32 NHWC [B,H,W,64] + tile statistics
 * (adm_blocks.py:319-340 cat_conditioning, :384-385). w fp32 [64, Cc+Cx, 3, 3] in the reference layout. */
MCEDM_API int mcedm_conv_in(const float* x, int Cx, const float* cond, int Cc, const float* w, const float* bias,
                            int B, int H, int W, float* out, float* stats_partial, void* stream);
/* dst NCHW fp32 [B,Cout,H,W] = first Cout channels of src NHWC fp32 [B,H,W,Cs] (out_conv result, :403). */
MCEDM_API int mcedm_head_to_nchw(const float* src, int Cs, int Cout, int B, int H, int W, float* dst, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K4/K5  EDM preconditioning and stochastic-Heun sampler updates with mask blending              */
/*        (models/mcedm.py:199-211, :443-461, :570-638)                                           */
/* -------------------------------------------------------------------------------------------- */
/* All tensors NCHW; state fp64, network I/O fp32, mask fp32 (1 = missing/generated, 0 = observed). */
/* x = cond[:, :C]*(1-mask) + (noise*t0)*mask                                   (mcedm.py:590-597) */
MCEDM_API int mcedm_edm_init(const float* noise, const float* cond, int Ccond, const float* mask, double t0, int B,
                             int C, int H, int W, double* x, void* stream);
/* x_hat = x_cur + coef*eps*mask ; x_in = c_in*float(x_hat)       coef = sqrt(t_hat^2-t_cur^2)*S_noise (:608) */
MCEDM_API int mcedm_edm_churn(const double* x_cur, const double* eps, const float* mask, double coef, float c_in,
                              long long total, double* x_hat, float* x_in, void* stream);
/* D = c_skip*float(x_hat)+c_out*F ; d_cur = (x_hat-D)/t_hat ; x_next = x_hat+(t_next-t_hat)*d_cur*mask ;
 * x_in = c_in_next*float(x_next) (x_in, D_out may be NULL)                                 (:612-618) */
MCEDM_API int mcedm_edm_euler(const double* x_hat, const float* F, const float* mask, double t_hat, double t_next,
                              float c_skip, float c_out, float c_in_next, long long total, double* d_cur,
                              double* x_next, float* x_in, float* D_out, void* stream);
/* second-order correction                                                                  (:621-628) */
MCEDM_API int mcedm_edm_correct(const double* x_hat, const double* x_e, const float* F2, const double* d_cur,
                                const float* mask, double t_hat, double t_next, float c_skip, float c_out,
                                long long total, double* x_next, float* D_out, void* stream);
/* x_in[b] = c_in[b*stride] * x[b]                                       (mcedm.py:208, :454) */
MCEDM_API int mcedm_edm_precond_in(const float* x, const float* c_in, int coef_stride, int B, long long chw,
                                   float* x_in, void* stream);
/* D[b] = c_skip[b*stride]*x[b] + c_out[b*stride]*F[b]   (mcedm.py:210, :460); chw = elements per sample */
MCEDM_API int mcedm_edm_precond_out(const float* x, const float* F, const float* c_skip, const float* c_out,
                                    int coef_stride, int B, long long chw, float* D, void* stream);
/* PDE-guided sampler (PlCondDdim.sample_edm with guide_dx, models/ddim.py:1566-1590):
 * D = c_skip*float(x) + c_out*F with scalar coefficients (get_denoised, ddim.py:1756-1766) */
MCEDM_API int mcedm_edm_denoised(const double* x, const float* F, float c_skip, float c_out, long long total, float* D,
                                 void* stream);
/* d_cur = (x_hat - D)/t_hat - (5*gdx)/t_hat [float32 term] ; x_next = x_hat + ((t_next-t_hat)*d_cur)*mask ;
 * x_in = c_in_next*float(x_next) (x_in may be NULL)                                            (ddim.py:1569-1573) */
MCEDM_API int mcedm_edm_euler_guided(const double* x_hat, const float* D, const float* gdx, const float* mask,
                                     double t_hat, double t_next, float c_in_next, long long total, double* d_cur,
                                     double* x_next, float* x_in, void* stream);
/* d' = (x_e - D2)/t_next - (5*gdx)/t_hat ; x_next = x_hat + ((t_next-t_hat)*(0.5 d_cur + 0.5 d'))*mask  (:1588-1592) */
MCEDM_API int mcedm_edm_correct_guided(const double* x_hat, const double* x_e, const float* D2, const float* gdx,
                                       const double* d_cur, const float* mask, double t_hat, double t_next,
                                       long long total, double* x_next, void* stream);
/* Classifier-free guidance: the network runs once on 2B rows, rows [0, B) with cond and rows [B, 2B) with the all-zero
 * condition, both on the same x_in; F (2*total elements) = [F_c | F_u].  The kernels below read
 *   F_w = (1+w)*F_c - w*F_u   (fp32; (1+w) and w rounded to fp32 in the call, two rounded products, one rounded
 *                              difference, no FMA)
 * where their siblings above read F, with otherwise the same arithmetic.  w must be finite.
 * churn_cfg: as edm_churn, writing x_in to both halves (2*total elements);
 * euler_cfg / correct_cfg: as edm_euler / edm_correct with F_w; euler_cfg writes x_in to both halves;
 * denoised_cfg: as edm_denoised with F_w (the PDE-guided sampler then runs edm_euler_guided / _correct_guided on D);
 * precond_out_cfg: as edm_precond_out with F_w (B rows), also writing F_w to F_w_out. */
MCEDM_API int mcedm_edm_churn_cfg(const double* x_cur, const double* eps, const float* mask, double coef, float c_in,
                                  long long total, double* x_hat, float* x_in, void* stream);
MCEDM_API int mcedm_edm_euler_cfg(const double* x_hat, const float* F, const float* mask, double t_hat, double t_next,
                                  float c_skip, float c_out, float c_in_next, double w, long long total, double* d_cur,
                                  double* x_next, float* x_in, float* D_out, void* stream);
MCEDM_API int mcedm_edm_correct_cfg(const double* x_hat, const double* x_e, const float* F2, const double* d_cur,
                                    const float* mask, double t_hat, double t_next, float c_skip, float c_out, double w,
                                    long long total, double* x_next, float* D_out, void* stream);
MCEDM_API int mcedm_edm_denoised_cfg(const double* x, const float* F, float c_skip, float c_out, double w,
                                     long long total, float* D, void* stream);
MCEDM_API int mcedm_edm_precond_out_cfg(const float* x, const float* F, const float* c_skip, const float* c_out,
                                        int coef_stride, double w, int B, long long chw, float* D, float* F_w_out,
                                        void* stream);
/* RePaint-style conditioning of PlDdim.sample_edm (models/ddim.py:959-1051; mask == 1 means KNOWN):
 * x0 = double((hu*sqrt_a + noise*sqrt_1ma)*mask + noise*(1-mask)) * t0                          (:987-993) */
MCEDM_API int mcedm_edm_vp_init(const float* hu, const float* noise, const float* mask, float sqrt_a, float sqrt_1ma,
                                double t0, long long total, double* x, void* stream);
/* x = double((sqrt_a*hu + sqrt_1ma*noise)*mask) + x*double(1-mask), in place (:1029-1031); sqrt_a = 1, sqrt_1ma = 0 is
 * the final replacement `hu*mask + x*(1-mask)` (:1040-1041) */
MCEDM_API int mcedm_edm_repaint_blend(const float* hu, const float* noise, const float* mask, float sqrt_a,
                                      float sqrt_1ma, long long total, double* x, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K6: PDE residual of sampled fields and its gradient (pde.cu)                                  */
/* -------------------------------------------------------------------------------------------- */
/* A field channel is a "plane": element (b,t,x) at base[b*strides[0] + t*strides[1] + x*strides[2]] (element units),
 * float32 or float64 (f64 flag), cast to float32 on load.  With apply_norm the un-normalised value is v*div + sub
 * (Normalizer(inverse=True), models/normalizer.py:26-27); div always supplies the residual scale div^2
 * (SweFvLoss.get_scaling, models/pde_loss.py:187-197).
 *
 * SweFvLoss.calculate_loss (models/pde_loss.py:199-215) as called by PlMcedm.get_pde_loss (models/mcedm.py:468-499)
 * and PlCondDdim.get_pde_loss (models/ddim.py:1388-1422): one FORCE finite-volume step (pde_loss.py:129-165) of every
 * row t, compared with row t+1 of gt (gt = NULL: with the un-normalised prediction itself); NaN -> 0.
 * half_dt = float32(0.5*Tn/T), dx = the float32 grid spacing of gen_x (:104-118).  loss [B,T,X,2] float32 (may be
 * NULL) is bit-identical to the reference's matrix; row_sums [B*T] float64 workspace; total (may be NULL) receives
 * the float64 sum of all entries (torch.sum in the reference). */
MCEDM_API int mcedm_swe_fv_loss(const void* h, int h_f64, const long long* h_strides, const void* u, int u_f64,
                                const long long* u_strides, int apply_norm, float h_div, float h_sub, float u_div,
                                float u_sub, const float* gt, int B, int T, int X, float half_dt, float dx, float g,
                                float* loss, double* row_sums, double* total, void* stream);
/* SweFvLoss.forward(return_d=True) (models/pde_loss.py:231-242): d mean(loss matrix)/d pred (un-normalised), gt held
 * constant, NaN -> 0; analytic adjoint instead of autograd.  mode 0: out [B,T,X,2]; 1: out [B,T,X] = channel mean
 * (PlCondDdim.get_dx_pde with calc_prob, models/ddim.py:1445-1446); 2: channel sum (:1448). */
MCEDM_API int mcedm_swe_fv_grad(const void* h, int h_f64, const long long* h_strides, const void* u, int u_f64,
                                const long long* u_strides, int apply_norm, float h_div, float h_sub, float u_div,
                                float u_sub, const float* gt, int B, int T, int X, float half_dt, float dx, float g,
                                int mode, float* out, void* stream);
/* DarcyLoss.calculate_loss + forward's /(t*n) (models/pde_loss.py:30-56, :81-84): a, u planes of [B,S,S];
 * loss [B,S-4,S-4] float32 (may be NULL), row_sums [B*(S-4)] float64 workspace, total as above. */
MCEDM_API int mcedm_darcy_loss(const void* a, int a_f64, const long long* a_strides, const void* u, int u_f64,
                               const long long* u_strides, int apply_norm, float a_div, float a_sub, float u_div,
                               float u_sub, int B, int S, float D, float* loss, double* row_sums, double* total,
                               void* stream);

/* -------------------------------------------------------------------------------------------- */
/* training-side small kernels (train_small.cu)                                                  */
/* -------------------------------------------------------------------------------------------- */
/* x_noise = x + mask*noise*sigma[b] ; x_in = c_in[b]*x_noise   (mcedm.py:216, :208); mask may be NULL */
MCEDM_API int mcedm_edm_noise_in(const float* x, const float* noise, const float* mask, const float* sigma,
                                 const float* c_in, int B, long long chw, float* x_noise, float* x_in, void* stream);
/* Batch preparation of PlMcedm.training_step in one pass (mcedm.py:257-265 data_transform + rearranges, :241-252
 * get_cond_in, normalizer.py:28-29): x = ((h - h_sub)/h_div | (u - u_sub)/u_div), cond = x*(1-mask) + randn*mask.
 * h, u [B,HW]; mask, randn [B,HW,2] channel-last; x, cond, mask_c [B,2,HW] channel-first.  Bit-identical to torch. */
MCEDM_API int mcedm_mcedm_prep(const float* h, const float* u, const float* mask, const float* randn, float h_sub,
                               float h_div, float u_sub, float u_div, int B, long long HW, float* x, float* cond,
                               float* mask_c, void* stream);
/* mcedm_mcedm_prep with the mask generated on the device (SURVEY 8f rank 3; h5_dataset.py:232-255, :306-393): every
 * mask of the reference's datasets is "channel c missing from time row obs_rows[b][c] on" (0 = whole channel missing,
 * H = observed), so obs_rows DEVICE int32 [B][2] replaces the [B,H,W,2] mask tensor.  mask_bhwc: NULL, or fp32 [B,H,W,2]
 * receiving the channel-last mask the module logs / scores with.  Bit-identical to mcedm_mcedm_prep on the expanded mask. */
MCEDM_API int mcedm_mcedm_prep_rows(const float* h, const float* u, const int* obs_rows, const float* randn, float h_sub,
                                    float h_div, float u_sub, float u_div, int B, int H, int W, float* x, float* cond,
                                    float* mask_c, float* mask_bhwc, void* stream);
/* channels [c_dst0, c_dst0+Ca+Cb) of a 64-channel bf16 NHWC tensor <- cat(a, b) (NCHW fp32; b may be NULL, Cb = 0) */
MCEDM_API int mcedm_nchw_to_nhwc_pad(const float* a, int Ca, const float* b, int Cb, int B, int H, int W,
                                     void* dst_bf16, int c_dst0, void* stream);
/* partial[cta][64] = column sums over the CTA's pixel range of channels [c_off, c_off+64) of bf16 [pixels, C] */
MCEDM_API int mcedm_colsum_bf16(const void* x_bf16, long long pixels, int C, int c_off, float* partial, int n_ctas,
                                void* stream);
/* The two helpers above for either 16-bit format (op_fmt 0 bf16, 1 fp16); the pad variant multiplies by `scale` first
 * (the loss scale of the fp16 training plan: dL/dF enters the backward as scale * dL/dF). */
MCEDM_API int mcedm_nchw_to_nhwc_pad16(const float* a, int Ca, const float* b, int Cb, int B, int H, int W, void* dst16,
                                       int c_dst0, float scale, int op_fmt, void* stream);
MCEDM_API int mcedm_colsum16(const void* x16, long long pixels, int C, int c_off, float* partial, int n_ctas, int op_fmt,
                             void* stream);
/* The pad variant under dynamic loss scaling: the scale is read from device memory (*scale, so a graph replay uses the
 * current one) and op_fmt must be MCEDM_FMT_F16_INF (scale * dL/dF beyond fp16's range becomes inf). */
MCEDM_API int mcedm_nchw_to_nhwc_pad16_scaled(const float* a, int Ca, const float* b, int Cb, int B, int H, int W,
                                              void* dst16, int c_dst0, const float* scale, int op_fmt, void* stream);
/* g <- g * (1 / *scale): the loss scale comes off the fp32 flat gradient (exact for power-of-two scales). */
MCEDM_API int mcedm_grad_unscale(float* g, long long n, const float* scale, void* stream);
/* backward of mcedm_emb_mlp: dss fp32 [n_aff][B][128] = gradient of every block's (scale | shift);
 * vec_scratch fp32 [B][320]; outputs in the reference parameter shapes (affine [n_aff][128][64] / [n_aff][128],
 * map_layer1, map_layer0 [64][64] / [64]) */
MCEDM_API int mcedm_emb_mlp_bwd(const float* c_noise, const float* freqs, const float* w0, const float* b0,
                                const float* w1, const float* b1, const float* aff_w, const float* dss, int n_aff, int B,
                                float* vec_scratch, float* d_aff_w, float* d_aff_b, float* d_w1, float* d_b1,
                                float* d_w0, float* d_b0, void* stream);
/* partial[i] = sum of squares of the i-th grid-stride slice of g (fp64); n_partial CTAs */
MCEDM_API int mcedm_sumsq_partial(const float* g, long long n, double* partial, int n_partial, void* stream);
/* torch.optim.Adam step on flat fp32 buffers (mcedm.py:141) with gradient-norm clipping folded in
 * (trainer_ddim.yaml:8-9: coef = min(1, max_norm / (grad_scale*||g|| + 1e-6)); norm_partial NULL = no clipping);
 * grad_scale multiplies g first (1/world_size after a sum all-reduce); norm_out NULL or receives the norm. */
MCEDM_API int mcedm_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                              float beta2, float eps, float weight_decay, int step, const double* norm_partial,
                              int n_partial, float max_norm, float grad_scale, float* norm_out, void* stream);
/* ema = ema*beta + (1-beta)*p   (ddim_blocks.py:48-56) */
MCEDM_API int mcedm_ema_update(float* ema, const float* p, long long n, float beta, void* stream);
/* mcedm_adam_step under dynamic loss scaling.  norm_partial (mcedm_sumsq_partial of g) is required; clipping runs iff
 * max_norm > 0.  A non-finite sum of squares sets *found_inf = 1 (else 0) and the step writes nothing to p, m, v.  The
 * bias corrections use step = *step_count + 1 (the applied-step count, in device memory; mcedm_loss_scale_update
 * advances it).  No host synchronisation. */
MCEDM_API int mcedm_adam_step_dyn(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                                  float beta2, float eps, float weight_decay, const int* step_count,
                                  const double* norm_partial, int n_partial, float max_norm, float grad_scale,
                                  float* norm_out, float* found_inf, void* stream);
/* torch._amp_update_scale_ on device words: found_inf != 0 -> scale *= backoff, tracker = 0; else tracker + 1 reaching
 * growth_interval -> scale *= growth (kept if finite), tracker = 0, otherwise tracker += 1.  When the step applied
 * (found_inf == 0) *step_count += 1 (step_count may be NULL).  One thread. */
MCEDM_API int mcedm_loss_scale_update(float* scale, int* growth_tracker, const float* found_inf, int* step_count,
                                      float growth_factor, float backoff_factor, int growth_interval, void* stream);
/* All packed operand copies of the parameters in one launch (replaces the per-tensor permute / flip / cast passes of
 * the weight re-pack after every optimizer step; adm_blocks.py:58 casts the weights per call in the reference).
 * dst16[i] = round16(base[idx_a[i]]) for i < n16 (fmt 0 bf16, 1 fp16; idx -1 = zero padding);
 * dst32[j] = base[idx_a[n16+j]] (+ base[idx_b[j]] when idx_b[j] >= 0) for j < n32. */
MCEDM_API int mcedm_pack_gather(const float* base, const long long* idx_a, const long long* idx_b, long long n16,
                                long long n32, int fmt, void* dst16, float* dst32, void* stream);

/* DDIM sampler with known-region replacement and repeats — PlDdim.sample_with_repeat (models/ddim.py:808-913).
 * fp32 state [total] elements, known_mask == 1 where the ground truth hu is imposed; bit-identical to the torch
 * expressions.  Scalars are the fp32 values of sqrt(a_t), sqrt(1 - a_t), sqrt(a_next), c1, c2 the reference forms
 * (:866-867, :885-891).
 *   mcedm_ddim_init: x = (hu*sqrt_a + noise*sqrt_1ma)*mask + noise*(1 - mask)                          (:842-843)
 *   mcedm_ddim_x0:   x0 = (xt - et*sqrt_1ma)/sqrt_a; x0 = hu*mask + x0*(1 - mask); xt_out (NULL: skip) =
 *                    sqrt_a*x0 + sqrt_1ma*et, the re-noised input of the next repeat                  (:876-883)
 *   mcedm_ddim_next: xt' = sqrt_a_next*x0 [+ c1*rand] + c2*et; x_next = (sqrt_a_next*hu + c2*noise)*mask + xt'*(1 - mask)
 *                    (rand_or_null NULL for eta == 0)                                                 (:885-895) */
MCEDM_API int mcedm_ddim_init(const float* hu, const float* noise, const float* known_mask, float sqrt_a, float sqrt_1ma,
                              long long total, float* x, void* stream);
MCEDM_API int mcedm_ddim_x0(const float* xt, const float* et, const float* hu, const float* known_mask, float sqrt_a,
                            float sqrt_1ma, long long total, float* x0_out, float* xt_out, void* stream);
MCEDM_API int mcedm_ddim_next(const float* x0, const float* et, const float* hu, const float* noise,
                              const float* known_mask, const float* rand_or_null, float sqrt_a_next, float c1, float c2,
                              long long total, float* x_next, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K7  DDPM U-Net pieces (models/ddim_blocks.py:222-470 `Model`; its convolutions and attention run   */
/*     on the K1f / K3 kernels above)                                                               */
/* -------------------------------------------------------------------------------------------- */
/* Per-(sample, channel) statistics of a raw 16-bit activation [B][positions_per_img][64] (dense NHWC: H*W positions;
 * padded-flat: block positions, whose stored zeros add nothing): partial fp32 [B][n_split][64][2] = (sum, sum of squares)
 * over the n_split position ranges of each image.  Replaces the statistics half of Normalize (ddim_blocks.py:60-61,
 * GroupNorm(32, eps 1e-6): 2 channels per group at 64 channels — finer than the conv epilogues' 4-channel records). */
MCEDM_API int mcedm_gn_stats16(const void* x16, long long positions_per_img, int B, int op_fmt, int n_split,
                               float* partial, void* stream);
/* coef_out fp32 [B][128] = (a | b) of y = act(a*x + b) == act(GroupNorm(x + shift)) for groups of channels_per_group
 * consecutive channels of this 64-channel tensor (gamma / beta fp32 [64]: the tensor's slice of a wider norm),
 * pixels_per_img = H*W data positions.  shift NULL, or fp32 [B or 1][64] (shift_batch_stride 64 or 0): the per-sample
 * temb_proj(swish(temb)) term ResnetBlock adds between conv1 and norm2 (ddim_blocks.py:140-146), folded into the
 * statistics and into b so that x + shift is never materialised. */
MCEDM_API int mcedm_gn_coef_groups(const float* partial, int n_split, long long pixels_per_img, const float* gamma,
                                   const float* beta, int channels_per_group, float eps, const float* shift,
                                   int shift_batch_stride, int B, float* coef_out, void* stream);
/* out16[b, i, j, :] = src16[b, 2i+1, 2j+1, :] (64 channels, 16-bit), each side dense NHWC (pitch 0) or padded-flat:
 * the sampling half of Downsample (ddim_blocks.py:97-101: pad (0,1,0,1) + stride-2 3x3 conv == the stride-1 same conv at
 * the odd positions). */
MCEDM_API int mcedm_decimate16(const void* src16, int in_pitch, int in_blk, int B, int H, int W, void* out16,
                               int out_pitch, int out_blk, void* stream);
/* Timestep embedding (ddim_blocks.py:12-30, :422-425) and every ResnetBlock's temb_proj(swish(temb)) (:140):
 * t fp32 [Bt]; w0 [256][64], w1 [256][256]; w_proj [n_blocks][64][256], b_proj [n_blocks][64];
 * out fp32 [n_blocks][Bt][64]. */
MCEDM_API int mcedm_ddpm_temb(const float* t, int Bt, const float* w0, const float* b0, const float* w1, const float* b1,
                              const float* w_proj, const float* b_proj, int n_blocks, float* out, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* K8  fused validation / test reductions (SURVEY 8f rank 4)                                       */
/* -------------------------------------------------------------------------------------------- */
/* One pass over the sampled fields for PlMcedm.test_step / validation_step (models/mcedm.py:385-408):
 *   mean over n_samples (mcedm.py:385-386), MaskedLoss('l1') on the normalised state and on the inverse-normalised
 *   state (losses.py:62-78, normalizer.py:28-29), restricted to channels [c0, c1) (`loss_dim`).
 * xs fp64 [n_samples][b][pixels][C] (channel-last, n-major as rearrange '(n b) ...'); gt fp32 [b][pixels][C];
 * gt_unnorm_a fp32 [b][pixels][Ca] and gt_unnorm_b fp32 [b][pixels][C-Ca] (h_unnorm, u_unnorm as the datamodule delivers
 * them; both NULL: skip the un-normalised error); mask fp32 [b][pixels][C] (1 = scored); sub / div DEVICE fp64 [C]
 * (Normalizer buffers per channel); clamp01: clamp to [0,1] before the inverse transform (min_max normalisation).
 * mean_out NULL or fp64 [b][pixels][C]; partial_scratch DEVICE fp64 [n_cta][3];
 * out3 DEVICE fp64 [3] = (masked MAE, masked MAE un-normalised, number of scored entries). */
MCEDM_API int mcedm_masked_mae_mean(const double* xs, int n_samples, int b, long long pixels, int C, const float* gt,
                                    const float* gt_unnorm_a, const float* gt_unnorm_b, int Ca, const float* mask, int c0,
                                    int c1, const double* sub, const double* div, int clamp01, double* mean_out,
                                    double* partial_scratch, int n_cta, double* out3, void* stream);
/* Per (sample, channel) of pred fp64 [b][pixels][C] vs target fp32 [b][pixels][C]: Pearson correlation exactly as
 * CorrelationLoss.calculate_correlation (losses.py:101-116: centred sums, zero denominators += 1e-7) into corr_bc fp64
 * [b][C] (NULL: skip; target may then be NULL), and min / max of pred into min_bc / max_bc fp64 [b][C] (NULL: skip) — the
 * reductions of scale_each_min_max (ddim.py:689-698). */
MCEDM_API int mcedm_corr_minmax(const double* pred, const float* target, int b, long long pixels, int C, double* corr_bc,
                                double* min_bc, double* max_bc, void* stream);

/* -------------------------------------------------------------------------------------------- */
/* bring-up instrumentation of the product kernels (the checker / probe kernels live in their own   */
/* library: include/mcedm_b200_check.h, libmcedm_b200_check.so)                                     */
/* -------------------------------------------------------------------------------------------- */
/* Saturation audit of the fp16 activation storage: with MCEDM_DBG=4 in the environment the fused 16-bit convolution
 * epilogues (conv_rows_fused N=64, conv_flat_fused fast paths) count every accumulator / output value whose magnitude
 * exceeds 65504 (clamped by the saturating conversion) or is NaN; *host_out receives the count since the last reset. */
MCEDM_API int mcedm_saturation_count(long long* host_out, int reset, void* stream);
/* bring-up: per-CTA cycles spent in each role's barrier waits by the last fused conv_rows launch run with MCEDM_DBG=32
 * (HOST int64 [160][8]: h_empty, acc_empty, h_ready, acc_full, h_full waits; epilogue, MMA, producer role totals) */
MCEDM_API int mcedm_debug_rows(long long* host_out);

#ifdef __cplusplus
}
#endif
#endif /* MCEDM_B200_H */
