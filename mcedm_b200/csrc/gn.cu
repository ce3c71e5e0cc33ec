// K2 — GroupNorm statistics and fused GroupNorm-apply + adaptive scale/shift + SiLU + resample.
//
// Replaces, per UNetBlock (models/adm_blocks.py:159-181):
//   silu(norm0(x))                                   :161  (+ the up/down resample conv0 performs
//                                                          before its 3x3 filter, :73-77)
//   silu(addcmul(shift, norm1(x), scale + 1))        :163-166
//   norm2(x)                                         :175
// and silu(out_norm(x)) (:403).  GroupNorm itself is models/adm_blocks.py:86-97: groups of 4
// consecutive channels, biased variance over 4*H*W values, eps 1e-5, per-channel affine.
//
// All kernels are HBM-bound streaming kernels (fp32 in -> bf16 out, 6 B per element): 128-bit
// loads/stores, one pass.  Statistics arrive as per-128-pixel-tile partial sums (sum, sum of
// squares per group) that the conv epilogue already produced (conv_igemm.cu); they are folded in
// fp64 in a fixed order here, so results are run-to-run deterministic.
#include "philox.cuh"
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

namespace mcedm {

// ---------------------------------------------------------------------------------------------
// stand-alone partial statistics (used for tensors not produced by conv_igemm, and by tests)
// x: fp32 [n_tiles*128, 64]; out: [n_tiles][16][2]
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gn_stats_kernel(const float* __restrict__ x, float* __restrict__ out) {
  const long long tile = blockIdx.x;
  const int unit = threadIdx.x & 15;      // 4-channel group
  const int r0 = threadIdx.x >> 4;        // 0..15
  const float4* xp = reinterpret_cast<const float4*>(x + tile * 128 * 64);
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float4 a = xp[(r0 + 16 * i) * 16 + unit];
    s1 += (a.x + a.y) + (a.z + a.w);
    s2 += (a.x * a.x + a.y * a.y) + (a.z * a.z + a.w * a.w);
  }
  // lanes l and l^16 of a warp share `unit`
  s1 += __shfl_xor_sync(0xffffffffu, s1, 16);
  s2 += __shfl_xor_sync(0xffffffffu, s2, 16);
  __shared__ float sm[8][16][2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane < 16) {
    sm[warp][lane][0] = s1;
    sm[warp][lane][1] = s2;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    const int g = threadIdx.x >> 1, k = threadIdx.x & 1;
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += sm[w][g][k];
    out[tile * 32 + threadIdx.x] = t;
  }
}

// ---------------------------------------------------------------------------------------------
// apply
// ---------------------------------------------------------------------------------------------
struct GnApplyParams {
  const float* x;            // fp32 NHWC [B, Hin, Win, 64]
  const float* partial;      // [B*tiles_per_img][16][2]
  int tiles_per_img;         // partial-sum records per image (Hin*Win/128, or 4x that from conv_rows)
  const float* gamma;        // [64]
  const float* beta;         // [64]
  const float* scale_shift;  // nullptr or [Bemb][2*C_emb]: scale at +c, shift at +C_emb+c
  int emb_batch_stride;      // 0 when one embedding row is broadcast over the batch
  int emb_shift_offset;      // distance (floats) from scale[c] to shift[c]
  float eps;
  int act;                   // 0 identity, 1 SiLU
  int resample;              // 0 same, 1 nearest x2 up (out is 2Hin x 2Win), 2 2x2 mean (out is Hin/2 x Win/2)
  int Hin, Win;
  void* out;                 // bf16 NHWC at the output resolution
  void* out_raw;             // nullptr or bf16 NHWC copy of x itself (same resolution only)
  int pix_per_cta;           // INPUT pixels per CTA for resample 0/1, OUTPUT pixels per CTA for resample 2
  float* meanrstd_out;       // nullptr or [B][16][2] receiving (mean, rstd) per group (saved for the backward)
  int fmt;                   // output operand format: 0 bf16, 1 fp16
  float* coef;               // [B][128]: per-channel (a | b) with y = act(a*x + b); written by gn_finalize_kernel
  int out_pitch;             // 0: dense NHWC output; > 0: padded flat layout of conv_flat.cu (row pitch)
  int out_blk;               // positions per image block of the padded layout
  void* out_lo;              // nullptr, or (fp32-accuracy mode) receives operand - float(rounded operand), same layout as out
  void* out_raw_lo;          // likewise for the raw copy
  int x16;                   // x is a 16-bit NHWC tensor in the operand format (inference: raw activations are 16-bit)
  int in_pitch, in_blk;      // x16 only: x itself is in the padded flat layout (0: dense)
  int fast_act;              // fp32 input: SiLU through MUFU.TANH as well (training forward: the operand is bf16 anyway)
};

// pixel index of output (b, y, x) in the dense NHWC layout or in the padded flat layout
__device__ __forceinline__ long long gn_out_index(const GnApplyParams& p, int b, int y, int x, int Ho, int Wo) {
  if (p.out_pitch > 0) return (long long)b * p.out_blk + (long long)(y + 1) * p.out_pitch + x;
  return ((long long)b * Ho + y) * Wo + x;
}

// FAST (the 16-bit inference instantiation): SiLU through one MUFU.TANH instead of ex2 + rcp, as in the fused convs
template <bool FAST = false>
__device__ __forceinline__ float4 gn_act4(float4 v, const float4 a, const float4 b, int act, bool fast = false) {
  v.x = fmaf(v.x, a.x, b.x);
  v.y = fmaf(v.y, a.y, b.y);
  v.z = fmaf(v.z, a.z, b.z);
  v.w = fmaf(v.w, a.w, b.w);
  if (act) {
    if (FAST || fast) {
      v.x = silu_from_half_arg(0.5f * v.x);
      v.y = silu_from_half_arg(0.5f * v.y);
      v.z = silu_from_half_arg(0.5f * v.z);
      v.w = silu_from_half_arg(0.5f * v.w);
    } else {
      v.x = silu_f(v.x);
      v.y = silu_f(v.y);
      v.z = silu_f(v.z);
      v.w = silu_f(v.w);
    }
  }
  return v;
}
__device__ __forceinline__ uint4 pack8(const float4 lo, const float4 hi, int fmt) {
  uint4 o;
  o.x = pack_op2(lo.x, lo.y, fmt);
  o.y = pack_op2(lo.z, lo.w, fmt);
  o.z = pack_op2(hi.x, hi.y, fmt);
  o.w = pack_op2(hi.z, hi.w, fmt);
  return o;
}
template <bool INF>
__device__ __forceinline__ uint4 pack8_g(const float4 lo, const float4 hi, int fmt) {
  uint4 o;
  o.x = pack_op2_g<INF>(lo.x, lo.y, fmt);
  o.y = pack_op2_g<INF>(lo.z, lo.w, fmt);
  o.z = pack_op2_g<INF>(hi.x, hi.y, fmt);
  o.w = pack_op2_g<INF>(hi.z, hi.w, fmt);
  return o;
}

// second term of the split operand: what the 16-bit rounding of (lo, hi) dropped (fp32-accuracy mode, fp16 only)
__device__ __forceinline__ uint4 pack8_rem(const float4 lo, const float4 hi, const uint4 r) {
  const float2 a = unpack_f16x2(r.x), b = unpack_f16x2(r.y), c = unpack_f16x2(r.z), d = unpack_f16x2(r.w);
  uint4 o;
  o.x = pack_f16x2(lo.x - a.x, lo.y - a.y);
  o.y = pack_f16x2(lo.z - b.x, lo.w - b.y);
  o.z = pack_f16x2(hi.x - c.x, hi.y - c.y);
  o.w = pack_f16x2(hi.z - d.x, hi.w - d.y);
  return o;
}

// grid = B: folds the partial-sum records of image b (fixed order, fp64) into per-channel coefficients.
// Done once per GroupNorm instead of once per streaming CTA, so the apply pass below is a pure stream.
__global__ void __launch_bounds__(256) gn_finalize_kernel(const GnApplyParams p) {
  pdl_wait();
  pdl_trigger();
  __shared__ float sMean[16], sRstd[16];
  const int b = blockIdx.x;
  // the affine parameters do not depend on the fold: requested first, so their latency overlaps the records'
  float pg = 0.f, pb = 0.f, psc = 0.f, psh = 0.f;
  if (threadIdx.x < 64) {
    pg = __ldg(p.gamma + threadIdx.x);
    pb = __ldg(p.beta + threadIdx.x);
    if (p.scale_shift) {
      const float* ss = p.scale_shift + (long long)b * p.emb_batch_stride;
      psc = ss[threadIdx.x];
      psh = ss[p.emb_shift_offset + threadIdx.x];
    }
  }
  {
    // fold the partial-sum records of image b: 16 threads per group, fixed order, fp64.
    // Loads are issued 8 at a time before any add so the L2 latency is paid once per batch, not per record.
    const int g = threadIdx.x >> 4, j = threadIdx.x & 15;
    double s1 = 0.0, s2 = 0.0;
    const float2* pp = reinterpret_cast<const float2*>(p.partial + (long long)b * p.tiles_per_img * 32 + g * 2);
    int t = j;
    for (; t + 7 * 16 < p.tiles_per_img; t += 8 * 16) {
      float2 v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = pp[(t + k * 16) * 16];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        s1 += (double)v[k].x;
        s2 += (double)v[k].y;
      }
    }
    for (; t < p.tiles_per_img; t += 16) {
      const float2 v = pp[t * 16];
      s1 += (double)v.x;
      s2 += (double)v.y;
    }
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, off);
      s2 += __shfl_xor_sync(0xffffffffu, s2, off);
    }
    if (j == 0) {
      const double cnt = 4.0 * (double)p.Hin * (double)p.Win;
      const double mean = s1 / cnt;
      double var = s2 / cnt - mean * mean;
      if (var < 0.0) var = 0.0;
      sMean[g] = (float)mean;
      sRstd[g] = (float)(1.0 / sqrt(var + (double)p.eps));
    }
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int c = threadIdx.x;
    float a = sRstd[c >> 2] * pg;
    float bb = pb - sMean[c >> 2] * a;
    if (p.scale_shift) {
      const float sc = 1.0f + psc;
      a *= sc;
      bb = fmaf(bb, sc, psh);
    }
    p.coef[(long long)b * 128 + c] = a;
    p.coef[(long long)b * 128 + 64 + c] = bb;
  } else if (threadIdx.x < 80 && p.meanrstd_out) {
    const int g = threadIdx.x - 64;
    *reinterpret_cast<float2*>(p.meanrstd_out + ((long long)b * 16 + g) * 2) = make_float2(sMean[g], sRstd[g]);
  }
}

// 8 consecutive channels of input pixel `pix` (dense index inside the whole tensor) as two float4
template <bool X16>
__device__ __forceinline__ void gn_load8(const GnApplyParams& p, long long pix, int c8, float4& lo, float4& hi) {
  if constexpr (X16) {
    const uint4 v = reinterpret_cast<const uint4*>(p.x)[pix * 8 + c8];
    if (p.fmt) {
      const float2 a = unpack_f16x2(v.x), b = unpack_f16x2(v.y), c = unpack_f16x2(v.z), d = unpack_f16x2(v.w);
      lo = make_float4(a.x, a.y, b.x, b.y);
      hi = make_float4(c.x, c.y, d.x, d.y);
    } else {
      lo = make_float4(bf16_lo(v.x), bf16_hi(v.x), bf16_lo(v.y), bf16_hi(v.y));
      hi = make_float4(bf16_lo(v.z), bf16_hi(v.z), bf16_lo(v.w), bf16_hi(v.w));
    }
  } else {
    const float4* xp = reinterpret_cast<const float4*>(p.x + pix * 64 + c8 * 8);
    lo = xp[0];
    hi = xp[1];
  }
}
// dense pixel index (b, y, x) of the INPUT tensor, or its padded-flat position when the 16-bit input is flat
__device__ __forceinline__ long long gn_in_index(const GnApplyParams& p, int b, int ip) {
  if (p.in_pitch > 0) {
    const int y = ip / p.Win;
    return (long long)b * p.in_blk + (long long)(y + 1) * p.in_pitch + (ip - y * p.Win);
  }
  return (long long)b * p.Hin * p.Win + ip;
}

// dropout of the training forward (gn_apply_dropout_kernel; mask definition in philox.cuh)
struct GnDropout {
  uint32_t thr;              // keep iff mask word >= thr
  float scale;               // 1 / (1 - p), rounded to fp32 on the host
  int layer;                 // the block's layer id (aff_index)
  const uint32_t* rng;       // device {seed_lo, seed_hi, step}
};

// DROP: resample 0 and SiLU only; SiLU in the exact form (not the MUFU.TANH one of the 16-bit inference instantiation),
// operand = fp16(silu(a*x + b) * s) where kept, 0 elsewhere.  DROP = false compiles to the kernel without dropout.
template <bool X16, bool DROP>
__device__ __forceinline__ void gn_apply_body(const GnApplyParams& p, const GnDropout& d) {
  pdl_wait();
  pdl_trigger();
  const int b = blockIdx.y;
  const int c8 = threadIdx.x & 7;          // 8-channel slice
  const int ps = threadIdx.x >> 3;         // 0..31
  const float4* cf = reinterpret_cast<const float4*>(p.coef + (long long)b * 128 + c8 * 8);
  const float4 a_lo = __ldg(cf), a_hi = __ldg(cf + 1), b_lo = __ldg(cf + 16), b_hi = __ldg(cf + 17);
  const long long in_img = (long long)b * p.Hin * p.Win;
  const int pix0 = blockIdx.x * p.pix_per_cta;
  uint4* out = reinterpret_cast<uint4*>(p.out);

  if (DROP || p.resample == 0) {
    // 4 pixels (8 x 128-bit loads) in flight per thread before any dependent work
    for (int i = ps; i < p.pix_per_cta; i += 128) {
      float4 lo[4], hi[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (i + 32 * k < p.pix_per_cta) gn_load8<X16>(p, gn_in_index(p, b, pix0 + i + 32 * k), c8, lo[k], hi[k]);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (i + 32 * k < p.pix_per_cta) {
          const int ip = pix0 + i + 32 * k;
          const long long pix = in_img + ip;
          if (p.out_raw) {
            const uint4 rw = pack8(lo[k], hi[k], p.fmt);
            reinterpret_cast<uint4*>(p.out_raw)[pix * 8 + c8] = rw;
            if (p.out_raw_lo) reinterpret_cast<uint4*>(p.out_raw_lo)[pix * 8 + c8] = pack8_rem(lo[k], hi[k], rw);
          }
          long long opix = pix;
          if (p.out_pitch > 0) {
            const int y = ip / p.Win;
            opix = gn_out_index(p, b, y, ip - y * p.Win, p.Hin, p.Win);
          }
          float4 yl = gn_act4<X16 && !DROP>(lo[k], a_lo, b_lo, p.act, p.fast_act),
                 yh = gn_act4<X16 && !DROP>(hi[k], a_hi, b_hi, p.act, p.fast_act);
          if constexpr (DROP) {
            // logical NHWC index of channel 8*c8 is pix*64 + 8*c8: Philox counters pix*16 + 2*c8 and the next one
            const unsigned long long q = (unsigned long long)pix * 16ull + 2ull * (unsigned)c8;
            yl = dropout_apply4(yl, dropout_words(q, d.layer, d.rng), d.thr, d.scale);
            yh = dropout_apply4(yh, dropout_words(q + 1, d.layer, d.rng), d.thr, d.scale);
          }
          const uint4 yo = pack8(yl, yh, p.fmt);
          out[opix * 8 + c8] = yo;
          if (p.out_lo) reinterpret_cast<uint4*>(p.out_lo)[opix * 8 + c8] = pack8_rem(yl, yh, yo);
        }
      }
    }
  } else if (p.resample == 1) {
    const int Wo = p.Win * 2, Ho = p.Hin * 2;
    const long long rstride = p.out_pitch > 0 ? p.out_pitch : Wo;
    for (int i = ps; i < p.pix_per_cta; i += 32) {
      const int ip = pix0 + i;
      const int y = ip / p.Win, x = ip - y * p.Win;
      float4 xl, xh;
      gn_load8<X16>(p, gn_in_index(p, b, ip), c8, xl, xh);
      const float4 yl = gn_act4<X16>(xl, a_lo, b_lo, p.act, p.fast_act), yh = gn_act4<X16>(xh, a_hi, b_hi, p.act, p.fast_act);
      const uint4 v = pack8(yl, yh, p.fmt);
      const long long o00 = gn_out_index(p, b, 2 * y, 2 * x, Ho, Wo);
      out[o00 * 8 + c8] = v;
      out[(o00 + 1) * 8 + c8] = v;
      out[(o00 + rstride) * 8 + c8] = v;
      out[(o00 + rstride + 1) * 8 + c8] = v;
      if (p.out_lo) {
        uint4* ol = reinterpret_cast<uint4*>(p.out_lo);
        const uint4 r = pack8_rem(yl, yh, v);
        ol[o00 * 8 + c8] = r;
        ol[(o00 + 1) * 8 + c8] = r;
        ol[(o00 + rstride) * 8 + c8] = r;
        ol[(o00 + rstride + 1) * 8 + c8] = r;
      }
      if (X16 && p.out_raw) {   // nearest-x2 copy of the RAW input: the skip path of an up block (adm_blocks.py:149-151)
        uint4* orw = reinterpret_cast<uint4*>(p.out_raw);
        const uint4 r = pack8(xl, xh, p.fmt);
        orw[o00 * 8 + c8] = r;
        orw[(o00 + 1) * 8 + c8] = r;
        orw[(o00 + rstride) * 8 + c8] = r;
        orw[(o00 + rstride + 1) * 8 + c8] = r;
      }
    }
  } else {
    const int Wo = p.Win >> 1, Ho = p.Hin >> 1;
    // two output pixels (8 loads) in flight per thread before any dependent work
    for (int i = ps; i < p.pix_per_cta; i += 64) {
      float4 xl[2][4], xh[2][4];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int op = pix0 + i + 32 * u;
        const int y = op / Wo, x = op - y * Wo;
        if (i + 32 * u < p.pix_per_cta) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            gn_load8<X16>(p, gn_in_index(p, b, (2 * y + (k >> 1)) * p.Win + 2 * x + (k & 1)), c8, xl[u][k], xh[u][k]);
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (i + 32 * u < p.pix_per_cta) {
          const int op = pix0 + i + 32 * u;
          const int y = op / Wo, x = op - y * Wo;
          float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float4 l = gn_act4<X16>(xl[u][k], a_lo, b_lo, p.act, p.fast_act), h = gn_act4<X16>(xh[u][k], a_hi, b_hi, p.act, p.fast_act);
            lo.x += l.x; lo.y += l.y; lo.z += l.z; lo.w += l.w;
            hi.x += h.x; hi.y += h.y; hi.z += h.z; hi.w += h.w;
          }
          lo.x *= 0.25f; lo.y *= 0.25f; lo.z *= 0.25f; lo.w *= 0.25f;
          hi.x *= 0.25f; hi.y *= 0.25f; hi.z *= 0.25f; hi.w *= 0.25f;
          const uint4 yo = pack8(lo, hi, p.fmt);
          const long long oi = gn_out_index(p, b, y, x, Ho, Wo);
          out[oi * 8 + c8] = yo;
          if (p.out_raw) {
            // 2x2 mean of the RAW input in the same layout: the residual of a down block's conv1 (Conv2d with
            // kernel=0, down=True on the skip path, adm_blocks.py:149-151), read there like a same-resolution residual
            const float4* r = xl[u];
            const float4* s = xh[u];
            const float4 rl = make_float4(0.25f * ((r[0].x + r[1].x) + (r[2].x + r[3].x)), 0.25f * ((r[0].y + r[1].y) + (r[2].y + r[3].y)),
                                          0.25f * ((r[0].z + r[1].z) + (r[2].z + r[3].z)), 0.25f * ((r[0].w + r[1].w) + (r[2].w + r[3].w)));
            const float4 rh = make_float4(0.25f * ((s[0].x + s[1].x) + (s[2].x + s[3].x)), 0.25f * ((s[0].y + s[1].y) + (s[2].y + s[3].y)),
                                          0.25f * ((s[0].z + s[1].z) + (s[2].z + s[3].z)), 0.25f * ((s[0].w + s[1].w) + (s[2].w + s[3].w)));
            reinterpret_cast<uint4*>(p.out_raw)[oi * 8 + c8] = pack8(rl, rh, p.fmt);
          }
          if (p.out_lo) reinterpret_cast<uint4*>(p.out_lo)[oi * 8 + c8] = pack8_rem(lo, hi, yo);
        }
      }
    }
  }
}

template <bool X16>
__global__ void __launch_bounds__(256) gn_apply_kernel(const GnApplyParams p) {
  gn_apply_body<X16, false>(p, GnDropout{});
}

struct GnApplyDropParams {
  GnApplyParams g;
  GnDropout d;
};
__global__ void __launch_bounds__(256) gn_apply_dropout_kernel(const GnApplyDropParams p) {
  gn_apply_body<true, true>(p.g, p.d);
}

// in-place g = fp16(g * keep * s) on a 16-bit [B, H, W, 64] tensor (dense, or padded-flat with row pitch `pitch` and
// `blk` positions per image); one thread per (pixel, 8-channel chunk), padding positions are never touched.
// INF: fp16 stores without saturation (op_fmt MCEDM_FMT_F16_INF, dynamic loss scaling)
template <bool INF = false>
__global__ void __launch_bounds__(256) dropout_bwd16_kernel(void* __restrict__ g, int pitch, int blk, int B, int H, int W,
                                                            GnDropout d, int fmt) {
  pdl_wait();
  pdl_trigger();
  const long long hw = (long long)H * W;
  const long long n_chunks = (long long)B * hw * 8;
  uint4* gp = reinterpret_cast<uint4*>(g);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_chunks; i += (long long)gridDim.x * blockDim.x) {
    const long long pix = i >> 3;
    const int c8 = (int)(i & 7);
    long long spix = pix;
    if (pitch > 0) {
      const long long b = pix / hw;
      const int ip = (int)(pix - b * hw);
      const int y = ip / W;
      spix = b * blk + (long long)(y + 1) * pitch + (ip - y * W);
    }
    const uint4 v = gp[spix * 8 + c8];
    float4 lo, hi;
    if (fmt) {
      const float2 a = unpack_f16x2(v.x), b = unpack_f16x2(v.y), c = unpack_f16x2(v.z), e = unpack_f16x2(v.w);
      lo = make_float4(a.x, a.y, b.x, b.y);
      hi = make_float4(c.x, c.y, e.x, e.y);
    } else {
      lo = make_float4(bf16_lo(v.x), bf16_hi(v.x), bf16_lo(v.y), bf16_hi(v.y));
      hi = make_float4(bf16_lo(v.z), bf16_hi(v.z), bf16_lo(v.w), bf16_hi(v.w));
    }
    const unsigned long long q = (unsigned long long)pix * 16ull + 2ull * (unsigned)c8;
    lo = dropout_apply4(lo, dropout_words(q, d.layer, d.rng), d.thr, d.scale);
    hi = dropout_apply4(hi, dropout_words(q + 1, d.layer, d.rng), d.thr, d.scale);
    gp[spix * 8 + c8] = pack8_g<INF>(lo, hi, fmt);
  }
}

// CTAs of <= 512 work pixels; keep >= ~4 CTAs per SM when the batch allows it (0: `work` cannot be tiled)
static int gn_apply16_pix_per_cta(int work, int B) {
  int per = 512;
  while (per > 32 && ((work % per) != 0 || (long long)(work / per) * B < 4LL * num_sms())) per >>= 1;
  if (per < 32) per = 32;
  while (per > 32 && (work % per) != 0) per >>= 1;
  return work % per == 0 ? per : 0;
}

}  // namespace mcedm

extern "C" int mcedm_gn_stats(const float* x, long long n_pixels, float* partial, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n_pixels > 0 && n_pixels % 128 == 0, "gn_stats: pixel count %lld must be a multiple of 128", n_pixels);
  gn_stats_kernel<<<(unsigned)(n_pixels / 128), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, partial);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

static int gn_apply_impl(const float* x, const float* partial, const float* gamma, const float* beta,
                         const float* scale_shift, int emb_batch_stride, int emb_shift_offset, float eps,
                         int act, int resample, int B, int Hin, int Win, int parts_per_img, int out_pitch,
                         int out_blk, void* out_bf16, void* out_raw_bf16, float* meanrstd_out, float* coef_scratch,
                         int op_fmt, void* out_lo, void* out_raw_lo, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && (Hin * Win) % 128 == 0, "gn_apply: Hin*Win=%d must be a multiple of 128", Hin * Win);
  MCEDM_REQUIRE(resample >= 0 && resample <= 2, "gn_apply: resample=%d", resample);
  MCEDM_REQUIRE(resample == 0 || out_raw_bf16 == nullptr, "gn_apply: raw copy only without resampling");
  MCEDM_REQUIRE(resample != 2 || (Hin % 2 == 0 && Win % 2 == 0), "gn_apply: 2x2 mean needs even H, W");
  GnApplyParams p;
  p.x = x;
  p.partial = partial;
  p.tiles_per_img = parts_per_img > 0 ? parts_per_img : Hin * Win / 128;
  p.gamma = gamma;
  p.beta = beta;
  p.scale_shift = scale_shift;
  p.emb_batch_stride = emb_batch_stride;
  p.emb_shift_offset = emb_shift_offset;
  p.eps = eps;
  p.act = act;
  p.resample = resample;
  p.Hin = Hin;
  p.Win = Win;
  p.out = out_bf16;
  p.out_raw = out_raw_bf16;
  p.out_pitch = out_pitch;
  p.out_blk = out_blk;
  p.meanrstd_out = meanrstd_out;
  p.coef = coef_scratch;
  p.fmt = op_fmt ? 1 : 0;
  p.x16 = 0;
  p.in_pitch = 0;
  p.in_blk = 0;
  p.out_lo = out_lo;
  p.out_raw_lo = out_raw_lo;
  // training forward (it saves mean / rstd for the backward): the operand is rounded to bf16 (2^-9) anyway, so SiLU may
  // take the one-MUFU tanh form (2^-11) of the inference kernels; the fp32-accuracy and fallback inference plans keep
  // the exact form
  p.fast_act = (meanrstd_out != nullptr && out_lo == nullptr) ? 1 : 0;
  MCEDM_REQUIRE(coef_scratch != nullptr, "gn_apply: coef_scratch (fp32 [B][128]) is required");
  const int work = (resample == 2) ? (Hin * Win / 4) : (Hin * Win);  // pixels iterated per image
  // streaming CTAs of <= 512 pixels (~200 KB of traffic each); keep >= ~4 CTAs per SM when the batch allows it
  int per = 512;
  while (per > 32 && ((work % per) != 0 || (long long)(work / per) * B < 4LL * num_sms())) per >>= 1;
  if (per < 32) per = 32;
  while (per > 32 && (work % per) != 0) per >>= 1;
  MCEDM_REQUIRE(work % per == 0, "gn_apply: cannot tile %d pixels", work);
  p.pix_per_cta = per;
  dim3 grid(work / per, B);
  MCEDM_CUDA(launch_pdl(gn_finalize_kernel, dim3(B), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), p));
  MCEDM_CUDA(launch_pdl(gn_apply_kernel<false>, grid, dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), p));
  return 0;
}

extern "C" int mcedm_gn_apply(const float* x, const float* partial, const float* gamma, const float* beta,
                              const float* scale_shift, int emb_batch_stride, int emb_shift_offset, float eps,
                              int act, int resample, int B, int Hin, int Win, int parts_per_img, int out_pitch,
                              int out_blk, void* out_bf16, void* out_raw_bf16, float* meanrstd_out, float* coef_scratch,
                              int op_fmt, void* stream) {
  return gn_apply_impl(x, partial, gamma, beta, scale_shift, emb_batch_stride, emb_shift_offset, eps, act, resample, B, Hin,
                       Win, parts_per_img, out_pitch, out_blk, out_bf16, out_raw_bf16, meanrstd_out, coef_scratch, op_fmt,
                       nullptr, nullptr, stream);
}

extern "C" int mcedm_gn_apply_split(const float* x, const float* partial, const float* gamma, const float* beta,
                                    const float* scale_shift, int emb_batch_stride, int emb_shift_offset, float eps,
                                    int act, int resample, int B, int Hin, int Win, int parts_per_img, int out_pitch,
                                    int out_blk, void* out_hi, void* out_lo, void* raw_hi, void* raw_lo,
                                    float* coef_scratch, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(out_lo != nullptr && (raw_hi == nullptr) == (raw_lo == nullptr), "gn_apply_split: hi and lo outputs go in pairs");
  return gn_apply_impl(x, partial, gamma, beta, scale_shift, emb_batch_stride, emb_shift_offset, eps, act, resample, B, Hin,
                       Win, parts_per_img, out_pitch, out_blk, out_hi, raw_hi, nullptr, coef_scratch, 1, out_lo, raw_lo,
                       stream);
}

extern "C" int mcedm_gn_coef(const float* partial, int parts_per_img, const float* gamma, const float* beta,
                             const float* scale_shift, int emb_batch_stride, int emb_shift_offset, float eps, int B,
                             int Hin, int Win, float* coef_out, float* meanrstd_out, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && parts_per_img >= 1 && coef_out != nullptr, "gn_coef: bad arguments");
  GnApplyParams p;
  memset(&p, 0, sizeof(p));
  p.partial = partial;
  p.tiles_per_img = parts_per_img;
  p.gamma = gamma;
  p.beta = beta;
  p.scale_shift = scale_shift;
  p.emb_batch_stride = emb_batch_stride;
  p.emb_shift_offset = emb_shift_offset;
  p.eps = eps;
  p.Hin = Hin;
  p.Win = Win;
  p.meanrstd_out = meanrstd_out;
  p.coef = coef_out;
  MCEDM_CUDA(launch_pdl(gn_finalize_kernel, dim3(B), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), p));
  return 0;
}

extern "C" int mcedm_gn_apply16(const void* x16, int in_pitch, int in_blk, const float* coef, int act, int resample,
                                int B, int Hin, int Win, int out_pitch, int out_blk, void* out16, void* out_pooled16,
                                int op_fmt, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && (Hin * Win) % 128 == 0, "gn_apply16: Hin*Win=%d must be a multiple of 128", Hin * Win);
  MCEDM_REQUIRE(resample >= 0 && resample <= 2, "gn_apply16: resample=%d", resample);
  MCEDM_REQUIRE(resample != 2 || (Hin % 2 == 0 && Win % 2 == 0), "gn_apply16: 2x2 mean needs even H, W");
  MCEDM_REQUIRE(coef != nullptr, "gn_apply16: coefficients (mcedm_gn_coef) are required");
  MCEDM_REQUIRE(out_pooled16 == nullptr || resample != 0, "gn_apply16: the raw resampled copy needs resample = 1 or 2");
  GnApplyParams p;
  memset(&p, 0, sizeof(p));
  p.x = reinterpret_cast<const float*>(x16);
  p.out_raw = out_pooled16;
  p.x16 = 1;
  p.in_pitch = in_pitch;
  p.in_blk = in_blk;
  p.act = act;
  p.resample = resample;
  p.Hin = Hin;
  p.Win = Win;
  p.out = out16;
  p.out_pitch = out_pitch;
  p.out_blk = out_blk;
  p.coef = const_cast<float*>(coef);
  p.fmt = op_fmt ? 1 : 0;
  const int work = (resample == 2) ? (Hin * Win / 4) : (Hin * Win);
  const int per = gn_apply16_pix_per_cta(work, B);
  MCEDM_REQUIRE(per > 0, "gn_apply16: cannot tile %d pixels", work);
  p.pix_per_cta = per;
  dim3 grid(work / per, B);
  MCEDM_CUDA(launch_pdl(gn_apply_kernel<true>, grid, dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), p));
  return 0;
}

extern "C" int mcedm_gn_apply16_dropout(const void* x16, int in_pitch, int in_blk, const float* coef, int B, int H, int W,
                                        int out_pitch, int out_blk, void* out16, unsigned int threshold, float scale,
                                        int layer, const unsigned int* rng, int op_fmt, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && (H * W) % 128 == 0, "gn_apply16_dropout: H*W=%d must be a multiple of 128", H * W);
  MCEDM_REQUIRE(coef != nullptr && rng != nullptr && x16 != nullptr && out16 != nullptr,
                "gn_apply16_dropout: input, coefficients, output and the rng words are required");
  MCEDM_REQUIRE(scale >= 1.f && layer >= 0, "gn_apply16_dropout: scale=%g layer=%d", (double)scale, layer);
  GnApplyDropParams p;
  memset(&p, 0, sizeof(p));
  p.g.x = reinterpret_cast<const float*>(x16);
  p.g.x16 = 1;
  p.g.in_pitch = in_pitch;
  p.g.in_blk = in_blk;
  p.g.act = 1;
  p.g.resample = 0;
  p.g.Hin = H;
  p.g.Win = W;
  p.g.out = out16;
  p.g.out_pitch = out_pitch;
  p.g.out_blk = out_blk;
  p.g.coef = const_cast<float*>(coef);
  p.g.fmt = op_fmt ? 1 : 0;
  p.d.thr = threshold;
  p.d.scale = scale;
  p.d.layer = layer;
  p.d.rng = rng;
  const int per = gn_apply16_pix_per_cta(H * W, B);
  MCEDM_REQUIRE(per > 0, "gn_apply16_dropout: cannot tile %d pixels", H * W);
  p.g.pix_per_cta = per;
  MCEDM_CUDA(launch_pdl(gn_apply_dropout_kernel, dim3(H * W / per, B), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), p));
  return 0;
}

extern "C" int mcedm_dropout_bwd16(void* g16, int pitch, int blk, int B, int H, int W, unsigned int threshold, float scale,
                                   int layer, const unsigned int* rng, int op_fmt, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(g16 != nullptr && rng != nullptr && B >= 1 && H >= 1 && W >= 1, "dropout_bwd16: bad arguments");
  MCEDM_REQUIRE(scale >= 1.f && layer >= 0, "dropout_bwd16: scale=%g layer=%d", (double)scale, layer);
  MCEDM_REQUIRE(pitch == 0 || (pitch >= W + 1 && blk >= (H + 1) * pitch), "dropout_bwd16: bad padded layout");
  const GnDropout d{threshold, scale, layer, rng};
  const long long chunks = (long long)B * H * W * 8;
  long long grid = (chunks + 255) / 256;
  if (grid > 8LL * num_sms()) grid = 8LL * num_sms();
  MCEDM_CUDA(launch_pdl(op_fmt == MCEDM_FMT_F16_INF ? dropout_bwd16_kernel<true> : dropout_bwd16_kernel<false>,
                        dim3((unsigned)grid), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), g16, pitch, blk, B, H, W,
                        d, op_fmt ? 1 : 0));
  return 0;
}
