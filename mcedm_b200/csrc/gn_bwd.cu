// K2-bwd / K6 — backward of the fused GroupNorm + (1+scale)/shift + SiLU + resample pass, and the masked
// mixed-conditioning EDM loss with its gradient.
//
// Forward (gn.cu; models/adm_blocks.py:86-97, :161, :163-166):
//     xh = (x - mu) * rstd          per (sample, group of 4 channels)
//     u  = (xh * gamma + beta) * (1 + s) + sh          s, sh = affine(emb) halves (0 when absent)
//     y  = resample(act(u))         act = SiLU | identity; resample = none | nearest x2 | 2x2 mean
// Backward, given dy (fp32, at the conv resolution):
//     du = resample^T(dy) * act'(u)
//     per (sample, channel):  A1 = sum_hw du,  A2 = sum_hw du * xh          (pass 1: gn_bwd_reduce)
//     d sh = A1,  d s = gamma*A2 + beta*A1,  d beta = sum_b (1+s) A1,  d gamma = sum_b (1+s) A2
//     dx = rstd * ( gamma (1+s) du - m1 - xh * m2 ),   m1, m2 = group means of gamma(1+s){A1, A2}
//                                                                         (finalize + pass 2: gn_bwd_apply)
// Pass 2 also adds up to two residual-path gradients, writes the fp32 total, a bf16 copy in the conv
// operand layout (dense NHWC or the padded-flat layout of conv_flat.cu) and per-CTA column sums of the
// total (= the bias gradient of the convolution that produced x).  All reductions are two-stage and
// ordered: results are deterministic.  Streaming, HBM-bound kernels (128-bit accesses).
//
// Loss (models/mcedm.py:213-239, :278; models/losses.py:48-53):
//     D = c_skip x_noise + c_out F ;  L = (1/B) sum_b w_b sum (m D - m x)^2 ;  dF = c_out (2/B) w_b m (m D - m x)
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

namespace mcedm {

struct GnBwdParams {
  const float* dy;           // fp32 NHWC [B, Ho, Wo, 64] gradient w.r.t. the operand written by gn_apply
  const float* x;            // fp32 NHWC [B, Hin, Win, 64] saved input of the GroupNorm
  const float* meanrstd;     // forward statistics of x saved by gn_apply: [B][16][2] = (mean, rstd)
  const float* gamma;
  const float* beta;
  const float* scale_shift;  // nullptr or scale at [b*stride + c], shift at [b*stride + off + c]
  int emb_batch_stride, emb_shift_offset;
  float eps;
  int act, resample;
  int B, Hin, Win;
  int ctas_per_img, pix_per_cta;   // INPUT pixels per CTA
  float* red_partial;        // pass 1 out: [B][ctas_per_img][64][2]
  // ---- pass 2 ----
  const float* coef;         // [B][64][4] = (k1, rstd*m1, rstd*m2, unused) from gn_bwd_finalize
  const float* add0;         // nullptr or fp32 [B,Hin,Win,64] added to dx (residual-path gradients)
  const float* add1;
  int add0_mode;             // how add0 maps onto x: 0 same res, 1 add0 is at 2x res (sum 2x2), 2 add0 at 1/2 res (0.25 * nearest)
  float* dx;                 // fp32 NHWC total gradient w.r.t. x (may be nullptr)
  void* dx_bf16;             // nullptr or bf16 copy (operand layout)
  int out_pitch, out_blk;    // padded-flat layout parameters of dx_bf16 (0 = dense)
  void* dx_bf16_dense;       // nullptr or a second, always dense NHWC bf16 copy (operand of the 1x1 convolutions)
  float* colsum_partial;     // nullptr or [B*ctas_per_img][64]
  int w_shift;               // log2(Win) when Win is a power of two (every level of the U-Net), else -1
  float* dgb_partial;        // [B][64][2] (d gamma, d beta) contributions of sample b (written by CTA 0 of the sample)
  float* d_scale_shift;      // nullptr or d(scale | shift) of sample b
  int dss_batch_stride;
};

// (y, x) of input pixel ip: a shift when the width is a power of two (the integer division was ~1/4 of the loop body)
__device__ __forceinline__ void gn_row_col(const GnBwdParams& p, int ip, int& y, int& x) {
  if (p.w_shift >= 0) {
    y = ip >> p.w_shift;
    x = ip & (p.Win - 1);
  } else {
    y = ip / p.Win;
    x = ip - y * p.Win;
  }
}

// d silu(u)/du = s*(1 + u*(1 - s)), s = sigmoid(u) = 0.5 + 0.5*tanh(u/2): ONE special-function op (MUFU.TANH, 2^-11)
// instead of ex2 + an IEEE reciprocal; the two GroupNorm backward passes were bound by that instruction stream.
__device__ __forceinline__ float silu_grad(float u) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * u));
  const float sg = fmaf(0.5f, t, 0.5f);
  return sg * fmaf(u, 1.0f - sg, 1.0f);
}

// mean / rstd of (b, g) as saved by the forward gn_apply (meanrstd[b][16][2])
__device__ __forceinline__ void gn_load_stats(const GnBwdParams& p, int b, float* sMean, float* sRstd) {
  if (threadIdx.x < 16) {
    const float2 v = *reinterpret_cast<const float2*>(p.meanrstd + ((long long)b * 16 + threadIdx.x) * 2);
    sMean[threadIdx.x] = v.x;
    sRstd[threadIdx.x] = v.y;
  }
}

// resample^T(dy) for 4 channels of input pixel (b, y, x)
__device__ __forceinline__ float4 gather_dy(const GnBwdParams& p, int b, int y, int x, int c) {
  if (p.resample == 0) {
    return *reinterpret_cast<const float4*>(p.dy + (((long long)b * p.Hin + y) * p.Win + x) * 64 + c);
  } else if (p.resample == 1) {   // forward upsampled: each input pixel fed 4 outputs
    const int Wo = p.Win * 2;
    const float* d0 = p.dy + (((long long)b * p.Hin * 2 + 2 * y) * Wo + 2 * x) * 64 + c;
    const float4 a = *reinterpret_cast<const float4*>(d0), bq = *reinterpret_cast<const float4*>(d0 + 64);
    const float4 cq = *reinterpret_cast<const float4*>(d0 + (long long)Wo * 64);
    const float4 dq = *reinterpret_cast<const float4*>(d0 + (long long)Wo * 64 + 64);
    return make_float4((a.x + bq.x) + (cq.x + dq.x), (a.y + bq.y) + (cq.y + dq.y), (a.z + bq.z) + (cq.z + dq.z),
                       (a.w + bq.w) + (cq.w + dq.w));
  } else {                        // forward 2x2 mean: each input pixel fed one output with weight 1/4
    const float4 a = *reinterpret_cast<const float4*>(
        p.dy + (((long long)b * (p.Hin >> 1) + (y >> 1)) * (p.Win >> 1) + (x >> 1)) * 64 + c);
    return make_float4(0.25f * a.x, 0.25f * a.y, 0.25f * a.z, 0.25f * a.w);
  }
}

struct ChanCoef {   // per-channel forward coefficients held in registers for 4 channels
  float4 a, bb, k;  // u = x*a + bb ;  xh = x*rs - mr (rs, mr are per group: same for the 4 channels)
};

// block = 256 threads: 16 channel-quads x 16 pixel lanes
__global__ void __launch_bounds__(256) gn_bwd_reduce_kernel(const GnBwdParams p) {
  __shared__ float sMean[16], sRstd[16];
  __shared__ float sA[64], sB[64];
  __shared__ float red[16][64][2];
  const int b = blockIdx.y;
  gn_load_stats(p, b, sMean, sRstd);
  __syncthreads();
  if (threadIdx.x < 64) {
    const int c = threadIdx.x;
    float a = sRstd[c >> 2] * p.gamma[c];
    float bb = p.beta[c] - sMean[c >> 2] * a;
    if (p.scale_shift) {
      const float* ss = p.scale_shift + (long long)b * p.emb_batch_stride;
      const float sc = 1.0f + ss[c];
      a *= sc;
      bb = fmaf(bb, sc, ss[p.emb_shift_offset + c]);
    }
    sA[c] = a;
    sB[c] = bb;
  }
  __syncthreads();
  const int cq = threadIdx.x & 15, pl = threadIdx.x >> 4;
  const int c = cq * 4;
  const float4 a4 = *reinterpret_cast<const float4*>(&sA[c]);
  const float4 b4 = *reinterpret_cast<const float4*>(&sB[c]);
  const float rs = sRstd[cq], mr = sMean[cq] * sRstd[cq];
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
  const int pix0 = blockIdx.x * p.pix_per_cta;
  for (int i = pl; i < p.pix_per_cta; i += 16) {
    const int ip = pix0 + i;
    int y, x;
    gn_row_col(p, ip, y, x);
    const float4 xv = *reinterpret_cast<const float4*>(p.x + (((long long)b * p.Hin + y) * p.Win + x) * 64 + c);
    float4 d = gather_dy(p, b, y, x, c);
    if (p.act) {
      d.x *= silu_grad(fmaf(xv.x, a4.x, b4.x));
      d.y *= silu_grad(fmaf(xv.y, a4.y, b4.y));
      d.z *= silu_grad(fmaf(xv.z, a4.z, b4.z));
      d.w *= silu_grad(fmaf(xv.w, a4.w, b4.w));
    }
    s1.x += d.x; s1.y += d.y; s1.z += d.z; s1.w += d.w;
    s2.x += d.x * fmaf(xv.x, rs, -mr);
    s2.y += d.y * fmaf(xv.y, rs, -mr);
    s2.z += d.z * fmaf(xv.z, rs, -mr);
    s2.w += d.w * fmaf(xv.w, rs, -mr);
  }
  red[pl][c + 0][0] = s1.x; red[pl][c + 0][1] = s2.x;
  red[pl][c + 1][0] = s1.y; red[pl][c + 1][1] = s2.y;
  red[pl][c + 2][0] = s1.z; red[pl][c + 2][1] = s2.z;
  red[pl][c + 3][0] = s1.w; red[pl][c + 3][1] = s2.w;
  __syncthreads();
  if (threadIdx.x < 128) {
    const int cc = threadIdx.x >> 1, k = threadIdx.x & 1;
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < 16; ++r) t += red[r][cc][k];
    p.red_partial[(((long long)b * p.ctas_per_img + blockIdx.x) * 64 + cc) * 2 + k] = t;
  }
}

__device__ __forceinline__ float4 gather_add(const float* add, int mode, int b, int y, int x, int H, int W, int c) {
  if (mode == 0) {
    return *reinterpret_cast<const float4*>(add + (((long long)b * H + y) * W + x) * 64 + c);
  } else if (mode == 1) {   // add is at 2x resolution (the block downsampled its skip path): 0.25 * sum of 4... no:
    // forward skip = 2x2 mean of x  ->  d x = 0.25 * g(y/2, x/2); handled by mode 2. mode 1: forward skip =
    // nearest-x2 upsample of x -> d x = sum of the 4 outputs
    const int Wo = W * 2;
    const float* d0 = add + (((long long)b * H * 2 + 2 * y) * Wo + 2 * x) * 64 + c;
    const float4 a = *reinterpret_cast<const float4*>(d0), bq = *reinterpret_cast<const float4*>(d0 + 64);
    const float4 cq = *reinterpret_cast<const float4*>(d0 + (long long)Wo * 64);
    const float4 dq = *reinterpret_cast<const float4*>(d0 + (long long)Wo * 64 + 64);
    return make_float4((a.x + bq.x) + (cq.x + dq.x), (a.y + bq.y) + (cq.y + dq.y), (a.z + bq.z) + (cq.z + dq.z),
                       (a.w + bq.w) + (cq.w + dq.w));
  } else {
    const float4 a =
        *reinterpret_cast<const float4*>(add + (((long long)b * (H >> 1) + (y >> 1)) * (W >> 1) + (x >> 1)) * 64 + c);
    return make_float4(0.25f * a.x, 0.25f * a.y, 0.25f * a.z, 0.25f * a.w);
  }
}

__global__ void __launch_bounds__(256) gn_bwd_apply_kernel(const GnBwdParams p) {
  __shared__ float sMean[16], sRstd[16];
  __shared__ float sA[64], sB[64];
  __shared__ float sG1[64], sG2[64], sK[64][3];
  __shared__ float red[16][64];
  const int b = blockIdx.y;
  gn_load_stats(p, b, sMean, sRstd);
  __syncthreads();
  if (threadIdx.x < 64) {
    const int c = threadIdx.x;
    float a = sRstd[c >> 2] * p.gamma[c];
    float bb = p.beta[c] - sMean[c >> 2] * a;
    if (p.scale_shift) {
      const float* ss = p.scale_shift + (long long)b * p.emb_batch_stride;
      const float sc = 1.0f + ss[c];
      a *= sc;
      bb = fmaf(bb, sc, ss[p.emb_shift_offset + c]);
    }
    sA[c] = a;
    sB[c] = bb;
  }
  __syncthreads();
  const int cq = threadIdx.x & 15, pl = threadIdx.x >> 4;
  const int c = cq * 4;
  const float4 a4 = *reinterpret_cast<const float4*>(&sA[c]);
  const float4 b4 = *reinterpret_cast<const float4*>(&sB[c]);
  const float rs = sRstd[cq], mr = sMean[cq] * sRstd[cq];
  // ---- fold of the pass-1 partials (formerly a separate B-CTA launch between the two passes: 41 latency-bound
  // launches per training step).  Every CTA of sample b folds the same records in the same order; CTA 0 of the sample
  // also emits the parameter-gradient rows.
  if (threadIdx.x < 64) {
    const int ch = threadIdx.x;
    double a1 = 0.0, a2 = 0.0;
    const float2* rp = reinterpret_cast<const float2*>(p.red_partial + ((long long)b * p.ctas_per_img * 64 + ch) * 2);
    int t = 0;
    for (; t + 8 <= p.ctas_per_img; t += 8) {
      float2 v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = rp[(t + k) * 64];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        a1 += (double)v[k].x;
        a2 += (double)v[k].y;
      }
    }
    for (; t < p.ctas_per_img; ++t) {
      const float2 v = rp[t * 64];
      a1 += (double)v.x;
      a2 += (double)v.y;
    }
    float sc = 1.0f;
    if (p.scale_shift) sc = 1.0f + p.scale_shift[(long long)b * p.emb_batch_stride + ch];
    const float g = p.gamma[ch], be = p.beta[ch];
    const float A1 = (float)a1, A2 = (float)a2;
    const float kk = g * sc;                      // d xh = kk * du
    sG1[ch] = kk * A1;
    sG2[ch] = kk * A2;
    sK[ch][0] = sRstd[ch >> 2] * kk;
    if (blockIdx.x == 0) {
      p.dgb_partial[((long long)b * 64 + ch) * 2 + 0] = sc * A2;     // d gamma contribution of sample b
      p.dgb_partial[((long long)b * 64 + ch) * 2 + 1] = sc * A1;     // d beta
      if (p.d_scale_shift) {
        p.d_scale_shift[(long long)b * p.dss_batch_stride + ch] = g * A2 + be * A1;                  // d scale
        p.d_scale_shift[(long long)b * p.dss_batch_stride + p.emb_shift_offset + ch] = A1;           // d shift
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int ch = threadIdx.x, g0 = ch & ~3;
    const float cnt = 4.0f * (float)p.Hin * (float)p.Win;
    const float m1 = ((sG1[g0] + sG1[g0 + 1]) + (sG1[g0 + 2] + sG1[g0 + 3])) / cnt;
    const float m2 = ((sG2[g0] + sG2[g0 + 1]) + (sG2[g0 + 2] + sG2[g0 + 3])) / cnt;
    sK[ch][1] = sRstd[ch >> 2] * m1;
    sK[ch][2] = sRstd[ch >> 2] * m2;
  }
  __syncthreads();
  const float4 k0 = make_float4(sK[c][0], sK[c][1], sK[c][2], 0.f), k1 = make_float4(sK[c + 1][0], sK[c + 1][1], sK[c + 1][2], 0.f);
  const float4 k2 = make_float4(sK[c + 2][0], sK[c + 2][1], sK[c + 2][2], 0.f), k3 = make_float4(sK[c + 3][0], sK[c + 3][1], sK[c + 3][2], 0.f);
  float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
  const int pix0 = blockIdx.x * p.pix_per_cta;
  for (int i = pl; i < p.pix_per_cta; i += 16) {
    const int ip = pix0 + i;
    int y, x;
    gn_row_col(p, ip, y, x);
    const long long pix = ((long long)b * p.Hin + y) * p.Win + x;
    const float4 xv = *reinterpret_cast<const float4*>(p.x + pix * 64 + c);
    float4 d = gather_dy(p, b, y, x, c);
    if (p.act) {
      d.x *= silu_grad(fmaf(xv.x, a4.x, b4.x));
      d.y *= silu_grad(fmaf(xv.y, a4.y, b4.y));
      d.z *= silu_grad(fmaf(xv.z, a4.z, b4.z));
      d.w *= silu_grad(fmaf(xv.w, a4.w, b4.w));
    }
    float4 o;
    o.x = k0.x * d.x - k0.y - fmaf(xv.x, rs, -mr) * k0.z;
    o.y = k1.x * d.y - k1.y - fmaf(xv.y, rs, -mr) * k1.z;
    o.z = k2.x * d.z - k2.y - fmaf(xv.z, rs, -mr) * k2.z;
    o.w = k3.x * d.w - k3.y - fmaf(xv.w, rs, -mr) * k3.z;
    if (p.add0) {
      const float4 r = gather_add(p.add0, p.add0_mode, b, y, x, p.Hin, p.Win, c);
      o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
    }
    if (p.add1) {
      const float4 r = *reinterpret_cast<const float4*>(p.add1 + pix * 64 + c);
      o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
    }
    cs.x += o.x; cs.y += o.y; cs.z += o.z; cs.w += o.w;
    if (p.dx) *reinterpret_cast<float4*>(p.dx + pix * 64 + c) = o;
    if (p.dx_bf16) {
      long long opix = pix;
      if (p.out_pitch > 0) opix = (long long)b * p.out_blk + (long long)(y + 1) * p.out_pitch + x;
      uint2 ob;
      ob.x = pack_bf16x2(o.x, o.y);
      ob.y = pack_bf16x2(o.z, o.w);
      *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(p.dx_bf16) + opix * 64 + c) = ob;
    }
    if (p.dx_bf16_dense) {
      uint2 ob;
      ob.x = pack_bf16x2(o.x, o.y);
      ob.y = pack_bf16x2(o.z, o.w);
      *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(p.dx_bf16_dense) + pix * 64 + c) = ob;
    }
  }
  if (p.colsum_partial) {
    red[pl][c + 0] = cs.x; red[pl][c + 1] = cs.y; red[pl][c + 2] = cs.z; red[pl][c + 3] = cs.w;
    __syncthreads();
    if (threadIdx.x < 64) {
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) t += red[r][threadIdx.x];
      p.colsum_partial[((long long)b * p.ctas_per_img + blockIdx.x) * 64 + threadIdx.x] = t;
    }
  }
}

// out[j] (+)= scale * sum_r in[r*stride_r + j*stride_j]: 64 columns x 16 row lanes per CTA, fp64, fixed order
// (folds per-CTA / per-sample partial sums; deterministic)
__global__ void __launch_bounds__(1024)
reduce_rows_kernel(const float* __restrict__ in, int n_rows, long long stride_r, int n_cols, long long stride_j,
                   float* __restrict__ out, int accumulate, float scale) {
  __shared__ double sm[16][64];
  const int c = threadIdx.x & 63, lane = threadIdx.x >> 6;
  const int j = blockIdx.x * 64 + c;
  double t = 0.0;
  if (j < n_cols)
    for (int r = lane; r < n_rows; r += 16) t += (double)in[r * stride_r + j * stride_j];
  sm[lane][c] = t;
  __syncthreads();
  if (lane == 0 && j < n_cols) {
    double a = 0.0;
#pragma unroll
    for (int l = 0; l < 16; ++l) a += sm[l][c];
    const float v = (float)a * scale;
    out[j] = accumulate ? out[j] + v : v;
  }
}

// The same fold for a table of jobs in ONE launch (grid.y = job): the backward of one training step issues ~60 of these
// folds (bias, gamma, beta gradients), each a 3-17 us latency-bound launch; none feeds anything but the flat gradient
// buffer, so they are queued and run together at the end of the backward.
__global__ void __launch_bounds__(1024) reduce_rows_batched_kernel(const mcedm_reduce_job* __restrict__ jobs) {
  __shared__ double sm[16][64];
  const mcedm_reduce_job jb = jobs[blockIdx.y];
  if ((int)blockIdx.x * 64 >= jb.n_cols) return;
  const int c = threadIdx.x & 63, lane = threadIdx.x >> 6;
  const int j = blockIdx.x * 64 + c;
  double t = 0.0;
  if (j < jb.n_cols)
    for (int r = lane; r < jb.n_rows; r += 16) t += (double)jb.in[r * jb.stride_r + j * jb.stride_j];
  sm[lane][c] = t;
  __syncthreads();
  if (lane == 0 && j < jb.n_cols) {
    double a = 0.0;
#pragma unroll
    for (int l = 0; l < 16; ++l) a += sm[l][c];
    const float v = (float)a * jb.scale;
    jb.out[j] = jb.accumulate ? jb.out[j] + v : v;
  }
}

// ------------------------------------------------------------------------------------------------ loss
// grid = (ctas_per_sample, B); NCHW fp32 tensors with chw elements per sample
__global__ void __launch_bounds__(256)
edm_loss_kernel(const float* __restrict__ F, const float* __restrict__ x_noise, const float* __restrict__ x,
                const float* __restrict__ mask, const float* __restrict__ c_skip, const float* __restrict__ c_out,
                const float* __restrict__ weight, long long chw, int B, float* __restrict__ dF,
                uint16_t* __restrict__ dF_pad, long long hw, float* __restrict__ loss_partial) {
  const int b = blockIdx.y;
  const float cs = c_skip[b], co = c_out[b], w = weight[b];
  const float gscale = 2.0f * w / (float)B;
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < chw; i += (long long)gridDim.x * 256) {
    const long long k = (long long)b * chw + i;
    const float m = mask ? mask[k] : 1.0f;
    const float D = __fadd_rn(__fmul_rn(cs, x_noise[k]), __fmul_rn(co, F[k]));
    const float diff = __fsub_rn(__fmul_rn(D, m), __fmul_rn(x[k], m));
    acc += w * diff * diff;
    const float gF = co * gscale * m * diff;
    if (dF) dF[k] = gF;
    if (dF_pad) {   // channel c of pixel (b, i % hw) in a 64-channel bf16 NHWC tensor
      const long long c = i / hw;
      dF_pad[((long long)b * hw + (i - c * hw)) * 64 + c] = (uint16_t)(pack_bf16x2(gF, 0.f) & 0xffffu);
    }
  }
  __shared__ float sm[256];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss_partial[(long long)b * gridDim.x + blockIdx.x] = sm[0];
}


// ------------------------------------------------------------------------------------------------ 16-bit plan
// The same two passes for the 16-bit training plan (train16_engine.py, plan "fused16"): x is the RAW 16-bit activation
// the fused forward stored (dense NHWC or padded-flat), dy the 16-bit output of a data-gradient conv (same layouts), the
// residual-path gradients are fp32 or 16-bit.  Every tensor carries its own (pitch, blk): 0 = dense NHWC, > 0 = the
// padded-flat layout of conv_flat.cu at that tensor's resolution.  The fold of the pass-1 partials is done ONCE per
// sample, by the last CTA of the sample to finish pass 1 (ticket counter; the fold order is
// fixed, so the result does not depend on which CTA that is); pass 2 reads three coefficients per channel.
struct GnBwd16Params {
  const void* dy; int dy_pitch, dy_blk;        // at the conv resolution (Hin x Win, 2x for resample 1, 1/2 for 2)
  const void* x; int x_pitch, x_blk;           // at Hin x Win; dx / dx16 / add1 share this layout
  int fmt;                                     // 16-bit format of x, dy, dx16 (and of 16-bit adds): 0 bf16, 1 fp16
  const float* meanrstd;
  const float* coef_ab;                        // [B][128] = (a | b) of u = a x + b, from the forward's mcedm_gn_coef
  const float* gamma;
  const float* beta;
  const float* scale_shift;
  int emb_batch_stride, emb_shift_offset;
  int act, resample;
  int B, Hin, Win, w_shift;
  int ctas_per_img, pix_per_cta;
  float* red_partial;                          // [B][ctas_per_img][64][2]
  float* kcoef;                                // [B][3][64] = rstd*k | rstd*m1 | rstd*m2 written by the fold
  unsigned int* ticket;                        // [3][B], zero before the launch, zero again after it (see the fused kernel)
  int fused;                                   // both passes in one kernel
  unsigned int* err;                           // watchdog word
  const void* add0; int add0_mode, add0_pitch, add0_blk;   // at ITS resolution (mode as in GnBwdParams)
  const void* add1;
  int add16;                                   // add0 / add1 are 16-bit (fmt) instead of fp32
  float* dx;
  void* dx16;
  void* dx16_dense;
  float* colsum_partial;
  float* dgb_partial;
  float* d_scale_shift;
  int dss_batch_stride;
};

__device__ __forceinline__ long long lay_index(int pitch, int blk, int b, int y, int x, int H, int W) {
  if (pitch > 0) return (long long)b * blk + (long long)(y + 1) * pitch + x;
  return ((long long)b * H + y) * W + x;
}
__device__ __forceinline__ void unpack8(const uint4 r, int fmt, float (&v)[8]) {
  if (fmt) {
    const float2 a = unpack_f16x2(r.x), b = unpack_f16x2(r.y), c = unpack_f16x2(r.z), d = unpack_f16x2(r.w);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
  } else {
    v[0] = bf16_lo(r.x); v[1] = bf16_hi(r.x); v[2] = bf16_lo(r.y); v[3] = bf16_hi(r.y);
    v[4] = bf16_lo(r.z); v[5] = bf16_hi(r.z); v[6] = bf16_lo(r.w); v[7] = bf16_hi(r.w);
  }
}
__device__ __forceinline__ uint4 pack8v(const float (&v)[8], int fmt) {
  uint4 o;
  o.x = pack_op2(v[0], v[1], fmt);
  o.y = pack_op2(v[2], v[3], fmt);
  o.z = pack_op2(v[4], v[5], fmt);
  o.w = pack_op2(v[6], v[7], fmt);
  return o;
}
template <bool INF>
__device__ __forceinline__ uint4 pack8v_g(const float (&v)[8], int fmt) {
  uint4 o;
  o.x = pack_op2_g<INF>(v[0], v[1], fmt);
  o.y = pack_op2_g<INF>(v[2], v[3], fmt);
  o.z = pack_op2_g<INF>(v[4], v[5], fmt);
  o.w = pack_op2_g<INF>(v[6], v[7], fmt);
  return o;
}
__device__ __forceinline__ uint4 ldg16(const void* base, long long pix, int oct) {
  return reinterpret_cast<const uint4*>(base)[pix * 8 + oct];
}
// 8 channels of a tensor that is fp32 or 16-bit
__device__ __forceinline__ void load8_any(const void* base, long long pix, int oct, int is16, int fmt, float (&v)[8]) {
  if (is16) {
    unpack8(ldg16(base, pix, oct), fmt, v);
  } else {
    const float4* q = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + pix * 64 + oct * 8);
    const float4 a = q[0], b = q[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
}
// resample^T(t) for 8 channels of input pixel (b, y, x): t lives at Hin x Win (mode 0), 2x (mode 1: sum of the four
// pixels the input fed) or 1/2 resolution (mode 2: a quarter of the one pixel it fed)
__device__ __forceinline__ void gather8(const void* t, int mode, int pitch, int blk, int is16, int fmt, int b, int y,
                                        int x, int H, int W, int oct, float (&d)[8]) {
  if (mode == 0) {
    load8_any(t, lay_index(pitch, blk, b, y, x, H, W), oct, is16, fmt, d);
  } else if (mode == 1) {
    const long long o00 = lay_index(pitch, blk, b, 2 * y, 2 * x, 2 * H, 2 * W);
    const long long rstride = pitch > 0 ? pitch : 2 * W;
    float t0[8], t1[8], t2[8], t3[8];
    load8_any(t, o00, oct, is16, fmt, t0);
    load8_any(t, o00 + 1, oct, is16, fmt, t1);
    load8_any(t, o00 + rstride, oct, is16, fmt, t2);
    load8_any(t, o00 + rstride + 1, oct, is16, fmt, t3);
#pragma unroll
    for (int k = 0; k < 8; ++k) d[k] = (t0[k] + t1[k]) + (t2[k] + t3[k]);
  } else {
    load8_any(t, lay_index(pitch, blk, b, y >> 1, x >> 1, H >> 1, W >> 1), oct, is16, fmt, d);
#pragma unroll
    for (int k = 0; k < 8; ++k) d[k] *= 0.25f;
  }
}

struct Gn16Coef {
  float a[8], bb[8];
  float rs0, mr0, rs1, mr1;      // the 8 channels span two 4-channel groups
};
// forward coefficients of the thread's 8 channels straight from global memory (independent loads, no barrier)
__device__ __forceinline__ void gn16_coef(const GnBwd16Params& p, int b, int oct, Gn16Coef& cf) {
  const float4* ab = reinterpret_cast<const float4*>(p.coef_ab + (long long)b * 128 + oct * 8);
  const float4 a0 = __ldg(ab), a1 = __ldg(ab + 1), b0 = __ldg(ab + 16), b1 = __ldg(ab + 17);
  const float4 m = __ldg(reinterpret_cast<const float4*>(p.meanrstd + ((long long)b * 16 + 2 * oct) * 2));
  cf.a[0] = a0.x; cf.a[1] = a0.y; cf.a[2] = a0.z; cf.a[3] = a0.w;
  cf.a[4] = a1.x; cf.a[5] = a1.y; cf.a[6] = a1.z; cf.a[7] = a1.w;
  cf.bb[0] = b0.x; cf.bb[1] = b0.y; cf.bb[2] = b0.z; cf.bb[3] = b0.w;
  cf.bb[4] = b1.x; cf.bb[5] = b1.y; cf.bb[6] = b1.z; cf.bb[7] = b1.w;
  cf.rs0 = m.y; cf.mr0 = m.x * m.y;
  cf.rs1 = m.w; cf.mr1 = m.z * m.w;
}

// 256 threads = 8 channel octets x 32 pixel lanes; FAST (no resampling anywhere): NP pixels' 128-bit loads are issued
// before any dependent work (a 16-bit stream has half the bytes per load of the fp32 kernels above: with one pixel in
// flight per thread these passes were latency-bound at a third of the HBM rate).
constexpr int kGnNP = 4;    // pass 1: two streams
constexpr int kGnNPa = 2;   // pass 2: up to four streams + the stores

// pass 1 of one CTA (sums of du and du * xh over its pixels) + the per-sample fold by the last CTA to arrive
// STAGED (one-kernel variant): the loads are per-thread cp.async copies into a 4-deep ring of thread-private shared-memory
// slots, three batches ahead of the arithmetic.  With register-resident batches a warp alternated a load phase and ~400
// instructions of arithmetic per thread (2.6 us per iteration at 14 resident warps per SM: 3.3 TB/s of algorithmic traffic);
// here the memory system always has 3 batches per thread in flight and the registers only hold the pixel being processed.
constexpr int kGnST = 4;                       // ring depth (batches)
constexpr int kGnStageBytes = kGnST * 4 * 4096;   // 4 slots of 256 threads x 16 B per batch

template <bool FAST, bool STAGED = false>
__device__ __forceinline__ void gn16_pass1(const GnBwd16Params& p, float (*red)[64][2], float* sG1, float* sG2,
                                           unsigned int* sLastp, uint32_t stage = 0) {
  unsigned int& sLast = *sLastp;
  const int b = blockIdx.y;
  const int oct = threadIdx.x & 7, pl = threadIdx.x >> 3;
  Gn16Coef cf;
  gn16_coef(p, b, oct, cf);
  float s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s1[k] = s2[k] = 0.f;
  const int pix0 = blockIdx.x * p.pix_per_cta;
  if (FAST && STAGED) {
    constexpr int NPS = 2;                                  // pixels per thread and batch: slots x0 x1 dy0 dy1
    const int n_it = p.pix_per_cta / (32 * NPS);            // pix_per_cta is a power of two >= 128
    const uint32_t sb = stage + threadIdx.x * 16;
    auto issue = [&](int it) {
      if (it < n_it) {
        const uint32_t sl = sb + (uint32_t)(it % kGnST) * (4 * 4096);
#pragma unroll
        for (int u = 0; u < NPS; ++u) {
          const int ip = pix0 + pl + 32 * (it * NPS + u);
          const int y = ip >> p.w_shift, x = ip & (p.Win - 1);
          cp_async16(sl + u * 4096, reinterpret_cast<const uint4*>(p.x) +
                                        lay_index(p.x_pitch, p.x_blk, b, y, x, p.Hin, p.Win) * 8 + oct);
          cp_async16(sl + (NPS + u) * 4096, reinterpret_cast<const uint4*>(p.dy) +
                                                lay_index(p.dy_pitch, p.dy_blk, b, y, x, p.Hin, p.Win) * 8 + oct);
        }
      }
      cp_async_commit();
    };
    issue(0);
    issue(1);
    issue(2);
    for (int it = 0; it < n_it; ++it) {
      issue(it + 3);
      cp_async_wait<3>();
      const uint32_t sl = sb + (uint32_t)(it % kGnST) * (4 * 4096);
#pragma unroll
      for (int u = 0; u < NPS; ++u) {
        float xv[8], d[8];
        unpack8(lds128(sl + u * 4096), p.fmt, xv);
        unpack8(lds128(sl + (NPS + u) * 4096), p.fmt, d);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          float dk = d[k];
          if (p.act) dk *= silu_grad(fmaf(xv[k], cf.a[k], cf.bb[k]));
          s1[k] += dk;
          s2[k] += dk * (k < 4 ? fmaf(xv[k], cf.rs0, -cf.mr0) : fmaf(xv[k], cf.rs1, -cf.mr1));
        }
      }
    }
    cp_async_wait<0>();
  } else if (FAST) {
    for (int i = pl; i < p.pix_per_cta; i += 32 * kGnNP) {
      uint4 xr[kGnNP], dr[kGnNP];
#pragma unroll
      for (int u = 0; u < kGnNP; ++u) {
        if (i + 32 * u < p.pix_per_cta) {
          const int ip = pix0 + i + 32 * u;
          const int y = ip >> p.w_shift, x = ip & (p.Win - 1);
          xr[u] = ldg16(p.x, lay_index(p.x_pitch, p.x_blk, b, y, x, p.Hin, p.Win), oct);
          dr[u] = ldg16(p.dy, lay_index(p.dy_pitch, p.dy_blk, b, y, x, p.Hin, p.Win), oct);
        }
      }
#pragma unroll
      for (int u = 0; u < kGnNP; ++u) {
        if (i + 32 * u < p.pix_per_cta) {
          float xv[8], d[8];
          unpack8(xr[u], p.fmt, xv);
          unpack8(dr[u], p.fmt, d);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float dk = d[k];
            if (p.act) dk *= silu_grad(fmaf(xv[k], cf.a[k], cf.bb[k]));
            s1[k] += dk;
            s2[k] += dk * (k < 4 ? fmaf(xv[k], cf.rs0, -cf.mr0) : fmaf(xv[k], cf.rs1, -cf.mr1));
          }
        }
      }
    }
  } else {
    for (int i = pl; i < p.pix_per_cta; i += 32) {
      const int ip = pix0 + i;
      const int y = ip >> p.w_shift, x = ip & (p.Win - 1);
      float xv[8], d[8];
      unpack8(ldg16(p.x, lay_index(p.x_pitch, p.x_blk, b, y, x, p.Hin, p.Win), oct), p.fmt, xv);
      gather8(p.dy, p.resample, p.dy_pitch, p.dy_blk, 1, p.fmt, b, y, x, p.Hin, p.Win, oct, d);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float dk = d[k];
        if (p.act) dk *= silu_grad(fmaf(xv[k], cf.a[k], cf.bb[k]));
        s1[k] += dk;
        s2[k] += dk * (k < 4 ? fmaf(xv[k], cf.rs0, -cf.mr0) : fmaf(xv[k], cf.rs1, -cf.mr1));
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    red[pl][oct * 8 + k][0] = s1[k];
    red[pl][oct * 8 + k][1] = s2[k];
  }
  __syncthreads();
  if (threadIdx.x < 128) {
    const int cc = threadIdx.x >> 1, k = threadIdx.x & 1;
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < 32; ++r) t += red[r][cc][k];
    p.red_partial[(((long long)b * p.ctas_per_img + blockIdx.x) * 64 + cc) * 2 + k] = t;
  }
  // ---- the last CTA of sample b folds the sample's records (fixed order, fp64) into the pass-2 coefficients and
  // the parameter-gradient rows
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) sLast = (atomicAdd(p.ticket + b, 1u) == (unsigned)p.ctas_per_img - 1u) ? 1u : 0u;
  __syncthreads();
  if (!sLast) return;            // (warp-uniform: the whole CTA leaves)
  __threadfence();
  float kk = 0.f, rstd_c = 0.f;
  if (threadIdx.x < 64) {
    const int ch = threadIdx.x;
    double a1 = 0.0, a2 = 0.0;
    const float2* rp = reinterpret_cast<const float2*>(p.red_partial + ((long long)b * p.ctas_per_img * 64 + ch) * 2);
    int t = 0;
    for (; t + 8 <= p.ctas_per_img; t += 8) {
      float2 v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = __ldcg(rp + (t + k) * 64);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        a1 += (double)v[k].x;
        a2 += (double)v[k].y;
      }
    }
    for (; t < p.ctas_per_img; ++t) {
      const float2 v = __ldcg(rp + t * 64);
      a1 += (double)v.x;
      a2 += (double)v.y;
    }
    float sc = 1.0f;
    if (p.scale_shift) sc = 1.0f + p.scale_shift[(long long)b * p.emb_batch_stride + ch];
    const float g = p.gamma[ch], be = p.beta[ch];
    const float A1 = (float)a1, A2 = (float)a2;
    kk = g * sc;                                  // d xh = kk * du
    rstd_c = p.meanrstd[((long long)b * 16 + (ch >> 2)) * 2 + 1];
    sG1[ch] = kk * A1;
    sG2[ch] = kk * A2;
    p.dgb_partial[((long long)b * 64 + ch) * 2 + 0] = sc * A2;     // d gamma contribution of sample b
    p.dgb_partial[((long long)b * 64 + ch) * 2 + 1] = sc * A1;     // d beta
    if (p.d_scale_shift) {
      p.d_scale_shift[(long long)b * p.dss_batch_stride + ch] = g * A2 + be * A1;                  // d scale
      p.d_scale_shift[(long long)b * p.dss_batch_stride + p.emb_shift_offset + ch] = A1;           // d shift
    }
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int ch = threadIdx.x, g0 = ch & ~3;
    const float cnt = 4.0f * (float)p.Hin * (float)p.Win;
    const float m1 = ((sG1[g0] + sG1[g0 + 1]) + (sG1[g0 + 2] + sG1[g0 + 3])) / cnt;
    const float m2 = ((sG2[g0] + sG2[g0 + 1]) + (sG2[g0 + 2] + sG2[g0 + 3])) / cnt;
    float* kc = p.kcoef + (long long)b * 192 + ch;
    kc[0] = rstd_c * kk;
    kc[64] = rstd_c * m1;
    kc[128] = rstd_c * m2;
  }
  if (threadIdx.x == 0) p.ticket[b] = 0u;         // ready for the next launch on this stream
  if (p.fused) {
    // one-kernel variant: publish "kcoef of sample b is complete" to the sample's other CTAs (spinning in the kernel)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) atomicExch(p.ticket + p.B + b, 1u);
  }
}

template <bool FAST>
__global__ void __launch_bounds__(256) gn_bwd16_reduce_kernel(const GnBwd16Params p) {
  __shared__ float red[32][64][2];
  __shared__ float sG1[64], sG2[64];
  __shared__ unsigned int sLast;
  gn16_pass1<FAST>(p, red, sG1, sG2, &sLast);
}

// pass 2 of one CTA: dx = k0 du - (k1 + xh k2) + residual-path gradients, 16-bit out, column sums
// INF: 16-bit gradient stores without saturation (op_fmt MCEDM_FMT_F16_INF, dynamic loss scaling)
template <bool FAST, bool STAGED = false, bool INF = false>
__device__ __forceinline__ void gn16_pass2(const GnBwd16Params& p, float (*red)[64], uint32_t stage = 0) {
  const int b = blockIdx.y;
  const int oct = threadIdx.x & 7, pl = threadIdx.x >> 3;
  Gn16Coef cf;
  gn16_coef(p, b, oct, cf);
  // dx = k0[c] du - (k1 + xh k2) with k1, k2 constant inside a 4-channel group
  float k0[8], cs[8];
  const float* kc = p.kcoef + (long long)b * 192 + oct * 8;
  {
    const float4 q0 = __ldcg(reinterpret_cast<const float4*>(kc)), q1 = __ldcg(reinterpret_cast<const float4*>(kc + 4));
    k0[0] = q0.x; k0[1] = q0.y; k0[2] = q0.z; k0[3] = q0.w; k0[4] = q1.x; k0[5] = q1.y; k0[6] = q1.z; k0[7] = q1.w;
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) cs[k] = 0.f;
  const float k1a = __ldcg(kc + 64), k2a = __ldcg(kc + 128), k1b = __ldcg(kc + 68), k2b = __ldcg(kc + 132);
  const int pix0 = blockIdx.x * p.pix_per_cta;
  if (FAST && STAGED) {
    // one pixel per thread and batch: slots x, dy, add0, add1
    const int n_it = p.pix_per_cta / 32;
    const uint32_t sb = stage + threadIdx.x * 16;
    auto issue = [&](int it) {
      if (it < n_it) {
        const uint32_t sl = sb + (uint32_t)(it % kGnST) * (4 * 4096);
        const int ip = pix0 + pl + 32 * it;
        const int y = ip >> p.w_shift, x = ip & (p.Win - 1);
        const long long px = lay_index(p.x_pitch, p.x_blk, b, y, x, p.Hin, p.Win);
        cp_async16(sl, reinterpret_cast<const uint4*>(p.x) + px * 8 + oct);
        cp_async16(sl + 4096, reinterpret_cast<const uint4*>(p.dy) +
                                  lay_index(p.dy_pitch, p.dy_blk, b, y, x, p.Hin, p.Win) * 8 + oct);
        if (p.add0)
          cp_async16(sl + 2 * 4096, reinterpret_cast<const uint4*>(p.add0) +
                                        lay_index(p.add0_pitch, p.add0_blk, b, y, x, p.Hin, p.Win) * 8 + oct);
        if (p.add1) cp_async16(sl + 3 * 4096, reinterpret_cast<const uint4*>(p.add1) + px * 8 + oct);
      }
      cp_async_commit();
    };
    issue(0);
    issue(1);
    issue(2);
    for (int it = 0; it < n_it; ++it) {
      issue(it + 3);
      cp_async_wait<3>();
      const uint32_t sl = sb + (uint32_t)(it % kGnST) * (4 * 4096);
      const int ip = pix0 + pl + 32 * it;
      const int y = ip >> p.w_shift, x = ip & (p.Win - 1);
      const long long px = lay_index(p.x_pitch, p.x_blk, b, y, x, p.Hin, p.Win);
      float xv[8], d[8], o[8];
      unpack8(lds128(sl), p.fmt, xv);
      unpack8(lds128(sl + 4096), p.fmt, d);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float dk = d[k];
        if (p.act) dk *= silu_grad(fmaf(xv[k], cf.a[k], cf.bb[k]));
        const float t = k < 4 ? fmaf(fmaf(xv[k], cf.rs0, -cf.mr0), k2a, k1a) : fmaf(fmaf(xv[k], cf.rs1, -cf.mr1), k2b, k1b);
        o[k] = fmaf(k0[k], dk, -t);
      }
      if (p.add0) {
        float r[8];
        unpack8(lds128(sl + 2 * 4096), p.fmt, r);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] += r[k];
      }
      if (p.add1) {
        float r[8];
        unpack8(lds128(sl + 3 * 4096), p.fmt, r);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] += r[k];
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) cs[k] += o[k];
      if (p.dx) {
        float4* q = reinterpret_cast<float4*>(p.dx + px * 64 + oct * 8);
        q[0] = make_float4(o[0], o[1], o[2], o[3]);
        q[1] = make_float4(o[4], o[5], o[6], o[7]);
      }
      const uint4 ov = pack8v_g<INF>(o, p.fmt);
      if (p.dx16) reinterpret_cast<uint4*>(p.dx16)[px * 8 + oct] = ov;
      if (p.dx16_dense) reinterpret_cast<uint4*>(p.dx16_dense)[((long long)b * p.Hin * p.Win + ip) * 8 + oct] = ov;
    }
    cp_async_wait<0>();
  } else if (FAST) {
    // no resampling, residual-path gradients (if any) 16-bit at the same resolution
    for (int i = pl; i < p.pix_per_cta; i += 32 * kGnNPa) {
      uint4 xr[kGnNPa], dr[kGnNPa], ar[kGnNPa], br[kGnNPa];
      long long pix[kGnNPa];
#pragma unroll
      for (int u = 0; u < kGnNPa; ++u) {
        if (i + 32 * u < p.pix_per_cta) {
          const int ip = pix0 + i + 32 * u;
          const int y = ip >> p.w_shift, x = ip & (p.Win - 1);
          pix[u] = lay_index(p.x_pitch, p.x_blk, b, y, x, p.Hin, p.Win);
          xr[u] = ldg16(p.x, pix[u], oct);
          dr[u] = ldg16(p.dy, lay_index(p.dy_pitch, p.dy_blk, b, y, x, p.Hin, p.Win), oct);
          if (p.add0) ar[u] = ldg16(p.add0, lay_index(p.add0_pitch, p.add0_blk, b, y, x, p.Hin, p.Win), oct);
          if (p.add1) br[u] = ldg16(p.add1, pix[u], oct);
        }
      }
#pragma unroll
      for (int u = 0; u < kGnNPa; ++u) {
        if (i + 32 * u < p.pix_per_cta) {
          float xv[8], d[8], o[8];
          unpack8(xr[u], p.fmt, xv);
          unpack8(dr[u], p.fmt, d);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float dk = d[k];
            if (p.act) dk *= silu_grad(fmaf(xv[k], cf.a[k], cf.bb[k]));
            const float t = k < 4 ? fmaf(fmaf(xv[k], cf.rs0, -cf.mr0), k2a, k1a) : fmaf(fmaf(xv[k], cf.rs1, -cf.mr1), k2b, k1b);
            o[k] = fmaf(k0[k], dk, -t);
          }
          if (p.add0) {
            float r[8];
            unpack8(ar[u], p.fmt, r);
#pragma unroll
            for (int k = 0; k < 8; ++k) o[k] += r[k];
          }
          if (p.add1) {
            float r[8];
            unpack8(br[u], p.fmt, r);
#pragma unroll
            for (int k = 0; k < 8; ++k) o[k] += r[k];
          }
#pragma unroll
          for (int k = 0; k < 8; ++k) cs[k] += o[k];
          if (p.dx) {
            float4* q = reinterpret_cast<float4*>(p.dx + pix[u] * 64 + oct * 8);
            q[0] = make_float4(o[0], o[1], o[2], o[3]);
            q[1] = make_float4(o[4], o[5], o[6], o[7]);
          }
          const uint4 ov = pack8v_g<INF>(o, p.fmt);
          if (p.dx16) reinterpret_cast<uint4*>(p.dx16)[pix[u] * 8 + oct] = ov;
          if (p.dx16_dense) {
            const int ip = pix0 + i + 32 * u;
            reinterpret_cast<uint4*>(p.dx16_dense)[((long long)b * p.Hin * p.Win + ip) * 8 + oct] = ov;
          }
        }
      }
    }
  } else {
    for (int i = pl; i < p.pix_per_cta; i += 32) {
      const int ip = pix0 + i;
      const int y = ip >> p.w_shift, x = ip & (p.Win - 1);
      const long long pix = lay_index(p.x_pitch, p.x_blk, b, y, x, p.Hin, p.Win);
      float xv[8], d[8], o[8];
      unpack8(ldg16(p.x, pix, oct), p.fmt, xv);
      gather8(p.dy, p.resample, p.dy_pitch, p.dy_blk, 1, p.fmt, b, y, x, p.Hin, p.Win, oct, d);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float dk = d[k];
        if (p.act) dk *= silu_grad(fmaf(xv[k], cf.a[k], cf.bb[k]));
        const float t = k < 4 ? fmaf(fmaf(xv[k], cf.rs0, -cf.mr0), k2a, k1a) : fmaf(fmaf(xv[k], cf.rs1, -cf.mr1), k2b, k1b);
        o[k] = fmaf(k0[k], dk, -t);
      }
      if (p.add0) {
        float r[8];
        gather8(p.add0, p.add0_mode, p.add0_pitch, p.add0_blk, p.add16, p.fmt, b, y, x, p.Hin, p.Win, oct, r);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] += r[k];
      }
      if (p.add1) {
        float r[8];
        load8_any(p.add1, pix, oct, p.add16, p.fmt, r);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] += r[k];
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) cs[k] += o[k];
      if (p.dx) {
        float4* q = reinterpret_cast<float4*>(p.dx + pix * 64 + oct * 8);
        q[0] = make_float4(o[0], o[1], o[2], o[3]);
        q[1] = make_float4(o[4], o[5], o[6], o[7]);
      }
      const uint4 ov = pack8v_g<INF>(o, p.fmt);
      if (p.dx16) reinterpret_cast<uint4*>(p.dx16)[pix * 8 + oct] = ov;
      if (p.dx16_dense) reinterpret_cast<uint4*>(p.dx16_dense)[((long long)b * p.Hin * p.Win + ip) * 8 + oct] = ov;
    }
  }
  if (p.colsum_partial) {
#pragma unroll
    for (int k = 0; k < 8; ++k) red[pl][oct * 8 + k] = cs[k];
    __syncthreads();
    if (threadIdx.x < 64) {
      float t = 0.f;
#pragma unroll
      for (int r = 0; r < 32; ++r) t += red[r][threadIdx.x];
      p.colsum_partial[((long long)b * p.ctas_per_img + blockIdx.x) * 64 + threadIdx.x] = t;
    }
  }
}

template <bool FAST, bool INF = false>
__global__ void __launch_bounds__(256, 2) gn_bwd16_apply_kernel(const GnBwd16Params p) {
  __shared__ float red[32][64];
  gn16_pass2<FAST, false, INF>(p, red);
}

// Both passes in ONE kernel (p.fused).  The grid is about one wave of co-resident CTAs (pick_pix_per_cta16; the launcher
// checks it against 2 x SM count), a sample's CTAs are neighbours in the launch order: each CTA runs pass 1 on its pixel
// slice, the last one of the sample folds the partial sums and raises the sample's flag, the others spin on it, then every
// CTA runs pass 2 on the SAME slice, which it finds in L2 (a sample is 2 x 2 MB at 128 x 128): 3 instead of 5 trips
// through HBM per element.  ticket[0..B) counts pass-1 arrivals, ticket[B..2B) is the flag, ticket[2B..3B) counts pass-2
// departures (the last one clears the flag): every word is zero again when the launch ends.  The spin is bounded like the
// mbarrier waits (a protocol bug must not hang the GPU): on timeout the CTA goes on with whatever kcoef holds and
// records the tag in *err.
template <bool FAST1, bool FAST2, bool INF = false>
__global__ void __launch_bounds__(256, 2) gn_bwd16_fused_kernel(const GnBwd16Params p) {
  __shared__ float red[32][64][2];
  __shared__ float sG1[64], sG2[64];
  __shared__ unsigned int sLast;
  extern __shared__ uint4 gn_stage[];
  const uint32_t stage = smem_u32(gn_stage);
  gn16_pass1<FAST1, FAST1>(p, red, sG1, sG2, &sLast, stage);
  const int b = blockIdx.y;
  if (threadIdx.x == 0) {
    volatile unsigned int* flag = p.ticket + p.B + b;
    if (*flag == 0u) {
      const long long t0 = clock64();
      while (*flag == 0u) {
        __nanosleep(64);
        if (clock64() - t0 > 2000000000LL) {
          atomicCAS(p.err, 0u, 0xdead7000u);
          break;
        }
      }
    }
    __threadfence();
  }
  __syncthreads();
  gn16_pass2<FAST2, FAST2, INF>(p, reinterpret_cast<float(*)[64]>(&red[0][0][0]), stage);
  __syncthreads();
  if (threadIdx.x == 0) {
    if (atomicAdd(p.ticket + 2 * p.B + b, 1u) == (unsigned)p.ctas_per_img - 1u) {
      p.ticket[2 * p.B + b] = 0u;
      p.ticket[p.B + b] = 0u;
    }
  }
}

// CTAs of the 16-bit passes: >= 128 pixels (32 lanes x 4 pixels in flight); about ONE wave of equal CTAs (2 resident per
// SM) when the batch allows it, so the per-CTA prologue (coefficient loads) is paid once
static int pick_pix_per_cta16(int work, int B) {
  int per = 2048;
  while (per > 128 && ((work % per) != 0 || 2LL * (work / per) * B < 3LL * num_sms())) per >>= 1;
  while (per > 16 && (work % per) != 0) per >>= 1;
  return per;
}

static int pick_pix_per_cta(int work, int B) {
  int per = 2048;
  while (per > 16 && ((work % per) != 0 || (long long)(work / per) * B < 4LL * num_sms())) per >>= 1;
  if (per < 16) per = 16;
  while (per > 16 && (work % per) != 0) per >>= 1;
  return per;
}

}  // namespace mcedm

extern "C" int mcedm_gn_bwd16_ctas_per_img(int Hin, int Win, int B) {
  const int work = Hin * Win;
  return work / mcedm::pick_pix_per_cta16(work, B);
}

extern "C" int mcedm_gn_bwd_ctas_per_img(int Hin, int Win, int B) {
  const int work = Hin * Win;
  return work / mcedm::pick_pix_per_cta(work, B);
}

extern "C" int mcedm_gn_bwd(const float* dy, const float* x, const float* meanrstd, const float* gamma, const float* beta, const float* scale_shift, int emb_batch_stride,
                            int emb_shift_offset, float eps, int act, int resample, int B, int Hin, int Win,
                            float* red_partial, float* coef, float* dgb_partial, float* d_scale_shift,
                            int dss_batch_stride, const float* add0, int add0_mode, const float* add1, float* dx,
                            void* dx_bf16, int out_pitch, int out_blk, void* dx_bf16_dense, float* colsum_partial,
                            void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && (Hin * Win) % 16 == 0, "gn_bwd: bad shape");
  MCEDM_REQUIRE(resample >= 0 && resample <= 2, "gn_bwd: resample=%d", resample);
  GnBwdParams p;
  memset(&p, 0, sizeof(p));
  p.dy = dy; p.x = x; p.meanrstd = meanrstd;
  p.gamma = gamma; p.beta = beta; p.scale_shift = scale_shift;
  p.emb_batch_stride = emb_batch_stride; p.emb_shift_offset = emb_shift_offset;
  p.eps = eps; p.act = act; p.resample = resample;
  p.B = B; p.Hin = Hin; p.Win = Win;
  const int work = Hin * Win;
  p.w_shift = (Win & (Win - 1)) == 0 ? __builtin_ctz((unsigned)Win) : -1;
  p.pix_per_cta = pick_pix_per_cta(work, B);
  p.ctas_per_img = work / p.pix_per_cta;
  p.red_partial = red_partial;
  p.coef = coef;   // unused since the fold moved into the apply pass (kept in the ABI as caller-owned scratch)
  p.add0 = add0; p.add0_mode = add0_mode; p.add1 = add1;
  p.dx = dx; p.dx_bf16 = dx_bf16; p.out_pitch = out_pitch; p.out_blk = out_blk;
  p.dx_bf16_dense = dx_bf16_dense;
  p.colsum_partial = colsum_partial;
  p.dgb_partial = dgb_partial;
  p.d_scale_shift = d_scale_shift;
  p.dss_batch_stride = dss_batch_stride;
  MCEDM_REQUIRE(dgb_partial != nullptr, "gn_bwd: dgb_partial ([B][64][2]) is required");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  dim3 grid(p.ctas_per_img, B);
  gn_bwd_reduce_kernel<<<grid, 256, 0, st>>>(p);
  MCEDM_CUDA(cudaGetLastError());
  gn_bwd_apply_kernel<<<grid, 256, 0, st>>>(p);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}


namespace mcedm {
template <bool INF>
static int gn_bwd16_launch(GnBwd16Params& p, dim3 grid, int resample, bool fast2, int split, cudaStream_t st) {
  // one kernel when every CTA of the grid is resident at once (2 per SM): the in-kernel wait needs the sample's CTAs live
  if (!split && (long long)p.ctas_per_img * p.B <= 2LL * num_sms() && p.pix_per_cta % 64 == 0) {   // (staged batches: 64 pixels)
    p.fused = 1;
    p.err = watchdog_ptr();
    MCEDM_REQUIRE(p.err != nullptr, "gn_bwd16: cannot allocate the watchdog word");
    static bool attr = false;
    if (!attr) {
      MCEDM_CUDA(cudaFuncSetAttribute(gn_bwd16_fused_kernel<true, true, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGnStageBytes));
      MCEDM_CUDA(cudaFuncSetAttribute(gn_bwd16_fused_kernel<true, false, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGnStageBytes));
      attr = true;
    }
    if (resample == 0 && fast2) gn_bwd16_fused_kernel<true, true, INF><<<grid, 256, kGnStageBytes, st>>>(p);
    else if (resample == 0) gn_bwd16_fused_kernel<true, false, INF><<<grid, 256, kGnStageBytes, st>>>(p);
    else gn_bwd16_fused_kernel<false, false, INF><<<grid, 256, 0, st>>>(p);
    MCEDM_CUDA(cudaGetLastError());
    return 0;
  }
  if (resample == 0) {
    gn_bwd16_reduce_kernel<true><<<grid, 256, 0, st>>>(p);
  } else {
    gn_bwd16_reduce_kernel<false><<<grid, 256, 0, st>>>(p);
  }
  MCEDM_CUDA(cudaGetLastError());
  if (fast2) {      // the batched pass takes 16-bit residual-path gradients at the same resolution only
    gn_bwd16_apply_kernel<true, INF><<<grid, 256, 0, st>>>(p);
  } else {
    gn_bwd16_apply_kernel<false, INF><<<grid, 256, 0, st>>>(p);
  }
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace mcedm

extern "C" int mcedm_gn_bwd16(const void* dy16, int dy_pitch, int dy_blk, const void* x16, int x_pitch, int x_blk,
                              int op_fmt, const float* meanrstd, const float* coef_ab, const float* gamma,
                              const float* beta, const float* scale_shift, int emb_batch_stride, int emb_shift_offset,
                              int act, int resample, int B, int Hin, int Win, float* red_partial, float* kcoef,
                              unsigned int* ticket, float* dgb_partial, float* d_scale_shift, int dss_batch_stride,
                              const void* add0, int add0_mode, int add0_pitch, int add0_blk, const void* add1,
                              int add16, float* dx, void* dx16, void* dx16_dense, float* colsum_partial,
                              void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && (Hin * Win) % 16 == 0 && (Win & (Win - 1)) == 0, "gn_bwd16: bad shape %dx%d", Hin, Win);
  MCEDM_REQUIRE(resample >= 0 && resample <= 2 && add0_mode >= 0 && add0_mode <= 2, "gn_bwd16: resample=%d add0_mode=%d",
                resample, add0_mode);
  MCEDM_REQUIRE(dy16 && x16 && meanrstd && coef_ab && red_partial && dgb_partial && kcoef && ticket,
                "gn_bwd16: missing buffers");
  GnBwd16Params p;
  memset(&p, 0, sizeof(p));
  p.dy = dy16; p.dy_pitch = dy_pitch; p.dy_blk = dy_blk;
  p.x = x16; p.x_pitch = x_pitch; p.x_blk = x_blk;
  p.fmt = op_fmt ? 1 : 0;
  p.meanrstd = meanrstd; p.coef_ab = coef_ab; p.gamma = gamma; p.beta = beta; p.scale_shift = scale_shift;
  p.emb_batch_stride = emb_batch_stride; p.emb_shift_offset = emb_shift_offset;
  p.act = act; p.resample = resample;
  p.B = B; p.Hin = Hin; p.Win = Win;
  p.w_shift = __builtin_ctz((unsigned)Win);
  const int work = Hin * Win;
  p.pix_per_cta = pick_pix_per_cta16(work, B);
  p.ctas_per_img = work / p.pix_per_cta;
  p.red_partial = red_partial;
  p.kcoef = kcoef;
  p.ticket = ticket;
  p.add0 = add0; p.add0_mode = add0_mode; p.add0_pitch = add0_pitch; p.add0_blk = add0_blk;
  p.add1 = add1;
  p.add16 = add16 ? 1 : 0;
  p.dx = dx; p.dx16 = dx16; p.dx16_dense = dx16_dense;
  p.colsum_partial = colsum_partial;
  p.dgb_partial = dgb_partial;
  p.d_scale_shift = d_scale_shift;
  p.dss_batch_stride = dss_batch_stride;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  dim3 grid(p.ctas_per_img, B);
  const bool fast2 = resample == 0 && (add0 == nullptr || (add0_mode == 0 && p.add16)) && (add1 == nullptr || p.add16);
  static int split = -1;
  if (split < 0) {
    const char* e = getenv("MCEDM_GNBWD_SPLIT");
    split = (e && atoi(e)) ? 1 : 0;
  }
  if (op_fmt == MCEDM_FMT_F16_INF) return gn_bwd16_launch<true>(p, grid, resample, fast2, split, st);
  return gn_bwd16_launch<false>(p, grid, resample, fast2, split, st);
}

extern "C" int mcedm_reduce_rows(const float* in, int n_rows, long long stride_r, int n_cols, long long stride_j,
                                 float* out, int accumulate, float scale, void* stream) {
  using namespace mcedm;
  reduce_rows_kernel<<<(n_cols + 63) / 64, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      in, n_rows, stride_r, n_cols, stride_j, out, accumulate, scale);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_reduce_rows_batched(const mcedm_reduce_job* jobs_dev, int n_jobs, int max_cols, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n_jobs >= 1 && n_jobs <= 65535 && max_cols >= 1, "reduce_rows_batched: bad sizes");
  dim3 grid((max_cols + 63) / 64, n_jobs);
  reduce_rows_batched_kernel<<<grid, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(jobs_dev);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_loss(const float* F, const float* x_noise, const float* x, const float* mask,
                              const float* c_skip, const float* c_out, const float* weight, int B, long long chw,
                              float* dF, void* dF_pad_bf16, long long hw, float* loss_partial, int ctas_per_sample,
                              void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && ctas_per_sample >= 1, "edm_loss: bad sizes");
  MCEDM_REQUIRE(dF_pad_bf16 == nullptr || (hw >= 1 && chw % hw == 0 && chw / hw <= 64), "edm_loss: bad padded output");
  dim3 grid(ctas_per_sample, B);
  edm_loss_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(F, x_noise, x, mask, c_skip, c_out, weight,
                                                                            chw, B, dF,
                                                                            reinterpret_cast<uint16_t*>(dF_pad_bf16), hw,
                                                                            loss_partial);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}
