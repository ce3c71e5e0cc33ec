// Small training-side kernels (HBM- or latency-bound; CUDA cores):
//   * edm_noise_in     — x_noise = x + mask*noise*sigma_b ; x_in = c_in_b * x_noise        (models/mcedm.py:216, :208)
//   * nchw_to_nhwc_pad — NCHW fp32 (<= 8 channels, up to two tensors concatenated) -> the first channels of a
//                        64-channel bf16 NHWC tensor (remaining channels stay zero): turns the first conv's
//                        input and dL/dF into tensor-core operands for conv_wgrad / the data-gradient convs
//   * colsum_bf16      — per-CTA column sums of a bf16 [pixels, C] tensor (bias gradients of qkv, out_conv)
//   * emb_mlp_bwd      — backward of emb_mlp (small.cu): per-sample pass + batch-reduction pass
//   * sumsq_partial / adam_step / ema_update — gradient-norm clipping (clip_grad_norm_ semantics,
//                        configs/trainer/trainer_ddim.yaml:8-9), torch.optim.Adam update (models/mcedm.py:141) and
//                        EmaModel.update (models/ddim_blocks.py:48-56) on flat fp32 buffers
//   * grad_accumulate  — the gradient-accumulation fold: window buffer (+)= micro-batch flat gradient / N
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace mcedm {

__global__ void __launch_bounds__(256)
edm_noise_in_kernel(const float* __restrict__ x, const float* __restrict__ noise, const float* __restrict__ mask,
                    const float* __restrict__ sigma, const float* __restrict__ c_in, long long chw,
                    float* __restrict__ x_noise, float* __restrict__ x_in) {
  const int b = blockIdx.y;
  const float s = sigma[b], ci = c_in[b];
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < chw; i += (long long)gridDim.x * 256) {
    const long long k = (long long)b * chw + i;
    // x + mask * noise * sigma, evaluated left to right as torch does (mcedm.py:216)
    const float t = mask ? __fmul_rn(__fmul_rn(mask[k], noise[k]), s) : __fmul_rn(noise[k], s);
    const float xn = __fadd_rn(x[k], t);
    x_noise[k] = xn;
    x_in[k] = __fmul_rn(ci, xn);
  }
}

// Batch preparation of PlMcedm.training_step (models/mcedm.py:257-265, :241-252; models/normalizer.py:28-29):
//   x[b,0] = (h - h_sub)/h_div ; x[b,1] = (u - u_sub)/u_div                      (data_transform, b h w c)
//   cond   = x*(1 - mask) + randn*mask                                            (get_cond_in)
// and the three `b h w c -> b c h w` rearranges, in one pass (the reference: ~10 elementwise / permute launches).
// Every float32 operation is the torch operation, individually rounded: outputs are bit-identical.
// h, u: [B,HW] ; mask, randn: [B,HW,2] (channel-last, as the datamodule / torch.randn_like produce them);
// x, cond, mask_c: [B,2,HW] (channel-first).  One thread per pixel: 8-byte channel-pair loads, coalesced plane stores.
__global__ void __launch_bounds__(256)
mcedm_prep_kernel(const float* __restrict__ h, const float* __restrict__ u, const float* __restrict__ mask,
                  const float* __restrict__ randn, float h_sub, float h_div, float u_sub, float u_div, long long HW,
                  long long total_pix, float* __restrict__ x, float* __restrict__ cond, float* __restrict__ mask_c) {
  const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
  if (pix >= total_pix) return;
  const long long b = pix / HW, hw = pix - b * HW;
  const float xh = __fdiv_rn(__fsub_rn(h[pix], h_sub), h_div);
  const float xu = __fdiv_rn(__fsub_rn(u[pix], u_sub), u_div);
  const float2 m = *reinterpret_cast<const float2*>(mask + pix * 2);
  const float2 r = *reinterpret_cast<const float2*>(randn + pix * 2);
  const long long o0 = (b * 2) * HW + hw, o1 = o0 + HW;
  x[o0] = xh;
  x[o1] = xu;
  cond[o0] = __fadd_rn(__fmul_rn(xh, __fsub_rn(1.0f, m.x)), __fmul_rn(r.x, m.x));
  cond[o1] = __fadd_rn(__fmul_rn(xu, __fsub_rn(1.0f, m.y)), __fmul_rn(r.y, m.y));
  mask_c[o0] = m.x;
  mask_c[o1] = m.y;
}

// The same with the mask GENERATED on the device (SURVEY section 8f rank 3): every mask the reference's datasets produce
// (h5_dataset.py:232-255 channel masks, :306-393 time masks) is "channel c is missing from time row obs_rows[b][c]
// on" (0: whole channel missing, H: fully observed, t_max: random observation horizon), so the DataLoader only has to
// deliver the two integers per item it drew with the reference's RNG calls; the [B,H,W,2] mask never crosses PCIe and
// the per-item torch.cat / ones_like / zeros_like work of the worker processes disappears.
__global__ void __launch_bounds__(256)
mcedm_prep_rows_kernel(const float* __restrict__ h, const float* __restrict__ u, const int* __restrict__ obs_rows,
                       const float* __restrict__ randn, float h_sub, float h_div, float u_sub, float u_div, long long HW,
                       int W, long long total_pix, float* __restrict__ x, float* __restrict__ cond,
                       float* __restrict__ mask_c, float* __restrict__ mask_bhwc) {
  const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
  if (pix >= total_pix) return;
  const long long b = pix / HW, hw = pix - b * HW;
  const int t = (int)(hw / W);
  const float xh = __fdiv_rn(__fsub_rn(h[pix], h_sub), h_div);
  const float xu = __fdiv_rn(__fsub_rn(u[pix], u_sub), u_div);
  const float2 m = make_float2(t >= obs_rows[b * 2] ? 1.0f : 0.0f, t >= obs_rows[b * 2 + 1] ? 1.0f : 0.0f);
  const float2 r = *reinterpret_cast<const float2*>(randn + pix * 2);
  const long long o0 = (b * 2) * HW + hw, o1 = o0 + HW;
  x[o0] = xh;
  x[o1] = xu;
  cond[o0] = __fadd_rn(__fmul_rn(xh, __fsub_rn(1.0f, m.x)), __fmul_rn(r.x, m.x));
  cond[o1] = __fadd_rn(__fmul_rn(xu, __fsub_rn(1.0f, m.y)), __fmul_rn(r.y, m.y));
  mask_c[o0] = m.x;
  mask_c[o1] = m.y;
  if (mask_bhwc) *reinterpret_cast<float2*>(mask_bhwc + pix * 2) = m;
}

// one thread per pixel; dst channels [c_dst0, c_dst0 + Ca + Cb) <- cat(a, b)[:, :, pix]
__global__ void __launch_bounds__(256)
nchw_to_nhwc_pad_kernel(const float* __restrict__ a, int Ca, const float* __restrict__ bsrc, int Cb, long long HW,
                        long long total_pix, unsigned short* __restrict__ dst, int c_dst0, float scale, int fmt) {
  const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
  if (pix >= total_pix) return;
  const long long b = pix / HW, hw = pix - b * HW;
  unsigned short* d = dst + pix * 64 + c_dst0;
  for (int c = 0; c < Ca; ++c) d[c] = (unsigned short)(pack_op2(scale * a[(b * Ca + c) * HW + hw], 0.f, fmt) & 0xffffu);
  for (int c = 0; c < Cb; ++c)
    d[Ca + c] = (unsigned short)(pack_op2(scale * bsrc[(b * Cb + c) * HW + hw], 0.f, fmt) & 0xffffu);
}

// the same for the loss-scaled dL/dF of dynamic loss scaling: the scale is read from device memory (a graph replay sees
// the current one) and the fp16 conversion does not saturate (S * dL/dF beyond 65504 becomes inf: the step skips)
__global__ void __launch_bounds__(256)
nchw_to_nhwc_pad_scaled_kernel(const float* __restrict__ a, int Ca, const float* __restrict__ bsrc, int Cb, long long HW,
                               long long total_pix, unsigned short* __restrict__ dst, int c_dst0,
                               const float* __restrict__ scale_dev) {
  const long long pix = (long long)blockIdx.x * 256 + threadIdx.x;
  if (pix >= total_pix) return;
  const float scale = *scale_dev;
  const long long b = pix / HW, hw = pix - b * HW;
  unsigned short* d = dst + pix * 64 + c_dst0;
  for (int c = 0; c < Ca; ++c) d[c] = (unsigned short)(pack_f16x2_inf(scale * a[(b * Ca + c) * HW + hw], 0.f) & 0xffffu);
  for (int c = 0; c < Cb; ++c)
    d[Ca + c] = (unsigned short)(pack_f16x2_inf(scale * bsrc[(b * Cb + c) * HW + hw], 0.f) & 0xffffu);
}

// grid = n_ctas, block = 256 = 8 channel-octets x 32 pixel lanes; x is [pixels][C] bf16, this launch sums the
// 64 channels starting at c_off.  partial[cta][64]
__global__ void __launch_bounds__(256)
colsum_bf16_kernel(const unsigned short* __restrict__ x, long long pixels, int C, int c_off,
                   float* __restrict__ partial, int fmt) {
  __shared__ float red[32][64];
  const int oct = threadIdx.x & 7, pl = threadIdx.x >> 3;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  const long long per = (pixels + gridDim.x - 1) / gridDim.x;
  const long long p0 = (long long)blockIdx.x * per;
  const long long p1 = p0 + per < pixels ? p0 + per : pixels;
  for (long long pix = p0 + pl; pix < p1; pix += 32) {
    const uint4 v = *reinterpret_cast<const uint4*>(x + pix * C + c_off + oct * 8);
    if (fmt) {
      const float2 a = unpack_f16x2(v.x), b = unpack_f16x2(v.y), c = unpack_f16x2(v.z), d = unpack_f16x2(v.w);
      acc[0] += a.x; acc[1] += a.y; acc[2] += b.x; acc[3] += b.y;
      acc[4] += c.x; acc[5] += c.y; acc[6] += d.x; acc[7] += d.y;
    } else {
      acc[0] += bf16_lo(v.x); acc[1] += bf16_hi(v.x);
      acc[2] += bf16_lo(v.y); acc[3] += bf16_hi(v.y);
      acc[4] += bf16_lo(v.z); acc[5] += bf16_hi(v.z);
      acc[6] += bf16_lo(v.w); acc[7] += bf16_hi(v.w);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) red[pl][oct * 8 + i] = acc[i];
  __syncthreads();
  if (threadIdx.x < 64) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < 32; ++r) t += red[r][threadIdx.x];
    partial[(long long)blockIdx.x * 64 + threadIdx.x] = t;
  }
}

// ------------------------------------------- emb MLP backward -------------------------------------------
__device__ __forceinline__ float silu_grad_f(float u) {
  const float sg = 1.0f / (1.0f + __expf(-u));
  return sg * (1.0f + u * (1.0f - sg));
}

// Pass 1, grid = B, block = 128: recompute the forward of sample b, back-propagate d(scale|shift) of all blocks
// to the two hidden layers.  vec[b] = (e | h0 | h1 | d_pre0 | d_pre1), 5 x 64 floats.
__global__ void __launch_bounds__(128)
emb_bwd_sample_kernel(const float* __restrict__ c_noise, const float* __restrict__ freqs, const float* __restrict__ w0,
                      const float* __restrict__ b0, const float* __restrict__ w1, const float* __restrict__ b1,
                      const float* __restrict__ aff_w, const float* __restrict__ dss, int n_aff, int B,
                      float* __restrict__ vec) {
  __shared__ float e[64], h0[64], pre0[64], pre1[64], h1[64], d1[64], dh0[64], g[128];
  const int b = blockIdx.x, t = threadIdx.x;
  if (t < 32) {
    const float ang = c_noise[b] * freqs[t];
    e[t] = cosf(ang);
    e[t + 32] = sinf(ang);
  }
  __syncthreads();
  if (t < 64) {
    float acc = 0.f;
    for (int k = 0; k < 64; ++k) acc = fmaf(e[k], w0[t * 64 + k], acc);
    pre0[t] = acc + b0[t];
    h0[t] = silu_f(pre0[t]);
  }
  __syncthreads();
  if (t < 64) {
    float acc = 0.f;
    for (int k = 0; k < 64; ++k) acc = fmaf(h0[k], w1[t * 64 + k], acc);
    pre1[t] = acc + b1[t];
    h1[t] = silu_f(pre1[t]);
  }
  // d h1[k] = sum_a sum_t dss[a][b][t] * aff_w[a][t][k]
  float acc = 0.f;
  for (int a = 0; a < n_aff; ++a) {
    __syncthreads();
    g[t] = dss[((long long)a * B + b) * 128 + t];
    __syncthreads();
    if (t < 64) {
      const float* w = aff_w + (long long)a * 128 * 64 + t;
      for (int r = 0; r < 128; ++r) acc = fmaf(g[r], w[r * 64], acc);
    }
  }
  if (t < 64) d1[t] = acc * silu_grad_f(pre1[t]);
  __syncthreads();
  if (t < 64) {
    float a2 = 0.f;
    for (int r = 0; r < 64; ++r) a2 = fmaf(d1[r], w1[r * 64 + t], a2);
    dh0[t] = a2 * silu_grad_f(pre0[t]);
  }
  __syncthreads();
  if (t < 64) {
    float* v = vec + (long long)b * 320;
    v[t] = e[t];
    v[64 + t] = h0[t];
    v[128 + t] = h1[t];
    v[192 + t] = dh0[t];
    v[256 + t] = d1[t];
  }
}

// Pass 2: every parameter gradient is sum_b u[b][t] * v[b][k] (or sum_b u[b][t] for biases); one thread per
// output element, ordered loop over the batch.
//   job 0 .. n_aff-1 : d aff_w[a][t][k] (128 x 64) and d aff_b[a][t];  job n_aff : d w1, d b1;  job n_aff+1 : d w0, d b0
__global__ void __launch_bounds__(256)
emb_bwd_param_kernel(const float* __restrict__ vec, const float* __restrict__ dss, int n_aff, int B,
                     float* __restrict__ d_aff_w, float* __restrict__ d_aff_b, float* __restrict__ d_w1,
                     float* __restrict__ d_b1, float* __restrict__ d_w0, float* __restrict__ d_b0) {
  const int job = blockIdx.y;
  const int idx = blockIdx.x * 256 + threadIdx.x;
  if (job < n_aff) {
    if (idx >= 128 * 64) return;
    const int t = idx >> 6, k = idx & 63;
    float acc = 0.f, accb = 0.f;
    for (int b = 0; b < B; ++b) {
      const float u = dss[((long long)job * B + b) * 128 + t];
      acc = fmaf(u, vec[(long long)b * 320 + 128 + k], acc);
      accb += u;
    }
    d_aff_w[(long long)job * 8192 + idx] = acc;
    if (k == 0) d_aff_b[job * 128 + t] = accb;
  } else {
    if (idx >= 64 * 64) return;
    const int t = idx >> 6, k = idx & 63;
    const int uoff = job == n_aff ? 256 : 192, voff = job == n_aff ? 64 : 0;
    float acc = 0.f, accb = 0.f;
    for (int b = 0; b < B; ++b) {
      const float u = vec[(long long)b * 320 + uoff + t];
      acc = fmaf(u, vec[(long long)b * 320 + voff + k], acc);
      accb += u;
    }
    (job == n_aff ? d_w1 : d_w0)[idx] = acc;
    if (k == 0) (job == n_aff ? d_b1 : d_b0)[t] = accb;
  }
}

// ------------------------------------------- optimiser -------------------------------------------
__global__ void __launch_bounds__(256)
sumsq_partial_kernel(const float* __restrict__ g, long long n, double* __restrict__ partial) {
  double acc = 0.0;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float v = g[i];
    acc += (double)v * (double)v;
  }
  __shared__ double sm[256];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = sm[0];
}

// torch.optim.Adam (single-tensor path, no amsgrad, coupled weight decay) with the clip_grad_norm_ coefficient
// folded in:  g <- g * min(1, max_norm / (||g|| + 1e-6)).  norm_partial may be NULL (no clipping).
// DYN (dynamic loss scaling): norm_partial is always given and clipping runs iff max_norm > 0; a non-finite sum of
// squares is found-inf (block 0 stores it) and the step writes nothing; the bias corrections come from the applied-step
// count in device memory (*step_count + 1; mcedm_loss_scale_update advances it).
template <bool DYN = false>
__global__ void __launch_bounds__(256)
adam_step_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                 long long n, float lr, float beta1, float beta2, float eps, float weight_decay, float bc1, float bc2_sqrt,
                 const double* __restrict__ norm_partial, int n_partial, float max_norm, float grad_scale,
                 float* __restrict__ norm_out, const int* __restrict__ step_count, float* __restrict__ found_inf) {
  __shared__ float s_coef, s_bc1, s_bc2;
  __shared__ int s_skip;
  if (threadIdx.x == 0) {
    float coef = grad_scale;
    if (norm_partial) {
      double t = 0.0;
      for (int i = 0; i < n_partial; ++i) t += norm_partial[i];
      const float nrm = (float)sqrt(t) * grad_scale;
      if (!DYN || max_norm > 0.f) {
        const float c = max_norm / (nrm + 1e-6f);
        coef *= c < 1.0f ? c : 1.0f;
        if (norm_out && blockIdx.x == 0) *norm_out = nrm;
      }
      if (DYN) {
        const bool inf = !isfinite(t);
        if (blockIdx.x == 0) *found_inf = inf ? 1.0f : 0.0f;
        s_skip = inf ? 1 : 0;
        const double step = (double)(*step_count + 1);
        s_bc1 = (float)(1.0 - pow((double)beta1, step));
        s_bc2 = (float)sqrt(1.0 - pow((double)beta2, step));
      }
    }
    s_coef = coef;
  }
  __syncthreads();
  if (DYN) {
    if (s_skip) return;
    bc1 = s_bc1;
    bc2_sqrt = s_bc2;
  }
  const float coef = s_coef;
  const float step_size = lr / bc1;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    float gi = g[i] * coef;
    const float pi = p[i];
    if (weight_decay != 0.f) gi = fmaf(weight_decay, pi, gi);
    const float mi = m[i] + (gi - m[i]) * (1.0f - beta1);          // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = fmaf(1.0f - beta2, gi * gi, v[i] * beta2);    // exp_avg_sq.mul_(b2).addcmul_(g, g, 1 - b2)
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - step_size * (mi / denom);
  }
}

// torch._amp_update_scale_ (aten/src/ATen/native/cuda/AmpKernels.cu) on one thread, plus the applied-step count of the
// fused Adam: +1 when the step applied
__global__ void __launch_bounds__(32)
loss_scale_update_kernel(float* __restrict__ scale, int* __restrict__ tracker, const float* __restrict__ found_inf,
                         int* __restrict__ step_count, float growth, float backoff, int interval) {
  if (threadIdx.x != 0) return;
  if (*found_inf != 0.0f) {
    *scale = *scale * backoff;
    *tracker = 0;
    return;
  }
  if (step_count) *step_count += 1;
  const int successful = *tracker + 1;
  if (successful == interval) {
    const float grown = *scale * growth;
    if (isfinite(grown)) *scale = grown;          // never grows past fp32's range
    *tracker = 0;
  } else {
    *tracker = successful;
  }
}

// g <- g * (1 / scale): the loss scale comes off the flat gradient (power-of-two scales: exact)
__global__ void __launch_bounds__(256)
grad_unscale_kernel(float* __restrict__ g, long long n, const float* __restrict__ scale) {
  const float inv = 1.0f / *scale;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) g[i] *= inv;
}

// Gradient accumulation: acc <- (first ? 0 : acc) + alpha * g over the flat fp32 gradient, four elements per
// 128-bit access.  `first` does not read acc (a window's first micro-batch overwrites whatever the buffer held);
// otherwise one fma per element.  inf / nan in g or acc stay non-finite, so an overflowed micro-batch still makes the
// window's gradient non-finite for the loss-scaled Adam step.
__global__ void __launch_bounds__(256)
grad_accumulate_kernel(float* __restrict__ acc, const float* __restrict__ g, long long n, float alpha, int first) {
  const long long n4 = n >> 2, tid = (long long)blockIdx.x * 256 + threadIdx.x, stride = (long long)gridDim.x * 256;
  float4* acc4 = reinterpret_cast<float4*>(acc);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  for (long long i = tid; i < n4; i += stride) {
    const float4 v = g4[i];
    float4 a;
    if (first) {
      a = make_float4(alpha * v.x, alpha * v.y, alpha * v.z, alpha * v.w);
    } else {
      a = acc4[i];
      a = make_float4(fmaf(alpha, v.x, a.x), fmaf(alpha, v.y, a.y), fmaf(alpha, v.z, a.z), fmaf(alpha, v.w, a.w));
    }
    acc4[i] = a;
  }
  for (long long i = 4 * n4 + tid; i < n; i += stride) acc[i] = first ? alpha * g[i] : fmaf(alpha, g[i], acc[i]);
}

__global__ void __launch_bounds__(256)
ema_update_kernel(float* __restrict__ ema, const float* __restrict__ p, long long n, float beta) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    ema[i] = ema[i] * beta + (1.0f - beta) * p[i];                  // ddim_blocks.py:53-56
}

// Weight packing in one launch: every tensor-core operand copy of the parameters (forward layout, flipped /
// transposed data-gradient layout, permuted qkv, padded head) is a gather from the fp32 parameter storage.
// idx_a[i] = element offset from `base` (or -1: zero padding); entries [0, n16) are rounded to the 16-bit operand
// format, entries [n16, n16 + n32) stay fp32 and may add a second source (conv1 bias + skip bias).
__global__ void __launch_bounds__(256)
pack_gather_kernel(const float* __restrict__ base, const long long* __restrict__ idx_a,
                   const long long* __restrict__ idx_b, long long n16, long long n32, int fmt,
                   unsigned short* __restrict__ dst16, float* __restrict__ dst32) {
  const long long n = n16 + n32;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const long long a = idx_a[i];
    float v = a >= 0 ? base[a] : 0.0f;
    if (i < n16) {
      dst16[i] = fmt ? __half_as_ushort(__float2half_rn(v)) : __bfloat16_as_ushort(__float2bfloat16_rn(v));
    } else {
      const long long b = idx_b[i - n16];
      if (b >= 0) v = __fadd_rn(v, base[b]);
      dst32[i - n16] = v;
    }
  }
}

}  // namespace mcedm

extern "C" int mcedm_pack_gather(const float* base, const long long* idx_a, const long long* idx_b, long long n16,
                                 long long n32, int fmt, void* dst16, float* dst32, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n16 >= 0 && n32 >= 0 && n16 + n32 >= 1 && (fmt == 0 || fmt == 1), "pack_gather: bad sizes");
  int grid = (int)((n16 + n32 + 255) / 256);
  if (grid > 8 * num_sms()) grid = 8 * num_sms();
  pack_gather_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      base, idx_a, idx_b, n16, n32, fmt, reinterpret_cast<unsigned short*>(dst16), dst32);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_noise_in(const float* x, const float* noise, const float* mask, const float* sigma,
                                  const float* c_in, int B, long long chw, float* x_noise, float* x_in, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && chw >= 1, "edm_noise_in: bad sizes");
  int gx = (int)((chw + 255) / 256);
  if (gx > 64) gx = 64;
  dim3 grid(gx, B);
  edm_noise_in_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, noise, mask, sigma, c_in, chw,
                                                                                x_noise, x_in);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_mcedm_prep(const float* h, const float* u, const float* mask, const float* randn, float h_sub,
                                float h_div, float u_sub, float u_div, int B, long long HW, float* x, float* cond,
                                float* mask_c, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && HW >= 1, "mcedm_prep: bad sizes");
  const long long total = HW * B;
  mcedm_prep_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      h, u, mask, randn, h_sub, h_div, u_sub, u_div, HW, total, x, cond, mask_c);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_mcedm_prep_rows(const float* h, const float* u, const int* obs_rows, const float* randn, float h_sub,
                                    float h_div, float u_sub, float u_div, int B, int H, int W, float* x, float* cond,
                                    float* mask_c, float* mask_bhwc, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && H >= 1 && W >= 1 && obs_rows != nullptr, "mcedm_prep_rows: bad arguments");
  const long long HW = (long long)H * W, total = HW * B;
  mcedm_prep_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      h, u, obs_rows, randn, h_sub, h_div, u_sub, u_div, HW, W, total, x, cond, mask_c, mask_bhwc);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_nchw_to_nhwc_pad16(const float* a, int Ca, const float* b, int Cb, int B, int H, int W, void* dst16,
                                        int c_dst0, float scale, int op_fmt, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(Ca >= 0 && Cb >= 0 && Ca + Cb >= 1 && c_dst0 >= 0 && c_dst0 + Ca + Cb <= 64, "nchw_to_nhwc_pad: channels");
  const long long HW = (long long)H * W, total = HW * B;
  nchw_to_nhwc_pad_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      a, Ca, b, Cb, HW, total, reinterpret_cast<unsigned short*>(dst16), c_dst0, scale, op_fmt ? 1 : 0);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_nchw_to_nhwc_pad16_scaled(const float* a, int Ca, const float* b, int Cb, int B, int H, int W,
                                               void* dst16, int c_dst0, const float* scale, int op_fmt, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(Ca >= 0 && Cb >= 0 && Ca + Cb >= 1 && c_dst0 >= 0 && c_dst0 + Ca + Cb <= 64, "nchw_to_nhwc_pad: channels");
  MCEDM_REQUIRE(scale && op_fmt == MCEDM_FMT_F16_INF, "nchw_to_nhwc_pad16_scaled: needs a device scale and op_fmt 3");
  const long long HW = (long long)H * W, total = HW * B;
  nchw_to_nhwc_pad_scaled_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      a, Ca, b, Cb, HW, total, reinterpret_cast<unsigned short*>(dst16), c_dst0, scale);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_nchw_to_nhwc_pad(const float* a, int Ca, const float* b, int Cb, int B, int H, int W, void* dst_bf16,
                                      int c_dst0, void* stream) {
  return mcedm_nchw_to_nhwc_pad16(a, Ca, b, Cb, B, H, W, dst_bf16, c_dst0, 1.0f, 0, stream);
}

extern "C" int mcedm_colsum16(const void* x16, long long pixels, int C, int c_off, float* partial, int n_ctas, int op_fmt,
                              void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(pixels >= 1 && C % 8 == 0 && c_off % 8 == 0 && c_off + 64 <= C && n_ctas >= 1, "colsum16: bad sizes");
  colsum_bf16_kernel<<<n_ctas, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const unsigned short*>(x16), pixels, C, c_off, partial, op_fmt ? 1 : 0);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_colsum_bf16(const void* x_bf16, long long pixels, int C, int c_off, float* partial, int n_ctas,
                                 void* stream) {
  return mcedm_colsum16(x_bf16, pixels, C, c_off, partial, n_ctas, 0, stream);
}

extern "C" int mcedm_emb_mlp_bwd(const float* c_noise, const float* freqs, const float* w0, const float* b0,
                                 const float* w1, const float* b1, const float* aff_w, const float* dss, int n_aff,
                                 int B, float* vec_scratch, float* d_aff_w, float* d_aff_b, float* d_w1, float* d_b1,
                                 float* d_w0, float* d_b0, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && n_aff >= 1, "emb_mlp_bwd: bad sizes");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  emb_bwd_sample_kernel<<<B, 128, 0, st>>>(c_noise, freqs, w0, b0, w1, b1, aff_w, dss, n_aff, B, vec_scratch);
  MCEDM_CUDA(cudaGetLastError());
  dim3 grid(32, n_aff + 2);
  emb_bwd_param_kernel<<<grid, 256, 0, st>>>(vec_scratch, dss, n_aff, B, d_aff_w, d_aff_b, d_w1, d_b1, d_w0, d_b0);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_sumsq_partial(const float* g, long long n, double* partial, int n_partial, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n >= 1 && n_partial >= 1, "sumsq_partial: bad sizes");
  sumsq_partial_kernel<<<n_partial, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(g, n, partial);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_adam_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                               float beta2, float eps, float weight_decay, int step, const double* norm_partial,
                               int n_partial, float max_norm, float grad_scale, float* norm_out, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n >= 1 && step >= 1, "adam_step: bad sizes");
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  int grid = (int)((n + 255) / 256);
  if (grid > 4 * num_sms()) grid = 4 * num_sms();
  adam_step_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, (float)bc1, (float)sqrt(bc2), norm_partial, n_partial,
      max_norm, grad_scale, norm_out, nullptr, nullptr);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_adam_step_dyn(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                                   float beta2, float eps, float weight_decay, const int* step_count,
                                   const double* norm_partial, int n_partial, float max_norm, float grad_scale,
                                   float* norm_out, float* found_inf, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n >= 1 && n_partial >= 1 && step_count && norm_partial && found_inf, "adam_step_dyn: bad arguments");
  int grid = (int)((n + 255) / 256);
  if (grid > 4 * num_sms()) grid = 4 * num_sms();
  adam_step_kernel<true><<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, 1.0f, 1.0f, norm_partial, n_partial, max_norm, grad_scale,
      norm_out, step_count, found_inf);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_loss_scale_update(float* scale, int* growth_tracker, const float* found_inf, int* step_count,
                                       float growth_factor, float backoff_factor, int growth_interval, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(scale && growth_tracker && found_inf && growth_interval >= 1, "loss_scale_update: bad arguments");
  loss_scale_update_kernel<<<1, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      scale, growth_tracker, found_inf, step_count, growth_factor, backoff_factor, growth_interval);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_grad_unscale(float* g, long long n, const float* scale, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n >= 1 && scale, "grad_unscale: bad arguments");
  int grid = (int)((n + 255) / 256);
  if (grid > 4 * num_sms()) grid = 4 * num_sms();
  grad_unscale_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(g, n, scale);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_grad_accumulate(float* acc, const float* g, long long n, float alpha, int first, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(acc && g && n >= 1, "grad_accumulate: bad arguments");
  MCEDM_REQUIRE(((reinterpret_cast<uintptr_t>(acc) | reinterpret_cast<uintptr_t>(g)) & 15) == 0,
                "grad_accumulate: buffers must be 16-byte aligned");
  int grid = (int)((n / 4 + 255) / 256);
  if (grid < 1) grid = 1;
  if (grid > 8 * num_sms()) grid = 8 * num_sms();
  grad_accumulate_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(acc, g, n, alpha, first);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_ema_update(float* ema, const float* p, long long n, float beta, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n >= 1, "ema_update: bad sizes");
  int grid = (int)((n + 255) / 256);
  if (grid > 4 * num_sms()) grid = 4 * num_sms();
  ema_update_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(ema, p, n, beta);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}
