// K5 — EDM stochastic-Heun sampler state updates with observed-state mask blending, and the EDM
// preconditioning arithmetic around the network (K4), fused into three elementwise kernels per step.
//
// Replaces the ~25 fp64 torch elementwise launches per step of PlMcedm.sample_edm
// (models/mcedm.py:594-628) and the preconditioning of PlMcedm.get_denoised (models/mcedm.py:443-461).
// The sampler state is fp64 NCHW [B,C,H,W] exactly as in the reference; the network I/O is fp32.
// Every arithmetic step mirrors the reference's torch expression order with explicit round-to-nearest
// intrinsics (no FMA contraction), so the fp64 updates are bit-reproducible against torch and pixels
// with mask == 0 keep their observed value bit-exactly for the whole trajectory.
//
// HBM-bound: ~60-100 B per element per kernel, 128-bit accesses where the dtype allows.
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

#include <cmath>

namespace mcedm {

// x0 = known*(1-m) [fp32 product, as torch computes it on fp32 tensors]  +  (double(noise)*t0) * m
// known = cond[:, :C] of a [B,Ccond,H,W] tensor (models/mcedm.py:590-597)
__global__ void edm_init_kernel(const float* __restrict__ noise, const float* __restrict__ cond, int Ccond, int C,
                                long long HW, const float* __restrict__ mask, double t0, long long total,
                                double* __restrict__ x) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long chw = (long long)C * HW;
  const long long b = i / chw, r = i - b * chw;
  const float m = mask[i];
  const float known = cond[b * (long long)Ccond * HW + r];
  const float t1 = __fmul_rn(known, __fsub_rn(1.0f, m));
  const double t2 = __dmul_rn(__dmul_rn((double)noise[i], t0), (double)m);
  x[i] = __dadd_rn((double)t1, t2);
}

// Classifier-free guidance (CFG): the network runs once on a batch of 2B rows, rows [0, B) with the condition and
// rows [B, 2B) with the all-zero condition, so F holds [F_c | F_u] with F_u starting `total` elements after F_c.
// Every kernel below that reads F takes a CFG flag and reads the guided output
//   F_w = (1+w)*F_c - w*F_u    (fp32; two products and one difference, each rounded: no FMA)
// in place of F; the CFG = false instantiation is the unguided kernel, with the same arithmetic as before.
// w_c = float(1+w) and w_u = float(w) are rounded on the host, so w = 0 gives the bits of F_c and w = -1 those of F_u.
template <bool CFG>
__device__ __forceinline__ float net_out(const float* __restrict__ F, long long i, long long total, float w_c,
                                         float w_u) {
  if constexpr (CFG) return __fsub_rn(__fmul_rn(w_c, F[i]), __fmul_rn(w_u, F[total + i]));
  else return F[i];
}

// x_hat = x_cur + ((coef * S_noise) * eps) * m ;  x_in = float(x_hat) * c_in   (models/mcedm.py:607-608, 444, 454)
// (CFG: x_in also to the unconditional half)
template <bool CFG>
__global__ void edm_churn_kernel(const double* __restrict__ x_cur, const double* __restrict__ eps,
                                 const float* __restrict__ mask, double coef, float c_in, long long total,
                                 double* __restrict__ x_hat, float* __restrict__ x_in) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const double xh = __dadd_rn(x_cur[i], __dmul_rn(__dmul_rn(coef, eps[i]), (double)mask[i]));
  x_hat[i] = xh;
  const float xi = __fmul_rn(c_in, (float)xh);
  x_in[i] = xi;
  if constexpr (CFG) x_in[total + i] = xi;
}

// D = c_skip*float(x_hat) + c_out*F (fp32) ; d_cur = (x_hat - double(D)) / t_hat ;
// x_next = x_hat + ((t_next - t_hat) * d_cur) * m ; x_in = float(x_next) * c_in_next   (models/mcedm.py:612-618)
// (CFG: F_w in place of F, x_in to both halves)
template <bool CFG>
__global__ void edm_euler_kernel(const double* __restrict__ x_hat, const float* __restrict__ F,
                                 const float* __restrict__ mask, double t_hat, double dt, float c_skip, float c_out,
                                 float c_in_next, float w_c, float w_u, long long total, double* __restrict__ d_cur,
                                 double* __restrict__ x_next, float* __restrict__ x_in, float* __restrict__ D_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const double xh = x_hat[i];
  const float D = __fadd_rn(__fmul_rn(c_skip, (float)xh), __fmul_rn(c_out, net_out<CFG>(F, i, total, w_c, w_u)));
  const double d = __ddiv_rn(__dsub_rn(xh, (double)D), t_hat);
  const double xn = __dadd_rn(xh, __dmul_rn(__dmul_rn(dt, d), (double)mask[i]));
  d_cur[i] = d;
  x_next[i] = xn;
  if (x_in) {
    const float xi = __fmul_rn(c_in_next, (float)xn);
    x_in[i] = xi;
    if constexpr (CFG) x_in[total + i] = xi;
  }
  if (D_out) D_out[i] = D;
}

// D2 = c_skip*float(x_e) + c_out*F2 ; d' = (x_e - double(D2)) / t_next ;
// x_next = x_hat + ((t_next - t_hat) * (0.5*d_cur + 0.5*d')) * m     (models/mcedm.py:621-628)
template <bool CFG>
__global__ void edm_correct_kernel(const double* __restrict__ x_hat, const double* __restrict__ x_e,
                                   const float* __restrict__ F2, const double* __restrict__ d_cur,
                                   const float* __restrict__ mask, double t_next, double dt, float c_skip,
                                   float c_out, float w_c, float w_u, long long total, double* __restrict__ x_next,
                                   float* __restrict__ D_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const double xe = x_e[i];
  const float D = __fadd_rn(__fmul_rn(c_skip, (float)xe), __fmul_rn(c_out, net_out<CFG>(F2, i, total, w_c, w_u)));
  const double dp = __ddiv_rn(__dsub_rn(xe, (double)D), t_next);
  const double avg = __dadd_rn(__dmul_rn(0.5, d_cur[i]), __dmul_rn(0.5, dp));
  x_next[i] = __dadd_rn(x_hat[i], __dmul_rn(__dmul_rn(dt, avg), (double)mask[i]));
  if (D_out) D_out[i] = D;
}

// D = c_skip[b]*x + c_out[b]*F with per-sample coefficients (training-time preconditioning,
// models/mcedm.py:203-210); also used by get_denoised with a single sigma (stride 0).  CFG: F_w in place of F, and
// F_w itself to F_out (get_denoised returns it)
template <bool CFG>
__global__ void edm_precond_out_kernel(const float* __restrict__ x, const float* __restrict__ F,
                                       const float* __restrict__ c_skip, const float* __restrict__ c_out,
                                       int coef_stride, float w_c, float w_u, long long chw, long long total,
                                       float* __restrict__ D, float* __restrict__ F_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long b = i / chw;
  const float f = net_out<CFG>(F, i, total, w_c, w_u);
  D[i] = __fadd_rn(__fmul_rn(c_skip[b * coef_stride], x[i]), __fmul_rn(c_out[b * coef_stride], f));
  if constexpr (CFG) F_out[i] = f;
}

// x_in = c_in[b] * x  (network input scaling, models/mcedm.py:208, :454)
__global__ void edm_precond_in_kernel(const float* __restrict__ x, const float* __restrict__ c_in, int coef_stride,
                                      long long chw, long long total, float* __restrict__ x_in) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  x_in[i] = __fmul_rn(c_in[(i / chw) * coef_stride], x[i]);
}

// ---- PDE-guided variants (PlCondDdim.sample_edm with guide_dx, models/ddim.py:1566-1590) -------------------------
// D = c_skip*float(x) + c_out*F, materialised because the guidance gradient is a stencil over D  (ddim.py:1756-1766)
// (CFG: F_w in place of F)
template <bool CFG>
__global__ void edm_denoised_kernel(const double* __restrict__ x, const float* __restrict__ F, float c_skip, float c_out,
                                    float w_c, float w_u, long long total, float* __restrict__ D) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  D[i] = __fadd_rn(__fmul_rn(c_skip, (float)x[i]), __fmul_rn(c_out, net_out<CFG>(F, i, total, w_c, w_u)));
}

// d_cur = (x_hat - double(D))/t_hat - double((5*dx)/float(t_hat)) ; x_next = x_hat + ((t_next - t_hat)*d_cur)*m
// (`weight * dx / t_hat` is a float32 tensor divided by a 0-dim float64 tensor: evaluated in float32, ddim.py:1571)
__global__ void edm_euler_guided_kernel(const double* __restrict__ x_hat, const float* __restrict__ D,
                                        const float* __restrict__ gdx, const float* __restrict__ mask, double t_hat,
                                        float t_div, double dt, float c_in_next, long long total,
                                        double* __restrict__ d_cur, double* __restrict__ x_next,
                                        float* __restrict__ x_in) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const double xh = x_hat[i];
  const float gterm = __fdiv_rn(__fmul_rn(5.0f, gdx[i]), t_div);
  const double d = __dsub_rn(__ddiv_rn(__dsub_rn(xh, (double)D[i]), t_hat), (double)gterm);
  const double xn = __dadd_rn(xh, __dmul_rn(__dmul_rn(dt, d), (double)mask[i]));
  d_cur[i] = d;
  x_next[i] = xn;
  if (x_in) x_in[i] = __fmul_rn(c_in_next, (float)xn);
}

// d' = (x_e - double(D2))/t_next - double((5*dx2)/float(t_hat))   [t_hat, not t_next: ddim.py:1590]
__global__ void edm_correct_guided_kernel(const double* __restrict__ x_hat, const double* __restrict__ x_e,
                                          const float* __restrict__ D2, const float* __restrict__ gdx,
                                          const double* __restrict__ d_cur, const float* __restrict__ mask,
                                          double t_next, float t_div, double dt, long long total,
                                          double* __restrict__ x_next) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float gterm = __fdiv_rn(__fmul_rn(5.0f, gdx[i]), t_div);
  const double dp = __dsub_rn(__ddiv_rn(__dsub_rn(x_e[i], (double)D2[i]), t_next), (double)gterm);
  const double avg = __dadd_rn(__dmul_rn(0.5, d_cur[i]), __dmul_rn(0.5, dp));
  x_next[i] = __dadd_rn(x_hat[i], __dmul_rn(__dmul_rn(dt, avg), (double)mask[i]));
}

// ---- RePaint-style known-region handling of PlDdim.sample_edm (models/ddim.py:959-1051) ---------------------------
// x0 = double( (hu*sa + noise*s1)*m + noise*(1-m) ) * t0 ; sa = sqrt(alpha_bar(t0)), s1 = sqrt(1 - alpha_bar(t0))
// float32 up to the cast, as torch evaluates :987-993 (mask == 1 means KNOWN here, the opposite of PlMcedm)
__global__ void edm_vp_init_kernel(const float* __restrict__ hu, const float* __restrict__ noise,
                                   const float* __restrict__ mask, float sa, float s1, double t0, long long total,
                                   double* __restrict__ x) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float m = mask[i], n = noise[i];
  const float known = __fadd_rn(__fmul_rn(hu[i], sa), __fmul_rn(n, s1));
  const float x32 = __fadd_rn(__fmul_rn(known, m), __fmul_rn(n, __fsub_rn(1.0f, m)));
  x[i] = __dmul_rn((double)x32, t0);
}

// x = double((sa*hu + s1*noise)*m) + x*double(1-m)   (replace the known part, :1029-1031; sa = 1, s1 = 0 gives the
// final `hu*m + x*(1-m)` of :1040-1041 exactly)
__global__ void edm_repaint_blend_kernel(const float* __restrict__ hu, const float* __restrict__ noise,
                                         const float* __restrict__ mask, float sa, float s1, long long total,
                                         double* __restrict__ x) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float m = mask[i];
  const float known = __fadd_rn(__fmul_rn(sa, hu[i]), __fmul_rn(s1, noise[i]));
  x[i] = __dadd_rn((double)__fmul_rn(known, m), __dmul_rn(x[i], (double)__fsub_rn(1.0f, m)));
}

static inline unsigned blocks_for(long long total) { return (unsigned)((total + 255) / 256); }

// ---- DDIM sampler with known-region replacement and repeats: PlDdim.sample_with_repeat (models/ddim.py:808-913) -------
// fp32 state, every operation in torch's evaluation order (explicit _rn intrinsics: bit-identical to the expressions).
// x = (hu*sa + noise*s1)*mask + noise*(1-mask)    (:842-843; sa = sqrt(a_T-1), s1 = sqrt(1 - a_T-1); mask == 1 KNOWN)
__global__ void ddim_init_kernel(const float* __restrict__ hu, const float* __restrict__ noise,
                                 const float* __restrict__ mask, float sa, float s1, long long total,
                                 float* __restrict__ x) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float m = mask[i], nz = noise[i];
  const float known = __fadd_rn(__fmul_rn(hu[i], sa), __fmul_rn(nz, s1));
  x[i] = __fadd_rn(__fmul_rn(known, m), __fmul_rn(nz, __fsub_rn(1.0f, m)));
}

// x0 = (xt - et*s1)/sa ; x0 = hu*mask + x0*(1-mask) ; optionally xt' = sa*x0 + s1*et   (:876-883)
__global__ void ddim_x0_kernel(const float* __restrict__ xt, const float* __restrict__ et, const float* __restrict__ hu,
                               const float* __restrict__ mask, float sa, float s1, long long total,
                               float* __restrict__ x0_out, float* __restrict__ xt_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float m = mask[i], e = et[i];
  float x0 = __fdiv_rn(__fsub_rn(xt[i], __fmul_rn(e, s1)), sa);
  x0 = __fadd_rn(__fmul_rn(hu[i], m), __fmul_rn(x0, __fsub_rn(1.0f, m)));
  x0_out[i] = x0;
  if (xt_out) xt_out[i] = __fadd_rn(__fmul_rn(sa, x0), __fmul_rn(s1, e));
}

// xt_next = sa_n*x0 [+ c1*rand] + c2*et ; known = sa_n*hu + c2*noise ; x = known*mask + xt_next*(1-mask)   (:885-895)
__global__ void ddim_next_kernel(const float* __restrict__ x0, const float* __restrict__ et, const float* __restrict__ hu,
                                 const float* __restrict__ noise, const float* __restrict__ mask,
                                 const float* __restrict__ rnd, float sa_n, float c1, float c2, long long total,
                                 float* __restrict__ x_next) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float m = mask[i];
  float xn = __fmul_rn(sa_n, x0[i]);
  if (rnd) xn = __fadd_rn(xn, __fmul_rn(c1, rnd[i]));
  xn = __fadd_rn(xn, __fmul_rn(c2, et[i]));
  const float known = __fadd_rn(__fmul_rn(sa_n, hu[i]), __fmul_rn(c2, noise[i]));
  x_next[i] = __fadd_rn(__fmul_rn(known, m), __fmul_rn(xn, __fsub_rn(1.0f, m)));
}

}  // namespace mcedm

extern "C" int mcedm_edm_init(const float* noise, const float* cond, int Ccond, const float* mask, double t0, int B,
                              int C, int H, int W, double* x, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(Ccond >= C && C >= 1, "edm_init: cond has %d channels, state has %d", Ccond, C);
  const long long HW = (long long)H * W, total = (long long)B * C * HW;
  edm_init_kernel<<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(noise, cond, Ccond, C, HW,
                                                                                         mask, t0, total, x);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_churn(const double* x_cur, const double* eps, const float* mask, double coef, float c_in,
                               long long total, double* x_hat, float* x_in, void* stream) {
  using namespace mcedm;
  edm_churn_kernel<false><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x_cur, eps, mask, coef, c_in,
                                                                                          total, x_hat, x_in);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_euler(const double* x_hat, const float* F, const float* mask, double t_hat, double t_next,
                               float c_skip, float c_out, float c_in_next, long long total, double* d_cur,
                               double* x_next, float* x_in, float* D_out, void* stream) {
  using namespace mcedm;
  edm_euler_kernel<false><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x_hat, F, mask, t_hat, t_next - t_hat, c_skip, c_out, c_in_next, 1.0f, 0.0f, total, d_cur, x_next, x_in, D_out);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_correct(const double* x_hat, const double* x_e, const float* F2, const double* d_cur,
                                 const float* mask, double t_hat, double t_next, float c_skip, float c_out,
                                 long long total, double* x_next, float* D_out, void* stream) {
  using namespace mcedm;
  edm_correct_kernel<false><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x_hat, x_e, F2, d_cur, mask, t_next, t_next - t_hat, c_skip, c_out, 1.0f, 0.0f, total, x_next, D_out);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_precond_out(const float* x, const float* F, const float* c_skip, const float* c_out,
                                     int coef_stride, int B, long long chw, float* D, void* stream) {
  using namespace mcedm;
  const long long total = (long long)B * chw;
  edm_precond_out_kernel<false><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, F, c_skip, c_out, coef_stride, 1.0f, 0.0f, chw, total, D, nullptr);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_precond_in(const float* x, const float* c_in, int coef_stride, int B, long long chw,
                                    float* x_in, void* stream) {
  using namespace mcedm;
  const long long total = (long long)B * chw;
  edm_precond_in_kernel<<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, c_in, coef_stride,
                                                                                               chw, total, x_in);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_denoised(const double* x, const float* F, float c_skip, float c_out, long long total, float* D,
                                  void* stream) {
  using namespace mcedm;
  edm_denoised_kernel<false><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, F, c_skip, c_out, 1.0f, 0.0f, total, D);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

// ---- classifier-free guidance: F = [F_c | F_u] of a 2B-row network batch; w is rounded to fp32 here --------------
static inline void cfg_weights(double w, float* w_c, float* w_u) {
  *w_c = (float)(1.0 + w);
  *w_u = (float)w;
}

extern "C" int mcedm_edm_churn_cfg(const double* x_cur, const double* eps, const float* mask, double coef, float c_in,
                                   long long total, double* x_hat, float* x_in, void* stream) {
  using namespace mcedm;
  edm_churn_kernel<true><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x_cur, eps, mask, coef, c_in, total, x_hat, x_in);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_euler_cfg(const double* x_hat, const float* F, const float* mask, double t_hat, double t_next,
                                   float c_skip, float c_out, float c_in_next, double w, long long total, double* d_cur,
                                   double* x_next, float* x_in, float* D_out, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(std::isfinite(w), "edm_euler_cfg: guidance weight is not finite");
  float w_c, w_u;
  cfg_weights(w, &w_c, &w_u);
  edm_euler_kernel<true><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x_hat, F, mask, t_hat, t_next - t_hat, c_skip, c_out, c_in_next, w_c, w_u, total, d_cur, x_next, x_in, D_out);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_correct_cfg(const double* x_hat, const double* x_e, const float* F2, const double* d_cur,
                                     const float* mask, double t_hat, double t_next, float c_skip, float c_out, double w,
                                     long long total, double* x_next, float* D_out, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(std::isfinite(w), "edm_correct_cfg: guidance weight is not finite");
  float w_c, w_u;
  cfg_weights(w, &w_c, &w_u);
  edm_correct_kernel<true><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x_hat, x_e, F2, d_cur, mask, t_next, t_next - t_hat, c_skip, c_out, w_c, w_u, total, x_next, D_out);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_denoised_cfg(const double* x, const float* F, float c_skip, float c_out, double w,
                                      long long total, float* D, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(std::isfinite(w), "edm_denoised_cfg: guidance weight is not finite");
  float w_c, w_u;
  cfg_weights(w, &w_c, &w_u);
  edm_denoised_kernel<true><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, F, c_skip, c_out, w_c, w_u, total, D);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_precond_out_cfg(const float* x, const float* F, const float* c_skip, const float* c_out,
                                         int coef_stride, double w, int B, long long chw, float* D, float* F_w,
                                         void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(std::isfinite(w), "edm_precond_out_cfg: guidance weight is not finite");
  float w_c, w_u;
  cfg_weights(w, &w_c, &w_u);
  const long long total = (long long)B * chw;
  edm_precond_out_kernel<true><<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, F, c_skip, c_out, coef_stride, w_c, w_u, chw, total, D, F_w);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_euler_guided(const double* x_hat, const float* D, const float* gdx, const float* mask,
                                      double t_hat, double t_next, float c_in_next, long long total, double* d_cur,
                                      double* x_next, float* x_in, void* stream) {
  using namespace mcedm;
  edm_euler_guided_kernel<<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x_hat, D, gdx, mask, t_hat, (float)t_hat, t_next - t_hat, c_in_next, total, d_cur, x_next, x_in);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_correct_guided(const double* x_hat, const double* x_e, const float* D2, const float* gdx,
                                        const double* d_cur, const float* mask, double t_hat, double t_next,
                                        long long total, double* x_next, void* stream) {
  using namespace mcedm;
  edm_correct_guided_kernel<<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x_hat, x_e, D2, gdx, d_cur, mask, t_next, (float)t_hat, t_next - t_hat, total, x_next);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_vp_init(const float* hu, const float* noise, const float* mask, float sqrt_a, float sqrt_1ma,
                                 double t0, long long total, double* x, void* stream) {
  using namespace mcedm;
  edm_vp_init_kernel<<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(hu, noise, mask, sqrt_a,
                                                                                            sqrt_1ma, t0, total, x);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_edm_repaint_blend(const float* hu, const float* noise, const float* mask, float sqrt_a,
                                       float sqrt_1ma, long long total, double* x, void* stream) {
  using namespace mcedm;
  edm_repaint_blend_kernel<<<blocks_for(total), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      hu, noise, mask, sqrt_a, sqrt_1ma, total, x);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_ddim_init(const float* hu, const float* noise, const float* known_mask, float sqrt_a, float sqrt_1ma,
                               long long total, float* x, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(total >= 1, "ddim_init: empty");
  ddim_init_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      hu, noise, known_mask, sqrt_a, sqrt_1ma, total, x);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_ddim_x0(const float* xt, const float* et, const float* hu, const float* known_mask, float sqrt_a,
                             float sqrt_1ma, long long total, float* x0_out, float* xt_out, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(total >= 1, "ddim_x0: empty");
  ddim_x0_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      xt, et, hu, known_mask, sqrt_a, sqrt_1ma, total, x0_out, xt_out);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int mcedm_ddim_next(const float* x0, const float* et, const float* hu, const float* noise,
                               const float* known_mask, const float* rand_or_null, float sqrt_a_next, float c1, float c2,
                               long long total, float* x_next, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(total >= 1, "ddim_next: empty");
  ddim_next_kernel<<<(unsigned)((total + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x0, et, hu, noise, known_mask, rand_or_null, sqrt_a_next, c1, c2, total, x_next);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}
