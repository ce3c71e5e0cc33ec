// K3-bwd — backward of the fused self-attention (attn.cu) on tcgen05.
//
// Autograd of AttentionOp (models/adm_blocks.py:103-118: forward softmax(q.k/8) in fp32, backward through
// torch._softmax_backward_data) and of the value einsum (:178).  With P = softmax(Q K^T / 8) saved only as
// its row-wise base-2 log-sum-exp (lse, written by attn_kernel) and D_i = sum_c dO[i,c] O[i,c]:
//
//     dV = P^T dO          dP = dO V^T          dS = P o (dP - D) / 8          dQ = dS K          dK = dS^T Q
//
// P and dS are L x L per sample (4 MB each in fp32 at L = 1024) and are recomputed tile by tile from Q, K, V
// on the tensor cores; they never reach HBM.  Two kernels from one template, one CTA per 128-row block:
//
//   MODE 0 (dQ)     : fixed X1 = Q_i, X2 = dO_i ; streamed Y1 = K_j, Y2 = V_j ; rows = queries
//                     T1 = X1 Y1^T = S,  T2 = X2 Y2^T = dP,  acc2 += dS Y1                (-> dQ_i)
//   MODE 1 (dK, dV) : fixed X1 = K_j, X2 = V_j  ; streamed Y1 = Q_i, Y2 = dO_i ; rows = keys
//                     T1 = S^T,  T2 = dP^T,  acc1 += P^T Y2 (-> dV_j),  acc2 += dS^T Y1     (-> dK_j)
//
// Each needs no atomics and no cross-CTA reduction (results are deterministic); the price is that S and dP are
// computed twice.  Attention is ~2 % of the network's FLOPs.
//   warp 0 : TMA producer (X tiles once, Y tiles through a 3-stage ring)
//   warp 1 : MMA issuer; T1/T2 of block it+1 are issued before the accumulating MMAs of block it, so the
//            element-wise warps never wait for the tensor pipe longer than one block
//   warps 2-5 : one T row per thread: P / dS -> bf16 -> SWIZZLE_128B K-major smem operand tiles
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

#include <cuda_bf16.h>

namespace mcedm {

constexpr int kBStages = 3;
constexpr int kBTile = 16384;   // 128 rows x 128 B

__device__ __forceinline__ float ex2b(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// D[b, i] = sum_c dO[b,i,c] * O[b,i,c]; one thread per (b, i) row of 64 bf16 (128 B).
__global__ void attn_bwd_prep_kernel(const uint4* __restrict__ o, const uint4* __restrict__ d_o, long long rows,
                                     float* __restrict__ dvec, int fmt) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float acc = 0.f;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const uint4 a = o[r * 8 + u], g = d_o[r * 8 + u];
    if (fmt) {
      const uint32_t av[4] = {a.x, a.y, a.z, a.w}, gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 x = unpack_f16x2(av[k]), y = unpack_f16x2(gv[k]);
        acc += x.x * y.x + x.y * y.y;
      }
      continue;
    }
    acc += bf16_lo(a.x) * bf16_lo(g.x) + bf16_hi(a.x) * bf16_hi(g.x);
    acc += bf16_lo(a.y) * bf16_lo(g.y) + bf16_hi(a.y) * bf16_hi(g.y);
    acc += bf16_lo(a.z) * bf16_lo(g.z) + bf16_hi(a.z) * bf16_hi(g.z);
    acc += bf16_lo(a.w) * bf16_lo(g.w) + bf16_hi(a.w) * bf16_hi(g.w);
  }
  dvec[r] = acc;
}

struct AttnBwdParams {
  int L;
  const float* lse;     // [B, L]
  const float* dvec;    // [B, L]
  __nv_bfloat16* out1;  // MODE 1: dV ; MODE 0: unused
  __nv_bfloat16* out2;  // MODE 1: dK ; MODE 0: dQ
  unsigned int* err;
  int fmt;              // 16-bit format of every operand / output: 0 bf16, 1 fp16
};

// INF: the dS tiles and the dQ / dK / dV stores in fp16 without saturation (op_fmt MCEDM_FMT_F16_INF)
template <int MODE, bool INF = false>
__global__ void __launch_bounds__(192, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_do,
                const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* x_smem = smem;                                   // X1 | X2            (32 KB)
  uint8_t* y_smem = x_smem + 2 * kBTile;                    // stages x (Y1 | Y2) (96 KB)
  uint8_t* p_smem = y_smem + kBStages * 2 * kBTile;         // P  : 2 atoms of 64 (32 KB), MODE 1 only
  uint8_t* ds_smem = p_smem + 2 * kBTile;                   // dS : 2 atoms of 64 (32 KB)
  float* col_stats = reinterpret_cast<float*>(ds_smem + 2 * kBTile);   // MODE 1: 2 buffers x (lse[128] | D[128])
  uint64_t* bars = reinterpret_cast<uint64_t*>(col_stats + 2 * 256);
  uint64_t* x_full = bars;
  uint64_t* acc_full = bars + 1;
  uint64_t* t_full = bars + 2;
  uint64_t* t_empty = bars + 3;
  uint64_t* p_full = bars + 4;
  uint64_t* p_empty = bars + 5;
  uint64_t* y_full = bars + 6;
  uint64_t* y_empty = bars + 6 + kBStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6 + 2 * kBStages);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = p.L / 128;
  const int b = blockIdx.x / nblk;
  const int r0 = (blockIdx.x - b * nblk) * 128;    // first row (query for MODE 0, key for MODE 1) of this CTA

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_qkv);
    prefetch_tmap(&tm_do);
    mbar_init(x_full, 1);
    mbar_init(acc_full, 1);
    mbar_init(t_full, 1);
    mbar_init(t_empty, 128);
    mbar_init(p_full, 128);
    mbar_init(p_empty, 1);
    for (int i = 0; i < kBStages; ++i) {
      mbar_init(&y_full[i], 1);
      mbar_init(&y_empty[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_t1 = tmem_base, tmem_t2 = tmem_base + 128;
  const uint32_t tmem_acc1 = tmem_base + 256, tmem_acc2 = tmem_base + 320;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(x_full, 2 * kBTile);
      if (MODE == 0) {
        tma_load_4d(x_smem, &tm_qkv, x_full, 0, r0, 0, b);                // Q_i
        tma_load_4d(x_smem + kBTile, &tm_do, x_full, 0, r0, 0, b);        // dO_i
      } else {
        tma_load_4d(x_smem, &tm_qkv, x_full, 64, r0, 0, b);               // K_j
        tma_load_4d(x_smem + kBTile, &tm_qkv, x_full, 128, r0, 0, b);     // V_j
      }
      for (int it = 0; it < nblk; ++it) {
        const uint32_t s = it % kBStages, n = it / kBStages;
        mbar_wait(&y_empty[s], (n & 1u) ^ 1u, p.err, 0x5100 + s);
        mbar_expect_tx(&y_full[s], 2 * kBTile);
        uint8_t* dst = y_smem + s * 2 * kBTile;
        if (MODE == 0) {
          tma_load_4d(dst, &tm_qkv, &y_full[s], 64, it * 128, 0, b);            // K_j
          tma_load_4d(dst + kBTile, &tm_qkv, &y_full[s], 128, it * 128, 0, b);  // V_j
        } else {
          tma_load_4d(dst, &tm_qkv, &y_full[s], 0, it * 128, 0, b);             // Q_i
          tma_load_4d(dst + kBTile, &tm_do, &y_full[s], 0, it * 128, 0, b);     // dO_i
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc_t = umma_idesc_16(128, 128, 0, 0, p.fmt);
    const uint32_t idesc_acc = umma_idesc_16(128, 64, 0, 1, p.fmt);    // B = streamed tile, MN-major
    mbar_wait(x_full, 0, p.err, 0x5200);
    tc_fence_after();
    const uint64_t x1d = umma_desc_k_sw128(smem_u32(x_smem));
    const uint64_t x2d = umma_desc_k_sw128(smem_u32(x_smem + kBTile));
    const uint32_t p_base = smem_u32(p_smem), ds_base = smem_u32(ds_smem);
    for (int it = 0; it <= nblk; ++it) {
      if (it < nblk) {
        const uint32_t s = it % kBStages, n = it / kBStages;
        mbar_wait(&y_full[s], n & 1u, p.err, 0x5300 + s);
        mbar_wait(t_empty, ((uint32_t)it & 1u) ^ 1u, p.err, 0x5400);
        tc_fence_after();
        const uint64_t y1d = umma_desc_k_sw128(smem_u32(y_smem + s * 2 * kBTile));
        const uint64_t y2d = umma_desc_k_sw128(smem_u32(y_smem + s * 2 * kBTile + kBTile));
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16(tmem_t1, x1d + 2 * k, y1d + 2 * k, idesc_t, (uint32_t)(k != 0));
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16(tmem_t2, x2d + 2 * k, y2d + 2 * k, idesc_t, (uint32_t)(k != 0));
          umma_commit(t_full);
        }
        __syncwarp();
      }
      if (it >= 1) {
        const int jp = it - 1;
        const uint32_t sp = jp % kBStages;
        mbar_wait(p_full, (uint32_t)jp & 1u, p.err, 0x5500);
        tc_fence_after();
        const uint32_t y1 = smem_u32(y_smem + sp * 2 * kBTile), y2 = y1 + kBTile;
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const uint32_t koff = (kk >> 2) * kBTile + (kk & 3) * 32;
            if (MODE == 1)
              umma_f16(tmem_acc1, umma_desc_k_sw128(p_base + koff), umma_desc_mn_sw128(y2 + kk * 2048, 8192), idesc_acc,
                       (uint32_t)((jp | kk) != 0));
            umma_f16(tmem_acc2, umma_desc_k_sw128(ds_base + koff), umma_desc_mn_sw128(y1 + kk * 2048, 8192), idesc_acc,
                     (uint32_t)((jp | kk) != 0));
          }
          umma_commit(p_empty);
          umma_commit(&y_empty[sp]);
        }
        __syncwarp();
      }
    }
    if (elect_one()) umma_commit(acc_full);
    __syncwarp();
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int tid = threadIdx.x - 64;     // 0..127
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float c1 = 0.125f * 1.4426950408889634f;
    float row_lse = 0.f, row_d = 0.f;
    if (MODE == 0) {
      row_lse = p.lse[(long long)b * p.L + r0 + row];
      row_d = p.dvec[(long long)b * p.L + r0 + row];
    }
    for (int it = 0; it < nblk; ++it) {
      float* cs = col_stats + (it & 1) * 256;
      if (MODE == 1) {
        // statistics of the 128 streamed queries (columns of T1/T2); double-buffered by block parity
        cs[tid] = p.lse[(long long)b * p.L + it * 128 + tid];
        cs[128 + tid] = p.dvec[(long long)b * p.L + it * 128 + tid];
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      mbar_wait(t_full, (uint32_t)it & 1u, p.err, 0x5600);
      mbar_wait(p_empty, ((uint32_t)it & 1u) ^ 1u, p.err, 0x5700);
      tc_fence_after();
      uint8_t* prow = p_smem + row * 128;
      uint8_t* dsrow = ds_smem + row * 128;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t s[32], g[32];
        tmem_ld_x32(tmem_t1 + lane_addr + c * 32, s);
        tmem_ld_x32(tmem_t2 + lane_addr + c * 32, g);
        tmem_wait_ld();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint4 po, dso;
          uint32_t* pp = reinterpret_cast<uint32_t*>(&po);
          uint32_t* dp = reinterpret_cast<uint32_t*>(&dso);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int i0 = u * 8 + 2 * e;
            float l0 = row_lse, l1 = row_lse, d0 = row_d, d1 = row_d;
            if (MODE == 1) {
              l0 = cs[c * 32 + i0];
              l1 = cs[c * 32 + i0 + 1];
              d0 = cs[128 + c * 32 + i0];
              d1 = cs[128 + c * 32 + i0 + 1];
            }
            const float p0 = ex2b(fmaf(__uint_as_float(s[i0]), c1, -l0));
            const float p1 = ex2b(fmaf(__uint_as_float(s[i0 + 1]), c1, -l1));
            const float ds0 = p0 * (__uint_as_float(g[i0]) - d0) * 0.125f;
            const float ds1 = p1 * (__uint_as_float(g[i0 + 1]) - d1) * 0.125f;
            pp[e] = pack_op2(p0, p1, p.fmt);
            dp[e] = pack_op2_g<INF>(ds0, ds1, p.fmt);
          }
          const int unit = ((c & 1) * 4 + u) ^ (row & 7);
          if (MODE == 1) *reinterpret_cast<uint4*>(prow + (c >> 1) * kBTile + unit * 16) = po;
          *reinterpret_cast<uint4*>(dsrow + (c >> 1) * kBTile + unit * 16) = dso;
        }
      }
      tc_fence_before();
      mbar_arrive(t_empty);
      fence_proxy_async_smem();
      mbar_arrive(p_full);
    }
    // ---------------- epilogue: accumulators -> bf16 ----------------
    mbar_wait(acc_full, 0, p.err, 0x5800);
    tc_fence_after();
    const long long orow = ((long long)b * p.L + r0 + row) * 64;
#pragma unroll 1
    for (int a = (MODE == 1 ? 0 : 1); a < 2; ++a) {
      __nv_bfloat16* dst = (a == 0 ? p.out1 : p.out2) + orow;
      const uint32_t tacc = a == 0 ? tmem_acc1 : tmem_acc2;
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t v[32];
        tmem_ld_x32(tacc + lane_addr + c * 32, v);
        tmem_wait_ld();
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint4 o;
          o.x = pack_op2_g<INF>(__uint_as_float(v[u * 8 + 0]), __uint_as_float(v[u * 8 + 1]), p.fmt);
          o.y = pack_op2_g<INF>(__uint_as_float(v[u * 8 + 2]), __uint_as_float(v[u * 8 + 3]), p.fmt);
          o.z = pack_op2_g<INF>(__uint_as_float(v[u * 8 + 4]), __uint_as_float(v[u * 8 + 5]), p.fmt);
          o.w = pack_op2_g<INF>(__uint_as_float(v[u * 8 + 6]), __uint_as_float(v[u * 8 + 7]), p.fmt);
          *reinterpret_cast<uint4*>(dst + c * 32 + u * 8) = o;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace mcedm

namespace mcedm {
template <bool INF>
static int attn_bwd_launch(const CUtensorMap& tm_qkv, const CUtensorMap& tm_do, int L, const float* lse, float* dvec,
                           void* dq_bf16, void* dk_bf16, void* dv_bf16, int op_fmt, int B, cudaStream_t st) {
  AttnBwdParams p;
  p.L = L;
  p.lse = lse;
  p.dvec = dvec;
  p.fmt = op_fmt ? 1 : 0;
  p.err = watchdog_ptr();
  MCEDM_REQUIRE(p.err != nullptr, "attention_bwd: no watchdog word");
  const int smem = 1024 + 2 * kBTile + kBStages * 2 * kBTile + 4 * kBTile + 2 * 256 * 4 + 256;
  static bool attr_set = false;
  if (!attr_set) {
    MCEDM_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<0, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    MCEDM_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<1, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set = true;
  }
  const unsigned grid = (unsigned)(B * (L / 128));
  p.out1 = nullptr;
  p.out2 = reinterpret_cast<__nv_bfloat16*>(dq_bf16);
  attn_bwd_kernel<0, INF><<<grid, 192, smem, st>>>(tm_qkv, tm_do, p);
  MCEDM_CUDA(cudaGetLastError());
  p.out1 = reinterpret_cast<__nv_bfloat16*>(dv_bf16);
  p.out2 = reinterpret_cast<__nv_bfloat16*>(dk_bf16);
  attn_bwd_kernel<1, INF><<<grid, 192, smem, st>>>(tm_qkv, tm_do, p);
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}
}  // namespace mcedm

extern "C" int mcedm_attention_bwd(const void* qkv_bf16, const void* out_bf16, const void* d_out_bf16,
                                   const float* lse, int B, int L, float* dvec, void* dq_bf16, void* dk_bf16,
                                   void* dv_bf16, void* stream) {
  return mcedm_attention_bwd16(qkv_bf16, out_bf16, d_out_bf16, lse, B, L, dvec, dq_bf16, dk_bf16, dv_bf16, 0, stream);
}

extern "C" int mcedm_attention_bwd16(const void* qkv_bf16, const void* out_bf16, const void* d_out_bf16,
                                     const float* lse, int B, int L, float* dvec, void* dq_bf16, void* dk_bf16,
                                     void* dv_bf16, int op_fmt, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && L >= 128 && L % 128 == 0, "attention_bwd: L=%d must be a positive multiple of 128", L);
  CUtensorMap tm_qkv, tm_do;
  int rc = make_tmap_nhwc_bf16(&tm_qkv, qkv_bf16, B, 1, L, 192, 128, 1);
  if (rc) return rc;
  rc = make_tmap_nhwc_bf16(&tm_do, d_out_bf16, B, 1, L, 64, 128, 1);
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long rows = (long long)B * L;
  attn_bwd_prep_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(
      reinterpret_cast<const uint4*>(out_bf16), reinterpret_cast<const uint4*>(d_out_bf16), rows, dvec, op_fmt ? 1 : 0);
  MCEDM_CUDA(cudaGetLastError());
  return op_fmt == MCEDM_FMT_F16_INF ? attn_bwd_launch<true>(tm_qkv, tm_do, L, lse, dvec, dq_bf16, dk_bf16, dv_bf16, 1, B, st)
                                   : attn_bwd_launch<false>(tm_qkv, tm_do, L, lse, dvec, dq_bf16, dk_bf16, dv_bf16, op_fmt, B, st);
}
