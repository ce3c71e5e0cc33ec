// K3 — fused single-head self-attention at the low-resolution U-Net levels on tcgen05.
//
// Replaces AttentionOp.forward + the value einsum of UNetBlock.forward
// (models/adm_blocks.py:103-109, :176-178):
//     w = softmax_j( sum_c q[c,i] * k[c,j] / sqrt(64) )   (fp32),   a[c,i] = sum_j w[i,j] * v[c,j]
// for one head of 64 channels over L = H*W tokens (L = 1024 at 32x32).  The reference materialises
// the L x L weight matrix in HBM (4 MB per sample per block); here it never leaves the SM.
//
// Input : qkv bf16 [B, L, 192] = (q | k | v) blocks of 64 channels, written by the qkv 1x1 conv
//         (conv_igemm with N = 192; the reference's per-channel q/k/v interleave,
//         adm_blocks.py:175-176, is undone by permuting the weight rows once at pack time).
// Output: a bf16 [B, L, 64] (operand of the proj 1x1 conv).
//
// One CTA = 128 queries of one sample. Two passes over the keys in blocks of 128:
//   pass 1: S = Q K^T on tensor cores -> TMEM; softmax warps keep the running row maximum (no exponentials);
//   pass 2: S again, P = exp2((S - max) * log2e/8) -> bf16 -> swizzled smem, O += P V on tensor cores; the row
//           sum is accumulated in fp32 from the same exponentials.
// The second QK^T costs 50 % more MMA work but removes every accumulator rescale; the kernel is
// bound by the exp/convert work of the 4 softmax warps, not by the tensor pipe.
//
// SINGLE-PASS variant (inference, round 2).  What bounds the two-pass kernel is not the exponentials but reading S out
// of TMEM twice (64 B per cycle per SM: 1024 cycles per 128 x 128 fp32 block, per pass — as long as the block's MUFU
// work).  Softmax is invariant to the shift, so the shift need not be the row maximum: the single-pass kernel takes
// m_ref = the exact row maximum of key block 0 and never rescales.  Later blocks may exceed m_ref; P = exp2(.) then
// exceeds 1, which fp16 holds up to 2^16.  A CTA whose exponent argument ever exceeds 15 (a score 83 above its first
// block's maximum: not seen on normalised inputs, but legal) raises its flag and the caller re-runs exactly those tiles
// with the two-pass kernel, whose CTAs return at once when their flag is clear.
//
// H2 (single pass, fp16 operands): after the single pass the softmax warps themselves were the pacer (per element: FFMA,
// MUFU.EX2, half of a pack, unpack + add for the row sum).  Now the exponent argument is rounded to fp16 PAIRS and one
// `ex2.approx.f16x2` produces two weights already in operand format (no pack), and the row sums of those ROUNDED weights
// (what the P V product sums) are three packed fp16 adds over 8 values, then fp32.
//   warp 0 : TMA producer (Q once; K blocks in pass 1; K and V blocks in pass 2; 3-stage ring)
//   warp 1 : MMA issuer (S double-buffered in TMEM so softmax of block j overlaps QK^T of block j+1)
//   warps 2.. : softmax / epilogue: KS warps per TMEM lane quarter (2, or 4 for H2), each owning 128 / KS keys of every
//               S block of its 32 query rows (TMEM lane == row: no shuffles); the slices' row maxima / row sums meet
//               once per pass through shared memory.  (With 4 softmax warps = one per scheduler, the dependent
//               ld -> ex2 -> cvt -> st chain had nothing to overlap with and set the kernel's pace.)
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

#include <cuda_bf16.h>
#include <cstdlib>

namespace mcedm {

constexpr int kKvStages = 3;
constexpr int kTile = 16384;  // 128 rows x 128 B

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// SINGLE: one pass over the keys (see the header); flags = per-CTA overflow flags, WRITTEN by the single-pass kernel and
// READ by the two-pass kernel launched after it (NULL: every CTA of the two-pass kernel runs).
// KS: softmax warps per TMEM lane quarter (each owns 128 / KS key columns of every S block).  2 for the two-pass /
// fp32-exponential kernels; 4 for H2, whose per-warp chain (tcgen05.ld -> FFMA -> cvt -> MUFU -> st.shared) was latency-
// bound at 10 resident warps (ncu: issue slots 29 % active, top stalls long scoreboard / wait / MIO throttle).
template <bool H2>
constexpr int attn_threads() {
  return 64 + 128 * (H2 ? 4 : 2);
}

template <bool SINGLE, bool H2>
__global__ void __launch_bounds__(attn_threads<H2>(), 1)
attn_kernel(const __grid_constant__ CUtensorMap tm_qkv, int L, __nv_bfloat16* __restrict__ out,
            float* __restrict__ lse_out, int fmt, unsigned int* err, unsigned int* __restrict__ flags, int n_tiles) {
  constexpr int KS = H2 ? 4 : 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* q_smem = smem;                                  // 16 KB
  uint8_t* kv_smem = q_smem + kTile;                       // stages x (K 16 KB | V 16 KB)
  uint8_t* p_smem = kv_smem + kKvStages * 2 * kTile;       // 2 buffers x 32 KB (2 atoms of 64 keys)
  uint64_t* bars = reinterpret_cast<uint64_t*>(p_smem + 2 * 2 * kTile);
  uint64_t* q_full = bars;            // 1
  uint64_t* o_full = bars + 1;        // 1
  uint64_t* s_full = bars + 2;        // 2
  uint64_t* s_empty = bars + 4;       // 2
  uint64_t* p_full = bars + 6;        // 2
  uint64_t* p_empty = bars + 8;       // 2
  uint64_t* kv_full = bars + 10;      // stages
  uint64_t* kv_empty = bars + 10 + kKvStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10 + 2 * kKvStages);
  float* xch_m = reinterpret_cast<float*>(bars) + 64;                      // [KS][128 rows] partial row maxima
  float* xch_l = xch_m + 128 * KS;                                         // [KS][128 rows] partial row sums

  pdl_wait();       // (the flag words written below are read by the previous call's fallback launch)
  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = L / 128;
  const int p2_start = SINGLE ? 0 : nblk;      // first iteration of the exponentiating pass
  const int n_it = p2_start + nblk;
  // One tile (128 queries of one sample) per CTA when the grid covers all tiles (the single-pass kernel and the
  // stand-alone two-pass kernel).  The FALLBACK launch of the two-pass kernel (flags != NULL) runs a small grid whose
  // CTAs stride over the tiles and redo only the flagged ones: with no flag raised — the normal case — it costs a
  // launch and a few flag reads per CTA instead of 2048 empty 180 KB-shared-memory CTAs (17 us).
  if (!SINGLE && flags != nullptr) {
    // fallback launch: all of this CTA's flags in ONE round trip (one thread per tile); nothing raised - the normal case -
    // and the CTA is gone (the loop below would read them one dependent load after the other: ~0.5 us per tile)
    int any = 0;
    for (int tile = (int)blockIdx.x + (int)threadIdx.x * (int)gridDim.x; tile < n_tiles; tile += (int)(blockDim.x * gridDim.x))
      any |= flags[tile] != 0u;
    if (!__syncthreads_or(any)) return;
  }
  // TMEM is allocated ONCE per CTA: tcgen05.relinquish_alloc_permit gives the right to allocate up for the rest of the
  // CTA's life, so a second allocation by a fallback CTA that redoes more than one flagged tile is a device exception
  // ("unspecified launch failure": seen at 256 samples per call, where a CTA strides over 14 tiles, as soon as one CTA had
  // two flagged tiles; the 2-sample test gave every CTA at most one).
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  bool first_tile = true;
  for (int tile = (int)blockIdx.x; tile < n_tiles; tile += (int)gridDim.x) {
  if (!SINGLE && flags != nullptr && flags[tile] == 0u) continue;
  const int b = tile / nblk;
  const int q0 = (tile - b * nblk) * 128;

  if (warp == 0 && lane == 0) {
    if (SINGLE && flags) flags[tile] = 0u;
    if (!first_tile) {                       // barriers of the previous tile: every role is past them (__syncthreads below)
      for (int i = 0; i < 10 + 2 * kKvStages; ++i) mbar_inval(&bars[i]);
    }
    prefetch_tmap(&tm_qkv);
    mbar_init(q_full, 1);
    mbar_init(o_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_empty[i], 4 * KS);                         // one arrival per softmax warp
      mbar_init(&p_full[i], 4 * KS);
      mbar_init(&p_empty[i], 1);
    }
    for (int i = 0; i < kKvStages; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    fence_barrier_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_o = tmem_base + 256;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(q_full, kTile);
      tma_load_4d(q_smem, &tm_qkv, q_full, 0, q0, 0, b);
      for (int it = 0; it < n_it; ++it) {
        const int pass = it >= p2_start ? 1 : 0, j = it - pass * p2_start;
        const uint32_t s = it % kKvStages, n = it / kKvStages;
        mbar_wait(&kv_empty[s], (n & 1u) ^ 1u, err, 0x1100 + s);
        mbar_expect_tx(&kv_full[s], pass ? 2 * kTile : kTile);
        tma_load_4d(kv_smem + s * 2 * kTile, &tm_qkv, &kv_full[s], 64, j * 128, 0, b);
        if (pass) tma_load_4d(kv_smem + s * 2 * kTile + kTile, &tm_qkv, &kv_full[s], 128, j * 128, 0, b);
      }
    }
  } else if (warp == 1) {
    // warp-uniform control flow; one elected lane issues the tcgen05 instructions
    {
      const uint32_t idesc_s = umma_idesc_16(128, 128, 0, 0, fmt);
      const uint32_t idesc_o = umma_idesc_16(128, 64, 0, 1, fmt);    // B = V, MN-major
      mbar_wait(q_full, 0, err, 0x1200);
      tc_fence_after();
      const uint32_t q_base = smem_u32(q_smem);
      for (int it = 0; it <= n_it; ++it) {
        if (it < n_it) {
          const int pass = it >= p2_start ? 1 : 0;
          const uint32_t sb = it & 1u, ns = (uint32_t)it >> 1;
          const uint32_t s = it % kKvStages, n = it / kKvStages;
          mbar_wait(&s_empty[sb], (ns & 1u) ^ 1u, err, 0x1300 + sb);
          mbar_wait(&kv_full[s], n & 1u, err, 0x1400 + s);
          tc_fence_after();
          const uint64_t qd = umma_desc_k_sw128(q_base);
          const uint64_t kd = umma_desc_k_sw128(smem_u32(kv_smem + s * 2 * kTile));
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16(tmem_base + sb * 128, qd + 2 * k, kd + 2 * k, idesc_s, (uint32_t)(k != 0));
            umma_commit(&s_full[sb]);
            if (pass == 0) umma_commit(&kv_empty[s]);
          }
          __syncwarp();
        }
        if (it >= p2_start + 1) {
          const int jp = it - 1 - p2_start;                // P V of the previous pass-2 block
          const uint32_t pb = jp & 1u, np = (uint32_t)jp >> 1;
          const uint32_t sp = (it - 1) % kKvStages;
          mbar_wait(&p_full[pb], np & 1u, err, 0x1500 + pb);
          tc_fence_after();
          // descriptor words formed in warp-uniform code, compile-time offsets inside the elected branch
          const uint64_t pd = umma_desc_k_sw128(smem_u32(p_smem + pb * 2 * kTile));
          const uint64_t vd = umma_desc_mn_sw128(smem_u32(kv_smem + sp * 2 * kTile + kTile), 8192);
          if (elect_one()) {
#pragma unroll
            for (int kk = 0; kk < 8; ++kk)
              umma_f16(tmem_o, pd + (uint64_t)(((kk >> 2) * kTile + (kk & 3) * 32) >> 4), vd + (uint64_t)((kk * 2048) >> 4),
                       idesc_o, (uint32_t)((jp | kk) != 0));
            umma_commit(&p_empty[pb]);
            umma_commit(&kv_empty[sp]);
          }
          __syncwarp();
        }
      }
      if (elect_one()) umma_commit(o_full);
      __syncwarp();
    }
  } else {
    const int q = warp & 3;
    const int hsel = (warp - 2) >> 2;          // which 128 / KS-key slice of every S block this warp owns
    constexpr int CPW = 4 / KS;                // 32-column chunks per warp and S block
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float c1 = 0.125f * 1.4426950408889634f;   // 1/sqrt(64) * log2(e)
    float m = -INFINITY, l = 0.f;
    // ---------------- pass 1: row maximum only (the row sum is accumulated from the pass-2 exponentials) -----
    for (int it = 0; it < p2_start; ++it) {
      const uint32_t sb = it & 1u, ns = (uint32_t)it >> 1;
      mbar_wait(&s_full[sb], ns & 1u, err, 0x1600 + sb);
      tc_fence_after();
#pragma unroll 1
      for (int c = CPW * hsel; c < CPW * hsel + CPW; ++c) {
        uint32_t v[32];
        tmem_ld_x32(tmem_base + lane_addr + sb * 128 + c * 32, v);
        tmem_wait_ld();
        float cm0 = __uint_as_float(v[0]), cm1 = __uint_as_float(v[1]);
#pragma unroll
        for (int i = 2; i < 32; i += 2) {
          cm0 = fmaxf(cm0, __uint_as_float(v[i]));
          cm1 = fmaxf(cm1, __uint_as_float(v[i + 1]));
        }
        m = fmaxf(m, fmaxf(cm0, cm1));
      }
      tc_fence_before();
      mbar_arrive_warp(&s_empty[sb]);
    }
    if constexpr (SINGLE) {
      // m_ref = exact row maximum of key block 0 (its S buffer is read again by the loop below; s_empty is not
      // arrived on here, so the buffer stays valid)
      mbar_wait(&s_full[0], 0u, err, 0x1650);
      tc_fence_after();
#pragma unroll 1
      for (int c = CPW * hsel; c < CPW * hsel + CPW; ++c) {
        uint32_t v[32];
        tmem_ld_x32(tmem_base + lane_addr + c * 32, v);
        tmem_wait_ld();
        float cm0 = __uint_as_float(v[0]), cm1 = __uint_as_float(v[1]);
#pragma unroll
        for (int i = 2; i < 32; i += 2) {
          cm0 = fmaxf(cm0, __uint_as_float(v[i]));
          cm1 = fmaxf(cm1, __uint_as_float(v[i + 1]));
        }
        m = fmaxf(m, fmaxf(cm0, cm1));
      }
    }
    // the two halves of a row exchange their partial maxima
    xch_m[hsel * 128 + row] = m;
    asm volatile("bar.sync 1, %0;" ::"n"(128 * KS) : "memory");
    m = xch_m[row];
#pragma unroll
    for (int k = 1; k < KS; ++k) m = fmaxf(m, xch_m[k * 128 + row]);
    const float mc = m * c1;
    float amax = 0.f;                         // SINGLE: largest exponent argument seen (0 at the reference maximum)
    uint32_t hmax = 0u;                       // H2: the same as a packed fp16 pair
    // ---------------- pass 2: P = exp2(S*c1 - m*c1) -> bf16 -> smem ----------------
    for (int j = 0; j < nblk; ++j) {
      const int it = p2_start + j;
      const uint32_t sb = it & 1u, ns = (uint32_t)it >> 1;
      const uint32_t pb = j & 1u, np = (uint32_t)j >> 1;
      mbar_wait(&s_full[sb], ns & 1u, err, 0x1700 + sb);
      mbar_wait(&p_empty[pb], (np & 1u) ^ 1u, err, 0x1800 + pb);
      tc_fence_after();
      uint8_t* prow = p_smem + pb * 2 * kTile + row * 128;
#pragma unroll 1
      for (int c = CPW * hsel; c < CPW * hsel + CPW; ++c) {
        uint32_t v[32];
        tmem_ld_x32(tmem_base + lane_addr + sb * 128 + c * 32, v);
        tmem_wait_ld();
        const uint32_t atom_row = smem_u32(prow) + (c >> 1) * kTile;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          uint4 o;
          uint32_t* op = reinterpret_cast<uint32_t*>(&o);
          if constexpr (H2) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float a0 = fmaf(__uint_as_float(v[u * 8 + 2 * e]), c1, -mc);
              const float a1 = fmaf(__uint_as_float(v[u * 8 + 2 * e + 1]), c1, -mc);
              uint32_t hh;
              asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(hh) : "f"(a1), "f"(a0));
              asm("max.NaN.f16x2 %0, %0, %1;" : "+r"(hmax) : "r"(hh));
              asm("ex2.approx.f16x2 %0, %1;" : "=r"(op[e]) : "r"(hh));
            }
            // row sum of the ROUNDED weights: three packed fp16 adds over the 8 values, then fp32 (the fp16 partial of 8
            // terms carries ~2^-11 relative error, random over the 128 partials of a row)
            uint32_t s01, s23, s4;
            asm("add.rn.f16x2 %0, %1, %2;" : "=r"(s01) : "r"(op[0]), "r"(op[1]));
            asm("add.rn.f16x2 %0, %1, %2;" : "=r"(s23) : "r"(op[2]), "r"(op[3]));
            asm("add.rn.f16x2 %0, %1, %2;" : "=r"(s4) : "r"(s01), "r"(s23));
            const float2 sf = unpack_f16x2(s4);
            l += sf.x + sf.y;
            const int unit = ((c & 1) * 4 + u) ^ (row & 7);
            sts128(atom_row + unit * 16, o);
            continue;
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float a0 = fmaf(__uint_as_float(v[u * 8 + 2 * e]), c1, -mc);
            const float a1 = fmaf(__uint_as_float(v[u * 8 + 2 * e + 1]), c1, -mc);
            if constexpr (SINGLE) amax = fmaxf(amax, fmaxf(a0, a1));
            const float p0 = ex2(a0);
            const float p1 = ex2(a1);
            op[e] = pack_op2(p0, p1, fmt);
            // normalise by what the P V product actually sums (the rounded weights)
            if (fmt) {
              const float2 r = unpack_f16x2(op[e]);
              l += r.x + r.y;
            } else {
              l += bf16_lo(op[e]) + bf16_hi(op[e]);
            }
          }
          const int unit = ((c & 1) * 4 + u) ^ (row & 7);
          sts128(atom_row + unit * 16, o);
        }
      }
      tc_fence_before();
      mbar_arrive_warp(&s_empty[sb]);
      fence_proxy_async_smem();     // generic-proxy P writes -> visible to the UMMA (async proxy) reads
      mbar_arrive_warp(&p_full[pb]);
    }
    if constexpr (H2) {
      const float2 hm = unpack_f16x2(hmax);
      amax = (hm.x != hm.x || hm.y != hm.y) ? __int_as_float(0x7fc00000) : fmaxf(hm.x, hm.y);
    }
    if constexpr (SINGLE) {
      // fp16 weights hold exp2(a) up to a < 16; beyond 15 (or a non-finite score) the tile is redone by the two-pass kernel
      if (__any_sync(0xffffffffu, !(amax <= 15.0f)) && lane == 0 && flags) flags[tile] = 1u;
    }
    // ---------------- epilogue: O / l -> bf16 ----------------
    xch_l[hsel * 128 + row] = l;
    asm volatile("bar.sync 1, %0;" ::"n"(128 * KS) : "memory");
    l = xch_l[row];
#pragma unroll
    for (int k = 1; k < KS; ++k) l += xch_l[k * 128 + row];
    mbar_wait(o_full, 0, err, 0x1900);
    tc_fence_after();
    const float inv_l = 1.0f / l;
    // saved for the backward: P[i][j] = exp2(S[i][j] * c1 - lse2[i])
    if (lse_out && hsel == 0) lse_out[(long long)b * L + q0 + row] = mc + log2f(l);
    __nv_bfloat16* orow = out + ((long long)b * L + q0 + row) * 64;
#pragma unroll 1
    for (int c = hsel; c < (hsel < 2 ? hsel + 1 : hsel); ++c) {      // O has two 32-column chunks: slices 0 and 1 store them
      uint32_t v[32];
      tmem_ld_x32(tmem_o + lane_addr + c * 32, v);
      tmem_wait_ld();
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        uint4 o;
        o.x = pack_op2(__uint_as_float(v[u * 8 + 0]) * inv_l, __uint_as_float(v[u * 8 + 1]) * inv_l, fmt);
        o.y = pack_op2(__uint_as_float(v[u * 8 + 2]) * inv_l, __uint_as_float(v[u * 8 + 3]) * inv_l, fmt);
        o.z = pack_op2(__uint_as_float(v[u * 8 + 4]) * inv_l, __uint_as_float(v[u * 8 + 5]) * inv_l, fmt);
        o.w = pack_op2(__uint_as_float(v[u * 8 + 6]) * inv_l, __uint_as_float(v[u * 8 + 7]) * inv_l, fmt);
        *reinterpret_cast<uint4*>(orow + c * 32 + u * 8) = o;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  first_tile = false;
  }   // tile loop
  if (warp == 1) tmem_dealloc(*tmem_slot, 512);
}

}  // namespace mcedm

namespace mcedm {
// per-CTA overflow flags of the single-pass kernel (device memory, grown on demand outside graph capture)
static unsigned int* attn_flags(long long n) {
  static unsigned int* buf = nullptr;
  static long long cap = 0;
  if (n > cap) {
    if (buf) cudaFree(buf);
    const long long want = n < 16384 ? 16384 : n;
    if (cudaMalloc(&buf, sizeof(unsigned int) * want) != cudaSuccess) {
      buf = nullptr;
      cap = 0;
      return nullptr;
    }
    cudaMemset(buf, 0, sizeof(unsigned int) * want);
    cap = want;
  }
  return buf;
}
}  // namespace mcedm

extern "C" int mcedm_attention(const void* qkv_bf16, int B, int L, void* out_bf16, float* lse_out, int op_fmt,
                               void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(B >= 1 && L >= 128 && L % 128 == 0, "attention: L=%d must be a positive multiple of 128", L);
  CUtensorMap tm;
  int rc = make_tmap_nhwc_bf16(&tm, qkv_bf16, B, 1, L, 192, 128, 1);
  if (rc) return rc;
  unsigned int* err = watchdog_ptr();
  MCEDM_REQUIRE(err != nullptr, "attention: no watchdog word");
  const int smem = 1024 + kTile + kKvStages * 2 * kTile + 4 * kTile + 256 + 4096;   // align | Q | K/V | P | barriers | row exchange
  static bool attr_set = false;
  if (!attr_set) {
    MCEDM_CUDA((cudaFuncSetAttribute(attn_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)));
    MCEDM_CUDA((cudaFuncSetAttribute(attn_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)));
    MCEDM_CUDA((cudaFuncSetAttribute(attn_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)));
    attr_set = true;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned grid = (unsigned)(B * (L / 128));
  // inference (no log-sum-exp requested): single pass over the keys + a fallback launch whose CTAs return at once
  // unless the single-pass CTA flagged an exponent beyond fp16's range; training runs the two-pass kernel
  auto* o = reinterpret_cast<__nv_bfloat16*>(out_bf16);
  const int fmt = op_fmt ? 1 : 0;
  if (lse_out == nullptr) {
    unsigned int* flags = attn_flags(grid);
    MCEDM_REQUIRE(flags != nullptr, "attention: cannot allocate the overflow flags");
    if (fmt)
      MCEDM_CUDA(launch_pdl(attn_kernel<true, true>, dim3(grid), dim3(attn_threads<true>()), (size_t)smem, st, tm, L, o,
                            nullptr, fmt, err, flags, (int)grid));
    else
      MCEDM_CUDA(launch_pdl(attn_kernel<true, false>, dim3(grid), dim3(attn_threads<false>()), (size_t)smem, st, tm, L, o,
                            nullptr, fmt, err, flags, (int)grid));
    MCEDM_CUDA(cudaGetLastError());
    const unsigned fb_grid = grid < (unsigned)num_sms() ? grid : (unsigned)num_sms();
    MCEDM_CUDA(launch_pdl(attn_kernel<false, false>, dim3(fb_grid), dim3(attn_threads<false>()), (size_t)smem, st, tm, L,
                          o, nullptr, fmt, err, flags, (int)grid));
    MCEDM_CUDA(cudaGetLastError());
    return 0;
  }
  MCEDM_CUDA(launch_pdl(attn_kernel<false, false>, dim3(grid), dim3(attn_threads<false>()), (size_t)smem, st, tm, L, o,
                        lse_out, fmt, err, nullptr, (int)grid));
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}

