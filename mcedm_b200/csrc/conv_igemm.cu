// K1 — 3x3 / 1x1 convolution as an implicit GEMM on the tcgen05 tensor cores (sm_100a).
//
// Replaces the reference's `Conv2d.forward` call sites (models/adm_blocks.py:65-81) for every
// 64-multiple-channel convolution of the ADM U-Net, plus the residual add of
// `UNetBlock.forward` (models/adm_blocks.py:171,179) and the channel concat of the decoder
// (models/adm_blocks.py:401), both of which are fused here.
//
// GEMM view:  D[pixels, N] = sum_seg  A_seg[pixels, 64] * W_seg[N, 64]^T
//   * one "segment" = one (source tensor, filter tap) pair = 64 input channels;
//     3x3 conv of one 64-ch source = 9 segments, two concatenated sources = 18,
//     conv1 + the block's 1x1 skip projection of the raw 128-ch input = 9 + 2.
//   * A tiles are fetched by TMA straight from the NHWC bf16 activation: a 4-D box
//     (64 ch, W, 128/W rows, 1 image) at coordinate (0, dx, y0+dy, b). Out-of-bounds
//     coordinates are zero-filled by the TMA unit = the conv's zero padding. The tile lands in
//     shared memory as 128 rows x 128 B, SWIZZLE_128B = the canonical K-major UMMA layout.
//   * all W_seg (bf16, [N,64] K-major each) stay resident in shared memory for the CTA's life.
//   * one thread issues tcgen05.mma (M=128, N, K=16) x4 per segment into a double-buffered
//     fp32 accumulator in TMEM; 4 epilogue warps drain it (tcgen05.ld), add bias / residual,
//     emit GroupNorm partial sums and store coalesced through a swizzled staging buffer.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner,
// warps 2..5 = epilogue (TMEM lane quarter = warp_id % 4).
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

#include <cuda_bf16.h>

namespace mcedm {

constexpr int kMaxSeg = 20;
constexpr int kTileM = 128;
constexpr int kATileBytes = kTileM * 128;  // 128 pixels x 64 bf16

struct ConvParams {
  int n_seg;
  int n_stages;
  int n_tiles;
  int H, W;
  int tiles_per_img;
  int rows_per_tile;
  signed char seg_src[kMaxSeg];
  signed char seg_dy[kMaxSeg];
  signed char seg_dx[kMaxSeg];
  const float* bias;      // [N] or nullptr
  void* out;              // [pixels, N] fp32 or bf16
  int out_bf16;
  int fmt;               // 16-bit operand format (inputs, weights and a 16-bit output): 0 bf16, 1 fp16
  const float* res;       // residual, fp32 NHWC with N channels (resolution per res_mode)
  int res_mode;           // 0 none, 1 same resolution, 2 nearest-x2 upsample of res, 3 2x2 mean of res
  float* stats;           // [n_tiles][N/4][2] (sum, sum of squares of the stored values) or nullptr
  unsigned int* err;
  // ---- 16-bit I/O variant (mcedm_conv_igemm16, inference)
  int res16;              // residual (res_mode 1) is 16-bit in the operand format and is prefetched
  int io_pitch, io_blk;   // > 0: out and res are padded-flat (conv_flat.cu layout) instead of dense NHWC
};

template <int N>
struct ConvCfg {
  static constexpr int CH = (N >= 32) ? 32 : 16;          // accumulator columns per epilogue chunk
  static constexpr int NCH = N / CH;
  static constexpr int U = CH / 4;                        // 16-byte units per staged row
  static constexpr int W_SEG_BYTES = N * 128;
  // epilogue column groups: G x 4 warps, each group drains NCH / G chunks of every tile (with 4 warps for N = 192 the
  // six chunks per tile made the epilogue the pacer of the 1x1 convs: 50 us for a 12 us memory job)
  static constexpr int G = (N >= 192) ? 3 : (N >= 64) ? 2 : 1;
  static constexpr int NLOC = NCH / G;                     // chunks per warp
  static constexpr int THREADS = 64 + 128 * G;
  static constexpr int STAGE_BYTES = 4 * G * 32 * CH * 4;  // per-CTA epilogue staging
  static constexpr int STAT_BYTES = 2 * 4 * (N / 4) * 2 * 4;
  static constexpr int ACC_STRIDE = (N == 192) ? 256 : N; // TMEM column stride between the two buffers
  static constexpr int TMEM_COLS = (2 * ACC_STRIDE <= 32) ? 32 : (2 * ACC_STRIDE <= 64) ? 64
                                   : (2 * ACC_STRIDE <= 128) ? 128 : (2 * ACC_STRIDE <= 256) ? 256 : 512;
};

template <int THREADS>
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(THREADS) : "memory"); }

// INF: 16-bit output without saturation (the 1x1 data gradients of dynamic loss scaling, op_fmt MCEDM_FMT_F16_INF)
template <int N, bool INF = false>
__global__ void __launch_bounds__(ConvCfg<N>::THREADS, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_a0,
                  const __grid_constant__ CUtensorMap tm_a1, const __grid_constant__ CUtensorMap tm_a2,
                  const __grid_constant__ CUtensorMap tm_a3, const ConvParams p) {
  using Cfg = ConvCfg<N>;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_smem = smem;
  uint8_t* a_smem = w_smem + p.n_seg * Cfg::W_SEG_BYTES;
  uint8_t* stage_smem = a_smem + p.n_stages * kATileBytes;
  float* stat_smem = reinterpret_cast<float*>(stage_smem + Cfg::STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(stat_smem) + Cfg::STAT_BYTES);
  uint64_t* w_full = bars;             // 1
  uint64_t* acc_full = bars + 1;       // 2
  uint64_t* acc_empty = bars + 3;      // 2
  uint64_t* a_full = bars + 5;         // n_stages
  uint64_t* a_empty = a_full + p.n_stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_empty + p.n_stages);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_w);
    prefetch_tmap(&tm_a0);
    mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4 * Cfg::G);                  // one arrival per epilogue warp
    }
    for (int i = 0; i < p.n_stages; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
    }
    fence_barrier_init();
    // weights before pdl_wait (not written by the preceding kernel): the prologue overlaps the previous kernel's tail
    mbar_expect_tx(w_full, (uint32_t)(p.n_seg * Cfg::W_SEG_BYTES));
    for (int s = 0; s < p.n_seg; ++s) tma_load_2d(w_smem + s * Cfg::W_SEG_BYTES, &tm_w, w_full, 0, s * N);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      const CUtensorMap* maps[4] = {&tm_a0, &tm_a1, &tm_a2, &tm_a3};
      uint32_t it = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const int b = tile / p.tiles_per_img;
        const int y0 = (tile - b * p.tiles_per_img) * p.rows_per_tile;
        for (int s = 0; s < p.n_seg; ++s, ++it) {
          const uint32_t stage = it % (uint32_t)p.n_stages;
          const uint32_t ph = (it / (uint32_t)p.n_stages) & 1u;
          mbar_wait(&a_empty[stage], ph ^ 1u, p.err, 0x100 + stage);
          mbar_expect_tx(&a_full[stage], kATileBytes);
          tma_load_4d(a_smem + stage * kATileBytes, maps[p.seg_src[s]], &a_full[stage], 0, (int)p.seg_dx[s],
                      y0 + (int)p.seg_dy[s], b);
        }
      }
    }
  } else if (warp == 1) {
    // ====================================== MMA issuer ======================================
    // warp-uniform control flow (descriptors stay in uniform registers); one elected lane issues
    {
      const uint32_t idesc = umma_idesc_16(kTileM, N, 0, 0, p.fmt);
      mbar_wait(w_full, 0, p.err, 0x200);
      tc_fence_after();
      uint32_t it = 0, tcount = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++tcount) {
        const uint32_t buf = tcount & 1u;
        const uint32_t aph = (tcount >> 1) & 1u;
        mbar_wait(&acc_empty[buf], aph ^ 1u, p.err, 0x300 + buf);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * Cfg::ACC_STRIDE;
        for (int s = 0; s < p.n_seg; ++s, ++it) {
          const uint32_t stage = it % (uint32_t)p.n_stages;
          const uint32_t ph = (it / (uint32_t)p.n_stages) & 1u;
          mbar_wait(&a_full[stage], ph, p.err, 0x400 + stage);
          tc_fence_after();
          const uint64_t ad = umma_desc_k_sw128(smem_u32(a_smem + stage * kATileBytes));
          const uint64_t bd = umma_desc_k_sw128(smem_u32(w_smem + s * Cfg::W_SEG_BYTES));
          if (elect_one()) {
            // advance 16 bf16 (32 B) along K inside the 128-byte swizzle row: +2 in the (address >> 4) field
            umma_f16(d_tmem, ad, bd, idesc, s != 0 ? 1u : 0u);
            umma_f16(d_tmem, ad + 2, bd + 2, idesc, 1u);
            umma_f16(d_tmem, ad + 4, bd + 4, idesc, 1u);
            umma_f16(d_tmem, ad + 6, bd + 6, idesc, 1u);
            umma_commit(&a_empty[stage]);  // smem stage reusable once these MMAs have read it
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(&acc_full[buf]);     // accumulator complete
        __syncwarp();
      }
    }
  } else {
    // ======================================= epilogue =======================================
    const int q = warp & 3;              // TMEM lane quarter this warp may access
    const int ew = warp - 2;             // staging slot
    const int cg = ew >> 2;              // column group: chunks [cg * NLOC, (cg + 1) * NLOC)
    const uint32_t my_stage = smem_u32(stage_smem) + ew * (32 * Cfg::CH * 4);
    const int unit = lane % Cfg::U;
    const int row_in_it = lane / Cfg::U;
    constexpr int ROWS_PER_IT = 32 / Cfg::U;
    const int wshift = __ffs(p.W) - 1;
    uint32_t tcount = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++tcount) {
      const uint32_t buf = tcount & 1u;
      const uint32_t aph = (tcount >> 1) & 1u;
      const long long pix0 = (long long)tile * kTileM + q * 32;
      // A tile never straddles images (tiles_per_img = H*W / 128) and W is a power of two (it divides 128): one 32-bit
      // division per tile, shifts per row.  (64-bit divisions per row made this epilogue the pacer of the 1x1 convs:
      // ~3000 issue cycles per tile.)
      const int img = tile / p.tiles_per_img;
      const int rem0 = (tile - img * p.tiles_per_img) * kTileM + q * 32;
      // output / residual pixel index of this lane's rows (dense, or padded-flat for the 16-bit I/O variant)
      long long opix[Cfg::U];
#pragma unroll
      for (int itr = 0; itr < Cfg::U; ++itr) {
        const int rem = rem0 + itr * ROWS_PER_IT + row_in_it;
        opix[itr] = pix0 + itr * ROWS_PER_IT + row_in_it;
        if (p.io_pitch > 0) {
          const int y = rem >> wshift;
          opix[itr] = (long long)img * p.io_blk + (long long)(y + 1) * p.io_pitch + (rem & (p.W - 1));
        }
      }
      // 16-bit residual prefetch (independent of the accumulator); N <= 64 only
      constexpr int NPRE = (N <= 64) ? Cfg::NLOC : 1;
      uint2 rh[NPRE][Cfg::U];
      if (N <= 64 && p.res16 && p.res_mode == 1) {
#pragma unroll
        for (int lc = 0; lc < NPRE; ++lc)
#pragma unroll
          for (int itr = 0; itr < Cfg::U; ++itr)
            rh[lc][itr] = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(p.res) + opix[itr] * N +
                                                          (cg * Cfg::NLOC + lc) * Cfg::CH + unit * 4);
      }
      mbar_wait(&acc_full[buf], aph, p.err, 0x500 + buf);
      tc_fence_after();
      float* my_stat = stat_smem + ((tcount & 1u) * 4 + q) * (N / 4) * 2;
      constexpr int kChUnroll = (N <= 64) ? Cfg::NLOC : 1;
#pragma unroll kChUnroll
      for (int lc = 0; lc < Cfg::NLOC; ++lc) {
        const int ch = cg * Cfg::NLOC + lc;
        uint32_t v[Cfg::CH];
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * Cfg::ACC_STRIDE + ch * Cfg::CH;
        if constexpr (Cfg::CH == 32) tmem_ld_x32(taddr, v); else tmem_ld_x16(taddr, v);
        tmem_wait_ld();
        if (lc == Cfg::NLOC - 1) {
          tc_fence_before();
          mbar_arrive_warp(&acc_empty[buf]);  // all of this warp's TMEM reads of this buffer are done
        }
        // registers (one pixel row per thread) -> swizzled staging rows
#pragma unroll
        for (int j = 0; j < Cfg::U; ++j) {
          const int pj = j ^ (lane & (Cfg::U - 1));
          sts128(my_stage + lane * (Cfg::CH * 4) + pj * 16, make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
        }
        __syncwarp();
        const int c0 = ch * Cfg::CH + unit * 4;
        float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) bz = *reinterpret_cast<const float4*>(p.bias + c0);
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int itr = 0; itr < Cfg::U; ++itr) {
          const int row = itr * ROWS_PER_IT + row_in_it;
          const int pu = unit ^ (row & (Cfg::U - 1));
          float4 a = lds128f(my_stage + row * (Cfg::CH * 4) + pu * 16);
          a.x += bz.x; a.y += bz.y; a.z += bz.z; a.w += bz.w;
          const long long pix = pix0 + row;
          if (p.res_mode == 1) {
            if (N <= 64 && p.res16) {
              const uint2 hv = rh[N <= 64 ? lc : 0][itr];
              float2 lo, hi;
              if (p.fmt) {
                lo = unpack_f16x2(hv.x);
                hi = unpack_f16x2(hv.y);
              } else {
                lo = make_float2(bf16_lo(hv.x), bf16_hi(hv.x));
                hi = make_float2(bf16_lo(hv.y), bf16_hi(hv.y));
              }
              a.x += lo.x; a.y += lo.y; a.z += hi.x; a.w += hi.y;
            } else {
              const float4 r = *reinterpret_cast<const float4*>(p.res + pix * N + c0);
              a.x += r.x; a.y += r.y; a.z += r.z; a.w += r.w;
            }
          } else if (p.res_mode != 0) {
            const int b = img;
            const int rem = rem0 + row;
            const int y = rem >> wshift, x = rem & (p.W - 1);
            if (p.res_mode == 2) {
              const int Hs = p.H >> 1, Ws = p.W >> 1;
              const float4 r = *reinterpret_cast<const float4*>(
                  p.res + (((long long)b * Hs + (y >> 1)) * Ws + (x >> 1)) * N + c0);
              a.x += r.x; a.y += r.y; a.z += r.z; a.w += r.w;
            } else {
              const int Hs = p.H << 1, Ws = p.W << 1;
              const float* r0 = p.res + (((long long)b * Hs + 2 * y) * Ws + 2 * x) * N + c0;
              const float4 r00 = *reinterpret_cast<const float4*>(r0);
              const float4 r01 = *reinterpret_cast<const float4*>(r0 + N);
              const float4 r10 = *reinterpret_cast<const float4*>(r0 + (long long)Ws * N);
              const float4 r11 = *reinterpret_cast<const float4*>(r0 + (long long)Ws * N + N);
              a.x += 0.25f * ((r00.x + r01.x) + (r10.x + r11.x));
              a.y += 0.25f * ((r00.y + r01.y) + (r10.y + r11.y));
              a.z += 0.25f * ((r00.z + r01.z) + (r10.z + r11.z));
              a.w += 0.25f * ((r00.w + r01.w) + (r10.w + r11.w));
            }
          }
          s1 += (a.x + a.y) + (a.z + a.w);
          s2 += (a.x * a.x + a.y * a.y) + (a.z * a.z + a.w * a.w);
          if (p.out_bf16) {
            uint2 o;
            o.x = pack_op2_g<INF>(a.x, a.y, p.fmt);
            o.y = pack_op2_g<INF>(a.z, a.w, p.fmt);
            *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + opix[itr] * N + c0) = o;
          } else {
            *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + opix[itr] * N + c0) = a;
          }
        }
        if (p.stats) {
          // lanes sharing `unit` hold the same 4-channel group: fold the row sub-blocks
#pragma unroll
          for (int off = Cfg::U; off < 32; off <<= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, off);
            s2 += __shfl_xor_sync(0xffffffffu, s2, off);
          }
          if (lane < Cfg::U) {
            my_stat[(ch * Cfg::U + lane) * 2 + 0] = s1;
            my_stat[(ch * Cfg::U + lane) * 2 + 1] = s2;
          }
        }
        __syncwarp();
      }
      if (p.stats) {
        epi_bar_sync<128 * Cfg::G>();
        const int t = threadIdx.x - 64;  // 0 .. 128 G - 1
        if (t < (N / 4) * 2) {
          const float* sb = stat_smem + (tcount & 1u) * 4 * (N / 4) * 2;
          const float tot = (sb[t] + sb[(N / 4) * 2 + t]) + (sb[2 * (N / 4) * 2 + t] + sb[3 * (N / 4) * 2 + t]);
          p.stats[(long long)tile * (N / 4) * 2 + t] = tot;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int N, bool INF = false>
static int launch_conv(const CUtensorMap& tm_w, const CUtensorMap* tm_a, const ConvParams& p, cudaStream_t stream) {
  using Cfg = ConvCfg<N>;
  ConvParams q = p;
  const int fixed = 1024 + q.n_seg * Cfg::W_SEG_BYTES + Cfg::STAGE_BYTES + Cfg::STAT_BYTES + 512;
  int stages = (232448 - fixed) / kATileBytes;
  if (stages > 8) stages = 8;
  MCEDM_REQUIRE(stages >= 2, "conv_igemm: %d segments x N=%d do not fit in shared memory", q.n_seg, N);
  q.n_stages = stages;
  const int smem = fixed + stages * kATileBytes;
  static bool attr_set = false;
  static int attr_smem = 0;
  if (!attr_set || smem > attr_smem) {
    MCEDM_CUDA(cudaFuncSetAttribute(conv_igemm_kernel<N, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    attr_set = true;
    attr_smem = 232448;
  }
  int grid = q.n_tiles < num_sms() ? q.n_tiles : num_sms();
  MCEDM_CUDA(launch_pdl(conv_igemm_kernel<N, INF>, dim3(grid), dim3(Cfg::THREADS), (size_t)smem, stream, tm_w, tm_a[0], tm_a[1], tm_a[2],
                        tm_a[3], q));
  return 0;
}

}  // namespace mcedm

static int conv_igemm_impl(const void* const* src, int n_src, const int* seg_src, const int* seg_dy,
                           const int* seg_dx, int n_seg, const void* w_packed, const float* bias, int B, int H,
                           int W, int N, void* out, int out_bf16, const float* res, int res_mode,
                           float* stats_partial, int op_fmt, int res16, int io_pitch, int io_blk, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(!res16 || (res_mode == 1 && N <= 64), "conv_igemm16: a 16-bit residual needs res_mode 1 and N <= 64");
  MCEDM_REQUIRE(io_pitch == 0 || (io_pitch >= W && io_blk >= (H + 2) * io_pitch), "conv_igemm16: bad padded-flat geometry");
  MCEDM_REQUIRE(n_src >= 1 && n_src <= 4, "conv_igemm: n_src=%d not in 1..4", n_src);
  MCEDM_REQUIRE(n_seg >= 1 && n_seg <= kMaxSeg, "conv_igemm: n_seg=%d not in 1..%d", n_seg, kMaxSeg);
  MCEDM_REQUIRE(W >= 8 && W <= 128 && (128 % W) == 0, "conv_igemm: W=%d must divide 128", W);
  MCEDM_REQUIRE(((long long)H * W) % 128 == 0, "conv_igemm: H*W=%d must be a multiple of 128", H * W);
  MCEDM_REQUIRE(B >= 1 && res_mode >= 0 && res_mode <= 3, "conv_igemm: bad B/res_mode");
  MCEDM_REQUIRE(res_mode == 0 || res != nullptr, "conv_igemm: res_mode=%d needs a residual tensor", res_mode);
  MCEDM_REQUIRE(res_mode != 2 || (H % 2 == 0 && W % 2 == 0), "conv_igemm: upsampled residual needs even H, W");
  ConvParams p;
  memset(&p, 0, sizeof(p));
  p.n_seg = n_seg;
  p.H = H;
  p.W = W;
  p.rows_per_tile = 128 / W;
  p.tiles_per_img = (H * W) / 128;
  p.n_tiles = B * p.tiles_per_img;
  for (int s = 0; s < n_seg; ++s) {
    MCEDM_REQUIRE(seg_src[s] >= 0 && seg_src[s] < n_src, "conv_igemm: segment %d names source %d", s, seg_src[s]);
    MCEDM_REQUIRE(seg_dy[s] >= -1 && seg_dy[s] <= 1 && seg_dx[s] >= -1 && seg_dx[s] <= 1,
                  "conv_igemm: segment %d tap (%d,%d) outside 3x3", s, seg_dy[s], seg_dx[s]);
    p.seg_src[s] = (signed char)seg_src[s];
    p.seg_dy[s] = (signed char)seg_dy[s];
    p.seg_dx[s] = (signed char)seg_dx[s];
  }
  p.bias = bias;
  p.out = out;
  p.out_bf16 = out_bf16;
  p.fmt = op_fmt ? 1 : 0;
  p.res = res;
  p.res_mode = res_mode;
  p.stats = stats_partial;
  p.res16 = res16 ? 1 : 0;
  p.io_pitch = io_pitch;
  p.io_blk = io_blk;
  p.err = watchdog_ptr();
  MCEDM_REQUIRE(p.err != nullptr, "conv_igemm: cannot allocate the watchdog word (no CUDA device?)");

  CUtensorMap tm_w, tm_a[4];
  int rc = make_tmap_rows64_bf16(&tm_w, w_packed, (long long)n_seg * N, N);
  if (rc) return rc;
  for (int i = 0; i < 4; ++i) {
    const void* ptr = src[i < n_src ? i : 0];
    rc = make_tmap_nhwc_bf16(&tm_a[i], ptr, B, H, W, 64, W, p.rows_per_tile);
    if (rc) return rc;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (op_fmt == MCEDM_FMT_F16_INF) {
    MCEDM_REQUIRE(N == 64 && out_bf16, "conv_igemm: op_fmt MCEDM_FMT_F16_INF is the N = 64 16-bit data-gradient launch");
    return launch_conv<64, true>(tm_w, tm_a, p, st);
  }
  switch (N) {
    case 16: return launch_conv<16>(tm_w, tm_a, p, st);
    case 64: return launch_conv<64>(tm_w, tm_a, p, st);
    case 128: return launch_conv<128>(tm_w, tm_a, p, st);
    case 192: return launch_conv<192>(tm_w, tm_a, p, st);
    default: return fail(-1, "conv_igemm: N=%d unsupported (16, 64, 128, 192)", N);
  }
}

extern "C" int mcedm_conv_igemm(const void* const* src, int n_src, const int* seg_src, const int* seg_dy,
                                const int* seg_dx, int n_seg, const void* w_packed, const float* bias, int B, int H,
                                int W, int N, void* out, int out_bf16, const float* res, int res_mode,
                                float* stats_partial, int op_fmt, void* stream) {
  return conv_igemm_impl(src, n_src, seg_src, seg_dy, seg_dx, n_seg, w_packed, bias, B, H, W, N, out, out_bf16, res,
                         res_mode, stats_partial, op_fmt, 0, 0, 0, stream);
}

extern "C" int mcedm_conv_igemm16(const void* const* src, int n_src, const int* seg_src, const int* seg_dy,
                                  const int* seg_dx, int n_seg, const void* w_packed, const float* bias, int B, int H,
                                  int W, int N, void* out16, const void* res16, int res_mode, int io_pitch, int io_blk,
                                  float* stats_partial, int op_fmt, void* stream) {
  return conv_igemm_impl(src, n_src, seg_src, seg_dy, seg_dx, n_seg, w_packed, bias, B, H, W, N, out16, 1,
                         reinterpret_cast<const float*>(res16), res_mode, stats_partial, op_fmt, res_mode == 1, io_pitch,
                         io_blk, stream);
}
