// K1c — 3x3 convolution for the narrow levels (W = 64, 32, 16): implicit GEMM on tcgen05 over a
// ZERO-PADDED FLAT pixel sequence, every input element fetched once.
//
// Same math as conv_igemm.cu / conv_rows.cu (models/adm_blocks.py:65-81 Conv2d.forward + fused residual
// :171).  A 128-row UMMA tile must be 128 consecutive shared-memory rows, which for W < 128 spans
// several image rows; with a dense layout a +-1 pixel shift would leak across row ends.  The bf16
// operand is therefore stored by the producing GroupNorm pass (gn.cu) in a padded layout:
//
//     image block (blk positions, a multiple of 128):  [P zeros][row 0: W px | 1 zero][row 1 ...] ... [zeros]
//     P = W + 1 = row pitch;  position(b, y, x) = b*blk + (y+1)*P + x
//
// so the whole tensor is ONE flat sequence of 128-byte pixels in which the filter tap (dy, dx) is the
// constant offset dy*P + dx and every out-of-image neighbour is a stored zero.  A tile = 128
// consecutive positions; its 9 A operands are row-shifted UMMA descriptors into a ring of 128-position
// chunks (chunk t-1, t, t+1 are adjacent in the ring; two mirror slots keep them adjacent across the
// wrap).  Each chunk is one 16 KB TMA load and serves 3 tiles x 9 taps.  Rows that fall on padding
// (6 % at 64x64, 12 % at 32x32; a pitch of W + 8 used to cost 19 % / 37 %) are computed and dropped by the epilogue.
//
// Warp roles / epilogue exactly as conv_rows.cu (8 epilogue warps, 4-deep TMEM accumulator ring,
// per-(tile, lane quarter) GroupNorm partial sums).
//
// FUSED variant (inference, mcedm_conv_flat_fused): as in conv_rows.cu, the source is the RAW 16-bit activation in
// the padded flat layout and four transform warps apply y = silu(a[b,c]*x + b[b,c]) (GroupNorm + scale/shift + SiLU,
// coefficients from mcedm_gn_coef) to every data position of a chunk in shared memory before its first MMA; padding
// positions are skipped so their zeros survive.  Output and residual are padded-flat too (output position == tile
// row position, so the epilogue stores are trivially coalesced): 16-bit, or fp32 for the K-split partial sum of the
// 128-channel decoder convs (pass 1 writes an fp32 partial, pass 2 adds it as its residual).
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

#include <cuda_bf16.h>
#include <cstdlib>

namespace mcedm {

constexpr int kChunkBytes = 16 * 1024;

struct FlatParams {
  int n_slots;             // ring depth S (physical slots = S + 2 mirrors)
  int H, W, P;             // image size, row pitch of the padded operand
  int tiles_per_img;       // blk / 128
  long long total_tiles;   // B * tiles_per_img
  const float* bias;
  float* out;              // fp32 NHWC [B,H,W,N] (unpadded)
  const float* res;
  int res_mode;            // 0 none, 1 same res, 2 nearest-x2 of [B,H/2,W/2,N], 3 2x2 mean of [B,2H,2W,N]
  float* stats;            // [total_tiles][4][N/4][2]
  int fmt;                 // 16-bit operand format: 0 bf16, 1 fp16
  unsigned int* err;
  // ---- FUSED variant only
  const float* coef;       // fp32 [B][128] = (a | b) of y = silu(a*x + b)
  int out_f32;             // out is fp32 padded-flat [B*blk][N] (K-split partial) instead of 16-bit padded-flat
  int res_f32;             // res (mode 1 only) is fp32 padded-flat
  int res_pitch, res_blk;  // layout of the 16-bit residual tensor at ITS resolution: 0,0 dense NHWC, else padded-flat
  int dbg;                 // bring-up switches (MCEDM_DBG): 4 saturation audit, 16 TMA-loaded chunks instead of direct loads
  const void* src;         // the padded-flat source itself (the transform warps' direct loads)
};

template <int N, bool FUSED>
struct FlatCfg {
  static constexpr int CH = 32;
  static constexpr int NCH = N / CH;
  static constexpr int U = 8;
  static constexpr int W_SEG_BYTES = N * 128;
  static constexpr int EPI_WARPS = 4 * NCH;
  static constexpr bool DUAL = FUSED;   // two MMA-issuing warps taking alternate tiles, see conv_rows.cu
  // WG (fused): roles laid out on warpgroup boundaries so that setmaxnreg can move registers between them:
  //   warps 0-3 TMA | MMA | MMA 2 | idle,  warps 4-11 epilogue,  warps 12-19 transform (EIGHT warps: with both MMA warps
  //   issuing, the four transform warps were this kernel's pacer).  640 threads launch at 96 registers; the transform
  //   groups and the first group drop to 80, the two epilogue groups take 120 (what they needed at 480 threads).
  //   setmaxnreg only moves registers INSIDE the CTA's launch allocation: 4 x 32 x 16 + 8 x 32 x 16 released = 8 x 32 x 24
  //   acquired (an inc that outruns the decs never returns).  `.aligned` means every warp of a warpgroup executes the SAME
  //   setmaxnreg instruction: each group has exactly one site (a dec per role branch of the first group - three
  //   different instructions - is undefined behaviour; it ran, and is the suspect of one launch failure in 8 x 99 x 8
  //   evaluations of an 8-GPU run).
  static constexpr bool WG = FUSED;
  static constexpr int XF_WARPS = FUSED ? 8 : 0;
  static constexpr int THREADS = WG ? 640 : 64 + 32 * EPI_WARPS;
  static constexpr int MMA2_WARP = WG ? 2 : -1;
  static constexpr int EPI_W0 = WG ? 4 : 2;
  static constexpr int XF_W0 = 12;
  static constexpr int STAGE_BYTES = EPI_WARPS * 32 * CH * 4;   // (the 16-bit fast-path epilogue uses half of it)
  static constexpr int ACC_BUFS = 4;
  static constexpr int TMEM_COLS = (ACC_BUFS * N <= 256) ? 256 : 512;
};

__device__ __forceinline__ uint64_t flat_desc(uint32_t addr) {
  constexpr uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
  const uint32_t lo = ((addr & 0x3FFFFu) >> 4) | (1u << 16);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

__device__ __forceinline__ float4 flat_residual(const FlatParams& p, int N, int b, int y, int x, int c0) {
  if (p.res_mode == 1) {
    return *reinterpret_cast<const float4*>(p.res + (((long long)b * p.H + y) * p.W + x) * N + c0);
  } else if (p.res_mode == 2) {
    return *reinterpret_cast<const float4*>(
        p.res + (((long long)b * (p.H >> 1) + (y >> 1)) * (p.W >> 1) + (x >> 1)) * N + c0);
  } else {
    const int Ws = p.W << 1;
    const float* r0 = p.res + (((long long)b * (p.H << 1) + 2 * y) * Ws + 2 * x) * N + c0;
    const float4 r00 = *reinterpret_cast<const float4*>(r0);
    const float4 r01 = *reinterpret_cast<const float4*>(r0 + N);
    const float4 r10 = *reinterpret_cast<const float4*>(r0 + (long long)Ws * N);
    const float4 r11 = *reinterpret_cast<const float4*>(r0 + (long long)Ws * N + N);
    return make_float4(0.25f * ((r00.x + r01.x) + (r10.x + r11.x)), 0.25f * ((r00.y + r01.y) + (r10.y + r11.y)),
                       0.25f * ((r00.z + r01.z) + (r10.z + r11.z)), 0.25f * ((r00.w + r01.w) + (r10.w + r11.w)));
  }
}

__device__ __forceinline__ float4 flat_unpack4(uint2 v, int fmt) {
  if (fmt) {
    const float2 lo = unpack_f16x2(v.x), hi = unpack_f16x2(v.y);
    return make_float4(lo.x, lo.y, hi.x, hi.y);
  }
  return make_float4(bf16_lo(v.x), bf16_hi(v.x), bf16_lo(v.y), bf16_hi(v.y));
}
// pixel index of (b, y, x) in a 16-bit tensor of height Hs / width Ws that is dense (pitch 0) or padded-flat
__device__ __forceinline__ long long flat_index(int pitch, int blk, int b, int y, int x, int Hs, int Ws) {
  if (pitch > 0) return (long long)b * blk + (long long)(y + 1) * pitch + x;
  return ((long long)b * Hs + y) * Ws + x;
}
// residual of the fused variant: 16-bit (any mode) or fp32 padded-flat (mode 1, the K-split partial sum)
__device__ __forceinline__ float4 flat_residual16(const FlatParams& p, int fmt, int N, int b, int y, int x, int c0,
                                                  long long pos) {
  const uint16_t* r16 = reinterpret_cast<const uint16_t*>(p.res);
  if (p.res_mode == 1) {
    if (p.res_f32) return *reinterpret_cast<const float4*>(p.res + pos * N + c0);
    return flat_unpack4(*reinterpret_cast<const uint2*>(r16 + pos * N + c0), fmt);
  } else if (p.res_mode == 2) {
    const long long i = flat_index(p.res_pitch, p.res_blk, b, y >> 1, x >> 1, p.H >> 1, p.W >> 1);
    return flat_unpack4(*reinterpret_cast<const uint2*>(r16 + i * N + c0), fmt);
  } else {
    const int Hs = p.H << 1, Ws = p.W << 1;
    const long long i00 = flat_index(p.res_pitch, p.res_blk, b, 2 * y, 2 * x, Hs, Ws);
    const long long rs = p.res_pitch > 0 ? p.res_pitch : Ws;
    const float4 r00 = flat_unpack4(*reinterpret_cast<const uint2*>(r16 + i00 * N + c0), fmt);
    const float4 r01 = flat_unpack4(*reinterpret_cast<const uint2*>(r16 + (i00 + 1) * N + c0), fmt);
    const float4 r10 = flat_unpack4(*reinterpret_cast<const uint2*>(r16 + (i00 + rs) * N + c0), fmt);
    const float4 r11 = flat_unpack4(*reinterpret_cast<const uint2*>(r16 + (i00 + rs + 1) * N + c0), fmt);
    return make_float4(0.25f * ((r00.x + r01.x) + (r10.x + r11.x)), 0.25f * ((r00.y + r01.y) + (r10.y + r11.y)),
                       0.25f * ((r00.z + r01.z) + (r10.z + r11.z)), 0.25f * ((r00.w + r01.w) + (r10.w + r11.w)));
  }
}
// 2 raw 16-bit values -> silu(a*x + b) (same arithmetic as conv_rows.cu xf_pair)
__device__ __forceinline__ uint32_t flat_xf_pair(uint32_t v, float a0, float b0, float a1, float b1, int fmt) {
  float x0, x1;
  if (fmt) {
    const float2 f = unpack_f16x2(v);
    x0 = f.x;
    x1 = f.y;
  } else {
    x0 = bf16_lo(v);
    x1 = bf16_hi(v);
  }
  // the coefficients arrive pre-halved: h = (a*x + b) / 2, silu(a*x + b) = h * (1 + tanh(h))
  return pack_op2(silu_from_half_arg(fmaf(x0, a0, b0)), silu_from_half_arg(fmaf(x1, a1, b1)), fmt);
}

// FM (fused only): epilogue variant folded at compile time: 0 fast path without residual, 1 fast path with a
// same-resolution 16-bit residual, 2 general path (resampled / fp32 residual, fp32 output); -1 = legacy unfused epilogue
// INF: fp16 stores without saturation (the data-gradient convs of dynamic loss scaling, op_fmt MCEDM_FMT_F16_INF)
template <int N, bool FUSED, int FM = -1, bool INF = false>
__global__ void __launch_bounds__(FlatCfg<N, FUSED>::THREADS, 1)
conv_flat_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_a,
                 const FlatParams p) {
  using Cfg = FlatCfg<N, FUSED>;
  const int fmt = FUSED ? 1 : p.fmt;      // the fused (inference) instantiation is fp16-only: folds at compile time
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int S = p.n_slots;
  uint8_t* w_smem = smem;
  uint8_t* ring = w_smem + 9 * Cfg::W_SEG_BYTES;               // (S + 2) chunk slots, contiguous
  uint8_t* stage_smem = ring + (S + 2) * kChunkBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_smem + Cfg::STAGE_BYTES);
  uint64_t* w_full = bars;
  uint64_t* acc_full = bars + 1;
  uint64_t* acc_empty = acc_full + Cfg::ACC_BUFS;
  uint64_t* c_full = acc_empty + Cfg::ACC_BUFS;                 // S
  uint64_t* c_empty = c_full + S;                               // S
  uint64_t* c_ready = c_empty + S;                              // S (FUSED: chunk transformed, visible to the MMA)
  uint64_t* turn = c_ready + S;                                 // 2 (DUAL: issue-order hand-over between the MMA warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(turn + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const long long t_begin = p.total_tiles * blockIdx.x / gridDim.x;
  const long long t_end = p.total_tiles * (blockIdx.x + 1) / gridDim.x;
  const int n_tiles = (int)(t_end - t_begin);
  // LDG mode: no TMA for the activation chunks.  The kernel is bounded by shared-memory traffic (operand fetch of the MMAs
  // + everything the warps move); TMA write + transform read + transform write cost 48 KB per chunk, a direct global load
  // into registers followed by ONE swizzled store costs 16.  (MCEDM_DBG & 16 selects TMA-loaded chunks instead: the path
  // that the direct loads are tested against.)
  const bool xf_ldg = FUSED && p.coef != nullptr && !(p.dbg & 16);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_w);
    prefetch_tmap(&tm_a);
    mbar_init(w_full, 1);
    for (int i = 0; i < Cfg::ACC_BUFS; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], Cfg::EPI_WARPS);              // one arrival per warp
    }
    for (int i = 0; i < S; ++i) {
      mbar_init(&c_full[i], 1);
      mbar_init(&c_empty[i], 1);
      mbar_init(&c_ready[i], FUSED ? Cfg::XF_WARPS : 1);
    }
    mbar_init(&turn[0], 1);
    mbar_init(&turn[1], 1);
    fence_barrier_init();
    // weights before pdl_wait (not written by the preceding kernel): the prologue overlaps the previous kernel's tail
    mbar_expect_tx(w_full, (uint32_t)(9 * Cfg::W_SEG_BYTES));
    for (int s = 0; s < 9; ++s) tma_load_2d(w_smem + s * Cfg::W_SEG_BYTES, &tm_w, w_full, 0, s * N);
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

  // (WG: every warpgroup has exactly ONE setmaxnreg site, and it dominates the group's role code so that ptxas budgets that
  // code accordingly: the first group's three roles therefore sit inside one block)
  const bool wg0 = Cfg::WG ? (warp < 4) : (warp == 0 || warp == 1 || warp == Cfg::MMA2_WARP);
  if (wg0) {
  if constexpr (Cfg::WG) setmaxnreg_dec<80>();
  if (warp == 0) {
    // ===================================== TMA producer =====================================
    // local chunk k (0 .. n_tiles+1) = global chunk t_begin - 1 + k; tile j uses chunks j, j+1, j+2
    if (lane == 0) {
      for (int k = 0; k < (xf_ldg ? 0 : n_tiles + 2); ++k) {
        const uint32_t slot = (uint32_t)k % (uint32_t)S, ph = ((uint32_t)k / (uint32_t)S) & 1u;
        mbar_wait(&c_empty[slot], ph ^ 1u, p.err, 0x3100 + slot);
        const bool mirror = slot < 2 && k >= S;
        mbar_expect_tx(&c_full[slot], mirror ? 2 * kChunkBytes : kChunkBytes);
        const long long row0 = (t_begin - 1 + k) * 128;       // may be -128 or past the end: zero-filled
        tma_load_2d(ring + slot * kChunkBytes, &tm_a, &c_full[slot], 0, (int)row0);
        if (mirror) tma_load_2d(ring + (S + slot) * kChunkBytes, &tm_a, &c_full[slot], 0, (int)row0);
      }
    }
  } else if (warp == 1 || warp == Cfg::MMA2_WARP) {
    // ====================================== MMA issuer ======================================
    // warp-uniform control flow, one elected lane issues (see conv_rows.cu)
    // DUAL (fused kernel): two warps take alternate tiles.  Tiles own separate accumulators, but the chunk ring is
    // released by commits that track only their own thread's MMAs, so the issue ORDER is handed over exactly as in
    // conv_rows.cu (the pipe executes in issue order: when tile j is complete so is tile j - 1).
    // lean issue loop (see conv_rows.cu): wrap-around ring counters, one election per tile, immediate offsets
    {
      const uint32_t idesc = umma_idesc_16(128, N, 0, 0, fmt);
      mbar_wait(w_full, 0, p.err, 0x3200);
      tc_fence_after();
      const uint32_t w_lo = (smem_u32(w_smem) >> 4) | (1u << 16);
      const uint32_t ring_lo = (smem_u32(ring) >> 4) | (1u << 16);
      constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
      auto desc = [&](uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; };
      // tap (ky, kx) = row offset ((ky-1)*P + (kx-1)) * 128 B from the centre chunk, in 16-byte units
      int tap_off[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) tap_off[t] = ((t / 3 - 1) * p.P + (t % 3 - 1)) * 8;
      uint32_t slot = 0, wslot = 0, wph = 0;
      int waited = 0;
      const uint32_t my_par = (warp == 1) ? 0u : 1u;
      uint32_t my_n = 0;
      for (int j = (!Cfg::DUAL && warp != 1) ? n_tiles : 0; j < n_tiles; ++j) {
        if (Cfg::DUAL && ((uint32_t)j & 1u) != my_par) {              // the other warp's tile: only the ring position moves
          slot = (slot + 1 == (uint32_t)S) ? 0u : slot + 1;
          continue;
        }
        const uint32_t buf = (uint32_t)j % Cfg::ACC_BUFS, aph = ((uint32_t)j / Cfg::ACC_BUFS) & 1u;
        mbar_wait(&acc_empty[buf], aph ^ 1u, p.err, 0x3300 + buf);
        while (waited < j + 3) {
          mbar_wait(FUSED ? &c_ready[wslot] : &c_full[wslot], wph, p.err, 0x3400 + wslot);
          ++waited;
          if (++wslot == (uint32_t)S) {
            wslot = 0;
            wph ^= 1u;
          }
        }
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * N;
        // window = slots slot, +1, +2 (mirrors keep them contiguous); the tile itself is the middle chunk
        const uint32_t centre = ring_lo + (slot + 1) * (kChunkBytes >> 4);
        const uint32_t s1 = (slot + 1 == (uint32_t)S) ? 0u : slot + 1;
        const uint32_t s2 = (s1 + 1 == (uint32_t)S) ? 0u : s1 + 1;
        // the nine A descriptor words are formed in warp-uniform code; the elected lane only issues
        uint32_t al[9];
#pragma unroll
        for (int t = 0; t < 9; ++t) al[t] = centre + (uint32_t)tap_off[t];
        if (Cfg::DUAL) {
          if (my_par == 1u) mbar_wait(&turn[1], my_n & 1u, p.err, 0x3a01);
          else if (my_n > 0) mbar_wait(&turn[0], (my_n - 1u) & 1u, p.err, 0x3a00);
        }
        if (elect_one()) {
#pragma unroll
          for (int t = 0; t < 9; ++t) {
            const uint64_t ad = desc(al[t]);
            const uint64_t bd = desc(w_lo + t * (Cfg::W_SEG_BYTES >> 4));
            umma_f16(d_tmem, ad, bd, idesc, t != 0 ? 1u : 0u);
            umma_f16(d_tmem, ad + 2, bd + 2, idesc, 1u);
            umma_f16(d_tmem, ad + 4, bd + 4, idesc, 1u);
            umma_f16(d_tmem, ad + 6, bd + 6, idesc, 1u);
          }
          if (Cfg::DUAL) mbar_arrive(&turn[my_par ^ 1u]);      // tile j issued: the other warp may issue tile j + 1
          umma_commit(&c_empty[slot]);        // chunk j has no further user
          if (j == n_tiles - 1) {
            umma_commit(&c_empty[s1]);
            umma_commit(&c_empty[s2]);
          }
          umma_commit(&acc_full[buf]);
        }
        __syncwarp();
        ++my_n;
        slot = s1;
      }
    }
  }
  } else if (!FUSED || (warp >= Cfg::EPI_W0 && warp < Cfg::EPI_W0 + Cfg::EPI_WARPS)) {
    // ======================================= epilogue =======================================
    if constexpr (Cfg::WG) setmaxnreg_inc<120>();     // (the ONE setmaxnreg instruction of the two epilogue warpgroups)
    const int q = warp & 3;
    const int ew = warp - Cfg::EPI_W0;
    const int ch = ew >> 2;
    const uint32_t my_stage = smem_u32(stage_smem) + ew * (32 * Cfg::CH * 4);
    const int unit = lane & 7;
    const int row_in_it = lane >> 3;
    const int c0 = ch * Cfg::CH + unit * 4;
    float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias) bz = *reinterpret_cast<const float4*>(p.bias + c0);
    // ---- fast path (FUSED, 16-bit output, residual none or same-resolution 16-bit: 22 of the 26 launches per
    // evaluation).  Output position == tile row position and the residual tensor has the same padded layout, so the
    // lane needs one base offset per tile and immediate offsets per row; padding rows are stored as zeros (which is
    // what they hold anyway) instead of being branched around, and add nothing to the statistics.
    if constexpr (FUSED && (FM == 0 || FM == 1)) {
      // 16-bit staging, as in conv_rows.cu (the kernel is bounded by shared-memory bytes per tile): the thread rounds
      // its position's 32 accumulators to fp16 and stages 64 B (XOR-swizzled 16-byte chunks); after the transposition a
      // lane owns 8 channels of 4 positions per pass, adds bias / residual in fp32, accumulates the GroupNorm sums,
      // rounds again and stores 16 B.  Half the staging bytes, half the shared / global memory instructions.
      const uint16_t* r16 = reinterpret_cast<const uint16_t*>(p.res);
      uint16_t* o16 = reinterpret_cast<uint16_t*>(p.out);
      constexpr bool has_res = FM == 1;
      const int u = lane & 3, rsub = lane >> 2;
      const int cc = ch * Cfg::CH + u * 8;                                   // first of this lane's 8 channels
      const uint32_t st16 = smem_u32(stage_smem) + ew * 2048;
      float bz8[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) bz8[e] = p.bias ? __ldg(p.bias + cc + e) : 0.f;
      uint4 rn[4];
      long long base = ((t_begin * 128) + q * 32 + rsub) * N + cc;          // element offset of this lane's first row
      if (has_res && n_tiles > 0) {
#pragma unroll
        for (int it = 0; it < 4; ++it) rn[it] = *reinterpret_cast<const uint4*>(r16 + base + it * 8 * N);
      }
      int tin = (int)(t_begin % p.tiles_per_img);                            // tile index inside its image
      for (int j = 0; j < n_tiles; ++j, base += 128 * N) {
        const long long tile = t_begin + j;
        const uint32_t buf = (uint32_t)j % Cfg::ACC_BUFS, aph = ((uint32_t)j / Cfg::ACC_BUFS) & 1u;
        // validity of the lane's 4 rows (8 positions apart; P >= 17: at most one row wrap per step): one division per tile
        const int pos = tin * 128 + q * 32 + rsub;
        int row = pos / p.P;
        int x = pos - row * p.P;
        uint32_t vmask = 0;
#pragma unroll
        for (int it = 0; it < 4; ++it, x += 8) {
          if (x >= p.P) {
            x -= p.P;
            ++row;
          }
          vmask |= ((row >= 1) && (row <= p.H) && (x < p.W)) ? (1u << it) : 0u;
        }
        if (++tin == p.tiles_per_img) tin = 0;
        uint4 rh[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) rh[it] = rn[it];
        if (has_res && j + 1 < n_tiles) {
#pragma unroll
          for (int it = 0; it < 4; ++it) rn[it] = *reinterpret_cast<const uint4*>(r16 + base + (128 + it * 8) * N);
        }
        mbar_wait(&acc_full[buf], aph, p.err, 0x3500 + buf);
        tc_fence_after();
        uint32_t v[32];
        tmem_ld_x32(tmem_base + ((uint32_t)(q * 32) << 16) + buf * N + ch * Cfg::CH, v);
        tmem_wait_ld();
        tc_fence_before();
        mbar_arrive_warp(&acc_empty[buf]);
        if (p.dbg & 4) {                          // the accumulator itself is rounded to fp16 for the staging tile
          float acc[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = __uint_as_float(v[i]);
          sat_audit(p.err, acc);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4 o;
          o.x = pack_f16x2_g<INF>(__uint_as_float(v[8 * c + 0]), __uint_as_float(v[8 * c + 1]));
          o.y = pack_f16x2_g<INF>(__uint_as_float(v[8 * c + 2]), __uint_as_float(v[8 * c + 3]));
          o.z = pack_f16x2_g<INF>(__uint_as_float(v[8 * c + 4]), __uint_as_float(v[8 * c + 5]));
          o.w = pack_f16x2_g<INF>(__uint_as_float(v[8 * c + 6]), __uint_as_float(v[8 * c + 7]));
          sts128(st16 + lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4), o);
        }
        __syncwarp();
        float sa1 = 0.f, sa2 = 0.f, sb1 = 0.f, sb2 = 0.f;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rr = it * 8 + rsub;
          const uint4 t = lds128(st16 + rr * 64 + ((u ^ ((rr >> 1) & 3)) << 4));
          const float m = (vmask >> it) & 1u ? 1.0f : 0.0f;                  // padding positions are stored as zeros
          float a[8];
          {
            const float2 t0 = unpack_f16x2(t.x), t1 = unpack_f16x2(t.y), t2 = unpack_f16x2(t.z), t3 = unpack_f16x2(t.w);
            a[0] = t0.x + bz8[0]; a[1] = t0.y + bz8[1]; a[2] = t1.x + bz8[2]; a[3] = t1.y + bz8[3];
            a[4] = t2.x + bz8[4]; a[5] = t2.y + bz8[5]; a[6] = t3.x + bz8[6]; a[7] = t3.y + bz8[7];
          }
          if (has_res) {
            const float2 r0 = unpack_f16x2(rh[it].x), r1 = unpack_f16x2(rh[it].y), r2 = unpack_f16x2(rh[it].z),
                         r3 = unpack_f16x2(rh[it].w);
            a[0] += r0.x; a[1] += r0.y; a[2] += r1.x; a[3] += r1.y;
            a[4] += r2.x; a[5] += r2.y; a[6] += r3.x; a[7] += r3.y;
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) a[e] *= m;
          if (p.dbg & 4) sat_audit(p.err, a);
          sa1 += (a[0] + a[1]) + (a[2] + a[3]);
          sa2 += (a[0] * a[0] + a[1] * a[1]) + (a[2] * a[2] + a[3] * a[3]);
          sb1 += (a[4] + a[5]) + (a[6] + a[7]);
          sb2 += (a[4] * a[4] + a[5] * a[5]) + (a[6] * a[6] + a[7] * a[7]);
          uint4 o;
          o.x = pack_f16x2_g<INF>(a[0], a[1]);
          o.y = pack_f16x2_g<INF>(a[2], a[3]);
          o.z = pack_f16x2_g<INF>(a[4], a[5]);
          o.w = pack_f16x2_g<INF>(a[6], a[7]);
          *reinterpret_cast<uint4*>(o16 + base + it * 8 * N) = o;
        }
        if (p.stats) {
#pragma unroll
          for (int off = 4; off < 32; off <<= 1) {
            sa1 += __shfl_xor_sync(0xffffffffu, sa1, off);
            sa2 += __shfl_xor_sync(0xffffffffu, sa2, off);
            sb1 += __shfl_xor_sync(0xffffffffu, sb1, off);
            sb2 += __shfl_xor_sync(0xffffffffu, sb2, off);
          }
          if (lane < 4)
            *reinterpret_cast<float4*>(p.stats + ((tile * 4 + q) * (N / 4) + ch * 8 + u * 2) * 2) =
                make_float4(sa1, sa2, sb1, sb2);
        }
        __syncwarp();
      }
    } else {
    // ---- general path
    // FUSED, 16-bit residual at the same or half resolution: the residual of tile j+1 is requested
    // before tile j is processed (raw register double buffer), otherwise every tile pays the DRAM latency in full.
    const bool pre = FUSED && ((p.res_mode == 1 && !p.res_f32) || p.res_mode == 2);
    uint2 rh_n[8];
    auto prefetch = [&](int j) {
      const long long tile = t_begin + j;
      const int b = (int)(tile / p.tiles_per_img);
      const int pos0 = (int)(tile - (long long)b * p.tiles_per_img) * 128 + q * 32;
      const uint16_t* r16 = reinterpret_cast<const uint16_t*>(p.res);
      int row = (pos0 + row_in_it) / p.P;            // one division per tile; the lane's rows are 4 positions apart
      int x = (pos0 + row_in_it) - row * p.P;
#pragma unroll
      for (int itr = 0; itr < 8; ++itr, x += 4) {
        if (x >= p.P) {
          x -= p.P;
          ++row;
        }
        rh_n[itr] = make_uint2(0u, 0u);
        if ((row >= 1) && (row <= p.H) && (x < p.W)) {
          const long long i = p.res_mode == 1 ? tile * 128 + q * 32 + itr * 4 + row_in_it
                                              : flat_index(p.res_pitch, p.res_blk, b, (row - 1) >> 1, x >> 1, p.H >> 1, p.W >> 1);
          rh_n[itr] = *reinterpret_cast<const uint2*>(r16 + i * N + c0);
        }
      }
    };
    if (pre && n_tiles > 0) prefetch(0);
    for (int j = 0; j < n_tiles; ++j) {
      const long long tile = t_begin + j;
      const uint32_t buf = (uint32_t)j % Cfg::ACC_BUFS, aph = ((uint32_t)j / Cfg::ACC_BUFS) & 1u;
      const int b = (int)(tile / p.tiles_per_img);
      const int pos0 = (int)(tile - (long long)b * p.tiles_per_img) * 128 + q * 32;
      // decode this lane's 8 rows (position -> image row / column; padding rows are dropped)
      long long opix[8];
      float4 rr[8];
      int row = (pos0 + row_in_it) / p.P;            // one division per tile; the lane's rows are 4 positions apart
      int x = (pos0 + row_in_it) - row * p.P;
#pragma unroll
      for (int itr = 0; itr < 8; ++itr, x += 4) {
        if (x >= p.P) {
          x -= p.P;
          ++row;
        }
        const bool valid = (row >= 1) && (row <= p.H) && (x < p.W);
        if constexpr (FUSED) {
          const long long gpos = tile * 128 + q * 32 + itr * 4 + row_in_it;    // padded-flat output position
          opix[itr] = valid ? gpos : -1;
          rr[itr] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (pre) rr[itr] = flat_unpack4(rh_n[itr], fmt);
          else if (valid && p.res_mode != 0) rr[itr] = flat_residual16(p, fmt, N, b, row - 1, x, c0, gpos);
        } else {
          opix[itr] = valid ? (((long long)b * p.H + (row - 1)) * p.W + x) : -1;
          rr[itr] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (valid && p.res_mode != 0) rr[itr] = flat_residual(p, N, b, row - 1, x, c0);
        }
      }
      if (pre && j + 1 < n_tiles) prefetch(j + 1);
      mbar_wait(&acc_full[buf], aph, p.err, 0x3500 + buf);
      tc_fence_after();
      uint32_t v[32];
      tmem_ld_x32(tmem_base + ((uint32_t)(q * 32) << 16) + buf * N + ch * Cfg::CH, v);
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive_warp(&acc_empty[buf]);
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const int pj = jj ^ (lane & 7);
        sts128(my_stage + lane * 128 + pj * 16, make_uint4(v[4 * jj], v[4 * jj + 1], v[4 * jj + 2], v[4 * jj + 3]));
      }
      __syncwarp();
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int itr = 0; itr < 8; ++itr) {
        const int row = itr * 4 + row_in_it;
        const int pu = unit ^ (row & 7);
        float4 a = lds128f(my_stage + row * 128 + pu * 16);
        if (opix[itr] >= 0) {
          a.x += bz.x; a.y += bz.y; a.z += bz.z; a.w += bz.w;
          a.x += rr[itr].x; a.y += rr[itr].y; a.z += rr[itr].z; a.w += rr[itr].w;
          s1 += (a.x + a.y) + (a.z + a.w);
          s2 += (a.x * a.x + a.y * a.y) + (a.z * a.z + a.w * a.w);
          if (FUSED && !p.out_f32) {
            uint2 o;
            o.x = pack_op2(a.x, a.y, fmt);
            o.y = pack_op2(a.z, a.w, fmt);
            *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(p.out) + opix[itr] * N + c0) = o;
          } else {
            *reinterpret_cast<float4*>(p.out + opix[itr] * N + c0) = a;
          }
        }
      }
      if (p.stats) {
#pragma unroll
        for (int off = 8; off < 32; off <<= 1) {
          s1 += __shfl_xor_sync(0xffffffffu, s1, off);
          s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        }
        if (lane < 8)
          *reinterpret_cast<float2*>(p.stats + ((tile * 4 + q) * (N / 4) + ch * 8 + lane) * 2) = make_float2(s1, s2);
      }
      __syncwarp();
    }
    }
  } else if (warp >= Cfg::XF_W0 && warp < Cfg::XF_W0 + Cfg::XF_WARPS) {
    // ============================ GroupNorm + SiLU transform (FUSED) ============================
    // thread t owns the logical 16-byte chunk jc = t & 7 (channels 8jc .. 8jc+7) of positions (t >> 3) + 16 i of every
    // 128-position chunk; physical 16-byte slot = jc ^ (position & 7) (SWIZZLE_128B, 1 KB-aligned chunk slots).
    if constexpr (Cfg::WG) setmaxnreg_dec<80>();      // (the ONE setmaxnreg instruction of the two transform warpgroups)
    const int t = (int)threadIdx.x - 32 * Cfg::XF_W0;
    const int jc = t & 7;
    const int prow = t >> 3;
    constexpr int XF_ROWS = FUSED ? 4 * Cfg::XF_WARPS : 16;   // positions covered per pass
    constexpr int XF_IT = 128 / XF_ROWS;
    int cur_b = -1;
    float ca[8], cb[8];
    // LDG mode: chunk k+1 is in flight in registers while chunk k is transformed (a chunk period is ~1.3 us)
    const uint4* srcp = reinterpret_cast<const uint4*>(p.src);
    uint4 n0[XF_IT];
    auto ldg_chunk = [&](int k, uint4 (&dst)[XF_IT]) {
      const long long g = t_begin - 1 + k;
      if (k < n_tiles + 2 && g >= 0 && g < p.total_tiles) {
        const uint4* a = srcp + (g * 128 + prow) * 8 + jc;
#pragma unroll
        for (int i = 0; i < XF_IT; ++i) dst[i] = ldg128_stream(a + (long long)i * XF_ROWS * 8);
      } else {
#pragma unroll
        for (int i = 0; i < XF_IT; ++i) dst[i] = make_uint4(0u, 0u, 0u, 0u);
      }
    };
    if (xf_ldg) ldg_chunk(0, n0);
    for (int k = 0; k < n_tiles + 2; ++k) {
      const uint32_t slot = (uint32_t)k % (uint32_t)S, ph = ((uint32_t)k / (uint32_t)S) & 1u;
      uint4 v[XF_IT];
      if (xf_ldg) {
#pragma unroll
        for (int i = 0; i < XF_IT; ++i) v[i] = n0[i];
        ldg_chunk(k + 1, n0);
        mbar_wait(&c_empty[slot], ph ^ 1u, p.err, 0x3100 + slot);     // the slot's previous chunk has no reader left
      } else {
        mbar_wait(&c_full[slot], ph, p.err, 0x3600 + slot);
      }
      const long long g = t_begin - 1 + k;                 // global chunk; outside the tensor = zero fill
      if (xf_ldg && !(g >= 0 && g < p.total_tiles)) {
        const uint32_t base = smem_u32(ring) + slot * kChunkBytes;
        const bool mirror = slot < 2 && k >= S;
#pragma unroll
        for (int i = 0; i < XF_IT; ++i) {
          const int pi = prow + XF_ROWS * i;
          const int off = pi * 128 + ((jc ^ (pi & 7)) << 4);
          sts128(base + off, make_uint4(0u, 0u, 0u, 0u));
          if (mirror) sts128(base + S * kChunkBytes + off, make_uint4(0u, 0u, 0u, 0u));
        }
        fence_proxy_async_smem();
      }
      if (g >= 0 && g < p.total_tiles && p.coef != nullptr) {
        const int b = (int)(g / p.tiles_per_img);
        const int base_pos = (int)(g - (long long)b * p.tiles_per_img) * 128;
        if (b != cur_b) {
          cur_b = b;
          const float4* cf = reinterpret_cast<const float4*>(p.coef + (long long)b * 128 + jc * 8);
          const float4 a0 = __ldg(cf), a1 = __ldg(cf + 1), b0 = __ldg(cf + 16), b1 = __ldg(cf + 17);
          ca[0] = a0.x; ca[1] = a0.y; ca[2] = a0.z; ca[3] = a0.w; ca[4] = a1.x; ca[5] = a1.y; ca[6] = a1.z; ca[7] = a1.w;
          cb[0] = b0.x; cb[1] = b0.y; cb[2] = b0.z; cb[3] = b0.w; cb[4] = b1.x; cb[5] = b1.y; cb[6] = b1.z; cb[7] = b1.w;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            ca[e] *= 0.5f;
            cb[e] *= 0.5f;
          }
        }
        const uint32_t base = smem_u32(ring) + slot * kChunkBytes;
        const bool mirror = slot < 2 && k >= S;
        bool ok[XF_IT];
        // (row, column) of this thread's first position; the next ones are XF_ROWS positions apart: one division per
        // chunk instead of one per position
        int row = (base_pos + prow) / p.P;
        int x = (base_pos + prow) - row * p.P;
#pragma unroll
        for (int i = 0; i < XF_IT; ++i) {
          const int pi = prow + XF_ROWS * i;
          ok[i] = (row >= 1) && (row <= p.H) && (x < p.W);
          if (!xf_ldg) v[i] = lds128(base + pi * 128 + ((jc ^ (pi & 7)) << 4));
          x += XF_ROWS;
          while (x >= p.P) {
            x -= p.P;
            ++row;
          }
        }
#pragma unroll
        for (int i = 0; i < XF_IT; ++i) {
          const int pi = prow + XF_ROWS * i;
          // branch-free (lanes of a warp sit on different positions): padding positions hold zeros and get them back
          uint4 o;
          o.x = flat_xf_pair(v[i].x, ca[0], cb[0], ca[1], cb[1], fmt);
          o.y = flat_xf_pair(v[i].y, ca[2], cb[2], ca[3], cb[3], fmt);
          o.z = flat_xf_pair(v[i].z, ca[4], cb[4], ca[5], cb[5], fmt);
          o.w = flat_xf_pair(v[i].w, ca[6], cb[6], ca[7], cb[7], fmt);
          if (!ok[i]) o = v[i];
          const int off = pi * 128 + ((jc ^ (pi & 7)) << 4);
          sts128(base + off, o);
          if (mirror) sts128(base + S * kChunkBytes + off, o);
        }
        fence_proxy_async_smem();
      }
      mbar_arrive_warp(&c_ready[slot]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace mcedm

extern "C" int mcedm_flat_geometry(int H, int W, int* pitch, int* block_positions) {
  using namespace mcedm;
  MCEDM_REQUIRE(W >= 16 && W <= 64 && H >= 1, "flat layout supports 16 <= W <= 64 (W=%d)", W);
  const int P = W + 1;     // one shared zero column between image rows is all the 3x3 taps need
  *pitch = P;
  *block_positions = ((H + 2) * P + 127) / 128 * 128;
  return 0;
}

namespace mcedm {
template <bool FUSED, int FM = -1, bool INF = false>
static int launch_flat(FlatParams p, const void* src_flat, const void* w_packed, int B, int blk, cudaStream_t st) {
  using Cfg = FlatCfg<64, FUSED>;
  const int N = 64;
  p.err = watchdog_ptr();
  p.src = src_flat;
  MCEDM_REQUIRE(p.err != nullptr, "conv_flat: cannot allocate the watchdog word");
  MCEDM_REQUIRE((long long)B * blk < (1LL << 31), "conv_flat: tensor too large for 32-bit TMA coordinates");
  const int fixed = 1024 + 9 * Cfg::W_SEG_BYTES + Cfg::STAGE_BYTES + 768;
  int slots = (232448 - fixed) / kChunkBytes - 2;
  if (slots > 6) slots = 6;
  MCEDM_REQUIRE(slots >= 3, "conv_flat: shared memory budget");
  p.n_slots = slots;
  const int smem = fixed + (slots + 2) * kChunkBytes;
  CUtensorMap tm_w, tm_a;
  int rc = make_tmap_rows64_bf16(&tm_w, w_packed, 9LL * N, N);
  if (rc) return rc;
  rc = make_tmap_rows64_bf16(&tm_a, src_flat, (long long)B * blk, 128);
  if (rc) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    MCEDM_CUDA(cudaFuncSetAttribute(conv_flat_kernel<64, FUSED, FM, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    attr_set = true;
  }
  long long grid = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
  MCEDM_CUDA(launch_pdl(conv_flat_kernel<64, FUSED, FM, INF>, dim3((unsigned)grid), dim3(Cfg::THREADS), (size_t)smem, st, tm_w, tm_a, p));
  return 0;
}
}  // namespace mcedm

extern "C" int mcedm_conv_flat(const void* src_flat, const void* w_packed, const float* bias, int B, int H, int W, int N,
                               float* out, const float* res, int res_mode, float* stats_partial, int op_fmt,
                               void* stream) {
  using namespace mcedm;
  int P = 0, blk = 0;
  int rc = mcedm_flat_geometry(H, W, &P, &blk);
  if (rc) return rc;
  MCEDM_REQUIRE(N == 64, "conv_flat: N=%d unsupported (64)", N);
  MCEDM_REQUIRE(res_mode >= 0 && res_mode <= 3 && (res_mode == 0 || res != nullptr), "conv_flat: bad residual mode");
  FlatParams p;
  memset(&p, 0, sizeof(p));
  p.H = H;
  p.W = W;
  p.P = P;
  p.tiles_per_img = blk / 128;
  p.total_tiles = (long long)B * p.tiles_per_img;
  p.bias = bias;
  p.out = out;
  p.res = res;
  p.res_mode = res_mode;
  p.stats = stats_partial;
  p.fmt = op_fmt ? 1 : 0;
  return launch_flat<false>(p, src_flat, w_packed, B, blk, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int mcedm_conv_flat_fused(const void* src_flat16, const float* coef, const void* w_packed, const float* bias,
                                     int B, int H, int W, int N, void* out_flat, int out_f32, const void* res,
                                     int res_mode, int res_f32, int res_pitch, int res_blk, float* stats_partial,
                                     int op_fmt, void* stream) {
  using namespace mcedm;
  int P = 0, blk = 0;
  int rc = mcedm_flat_geometry(H, W, &P, &blk);
  if (rc) return rc;
  MCEDM_REQUIRE(N == 64, "conv_flat_fused: N=%d unsupported (64)", N);
  MCEDM_REQUIRE(op_fmt == 1 || op_fmt == MCEDM_FMT_F16_INF,
                "conv_flat_fused: the fused inference kernels are fp16-only (op_fmt = 1)");
  MCEDM_REQUIRE(res_mode >= 0 && res_mode <= 3 && (res_mode == 0 || res != nullptr), "conv_flat_fused: bad residual mode");
  MCEDM_REQUIRE(!res_f32 || res_mode == 1, "conv_flat_fused: an fp32 residual must be same-resolution padded-flat");
  FlatParams p;
  memset(&p, 0, sizeof(p));
  p.H = H;
  p.W = W;
  p.P = P;
  p.tiles_per_img = blk / 128;
  p.total_tiles = (long long)B * p.tiles_per_img;
  p.bias = bias;
  p.out = reinterpret_cast<float*>(out_flat);
  p.out_f32 = out_f32 ? 1 : 0;
  p.res = reinterpret_cast<const float*>(res);
  p.res_mode = res_mode;
  p.res_f32 = res_f32 ? 1 : 0;
  p.res_pitch = res_pitch;
  p.res_blk = res_blk;
  p.stats = stats_partial;
  p.fmt = op_fmt ? 1 : 0;
  p.coef = coef;
  if (const char* e = getenv("MCEDM_DBG")) p.dbg = atoi(e);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (op_fmt == MCEDM_FMT_F16_INF) {
    // the data gradient of a 3x3 conv (no transform, no residual) is the one gradient this kernel writes
    MCEDM_REQUIRE(!p.out_f32 && p.res_mode == 0 && coef == nullptr,
                  "conv_flat_fused: op_fmt MCEDM_FMT_F16_INF is the data-gradient launch (16-bit out, no coefficients, no residual)");
    return launch_flat<true, 0, true>(p, src_flat16, w_packed, B, blk, st);
  }
  if (!p.out_f32 && p.res_mode == 0) return launch_flat<true, 0>(p, src_flat16, w_packed, B, blk, st);
  if (!p.out_f32 && p.res_mode == 1 && !p.res_f32) return launch_flat<true, 1>(p, src_flat16, w_packed, B, blk, st);
  return launch_flat<true, 2>(p, src_flat16, w_packed, B, blk, st);
}
