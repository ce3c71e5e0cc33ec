// K1b — 3x3 convolution for 128-pixel-wide images: implicit GEMM on tcgen05 with ROW-RESIDENT input.
//
// Same math and same packed-weight layout as conv_igemm.cu (models/adm_blocks.py:65-81 Conv2d.forward,
// fused residual :171 and 1x1 skip :150-151), specialised for the level that carries 68 % of the
// network's FLOPs (W = 128, one output tile = one image row).  conv_igemm fetches one 16 KB A tile per
// filter tap (9 L2->SMEM loads per tile) and measured L2-bandwidth bound at ~330 TFLOP/s; here every
// input row is fetched ONCE:
//
//   * a CTA owns a contiguous range of output rows (balanced over the grid: one wave, no tail);
//   * input row y of a source is one TMA box (64 ch, 130 px, 1, 1) at x = -1: 130 x 128 B with the
//     left/right zero padding supplied by TMA out-of-bounds fill, kept in a ring of row slots;
//   * the tap (dy, dx) of output row y is the SAME slot (input row y+dy) addressed through a UMMA
//     descriptor whose start address is advanced by (dx+1) * 128 B — SWIZZLE_128B is a function of the
//     absolute shared-memory address, so a row-shifted view of a swizzled tile is still a valid
//     K-major operand (pinned on silicon by tests/test_gpu_parity.py::test_umma_row_shifted_descriptor);
//   * each input row is used by 3 output rows x 3 dx taps = 9 segments before its slot is recycled:
//     L2->SMEM traffic drops from 147 KB to ~17 KB per tile.
//   * optional "centre" sources (the raw bf16 block input of the 1x1 skip projection) are plain
//     128 x 128 B tiles loaded once per output row.
//
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer / TMEM owner, warps 2-9 epilogue: two warps per
// TMEM lane quarter, each draining one 32-column half of the tile (4-deep TMEM accumulator ring; the
// residual tile is prefetched before the accumulator is waited for; GroupNorm partial sums are written
// per (tile, lane quarter) so the epilogue warps never synchronise with each other).
//
// FUSED variant (inference, mcedm_conv_rows_fused): the halo sources are RAW 16-bit activations (the residual stream
// or a conv0 output exactly as the producing conv stored it) and the GroupNorm + (1+scale)/shift + SiLU of
// adm_blocks.py:161/:166/:403 is applied IN SHARED MEMORY by four extra "transform" warps between the TMA load of a
// row and its first MMA: y = silu(a[b,c]*x + b[b,c]) with per-(sample, channel) coefficients from mcedm_gn_coef.
// The normalised operand therefore never exists in HBM (the separate gn_apply pass read 4 B and wrote 2 B per element
// per conv).  The transform rewrites each 16-byte chunk in place (same swizzled address), skips the two zero-padding
// pixel columns and the out-of-image rows (their zeros must stay zeros), then fence.proxy.async + mbarrier-arrives on
// h_ready[slot], which is what the MMA warp waits for in this variant.  Output, residual and the centre sources are
// 16-bit too; an output-channel window (n_off, n_total) lets a 128-channel conv run as two N=32 passes whose weights
// (72 KB each) stay resident.
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

#include <cuda_bf16.h>
#include <cstdlib>

namespace mcedm {

constexpr int kHaloRows = 130;
constexpr int kHaloBytes = 17 * 1024;          // 130 x 128 B = 16640, padded to a 1024 multiple
constexpr int kHaloTx = kHaloRows * 128;
constexpr int kCtrBytes = 16 * 1024;

struct RowsParams {
  int n_halo;            // 1..2 sources with 9 taps each
  int n_ctr;             // 0..2 centre-tap sources
  int n_slots;           // halo ring depth (input rows)
  int n_cslots;          // centre ring depth in 16 KB TILES (one tile = one centre source of one output row)
  int H;                 // image height; W == 128
  long long total_rows;  // B * H
  const float* bias;
  void* out;
  int out_bf16;
  int fmt;               // 16-bit operand format: 0 bf16, 1 fp16
  const float* res;
  int res_mode;          // 0 none, 1 same resolution, 2 nearest-x2 upsample of res
  float* stats;          // [total_rows][4 lane quarters][n_total/4][2]
  unsigned int* err;
  int n_off;             // first output channel of this launch inside the n_total-channel out / res / stats rows
  int n_total;           // channels per pixel of out / res (== N unless an output-channel window is used)
  int w_rows;            // rows per segment of the packed weight matrix (== n_total)
  const float* coef[2];  // FUSED: per halo source, fp32 [B][128] = (a | b) of y = silu(a*x + b); NULL = no transform
  int nchw_c;            // FUSED N = 16 head: > 0 -> out is fp32 NCHW [B, nchw_c, H, 128] (the network output F_x)
  int dbg;               // bring-up instrumentation (MCEDM_DBG): 2 drain-only epilogue, 4 saturation audit, 32 time every
                         // role's barrier waits, 64 time MMA issue / commits
  int res_pitch, res_blk; // FUSED, res_mode 2: the half-resolution residual is padded-flat (0,0: dense NHWC)
  int row_align;          // CTA row ranges are multiples of this many rows (1, or 4: see r_begin)
};

template <int N, bool FUSED>
struct RowsCfg {
  static constexpr int CH = N >= 32 ? 32 : 16;
  static constexpr int NCH = N / CH;
  static constexpr int U = CH / 4;
  static constexpr int W_SEG_BYTES = N * 128;
  static constexpr int EPI_WARPS = 4 * NCH;                 // one warp per (lane quarter, column chunk)
  // GroupNorm+SiLU transform warps (after the epilogue warps); the 16-wide head conv has a quarter of the MMA / epilogue
  // work per row, so there the transform is the pacer and gets eight
  // WG (fused N = 64): warps 0-3 TMA | MMA | MMA 2 | idle, 4-11 epilogue, 12-19 transform; 640 threads launch at 96
  // registers and setmaxnreg re-balances them (first group stays at 96, epilogue 128, transform 64: releases = acquisitions).
  // EIGHT transform warps without the spills that the plain 608-thread layout (104 registers for everybody) had.
  static constexpr bool WG = FUSED && N == 64;
  static constexpr int XF_WARPS = FUSED ? (N == 16 || WG ? 8 : 4) : 0;
  // A row's transform is a latency chain (wait for the TMA, shared-memory load, MUFU, store, proxy fence, hand-over) that
  // takes ~1300 cycles however many warps share it (head kernel: the same with 8 warps as the N = 64 kernel with 4), and
  // with all transform warps on the same row nothing overlaps it.  XF_SETS sets take alternate rows instead: the head
  // (8 warps, the transform is its pacer) goes from 185 to 159 us per launch at 256 samples; the N = 64 kernels lose
  // (two sets of two warps: 313 vs 302 us, 423 vs 363 with the residual - each thread then carries 16 chunks per row).
  static constexpr int XF_SETS = FUSED && N == 16 ? 2 : 1;
  static constexpr int XF_SET_WARPS = FUSED ? XF_WARPS / XF_SETS : 1;
  // DUAL: a second MMA-issuing warp (the last warp of the CTA) for the stacked kernels
  static constexpr bool DUAL = FUSED && (N == 64 || N == 16);
  static constexpr int THREADS = WG ? 640 : 64 + 32 * EPI_WARPS + 32 * XF_WARPS + (DUAL ? 32 : 0);
  static constexpr int MMA2_WARP = WG ? 2 : (DUAL ? THREADS / 32 - 1 : -1);
  static constexpr int EPI_W0 = WG ? 4 : 2;                  // first epilogue warp
  static constexpr int XF_W0 = WG ? 12 : 2 + EPI_WARPS;      // first transform warp
  // fused N = 64: the epilogue transposes through a 16-BIT staging tile (32 pixels x 64 B per warp), see the epilogue
  static constexpr bool EPI_H16 = FUSED && N == 64;
  static constexpr int STAGE_BYTES = EPI_H16 ? EPI_WARPS * 2048 : EPI_WARPS * 32 * CH * 4;
  // STACK (fused N = 64): the three vertical taps of a filter column are stacked into ONE N = 192 MMA per input row
  // (see the MMA issuer); eight 64-column accumulators then rotate through all 512 TMEM columns.
  static constexpr bool STACK = FUSED && (N == 64 || N == 16);   // N = 16: the head conv, 48 stacked B-rows
  static constexpr int ACC_BUFS = STACK ? 8 : 4;
  static constexpr int TMEM_COLS = (ACC_BUFS * N <= 32) ? 32 : (ACC_BUFS * N <= 64) ? 64 : (ACC_BUFS * N <= 128) ? 128
                                   : (ACC_BUFS * N <= 256) ? 256 : 512;
};

// bring-up instrumentation (MCEDM_DBG & 32): cycles each role spends inside its barrier waits, per CTA
__device__ long long g_rows_dbg[160][8];
__device__ __forceinline__ void timed_wait(uint64_t* bar, uint32_t parity, unsigned int* err, uint32_t tag, long long& acc,
                                           bool on) {
  if (!on) {
    mbar_wait(bar, parity, err, tag);
    return;
  }
  const long long t0 = clock64();
  mbar_wait(bar, parity, err, tag);
  acc += clock64() - t0;
}

// UMMA descriptor = constant high word | (address >> 4): the issuing thread only does 32-bit adds
__device__ __forceinline__ uint64_t desc_from_lo(uint32_t addr) {
  constexpr uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO=1024 | version 1 | SWIZZLE_128B
  const uint32_t lo = ((addr & 0x3FFFFu) >> 4) | (1u << 16);         // start address | LBO = 1
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

// 8 raw 16-bit values -> silu(a*x + b) -> 8 16-bit values (fp32 math; e^-v through one ex2 and one rcp)
__device__ __forceinline__ uint32_t xf_pair(uint32_t v, float a0, float b0, float a1, float b1, int fmt) {
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

// RM: residual mode folded at compile time (fused N = 64 instantiations; -1 = runtime p.res_mode)
// INF: fp16 stores without saturation (the data-gradient convs of dynamic loss scaling, op_fmt MCEDM_FMT_F16_INF)
template <int N, bool FUSED, int RM = -1, bool INF = false>
__global__ void __launch_bounds__(RowsCfg<N, FUSED>::THREADS, 1)
conv_rows_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_h0,
                 const __grid_constant__ CUtensorMap tm_h1, const __grid_constant__ CUtensorMap tm_c0,
                 const __grid_constant__ CUtensorMap tm_c1, const RowsParams p) {
  using Cfg = RowsCfg<N, FUSED>;
  // the fused (inference) instantiations are fp16-only (bf16 storage misses the 1e-2 bar): the format folds at compile time
  const int fmt = FUSED ? 1 : p.fmt;
  const int res_mode = RM >= 0 ? RM : p.res_mode;
  // fused N = 16 / 64 take exactly one halo source (128-channel convs are K-split): their source loops fold away
  const int n_halo = (FUSED && N != 32) ? 1 : p.n_halo;
  const bool out16 = (FUSED && N == 64) ? true : (p.out_bf16 != 0);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int n_seg = n_halo * 9 + p.n_ctr;
  const int slot_bytes = n_halo * kHaloBytes;
  uint8_t* w_smem = smem;
  uint8_t* h_smem = w_smem + n_seg * Cfg::W_SEG_BYTES;
  uint8_t* c_smem = h_smem + p.n_slots * slot_bytes;
  uint8_t* stage_smem = c_smem + p.n_cslots * kCtrBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_smem + Cfg::STAGE_BYTES);
  uint64_t* w_full = bars;
  uint64_t* acc_full = bars + 1;                     // ACC_BUFS
  uint64_t* acc_empty = acc_full + Cfg::ACC_BUFS;    // ACC_BUFS
  uint64_t* h_full = acc_empty + Cfg::ACC_BUFS;      // n_slots
  uint64_t* h_empty = h_full + p.n_slots;
  uint64_t* c_full = h_empty + p.n_slots;   // n_cslots
  uint64_t* c_empty = c_full + p.n_cslots;
  uint64_t* h_ready = c_empty + p.n_cslots;   // n_slots (FUSED: row transformed and visible to the async proxy)
  uint64_t* turn = h_ready + p.n_slots;       // 2 (DUAL: hand-over of the issue order between the two MMA warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(turn + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // balanced contiguous row range of this CTA, in units of `row_align` rows (4 for the fused N = 64 kernel, whose
  // GroupNorm partial sums are accumulated per 4-row block of an image: blocks must not straddle CTAs, and a record's
  // summation order must not depend on the batch size, which is what keeps row sharding bit-exact)
  const long long n_units = p.total_rows / p.row_align;
  const long long r_begin = n_units * blockIdx.x / gridDim.x * p.row_align;
  const long long r_end = n_units * (blockIdx.x + 1) / gridDim.x * p.row_align;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_w);
    prefetch_tmap(&tm_h0);
    mbar_init(w_full, 1);
    for (int i = 0; i < Cfg::ACC_BUFS; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], Cfg::EPI_WARPS);              // one arrival per warp
    }
    for (int i = 0; i < p.n_slots; ++i) {
      mbar_init(&h_full[i], 1);
      mbar_init(&h_empty[i], 1);
      mbar_init(&h_ready[i], FUSED ? Cfg::XF_SET_WARPS : 1);
    }
    for (int i = 0; i < p.n_cslots; ++i) {
      mbar_init(&c_full[i], 1);
      mbar_init(&c_empty[i], 1);
    }
    mbar_init(&turn[0], 1);
    mbar_init(&turn[1], 1);
    fence_barrier_init();
    // the packed weights are not written by the preceding kernel: their load is issued BEFORE pdl_wait, so under a
    // programmatic dependent launch it (and the whole prologue) overlaps the previous kernel's tail
    mbar_expect_tx(w_full, (uint32_t)(n_seg * Cfg::W_SEG_BYTES));
    for (int s = 0; s < n_seg; ++s) {
      // STACK keeps the taps of one filter column contiguous: slot (kx*3 + ky) holds tap (ky, kx)
      const int slot = (Cfg::STACK && s < 9) ? (s % 3) * 3 + s / 3 : s;
      tma_load_2d(w_smem + slot * Cfg::W_SEG_BYTES, &tm_w, w_full, 0, s * p.w_rows + p.n_off);
    }
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
      uint32_t hl = 0, cl = 0;   // halo rows / centre tiles loaded so far
      long long dbg_w0 = 0;
      const long long dbg_t0 = clock64();
      long long r = r_begin;
      while (r < r_end) {
        const int b = (int)(r / p.H);
        const int y0 = (int)(r - (long long)b * p.H);
        const int R = (int)((r_end - r) < (long long)(p.H - y0) ? (r_end - r) : (long long)(p.H - y0));
        for (int k = 0; k < R + 2; ++k) {
          const uint32_t slot = hl % (uint32_t)p.n_slots, ph = (hl / (uint32_t)p.n_slots) & 1u;
          timed_wait(&h_empty[slot], ph ^ 1u, p.err, 0x2100 + slot, dbg_w0, (p.dbg & 32) != 0);
          mbar_expect_tx(&h_full[slot], (uint32_t)(n_halo * kHaloTx));
          tma_load_4d(h_smem + slot * slot_bytes, &tm_h0, &h_full[slot], 0, -1, y0 - 1 + k, b);
          if (n_halo > 1)
            tma_load_4d(h_smem + slot * slot_bytes + kHaloBytes, &tm_h1, &h_full[slot], 0, -1, y0 - 1 + k, b);
          ++hl;
          if (p.n_ctr > 0 && k >= 2) {
            // the centre ring is tile-granular (one 16 KB tile per source and output row), so with n_ctr + 1 tiles the
            // next row's first source is already in flight while this row's tiles are consumed (a ring of whole rows
            // needed 2 x n_ctr tiles for any overlap, which the resident weights leave no room for)
            for (int s = 0; s < p.n_ctr; ++s, ++cl) {
              const uint32_t cs = cl % (uint32_t)p.n_cslots, cph = (cl / (uint32_t)p.n_cslots) & 1u;
              mbar_wait(&c_empty[cs], cph ^ 1u, p.err, 0x2200 + cs);
              mbar_expect_tx(&c_full[cs], (uint32_t)kCtrBytes);
              tma_load_4d(c_smem + cs * kCtrBytes, s == 0 ? &tm_c0 : &tm_c1, &c_full[cs], 0, 0, y0 + k - 2, b);
            }
          }
        }
        r += R;
      }
      if (p.dbg & 32) {
        g_rows_dbg[blockIdx.x][0] = dbg_w0;
        g_rows_dbg[blockIdx.x][7] = clock64() - dbg_t0;
      }
    }
  } else if (warp == 1 || warp == Cfg::MMA2_WARP) {
    // ====================================== MMA issuer ======================================
    // The whole warp runs the (warp-uniform) control flow so descriptors live in uniform registers; one
    // elected lane issues each tcgen05 instruction.  (Running this under `if (lane == 0)` made ptxas
    // emit an election loop + R2UR moves per MMA: ~4K issue cycles per tile on one thread, which was
    // the kernel's bottleneck.)
    if constexpr (Cfg::STACK) {
      // ---------------------------------------------------------------------------------------------------------
      // ky-stacked issue (N = 192).  With N = 64 every MMA re-reads its 4 KB A tile for 2 KB of weights and the pure
      // issue loop tops out at 1865 cycles per tile against 1152 of tensor time (scripts/probe_mma_rate.py: shared-
      // memory operand fetch); N = 128..192 runs at 96 % of the pipe.  So the loop is turned inside out: instead of
      // "output row <- 3 input rows x 3 taps" it is "input row k -> the three output rows k, k-1, k-2 it feeds", ONE
      // MMA per (kx, K step) with the weights of ky = 0, 1, 2 stacked as 192 B-rows.  Its 192 accumulator columns are
      // the 64-column accumulators of those three output rows, laid out in DESCENDING tile order around the 512 TMEM
      // columns so that they are adjacent; 12 MMAs per row instead of 36, A traffic cut 3x.  Splits: the very first
      // MMA into a fresh accumulator must not accumulate (single flag per instruction -> ky = 0 goes alone on
      // (kx, ks) = (0, 0)); a window that wraps past column 511 is issued in two pieces; segment edges drop the
      // sub-blocks whose output row is outside the CTA's range.
      // ---------------------------------------------------------------------------------------------------------
      const uint32_t idesc1 = umma_idesc_16(128, N, 0, 0, fmt), idesc2 = umma_idesc_16(128, 2 * N, 0, 0, fmt),
                     idesc3 = umma_idesc_16(128, 3 * N, 0, 0, fmt);
      mbar_wait(w_full, 0, p.err, 0x2300);
      tc_fence_after();
      const uint32_t ns = (uint32_t)p.n_slots;
      const uint32_t w_lo = (smem_u32(w_smem) >> 4) | (1u << 16);
      const uint32_t h_lo = (smem_u32(h_smem) >> 4) | (1u << 16);
      const uint32_t c_lo = (smem_u32(c_smem) >> 4) | (1u << 16);
      const uint32_t slot16 = (uint32_t)slot_bytes >> 4;
      constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
      auto desc = [&](uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; };
      uint32_t hs = 0, hph = 0;             // ring slot / phase of the next input row
      uint32_t cs = 0, cph = 0;
      uint32_t t0 = 0;                      // tile counter of the current segment's first output row
      long long dbg_w1 = 0, dbg_w2 = 0;
      const long long dbg_t0 = clock64();
      // ---------------------------------------------------------------------------------------------------------
      // DUAL issue.  tcgen05.mma queues only ~2 instructions deep (scripts/probe_mma_queue.py: cycles per row = tensor
      // time + whatever the issuing thread spends NOT issuing), and one row costs this warp ~1100 cycles of waits,
      // descriptor arithmetic, commits and loop control next to its 1152 cycles of MMAs: the tensor pipe idled for
      // almost half of every row.  Two warps now take alternate input rows ("steps").  Both run the identical control
      // flow and counters; a warp executes only the steps of its parity.  Accumulation order matters (the first MMA
      // into an output row's accumulator must precede every later contribution, and those come from the next two
      // steps), so the issue ORDER is handed over through two mbarriers: after its last MMA of step s the issuing lane
      // arrives on turn[other], which the other warp waits for before issuing step s + 1; while it issues, this warp
      // does its commits and the waits / arithmetic of step s + 2.  A commit tracks only its own thread's MMAs, but the
      // pipe executes in issue order, so when step s's MMAs are complete so are those of step s - 1.
      // ---------------------------------------------------------------------------------------------------------
      static_assert(Cfg::DUAL, "the stacked issue loop runs on two MMA warps");
      const uint32_t my_par = (warp == 1) ? 0u : 1u;
      uint32_t step = 0, my_n = 0;          // global step counter / steps issued by this warp
      long long r = r_begin;
      while (r < r_end) {
        const int b = (int)(r / p.H);
        const int y0 = (int)(r - (long long)b * p.H);
        const int R = (int)((r_end - r) < (long long)(p.H - y0) ? (r_end - r) : (long long)(p.H - y0));
        for (int k = 0; k < R + 2; ++k, ++step) {
          const bool ctr_step = p.n_ctr > 0 && k >= 2;
          if ((step & 1u) != my_par) {               // the other warp's step: advance the ring counters only
            if (++hs == ns) {
              hs = 0;
              hph ^= 1u;
            }
            if (ctr_step) {
              for (int s = 0; s < p.n_ctr; ++s) {
                if (++cs == (uint32_t)p.n_cslots) {
                  cs = 0;
                  cph ^= 1u;
                }
              }
            }
            continue;
          }
          if (k < R) {                      // output row k receives its first contribution from this input row
            const uint32_t tn = t0 + (uint32_t)k;
            timed_wait(&acc_empty[tn & 7u], ((tn >> 3) & 1u) ^ 1u, p.err, 0x2400 + (tn & 7u), dbg_w1, (p.dbg & 32) != 0);
          }
          timed_wait(&h_ready[hs], hph, p.err, 0x2500 + hs, dbg_w2, (p.dbg & 32) != 0);
          const bool ctr_now = p.n_ctr > 0 && k >= 2;      // centre tiles of output row k-2, just before it completes
          uint32_t cidx[2] = {0u, 0u};
          if (ctr_now) {
            uint32_t c = cs, ph = cph;
            for (int s = 0; s < p.n_ctr; ++s) {
              mbar_wait(&c_full[c], ph, p.err, 0x2600 + c);
              cidx[s] = c;
              if (++c == (uint32_t)p.n_cslots) {
                c = 0;
                ph ^= 1u;
              }
            }
          }
          tc_fence_after();
          const uint32_t a_row = h_lo + hs * slot16;
          const int kyA = k - (R - 1) > 0 ? k - (R - 1) : 0;   // output row k - ky must lie in [0, R)
          const int kyB = k < 2 ? k : 2;
          // Straight-line issue: every descriptor word below is (a value formed once per row in warp-uniform code) +
          // (a compile-time constant), so the elected lane executes little more than the tcgen05.mma themselves.
          // (A first version computed windows / splits inside the elected branch: ~165 cycles of dependent scalar
          // code per MMA, 2000 cycles per row before a single MMA was issued.)
          const uint32_t blk0 = (8u - ((t0 + (uint32_t)(k - kyA)) & 7u)) & 7u;      // accumulator block of B-row kyA
          const int nky = kyB - kyA + 1;
          const int split = (int)(8u - blk0) < nky ? (int)(8u - blk0) : nky;        // B-rows before the window wraps
          const uint32_t d0 = tmem_base + blk0 * (uint32_t)N;                        // first piece
          const uint32_t d1 = tmem_base + ((blk0 + (uint32_t)split) & 7u) * (uint32_t)N;   // piece after the wrap
          const uint32_t wrow = w_lo + (uint32_t)kyA * (Cfg::W_SEG_BYTES >> 4);
          const bool fresh = kyA == 0;        // output row k starts here: its very first MMA must not accumulate
          // issue order: step s - 1 (other warp) must have been issued.  Warp 0's n-th step waits for the other's n-th
          // arrival (none for n = 0), warp 1's n-th step for the (n + 1)-th.
          if (my_par == 1u) mbar_wait(&turn[1], my_n & 1u, p.err, 0x2a01);
          else if (my_n > 0) mbar_wait(&turn[0], (my_n - 1u) & 1u, p.err, 0x2a00);
          const long long dbg_c0 = (p.dbg & 64) ? clock64() : 0;
          if (nky == 3 && split == 3) {
            // interior row, contiguous window: N = 64 (fresh) + N = 128, then 11 x N = 192
            if (elect_one()) {
              umma_f16(d0, desc(a_row), desc(wrow), idesc1, 0u);
              umma_f16(d0 + (uint32_t)N, desc(a_row), desc(wrow + (Cfg::W_SEG_BYTES >> 4)), idesc2, 1u);
#pragma unroll
              for (int i = 1; i < 12; ++i) {
                const int kx = i >> 2, ks = i & 3;
                umma_f16(d0, desc(a_row + kx * 8 + ks * 2), desc(wrow + kx * 3 * (Cfg::W_SEG_BYTES >> 4) + ks * 2), idesc3, 1u);
              }
            }
          } else {
            // edge rows (fewer B-rows) and wrapped windows: pieces [kyA, kyA+split) at d0 and [kyA+split, kyB] at d1;
            // a fresh accumulator additionally takes ky = 0 alone on the first MMA
            const int n0 = split, n1 = nky - split;
            const uint32_t i0 = n0 == 1 ? idesc1 : n0 == 2 ? idesc2 : idesc3;
            const uint32_t i1 = n1 == 1 ? idesc1 : idesc2;
            const uint32_t w1 = wrow + (uint32_t)n0 * (Cfg::W_SEG_BYTES >> 4);
            if (elect_one()) {
#pragma unroll
              for (int i = 0; i < 12; ++i) {
                const int kx = i >> 2, ks = i & 3;
                const uint64_t ad = desc(a_row + kx * 8 + ks * 2);
                const uint32_t wo = kx * 3 * (Cfg::W_SEG_BYTES >> 4) + ks * 2;
                if (i == 0 && fresh && n0 > 1) {
                  // split the first piece: ky = 0 fresh, the rest of it accumulating
                  umma_f16(d0, ad, desc(wrow), idesc1, 0u);
                  umma_f16(d0 + (uint32_t)N, ad, desc(wrow + (Cfg::W_SEG_BYTES >> 4)), n0 == 2 ? idesc1 : idesc2, 1u);
                } else {
                  umma_f16(d0, ad, desc(wrow + wo), i0, (i == 0 && fresh) ? 0u : 1u);
                }
                if (n1 > 0) umma_f16(d1, ad, desc(w1 + wo), i1, 1u);
              }
            }
          }
          const long long dbg_c1 = (p.dbg & 64) ? clock64() : 0;
          if (elect_one()) {
            if (!ctr_now) mbar_arrive(&turn[my_par ^ 1u]);   // hand the issue order over
            umma_commit(&h_empty[hs]);                       // an input row is consumed entirely by its own step
            if (k >= 2) {
              const uint32_t td = t0 + (uint32_t)(k - 2);    // output row k-2 is complete after this step
              if (ctr_now) {
                const uint32_t blk = (8u - (td & 7u)) & 7u;
                for (int s = 0; s < p.n_ctr; ++s) {
                  const uint64_t ad = desc(c_lo + cidx[s] * (uint32_t)(kCtrBytes >> 4));
                  const uint64_t bd = desc(w_lo + (9 + s) * (Cfg::W_SEG_BYTES >> 4));
#pragma unroll
                  for (int ks = 0; ks < 4; ++ks) umma_f16(tmem_base + blk * (uint32_t)N, ad + 2 * ks, bd + 2 * ks, idesc1, 1u);
                  umma_commit(&c_empty[cidx[s]]);
                }
                mbar_arrive(&turn[my_par ^ 1u]);   // (centre MMAs of this step issued: hand over now)
              }
              umma_commit(&acc_full[td & 7u]);
            }
          }
          if (p.dbg & 64) {
            const long long dbg_c2 = clock64();
            dbg_w1 += dbg_c1 - dbg_c0;                       // MMA issue
            dbg_w2 += dbg_c2 - dbg_c1;                       // commits
          }
          __syncwarp();
          ++my_n;
          if (++hs == ns) {
            hs = 0;
            hph ^= 1u;
          }
          if (ctr_now) {
            for (int s = 0; s < p.n_ctr; ++s) {
              if (++cs == (uint32_t)p.n_cslots) {
                cs = 0;
                cph ^= 1u;
              }
            }
          }
        }
        t0 += (uint32_t)R;
        r += R;
      }
      if (warp == 1 && (p.dbg & 64)) {   // only the first issuer's elected lane measured: take the warp maximum
        for (int off = 16; off; off >>= 1) {
          const long long o1 = __shfl_xor_sync(0xffffffffu, dbg_w1, off), o2 = __shfl_xor_sync(0xffffffffu, dbg_w2, off);
          dbg_w1 = o1 > dbg_w1 ? o1 : dbg_w1;
          dbg_w2 = o2 > dbg_w2 ? o2 : dbg_w2;
        }
      }
      if ((p.dbg & 96) && lane == 0 && warp == 1) {
        g_rows_dbg[blockIdx.x][1] = dbg_w1;
        g_rows_dbg[blockIdx.x][2] = dbg_w2;
        g_rows_dbg[blockIdx.x][6] = clock64() - dbg_t0;
      }
    } else
    // Kept lean on purpose: this single warp's instruction stream paces the tensor pipe.  Ring positions are
    // wrap-around counters (no integer division), the three input rows' descriptor words are formed once per tile,
    // and ONE elected lane issues the tile's 36 tcgen05.mma back to back with immediate descriptor offsets
    // (the previous per-tap election + per-tap address arithmetic cost ~510 instructions per tile, which measured
    // as the limiter: tensor pipe 35 % active with every other role waiting).
    {
      const uint32_t idesc = umma_idesc_16(128, N, 0, 0, fmt);
      mbar_wait(w_full, 0, p.err, 0x2300);
      tc_fence_after();
      const uint32_t ns = (uint32_t)p.n_slots;
      const uint32_t w_lo = (smem_u32(w_smem) >> 4) | (1u << 16);          // descriptor low words: address >> 4 | LBO
      const uint32_t h_lo = (smem_u32(h_smem) >> 4) | (1u << 16);
      const uint32_t c_lo = (smem_u32(c_smem) >> 4) | (1u << 16);
      const uint32_t slot16 = (uint32_t)slot_bytes >> 4;
      constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO = 1024 | version 1 | SWIZZLE_128B
      auto desc = [&](uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; };
      uint32_t s0 = 0;                      // ring slot of the current tile's first input row
      uint32_t wslot = 0, wph = 0;          // next ring slot to wait for and its phase
      uint32_t waited = 0, need = 3;        // rows known to have landed / rows the current tile needs
      uint32_t cs = 0, cph = 0, tcount = 0;
      long long r = r_begin;
      while (r < r_end) {
        const int b = (int)(r / p.H);
        const int y0 = (int)(r - (long long)b * p.H);
        const int R = (int)((r_end - r) < (long long)(p.H - y0) ? (r_end - r) : (long long)(p.H - y0));
        for (int j = 0; j < R; ++j, ++tcount, ++need) {
          const uint32_t buf = tcount % Cfg::ACC_BUFS, aph = (tcount / Cfg::ACC_BUFS) & 1u;
          mbar_wait(&acc_empty[buf], aph ^ 1u, p.err, 0x2400 + buf);
          while (waited < need) {
            mbar_wait(FUSED ? &h_ready[wslot] : &h_full[wslot], wph, p.err, 0x2500 + wslot);
            ++waited;
            if (++wslot == ns) {
              wslot = 0;
              wph ^= 1u;
            }
          }
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + buf * N;
          const uint32_t s1 = (s0 + 1 == ns) ? 0u : s0 + 1;
          const uint32_t s2 = (s1 + 1 == ns) ? 0u : s1 + 1;
          const uint32_t a_lo[3] = {h_lo + s0 * slot16, h_lo + s1 * slot16, h_lo + s2 * slot16};
          if (elect_one()) {
#pragma unroll
            for (int s = 0; s < 2; ++s) {
              if (s < n_halo) {
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
                  for (int kx = 0; kx < 3; ++kx) {
                    // (dx + 1) pixel rows into the halo'd row = +8 in the (address >> 4) field; +32 B along K = +2
                    const uint64_t ad = desc(a_lo[ky] + s * (kHaloBytes >> 4) + kx * 8);
                    const uint64_t bd = desc(w_lo + (s * 9 + ky * 3 + kx) * (Cfg::W_SEG_BYTES >> 4));
                    umma_f16(d_tmem, ad, bd, idesc, (s | ky | kx) != 0 ? 1u : 0u);
                    umma_f16(d_tmem, ad + 2, bd + 2, idesc, 1u);
                    umma_f16(d_tmem, ad + 4, bd + 4, idesc, 1u);
                    umma_f16(d_tmem, ad + 6, bd + 6, idesc, 1u);
                  }
                }
              }
            }
          }
          uint32_t cidx[2] = {0u, 0u};
          if (p.n_ctr > 0) {
            // centre tiles last: they are the ones most likely to be late
            uint32_t c = cs, ph = cph;
            for (int s = 0; s < p.n_ctr; ++s) {
              mbar_wait(&c_full[c], ph, p.err, 0x2600 + c);
              cidx[s] = c;
              if (++c == (uint32_t)p.n_cslots) {
                c = 0;
                ph ^= 1u;
              }
            }
            tc_fence_after();
          }
          if (elect_one()) {
            if (p.n_ctr > 0) {
              for (int s = 0; s < p.n_ctr; ++s) {
                const uint64_t ad = desc(c_lo + cidx[s] * (uint32_t)(kCtrBytes >> 4));
                const uint64_t bd = desc(w_lo + (n_halo * 9 + s) * (Cfg::W_SEG_BYTES >> 4));
#pragma unroll
                for (int k = 0; k < 4; ++k) umma_f16(d_tmem, ad + 2 * k, bd + 2 * k, idesc, 1u);
                umma_commit(&c_empty[cidx[s]]);
              }
            }
            // input row s0 has no further user; the last output row of a segment also frees the two rows below it
            umma_commit(&h_empty[s0]);
            if (j == R - 1) {
              umma_commit(&h_empty[s1]);
              umma_commit(&h_empty[s2]);
            }
            umma_commit(&acc_full[buf]);
          }
          __syncwarp();
          s0 = s1;
          for (int s = 0; s < p.n_ctr; ++s) {
            if (++cs == (uint32_t)p.n_cslots) {
              cs = 0;
              cph ^= 1u;
            }
          }
        }
        // the next segment starts two rows further on (its own top halo row and the one above it)
        s0 = (s0 + 1 == ns) ? 0u : s0 + 1;
        s0 = (s0 + 1 == ns) ? 0u : s0 + 1;
        need += 2;
        r += R;
      }
    }
  } else if (Cfg::WG && warp == 3) {
    // the idle fourth warp of the first group (TMA | MMA | MMA 2 | idle keep their 96 registers)
  } else if (!FUSED || (warp >= Cfg::EPI_W0 && warp < Cfg::EPI_W0 + Cfg::EPI_WARPS)) {
    if constexpr (Cfg::WG) setmaxnreg_inc<128>();
    // ======================================= epilogue =======================================
    const int q = warp & 3;                 // TMEM lane quarter
    const int ew = warp - Cfg::EPI_W0;      // 0 .. EPI_WARPS-1
    const int ch = ew >> 2;                 // column chunk drained by this warp
    if constexpr (Cfg::EPI_H16) {
      // ---------------------------------------------------------------------------------------------------------
      // 16-bit staging.  (Also measured and dropped: the 8 warps as two SETS of 4 on alternate tiles, each warp draining
      // both 32-column halves of its lane quarter, so that consecutive tiles' latency chains overlap: 317 vs 301 us.)  The kernel is bounded by shared-memory BYTES per row (MMA operand fetch 120 KB + TMA 17 KB +
      // transform 32 KB + epilogue staging; scripts/rows_ablate.py: 9.7 cycles per KB), and the fp32 staging tile
      // (32 KB written + 32 KB read back per row) was the largest item the kernel itself controls.  Now each thread
      // rounds its pixel's 32 accumulators to fp16 FIRST and stages 64 B (4 x 16-byte chunks, XOR-swizzled with
      // (pixel >> 1) & 3: conflict-free both ways); after the transposition a lane owns 8 channels (16 B) of 4
      // pixels per pass, adds bias and the residual in fp32, accumulates the GroupNorm sums, rounds again and stores
      // 16 B (4 lanes = one pixel's 64-byte chunk, 8 pixels per store instruction).  16 KB + 16 KB per row instead of
      // 32 + 32; half as many shared and global memory instructions.  Price: the accumulator is rounded to fp16
      // before bias / residual are added (one extra 2^-12 relative rounding on a tensor that is stored in fp16 anyway).
      // GroupNorm partial sums are kept in registers across the 4 rows of an image-row block and written once per
      // block: one record per (4-row block, lane quarter) = H records per image instead of 4 H.
      // ---------------------------------------------------------------------------------------------------------
      const int u = lane & 3, rsub = lane >> 2;      // 16-byte channel chunk / pixel inside an 8-pixel pass
      const int NT = p.n_total;
      const int cg = p.n_off + ch * 32 + u * 8;      // first of this lane's 8 channels inside the out / res rows
      float bz[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) bz[e] = p.bias ? __ldg(p.bias + cg + e) : 0.f;
      const uint16_t* res16 = reinterpret_cast<const uint16_t*>(p.res);
      uint16_t* out16p = reinterpret_cast<uint16_t*>(p.out);
      const uint32_t st16 = smem_u32(stage_smem) + ew * 2048;
      uint4 rn[4];                                   // residual of the NEXT tile (requested one tile ahead)
      auto load_res = [&](long long r) {
        if (res_mode == 1) {
          const long long o = (r * 128 + q * 32 + rsub) * NT + cg;
#pragma unroll
          for (int it = 0; it < 4; ++it) rn[it] = *reinterpret_cast<const uint4*>(res16 + o + (long long)it * 8 * NT);
        } else if (res_mode == 2) {
          const int bimg = (int)(r / p.H);
          const int y = (int)(r - (long long)bimg * p.H);
          const long long rrow = (p.res_pitch > 0)
                                     ? ((long long)bimg * p.res_blk + (long long)((y >> 1) + 1) * p.res_pitch) * NT + cg
                                     : ((long long)bimg * (p.H >> 1) + (y >> 1)) * 64 * NT + cg;
#pragma unroll
          for (int it = 0; it < 4; ++it)
            rn[it] = *reinterpret_cast<const uint4*>(res16 + rrow + ((q * 32 + it * 8 + rsub) >> 1) * NT);
        }
      };
      if (r_begin < r_end) load_res(r_begin);
      float sa1 = 0.f, sa2 = 0.f, sb1 = 0.f, sb2 = 0.f;     // (sum, sum of squares) of this lane's two 4-channel groups
      long long dbg_w3 = 0;
      const long long dbg_t0 = clock64();
      uint32_t tcount = 0;
      for (long long r = r_begin; r < r_end; ++r, ++tcount) {
        const uint32_t buf = tcount % Cfg::ACC_BUFS, aph = (tcount / Cfg::ACC_BUFS) & 1u;
        uint4 rh[4];
#pragma unroll
        for (int it = 0; it < 4; ++it) rh[it] = rn[it];
        if (r + 1 < r_end) load_res(r + 1);
        timed_wait(&acc_full[buf], aph, p.err, 0x2700 + buf, dbg_w3, (p.dbg & 32) != 0);
        tc_fence_after();
        uint32_t v[32];
        const uint32_t acc_col = ((8u - buf) & 7u) * (uint32_t)N;          // STACK: descending tile order
        tmem_ld_x32(tmem_base + ((uint32_t)(q * 32) << 16) + acc_col + ch * 32, v);
        tmem_wait_ld();
        tc_fence_before();
        mbar_arrive_warp(&acc_empty[buf]);
        if (p.dbg & 2) continue;                  // bring-up: drain-only epilogue
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
        const long long pix0 = r * 128 + q * 32;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int rr = it * 8 + rsub;
          const uint4 t = lds128(st16 + rr * 64 + ((u ^ ((rr >> 1) & 3)) << 4));
          float a[8];
          {
            const float2 t0 = unpack_f16x2(t.x), t1 = unpack_f16x2(t.y), t2 = unpack_f16x2(t.z), t3 = unpack_f16x2(t.w);
            a[0] = t0.x + bz[0]; a[1] = t0.y + bz[1]; a[2] = t1.x + bz[2]; a[3] = t1.y + bz[3];
            a[4] = t2.x + bz[4]; a[5] = t2.y + bz[5]; a[6] = t3.x + bz[6]; a[7] = t3.y + bz[7];
          }
          if (res_mode != 0) {
            const float2 r0 = unpack_f16x2(rh[it].x), r1 = unpack_f16x2(rh[it].y), r2 = unpack_f16x2(rh[it].z),
                         r3 = unpack_f16x2(rh[it].w);
            a[0] += r0.x; a[1] += r0.y; a[2] += r1.x; a[3] += r1.y;
            a[4] += r2.x; a[5] += r2.y; a[6] += r3.x; a[7] += r3.y;
          }
          sa1 += (a[0] + a[1]) + (a[2] + a[3]);
          sa2 += (a[0] * a[0] + a[1] * a[1]) + (a[2] * a[2] + a[3] * a[3]);
          sb1 += (a[4] + a[5]) + (a[6] + a[7]);
          sb2 += (a[4] * a[4] + a[5] * a[5]) + (a[6] * a[6] + a[7] * a[7]);
          if (p.dbg & 4) sat_audit(p.err, a);
          uint4 o;
          o.x = pack_f16x2_g<INF>(a[0], a[1]);
          o.y = pack_f16x2_g<INF>(a[2], a[3]);
          o.z = pack_f16x2_g<INF>(a[4], a[5]);
          o.w = pack_f16x2_g<INF>(a[6], a[7]);
          *reinterpret_cast<uint4*>(out16p + (pix0 + rr) * NT + cg) = o;
        }
        if ((r & 3) == 3) {
          // end of a 4-row block (ranges are block-aligned and H % 4 == 0, so blocks never straddle images or CTAs):
          // lanes with equal `u` hold the same two groups
          if (p.stats) {
#pragma unroll
            for (int off = 4; off < 32; off <<= 1) {
              sa1 += __shfl_xor_sync(0xffffffffu, sa1, off);
              sa2 += __shfl_xor_sync(0xffffffffu, sa2, off);
              sb1 += __shfl_xor_sync(0xffffffffu, sb1, off);
              sb2 += __shfl_xor_sync(0xffffffffu, sb2, off);
            }
            if (lane < 4)
              *reinterpret_cast<float4*>(p.stats + (((r >> 2) * 4 + q) * (NT / 4) + (cg >> 2)) * 2) =
                  make_float4(sa1, sa2, sb1, sb2);
          }
          sa1 = sa2 = sb1 = sb2 = 0.f;
        }
        __syncwarp();                              // the staging tile is rewritten by the next tile
      }
      if ((p.dbg & 32) && warp == Cfg::EPI_W0 && lane == 0) {
        g_rows_dbg[blockIdx.x][3] = dbg_w3;
        g_rows_dbg[blockIdx.x][5] = clock64() - dbg_t0;
      }
    } else {
    const uint32_t my_stage = smem_u32(stage_smem) + ew * (32 * Cfg::CH * 4);
    const int unit = lane % Cfg::U;
    const int row_in_it = lane / Cfg::U;
    constexpr int ROWS_PER_IT = 32 / Cfg::U;
    const int c0 = ch * Cfg::CH + unit * 4;          // column inside this launch's N-wide window
    const int NT = p.n_total;                        // channels per pixel of out / res
    const int cg = p.n_off + c0;                     // column inside the out / res rows
    float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias) bz = *reinterpret_cast<const float4*>(p.bias + cg);
    const uint16_t* res16 = reinterpret_cast<const uint16_t*>(p.res);
    // The residual of tile r+1 is requested before tile r is processed (register double buffer): with all epilogue
    // warps on the same tile, a load issued at the top of its own tile would expose the full DRAM latency per tile.
    float4 rr_n[FUSED ? 1 : Cfg::U];      // fp32 residual (training / unfused path)
    uint2 rh_n[FUSED ? Cfg::U : 1];       // 16-bit residual (fused path)
    auto load_res = [&](long long r) {
      const long long pix0 = r * 128 + q * 32;
      if (res_mode == 1) {
#pragma unroll
        for (int itr = 0; itr < Cfg::U; ++itr) {
          const long long o = (pix0 + itr * ROWS_PER_IT + row_in_it) * NT + cg;
          if constexpr (FUSED) rh_n[itr] = *reinterpret_cast<const uint2*>(res16 + o);
          else rr_n[itr] = *reinterpret_cast<const float4*>(p.res + o);
        }
      } else if (res_mode == 2) {
        const int bimg = (int)(r / p.H);
        const int y = (int)(r - (long long)bimg * p.H);
        const long long rrow = (FUSED && p.res_pitch > 0)
                                   ? ((long long)bimg * p.res_blk + (long long)((y >> 1) + 1) * p.res_pitch) * NT + cg
                                   : ((long long)bimg * (p.H >> 1) + (y >> 1)) * 64 * NT + cg;
#pragma unroll
        for (int itr = 0; itr < Cfg::U; ++itr) {
          const long long o = rrow + ((q * 32 + itr * ROWS_PER_IT + row_in_it) >> 1) * NT;
          if constexpr (FUSED) rh_n[itr] = *reinterpret_cast<const uint2*>(res16 + o);
          else rr_n[itr] = *reinterpret_cast<const float4*>(p.res + o);
        }
      }
    };
    if (r_begin < r_end) load_res(r_begin);
    long long dbg_w3 = 0;
    const long long dbg_t0 = clock64();
    uint32_t tcount = 0;
    for (long long r = r_begin; r < r_end; ++r, ++tcount) {
      const uint32_t buf = tcount % Cfg::ACC_BUFS, aph = (tcount / Cfg::ACC_BUFS) & 1u;
      const long long pix0 = r * 128 + q * 32;
      float4 rr[FUSED ? 1 : Cfg::U];
      uint2 rh[FUSED ? Cfg::U : 1];
#pragma unroll
      for (int itr = 0; itr < (FUSED ? 1 : Cfg::U); ++itr) rr[itr] = rr_n[itr];
#pragma unroll
      for (int itr = 0; itr < (FUSED ? Cfg::U : 1); ++itr) rh[itr] = rh_n[itr];
      if (r + 1 < r_end) load_res(r + 1);
      timed_wait(&acc_full[buf], aph, p.err, 0x2700 + buf, dbg_w3, (p.dbg & 32) != 0);
      tc_fence_after();
      uint32_t v[Cfg::CH];
      const uint32_t acc_col = Cfg::STACK ? ((8u - buf) & 7u) * (uint32_t)N : buf * N;   // STACK: descending tile order
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc_col + ch * Cfg::CH;
      if constexpr (Cfg::CH == 32) tmem_ld_x32(taddr, v); else tmem_ld_x16(taddr, v);
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive_warp(&acc_empty[buf]);
      if (FUSED && (p.dbg & 2)) continue;       // bring-up: drain-only epilogue (what would a free epilogue buy?)
      if constexpr (FUSED && N == 16) {
        if (p.nchw_c > 0) {
          // output head (adm_blocks.py:403): the TMEM layout (lane = pixel) IS the NCHW order along x, so the first
          // nchw_c accumulator columns go straight to F_x[b, c, y, :] as coalesced 128-byte rows - no staging, no
          // 16-channel NHWC intermediate, no separate head_to_nchw pass
          // (one 32-bit division per row; the 16 predicated stores with their own 64-bit address arithmetic and bias
          // loads cost the epilogue ~1100 cycles per row and made it this kernel's pacer)
          const int bimg = (int)((unsigned long long)r / (unsigned)p.H);
          const int y = (int)(r - (long long)bimg * p.H);
          float* F = reinterpret_cast<float*>(p.out) + ((long long)bimg * p.nchw_c * p.H + y) * 128 + q * 32 + lane;
          const long long cstride = (long long)p.H * 128;
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            if (c >= p.nchw_c) break;
            F[c * cstride] = __uint_as_float(v[c]) + __ldg(p.bias + c);
          }
          continue;
        }
      }
#pragma unroll
      for (int j = 0; j < Cfg::U; ++j) {
        const int pj = j ^ (lane & (Cfg::U - 1));
        sts128(my_stage + lane * (Cfg::CH * 4) + pj * 16, make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
      }
      __syncwarp();
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int itr = 0; itr < Cfg::U; ++itr) {
        const int row = itr * ROWS_PER_IT + row_in_it;
        const int pu = unit ^ (row & (Cfg::U - 1));
        float4 a = lds128f(my_stage + row * (Cfg::CH * 4) + pu * 16);
        a.x += bz.x; a.y += bz.y; a.z += bz.z; a.w += bz.w;
        if (res_mode != 0) {
          if constexpr (FUSED) {
            float2 lo, hi;
            if (fmt) {
              lo = unpack_f16x2(rh[itr].x);
              hi = unpack_f16x2(rh[itr].y);
            } else {
              lo = make_float2(bf16_lo(rh[itr].x), bf16_hi(rh[itr].x));
              hi = make_float2(bf16_lo(rh[itr].y), bf16_hi(rh[itr].y));
            }
            a.x += lo.x; a.y += lo.y; a.z += hi.x; a.w += hi.y;
          } else {
            a.x += rr[itr].x; a.y += rr[itr].y; a.z += rr[itr].z; a.w += rr[itr].w;
          }
        }
        s1 += (a.x + a.y) + (a.z + a.w);
        s2 += (a.x * a.x + a.y * a.y) + (a.z * a.z + a.w * a.w);
        const long long pix = pix0 + row;
        if (out16) {
          uint2 o;
          o.x = pack_op2(a.x, a.y, fmt);
          o.y = pack_op2(a.z, a.w, fmt);
          *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + pix * NT + cg) = o;
        } else {
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + pix * NT + cg) = a;
        }
      }
      if (p.stats) {
        // lanes sharing `unit` hold the same 4-channel group; partial = (tile, lane quarter, group)
#pragma unroll
        for (int off = Cfg::U; off < 32; off <<= 1) {
          s1 += __shfl_xor_sync(0xffffffffu, s1, off);
          s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        }
        if (lane < Cfg::U)
          *reinterpret_cast<float2*>(p.stats + ((r * 4 + q) * (NT / 4) + (cg >> 2)) * 2) = make_float2(s1, s2);
      }
      __syncwarp();
    }
    if ((p.dbg & 32) && warp == Cfg::EPI_W0 && lane == 0) {
      g_rows_dbg[blockIdx.x][3] = dbg_w3;
      g_rows_dbg[blockIdx.x][5] = clock64() - dbg_t0;
    }
    }
  } else if (warp >= Cfg::XF_W0 && warp < Cfg::XF_W0 + Cfg::XF_WARPS) {
    if constexpr (Cfg::WG) setmaxnreg_dec<64>();
    // ============================ GroupNorm + SiLU transform (FUSED) ============================
    // thread t owns the logical 16-byte chunk j = t & 7 (channels 8j .. 8j+7) of pixels 1 + (t >> 3) + 16 i of every
    // halo row; the chunk's physical position follows SWIZZLE_128B: chunk ^ (pixel row & 7) (slots are 1 KB aligned).
    const int t0 = (int)threadIdx.x - 32 * Cfg::XF_W0;
    const int xset = t0 / (32 * Cfg::XF_SET_WARPS);           // this thread's set: input rows hl = xset (mod XF_SETS)
    const int t = t0 - xset * (32 * Cfg::XF_SET_WARPS);
    const int j = t & 7;
    const int prow = t >> 3;                // 0 .. XF_ROWS-1
    constexpr int XF_ROWS = FUSED ? 4 * Cfg::XF_SET_WARPS : 16;   // pixels covered per pass by one set's threads
    constexpr int XF_IT = 128 / XF_ROWS;
    constexpr int XF_SUB = XF_IT > 8 ? 8 : XF_IT;                 // 16-byte chunks in flight per thread
    uint32_t hl = 0;
    long long dbg_w4 = 0;
    long long r = r_begin;
    while (r < r_end) {
      const int b = (int)(r / p.H);
      const int y0 = (int)(r - (long long)b * p.H);
      const int R = (int)((r_end - r) < (long long)(p.H - y0) ? (r_end - r) : (long long)(p.H - y0));
      float ca[2][8], cb[2][8];
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        if (s < n_halo && p.coef[0] != nullptr) {
          const float4* cf = reinterpret_cast<const float4*>(p.coef[s] + (long long)b * 128 + j * 8);
          const float4 a0 = __ldg(cf), a1 = __ldg(cf + 1), b0 = __ldg(cf + 16), b1 = __ldg(cf + 17);
          ca[s][0] = a0.x; ca[s][1] = a0.y; ca[s][2] = a0.z; ca[s][3] = a0.w;
          ca[s][4] = a1.x; ca[s][5] = a1.y; ca[s][6] = a1.z; ca[s][7] = a1.w;
          cb[s][0] = b0.x; cb[s][1] = b0.y; cb[s][2] = b0.z; cb[s][3] = b0.w;
          cb[s][4] = b1.x; cb[s][5] = b1.y; cb[s][6] = b1.z; cb[s][7] = b1.w;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            ca[s][e] *= 0.5f;
            cb[s][e] *= 0.5f;
          }
        }
      }
      for (int k = 0; k < R + 2; ++k, ++hl) {
        if ((int)(hl % (uint32_t)Cfg::XF_SETS) != xset) continue;
        const uint32_t slot = hl % (uint32_t)p.n_slots, ph = (hl / (uint32_t)p.n_slots) & 1u;
        timed_wait(&h_full[slot], ph, p.err, 0x2800 + slot, dbg_w4, (p.dbg & 32) != 0);
        const int y = y0 - 1 + k;
        if (y >= 0 && y < p.H && p.coef[0] != nullptr) {   // out-of-image rows are TMA zero fill and must stay zero
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            if (s < n_halo) {
              const uint32_t base = smem_u32(h_smem) + slot * slot_bytes + s * kHaloBytes;
#pragma unroll
              for (int i0 = 0; i0 < XF_IT; i0 += XF_SUB) {
              uint4 v[XF_SUB];
#pragma unroll
              for (int i = 0; i < XF_SUB; ++i) {
                const int px = 1 + prow + XF_ROWS * (i0 + i);
                v[i] = lds128(base + px * 128 + ((j ^ (px & 7)) << 4));
              }
#pragma unroll
              for (int i = 0; i < XF_SUB; ++i) {
                const int px = 1 + prow + XF_ROWS * (i0 + i);
                uint4 o;
                o.x = xf_pair(v[i].x, ca[s][0], cb[s][0], ca[s][1], cb[s][1], fmt);
                o.y = xf_pair(v[i].y, ca[s][2], cb[s][2], ca[s][3], cb[s][3], fmt);
                o.z = xf_pair(v[i].z, ca[s][4], cb[s][4], ca[s][5], cb[s][5], fmt);
                o.w = xf_pair(v[i].w, ca[s][6], cb[s][6], ca[s][7], cb[s][7], fmt);
                sts128(base + px * 128 + ((j ^ (px & 7)) << 4), o);
              }
              }
            }
          }
          fence_proxy_async_smem();
        }
        mbar_arrive_warp(&h_ready[slot]);
      }
      r += R;
    }
    if ((p.dbg & 32) && t == 0) g_rows_dbg[blockIdx.x][4] = dbg_w4;
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int N, bool FUSED, int RM = -1, bool INF = false>
static int launch_rows(const CUtensorMap& tm_w, const CUtensorMap* tm_h, const CUtensorMap* tm_c, RowsParams p,
                       cudaStream_t stream) {
  using Cfg = RowsCfg<N, FUSED>;
  const int n_seg = p.n_halo * 9 + p.n_ctr;
  const int fixed = 1024 + n_seg * Cfg::W_SEG_BYTES + Cfg::STAGE_BYTES + 512;
  const int slot_bytes = p.n_halo * kHaloBytes;
  // centre ring: 2 x n_ctr tiles if the halo ring keeps its preferred depth, else n_ctr + 1 (still one tile of
  // look-ahead), else n_ctr
  const int min_pref = FUSED ? 5 : 4, min_ok = FUSED ? 4 : 3;
  int slots = 0;
  p.n_cslots = 0;
  const int cand[3] = {2 * p.n_ctr, p.n_ctr + 1, p.n_ctr};
  for (int i = 0; i < 3; ++i) {
    const int nc = cand[i];
    const int sl = (232448 - fixed - nc * kCtrBytes) / slot_bytes;
    if (sl >= (i == 0 ? min_pref : min_ok) || i == 2) {
      p.n_cslots = nc;
      slots = sl;
      break;
    }
  }
  if (slots > 8) slots = 8;
  MCEDM_REQUIRE(slots >= (FUSED ? 4 : 3),
                "conv_rows: %d halo sources + %d centre sources with N=%d do not fit in shared memory", p.n_halo,
                p.n_ctr, N);
  p.n_slots = slots;
  const int smem = fixed + slots * slot_bytes + p.n_cslots * kCtrBytes;
  static bool attr_set = false;
  if (!attr_set) {
    MCEDM_CUDA(cudaFuncSetAttribute(conv_rows_kernel<N, FUSED, RM, INF>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    attr_set = true;
  }
  const long long units = p.total_rows / p.row_align;
  long long grid = units < num_sms() ? units : num_sms();
  MCEDM_CUDA(launch_pdl(conv_rows_kernel<N, FUSED, RM, INF>, dim3((unsigned)grid), dim3(Cfg::THREADS), (size_t)smem, stream, tm_w,
                        tm_h[0], tm_h[1], tm_c[0], tm_c[1], p));
  return 0;
}

static int rows_common(RowsParams& p, CUtensorMap& tm_w, CUtensorMap* tm_h, CUtensorMap* tm_c,
                       const void* const* halo_src, int n_halo, const void* const* ctr_src, int n_ctr,
                       const void* w_packed, int B, int H, int N) {
  MCEDM_REQUIRE(n_halo >= 1 && n_halo <= 2 && n_ctr >= 0 && n_ctr <= 2, "conv_rows: n_halo=%d n_ctr=%d", n_halo, n_ctr);
  MCEDM_REQUIRE(B >= 1 && H >= 1, "conv_rows: bad B/H");
  MCEDM_REQUIRE(p.res_mode >= 0 && p.res_mode <= 2 && (p.res_mode == 0 || p.res != nullptr), "conv_rows: bad residual mode");
  MCEDM_REQUIRE(p.res_mode != 2 || H % 2 == 0, "conv_rows: upsampled residual needs even H");
  p.n_halo = n_halo;
  p.n_ctr = n_ctr;
  p.H = H;
  p.total_rows = (long long)B * H;
  if (p.row_align < 1) p.row_align = 1;
  MCEDM_REQUIRE(H % p.row_align == 0, "conv_rows: H=%d must be a multiple of %d for this kernel", H, p.row_align);
  p.err = watchdog_ptr();
  MCEDM_REQUIRE(p.err != nullptr, "conv_rows: cannot allocate the watchdog word");
  int rc = make_tmap_rows64_bf16(&tm_w, w_packed, (long long)(n_halo * 9 + n_ctr) * p.w_rows, N);
  if (rc) return rc;
  for (int i = 0; i < 2; ++i) {
    rc = make_tmap_nhwc_bf16(&tm_h[i], halo_src[i < n_halo ? i : 0], B, H, 128, 64, kHaloRows, 1);
    if (rc) return rc;
    rc = make_tmap_nhwc_bf16(&tm_c[i], n_ctr ? ctr_src[i < n_ctr ? i : 0] : halo_src[0], B, H, 128, 64, 128, 1);
    if (rc) return rc;
  }
  return 0;
}

}  // namespace mcedm

extern "C" int mcedm_conv_rows(const void* const* halo_src, int n_halo, const void* const* ctr_src, int n_ctr,
                               const void* w_packed, const float* bias, int B, int H, int N, void* out, int out_bf16,
                               const float* res, int res_mode, float* stats_partial, int op_fmt, void* stream) {
  using namespace mcedm;
  RowsParams p;
  memset(&p, 0, sizeof(p));
  p.bias = bias;
  p.out = out;
  p.out_bf16 = out_bf16;
  p.fmt = op_fmt ? 1 : 0;
  p.res = res;
  p.res_mode = res_mode;
  p.stats = stats_partial;
  p.n_off = 0;
  p.n_total = N;
  p.w_rows = N;
  CUtensorMap tm_w, tm_h[2], tm_c[2];
  int rc = rows_common(p, tm_w, tm_h, tm_c, halo_src, n_halo, ctr_src, n_ctr, w_packed, B, H, N);
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  switch (N) {
    case 16: return launch_rows<16, false>(tm_w, tm_h, tm_c, p, st);
    case 64: return launch_rows<64, false>(tm_w, tm_h, tm_c, p, st);
    default: return fail(-1, "conv_rows: N=%d unsupported (16, 64)", N);
  }
}

extern "C" int mcedm_conv_rows_fused(const void* const* halo_src, const float* const* halo_coef, int n_halo,
                                     const void* const* ctr_src, int n_ctr, const void* w_packed, const float* bias,
                                     int B, int H, int N, int n_off, int n_total, void* out, int out_16,
                                     const void* res16, int res_mode, int res_pitch, int res_blk,
                                     float* stats_partial, int op_fmt, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(n_total >= N && n_off >= 0 && n_off + N <= n_total && n_off % 4 == 0 && n_total % 4 == 0,
                "conv_rows_fused: bad output window (N=%d n_off=%d n_total=%d)", N, n_off, n_total);
  RowsParams p;
  memset(&p, 0, sizeof(p));
  p.bias = bias;
  p.out = out;
  p.out_bf16 = out_16;
  p.fmt = op_fmt ? 1 : 0;
  p.res = reinterpret_cast<const float*>(res16);
  p.res_mode = res_mode;
  p.stats = stats_partial;
  p.n_off = n_off;
  p.n_total = n_total;
  p.w_rows = n_total;
  p.res_pitch = res_pitch;
  p.res_blk = res_blk;
  p.row_align = N == 64 ? 4 : 1;     // GroupNorm records per 4-row block (see the epilogue)
  if (const char* e = getenv("MCEDM_DBG")) p.dbg = atoi(e);
  for (int i = 0; i < n_halo && i < 2; ++i) {
    p.coef[i] = halo_coef ? halo_coef[i] : nullptr;      // all NULL: the sources are already-normalised operands
    MCEDM_REQUIRE((p.coef[i] != nullptr) == (p.coef[0] != nullptr), "conv_rows_fused: coefficients for all sources or none");
  }
  CUtensorMap tm_w, tm_h[2], tm_c[2];
  int rc = rows_common(p, tm_w, tm_h, tm_c, halo_src, n_halo, ctr_src, n_ctr, w_packed, B, H, N);
  if (rc) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  MCEDM_REQUIRE(op_fmt == 1 || op_fmt == MCEDM_FMT_F16_INF,
                "conv_rows_fused: the fused inference kernels are fp16-only (op_fmt = 1)");
  MCEDM_REQUIRE(N != 64 || out_16 == 1, "conv_rows_fused: N = 64 writes 16-bit output");
  MCEDM_REQUIRE(N == 32 || n_halo == 1, "conv_rows_fused: N = 16 / 64 take one halo source (K-split 128-channel convs)");
  if (op_fmt == MCEDM_FMT_F16_INF) {
    // the data gradient of a 3x3 conv (no transform, no residual) is the one gradient this kernel writes
    MCEDM_REQUIRE(N == 64 && res_mode == 0 && p.coef[0] == nullptr,
                  "conv_rows_fused: op_fmt MCEDM_FMT_F16_INF is the N = 64 data-gradient launch (no coefficients, no residual)");
    return launch_rows<64, true, 0, true>(tm_w, tm_h, tm_c, p, st);
  }
  switch (N) {
    case 16: return launch_rows<16, true>(tm_w, tm_h, tm_c, p, st);
    case 32: return launch_rows<32, true>(tm_w, tm_h, tm_c, p, st);
    case 64:
      if (res_mode == 0) return launch_rows<64, true, 0>(tm_w, tm_h, tm_c, p, st);
      if (res_mode == 1) return launch_rows<64, true, 1>(tm_w, tm_h, tm_c, p, st);
      return launch_rows<64, true, 2>(tm_w, tm_h, tm_c, p, st);
    default: return fail(-1, "conv_rows_fused: N=%d unsupported (16, 32, 64)", N);
  }
}

extern "C" int mcedm_debug_rows(long long* host_out) {
  using namespace mcedm;
  MCEDM_CUDA(cudaDeviceSynchronize());
  MCEDM_CUDA(cudaMemcpyFromSymbol(host_out, g_rows_dbg, sizeof(long long) * 160 * 8));
  return 0;
}

extern "C" int mcedm_conv_head_fused(const void* src16, const float* coef, const void* w_packed, const float* bias, int B,
                                     int H, int c_out, float* F_nchw, int op_fmt, void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(c_out >= 1 && c_out <= 16 && coef != nullptr && bias != nullptr, "conv_head_fused: bad arguments");
  RowsParams p;
  memset(&p, 0, sizeof(p));
  p.bias = bias;
  p.out = F_nchw;
  p.out_bf16 = 0;
  p.fmt = op_fmt ? 1 : 0;
  p.n_total = 16;
  p.w_rows = 16;
  p.nchw_c = c_out;
  p.coef[0] = coef;
  if (const char* e = getenv("MCEDM_DBG")) p.dbg = atoi(e);
  CUtensorMap tm_w, tm_h[2], tm_c[2];
  const void* halo[1] = {src16};
  int rc = rows_common(p, tm_w, tm_h, tm_c, halo, 1, nullptr, 0, w_packed, B, H, 16);
  if (rc) return rc;
  return launch_rows<16, true>(tm_w, tm_h, tm_c, p, reinterpret_cast<cudaStream_t>(stream));
}
