// First convolution of the U-Net on the tensor cores (inference): 3x3 conv of cat([cond, x]) (NCHW fp32, Cin <= 5
// channels) -> raw 16-bit NHWC [B,H,128,64] + GroupNorm partial sums
// (models/adm_blocks.py:319-340 cat_conditioning, :384-385; same math as small.cu conv_in_kernel).
//
// The CUDA-core version is bound by 4.8 G fp32 FMAs per 128 samples (360 us measured, ~134 us at the FMA roofline)
// for a layer whose memory traffic is 33 MB in + 268 MB out.  Here the layer is ONE K = 16 tensor-core step per
// input row:
//   * four "builder" warps (one thread per pixel) read the Cin input values of pixel p-1, p, p+1 of image row y and
//     write the operand row  A[p][k = kx*Cin + c] = in[c][y][p + kx - 1]  (fp16, zero outside the image, zero-padded to
//     16) into the first 32 bytes of a 128-byte SWIZZLE_128B row: the horizontal taps are folded into K;
//   * the vertical taps are stacked into N exactly as in conv_rows.cu (STACK): input row k feeds output rows k, k-1,
//     k-2 with the weights of ky = 0, 1, 2 as 192 B-rows [ky][co][k], so an input row costs one N = 64 (fresh
//     accumulator) + one N = 128 MMA; eight 64-column accumulators rotate through TMEM in descending tile order;
//   * epilogue as conv_rows.cu (bias, GroupNorm partial sums per (row, lane quarter), coalesced 16-bit stores).
// The inputs are rounded to fp16 once, like every other activation of the inference plan.
#include "ptx.cuh"
#include "runtime.cuh"
#include "../../include/mcedm_b200.h"

namespace mcedm {

constexpr int kInSlots = 8;                 // ring of operand rows (16 KB each: only bytes [0, 32) of a row are used)
constexpr int kInTile = 16 * 1024;
// The layer is one MMA per input row and its pacer was the BUILDER: a row's 12-15 scalar loads, the operand store and the
// hand-over ran back to back, so every input row exposed one full global-memory latency (1.1 us per row: 242 us per launch at
// 256 samples; doubling the epilogue warps changed nothing).  Two sets of 4 builder warps now take alternate input rows and
// each thread requests its NEXT row's values before it packs and stores the current one: four rows in flight per CTA.
template <int CIN>
struct InTcCfg {
  static constexpr int SETS = 1;                       // epilogue warp sets (alternate output rows): 2 measured slower (184 vs 169 us)
  static constexpr int EPI_WARPS = 8 * SETS;
  static constexpr int BSETS = 2;                      // builder warp sets (alternate input rows)
  static constexpr int THREADS = 64 + 32 * EPI_WARPS + BSETS * 4 * 32;
  static constexpr int STAGE_BYTES = EPI_WARPS * 4096;
};

struct InTcParams {
  const float* x;        // [B, Cx, H, 128]
  const float* cond;     // [B, Cc, H, 128] or nullptr
  int Cx, Cc, H;
  long long total_rows;  // B * H
  const float* bias;     // [64]
  void* out;             // 16-bit NHWC [B, H, 128, 64]
  float* stats;          // [B*H][4][16][2] or nullptr
  int fmt;
  unsigned int* err;
};

template <int CIN>
__global__ void __launch_bounds__(InTcCfg<CIN>::THREADS, 1)
conv_in_tc_kernel(const __grid_constant__ CUtensorMap tm_w, const InTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* w_smem = smem;                                   // 3 x [64 co][64 k] fp16 = 24 KB, ky-major
  uint8_t* a_smem = w_smem + 3 * 8192;                      // kInSlots x 16 KB
  uint8_t* stage_smem = a_smem + kInSlots * kInTile;        // 8 warps x 4 KB
  using Cfg = InTcCfg<CIN>;
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_smem + Cfg::STAGE_BYTES);
  uint64_t* w_full = bars;
  uint64_t* acc_full = bars + 1;           // 8
  uint64_t* acc_empty = acc_full + 8;      // 8
  uint64_t* a_ready = acc_empty + 8;       // kInSlots
  uint64_t* a_empty = a_ready + kInSlots;  // kInSlots
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_empty + kInSlots);

  pdl_wait();
  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long r_begin = p.total_rows * blockIdx.x / gridDim.x;
  const long long r_end = p.total_rows * (blockIdx.x + 1) / gridDim.x;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_w);
    mbar_init(w_full, 1);
    for (int i = 0; i < 8; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 8);         // one arrival per epilogue warp
    }
    for (int i = 0; i < kInSlots; ++i) {
      mbar_init(&a_ready[i], 4);           // one arrival per builder warp
      mbar_init(&a_empty[i], 1);
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

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(w_full, 3 * 8192);
      for (int ky = 0; ky < 3; ++ky) tma_load_2d(w_smem + ky * 8192, &tm_w, w_full, 0, ky * 64);
    }
  } else if (warp == 1) {
    // ====================================== MMA issuer ======================================
    const uint32_t idesc1 = umma_idesc_16(128, 64, 0, 0, p.fmt), idesc2 = umma_idesc_16(128, 128, 0, 0, p.fmt),
                   idesc3 = umma_idesc_16(128, 192, 0, 0, p.fmt);
    mbar_wait(w_full, 0, p.err, 0x4300);
    tc_fence_after();
    const uint32_t w_lo = (smem_u32(w_smem) >> 4) | (1u << 16);
    const uint32_t a_lo = (smem_u32(a_smem) >> 4) | (1u << 16);
    constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
    auto desc = [&](uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; };
    uint32_t hs = 0, hph = 0, t0 = 0;
    long long r = r_begin;
    while (r < r_end) {
      const int b = (int)(r / p.H);
      const int y0 = (int)(r - (long long)b * p.H);
      const int R = (int)((r_end - r) < (long long)(p.H - y0) ? (r_end - r) : (long long)(p.H - y0));
      for (int k = 0; k < R + 2; ++k) {
        if (k < R) {
          const uint32_t tn = t0 + (uint32_t)k;
          mbar_wait(&acc_empty[tn & 7u], ((tn >> 3) & 1u) ^ 1u, p.err, 0x4400 + (tn & 7u));
        }
        mbar_wait(&a_ready[hs], hph, p.err, 0x4500 + hs);
        tc_fence_after();
        const int kyA = k - (R - 1) > 0 ? k - (R - 1) : 0;   // output row k - ky must lie in [0, R)
        const int kyB = k < 2 ? k : 2;
        const uint32_t blk0 = (8u - ((t0 + (uint32_t)(k - kyA)) & 7u)) & 7u;
        const int nky = kyB - kyA + 1;
        const int split = (int)(8u - blk0) < nky ? (int)(8u - blk0) : nky;
        const uint32_t d0 = tmem_base + blk0 * 64u;
        const uint32_t d1 = tmem_base + ((blk0 + (uint32_t)split) & 7u) * 64u;
        const uint64_t ad = desc(a_lo + hs * (kInTile >> 4));
        const uint32_t wrow = w_lo + (uint32_t)kyA * (8192 >> 4);
        const bool fresh = kyA == 0;
        const int n0 = split, n1 = nky - split;
        if (elect_one()) {
          // the whole K (3 taps x Cin <= 16) is one MMA step; a fresh accumulator takes ky = 0 alone, non-accumulating
          if (fresh && n0 > 1) {
            umma_f16(d0, ad, desc(wrow), idesc1, 0u);
            umma_f16(d0 + 64u, ad, desc(wrow + (8192 >> 4)), n0 == 2 ? idesc1 : idesc2, 1u);
          } else {
            umma_f16(d0, ad, desc(wrow), n0 == 1 ? idesc1 : n0 == 2 ? idesc2 : idesc3, fresh ? 0u : 1u);
          }
          if (n1 > 0) umma_f16(d1, ad, desc(wrow + (uint32_t)n0 * (8192 >> 4)), n1 == 1 ? idesc1 : idesc2, 1u);
          umma_commit(&a_empty[hs]);
          if (k >= 2) umma_commit(&acc_full[(t0 + (uint32_t)(k - 2)) & 7u]);
        }
        __syncwarp();
        if (++hs == kInSlots) {
          hs = 0;
          hph ^= 1u;
        }
      }
      t0 += (uint32_t)R;
      r += R;
    }
  } else if (warp < 2 + Cfg::EPI_WARPS) {
    // ======================================= epilogue =======================================
    const int q = warp & 3, ew = warp - 2, ch = (ew & 7) >> 2, set = ew >> 3;
    const uint32_t my_stage = smem_u32(stage_smem) + ew * 4096;
    const int unit = lane & 7, row_in_it = lane >> 3;
    const int c0 = ch * 32 + unit * 4;
    float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.bias) bz = *reinterpret_cast<const float4*>(p.bias + c0);
    uint16_t* o16 = reinterpret_cast<uint16_t*>(p.out);
    uint32_t tcount = (uint32_t)set;
    for (long long r = r_begin + set; r < r_end; r += Cfg::SETS, tcount += Cfg::SETS) {
      const uint32_t buf = tcount & 7u, aph = (tcount >> 3) & 1u;
      const long long pix0 = r * 128 + q * 32;
      mbar_wait(&acc_full[buf], aph, p.err, 0x4700 + buf);
      tc_fence_after();
      uint32_t v[32];
      tmem_ld_x32(tmem_base + ((uint32_t)(q * 32) << 16) + ((8u - buf) & 7u) * 64u + ch * 32, v);
      tmem_wait_ld();
      tc_fence_before();
      mbar_arrive_warp(&acc_empty[buf]);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int pj = j ^ (lane & 7);
        sts128(my_stage + lane * 128 + pj * 16, make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
      }
      __syncwarp();
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int itr = 0; itr < 8; ++itr) {
        const int row = itr * 4 + row_in_it;
        const int pu = unit ^ (row & 7);
        float4 a = lds128f(my_stage + row * 128 + pu * 16);
        a.x += bz.x; a.y += bz.y; a.z += bz.z; a.w += bz.w;
        s1 += (a.x + a.y) + (a.z + a.w);
        s2 += (a.x * a.x + a.y * a.y) + (a.z * a.z + a.w * a.w);
        uint2 o;
        o.x = pack_op2(a.x, a.y, p.fmt);
        o.y = pack_op2(a.z, a.w, p.fmt);
        *reinterpret_cast<uint2*>(o16 + (pix0 + row) * 64 + c0) = o;
      }
      if (p.stats) {
#pragma unroll
        for (int off = 8; off < 32; off <<= 1) {
          s1 += __shfl_xor_sync(0xffffffffu, s1, off);
          s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        }
        if (lane < 8) *reinterpret_cast<float2*>(p.stats + ((r * 4 + q) * 16 + ch * 8 + lane) * 2) = make_float2(s1, s2);
      }
      __syncwarp();
    }
  } else {
    // ======================================= builders =======================================
    const int bt = (int)threadIdx.x - 32 * (2 + Cfg::EPI_WARPS);
    const int px = bt & 127;                                 // this thread's pixel 0..127
    const int bset = bt >> 7;                                // builder set: input rows hl = bset (mod BSETS)
    const uint32_t a_base = smem_u32(a_smem);
    const long long HW = (long long)p.H * 128;
    // cursor over the CTA's input rows in the MMA warp's order: segment (image b, rows y0 .. y0+R-1) -> R + 2 input rows
    long long r = r_begin;
    int b = 0, y0 = 0, R = 0, k = 0;
    uint32_t hl = 0;
    bool done = r >= r_end;
    auto seg = [&]() {
      b = (int)(r / p.H);
      y0 = (int)(r - (long long)b * p.H);
      R = (int)((r_end - r) < (long long)(p.H - y0) ? (r_end - r) : (long long)(p.H - y0));
      k = 0;
    };
    auto advance = [&]() {
      ++hl;
      if (++k == R + 2) {
        r += R;
        if (r >= r_end) done = true;
        else seg();
      }
    };
    auto load_row = [&](float (&v)[16]) {
      // operand row of pixel px: value index kx*Cin + c = in[c][y][px + kx - 1]
      const int y = y0 - 1 + k;
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = 0.f;
      if (y >= 0 && y < p.H) {
#pragma unroll
        for (int c = 0; c < CIN; ++c) {
          const float* src = (c < p.Cc) ? p.cond + ((long long)b * p.Cc + c) * HW + (long long)y * 128
                                        : p.x + ((long long)b * p.Cx + (c - p.Cc)) * HW + (long long)y * 128;
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            const int xx = px + kx - 1;
            v[kx * CIN + c] = (xx >= 0 && xx < 128) ? __ldg(src + xx) : 0.f;
          }
        }
      }
    };
    if (!done) seg();
    for (int i = 0; i < bset && !done; ++i) advance();
    float v[16], vn[16];
    if (!done) load_row(v);
    while (!done) {
      const uint32_t hs = hl % (uint32_t)kInSlots, hph = (hl / (uint32_t)kInSlots) & 1u;
      for (int i = 0; i < Cfg::BSETS && !done; ++i) advance();
      if (!done) load_row(vn);                               // the next row's loads fly while this one is stored
      uint4 lo4, hi4;
      lo4.x = pack_op2(v[0], v[1], p.fmt);   lo4.y = pack_op2(v[2], v[3], p.fmt);
      lo4.z = pack_op2(v[4], v[5], p.fmt);   lo4.w = pack_op2(v[6], v[7], p.fmt);
      hi4.x = pack_op2(v[8], v[9], p.fmt);   hi4.y = pack_op2(v[10], v[11], p.fmt);
      hi4.z = pack_op2(v[12], v[13], p.fmt); hi4.w = pack_op2(v[14], v[15], p.fmt);
      mbar_wait(&a_empty[hs], hph ^ 1u, p.err, 0x4800 + hs);
      const uint32_t rowa = a_base + hs * kInTile + px * 128;
      sts128(rowa + ((0 ^ (px & 7)) << 4), lo4);
      sts128(rowa + ((1 ^ (px & 7)) << 4), hi4);
      fence_proxy_async_smem();
      mbar_arrive_warp(&a_ready[hs]);
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = vn[i];
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

extern "C" int mcedm_conv_in_tc16(const float* x, int Cx, const float* cond, int Cc, const void* w16_packed,
                                  const float* bias, int B, int H, void* out16, float* stats_partial, int op_fmt,
                                  void* stream) {
  using namespace mcedm;
  MCEDM_REQUIRE(Cx >= 1 && Cc >= 0 && Cx + Cc <= 5, "conv_in_tc16: %d+%d input channels (3*Cin must fit in K = 16)", Cx, Cc);
  MCEDM_REQUIRE(Cc == 0 || cond != nullptr, "conv_in_tc16: cond channels without a cond tensor");
  MCEDM_REQUIRE(B >= 1 && H >= 1, "conv_in_tc16: bad B/H");
  InTcParams p;
  memset(&p, 0, sizeof(p));
  p.x = x;
  p.cond = cond;
  p.Cx = Cx;
  p.Cc = Cc;
  p.H = H;
  p.total_rows = (long long)B * H;
  p.bias = bias;
  p.out = out16;
  p.stats = stats_partial;
  p.fmt = op_fmt ? 1 : 0;
  p.err = watchdog_ptr();
  MCEDM_REQUIRE(p.err != nullptr, "conv_in_tc16: cannot allocate the watchdog word");
  CUtensorMap tm_w;
  int rc = make_tmap_rows64_bf16(&tm_w, w16_packed, 3 * 64, 64);
  if (rc) return rc;
  const int smem = 1024 + 3 * 8192 + kInSlots * kInTile + 8 * 4096 + 512;
  long long grid = p.total_rows < num_sms() ? p.total_rows : num_sms();
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
#define MCEDM_IN_TC_CASE(C)                                                                                          \
  case C:                                                                                                            \
    MCEDM_CUDA(cudaFuncSetAttribute(conv_in_tc_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));       \
    MCEDM_CUDA(launch_pdl(conv_in_tc_kernel<C>, dim3((unsigned)grid), dim3(InTcCfg<C>::THREADS), (size_t)smem, st, tm_w, p)); \
    break;
  switch (Cx + Cc) {
    MCEDM_IN_TC_CASE(1) MCEDM_IN_TC_CASE(2) MCEDM_IN_TC_CASE(3) MCEDM_IN_TC_CASE(4) MCEDM_IN_TC_CASE(5)
  }
#undef MCEDM_IN_TC_CASE
  MCEDM_CUDA(cudaGetLastError());
  return 0;
}
