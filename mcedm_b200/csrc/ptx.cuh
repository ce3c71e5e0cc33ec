// Inline-PTX wrappers for the sm_100a features the kernels use: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and proxy fences.
// Torch-free; every kernel TU in csrc/ includes this.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace mcedm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// Explicit shared-space 128-bit accesses.  Pointers derived from the 1 KB-aligned dynamic shared-memory base go
// through a uintptr_t round trip, after which nvcc no longer knows their address space and emits GENERIC LD/ST
// (L1TEX path, long-scoreboard latency) instead of LDS/STS — measured as the top stall of the conv epilogues.
__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr)
               : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t saddr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
// Programmatic dependent launch (launch_pdl in runtime.cuh).  pdl_wait: returns once the preceding kernel of the stream
// has completed and its writes are visible (no-op for a plain launch); everything a kernel reads that an earlier kernel
// wrote must come after it.  pdl_trigger: lets the NEXT kernel's CTAs become resident as soon as every CTA of this grid
// has executed it (or exited): their prologue (barrier init, TMEM allocation, weight loads) then overlaps this kernel's
// tail; placed after pdl_wait, so whatever precedes this kernel is complete by the time a dependent's prologue runs.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// register re-allocation between warpgroups (all four warps of an aligned group execute it)
template <int R>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R)); }
template <int R>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R)); }
// streaming 128-bit global load (read once: do not allocate in L1)
__device__ __forceinline__ uint4 ldg128_stream(const void* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
// per-thread asynchronous 16-byte copies global -> shared (LDGSTS, L1 bypassed), grouped and awaited by the issuing thread
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// 256-bit global accesses (sm_100: LDG/STG.256), 32-byte aligned
__device__ __forceinline__ void ldg256(const void* p, uint32_t* v) {
  asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void stg256(void* p, const uint32_t* v) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
               "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ float4 lds128f(uint32_t saddr) {
  const uint4 v = lds128(saddr);
  return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
}

// ------------------------------------------ mbarrier ------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_inval(uint64_t* bar) {
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// One arrival per WARP (count the barrier in warps): 32 lanes arriving individually are 32 serialised shared-memory
// atomics on one address; with 128-256 arriving threads per tile that storm alone cost ~1 us per tile.
// All lanes must have finished (and fenced) their work: __syncwarp orders it before lane 0's arrive.
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must not hang the GPU (a hung box is a strike). On timeout (~1 s) the
// waiter records a tag in *err and returns; once *err is set every later wait returns at once, so the
// kernel drains quickly with garbage results and the host sees the flag (mcedm_check_error()).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, unsigned int* err, uint32_t tag) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 63u) == 0) {
      if (*reinterpret_cast<volatile unsigned int*>(err) != 0u) return;
      if (clock64() - t0 > 2000000000LL) {
        atomicCAS(err, 0u, 0xdead0000u | (tag & 0xffffu));
        __threadfence();
        return;
      }
    }
  }
}

// -------------------------------------------- TMA ---------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// generic-proxy smem writes -> visible to the async proxy (UMMA / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------- tcgen05 ------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers bf16/fp16 inputs with fp32 accumulate.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once every previously issued tcgen05.mma of this thread has completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (base_lane + t), columns c..c+31
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// ----------------------------------- UMMA descriptors -----------------------------------------
// Shared-memory matrix descriptor (tcgen05), SWIZZLE_128B. Bit layout (cute::UMMA::SmemDescriptor):
//   [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [49,52) base_offset |
//   [61,64) layout (2 = SWIZZLE_128B)
// K-major operand with 64 bf16 (=128 B) per row: rows are 128 B apart, 8-row groups SBO = 1024 B apart.
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t saddr, uint32_t base_offset = 0) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;             // LBO (ignored for swizzled K-major; canonical value 1)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;     // SBO
  d |= static_cast<uint64_t>(1) << 46;             // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(base_offset & 7u) << 49;
  d |= static_cast<uint64_t>(2) << 61;             // SWIZZLE_128B
  return d;
}
// MN-major operand, SWIZZLE_128B, one 64-element (128 B) MN block: each K index is one 128-B row,
// 8-K groups are SBO = 1024 B apart; LBO (stride between 64-element MN blocks) given by caller.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16, bf16 x bf16 -> fp32 (cute::UMMA::InstrDescriptor):
//   [4,6) D fmt (1=f32) | [7,10) A fmt (1=bf16) | [10,13) B fmt | 15 A major | 16 B major (0=K,1=MN) |
//   [17,23) N>>3 | [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major = 0, int b_mn_major = 0) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// Operand format of the 16-bit tensor-core operands: 0 = bf16 (training: gradients need the range), 1 = fp16
// (inference: activations are normalised and weights are O(1), and fp16's 11 significand bits cut the
// operand-rounding error of the network output ~8x at the same tensor throughput).  Same instruction kind.
__host__ __device__ constexpr uint32_t umma_idesc_16(int M, int N, int a_mn_major, int b_mn_major, int fmt) {
  const uint32_t f = fmt ? 0u : 1u;       // descriptor format code: 0 = f16, 1 = bf16
  return (1u << 4) | (f << 7) | (f << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}
// (kind::f16 requires A and B to share one 16-bit format: a bf16 x fp16 mix raises an illegal-instruction fault
// on sm_100a — tried, to keep the weights at 11 significand bits.)

// -------------------------------------- misc numerics -----------------------------------------
__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + __expf(-x)); }

// silu(2h) = h * (1 + tanh(h)) with ONE special-function op (MUFU.TANH, max relative error 2^-11 on tanh) instead of
// ex2 + rcp: the in-shared-memory GroupNorm+SiLU transform of the fused convs is instruction-bound.
__device__ __forceinline__ float silu_from_half_arg(float h) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  // satfinite: a value beyond the fp16 range (65504) clamps instead of becoming inf (16-bit activation storage)
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_op2(float lo, float hi, int fmt) {
  return fmt ? pack_f16x2(lo, hi) : pack_bf16x2(lo, hi);
}
// Gradient stores of dynamic loss scaling (op_fmt MCEDM_FMT_F16_INF): no `satfinite`, so a value beyond fp16's range
// becomes inf, reaches the fp32 flat gradient through the weight-gradient contractions and makes the step skip.
// INF = false is the saturating conversion above, instruction for instruction.
__device__ __forceinline__ uint32_t pack_f16x2_inf(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
template <bool INF>
__device__ __forceinline__ uint32_t pack_f16x2_g(float lo, float hi) {
  return INF ? pack_f16x2_inf(lo, hi) : pack_f16x2(lo, hi);
}
template <bool INF>
__device__ __forceinline__ uint32_t pack_op2_g(float lo, float hi, int fmt) {
  return INF ? pack_f16x2_inf(lo, hi) : pack_op2(lo, hi, fmt);
}
__device__ __forceinline__ float2 unpack_f16x2(uint32_t v) {
  float lo, hi;
  asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}\n"
      : "=f"(lo), "=f"(hi) : "r"(v));
  return make_float2(lo, hi);
}
// Saturation audit of the fp16 activation storage (MCEDM_DBG & 4): counts values whose magnitude exceeds the largest
// finite fp16 (65504; the packing conversions clamp them, `satfinite`) into word 8 of the watchdog buffer, so that a
// residual stream drifting out of fp16's range is REPORTED (mcedm_saturation_count) instead of silently clipped.
template <int NV>
__device__ __forceinline__ void sat_audit(unsigned int* err, const float (&a)[NV]) {
  unsigned int c = 0;
#pragma unroll
  for (int i = 0; i < NV; ++i) c += (fabsf(a[i]) > 65504.0f || a[i] != a[i]) ? 1u : 0u;
  if (c) atomicAdd(err + 8, c);
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

}  // namespace mcedm
