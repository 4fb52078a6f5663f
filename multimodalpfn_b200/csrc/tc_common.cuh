// tc_common.cuh — inline-PTX wrappers shared by the tcgen05 kernels (kernels_tc.cu, kernels_mlp.cu):
// mbarrier, TMA (cp.async.bulk.tensor), TMEM allocation / load / store, tcgen05.mma + commit, UMMA
// shared-memory and instruction descriptors, packed fp32x2 arithmetic.  Everything lives in an
// anonymous namespace: each translation unit gets its own copy.
#pragma once
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"

namespace mmpfn {
namespace {

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// One arrival per WARP: the lanes synchronise (which also orders their prior shared-memory / TMEM
// accesses before lane 0's release-arrive) and lane 0 arrives.  128 threads arriving one by one are
// 128 serialised atomics on one shared-memory word — several hundred cycles per hand-off.
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
__device__ __noinline__ void mbar_timeout() {
  printf("mmpfn: mbarrier timeout (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y, threadIdx.x);
  __trap();
}
// try_wait suspends the thread in hardware for a bounded time per probe (the 20 us hint), so the poll
// loop is three instructions; the clock is consulted once every 2^12 failed probes and a wait that
// lasts ~2 s traps (a protocol bug, not a slow tile) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  long long t0 = 0;
  while (true) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .u32 n;\n\t"
        "mov.u32 n, 0;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "@p bra DONE_%=;\n\t"
        "add.u32 n, n, 1;\n\t"
        "setp.lt.u32 p, n, 4096;\n\t"
        "@p bra WAIT_%=;\n\t"
        "mov.u32 %0, 0;\n\t"
        "bra EXIT_%=;\n\t"
        "DONE_%=:\n\t"
        "mov.u32 %0, 1;\n\t"
        "EXIT_%=:\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(20000u)
        : "memory");
    if (done) return;
    const long long now = clock64();
    if (t0 == 0) t0 = now;
    else if (now - t0 > 4000000000LL) mbar_timeout();
  }
}
// One lane of a converged warp.  Guarding a single-thread role with elect.sync (instead of lane == 0) lets
// ptxas know that exactly one thread is active inside: the uniform-register operands of UTCHMMA / UTMALDG
// are then filled by plain R2UR moves instead of a per-operand election loop (~70 cycles per MMA issue).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// Non-blocking probe: has the phase with this parity completed?  The answer can be consumed much later
// (the probe's ~200-cycle round trip then hides under other work) and a positive one replaces the wait.
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
// Wait for two barriers at once.  Even a wait that is already satisfied costs the calling thread
// ~200-250 cycles (SYNCS round trip): a single-thread issue loop that checks two barriers per step
// pays it once instead of twice when both probes are in flight together.
__device__ __forceinline__ void mbar_wait2(uint64_t* bar_a, uint32_t parity_a, uint64_t* bar_b, uint32_t parity_b) {
  const uint32_t a = smem_u32(bar_a), b = smem_u32(bar_b);
  uint32_t n = 0;
  long long t0 = 0;
  while (true) {
    uint32_t da, db;
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%2], %3, %6;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 q, [%4], %5, %6;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "selp.u32 %1, 1, 0, q;\n\t}"
        : "=r"(da), "=r"(db)
        : "r"(a), "r"(parity_a), "r"(b), "r"(parity_b), "r"(20000u)
        : "memory");
    if (da & db) return;
    if ((++n & 4095u) == 0) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000LL) mbar_timeout();
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
// bytes (a multiple of 16, 16-byte aligned address) of global memory into L2, asynchronously
__device__ __forceinline__ void l2_prefetch(const void* gptr, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32; one thread issues for the CTA
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T: the A operand (M = 128 rows = TMEM lanes, K bf16 elements packed two per
// 32-bit column) is read from tensor memory — 8 columns per K = 16 step
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every tcgen05 op issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets TMEM lane (base lane + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// 2^x on the FMA/ALU pipes (no MUFU): x = n + f with n = round(x), f in [-0.5, 0.5]; 2^f by a
// degree-3 minimax polynomial (max relative error 7.6e-5, far below the bf16 rounding of P), the
// integer part spliced into the exponent field.  x is clamped to [-126, 126]: below, the result is
// ~1e-38 ~ 0; above, it saturates at ~2^126 instead of wrapping the exponent into the sign bit (the
// item attention detects scores far above its reference by the row sum: that must come out huge,
// never negative).
__device__ __forceinline__ float poly_exp2(float x) {
  x = fminf(fmaxf(x, -126.0f), 126.0f);
  const float r = x + 12582912.0f;            // 1.5 * 2^23: round(x) lands in the low mantissa bits
  const float f = x - (r - 12582912.0f);
  float p = fmaf(0.05520550534129143f, f, 0.24261397123336792f);
  p = fmaf(p, f, 0.6932547688484192f);
  p = fmaf(p, f, 0.9999276995658875f);
  return __uint_as_float(__float_as_uint(p) + (__float_as_uint(r) << 23));
}
// which of the 32 elements of a register chunk take the polynomial: PN of 32, evenly spread
__host__ __device__ constexpr bool poly_sel(int i, int PN) { return ((i + 1) * PN) / 32 != (i * PN) / 32; }

// packed fp32 pairs (FFMA2 / FADD2): one issue slot for two lanes of the softmax arithmetic
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

__device__ __forceinline__ void st_shared_v4(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// ---- epilogue staging: shared memory -> global by TMA (bulk async-group), named barrier of the 128 epilogue threads
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void st_shared_u16(uint32_t saddr, uint16_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(saddr), "h"(v) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

// UMMA shared-memory operand descriptor, K-major, swizzled (cute::UMMA::SmemDescriptor layout):
// start address >> 4 in [0,14), LBO (=1, unused for swizzled K-major) in [16,30), SBO >> 4 in [32,46),
// version 1 in [46,48), layout type in [61,64) (2 = 128B swizzle, 4 = 64B swizzle).
constexpr uint32_t kSw128 = 2, kSw64 = 4;
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): fp32 accumulate, bf16 A/B, both K-major
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// the same for A/B of format FMT: format bits [7,10) / [10,13) are 1 for bf16 (FMT_BF16), 0 for fp16 (FMT_F16)
template <int FMT>
__host__ __device__ constexpr uint32_t make_idesc_fmt(int M, int N) {
  return FMT == FMT_F16 ? make_idesc(M, N) & ~((7u << 7) | (7u << 10)) : make_idesc(M, N);
}

// ---------------------------------------------------------------------------------------------
// LayerNorm statistics of the residual + LayerNorm epilogues (kernels_mlp.cu, kernels_rowgemm.cu,
// kernels_tc.cu): one thread owns one kE-wide row, which arrives as six 32-column chunks in order.
// The variance is taken about the mean, not as sq/kE - mean^2: that one-pass form cancels when a row's
// |mean| is large against its spread (the error grows with the square of mean/std; past ~1000 the
// variance comes out 0: a row of mean -4096, std 1.6 came out off by ~2e3).  Every value enters shifted
// by K = the mean of the row's first chunk, within ~std/sqrt(32) of the row mean, so that
// var = E[(a-K)^2] - E[a-K]^2 cancels only by (mean - K)^2 / var ~ 1/32, whatever the mean.  The sums are
// one pass over registers in packed fp32x2 arithmetic; the epilogues take them after a chunk's sum has
// gone back to TMEM and its residual slot to the producer, off the path of the residual ring.
// A row of exact zeros gives mean 0, variance 0 and normalises to exact zeros (the pad-row contract).
// ---------------------------------------------------------------------------------------------
struct LnRowStats {
  float k = 0.f;
  uint64_t s2 = 0ull, q2a = 0ull, q2b = 0ull;     // sum of (a - K) and of (a - K)^2, two lanes each
  // chunk c (0-based) of the row: 32 fp32 values as bits
  __device__ __forceinline__ void add32(const uint32_t (&v)[32], int c) {
    uint64_t a2[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a2[i] = pack_f32x2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
    if (c == 0) {
      uint64_t t2[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
      for (int i = 0; i < 16; ++i) t2[i & 3] = add_f32x2(t2[i & 3], a2[i]);
      float t0, t1;
      unpack_f32x2(add_f32x2(add_f32x2(t2[0], t2[1]), add_f32x2(t2[2], t2[3])), t0, t1);
      k = (t0 + t1) * (1.0f / 32);
    }
    const uint64_t nk2 = pack_f32x2(-k, -k);
    uint64_t sa = 0ull, sb = 0ull;
#pragma unroll
    for (int i = 0; i < 16; i += 2) {
      const uint64_t d0 = add_f32x2(a2[i], nk2), d1 = add_f32x2(a2[i + 1], nk2);
      sa = add_f32x2(sa, d0);
      sb = add_f32x2(sb, d1);
      q2a = fma_f32x2(d0, d0, q2a);
      q2b = fma_f32x2(d1, d1, q2b);
    }
    s2 = add_f32x2(s2, add_f32x2(sa, sb));
  }
  // after the last chunk
  __device__ __forceinline__ void finish(float& mean, float& rstd) const {
    float s0, s1, q0, q1;
    unpack_f32x2(s2, s0, s1);
    unpack_f32x2(add_f32x2(q2a, q2b), q0, q1);
    const float dm = (s0 + s1) * (1.0f / kE);
    mean = k + dm;
    rstd = rsqrtf(fmaxf((q0 + q1) * (1.0f / kE) - dm * dm, 0.f) + kLnEps);
  }
};


// ---------------------------------------------------------------------------------------------
// host: tensor maps
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

// dims innermost first; strides in bytes for dims 1..rank-1; elements are bf16 unless dtype says otherwise
int encode_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
               const cuuint32_t* box, CUtensorMapSwizzle sw,
               CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  EncodeTiledFn fn = get_encode();
  if (!fn) { set_error("cuTensorMapEncodeTiled not available"); return MMPFN_ECUDA; }
  cuuint32_t ones[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(m, dtype, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box,
                  ones, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) rank %d dims %llu,%llu box %u,%u", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
    return MMPFN_ECUDA;
  }
  return MMPFN_OK;
}

}  // namespace
}  // namespace mmpfn
