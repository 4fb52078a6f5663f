// kernels_attn.cu — attention across items (layer.py:341-379, multi_head_attention.py:547-736) as a
// flash-attention kernel written directly against sm_100a, d = 32:
//
//   S = Q K^T and O += P V on tcgen05 (accumulators in TMEM, operands staged by TMA), online softmax
//   in fp32 by four warps (thread = query row).  P goes back into tensor memory over the S columns it
//   came from (bf16 pairs; fp16 pairs in the fp16 instantiation) and the second MMA reads its A operand there: no
//   st.shared, no proxy fence.
//
// At d = 32 every exponential buys only 128 tensor FLOP, so the kernel lives on the MUFU pipe
// (16 ex2/clk/SM = 595 TFLOP/s at 1965 MHz if every exponential went there) and on the issue slots of
// the four schedulers, not on the tensor pipe.  Round-1 profile (profiles/r01_ncu_stalls_v6_*): the
// TMA and MMA role warps executed 117 and 164 instructions per key tile (bounded two-barrier polls,
// descriptor arithmetic, four commits) on schedulers 0 and 1, next to a softmax warp that needs ~230 of
// the 336 MUFU-bound cycles of a tile: scheduler 1 was ISSUE bound and, the four softmax warps of a CTA
// moving in lockstep, held the MUFU pipe of all four at 76 %.  This version
//   * hands every per-tile event to ONE barrier per S buffer: the MMA thread commits once per tile
//     (done[s]: "P V(j) and S(j+2) have completed") and the TMA thread refills V(j+2) and K(j+4) on one
//     barrier (kv_full[s]) behind it — 1 wait + 1 expect_tx + 2 loads, and 2 waits + 5 MMAs + 1 commit;
//   * takes PP of every 24 key PAIRS through a packed (FFMA2/FADD2) degree-3 polynomial 2^x on the FMA
//     pipe — 5 issue slots per exponential instead of 9 for the scalar form — with the exponent splice
//     clamped by one VIADDMNMX.RELU instead of two FMNMX.
//
// Tile: BK = 48 keys, 4 CTAs/SM.  TMEM: S0 [0,48)  S1 [48,96)  O [96,128).
// Test pass (every query head of a column reads that column's head-0 K/V): the six heads are stacked on
// the tile's row axis, so 6 x 300 query rows fill 15 tiles of 128 instead of 18.
// Every mbarrier wait is bounded (trap) so that a protocol bug cannot hang the GPU.
#include "tc_common.cuh"

namespace mmpfn {
namespace {

constexpr int A_BQ = 128;
constexpr int A_Q_BYTES = A_BQ * kD * 2;          // 8 KB  (64B rows, 64B swizzle)
constexpr int A_THREADS = 192;
#ifndef ATTN_PP
#define ATTN_PP 7
#endif
constexpr int kPolyPairsDefault = ATTN_PP;        // of 24 pairs per tile (measured optimum, see DESIGN.md)
#ifndef ATTN_KAHEAD
#define ATTN_KAHEAD 4
#endif
#ifndef ATTN_KBEHIND
#define ATTN_KBEHIND 5
#endif
#ifndef ATTN_PROBE_AT
#define ATTN_PROBE_AT 1000                        // pair step of the sweep at which the next tile's S is probed (>= NP: after it)
#endif
#ifndef ATTN_PIN
#define ATTN_PIN 1
#endif
#ifndef ATTN_ONE_ARRIVE
#define ATTN_ONE_ARRIVE 0                         // 1: the four softmax warps meet at a named barrier and ONE thread arrives on p_full
#endif
// a value the compiler must keep in a register instead of recomputing it from special registers at every use
__device__ __forceinline__ uint32_t pin_u32(uint32_t v) {
#if ATTN_PIN
  asm volatile("mov.u32 %0, %0;" : "+r"(v));
#endif
  return v;
}

template <int BK>
struct AttnCfg {
  static constexpr int kNKB = (BK + 63) / 64;                 // 64-key k-blocks of the V^T tile
  static constexpr int kKTx = BK * kD * 2;                    // bytes of one K tile (64 B per key)
  static constexpr int kKSlot = (kKTx + 511) / 512 * 512;     // slot stride: a multiple of the 64B-swizzle atom
  static constexpr int kVtBytes = kNKB * kD * 128;            // [32 d][64 keys = 128 B] per k-block, 128B swizzle
  static constexpr int kOffK = A_Q_BYTES;
  static constexpr int kOffVt = (kOffK + 2 * kKSlot + 1023) / 1024 * 1024;
  static constexpr int kOffBar = kOffVt + 2 * kVtBytes;
  static constexpr int kSmem = kOffBar + 128 + 1024;
  static constexpr int kTmemCols = 2 * BK + kD <= 128 ? 128 : 256;
  static constexpr int kMinCtas = 512 / kTmemCols;
  static_assert(2 * BK + kD <= 256, "two S accumulators and O must fit the CTA's TMEM share");
  static_assert(BK % 16 == 0, "tile shape");
};

struct AttnArgs {
  uint16_t* out;
  int T, n_q, n_kv, shared_kv, q_tiles;
  int stack_rows;   // > 0: the six query heads of a (b, t) column are stacked on the tile's row axis, Sq_pad rows each
  int kv_slots;     // shared_kv: estimators per rank chunk of the K/V context (>= 1; B when the context is dense)
  int tiles_per_seg;   // key tiles per row segment (row-sharded context: keys stored in per-rank chunks); 2^30 = one range
  // per-entry counts (the RAGGED instantiation only; entry = bt / T): query rows and keys of entry b, or NULL = n_q / n_kv
  const int* q_len;
  const int* kv_len;
};

#ifdef MMPFN_DEBUG
// tuning build only: clock64 stamps of one CTA (tools/attn_trace.py)
__device__ long long g_attn_trace[8192];
#define ATTN_TRACE(slot)                                                      \
  do {                                                                        \
    if (blockIdx.x == 5001 && (slot) < 8192) g_attn_trace[(slot)] = clock64(); \
  } while (0)
#else
#define ATTN_TRACE(slot) do {} while (0)
#endif

// try_wait parks the thread in hardware until the barrier completes its phase, the hint expires, or — measured:
// ~18 wake-ups per key tile and CTA — ANY mbarrier of the CTA sees an arrival.  A woken thread that finds its phase
// incomplete must go back to sleep cheaply: eight bare probes (four instructions each) per visit of the bounded
// counter; a wait that outlives ~2^20 probes traps instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait_lean(uint32_t addr, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .u32 n;\n\t"
      "mov.u32 n, 0;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t@p bra DONE_%=;\n\t"
      "add.u32 n, n, 1;\n\t"
      "setp.lt.u32 p, n, 131072;\n\t"
      "@p bra WAIT_%=;\n\t"
      "trap;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(addr), "r"(parity), "r"(20000u)
      : "memory");
}
__device__ __forceinline__ bool mbar_test_addr(uint32_t addr, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(addr), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ void mbar_expect_tx_addr(uint32_t addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void umma_commit_addr(uint32_t addr) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void tma_load_3d_addr(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d_addr(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                                 int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ uint64_t sub_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// 2^x for a PAIR of scores on the FMA / ALU pipes (no MUFU), ten instructions:
//   r = x + 1.5*2^23 (round(x) lands in the low mantissa bits), f = x - (r - 1.5*2^23) in [-0.5, 0.5]   3 FADD2
//   2^f * 2^-100 by a degree-3 minimax polynomial (max relative error 7.6e-5 << bf16 rounding of P)        3 FFMA2
//   t = clamp(round(x) + 100, 0, 226) by one VIADDMNMX.RELU each; result bits = poly bits + (t << 23)       2 + 2 LEA
// i.e. 2^x for x in [-100, 126]; below, the result saturates at ~2^-100 (nothing: the row reference is at
// most 2^8 above), above at ~2^126 (the row sum overflows the limit and the tile is repeated against the
// true maximum — never a wrapped exponent).  NaN / +inf in give NaN out, which fails the row-sum test too.
constexpr float kPolyScale = 7.888609052210118e-31f;     // 2^-100
__device__ __forceinline__ void poly_exp2_pair(uint32_t& a, uint32_t& b) {
  const uint64_t x2 = pack_f32x2(__uint_as_float(a), __uint_as_float(b));
  const uint64_t m2 = pack_f32x2(12582912.0f, 12582912.0f);
  const uint64_t r2 = add_f32x2(x2, m2);
  const uint64_t f2 = sub_f32x2(x2, sub_f32x2(r2, m2));
  uint64_t p2 = fma_f32x2(pack_f32x2(0.05520550534129143f * kPolyScale, 0.05520550534129143f * kPolyScale), f2,
                          pack_f32x2(0.24261397123336792f * kPolyScale, 0.24261397123336792f * kPolyScale));
  p2 = fma_f32x2(p2, f2, pack_f32x2(0.6932547688484192f * kPolyScale, 0.6932547688484192f * kPolyScale));
  p2 = fma_f32x2(p2, f2, pack_f32x2(0.9999276995658875f * kPolyScale, 0.9999276995658875f * kPolyScale));
  float pl, ph, rl, rh;
  unpack_f32x2(p2, pl, ph);
  unpack_f32x2(r2, rl, rh);
  const int tl = __viaddmin_s32_relu(__float_as_int(rl), 100 - 0x4B400000, 226);
  const int th = __viaddmin_s32_relu(__float_as_int(rh), 100 - 0x4B400000, 226);
  a = (uint32_t)(tl * 0x800000 + __float_as_int(pl));
  b = (uint32_t)(th * 0x800000 + __float_as_int(ph));
}
// which of the NP key pairs of a tile take the polynomial: PP of NP, evenly spread
__host__ __device__ constexpr bool poly_pair(int k, int PP, int NP) { return ((k + 1) * PP) / NP != (k * PP) / NP; }

// n consecutive fp32 columns of this warp's 32 TMEM lanes into v[0..n)
template <int N>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, uint32_t* v) {
  static_assert(N % 16 == 0, "columns come in chunks of 16");
#pragma unroll
  for (int c = 0; c + 32 <= N; c += 32) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[c + 0]), "=r"(v[c + 1]), "=r"(v[c + 2]), "=r"(v[c + 3]), "=r"(v[c + 4]), "=r"(v[c + 5]),
          "=r"(v[c + 6]), "=r"(v[c + 7]), "=r"(v[c + 8]), "=r"(v[c + 9]), "=r"(v[c + 10]), "=r"(v[c + 11]),
          "=r"(v[c + 12]), "=r"(v[c + 13]), "=r"(v[c + 14]), "=r"(v[c + 15]), "=r"(v[c + 16]), "=r"(v[c + 17]),
          "=r"(v[c + 18]), "=r"(v[c + 19]), "=r"(v[c + 20]), "=r"(v[c + 21]), "=r"(v[c + 22]), "=r"(v[c + 23]),
          "=r"(v[c + 24]), "=r"(v[c + 25]), "=r"(v[c + 26]), "=r"(v[c + 27]), "=r"(v[c + 28]), "=r"(v[c + 29]),
          "=r"(v[c + 30]), "=r"(v[c + 31])
        : "r"(taddr + c)
        : "memory");
  }
  if (N % 32 == 16) {
    constexpr int c = N - 16;
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[c + 0]), "=r"(v[c + 1]), "=r"(v[c + 2]), "=r"(v[c + 3]), "=r"(v[c + 4]), "=r"(v[c + 5]),
          "=r"(v[c + 6]), "=r"(v[c + 7]), "=r"(v[c + 8]), "=r"(v[c + 9]), "=r"(v[c + 10]), "=r"(v[c + 11]),
          "=r"(v[c + 12]), "=r"(v[c + 13]), "=r"(v[c + 14]), "=r"(v[c + 15])
        : "r"(taddr + c)
        : "memory");
  }
}

// n consecutive 32-bit columns of this warp's 32 TMEM lanes from v[0..n), n a multiple of 8
template <int N>
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t* v) {
  static_assert(N % 8 == 0, "columns go in chunks of 8");
  int c = 0;
#pragma unroll
  for (; c + 16 <= N; c += 16) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr + c), "r"(v[c + 0]), "r"(v[c + 1]), "r"(v[c + 2]), "r"(v[c + 3]), "r"(v[c + 4]), "r"(v[c + 5]),
          "r"(v[c + 6]), "r"(v[c + 7]), "r"(v[c + 8]), "r"(v[c + 9]), "r"(v[c + 10]), "r"(v[c + 11]), "r"(v[c + 12]),
          "r"(v[c + 13]), "r"(v[c + 14]), "r"(v[c + 15])
        : "memory");
  }
  if (N % 16 == 8) {
    constexpr int c8 = N - 8;
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr + c8), "r"(v[c8 + 0]), "r"(v[c8 + 1]), "r"(v[c8 + 2]), "r"(v[c8 + 3]), "r"(v[c8 + 4]),
                   "r"(v[c8 + 5]), "r"(v[c8 + 6]), "r"(v[c8 + 7])
                 : "memory");
  }
}

// Barriers (phase n of each counts from 0):
//   q_full        Q, K(0), K(1) have landed
//   kv_full[s]    n-th refill of slot s: V^T(2n+s) and K(2n+s+2) have landed
//   p_full[s]     n-th time the four softmax warps have written P(2n+s) into TMEM buffer s
//   done[s]       n = 0: S(s) of the prologue has completed; n >= 1: iteration j = 2(n-1)+s of the MMA
//                 thread — P V(j), then S(j+2) into buffer s — has.  One arrival tells the softmax
//                 that S(j+2) is in TMEM and that O holds P V(j), and the TMA thread that V slot s and
//                 K slot s (K(j+2), just consumed) are free.
//   warps 0-3  softmax, thread = query row (TMEM lane quarter = warp)
//   warp 4     TMA producer + TMEM allocation
//   warp 5     MMA issue
// RAGGED: entry b has its own key count kv_len[b] (tiles past it are not visited; its last tile is masked like the
// tail tile) and query count q_len[b] (output rows from there up to n_q are written as zeros; a tile holding only
// such rows stores its zeros and issues nothing else).  The other instantiation is the one the layer passes use.
template <int BK, int PP, bool RAGGED, int FMT>
__global__ void __launch_bounds__(A_THREADS, AttnCfg<BK>::kMinCtas)
    tc_item_attn_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                        const __grid_constant__ CUtensorMap map_vt, const AttnArgs p) {
  using C = AttnCfg<BK>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + C::kOffBar);
  const uint32_t sbase = pin_u32(smem_u32(smem));
  const uint32_t bar0 = pin_u32(sbase + C::kOffBar);
  const uint32_t q_full = bar0, kv_full = bar0 + 8, p_full = bar0 + 24, done = bar0 + 40;   // [2] each after q_full
  uint32_t* tmem_slot = (uint32_t*)(bars + 8);

  const int warp = threadIdx.x >> 5, lane = (int)pin_u32(threadIdx.x & 31);
  // Train pass: plane = (b*T + t)*kH + h, q tiles of a plane are adjacent CTAs.  Test pass (all six query
  // heads read the head-0 K/V of their column, multi_head_attention.py:436-445): the heads are stacked on
  // the row axis — row = h * Sq_pad + s of column bt — so that 6 x 300 rows fill 15 tiles instead of 18.
  const int plane = blockIdx.x / p.q_tiles;
  const int q0 = (blockIdx.x % p.q_tiles) * A_BQ;
  const int h = p.stack_rows ? 0 : plane % kH;
  const int bt = p.stack_rows ? plane : plane / kH;
  // K / V^T planes through 5-D tensor maps {.., .., c2, c3, c4}: own planes (train pass) are (plane, 0, 0); the
  // shared head-0 context (test pass) is (token column, slot, rank) — dense or inside an all-gather buffer
  const int kb = bt / p.T;
  const int kc2 = p.shared_kv ? bt - kb * p.T : plane;
  const int kc3 = p.shared_kv ? kb % p.kv_slots : 0;
  const int kc4 = p.shared_kv ? kb / p.kv_slots : 0;
  int n_kv = p.n_kv, n_q = p.n_q;
  if constexpr (RAGGED) {
    if (p.kv_len) n_kv = min(max(p.kv_len[kb], 1), p.n_kv);
    if (p.q_len) n_q = min(max(p.q_len[kb], 0), p.n_q);
    // does the tile hold a row of this entry (stacked: of any head)?
    bool live = q0 < n_q;
    if (p.stack_rows) {
      live = false;
      for (int hh = 0; hh < kH; ++hh) live |= hh * p.stack_rows < q0 + A_BQ && hh * p.stack_rows + n_q > q0;
    }
    if (!live) {
      if (threadIdx.x < A_BQ) {
        int qi = q0 + threadIdx.x, hh = h;
        if (p.stack_rows) {
          hh = qi / p.stack_rows;
          qi = hh < kH ? qi - hh * p.stack_rows : p.n_q;
        }
        if (qi < p.n_q) {
          uint4* d4 = reinterpret_cast<uint4*>(p.out + (((long long)kb * p.n_q + qi) * p.T + (bt - kb * p.T)) * kE + hh * kD);
#pragma unroll
          for (int i = 0; i < 4; ++i) d4[i] = make_uint4(0, 0, 0, 0);
        }
      }
      return;
    }
  }
  const int nkt = (n_kv + BK - 1) / BK;

  if (threadIdx.x == 0) {
    prefetch_tmap(&map_q);
    prefetch_tmap(&map_k);
    prefetch_tmap(&map_vt);
    mbar_init(bars, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(bars + 1 + s, 1);     // kv_full
      mbar_init(bars + 3 + s, ATTN_ONE_ARRIVE ? 1 : 4);     // p_full: one arrival per softmax warp (or one in all)
      mbar_init(bars + 5 + s, 1);     // done
    }
    fence_barrier_init();
  }
  if (warp == 4) tmem_alloc(tmem_slot, C::kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_o = tmem + 2 * BK;

  if (warp == 4) {
    if (elect_one()) {
      mbar_expect_tx_addr(q_full, A_Q_BYTES + (nkt > 1 ? 2 : 1) * C::kKTx);
      tma_load_3d_addr(sbase, &map_q, q_full, 0, q0, plane);
      // key tile j = rows [row, row + BK) of row segment seg (one segment unless the context build is row-sharded)
      const int tps = p.tiles_per_seg;
      auto seg_of = [&](int j, int& row) { const int sg = j / tps; row = (j - sg * tps) * BK; return sg; };
      int row, sg = seg_of(0, row);
      tma_load_5d_addr(sbase + C::kOffK, &map_k, q_full, 0, row, kc2, kc3 + sg, kc4);
      if (nkt > 1) {
        sg = seg_of(1, row);
        tma_load_5d_addr(sbase + C::kOffK + C::kKSlot, &map_k, q_full, 0, row, kc2, kc3 + sg, kc4);
      }
      // refill g: V^T(g) and K(g+2) into slot g & 1 once done[g & 1] has completed g/2 + 1 times
      for (int g = 0; g < nkt; ++g) {
        const uint32_t s = g & 1;
        const bool has_k = g + 2 < nkt;
        mbar_wait_lean(done + s * 8, (g >> 1) & 1);
        mbar_expect_tx_addr(kv_full + s * 8, C::kVtBytes + (has_k ? C::kKTx : 0));
        sg = seg_of(g, row);
#pragma unroll
        for (int kb = 0; kb < C::kNKB; ++kb)
          tma_load_5d_addr(sbase + C::kOffVt + s * C::kVtBytes + kb * (kD * 128), &map_vt, kv_full + s * 8,
                           row + kb * 64, 0, kc2, kc3 + sg, kc4);
        if (has_k) {
          sg = seg_of(g + 2, row);
          tma_load_5d_addr(sbase + C::kOffK + s * C::kKSlot, &map_k, kv_full + s * 8, 0, row, kc2, kc3 + sg, kc4);
        }
      }
    }
  } else if (warp == 5) {
    if (elect_one()) {
      constexpr uint32_t idesc_s = make_idesc_fmt<FMT>(A_BQ, BK);
      constexpr uint32_t idesc_o = make_idesc_fmt<FMT>(A_BQ, kD);
      const uint64_t qdesc = make_desc(sbase, 512, kSw64);
      const uint64_t kdesc0 = make_desc(sbase + C::kOffK, 512, kSw64);
      const uint64_t vdesc0 = make_desc(sbase + C::kOffVt, 1024, kSw128);
      // S = Q K^T of the tile whose K sits in slot s, into TMEM buffer s
      auto issue_s = [&](uint32_t s) {
        const uint64_t kdesc = kdesc0 + (uint64_t)((s * C::kKSlot) >> 4);
#pragma unroll
        for (int k = 0; k < kD / 16; ++k)
          umma_bf16(tmem + s * BK, qdesc + (uint64_t)(k * 2), kdesc + (uint64_t)(k * 2), idesc_s, k != 0);
      };
      mbar_wait_lean(q_full, 0);
      tc_fence_after();
      issue_s(0);
      umma_commit_addr(done);
      if (nkt > 1) {
        issue_s(1);
        umma_commit_addr(done + 8);
      }
      for (int j = 0; j < nkt; ++j) {
        const uint32_t s = j & 1, ph = (j >> 1) & 1;
        mbar_wait_lean(kv_full + s * 8, ph);      // V^T(j) and K(j+2): landed long ago, off the critical path
        mbar_wait_lean(p_full + s * 8, ph);       // P(j) is in TMEM buffer s
        tc_fence_after();
        ATTN_TRACE(4096 + j * 2);
        const uint64_t vdesc = vdesc0 + (uint64_t)((s * C::kVtBytes) >> 4);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)
          umma_bf16_ts(tmem_o, tmem + s * BK + k * 8, vdesc + (uint64_t)((k / 4) * ((kD * 128) >> 4) + (k % 4) * 2),
                       idesc_o, (j | k) != 0);
        // S(j+2) overwrites the columns P(j) sits in: issued behind P V(j) (tcgen05 ops of one thread
        // execute in order)
        if (j + 2 < nkt) issue_s(s);
        umma_commit_addr(done + s * 8);
        ATTN_TRACE(4096 + j * 2 + 1);
      }
    }
  } else {
    // ---- softmax warps: thread = one query row ----
    const int r = warp * 32 + lane;
    const uint32_t lane_off = pin_u32((uint32_t)(warp * 32) << 16);
    const float c = 0.17677669529663687f * 1.4426950408889634f;   // log2(e)/sqrt(d)
    // m_ref is the score the exponent of this row is measured from.  It only follows the running
    // maximum when that has grown by more than kTau (log2 units): p = 2^((s - m_ref) c) then stays
    // below 2^kTau, which fp32 sums and bf16 P hold without loss, and the round trip that rescales O
    // in TMEM (needed on nearly every tile otherwise) becomes rare after the first tiles.
    constexpr float kSumLimit = 256.0f;          // 2^kTau, kTau = 8
    constexpr float kMasked = -1.0e30f;          // a key past n_kv: 2^x of it is 0 (MUFU) or 2^-100 (polynomial), V^T is 0 there
    constexpr int kNP = BK / 2;                  // pairs of keys per row and tile
    constexpr int kAhead = ATTN_KAHEAD;          // pairs whose scaled argument is ready ahead of their ex2
    constexpr int kBehind = ATTN_KBEHIND;        // pairs whose ex2 is in flight before the first consumer reads one
    float m_ref = -INFINITY, l_run = 0.f;
    bool next_ready = false;
    uint32_t sv[BK];
    for (int j = 0; j < nkt; ++j) {
      const int sb = j & 1;
      const uint32_t tmem_s = tmem + sb * BK + lane_off;
      const int valid = n_kv - j * BK;           // keys of this tile that exist
      // S(j) is in TMEM (and P V(j-2) has drained buffer sb).  Usually the probe made at the end of the
      // previous tile has already said so.
      if (threadIdx.x == 0) ATTN_TRACE(j * 8 + 0);
      if (!next_ready) mbar_wait_lean(done + sb * 8, (j >> 1) & 1);
      tc_fence_after();
      if (threadIdx.x == 0) ATTN_TRACE(j * 8 + 1);

      // the whole row of S into registers (masking the keys a partial last tile does not have)
      auto load_row = [&]() {
        tmem_ld_cols<BK>(tmem_s, sv);
        tmem_ld_wait();
        if (valid < BK) {
#pragma unroll
          for (int i = 0; i < BK; ++i)
            if (i >= valid) sv[i] = __float_as_uint(kMasked);
        }
      };
      // One software-pipelined sweep over the row: step k scales pair k+kAhead (FFMA2), starts the
      // exponentials of pair k (two MUFU.EX2, or the packed polynomial), and retires pair k-kBehind
      // (row sum FADD2, bf16 pack F2FP, in place: slot k of sv then holds the packed pair).  Values are
      // transformed in place: s -> x -> p.  No row maximum is tracked here.
      const uint64_t c2 = pack_f32x2(c, c);
      bool probe = false;
      const uint32_t probe_bar = done + (sb ^ 1) * 8, probe_par = ((j + 1) >> 1) & 1;
      auto sweep = [&](float mc, bool with_probe) -> float {
        const uint64_t nmc2 = pack_f32x2(-mc, -mc);
        uint64_t lsum2 = 0ull;                                // (0.f, 0.f)
        auto scale = [&](int k) {
          float xa, xb;
          unpack_f32x2(fma_f32x2(pack_f32x2(__uint_as_float(sv[2 * k]), __uint_as_float(sv[2 * k + 1])), c2, nmc2), xa, xb);
          sv[2 * k] = __float_as_uint(xa);
          sv[2 * k + 1] = __float_as_uint(xb);
        };
        auto expo = [&](int k) {
          if (poly_pair(k, PP, kNP)) {
            poly_exp2_pair(sv[2 * k], sv[2 * k + 1]);
          } else {
            sv[2 * k] = __float_as_uint(fast_exp2(__uint_as_float(sv[2 * k])));
            sv[2 * k + 1] = __float_as_uint(fast_exp2(__uint_as_float(sv[2 * k + 1])));
          }
        };
        auto retire = [&](int k) {
          const float a = __uint_as_float(sv[2 * k]), b = __uint_as_float(sv[2 * k + 1]);
          lsum2 = add_f32x2(lsum2, pack_f32x2(a, b));
          sv[k] = pack16x2<FMT>(a, b);       // slot k belonged to pair k / 2, retired no later than this one
        };
#pragma unroll
        for (int k = 0; k < kAhead; ++k) scale(k);
#pragma unroll
        for (int k = 0; k < kNP + kBehind; ++k) {
          if (k + kAhead < kNP) scale(k + kAhead);
          if (k < kNP) expo(k);
          if (k >= kBehind) retire(k - kBehind);
          // the probe's ~200-cycle round trip runs under the rest of the sweep
          if (k == ATTN_PROBE_AT && with_probe) probe = j + 1 < nkt && mbar_test_addr(probe_bar, probe_par);
        }
        float lsum0, lsum1;
        unpack_f32x2(lsum2, lsum0, lsum1);
        return lsum0 + lsum1;
      };
      // the true maximum of the row of S held in sv (first tile, and the rare repeat below)
      auto row_max = [&]() -> float {
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
#pragma unroll
        for (int i = 0; i < BK; i += 8) {
          mx0 = fmaxf(mx0, fmaxf(__uint_as_float(sv[i]), __uint_as_float(sv[i + 1])));
          mx1 = fmaxf(mx1, fmaxf(__uint_as_float(sv[i + 2]), __uint_as_float(sv[i + 3])));
          mx2 = fmaxf(mx2, fmaxf(__uint_as_float(sv[i + 4]), __uint_as_float(sv[i + 5])));
          mx3 = fmaxf(mx3, fmaxf(__uint_as_float(sv[i + 6]), __uint_as_float(sv[i + 7])));
        }
        return fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
      };
      load_row();
      if (threadIdx.x == 0) ATTN_TRACE(j * 8 + 2);
      if (j == 0) m_ref = row_max();             // first tile: the reference is the true maximum of the tile
      // Later tiles: exponentials are taken against the reference of the earlier tiles, and no maximum
      // is computed at all: a score more than kTau (log2 units) above the reference shows up as a row
      // sum above 2^kTau (p <= sum p; inf and NaN fail the comparison too).  Only then — rare: the
      // running maximum of n keys moves ~ log n times, and a sum that merely crowds the limit just
      // refreshes the reference — is the true maximum taken and the sweep repeated.  S was consumed in
      // place, so the repeat reads it from TMEM again: P only overwrites the S columns after the decision.
      float lsum = sweep(m_ref * c, true);
      // early probe of the next tile's S: consumed at the top of the next iteration
      if (ATTN_PROBE_AT >= kNP + kBehind) probe = j + 1 < nkt && mbar_test_addr(probe_bar, probe_par);
      if (threadIdx.x == 0) ATTN_TRACE(j * 8 + 3);
      const bool moved = !(lsum <= kSumLimit);
      const bool any_moved = __any_sync(0xffffffffu, moved);   // tcgen05.ld is warp-collective
      float alpha = 1.0f;
      if (any_moved) {
        load_row();
        if (moved) {
          const float mx = fmaxf(row_max(), m_ref);
          alpha = fast_exp2((m_ref - mx) * c);
          m_ref = mx;
        }
        lsum = sweep(m_ref * c, false);
      }
      tmem_st_cols<BK / 2>(tmem_s, sv);          // P(j) over the first half of the S(j) columns
      l_run = l_run * alpha + lsum;
      if (threadIdx.x == 0) ATTN_TRACE(j * 8 + 4);
      // rescale the running output when some row of this warp moved its reference: needs P V(j-1),
      // i.e. iteration j-1 of the MMA thread = completion (j-1)/2 + 1 of done[(j-1) & 1]
      if (any_moved) {
        mbar_wait_lean(done + ((j - 1) & 1) * 8, (((j - 1) >> 1) + 1) & 1);   // j >= 1 here: tile 0 never moves
        tc_fence_after();
        uint32_t o[32];
        tmem_ld32(tmem_o + lane_off, o);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
        tmem_st32(tmem_o + lane_off, o);
      }
      // hand-off: P(j) (and a rescaled O) are in TMEM -> one arrival per warp on p_full.  (Deferring this under the
      // next tile's TMEM load was measured: 446 instead of 471 TFLOP/s — the MMA thread starts P V(j) later.)
      tmem_st_wait();
      if (threadIdx.x == 0) ATTN_TRACE(j * 8 + 5);
      tc_fence_before();
#if ATTN_ONE_ARRIVE
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (threadIdx.x == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(p_full + sb * 8) : "memory");
#else
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(p_full + sb * 8) : "memory");
#endif
      if (threadIdx.x == 0) ATTN_TRACE(j * 8 + 6);
      next_ready = __all_sync(0xffffffffu, probe);
      if (threadIdx.x == 0) ATTN_TRACE(j * 8 + 7);
    }
    uint32_t v[32];
    // the last iteration of the MMA thread: tcgen05 ops complete in order, so this covers all P V
    mbar_wait_lean(done + ((nkt - 1) & 1) * 8, (((nkt - 1) >> 1) + 1) & 1);
    tc_fence_after();
    tmem_ld32(tmem_o + lane_off, v);
    tmem_ld_wait();
    int qi = q0 + r, hh = h;
    if (p.stack_rows) {
      hh = qi / p.stack_rows;
      qi = hh < kH ? qi - hh * p.stack_rows : p.n_q;      // rows past the last head: nothing to store
    }
    if (qi < p.n_q) {
      float inv = 1.0f / l_run;
      if constexpr (RAGGED) {
        if (qi >= n_q) {                         // a pad row of this entry
          inv = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0u;
        }
      }
      const int b = bt / p.T, t = bt % p.T;
      uint16_t* dst = p.out + (((long long)b * p.n_q + qi) * p.T + t) * kE + hh * kD;
      uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        d4[i] = make_uint4(pack16x2<FMT>(__uint_as_float(v[8 * i]) * inv, __uint_as_float(v[8 * i + 1]) * inv),
                           pack16x2<FMT>(__uint_as_float(v[8 * i + 2]) * inv, __uint_as_float(v[8 * i + 3]) * inv),
                           pack16x2<FMT>(__uint_as_float(v[8 * i + 4]) * inv, __uint_as_float(v[8 * i + 5]) * inv),
                           pack16x2<FMT>(__uint_as_float(v[8 * i + 6]) * inv, __uint_as_float(v[8 * i + 7]) * inv));
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem, C::kTmemCols);
  }
}

template <int BK, int PP, bool RAGGED = false, int FMT = FMT_BF16>
int launch_attn_t(const CUtensorMap& mq, const CUtensorMap& mk, const CUtensorMap& mvt, const AttnArgs& a, dim3 grid,
                  cudaStream_t st) {
  using C = AttnCfg<BK>;
  MMPFN_OPT_IN_SMEM((tc_item_attn_kernel<BK, PP, RAGGED, FMT>), C::kSmem);
  tc_item_attn_kernel<BK, PP, RAGGED, FMT><<<grid, A_THREADS, C::kSmem, st>>>(mq, mk, mvt, a);
  return count_launch();
}

}  // namespace

int launch_tc_item_attn(const TcItemAttn& p, cudaStream_t st, int fmt) {
  constexpr int BK = 48;
  if (p.n_q <= 0 || p.B <= 0) return MMPFN_OK;
  if (p.n_kv <= 0) { set_error("item attention: empty key set"); return MMPFN_EINVAL; }
  const long long planes_q = (long long)p.B * p.T * kH;
  const long long planes_kv = p.shared_kv ? (long long)p.B * p.T : planes_q;
  // stacking pays when it saves tiles; the rows between n_q and Sq_pad of every head are then computed
  // (and dropped), so they should hold finite values (the QKV projection writes zeros there)
  const bool stack = p.shared_kv && (kH * p.Sq_pad + A_BQ - 1) / A_BQ < kH * ((p.n_q + A_BQ - 1) / A_BQ);
  const int q_tiles = stack ? (kH * p.Sq_pad + A_BQ - 1) / A_BQ : (p.n_q + A_BQ - 1) / A_BQ;
  const long long grid_planes = stack ? planes_kv : planes_q;
  if (grid_planes * q_tiles > 2147483647LL) { set_error("item attention: grid too large"); return MMPFN_EUNSUPPORTED; }
  CUtensorMap mq, mk, mvt;
  {
    const cuuint64_t dims[3] = {(cuuint64_t)kD, (cuuint64_t)(stack ? kH * p.Sq_pad : p.n_q),
                                (cuuint64_t)(stack ? planes_kv : planes_q)};
    const cuuint64_t strides[2] = {(cuuint64_t)kD * 2, (cuuint64_t)(stack ? kH : 1) * p.Sq_pad * kD * 2};
    const cuuint32_t box[3] = {kD, A_BQ, 1};
    MMPFN_TRY(encode_map(&mq, p.q, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B));
  }
  // K / V^T: {.., rows, c2, c3, c4} = (plane, row segment, 0) for own planes; for the shared context
  // (token column, slot, rank) when it sits in the estimator gather buffer or (token column, row segment, estimator)
  // when it was built row-sharded
  int slots = 1, tiles_per_seg = 1 << 30;
  cuuint64_t n2 = (cuuint64_t)planes_kv, n3 = 1, n4 = 1;
  const cuuint64_t plane_bytes = (cuuint64_t)p.Skv_pad * kD * 2;
  cuuint64_t s3 = plane_bytes * n2, s4 = plane_bytes * n2;
  cuuint64_t rows_extent = (cuuint64_t)p.n_kv;
  if (p.kv_seg_rows > 0) {
    if (p.kv_seg_rows % BK != 0 || p.kv_seg_rows > p.Skv_pad || p.kv_slots > 0 || (p.kv_seg_stride * 2) % 16 != 0) {
      set_error("item attention: row segments of %d rows (must be a multiple of %d, <= %d allocated rows)", p.kv_seg_rows, BK, p.Skv_pad);
      return MMPFN_EINVAL;
    }
    tiles_per_seg = p.kv_seg_rows / BK;
    rows_extent = (cuuint64_t)p.kv_seg_rows;      // pad rows of a short last segment are read: the caller keeps them finite
    n3 = (cuuint64_t)((p.n_kv + p.kv_seg_rows - 1) / p.kv_seg_rows);
    s3 = (cuuint64_t)p.kv_seg_stride * 2;
    if (p.shared_kv) { n2 = (cuuint64_t)p.T; n4 = (cuuint64_t)p.B; s4 = plane_bytes * p.T; }
  } else if (p.shared_kv) {
    slots = p.kv_slots > 0 ? p.kv_slots : p.B;
    if (p.B % slots != 0) { set_error("item attention: %d estimators do not fill chunks of %d", p.B, slots); return MMPFN_EINVAL; }
    n2 = (cuuint64_t)p.T; n3 = (cuuint64_t)slots; n4 = (cuuint64_t)(p.B / slots);
    s3 = plane_bytes * p.T;
    s4 = p.kv_slots > 0 ? (cuuint64_t)p.kv_rank_stride * 2 : s3 * slots;
    if (s4 % 16 != 0 || (n4 > 1 && s4 < s3 * slots)) { set_error("item attention: bad rank stride of the K/V context"); return MMPFN_EINVAL; }
  }
  {
    const cuuint64_t dims[5] = {(cuuint64_t)kD, rows_extent, n2, n3, n4};
    const cuuint64_t strides[4] = {(cuuint64_t)kD * 2, plane_bytes, s3, s4};
    const cuuint32_t box[5] = {kD, BK, 1, 1, 1};
    MMPFN_TRY(encode_map(&mk, p.k, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B));
  }
  {
    const cuuint64_t dims[5] = {rows_extent, (cuuint64_t)kD, n2, n3, n4};
    const cuuint64_t strides[4] = {(cuuint64_t)p.Skv_pad * 2, plane_bytes, s3, s4};
    const cuuint32_t box[5] = {64, kD, 1, 1, 1};
    MMPFN_TRY(encode_map(&mvt, p.vt, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  AttnArgs a{p.out, p.T, p.n_q, p.n_kv, p.shared_kv, q_tiles, stack ? p.Sq_pad : 0, slots, tiles_per_seg, p.q_len, p.kv_len};
  const dim3 grid((unsigned)(grid_planes * q_tiles));
  if (fmt == FMT_F16) {
    // fp16: P is stored only after the row-sum decision, so every stored p is <= kSumLimit (2^8), far inside fp16's range
    if (p.q_len || p.kv_len) return launch_attn_t<BK, kPolyPairsDefault, true, FMT_F16>(mq, mk, mvt, a, grid, st);
    return launch_attn_t<BK, kPolyPairsDefault, false, FMT_F16>(mq, mk, mvt, a, grid, st);
  }
  if (p.q_len || p.kv_len) return launch_attn_t<BK, kPolyPairsDefault, true>(mq, mk, mvt, a, grid, st);
#ifdef MMPFN_DEBUG
  // tuning builds only (-DMMPFN_DEBUG): MMPFN_ATTN_PP = polynomial pairs of every 24.  The product
  // library has exactly one variant and reads no environment variable.
  static int pp = -1;
  if (pp < 0) {
    const char* e = getenv("MMPFN_ATTN_PP");
    pp = e ? atoi(e) : kPolyPairsDefault;
  }
  switch (pp) {
    case 0: return launch_attn_t<BK, 0>(mq, mk, mvt, a, grid, st);
    case 3: return launch_attn_t<BK, 3>(mq, mk, mvt, a, grid, st);
    case 4: return launch_attn_t<BK, 4>(mq, mk, mvt, a, grid, st);
    case 8: return launch_attn_t<BK, 8>(mq, mk, mvt, a, grid, st);
    case 10: return launch_attn_t<BK, 10>(mq, mk, mvt, a, grid, st);
    case 12: return launch_attn_t<BK, 12>(mq, mk, mvt, a, grid, st);
    default: break;
  }
#endif
  return launch_attn_t<BK, kPolyPairsDefault>(mq, mk, mvt, a, grid, st);
}

}  // namespace mmpfn

#ifdef MMPFN_DEBUG
extern "C" int mmpfn_debug_attn_trace(long long* host_out, int n) {
  if (n > 8192) n = 8192;
  return cudaMemcpyFromSymbol(host_out, mmpfn::g_attn_trace, sizeof(long long) * n) == cudaSuccess ? 0 : MMPFN_ECUDA;
}
#endif
