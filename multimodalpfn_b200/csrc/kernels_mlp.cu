// kernels_mlp.cu — the whole MLP sublayer of a PerFeatureEncoderLayer in ONE persistent kernel:
//
//     state <- LayerNorm(state + W2 gelu(W1 state))            (mlp.py:93-138, layer.py:437-455)
//
// The 768-wide hidden activation never leaves the SM.  Per 128-token tile the hidden axis is walked
// in 12 chunks of 64: GEMM1 (tcgen05, 128 x 64 x 192) leaves the chunk in TMEM, eight GELU warps
// turn it into a bf16 K-major operand tile in shared memory, GEMM2 (128 x 192 x 64) accumulates it
// into the output tile in TMEM, and four epilogue warps add the fp32 residual, normalise and write
// the fp32 state and its bf16 shadow.  HBM traffic per token is 192 x (2 + 4 + 4 + 2) B instead of
// the 192 x 28 B of the two-GEMM form (the 768 x 2 B hidden row written and read back).
//
// One CTA per SM, all 512 TMEM columns: two output accumulators (the epilogue of tile i runs under
// the MMAs of tile i+1) and two hidden-chunk accumulators (GEMM1 of chunk g+1 runs under the GELU
// of chunk g).
//
//   warp 0        TMA producer: activation tile (1 buffer), W1 and W2 chunks (separate 2-slot rings)
//   warp 1        GEMM1 issue
//   warp 2        TMEM allocation, then TMA producer of the fp32 residual chunks
//   warp 3        GEMM2 issue
//   warps 4-11    GELU: TMEM lane quarter = warp % 4, chunk parity = (warp - 4) / 4
//   warps 12-15   epilogue: residual + LayerNorm, thread = token row
//
// The epilogue never touches global memory with thread-private accesses (16-byte pieces at a 768-byte
// stride: one L1 wavefront each, ~15k per tile, which also starved the GELU warps' shared-memory
// stores): the fp32 residual arrives by TMA as 128B-swizzled [128 x 32] chunks through a 3-slot ring,
// and the fp32 state / bf16 shadow leave through swizzled staging slots and TMA stores.  Ring and
// staging share the same 48 KB (pass 1 consumes, pass 2 produces); the next tile's first three
// residual chunks are requested when pass 2 has released the memory, ten chunks before they are read.
//
// GELU: 0.5 x (1 + erf(x / sqrt 2)) with erf(z) = tanh(g(z)), g an odd polynomial fitted to
// atanh(erf) (max |error| of the GELU 3e-5 before the hardware tanh, whose 2^-11 relative error is
// a quarter of the bf16 rounding the hidden activation gets anyway, and about the size of the fp16
// one); one MUFU.TANH and ~5 issue slots per element with packed f32x2 arithmetic, against ~30 for erff().
// The kernel is instantiated for bf16 and for fp16 operands (FMT): the tiles and bytes are the same.
#include "tc_common.cuh"

namespace mmpfn {
namespace {

constexpr int F_BM = 128;                         // tokens per tile
constexpr int F_CH = 64;                          // hidden columns per chunk
constexpr int F_NCH = kHid / F_CH;                // 12
constexpr int F_A_BYTES = F_BM * kE * 2;          // 48 KB: 3 k-blocks [128][64] bf16, 128B swizzle
constexpr int F_W1_BYTES = F_CH * kE * 2;         // 24 KB: 3 k-blocks [64][64]
constexpr int F_W2_BYTES = kE * F_CH * 2;         // 24 KB: [192][64]
constexpr int F_WSTAGE = F_W1_BYTES + F_W2_BYTES;
constexpr int F_HS_BYTES = F_BM * F_CH * 2;       // 16 KB: [128][64] bf16, 128B swizzle
constexpr int F_RC = 32;                          // residual / output chunk: 32 columns
constexpr int F_NRC = kE / F_RC;                  // 6 per row
constexpr int F_R_BYTES = F_BM * F_RC * 4;        // 16 KB: [128][128 B] fp32, 128B swizzle
constexpr int F_R_SLOTS = 3;
constexpr int F_OFF_A = 0;
constexpr int F_OFF_W = F_A_BYTES;
constexpr int F_OFF_HS = F_OFF_W + 2 * F_WSTAGE;
constexpr int F_OFF_RY = F_OFF_HS + 2 * F_HS_BYTES;              // residual ring; in pass 2: staging
constexpr int F_OFF_Y32 = F_OFF_RY;                              //   2 x 16 KB fp32 [128][128 B], 128B swizzle
constexpr int F_OFF_Y16 = F_OFF_RY + 2 * F_R_BYTES;              //   2 x 8 KB bf16 [128][64 B], 64B swizzle
constexpr int F_OFF_BAR = F_OFF_RY + F_R_SLOTS * F_R_BYTES;
constexpr int F_SMEM = F_OFF_BAR + 512 + 1024;
constexpr int F_THREADS = 512;
constexpr uint32_t F_TM_OUT = 0;                  // 2 x 192 columns
constexpr uint32_t F_TM_H = 384;                  // 2 x 64 columns

struct MlpArgs {
  int M, n_tiles;
  const uint16_t* state_b;
};

__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint64_t mul_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// gelu of two values; returns them packed as a 16-bit pair of format FMT (lo = first)
template <int FMT>
__device__ __forceinline__ uint32_t gelu2_16(float x0, float x1) {
  const uint64_t x = pack_f32x2(x0, x1);
  float q0, q1;
  unpack_f32x2(mul_f32x2(x, x), q0, q1);
  // beyond |x| = 6 the polynomial is frozen: u = 1.67 x there, tanh(u) = +-1 in fp32
  const uint64_t x2 = pack_f32x2(fminf(q0, 36.0f), fminf(q1, 36.0f));
  const uint64_t a0 = pack_f32x2(0.7974578142166138f, 0.7974578142166138f);
  const uint64_t a1 = pack_f32x2(0.03705103322863579f, 0.03705103322863579f);
  const uint64_t a2 = pack_f32x2(-0.0003588674298953265f, -0.0003588674298953265f);
  const uint64_t half = pack_f32x2(0.5f, 0.5f);
  uint64_t p = fma_f32x2(a2, x2, a1);
  p = fma_f32x2(p, x2, a0);
  float u0, u1;
  unpack_f32x2(mul_f32x2(p, x), u0, u1);
  const uint64_t t = pack_f32x2(tanh_approx(u0), tanh_approx(u1));
  const uint64_t h = mul_f32x2(x, half);
  float y0, y1;
  unpack_f32x2(fma_f32x2(h, t, h), y0, y1);
  return pack16x2<FMT>(y0, y1);
}

// DBG = 1: clock64 trace of the MMA thread of CTA 0 (8 stamps per chunk: before / after each wait)
#ifdef MMPFN_DEBUG
__device__ long long g_mlp_trace[4096];
#define MLP_TRACE_BODY(slot) if (DBG && blockIdx.x == 0 && (slot) < 4096) g_mlp_trace[(slot)] = clock64();
#else
#define MLP_TRACE_BODY(slot)
#endif
#define MLP_TRACE(slot)                                                                    \
  do {                                                                                     \
    MLP_TRACE_BODY(slot)                                                                   \
  } while (0)

template <int DBG, int FMT>
__global__ void __launch_bounds__(F_THREADS, 1) tc_mlp_kernel(const __grid_constant__ CUtensorMap map_a,
                                                            const __grid_constant__ CUtensorMap map_w1,
                                                            const __grid_constant__ CUtensorMap map_w2,
                                                            const __grid_constant__ CUtensorMap map_r,
                                                            const __grid_constant__ CUtensorMap map_y,
                                                            const MlpArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + F_OFF_BAR);
  uint64_t* a_full = bars;             // activation tile landed
  uint64_t* a_empty = bars + 2;        // ... and all GEMM1 of its tile have completed
  uint64_t* w1_full = bars + 4;        // [2] W1 chunk landed
  uint64_t* w1_empty = bars + 6;       // [2] ... and GEMM1 of its chunk has completed
  uint64_t* h_full = bars + 8;         // [2] hidden chunk accumulator complete in TMEM
  uint64_t* h_free = bars + 10;        // [2] ... and read out by the GELU warps (one arrival per warp: 4)
  uint64_t* hs_full = bars + 12;       // [2] gelu(chunk) is in shared memory (one arrival per warp: 4)
  uint64_t* hs_empty = bars + 14;      // [2] ... and GEMM2 has consumed it
  uint64_t* out_full = bars + 16;      // [2] output accumulator of a tile complete
  uint64_t* out_empty = bars + 18;     // [2] ... and drained by the epilogue (one arrival per warp: 4)
  uint64_t* w2_full = bars + 20;       // [2] W2 chunk landed
  uint64_t* w2_empty = bars + 22;      // [2] ... and GEMM2 of its chunk has completed
  uint64_t* r_full = bars + 24;        // [3] residual chunk landed
  uint64_t* r_empty = bars + 27;       // [3] ... and its slot may be refilled (one arrival per warp: 4)
  uint32_t* tmem_slot = (uint32_t*)(bars + 30);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // tiles of this CTA: blockIdx.x, blockIdx.x + gridDim.x, ...
  const int my_tiles = (p.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int G = my_tiles * F_NCH;      // chunks this CTA walks, flat over its tiles

  if (threadIdx.x == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_w1);
    prefetch_tmap(&map_w2);
    prefetch_tmap(&map_r);
    prefetch_tmap(&map_y);
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int s = 0; s < F_R_SLOTS; ++s) {
      mbar_init(&r_full[s], 1);
      mbar_init(&r_empty[s], 4);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&w1_full[s], 1);
      mbar_init(&w1_empty[s], 1);
      mbar_init(&w2_full[s], 1);
      mbar_init(&w2_empty[s], 1);
      mbar_init(&h_full[s], 1);
      mbar_init(&h_free[s], 4);
      mbar_init(&hs_full[s], 4);
      mbar_init(&hs_empty[s], 1);
      mbar_init(&out_full[s], 1);
      mbar_init(&out_empty[s], 4);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      auto load_a = [&](int i) {
        const int tile = (int)blockIdx.x + i * (int)gridDim.x;
        mbar_wait(a_empty, (i & 1) ^ 1);
        mbar_expect_tx(a_full, F_A_BYTES);
        uint8_t* a_dst = smem + F_OFF_A;
#pragma unroll
        for (int kb = 0; kb < 3; ++kb) tma_load_2d(a_dst + kb * (F_BM * 128), &map_a, a_full, kb * 64, tile * F_BM);
      };
      // the activation buffer is single: the tile after next is pulled into L2 early so that the
      // reload between the last GEMM1 of a tile and the first of the next one is an L2 hit
      auto prefetch_a = [&](int i) {
        const long long m0 = ((long long)blockIdx.x + (long long)i * gridDim.x) * F_BM;
        const long long rows = p.M - m0 < F_BM ? p.M - m0 : F_BM;
        if (rows > 0) l2_prefetch(p.state_b + m0 * kE, (uint32_t)(rows * kE * 2));
      };
      // W1 and W2 chunks travel on separate 2-slot rings: the W1 slot of chunk g is free as soon as
      // GEMM1(g) has completed (before the GELU of the chunk), the W2 slot once GEMM2(g) has, so both
      // loads of chunk g+2 have two chunk periods to land.  (One shared stage held until GEMM2(g)
      // left GEMM1(g+2) a single period: the TMA round trip sat on the critical path.)
      auto load_w1 = [&](int g) {
        const int ws = g & 1, c = g % F_NCH;
        mbar_wait(&w1_empty[ws], ((g >> 1) & 1) ^ 1);
        mbar_expect_tx(&w1_full[ws], F_W1_BYTES);
        uint8_t* w_dst = smem + F_OFF_W + ws * F_WSTAGE;
#pragma unroll
        for (int kb = 0; kb < 3; ++kb) tma_load_2d(w_dst + kb * (F_CH * 128), &map_w1, &w1_full[ws], kb * 64, c * F_CH);
      };
      auto load_w2 = [&](int g) {
        const int ws = g & 1, c = g % F_NCH;
        mbar_wait(&w2_empty[ws], ((g >> 1) & 1) ^ 1);
        mbar_expect_tx(&w2_full[ws], F_W2_BYTES);
        tma_load_2d(smem + F_OFF_W + ws * F_WSTAGE + F_W1_BYTES, &map_w2, &w2_full[ws], c * F_CH, 0);
      };
      if (my_tiles > 0) load_a(0);
      for (int g = 0; g < G; ++g) {
        const int i = g / F_NCH, c = g % F_NCH;
        if (c == 0 && i + 1 < my_tiles) prefetch_a(i + 1);
        load_w1(g);
        if (g > 0 && c != 0) load_w2(g - 1);
        // last chunk of a tile: every weight chunk of the tile is requested (its own W2 chunk one
        // iteration early) before this thread blocks on the tile's last GEMM1 to reload the A buffer
        if (c == F_NCH - 1) {
          load_w2(g);
          if (i + 1 < my_tiles) load_a(i + 1);
        }
      }
    }
  } else if (warp == 1) {
    // ---- GEMM1 issue: hidden chunk g = A(tile) W1c^T into TMEM H[g & 1] ----
    // GEMM1 and GEMM2 are issued by two different threads (warps 1 and 3): every hand-off of this
    // kernel costs the issuing thread ~200 cycles even when the barrier is already complete, and one
    // thread walking all four per chunk (w1_full, h_free, w2_full, hs_full) was the critical path
    // (~1900 cycles per chunk against 768 of tensor work).  The two streams only meet through
    // mbarriers (h_full/h_free via the GELU warps), so no ordering between the threads is needed.
    if (elect_one()) {
      constexpr uint32_t idesc1 = make_idesc_fmt<FMT>(F_BM, F_CH);
      const uint32_t sbase = smem_u32(smem);
      for (int g = 0; g < G; ++g) {
        const int i = g / F_NCH, c = g % F_NCH;
        const int hb = g & 1;
        MLP_TRACE(g * 8 + 0);
        if (c == 0) mbar_wait(a_full, i & 1);
        mbar_wait2(&w1_full[hb], (g >> 1) & 1, &h_free[hb], ((g >> 1) & 1) ^ 1);
        MLP_TRACE(g * 8 + 1);
        MLP_TRACE(g * 8 + 2);
        tc_fence_after();
        const uint32_t a_addr = sbase + F_OFF_A;
        const uint32_t w_addr = sbase + F_OFF_W + hb * F_WSTAGE;
#pragma unroll
        for (int kb = 0; kb < 3; ++kb) {
          const uint64_t adesc = make_desc(a_addr + kb * (F_BM * 128), 1024, kSw128);
          const uint64_t bdesc = make_desc(w_addr + kb * (F_CH * 128), 1024, kSw128);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem + F_TM_H + hb * F_CH, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc1,
                      (kb | k) != 0);
        }
        umma_commit(&w1_empty[hb]);
        umma_commit(&h_full[hb]);
        MLP_TRACE(g * 8 + 3);
        if (c == F_NCH - 1) umma_commit(a_empty);          // last GEMM1 of the tile: A buffer is free
      }
    }
  } else if (warp == 3) {
    // ---- GEMM2 issue: OUT[tile & 1] (+)= gelu(chunk g) W2c^T ----
    if (elect_one()) {
      constexpr uint32_t idesc2 = make_idesc_fmt<FMT>(F_BM, kE);
      const uint32_t sbase = smem_u32(smem);
      for (int g = 0; g < G; ++g) {
        const int i = g / F_NCH, c = g % F_NCH;
        const int hb = g & 1, ob = i & 1;
        MLP_TRACE(g * 8 + 4);
        if (c == 0) mbar_wait(&out_empty[ob], ((i >> 1) & 1) ^ 1);
        mbar_wait2(&w2_full[hb], (g >> 1) & 1, &hs_full[hb], (g >> 1) & 1);
        MLP_TRACE(g * 8 + 5);
        MLP_TRACE(g * 8 + 6);
        tc_fence_after();
        const uint64_t adesc = make_desc(sbase + F_OFF_HS + hb * F_HS_BYTES, 1024, kSw128);
        const uint64_t bdesc = make_desc(sbase + F_OFF_W + hb * F_WSTAGE + F_W1_BYTES, 1024, kSw128);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16(tmem + F_TM_OUT + ob * kE, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc2, (c | k) != 0);
        umma_commit(&w2_empty[hb]);
        umma_commit(&hs_empty[hb]);
        if (c == F_NCH - 1) umma_commit(&out_full[ob]);
        MLP_TRACE(g * 8 + 7);
      }
    }
  } else if (warp == 2) {
    // ---- residual producer: chunk c of tile i -> ring slot (6 i + c) % 3 ----
    if (elect_one()) {
      for (int i = 0; i < my_tiles; ++i) {
        const int m0 = ((int)blockIdx.x + i * (int)gridDim.x) * F_BM;
        for (int c = 0; c < F_NRC; ++c) {
          const int q = i * F_NRC + c;
          const int slot = q % F_R_SLOTS;
          mbar_wait(&r_empty[slot], ((q / F_R_SLOTS) & 1) ^ 1);
          mbar_expect_tx(&r_full[slot], F_R_BYTES);
          tma_load_2d(smem + F_OFF_RY + slot * F_R_BYTES, &map_r, &r_full[slot], c * F_RC, m0);
        }
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ---- GELU warps: two groups of four; group = parity of the chunk, so that the fixed costs of a
    // chunk (barrier wake-up, TMEM load, proxy fence: ~700 cycles) of one group hide under the
    // arithmetic of the other.  Thread = token row, all 64 hidden columns of the chunk. ----
    const int grp = (warp - 4) >> 2, quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int hb = grp;
    const uint32_t trow = tmem + F_TM_H + hb * F_CH + ((uint32_t)(quarter * 32) << 16);
    const uint32_t dst = smem_u32(smem) + F_OFF_HS + hb * F_HS_BYTES + r * 128;
    const int rsw = r & 7;
    uint32_t v0[32], v1[32];
    for (int g = grp; g < G; g += 2) {
      const uint32_t ph = (g >> 1) & 1;
      mbar_wait(&h_full[hb], ph);
      tc_fence_after();
      tmem_ld32(trow, v0);
      tmem_ld32(trow + 32, v1);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive_warp(&h_free[hb]);
      uint32_t pk[32];
#pragma unroll
      for (int i = 0; i < 16; ++i) pk[i] = gelu2_16<FMT>(__uint_as_float(v0[2 * i]), __uint_as_float(v0[2 * i + 1]));
#pragma unroll
      for (int i = 0; i < 16; ++i) pk[16 + i] = gelu2_16<FMT>(__uint_as_float(v1[2 * i]), __uint_as_float(v1[2 * i + 1]));
      mbar_wait(&hs_empty[hb], ph ^ 1);          // GEMM2 of chunk g-2 has released this buffer
      // 64 hidden columns = the row's 128 B = eight 16-byte pieces, XOR-swizzled
#pragma unroll
      for (int q = 0; q < 8; ++q)
        st_shared_v4(dst + ((q ^ rsw) << 4), pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
      fence_proxy_async();
      mbar_arrive_warp(&hs_full[hb]);
    }
  } else if (warp >= 12) {
    // ---- epilogue warps: state = LN(state + acc), fp32 state and bf16 shadow; thread = row ----
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int rsw = r & 7;
    const bool store_leader = warp == 12 && elect_one();
    const uint32_t sbase = smem_u32(smem);
    uint32_t v[32];
    for (int i = 0; i < my_tiles; ++i) {
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      const int ob = i & 1;
      const uint32_t trow = tmem + F_TM_OUT + ob * kE + ((uint32_t)(quarter * 32) << 16);
      mbar_wait(&out_full[ob], (i >> 1) & 1);
      tc_fence_after();
      // pass 1: add the residual chunk (16-byte piece j of row r sits at piece j ^ (r & 7)), keep the
      // sum in TMEM, accumulate the statistics.  The slots of chunks 0-2 go straight back to the
      // producer (chunks 3-5 of this tile); those of chunks 3-5 only after pass 2, which reuses them.
      LnRowStats stats;
#pragma unroll 1
      for (int c = 0; c < F_NRC; ++c) {
        const int q = i * F_NRC + c;
        const int slot = q % F_R_SLOTS;
        tmem_ld32(trow + c * 32, v);
        mbar_wait(&r_full[slot], (q / F_R_SLOTS) & 1);
        const uint32_t rrow = sbase + F_OFF_RY + slot * F_R_BYTES + r * 128;
        float4 rr[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) rr[k] = lds128(rrow + ((k ^ rsw) << 4));
        tmem_ld_wait();
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float a0 = __uint_as_float(v[4 * k]) + rr[k].x, a1 = __uint_as_float(v[4 * k + 1]) + rr[k].y,
                      a2 = __uint_as_float(v[4 * k + 2]) + rr[k].z, a3 = __uint_as_float(v[4 * k + 3]) + rr[k].w;
          v[4 * k] = __float_as_uint(a0); v[4 * k + 1] = __float_as_uint(a1);
          v[4 * k + 2] = __float_as_uint(a2); v[4 * k + 3] = __float_as_uint(a3);
        }
        tmem_st32(trow + c * 32, v);
        // The slot goes back to the producer only HERE, behind the store that consumed the residual values: an arrival
        // right after the ld.shared instructions were issued does not wait for their data, and the producer's next TMA
        // load then overwrites the slot under loads still in flight (a few rows per launch read the wrong chunk when
        // other work delays the warp: profiles/r02_interleaved_test_layers_experiment.txt).
        if (c < F_R_SLOTS) mbar_arrive_warp(&r_empty[slot]);
        stats.add32(v, c);
      }
      tmem_st_wait();
      float mean, rstd;
      stats.finish(mean, rstd);
      epi_bar();      // every row of the ring has been read: its memory becomes the staging area
      // pass 2: chunk c goes through staging slot c & 1 and out by TMA (rows past M are clipped by
      // the tensor maps).  One named barrier per chunk: before it the store leader has waited until
      // the store of chunk c-1 has read its slot, so after it that slot may take chunk c+1.
#pragma unroll 1
      for (int c = 0; c < F_NRC; ++c) {
        tmem_ld32(trow + c * 32, v);
        tmem_ld_wait();
        const uint32_t y32 = sbase + F_OFF_Y32 + (c & 1) * F_R_BYTES + r * 128;
        const uint32_t y16 = sbase + F_OFF_Y16 + (c & 1) * (F_R_BYTES / 2) + r * 64;
        float y[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) y[k] = (__uint_as_float(v[k]) - mean) * rstd;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          st_shared_v4(y32 + ((k ^ rsw) << 4), __float_as_uint(y[4 * k]), __float_as_uint(y[4 * k + 1]),
                       __float_as_uint(y[4 * k + 2]), __float_as_uint(y[4 * k + 3]));
#pragma unroll
        for (int k = 0; k < 4; ++k)
          st_shared_v4(y16 + ((k ^ ((r >> 1) & 3)) << 4), pack16x2<FMT>(y[8 * k], y[8 * k + 1]),
                       pack16x2<FMT>(y[8 * k + 2], y[8 * k + 3]), pack16x2<FMT>(y[8 * k + 4], y[8 * k + 5]),
                       pack16x2<FMT>(y[8 * k + 6], y[8 * k + 7]));
        fence_proxy_async();
        if (store_leader) bulk_wait_read0();
        epi_bar();
        if (store_leader) {
          tma_store_2d(&map_r, smem + F_OFF_Y32 + (c & 1) * F_R_BYTES, c * F_RC, tile * F_BM);
          tma_store_2d(&map_y, smem + F_OFF_Y16 + (c & 1) * (F_R_BYTES / 2), c * F_RC, tile * F_BM);
          bulk_commit();
        }
      }
      tc_fence_before();
      mbar_arrive_warp(&out_empty[ob]);
      // the staging memory goes back to the residual producer once the last stores have read it
      if (store_leader) bulk_wait_read0();
      epi_bar();
#pragma unroll
      for (int s = 0; s < F_R_SLOTS; ++s) mbar_arrive_warp(&r_empty[s]);
    }
    if (store_leader) bulk_wait0();       // shared memory must outlive the last bulk stores
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

}  // namespace

int launch_tc_mlp(const TcMlp& p, cudaStream_t st, int fmt) {
  if (p.M <= 0) return MMPFN_OK;
  if (!p.state_b || !p.w1 || !p.w2 || !p.resid_f32 || !p.state_b_out) { set_error("tc_mlp: null argument"); return MMPFN_EINVAL; }
  CUtensorMap ma, mw1, mw2, mr, my;
  {
    const cuuint64_t dims[2] = {(cuuint64_t)kE, (cuuint64_t)p.M};
    const cuuint64_t strides[1] = {(cuuint64_t)kE * 4};
    const cuuint32_t box[2] = {F_RC, F_BM};
    MMPFN_TRY(encode_map(&mr, p.resid_f32, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_DATA_TYPE_FLOAT32));
  }
  {
    const cuuint64_t dims[2] = {(cuuint64_t)kE, (cuuint64_t)p.M};
    const cuuint64_t strides[1] = {(cuuint64_t)kE * 2};
    const cuuint32_t box[2] = {F_RC, F_BM};
    MMPFN_TRY(encode_map(&my, p.state_b_out, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B));
  }
  {
    const cuuint64_t dims[2] = {(cuuint64_t)kE, (cuuint64_t)p.M};
    const cuuint64_t strides[1] = {(cuuint64_t)kE * 2};
    const cuuint32_t box[2] = {64, F_BM};
    MMPFN_TRY(encode_map(&ma, p.state_b, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  {
    const cuuint64_t dims[2] = {(cuuint64_t)kE, (cuuint64_t)kHid};
    const cuuint64_t strides[1] = {(cuuint64_t)kE * 2};
    const cuuint32_t box[2] = {64, F_CH};
    MMPFN_TRY(encode_map(&mw1, p.w1, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  {
    const cuuint64_t dims[2] = {(cuuint64_t)kHid, (cuuint64_t)kE};
    const cuuint64_t strides[1] = {(cuuint64_t)kHid * 2};
    const cuuint32_t box[2] = {F_CH, kE};
    MMPFN_TRY(encode_map(&mw2, p.w2, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  const int n_sm = device_sm_count();
  MlpArgs a{};
  a.M = p.M;
  a.n_tiles = (p.M + F_BM - 1) / F_BM;
  a.state_b = p.state_b;
  const int grid = a.n_tiles < n_sm ? a.n_tiles : n_sm;
  if (fmt == FMT_F16) {
    MMPFN_OPT_IN_SMEM((tc_mlp_kernel<0, FMT_F16>), F_SMEM);
    tc_mlp_kernel<0, FMT_F16><<<grid, F_THREADS, F_SMEM, st>>>(ma, mw1, mw2, mr, my, a);
    return count_launch();
  }
  MMPFN_OPT_IN_SMEM((tc_mlp_kernel<0, FMT_BF16>), F_SMEM);
#ifdef MMPFN_DEBUG
  MMPFN_OPT_IN_SMEM((tc_mlp_kernel<1, FMT_BF16>), F_SMEM);
  static int dbg = -1;
  if (dbg < 0) {
    const char* e = getenv("MMPFN_MLP_DBG");          // tuning build only: clock64 trace variant
    dbg = e ? atoi(e) : 0;
  }
  if (dbg) {
    tc_mlp_kernel<1, FMT_BF16><<<grid, F_THREADS, F_SMEM, st>>>(ma, mw1, mw2, mr, my, a);
    return count_launch();
  }
#endif
  tc_mlp_kernel<0, FMT_BF16><<<grid, F_THREADS, F_SMEM, st>>>(ma, mw1, mw2, mr, my, a);
  return count_launch();
}

}  // namespace mmpfn

#ifdef MMPFN_DEBUG
// tuning build only: copy the clock64 trace of CTA 0's MMA thread to the host (MMPFN_MLP_DBG=1 runs)
extern "C" int mmpfn_debug_mlp_trace(long long* host_out, int n) {
  if (n > 4096) n = 4096;
  return cudaMemcpyFromSymbol(host_out, mmpfn::g_mlp_trace, sizeof(long long) * n) == cudaSuccess ? 0 : MMPFN_ECUDA;
}
#endif
