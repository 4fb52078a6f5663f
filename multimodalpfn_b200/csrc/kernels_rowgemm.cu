// kernels_rowgemm.cu — the K = 192 projections of a PerFeatureEncoderLayer as ONE persistent kernel:
//
//     out = epi(A W^T),  A [M][192] bf16,  W [N][192] bf16,  N in {192, 576}
//
// used for the fused QKV projections (multi_head_attention.py:430-434) and, with the residual +
// LayerNorm epilogue (layer.py:437-455), for both attention output projections
// (multi_head_attention.py:513-517).  These GEMMs are far below the tensor ridge (<= 410 FLOP/B):
// what they need is bytes in flight, not MMA issue rate.  So:
//
//   * one CTA per SM, persistent; a CTA owns ONE 192-wide n-tile and keeps its W tile (72 KB)
//     resident in shared memory for its whole life; it walks the 128-row m-tiles with a stride;
//   * the accumulator (192 fp32 columns) is double buffered in TMEM: the MMAs of tile i+1 run under
//     the epilogue of tile i (the A tile, 48 KB, is single buffered: its MMAs take ~0.6 us of a
//     ~7 us tile period, the next load starts as soon as they have completed);
//   * the fp32 residual of the LayerNorm epilogue is streamed by TMA through a 3-slot ring of
//     [128 rows x 32 floats] 128B-swizzled chunks, prefetched across tile boundaries, so that the
//     epilogue threads (thread = row, like the TMEM lanes) read their row from shared memory without
//     bank conflicts instead of issuing 16-byte global loads with a 768-byte stride and waiting for
//     each batch (the old epilogue: ~2x off the HBM roofline);
//   * results leave through shared memory too: the epilogue threads write their row of a 32- or
//     64-column chunk into a swizzled staging slot and one thread hands it to a TMA store (full
//     128-byte lines, rows past the end clipped by the tensor map) — a thread = row epilogue storing
//     straight to global memory issues 16-byte pieces with a 384..1152-byte stride, which costs one
//     L1 wavefront per piece and stalls every other user of the SM's load/store path.
//
//   warp 0   TMA producer (W once, A tiles, residual chunks)
//   warp 1   MMA issue
//   warp 2   TMEM allocation
//   warps 4-7 epilogue, thread = tile row
#include "tc_common.cuh"

namespace mmpfn {
namespace {

constexpr int R_BM = 128, R_BN = 192, R_K = 192;
constexpr int R_W_BYTES = R_BN * R_K * 2;            // 72 KB: 3 k-blocks [192][64] bf16, 128B swizzle
constexpr int R_A_BYTES = R_BM * R_K * 2;            // 48 KB: 3 k-blocks [128][64]
constexpr int R_RC = 32;                             // residual chunk: 32 fp32 columns = 128 B
constexpr int R_R_BYTES = R_BM * R_RC * 4;           // 16 KB
constexpr int R_R_SLOTS = 3;
constexpr int R_NCH = kE / R_RC;                     // 6 chunks per row
constexpr int R_Y32_BYTES = R_BM * 128;              // 16 KB staging slot: [128 rows][128 B], 128B swizzle
constexpr int R_Y16_BYTES = R_BM * 64;               // 8 KB staging slot: [128 rows][64 B], 64B swizzle
constexpr int R_OFF_W = 0;
constexpr int R_OFF_A = R_W_BYTES;
constexpr int R_OFF_R = R_OFF_A + R_A_BYTES;
constexpr int R_OFF_Y32 = R_OFF_R + R_R_SLOTS * R_R_BYTES;      // 2 slots
constexpr int R_OFF_Y16 = R_OFF_Y32 + 2 * R_Y32_BYTES;          // 2 slots
constexpr int R_OFF_BAR = R_OFF_Y16 + 2 * R_Y16_BYTES;
constexpr int R_SMEM = R_OFF_BAR + 256 + 1024;
constexpr int R_THREADS = 256;

struct RowGemmArgs {
  int M, n_tiles, m_tiles, ctas_per_n;
  int items, B, S, T, tiles_s;
  uint16_t* out_bf16;
  int ldo;
  float* resid;
  uint16_t* ln_bf16;
  uint16_t *q_out, *k_out, *vt_out, *k0_out, *vt0_out;
  int S_pad;
};

// destinations of the item-attention QKV scatter (TC_EPI_QKV_ITEMS): q/k planes [plane][S][32] (row pitch
// 64 B), v^T planes [plane][32][S], and the head-0 context copies (planes = (b, t))
struct alignas(64) ItemMaps {
  CUtensorMap q, k, vt, k0, vt0;
};

template <int EPI, int FMT>
__global__ void __launch_bounds__(R_THREADS, 1) tc_rowgemm_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                  const __grid_constant__ CUtensorMap map_w,
                                                                  const __grid_constant__ CUtensorMap map_r,
                                                                  const __grid_constant__ CUtensorMap map_y,
                                                                  const __grid_constant__ ItemMaps im,
                                                                  const RowGemmArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + R_OFF_BAR);
  uint64_t* w_full = bars;             // W tile landed (once)
  uint64_t* a_full = bars + 1;         // [kAStages] A tile landed
  uint64_t* a_empty = bars + 3;        // [kAStages] ... and its MMAs have completed
  // The LayerNorm variant is HBM bound at ~7 us per tile and needs the shared memory for the residual
  // ring: one A buffer.  The plain projections move a third of the bytes per tile: there the load of
  // tile i+1 must not wait for the MMAs of tile i, and the second A buffer takes the ring's place.
  constexpr int kAStages = EPI == TC_EPI_RESID_LN ? 1 : 2;
  static_assert(R_R_SLOTS * R_R_BYTES == R_A_BYTES, "the second A buffer aliases the residual ring");
  static_assert(kH * R_BM * 64 == 2 * R_Y32_BYTES + 2 * R_Y16_BYTES, "six staged heads fill the staging area");
  uint64_t* acc_full = bars + 5;       // [2] accumulator complete in TMEM
  uint64_t* acc_empty = bars + 7;      // [2] ... and drained by the epilogue (one arrival per warp: 4)
  uint64_t* r_full = bars + 9;         // [3] residual chunk landed
  uint64_t* r_empty = bars + 12;       // [3] ... and consumed (one arrival per warp: 4)
  uint32_t* tmem_slot = (uint32_t*)(bars + 15);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int jn = (int)blockIdx.x % p.n_tiles;          // this CTA's n-tile
  const int cid = (int)blockIdx.x / p.n_tiles;         // its position among the CTAs of that n-tile
  const int my_tiles = cid < p.m_tiles ? (p.m_tiles - cid + p.ctas_per_n - 1) / p.ctas_per_n : 0;

  if (threadIdx.x == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_w);
    if (EPI == TC_EPI_RESID_LN) prefetch_tmap(&map_r);
    if (EPI != TC_EPI_QKV_ITEMS) prefetch_tmap(&map_y);
    if (EPI == TC_EPI_QKV_ITEMS) {
      prefetch_tmap(&im.q);
      prefetch_tmap(&im.k);
      prefetch_tmap(&im.vt);
    }
    mbar_init(w_full, 1);
    for (int s = 0; s < kAStages; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&acc_full[s], 1);
      mbar_init(&acc_empty[s], 4);
    }
    for (int s = 0; s < R_R_SLOTS; ++s) {
      mbar_init(&r_full[s], 1);
      mbar_init(&r_empty[s], 4);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // m-tile index -> coordinates.  FLAT: rows m0 .. m0+127.  ITEMS: 128 rows s at fixed (b, t).
  auto tile_of = [&](int i) { return cid + i * p.ctas_per_n; };

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(w_full, R_W_BYTES);
#pragma unroll
      for (int kb = 0; kb < 3; ++kb) tma_load_2d(smem + R_OFF_W + kb * (R_BN * 128), &map_w, w_full, kb * 64, jn * R_BN);
      auto load_a = [&](int i) {
        const int mt = tile_of(i);
        const int as = i % kAStages;
        uint64_t* full = &a_full[as];
        mbar_wait(&a_empty[as], ((i / kAStages) & 1) ^ 1);
        mbar_expect_tx(full, R_A_BYTES);
        uint8_t* dst = smem + R_OFF_A + as * R_A_BYTES;
        if (p.items) {
          const int per_b = p.T * p.tiles_s;
          const int tb = mt / per_b, r = mt % per_b;
          const int tt = r / p.tiles_s, s0 = (r % p.tiles_s) * R_BM;
#pragma unroll
          for (int kb = 0; kb < 3; ++kb) tma_load_4d(dst + kb * (R_BM * 128), &map_a, full, kb * 64, tt, s0, tb);
        } else {
#pragma unroll
          for (int kb = 0; kb < 3; ++kb) tma_load_2d(dst + kb * (R_BM * 128), &map_a, full, kb * 64, mt * R_BM);
        }
      };
      if (my_tiles > 0) load_a(0);
      for (int i = 0; i < my_tiles; ++i) {
        if (i + 1 < my_tiles) load_a(i + 1);      // blocks until its buffer's previous MMAs have completed
        if (EPI == TC_EPI_RESID_LN) {
          const int m0 = tile_of(i) * R_BM;
          for (int c = 0; c < R_NCH; ++c) {
            const int q = i * R_NCH + c;
            const int slot = q % R_R_SLOTS;
            mbar_wait(&r_empty[slot], ((q / R_R_SLOTS) & 1) ^ 1);
            mbar_expect_tx(&r_full[slot], R_R_BYTES);
            tma_load_2d(smem + R_OFF_R + slot * R_R_BYTES, &map_r, &r_full[slot], c * R_RC, m0);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_fmt<FMT>(R_BM, R_BN);
      const uint32_t sbase = smem_u32(smem);
      mbar_wait(w_full, 0);
      for (int i = 0; i < my_tiles; ++i) {
        const int ab = i & 1;
        const uint32_t ph = (i >> 1) & 1;
        const int as = i % kAStages;
        mbar_wait(&a_full[as], (i / kAStages) & 1);
        mbar_wait(&acc_empty[ab], ph ^ 1);
        tc_fence_after();
        if (EPI == TC_EPI_QKV_ITEMS && jn == 2) {
          // V is wanted transposed ([d][s] planes): swap the operand roles — W_v rows (d) on the M side, the 128 table
          // rows (s) on the N side — so that the accumulator already IS V^T (lane = d, column = s) and the epilogue
          // writes whole 16-byte pieces of a d row instead of 2-byte elements.  192 d rows = two M = 128 MMAs (the
          // second one's upper 64 lanes multiply whatever follows the W tile in shared memory and are never read).
          constexpr uint32_t idesc_t = make_idesc_fmt<FMT>(128, R_BM);
#pragma unroll
          for (int half = 0; half < 2; ++half)
#pragma unroll
            for (int kb = 0; kb < 3; ++kb) {
              const uint64_t wdesc = make_desc(sbase + R_OFF_W + kb * (R_BN * 128) + half * (128 * 128), 1024, kSw128);
              const uint64_t sdesc = make_desc(sbase + R_OFF_A + as * R_A_BYTES + kb * (R_BM * 128), 1024, kSw128);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_bf16(tmem + ab * 256 + half * 128, wdesc + (uint64_t)(k * 2), sdesc + (uint64_t)(k * 2), idesc_t,
                          (kb | k) != 0);
            }
        } else {
#pragma unroll
          for (int kb = 0; kb < 3; ++kb) {
            const uint64_t adesc = make_desc(sbase + R_OFF_A + as * R_A_BYTES + kb * (R_BM * 128), 1024, kSw128);
            const uint64_t bdesc = make_desc(sbase + R_OFF_W + kb * (R_BN * 128), 1024, kSw128);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(tmem + ab * R_BN, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
          }
        }
        umma_commit(&a_empty[as]);
        umma_commit(&acc_full[ab]);
      }
    }
  } else if (warp >= 4) {
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int rsw = r & 7;
    const bool store_leader = warp == 4 && elect_one();
    uint32_t v[32];
    for (int i = 0; i < my_tiles; ++i) {
      const int mt = tile_of(i);
      const int ab = i & 1;
      const uint32_t trow = tmem + ab * R_BN + ((uint32_t)(quarter * 32) << 16);
      mbar_wait(&acc_full[ab], (i >> 1) & 1);
      tc_fence_after();
      if (EPI == TC_EPI_BF16) {
        // 64-column chunks (128 B of bf16 per row) through the two fp32-sized staging slots
#pragma unroll 1
        for (int c = 0; c < R_BN / 64; ++c) {
          const int ys = (i * (R_BN / 64) + c) & 1;   // three chunks per tile: alternate across tiles too
          const uint32_t yrow = smem_u32(smem) + R_OFF_Y32 + ys * R_Y32_BYTES + r * 128;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            tmem_ld32(trow + c * 64 + hh * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 4; ++k)
              st_shared_v4(yrow + (((hh * 4 + k) ^ rsw) << 4),
                           pack16x2<FMT>(__uint_as_float(v[8 * k]), __uint_as_float(v[8 * k + 1])),
                           pack16x2<FMT>(__uint_as_float(v[8 * k + 2]), __uint_as_float(v[8 * k + 3])),
                           pack16x2<FMT>(__uint_as_float(v[8 * k + 4]), __uint_as_float(v[8 * k + 5])),
                           pack16x2<FMT>(__uint_as_float(v[8 * k + 6]), __uint_as_float(v[8 * k + 7])));
          }
          fence_proxy_async();
          if (store_leader) bulk_wait_read0();        // the previous chunk's store has read the other slot
          epi_bar();
          if (store_leader) {
            tma_store_2d(&map_y, smem + R_OFF_Y32 + ys * R_Y32_BYTES, jn * R_BN + c * 64, mt * R_BM);
            bulk_commit();
          }
        }
      } else if (EPI == TC_EPI_RESID_LN) {
        // state = LN(state + acc).  Pass 1: add the residual chunk (shared memory, 128B swizzle: 16-byte
        // chunk j of row r sits at chunk j ^ (r & 7)), keep the sum in TMEM, accumulate the statistics.
        // Pass 2: normalise, write the fp32 state and its bf16 shadow.
        LnRowStats stats;
#pragma unroll 1
        for (int c = 0; c < R_NCH; ++c) {
          const int q = i * R_NCH + c;
          const int slot = q % R_R_SLOTS;
          tmem_ld32(trow + c * 32, v);
          mbar_wait(&r_full[slot], (q / R_R_SLOTS) & 1);
          const uint32_t rrow = smem_u32(smem) + R_OFF_R + slot * R_R_BYTES + r * 128;
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
          // (released behind the store that consumed the residual values: an arrival issued right after the ld.shared
          // instructions does not wait for their data — see kernels_mlp.cu)
          mbar_arrive_warp(&r_empty[slot]);
          stats.add32(v, c);
        }
        tmem_st_wait();
        float mean, rstd;
        stats.finish(mean, rstd);
        // pass 2: chunk c goes through staging slot c & 1 (fp32 and bf16 halves) and out by TMA.  One
        // named barrier per chunk: before it the store leader has waited until the store of chunk c-1
        // has read its slot, so after it every thread may overwrite that slot with chunk c+1.
#pragma unroll 1
        for (int c = 0; c < R_NCH; ++c) {
          tmem_ld32(trow + c * 32, v);
          tmem_ld_wait();
          const uint32_t y32 = smem_u32(smem) + R_OFF_Y32 + (c & 1) * R_Y32_BYTES + r * 128;
          const uint32_t y16 = smem_u32(smem) + R_OFF_Y16 + (c & 1) * R_Y16_BYTES + r * 64;
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
            tma_store_2d(&map_r, smem + R_OFF_Y32 + (c & 1) * R_Y32_BYTES, c * R_RC, mt * R_BM);
            tma_store_2d(&map_y, smem + R_OFF_Y16 + (c & 1) * R_Y16_BYTES, c * R_RC, mt * R_BM);
            bulk_commit();
          }
        }
      } else {  // TC_EPI_QKV_ITEMS: n-tile jn in {q,k,v}; 32-column chunk = head
        // Every head's [128 rows x 32] block goes through an 8 KB staging block and out by TMA: q and k
        // as [128][64 B] rows (64B swizzle) into their plane, v transposed ([32 d][128 s], two 128B-
        // swizzled 64-column blocks) so that P V is a K-major x K-major MMA.  Rows past S_pad (v: columns past
        // S) are clipped by the tensor maps.  Head 0 of k and v is stored a second time into the layer's context.
        const int per_b = p.T * p.tiles_s;
        const int tb = mt / per_b, rem = mt % per_b;
        const int tt = rem / p.tiles_s, s0 = (rem % p.tiles_s) * R_BM;
        const int bt = tb * p.T + tt;
        // all six heads are staged (6 x 8 KB = the whole staging area) before one fence, one barrier
        // and one group of stores per tile; the stores of the previous tile must have read it first
        if (store_leader) bulk_wait_read0();
        epi_bar();
        if (jn < 2) {
#pragma unroll 1
          for (int h = 0; h < kH; ++h) {
            const uint32_t slot = smem_u32(smem) + R_OFF_Y32 + h * (R_BM * 64);
            tmem_ld32(trow + h * 32, v);
            tmem_ld_wait();
            const uint32_t yrow = slot + r * 64;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              st_shared_v4(yrow + ((k ^ ((r >> 1) & 3)) << 4),
                           pack16x2<FMT>(__uint_as_float(v[8 * k]), __uint_as_float(v[8 * k + 1])),
                           pack16x2<FMT>(__uint_as_float(v[8 * k + 2]), __uint_as_float(v[8 * k + 3])),
                           pack16x2<FMT>(__uint_as_float(v[8 * k + 4]), __uint_as_float(v[8 * k + 5])),
                           pack16x2<FMT>(__uint_as_float(v[8 * k + 6]), __uint_as_float(v[8 * k + 7])));
          }
        } else {
          // the accumulators hold V^T: lanes of half 0 = d rows of heads 0-3 (warp = head), half 1 = heads 4, 5 (warps
          // 0, 1).  Thread = (head, d = lane): its 128 s values leave as 16 pieces of 16 B — 64-column block c / 2,
          // row d (128 B), piece ((c & 1) * 4 + k) ^ (d & 7)
#pragma unroll 1
          for (int half = 0; half < 2; ++half) {
            const int h = half * 4 + quarter;
            if (h >= kH) break;
            const uint32_t tv = tmem + ab * 256 + half * 128 + ((uint32_t)(quarter * 32) << 16);
            const uint32_t drow = smem_u32(smem) + R_OFF_Y32 + h * (R_BM * 64) + lane * 128;
#pragma unroll 1
            for (int c = 0; c < R_BM / 32; ++c) {
              tmem_ld32(tv + c * 32, v);
              tmem_ld_wait();
#pragma unroll
              for (int k = 0; k < 4; ++k)
                st_shared_v4(drow + (c >> 1) * (kD * 128) + ((((c & 1) * 4 + k) ^ (lane & 7)) << 4),
                             pack16x2<FMT>(__uint_as_float(v[8 * k]), __uint_as_float(v[8 * k + 1])),
                             pack16x2<FMT>(__uint_as_float(v[8 * k + 2]), __uint_as_float(v[8 * k + 3])),
                             pack16x2<FMT>(__uint_as_float(v[8 * k + 4]), __uint_as_float(v[8 * k + 5])),
                             pack16x2<FMT>(__uint_as_float(v[8 * k + 6]), __uint_as_float(v[8 * k + 7])));
            }
          }
        }
        fence_proxy_async();
        epi_bar();
        if (store_leader) {
#pragma unroll 1
          for (int h = 0; h < kH; ++h) {
            const uint8_t* slot = smem + R_OFF_Y32 + h * (R_BM * 64);
            const int plane = bt * kH + h;
            if (jn == 0) {
              tma_store_3d(&im.q, slot, 0, s0, plane);
            } else if (jn == 1) {
              tma_store_3d(&im.k, slot, 0, s0, plane);
              if (h == 0 && p.k0_out) tma_store_3d(&im.k0, slot, 0, s0, bt);
            } else {
#pragma unroll
              for (int kb = 0; kb < 2; ++kb) {
                if (s0 + kb * 64 < p.S) {
                  tma_store_3d(&im.vt, slot + kb * (kD * 128), s0 + kb * 64, 0, plane);
                  if (h == 0 && p.vt0_out) tma_store_3d(&im.vt0, slot + kb * (kD * 128), s0 + kb * 64, 0, bt);
                }
              }
            }
          }
          bulk_commit();
        }
      }
      tc_fence_before();
      mbar_arrive_warp(&acc_empty[ab]);
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

template <int EPI, int FMT>
int launch_rowgemm_t(const CUtensorMap& ma, const CUtensorMap& mw, const CUtensorMap& mr, const CUtensorMap& my,
                     const ItemMaps& im, const RowGemmArgs& a, int grid, cudaStream_t st) {
  MMPFN_OPT_IN_SMEM((tc_rowgemm_kernel<EPI, FMT>), R_SMEM);
  tc_rowgemm_kernel<EPI, FMT><<<grid, R_THREADS, R_SMEM, st>>>(ma, mw, mr, my, im, a);
  return count_launch();
}

}  // namespace

// Same contract as launch_tc_gemm for K = 192, N % 192 == 0 and the BF16 / RESID_LN / QKV_ITEMS epilogues; with
// fmt = FMT_F16 every 16-bit operand and output is fp16 instead of bf16 (the epilogue names keep saying "BF16").
int launch_tc_rowgemm(const TcGemm& p, cudaStream_t st, int fmt) {
  if (p.K != R_K || p.N % R_BN != 0 || p.N <= 0) {
    set_error("tc_rowgemm: needs K=%d and N a multiple of %d (got N=%d K=%d)", R_K, R_BN, p.N, p.K);
    return MMPFN_EUNSUPPORTED;
  }
  if (p.epi == TC_EPI_RESID_LN && p.N != kE) { set_error("tc_rowgemm: LN epilogue needs N=%d", kE); return MMPFN_EINVAL; }
  RowGemmArgs a{};
  a.M = p.M; a.items = p.items; a.B = p.B; a.S = p.S; a.T = p.T;
  a.out_bf16 = p.out_bf16; a.ldo = p.N; a.resid = p.resid_f32; a.ln_bf16 = p.ln_bf16;
  a.q_out = p.q_out; a.k_out = p.k_out; a.vt_out = p.vt_out; a.k0_out = p.k0_out; a.vt0_out = p.vt0_out;
  a.S_pad = p.S_pad;
  a.n_tiles = p.N / R_BN;
  CUtensorMap ma, mw, mr;
  if (p.items) {
    if (p.epi != TC_EPI_QKV_ITEMS) { set_error("tc_rowgemm: item tiles need the QKV epilogue"); return MMPFN_EINVAL; }
    a.tiles_s = (p.S + R_BM - 1) / R_BM;
    a.m_tiles = p.B * p.T * a.tiles_s;
    const cuuint64_t dims[4] = {(cuuint64_t)p.K, (cuuint64_t)p.T, (cuuint64_t)p.S, (cuuint64_t)p.B};
    const cuuint64_t strides[3] = {(cuuint64_t)p.K * 2, (cuuint64_t)p.T * p.K * 2, (cuuint64_t)p.S * p.T * p.K * 2};
    const cuuint32_t box[4] = {64, 1, R_BM, 1};
    MMPFN_TRY(encode_map(&ma, p.A, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  } else {
    if (p.M <= 0) return MMPFN_OK;
    a.m_tiles = (p.M + R_BM - 1) / R_BM;
    const cuuint64_t dims[2] = {(cuuint64_t)p.K, (cuuint64_t)p.M};
    const cuuint64_t strides[1] = {(cuuint64_t)p.K * 2};
    const cuuint32_t box[2] = {64, R_BM};
    MMPFN_TRY(encode_map(&ma, p.A, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  if (a.m_tiles <= 0) return MMPFN_OK;
  {
    const cuuint64_t dims[2] = {(cuuint64_t)p.K, (cuuint64_t)p.N};
    const cuuint64_t strides[1] = {(cuuint64_t)p.K * 2};
    const cuuint32_t box[2] = {64, R_BN};
    MMPFN_TRY(encode_map(&mw, p.W, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  mr = mw;
  CUtensorMap my = mw;
  if (p.epi == TC_EPI_BF16) {
    const cuuint64_t dims[2] = {(cuuint64_t)p.N, (cuuint64_t)p.M};
    const cuuint64_t strides[1] = {(cuuint64_t)p.N * 2};
    const cuuint32_t box[2] = {64, R_BM};
    MMPFN_TRY(encode_map(&my, p.out_bf16, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  if (p.epi == TC_EPI_RESID_LN) {
    {
      const cuuint64_t dims[2] = {(cuuint64_t)kE, (cuuint64_t)p.M};
      const cuuint64_t strides[1] = {(cuuint64_t)kE * 2};
      const cuuint32_t box[2] = {R_RC, R_BM};
      MMPFN_TRY(encode_map(&my, p.ln_bf16, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B));
    }
    const cuuint64_t dims[2] = {(cuuint64_t)kE, (cuuint64_t)p.M};
    const cuuint64_t strides[1] = {(cuuint64_t)kE * 4};
    const cuuint32_t box[2] = {R_RC, R_BM};
    MMPFN_TRY(encode_map(&mr, p.resid_f32, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_DATA_TYPE_FLOAT32));
  }
  ItemMaps im;
  im.q = im.k = im.vt = im.k0 = im.vt0 = mw;
  if (p.epi == TC_EPI_QKV_ITEMS) {
    const cuuint64_t planes = (cuuint64_t)p.B * p.T * kH, planes0 = (cuuint64_t)p.B * p.T;
    // rows S .. S_pad-1 of a plane receive zeros (their A rows are out of bounds = zero filled): the test
    // pass of the item attention stacks the heads of a column and runs over those rows too
    auto rows_map = [&](CUtensorMap* m, const void* base, cuuint64_t np) {      // [plane][S_pad][32]
      const cuuint64_t dims[3] = {(cuuint64_t)kD, (cuuint64_t)p.S_pad, np};
      const cuuint64_t strides[2] = {(cuuint64_t)kD * 2, (cuuint64_t)p.S_pad * kD * 2};
      const cuuint32_t box[3] = {kD, R_BM, 1};
      return encode_map(m, base, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
    };
    auto cols_map = [&](CUtensorMap* m, const void* base, cuuint64_t np) {      // [plane][32][S (pitch S_pad)]
      const cuuint64_t dims[3] = {(cuuint64_t)p.S, (cuuint64_t)kD, np};
      const cuuint64_t strides[2] = {(cuuint64_t)p.S_pad * 2, (cuuint64_t)p.S_pad * kD * 2};
      const cuuint32_t box[3] = {64, kD, 1};
      return encode_map(m, base, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
    };
    if (!p.q_out || (a.n_tiles == 3 && (!p.k_out || !p.vt_out))) { set_error("tc_rowgemm: null QKV destination"); return MMPFN_EINVAL; }
    MMPFN_TRY(rows_map(&im.q, p.q_out, planes));
    if (p.k_out) MMPFN_TRY(rows_map(&im.k, p.k_out, planes));
    if (p.vt_out) MMPFN_TRY(cols_map(&im.vt, p.vt_out, planes));
    if (p.k0_out) MMPFN_TRY(rows_map(&im.k0, p.k0_out, planes0));
    if (p.vt0_out) MMPFN_TRY(cols_map(&im.vt0, p.vt0_out, planes0));
  }
  const int n_sm = device_sm_count();
  int per_n = n_sm / a.n_tiles;
  if (per_n > a.m_tiles) per_n = a.m_tiles;
  if (per_n < 1) per_n = 1;
  a.ctas_per_n = per_n;
  const int grid = per_n * a.n_tiles;
  const bool f16 = fmt == FMT_F16;
  switch (p.epi) {
    case TC_EPI_BF16:
      return f16 ? launch_rowgemm_t<TC_EPI_BF16, FMT_F16>(ma, mw, mr, my, im, a, grid, st)
                 : launch_rowgemm_t<TC_EPI_BF16, FMT_BF16>(ma, mw, mr, my, im, a, grid, st);
    case TC_EPI_RESID_LN:
      return f16 ? launch_rowgemm_t<TC_EPI_RESID_LN, FMT_F16>(ma, mw, mr, my, im, a, grid, st)
                 : launch_rowgemm_t<TC_EPI_RESID_LN, FMT_BF16>(ma, mw, mr, my, im, a, grid, st);
    case TC_EPI_QKV_ITEMS:
      return f16 ? launch_rowgemm_t<TC_EPI_QKV_ITEMS, FMT_F16>(ma, mw, mr, my, im, a, grid, st)
                 : launch_rowgemm_t<TC_EPI_QKV_ITEMS, FMT_BF16>(ma, mw, mr, my, im, a, grid, st);
  }
  set_error("tc_rowgemm: unsupported epilogue %d", p.epi);
  return MMPFN_EINVAL;
}

}  // namespace mmpfn
