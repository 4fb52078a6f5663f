// kernels_featfused.cu — QKV projection + attention between the features of a table row in ONE persistent kernel
// (layer.py:332-339 with multi_head_attention.py:430-434, 547-736 for the feature axis):
//
//     att[token][h*32 .. h*32+32) = softmax(q_h k_h^T / sqrt 32) v_h  over the T tokens of the token's table row,
//     (q | k | v) = x W_qkv^T,  x [M][192] bf16 (M = rows * T),  W_qkv [576][192] bf16
//
// The two-kernel form writes the [M][576] qkv block (1 152 B per token) and reads it back: three quarters of the
// HBM traffic of this sublayer's first half.  Here the block never leaves the SM:
//
//   * a CTA owns ONE PAIR OF HEADS: its 72 KB slice of W_qkv (q, k and v rows of the two heads) stays resident in
//     shared memory for the CTA's whole life (the K = 192 projections live on bytes in flight, not on MMA rate:
//     kernels_rowgemm.cu), and it walks tiles of G = 128 / T whole table rows (G T <= 128 tokens; T <= 64);
//   * tcgen05: one 128 x 192 x 192 MMA group per tile into TMEM (accumulators double buffered), A tile by TMA;
//   * four epilogue warps (thread = token) round the accumulators to bf16 into a shared-memory block of token rows
//     [q0 q1 k0 k1 v0 v1] (400-byte pitch: conflict-free ldmatrix), head 0's three column blocks first;
//   * two groups of eight attention warps, one per head of the pair, run the mma.sync core (feat_attn_core.cuh) per
//     (table row, 16-query tile) on that block, write the normalised output over the item's q block and send those
//     16 x 64 bytes to att[token][head * 32 ..] right away.  The block is DOUBLE BUFFERED and handed over per head
//     (full / empty barrier pair each): the attention — the long pole: ~1.4 us per tile on the legacy mma.sync path,
//     measured by knock-out builds — runs back to back while the load, MMA and conversion of the next tile and all
//     their barrier hand-offs (~1.3 us in series) happen beside it.
//
// HBM per token: 384 B in (the three head-pair CTAs of a tile read the same A tile within microseconds: one trip
// to HBM, two to L2) + 384 B out, against 384 + 1 152 + 1 152 + 384.
//
//   warp 0      TMA producer (W slice once, A tiles)
//   warp 1      MMA issue
//   warp 2      TMEM allocation
//   warps 4-7   epilogue: TMEM -> bf16 -> shared memory, thread = token
//   warps 8-15  attention + output store of the pair's first head, warps 16-23 of its second head
#include "feat_attn_core.cuh"
#include "tc_common.cuh"

namespace mmpfn {
namespace {

constexpr int U_BM = 128, U_BN = 192, U_K = 192;
constexpr int U_W_BYTES = U_BN * U_K * 2;            // 72 KB: 3 k-blocks [192][64] bf16, 128B swizzle
constexpr int U_A_BYTES = U_BM * U_K * 2;            // 48 KB: 3 k-blocks [128][64]
constexpr int U_ROW = 2 * 3 * kD * 2 + 16;           // 400 B per token: q0 q1 k0 k1 v0 v1 (64 B each) + 16 B pad
constexpr int U_QKV_BYTES = U_BM * U_ROW;            // 51 200 B per tile
constexpr int U_PAD_ROWS = 12;                       // the last table row's second 16-token tile may reach past the tile
constexpr int U_OFF_W = 0;
constexpr int U_OFF_A = U_W_BYTES;                   // one stage: its MMAs take ~0.3 us of a ~1.5 us tile period
constexpr int U_OFF_QKV = U_OFF_A + U_A_BYTES;       // two tiles back to back, then the pad rows (122 880: 1024-aligned)
constexpr int U_OFF_BAR = U_OFF_QKV + 2 * U_QKV_BYTES + U_PAD_ROWS * U_ROW;
constexpr int U_SMEM = U_OFF_BAR + 128 + 1024;
constexpr int U_THREADS = 768;
static_assert(U_SMEM <= 227 * 1024, "shared memory budget");
static_assert(U_ROW % 16 == 0 && U_ROW % 128 == 16, "ldmatrix rows: 16-byte aligned, 16 bytes apart modulo 128");

struct FusedArgs {
  uint16_t* att;            // [M][192] bf16
  long long M;              // tokens
  long long n_rows;         // table rows (M / T)
  int T, G;                 // tokens per table row, table rows per tile
  int m_tiles, ctas_per_pair;
};

template <int KT, int FMT>
__global__ void __launch_bounds__(U_THREADS, 1) feat_qkv_attn_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                    const __grid_constant__ CUtensorMap map_w,
                                                                    const FusedArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + U_OFF_BAR);
  uint64_t* w_full = bars;             // W slice landed (once)
  uint64_t* a_full = bars + 1;         // A tile landed
  uint64_t* a_empty = bars + 2;        // ... and its MMAs have completed
  uint64_t* acc_full = bars + 3;       // [2] accumulator complete in TMEM
  uint64_t* acc_empty = bars + 5;      // [2] ... and drained by the epilogue (one arrival per warp: 4)
  uint64_t* qkv_full = bars + 7;       // [buffer][head]: the head's q/k/v columns of a tile are in shared memory (4 arrivals)
  uint64_t* qkv_empty = bars + 11;     // [buffer][head]: ... and the head's attention warps are done with them (8 arrivals)
  uint32_t* tmem_slot = (uint32_t*)(bars + 15);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pair = (int)blockIdx.x % 3;               // heads 2 pair, 2 pair + 1
  const int cid = (int)blockIdx.x / 3;
  const int my_tiles = cid < p.m_tiles ? (p.m_tiles - cid + p.ctas_per_pair - 1) / p.ctas_per_pair : 0;
  const int tile_tokens = p.G * p.T;
  auto tile_of = [&](int i) { return cid + i * p.ctas_per_pair; };

  if (threadIdx.x == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_w);
    mbar_init(w_full, 1);
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&acc_full[s], 1);
      mbar_init(&acc_empty[s], 4);
    }
    for (int s = 0; s < 4; ++s) {
      mbar_init(&qkv_full[s], 4);
      mbar_init(&qkv_empty[s], 8);
    }
    fence_barrier_init();
  }
  // token rows past a tile (the other tile's first rows, or the pad rows) are only ever read as masked keys, but they
  // must be finite from the start (0 x NaN in P V)
  for (int i = threadIdx.x; i < (2 * U_QKV_BYTES + U_PAD_ROWS * U_ROW) / 16; i += U_THREADS)
    *reinterpret_cast<uint4*>(smem + U_OFF_QKV + i * 16) = make_uint4(0, 0, 0, 0);
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      // W slice rows [part * 64, part * 64 + 64) = part (q / k / v) of the two heads: rows part * 192 + pair * 64 .. of W_qkv
      mbar_expect_tx(w_full, U_W_BYTES);
#pragma unroll
      for (int kb = 0; kb < 3; ++kb)
#pragma unroll
        for (int part = 0; part < 3; ++part)
          tma_load_2d(smem + U_OFF_W + kb * (U_BN * 128) + part * (64 * 128), &map_w, w_full, kb * 64,
                      part * kE + pair * 64);
      for (int i = 0; i < my_tiles; ++i) {
        mbar_wait(a_empty, (i & 1) ^ 1);
        mbar_expect_tx(a_full, U_A_BYTES);
        uint8_t* dst = smem + U_OFF_A;
        const int tok0 = tile_of(i) * tile_tokens;     // (tokens past M are zero filled by the tensor map)
#pragma unroll
        for (int kb = 0; kb < 3; ++kb) tma_load_2d(dst + kb * (U_BM * 128), &map_a, a_full, kb * 64, tok0);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_fmt<FMT>(U_BM, U_BN);
      const uint32_t sbase = smem_u32(smem);
      mbar_wait(w_full, 0);
      for (int i = 0; i < my_tiles; ++i) {
        const int ab = i & 1;
        const uint32_t ph = (i >> 1) & 1;
        mbar_wait(a_full, i & 1);
        mbar_wait(&acc_empty[ab], ph ^ 1);
        tc_fence_after();
#pragma unroll
        for (int kb = 0; kb < 3; ++kb) {
          const uint64_t adesc = make_desc(sbase + U_OFF_A + kb * (U_BM * 128), 1024, kSw128);
          const uint64_t bdesc = make_desc(sbase + U_OFF_W + kb * (U_BN * 128), 1024, kSw128);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem + ab * U_BN, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
        }
        umma_commit(a_empty);
        umma_commit(&acc_full[ab]);
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ---- epilogue: accumulator row (token) -> bf16 -> its 384 bytes of the shared q/k/v block ----
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    uint32_t v[32];
    for (int i = 0; i < my_tiles; ++i) {
      const int ab = i & 1;
      const uint32_t row = smem_u32(smem) + U_OFF_QKV + ab * U_QKV_BYTES + r * U_ROW;
      const uint32_t trow = tmem + ab * U_BN + ((uint32_t)(quarter * 32) << 16);
      mbar_wait(&acc_full[ab], (i >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int h2 = 0; h2 < 2; ++h2) {
        mbar_wait(&qkv_empty[ab * 2 + h2], ((i >> 1) & 1) ^ 1);   // the head's attention warps are done with tile i - 2
#pragma unroll 1
        for (int part = 0; part < 3; ++part) {    // accumulator columns: q0 q1 k0 k1 v0 v1, 32 each
          const int c = part * 2 + h2;
          tmem_ld32(trow + c * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int k = 0; k < 4; ++k)
            st_shared_v4(row + c * 64 + k * 16, pack16x2<FMT>(__uint_as_float(v[8 * k]), __uint_as_float(v[8 * k + 1])),
                         pack16x2<FMT>(__uint_as_float(v[8 * k + 2]), __uint_as_float(v[8 * k + 3])),
                         pack16x2<FMT>(__uint_as_float(v[8 * k + 4]), __uint_as_float(v[8 * k + 5])),
                         pack16x2<FMT>(__uint_as_float(v[8 * k + 6]), __uint_as_float(v[8 * k + 7])));
        }
        mbar_arrive_warp(&qkv_full[ab * 2 + h2]);
      }
      tc_fence_before();
      mbar_arrive_warp(&acc_empty[ab]);
    }
  } else if (warp >= 8) {
    // ---- attention: group h2 = one head of the pair; items (table row g, 16-query tile mt); then the head's output
    // columns leave ----
    const int h2 = (warp - 8) >> 3, aw = (warp - 8) & 7;
    const int n_kt = (p.T + 15) >> 4;
    for (int i = 0; i < my_tiles; ++i) {
      const int qb = i & 1;
      const uint32_t qbase = smem_u32(smem) + U_OFF_QKV + qb * U_QKV_BYTES;
      const long long row0 = (long long)tile_of(i) * p.G;
      const int g_valid = (int)(p.n_rows - row0 < p.G ? p.n_rows - row0 : p.G);
      mbar_wait(&qkv_full[qb * 2 + h2], (i >> 1) & 1);
      const int n_items = g_valid * n_kt;
      uint8_t* dst = reinterpret_cast<uint8_t*>(p.att + (row0 * p.T) * kE + pair * 64 + h2 * 32);
      for (int item = aw; item < n_items; item += 8) {
        const int g = item / n_kt, mt = item % n_kt;
        const uint32_t rbase = qbase + g * p.T * U_ROW;
        feat_attn_item<KT, FMT>(rbase, U_ROW, h2 * 64, 128 + h2 * 64, 256 + h2 * 64, p.T, n_kt, mt, lane);
        // the item's 16 query rows x 64 B sit over its q block: they leave from this warp right away (two 16-byte
        // pieces per lane), no barrier across the group
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int idx = lane + 32 * k, t = mt * 16 + (idx >> 2), c = idx & 3;
          if (t < p.T) {
            uint4 o;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(o.x), "=r"(o.y), "=r"(o.z), "=r"(o.w)
                         : "r"(rbase + t * U_ROW + h2 * 64 + c * 16));
            *reinterpret_cast<uint4*>(dst + (long long)(g * p.T + t) * (kE * 2) + c * 16) = o;
          }
        }
      }
      mbar_arrive_warp(&qkv_empty[qb * 2 + h2]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

template <int KT, int FMT>
int launch_fused_t(const CUtensorMap& ma, const CUtensorMap& mw, const FusedArgs& a, int grid, cudaStream_t st) {
  MMPFN_OPT_IN_SMEM((feat_qkv_attn_kernel<KT, FMT>), U_SMEM);
  feat_qkv_attn_kernel<KT, FMT><<<grid, U_THREADS, U_SMEM, st>>>(ma, mw, a);
  return count_launch();
}

}  // namespace

bool feat_qkv_attn_supported(int T) { return T >= 2 && T <= 64; }

// x [M][192] bf16 (M = n_rows * T), w_qkv [576][192] bf16 -> att [M][192] bf16; all three fp16 with fmt = FMT_F16
int launch_feat_qkv_attn(const uint16_t* x, const uint16_t* w_qkv, long long M, int T, uint16_t* att, cudaStream_t st,
                         int fmt) {
  if (M <= 0) return MMPFN_OK;
  if (!feat_qkv_attn_supported(T) || M % T != 0 || M > 2147483647LL) {
    set_error("feat_qkv_attn: unsupported shape (M %lld, T %d)", M, T);
    return MMPFN_EUNSUPPORTED;
  }
  FusedArgs a{};
  a.att = att; a.M = M; a.T = T; a.n_rows = M / T;
  a.G = U_BM / T;
  const int n_kt = (T + 15) / 16;
  while (a.G > 1 && (a.G - 1) * T + 16 * n_kt > U_BM + U_PAD_ROWS) --a.G;     // the last row's key tiles stay inside the pad rows
  a.m_tiles = (int)((a.n_rows + a.G - 1) / a.G);
  CUtensorMap ma, mw;
  {
    const cuuint64_t dims[2] = {(cuuint64_t)U_K, (cuuint64_t)M};
    const cuuint64_t strides[1] = {(cuuint64_t)U_K * 2};
    const cuuint32_t box[2] = {64, U_BM};
    MMPFN_TRY(encode_map(&ma, x, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  {
    const cuuint64_t dims[2] = {(cuuint64_t)U_K, (cuuint64_t)(3 * kE)};
    const cuuint64_t strides[1] = {(cuuint64_t)U_K * 2};
    const cuuint32_t box[2] = {64, 64};
    MMPFN_TRY(encode_map(&mw, w_qkv, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  int per = device_sm_count() / 3;
  if (per > a.m_tiles) per = a.m_tiles;
  if (per < 1) per = 1;
  a.ctas_per_pair = per;
  if (fmt == FMT_F16)
    return T <= 32 ? launch_fused_t<2, FMT_F16>(ma, mw, a, per * 3, st) : launch_fused_t<4, FMT_F16>(ma, mw, a, per * 3, st);
  return T <= 32 ? launch_fused_t<2, FMT_BF16>(ma, mw, a, per * 3, st) : launch_fused_t<4, FMT_BF16>(ma, mw, a, per * 3, st);
}

}  // namespace mmpfn
