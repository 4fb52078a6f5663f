// kernels_tc.cu — the tensor-core path (bf16 operands, fp32 accumulation) written directly against
// sm_100a: TMA (cp.async.bulk.tensor) stages 128B/64B-swizzled tiles in shared memory, a single
// elected thread issues tcgen05.mma with accumulators in TMEM, epilogue / softmax warps read them
// back with tcgen05.ld.
//
//   tc_gemm_kernel       out = epi(A W^T), 128 x 192 x 64 tiles.  Serves the QKV / output
//                        projections (multi_head_attention.py:430, :513-517) and the MLP
//                        (mlp.py:93-104).  Epilogues: bf16 store, exact GELU, residual + LayerNorm
//                        (layer.py:437-455), and the item-attention QKV scatter.
//   (the item attention itself: kernels_attn.cu; the fused MLP sublayer: kernels_mlp.cu)
//
// Every mbarrier wait is bounded (trap after ~2 s) so that a protocol bug cannot hang the GPU.
#include "tc_common.cuh"

namespace mmpfn {
namespace {

// ---------------------------------------------------------------------------------------------
// GEMM
// ---------------------------------------------------------------------------------------------
constexpr int G_BM = 128, G_BN = 192, G_BK = 64, G_STAGES = 2;
constexpr int G_A_BYTES = G_BM * G_BK * 2;           // 16 KB
constexpr int G_B_BYTES = G_BN * G_BK * 2;           // 24 KB
constexpr int G_STAGE_BYTES = G_A_BYTES + G_B_BYTES;
constexpr int G_SMEM = G_STAGES * G_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
constexpr int G_TMEM_COLS = 256;
constexpr int G_THREADS = 192;

struct GemmArgs {
  int M, N, K;
  int items, B, S, T, tiles_s;
  uint16_t* out_bf16;
  float* resid;
  uint16_t* ln_bf16;
  uint16_t *q_out, *k_out, *vt_out, *k0_out, *vt0_out;
  int S_pad;
  const float* bias;
  float* out_f32;
};

template <int EPI>
__global__ void __launch_bounds__(G_THREADS) tc_gemm_kernel(const __grid_constant__ CUtensorMap map_a,
                                                            const __grid_constant__ CUtensorMap map_w,
                                                            const GemmArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + G_STAGES * G_STAGE_BYTES);
  uint64_t* empty = full + G_STAGES;
  uint64_t* acc_full = empty + G_STAGES;
  uint32_t* tmem_slot = (uint32_t*)(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KB = p.K / G_BK;
  const int n_tiles = p.N / G_BN;
  const int n0 = (blockIdx.x % n_tiles) * G_BN;
  const int m_tile = blockIdx.x / n_tiles;

  // tile coordinates
  int m0 = 0, tb = 0, tt = 0, s0 = 0;
  if (p.items) {
    const int mt = m_tile;
    const int per_b = p.T * p.tiles_s;
    tb = mt / per_b;
    const int r = mt % per_b;
    tt = r / p.tiles_s;
    s0 = (r % p.tiles_s) * G_BM;
  } else {
    m0 = m_tile * G_BM;
  }

  if (threadIdx.x == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_w);
    for (int s = 0; s < G_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, G_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      for (int kb = 0; kb < KB; ++kb) {
        const int s = kb % G_STAGES;
        mbar_wait(&empty[s], ((kb / G_STAGES) & 1) ^ 1);
        uint8_t* a_dst = smem + s * G_STAGE_BYTES;
        uint8_t* b_dst = a_dst + G_A_BYTES;
        mbar_expect_tx(&full[s], G_STAGE_BYTES);
        if (p.items) tma_load_4d(a_dst, &map_a, &full[s], kb * G_BK, tt, s0, tb);
        else tma_load_2d(a_dst, &map_a, &full[s], kb * G_BK, m0);
        tma_load_2d(b_dst, &map_w, &full[s], kb * G_BK, n0);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc(G_BM, G_BN);
      for (int kb = 0; kb < KB; ++kb) {
        const int s = kb % G_STAGES;
        mbar_wait(&full[s], (kb / G_STAGES) & 1);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * G_STAGE_BYTES);
        const uint64_t adesc = make_desc(a_addr, 1024, kSw128);
        const uint64_t bdesc = make_desc(a_addr + G_A_BYTES, 1024, kSw128);
#pragma unroll
        for (int k = 0; k < G_BK / 16; ++k)
          umma_bf16(tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
        umma_commit(&empty[s]);
      }
      umma_commit(acc_full);
    }
  } else {
    // ---- epilogue: 4 warps, warp w owns TMEM lanes [32*(w%4), +32) = tile rows ----
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t trow = tmem + ((uint32_t)(quarter * 32) << 16);
    mbar_wait(acc_full, 0);
    tc_fence_after();
    uint32_t v[32];
    if (EPI == TC_EPI_BF16 || EPI == TC_EPI_GELU_BF16) {
      const long long m = (long long)m0 + r;
      const bool ok = m < p.M;
      uint16_t* dst = p.out_bf16 + m * p.N + n0;
#pragma unroll 1
      for (int c = 0; c < G_BN / 32; ++c) {
        tmem_ld32(trow + c * 32, v);
        tmem_ld_wait();
        if (ok) {
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float a = __uint_as_float(v[2 * i]), b = __uint_as_float(v[2 * i + 1]);
            if (EPI == TC_EPI_GELU_BF16) { a = gelu_exact(a); b = gelu_exact(b); }
            pk[i] = pack_bf16x2(a, b);
          }
          uint4* d4 = reinterpret_cast<uint4*>(dst + c * 32);
#pragma unroll
          for (int i = 0; i < 4; ++i) d4[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
        }
      }
    } else if (EPI == TC_EPI_GLU_PAIR_F32) {
      // nn.GLU of the MGM stem (transformer.py:38-41): adjacent columns are (value, gate); fp32 out [M][N/2]
      const long long m = (long long)m0 + r;
      const bool ok = m < p.M;
      float* dst = p.out_f32 + m * (p.N / 2) + n0 / 2;
      const float* bias = p.bias + n0;
#pragma unroll 1
      for (int c = 0; c < G_BN / 32; ++c) {
        tmem_ld32(trow + c * 32, v);
        tmem_ld_wait();
        if (ok) {
          float o[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float a = __uint_as_float(v[2 * i]) + __ldg(bias + c * 32 + 2 * i);
            const float g = __uint_as_float(v[2 * i + 1]) + __ldg(bias + c * 32 + 2 * i + 1);
            o[i] = a * (1.0f / (1.0f + __expf(-g)));
          }
          float4* d4 = reinterpret_cast<float4*>(dst + c * 16);
#pragma unroll
          for (int i = 0; i < 4; ++i) d4[i] = make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
        }
      }
    } else if (EPI == TC_EPI_RESID_LN) {
      // state = LN(state + acc): pass 1 adds the residual, keeps v in TMEM and accumulates the
      // statistics; pass 2 normalises and writes the fp32 state and its bf16 shadow.
      const long long m = (long long)m0 + r;
      const bool ok = m < p.M;
      float* res = p.resid + m * kE;
      LnRowStats stats;
#pragma unroll 1
      for (int c = 0; c < kE / 32; ++c) {
        tmem_ld32(trow + c * 32, v);
        tmem_ld_wait();
        if (ok) {
          const float4* r4 = reinterpret_cast<const float4*>(res + c * 32);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 rr = r4[i];
            const float a0 = __uint_as_float(v[4 * i]) + rr.x, a1 = __uint_as_float(v[4 * i + 1]) + rr.y,
                        a2 = __uint_as_float(v[4 * i + 2]) + rr.z, a3 = __uint_as_float(v[4 * i + 3]) + rr.w;
            v[4 * i] = __float_as_uint(a0); v[4 * i + 1] = __float_as_uint(a1);
            v[4 * i + 2] = __float_as_uint(a2); v[4 * i + 3] = __float_as_uint(a3);
          }
          stats.add32(v, c);
        }
        tmem_st32(trow + c * 32, v);
      }
      tmem_st_wait();
      float mean, rstd;
      stats.finish(mean, rstd);
      uint16_t* lnb = p.ln_bf16 + m * kE;
#pragma unroll 1
      for (int c = 0; c < kE / 32; ++c) {
        tmem_ld32(trow + c * 32, v);
        tmem_ld_wait();
        if (ok) {
          float y[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) y[i] = (__uint_as_float(v[i]) - mean) * rstd;
          float4* o4 = reinterpret_cast<float4*>(res + c * 32);
#pragma unroll
          for (int i = 0; i < 8; ++i) o4[i] = make_float4(y[4 * i], y[4 * i + 1], y[4 * i + 2], y[4 * i + 3]);
          uint4* b4 = reinterpret_cast<uint4*>(lnb + c * 32);
#pragma unroll
          for (int i = 0; i < 4; ++i)
            b4[i] = make_uint4(pack_bf16x2(y[8 * i], y[8 * i + 1]), pack_bf16x2(y[8 * i + 2], y[8 * i + 3]),
                               pack_bf16x2(y[8 * i + 4], y[8 * i + 5]), pack_bf16x2(y[8 * i + 6], y[8 * i + 7]));
        }
      }
    } else {  // TC_EPI_QKV_ITEMS: n-tile j in {q,k,v}; 32-column chunk c = head
      const int s = s0 + r;
      const bool ok = s < p.S;
      const int j = blockIdx.x % n_tiles;
      const long long bt = (long long)tb * p.T + tt;
#pragma unroll 1
      for (int h = 0; h < kH; ++h) {
        tmem_ld32(trow + h * 32, v);
        tmem_ld_wait();
        if (!ok) continue;
        const long long plane = bt * kH + h;
        if (j < 2) {
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) pk[i] = pack_bf16x2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
          uint16_t* dst = (j == 0 ? p.q_out : p.k_out) + (plane * p.S_pad + s) * kD;
          uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
          for (int i = 0; i < 4; ++i) d4[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
          if (j == 1 && h == 0 && p.k0_out) {
            uint4* c4 = reinterpret_cast<uint4*>(p.k0_out + (bt * p.S_pad + s) * kD);
#pragma unroll
            for (int i = 0; i < 4; ++i) c4[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
          }
        } else {
          // V is stored transposed ([d][s]) so that P V is a K-major x K-major MMA; consecutive
          // lanes hold consecutive s -> 64 B coalesced per d
          uint16_t* dst = p.vt_out + plane * kD * p.S_pad + s;
          uint16_t* dst0 = (h == 0 && p.vt0_out) ? p.vt0_out + bt * kD * p.S_pad + s : nullptr;
#pragma unroll
          for (int d = 0; d < kD; ++d) {
            __nv_bfloat16 bv = __float2bfloat16_rn(__uint_as_float(v[d]));
            const uint16_t bits = *reinterpret_cast<uint16_t*>(&bv);
            dst[(long long)d * p.S_pad] = bits;
            if (dst0) dst0[(long long)d * p.S_pad] = bits;
          }
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, G_TMEM_COLS);
  }
}

template <int EPI>
int launch_gemm_t(const CUtensorMap& ma, const CUtensorMap& mw, const GemmArgs& a, dim3 grid, cudaStream_t st) {
  MMPFN_OPT_IN_SMEM(tc_gemm_kernel<EPI>, G_SMEM);
  tc_gemm_kernel<EPI><<<grid, G_THREADS, G_SMEM, st>>>(ma, mw, a);
  return count_launch();
}

}  // namespace

int launch_tc_gemm(const TcGemm& p, cudaStream_t st) {
  if (p.K % G_BK != 0 || p.N % G_BN != 0) {
    set_error("tc_gemm: N=%d must be a multiple of %d and K=%d of %d", p.N, G_BN, p.K, G_BK);
    return MMPFN_EUNSUPPORTED;
  }
  if (p.epi == TC_EPI_RESID_LN && p.N != kE) { set_error("tc_gemm: LN epilogue needs N=%d", kE); return MMPFN_EINVAL; }
  GemmArgs a{};
  a.M = p.M; a.N = p.N; a.K = p.K; a.items = p.items; a.B = p.B; a.S = p.S; a.T = p.T;
  a.out_bf16 = p.out_bf16; a.resid = p.resid_f32; a.ln_bf16 = p.ln_bf16;
  a.q_out = p.q_out; a.k_out = p.k_out; a.vt_out = p.vt_out; a.k0_out = p.k0_out; a.vt0_out = p.vt0_out;
  a.S_pad = p.S_pad;
  a.bias = p.bias; a.out_f32 = p.out_f32;
  if (p.epi == TC_EPI_GLU_PAIR_F32 && (!p.bias || !p.out_f32)) { set_error("tc_gemm: GLU epilogue needs bias and fp32 output"); return MMPFN_EINVAL; }
  CUtensorMap ma, mw;
  dim3 grid;
  if (p.items) {
    if (p.epi != TC_EPI_QKV_ITEMS) { set_error("tc_gemm: item tiles need the QKV epilogue"); return MMPFN_EINVAL; }
    a.tiles_s = (p.S + G_BM - 1) / G_BM;
    const cuuint64_t dims[4] = {(cuuint64_t)p.K, (cuuint64_t)p.T, (cuuint64_t)p.S, (cuuint64_t)p.B};
    const cuuint64_t strides[3] = {(cuuint64_t)p.K * 2, (cuuint64_t)p.T * p.K * 2, (cuuint64_t)p.S * p.T * p.K * 2};
    const cuuint32_t box[4] = {G_BK, 1, G_BM, 1};
    MMPFN_TRY(encode_map(&ma, p.A, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
    grid = dim3((unsigned)(p.B * p.T * a.tiles_s) * (p.N / G_BN));
  } else {
    if (p.M <= 0) return MMPFN_OK;
    const cuuint64_t dims[2] = {(cuuint64_t)p.K, (cuuint64_t)p.M};
    const cuuint64_t strides[1] = {(cuuint64_t)p.K * 2};
    const cuuint32_t box[2] = {G_BK, G_BM};
    MMPFN_TRY(encode_map(&ma, p.A, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
    grid = dim3((unsigned)((p.M + G_BM - 1) / G_BM) * (p.N / G_BN));
  }
  {
    const cuuint64_t dims[2] = {(cuuint64_t)p.K, (cuuint64_t)p.N};
    const cuuint64_t strides[1] = {(cuuint64_t)p.K * 2};
    const cuuint32_t box[2] = {G_BK, G_BN};
    MMPFN_TRY(encode_map(&mw, p.W, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B));
  }
  switch (p.epi) {
    case TC_EPI_BF16: return launch_gemm_t<TC_EPI_BF16>(ma, mw, a, grid, st);
    case TC_EPI_GELU_BF16: return launch_gemm_t<TC_EPI_GELU_BF16>(ma, mw, a, grid, st);
    case TC_EPI_RESID_LN: return launch_gemm_t<TC_EPI_RESID_LN>(ma, mw, a, grid, st);
    case TC_EPI_QKV_ITEMS: return launch_gemm_t<TC_EPI_QKV_ITEMS>(ma, mw, a, grid, st);
    case TC_EPI_GLU_PAIR_F32: return launch_gemm_t<TC_EPI_GLU_PAIR_F32>(ma, mw, a, grid, st);
  }
  set_error("tc_gemm: bad epilogue %d", p.epi);
  return MMPFN_EINVAL;
}

}  // namespace mmpfn
