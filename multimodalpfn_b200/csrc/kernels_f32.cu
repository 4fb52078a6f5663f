// kernels_f32.cu — fp32 FFMA building blocks: the 1e-5 parity mode of the layers, and the
// (row-count-bound, small) stem / decoder GEMMs in both modes.
//
//   sgemm_kernel        out = epi(A W^T + bias)            reference: einsum / nn.Linear call sites
//                                                         (multi_head_attention.py:430,:513-517; mlp.py:93-104)
//   layernorm_kernel    y = LN(x + res) [* gamma + beta]   layer.py:40-64 (no affine), nn.LayerNorm in the stem
//   feat_attn_kernel    per-row attention across tokens    layer.py:332-339
//   item_attn_f32       flash attention across items       layer.py:341-379
#include "common.cuh"
#include "feat_attn_core.cuh"

namespace mmpfn {

// ---------------------------------------------------------------------------------------------
// SGEMM: C[M][N] = epi(A[M][K] * W[N][K]^T + bias).  128x64x16 tiles, 256 threads, 8x4 per thread.
// ---------------------------------------------------------------------------------------------
namespace {
constexpr int BM = 128, BN = 64, BK = 16;

template <int EPI>
__global__ void __launch_bounds__(256) sgemm_kernel(SgemmParams p) {
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  const int z = blockIdx.z;
  const float* __restrict__ A = p.A + z * p.a_batch;
  const float* __restrict__ W = p.W + z * p.w_batch;
  const float* __restrict__ bias = p.bias ? p.bias + z * p.bias_batch : nullptr;
  float* __restrict__ C = p.C + z * p.c_batch;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;

  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int lr = tid >> 2;         // 0..63
  const int lk = (tid & 3) * 4;    // 0,4,8,12
  for (int k0 = 0; k0 < p.K; k0 += BK) {
    float4 a0 = make_float4(0, 0, 0, 0), a1 = a0, b0 = a0;
    if (m0 + lr < p.M) a0 = *reinterpret_cast<const float4*>(A + (long long)(m0 + lr) * p.lda + k0 + lk);
    if (m0 + lr + 64 < p.M) a1 = *reinterpret_cast<const float4*>(A + (long long)(m0 + lr + 64) * p.lda + k0 + lk);
    if (n0 + lr < p.N) b0 = *reinterpret_cast<const float4*>(W + (long long)(n0 + lr) * p.ldw + k0 + lk);
    __syncthreads();
    As[lk + 0][lr] = a0.x; As[lk + 1][lr] = a0.y; As[lk + 2][lr] = a0.z; As[lk + 3][lr] = a0.w;
    As[lk + 0][lr + 64] = a1.x; As[lk + 1][lr + 64] = a1.y; As[lk + 2][lr + 64] = a1.z; As[lk + 3][lr + 64] = a1.w;
    Bs[lk + 0][lr] = b0.x; Bs[lk + 1][lr] = b0.y; Bs[lk + 2][lr] = b0.z; Bs[lk + 3][lr] = b0.w;
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 x0 = *reinterpret_cast<const float4*>(&As[kk][ty * 8]);
      const float4 x1 = *reinterpret_cast<const float4*>(&As[kk][ty * 8 + 4]);
      const float4 w0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
      const float b[4] = {w0.x, w0.y, w0.z, w0.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
  }

  const int nb = n0 + tx * 4;
  float bv[4] = {0.f, 0.f, 0.f, 0.f};
  if (bias) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (nb + j < p.N) bv[j] = bias[nb + j];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + ty * 8 + i;
    if (m >= p.M) continue;
    const long long orow = (long long)(m / p.row_inner) * p.row_outer + (m % p.row_inner);
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = acc[i][j] + bv[j];
    if (EPI == EPI_GLU_PAIR) {
      // columns (2c, 2c+1) = (value, gate) -> out column c = value * sigmoid(gate)   (nn.GLU)
#pragma unroll
      for (int j = 0; j < 4; j += 2) {
        const int n = nb + j;
        if (n + 1 < p.N) C[orow * p.ldc + (n >> 1)] = v[j] * (1.0f / (1.0f + expf(-v[j + 1])));
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = nb + j;
        if (n >= p.N) continue;
        float o = v[j];
        if (EPI == EPI_GELU) o = gelu_exact(o);
        if (EPI == EPI_ADD_C) o += C[orow * p.ldc + n];
        C[orow * p.ldc + n] = o;
      }
    }
  }
}
}  // namespace

int launch_sgemm(const SgemmParams& p, int epi, cudaStream_t st) {
  if (p.M <= 0 || p.N <= 0) return MMPFN_OK;
  if (p.K % BK != 0 || p.lda % 4 != 0 || p.ldw % 4 != 0) {
    set_error("sgemm: K=%d lda=%d ldw=%d must be multiples of 16/4/4", p.K, p.lda, p.ldw);
    return MMPFN_EINVAL;
  }
  dim3 grid((p.M + BM - 1) / BM, (p.N + BN - 1) / BN, p.batches > 0 ? p.batches : 1);
  switch (epi) {
    case EPI_NONE: sgemm_kernel<EPI_NONE><<<grid, 256, 0, st>>>(p); break;
    case EPI_GELU: sgemm_kernel<EPI_GELU><<<grid, 256, 0, st>>>(p); break;
    case EPI_GLU_PAIR: sgemm_kernel<EPI_GLU_PAIR><<<grid, 256, 0, st>>>(p); break;
    case EPI_ADD_C: sgemm_kernel<EPI_ADD_C><<<grid, 256, 0, st>>>(p); break;
    default: set_error("sgemm: bad epilogue %d", epi); return MMPFN_EINVAL;
  }
  return count_launch();
}

// ---------------------------------------------------------------------------------------------
// LayerNorm: one warp per row, the row lives in registers (two-pass variance), float2 accesses.
// Bandwidth-bound: reads x (+res) once, writes y once (+ bf16 shadow).
// ---------------------------------------------------------------------------------------------
namespace {
template <int W>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ res,
                                                        const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, long long rows,
                                                        float* __restrict__ y, uint16_t* __restrict__ yb,
                                                        long long x_stride) {
  constexpr int V = W / 64;  // float2 per lane
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float2* xr = reinterpret_cast<const float2*>(x + row * x_stride);
  float2 v[V];
#pragma unroll
  for (int i = 0; i < V; ++i) v[i] = xr[lane + 32 * i];
  if (res) {
    const float2* rr = reinterpret_cast<const float2*>(res + row * W);
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const float2 r = rr[lane + 32 * i];
      v[i].x += r.x;
      v[i].y += r.y;
    }
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) s += v[i].x + v[i].y;
  const float mean = warp_sum(s) * (1.0f / W);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean;
    q = fmaf(a, a, q);
    q = fmaf(b, b, q);
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / W) + kLnEps);
#pragma unroll
  for (int i = 0; i < V; ++i) {
    float a = (v[i].x - mean) * rstd, b = (v[i].y - mean) * rstd;
    if (gamma) {
      const float2 g = reinterpret_cast<const float2*>(gamma)[lane + 32 * i];
      const float2 be = reinterpret_cast<const float2*>(beta)[lane + 32 * i];
      a = fmaf(a, g.x, be.x);
      b = fmaf(b, g.y, be.y);
    }
    if (y) reinterpret_cast<float2*>(y + row * W)[lane + 32 * i] = make_float2(a, b);
    if (yb) reinterpret_cast<uint32_t*>(yb + row * W)[lane + 32 * i] = pack_bf16x2(a, b);
  }
}
}  // namespace

int launch_layernorm(const float* x, const float* res, const float* gamma, const float* beta, long long rows,
                     int width, float* y_f32, uint16_t* y_bf16, cudaStream_t st, long long x_stride) {
  if (rows <= 0) return MMPFN_OK;
  if (x_stride == 0) x_stride = width;
  const int wpb = 8;
  const unsigned grid = (unsigned)((rows + wpb - 1) / wpb);
  switch (width) {
    case 192: layernorm_kernel<192><<<grid, wpb * 32, 0, st>>>(x, res, gamma, beta, rows, y_f32, y_bf16, x_stride); break;
    case 384: layernorm_kernel<384><<<grid, wpb * 32, 0, st>>>(x, res, gamma, beta, rows, y_f32, y_bf16, x_stride); break;
    case 768: layernorm_kernel<768><<<grid, wpb * 32, 0, st>>>(x, res, gamma, beta, rows, y_f32, y_bf16, x_stride); break;
    default: set_error("layernorm: unsupported width %d", width); return MMPFN_EUNSUPPORTED;
  }
  return count_launch();
}

// ---------------------------------------------------------------------------------------------
// Attention between features (layer.py:332-339): for every row (b,s) a T x T attention per head,
// d = 32.  One CTA per (row, head); q/k/v of that head staged in shared memory in fp32; one warp
// per query token: lanes over keys for the scores, lanes over d for the output.
// ---------------------------------------------------------------------------------------------
namespace {
template <typename TIn>
__device__ __forceinline__ float ld_as_float(const TIn* p);
template <>
__device__ __forceinline__ float ld_as_float<float>(const float* p) { return *p; }
template <>
__device__ __forceinline__ float ld_as_float<uint16_t>(const uint16_t* p) { return bf16_bits_to_float(*p); }
__device__ __forceinline__ void st_from_float(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_from_float(uint16_t* p, float v) {
  __nv_bfloat16 b = __float2bfloat16_rn(v);
  *p = *reinterpret_cast<uint16_t*>(&b);
}

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(128) feat_attn_kernel(const TIn* __restrict__ qkv, TOut* __restrict__ att,
                                                        int T) {
  extern __shared__ float sm[];
  constexpr int P = kD + 1;
  float* qs = sm;                // [T][33]
  float* ks = qs + T * P;        // [T][33]
  float* vs = ks + T * P;        // [T][33]
  float* ps = vs + T * P;        // [4 warps][T]
  const long long row = blockIdx.x;
  const int h = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const TIn* base = qkv + row * T * (3 * kE) + h * kD;
  for (int i = threadIdx.x; i < T * kD; i += blockDim.x) {
    const int t = i / kD, d = i % kD;
    const TIn* r = base + (long long)t * (3 * kE) + d;
    qs[t * P + d] = ld_as_float<TIn>(r);
    ks[t * P + d] = ld_as_float<TIn>(r + kE);
    vs[t * P + d] = ld_as_float<TIn>(r + 2 * kE);
  }
  __syncthreads();
  const float scale = 0.17677669529663687f;  // 1/sqrt(32)
  float* pw = ps + warp * T;
  for (int i = warp; i < T; i += 4) {
    float mx = -INFINITY;
    for (int j = lane; j < T; j += 32) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < kD; ++d) s = fmaf(qs[i * P + d], ks[j * P + d], s);
      s *= scale;
      pw[j] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < T; j += 32) {
      const float e = expf(pw[j] - mx);
      pw[j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    __syncwarp();
    float o = 0.f;
    for (int j = 0; j < T; ++j) o = fmaf(pw[j], vs[j * P + lane], o);
    st_from_float(att + (row * T + i) * kE + h * kD + lane, o / sum);
    __syncwarp();
  }
}

template <typename TIn, typename TOut>
int launch_feat_attn(const TIn* qkv, TOut* att, long long n_seq, int T, cudaStream_t st) {
  if (n_seq <= 0) return MMPFN_OK;
  const size_t smem = (size_t)(3 * T * (kD + 1) + 4 * T) * sizeof(float);
  if (smem > 200 * 1024) {
    set_error("feature attention: %d tokens per row exceed the shared-memory tile", T);
    return MMPFN_EUNSUPPORTED;
  }
  auto kern = feat_attn_kernel<TIn, TOut>;
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    set_error("feature attention: cannot opt in to %zu bytes of shared memory: %s", smem, cudaGetErrorString(cudaGetLastError()));
    return MMPFN_ECUDA;
  }
  // grid.x carries the rows (up to 2^31-1)
  kern<<<dim3((unsigned)n_seq, kH), 128, smem, st>>>(qkv, att, T);
  return count_launch();
}
}  // namespace

// ---------------------------------------------------------------------------------------------
// Attention between features, bf16 tensor-core version (mma.sync m16n8k16, fp32 accumulate).
// One CTA per table row: the row's whole qkv block ([T][576] bf16, contiguous in HBM) is staged in
// shared memory once (16 B cp.async, rows padded to 1168 B so that ldmatrix is conflict free), then
// each warp owns (head, 16-query tile) work items: S = Q K^T in registers, softmax in registers,
// P re-used as the A fragments of O = P V.  HBM-bound: reads qkv once, writes att once.
// ---------------------------------------------------------------------------------------------
namespace {
constexpr int FA_ROW_BYTES = 3 * kE * 2 + 16;   // 1168

// KT = number of 16-key tiles the register file is sized for (T <= 16*KT).
// A CTA walks table rows blockIdx.x, blockIdx.x + gridDim.x, ... with two staging buffers: the qkv block
// of the next row streams in (cp.async) while the current row is computed, so the DRAM latency of a row is
// paid under the previous row's arithmetic instead of once per CTA.
template <int KT>
__global__ void __launch_bounds__(384) feat_attn_mma_kernel(const uint16_t* __restrict__ qkv,
                                                            uint16_t* __restrict__ att, int T, long long n_rows,
                                                            int n_buf) {
  extern __shared__ __align__(16) uint8_t fsm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_kt = (T + 15) >> 4;               // 16-key tiles actually present
  const int Tp = n_kt * 16;
  const uint32_t buf_bytes = (uint32_t)Tp * FA_ROW_BYTES;
  const uint32_t sbase0 = (uint32_t)__cvta_generic_to_shared(fsm);
  constexpr int CH = 3 * kE * 2 / 16;           // 72 chunks of 16 B per token

  // stage [T][576] bf16 of one table row -> smem rows of FA_ROW_BYTES
  auto stage = [&](long long row, int b) {
    const uint8_t* src = reinterpret_cast<const uint8_t*>(qkv + row * T * (3 * kE));
    const uint32_t dst = sbase0 + b * buf_bytes;
    for (int i = threadIdx.x; i < T * CH; i += blockDim.x) {
      const int t = i / CH, c = i % CH;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + t * FA_ROW_BYTES + c * 16),
                   "l"(src + (long long)t * (3 * kE * 2) + c * 16));
    }
    asm volatile("cp.async.commit_group;");
  };
  // the padded token rows of the buffers stay zero for the CTA's whole life.  n_buf = 1 (wide rows: two
  // buffers would not fit shared memory): load, compute, load, ... without the overlap.
  for (int b = 0; b < n_buf; ++b)
    for (int i = threadIdx.x; i < (Tp - T) * CH; i += blockDim.x) {
      const int t = T + i / CH, c = i % CH;
      *reinterpret_cast<uint4*>(fsm + b * buf_bytes + t * FA_ROW_BYTES + c * 16) = make_uint4(0, 0, 0, 0);
    }
  long long row = blockIdx.x;
  if (row < n_rows) stage(row, 0);
  for (int it = 0; row < n_rows; row += gridDim.x, ++it) {
  const int cur = n_buf == 2 ? (it & 1) : 0;
  const long long nxt = row + gridDim.x;
  if (n_buf == 2 && nxt < n_rows) {
    stage(nxt, cur ^ 1);                         // (its previous reader finished before the barrier below)
    asm volatile("cp.async.wait_group 1;");
  } else {
    asm volatile("cp.async.wait_group 0;");
  }
  __syncthreads();
  const uint32_t sbase = sbase0 + cur * buf_bytes;

  const int n_items = kH * n_kt;
  for (int item = warp; item < n_items; item += (blockDim.x >> 5)) {
    const int h = item / n_kt, mt = item % n_kt;
    // (the output block of the item overwrites the item's own Q block in shared memory: the row then leaves as whole
    // 16-byte pieces, coalesced, instead of 4-byte stores scattered over 8 token rows)
    feat_attn_item<KT>(sbase, FA_ROW_BYTES, h * kD * 2, (kE + h * kD) * 2, (2 * kE + h * kD) * 2, T, n_kt, mt, lane);
  }
  __syncthreads();
  {
    constexpr int OC = kE * 2 / 16;               // 24 pieces of 16 B per token
    uint8_t* dst = reinterpret_cast<uint8_t*>(att + row * T * kE);
    for (int i = threadIdx.x; i < T * OC; i += blockDim.x) {
      const int t = i / OC, c = i % OC;
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                   : "r"(sbase + t * FA_ROW_BYTES + c * 16));
      *reinterpret_cast<uint4*>(dst + (long long)t * (kE * 2) + c * 16) = v;
    }
  }
  __syncthreads();                               // everyone is done with this buffer before it is refilled
  if (n_buf == 1 && nxt < n_rows) stage(nxt, 0);
  }
}

template <int KT>
int launch_feat_attn_mma_t(const uint16_t* qkv, uint16_t* att, long long n_seq, int T, cudaStream_t st) {
  const int Tp = (T + 15) / 16 * 16;
  const int n_buf = (size_t)2 * Tp * FA_ROW_BYTES <= 200 * 1024 ? 2 : 1;
  const size_t smem = (size_t)n_buf * Tp * FA_ROW_BYTES;
  auto kern = feat_attn_mma_kernel<KT>;
  MMPFN_OPT_IN_SMEM(kern, 227 * 1024);
  const int n_sm = device_sm_count();
  const int n_items = kH * (Tp / 16);
  const int warps = n_items < 12 ? n_items : 12;
  // CTAs resident per SM: shared memory (two staging buffers each) and 2048 threads
  int per_sm = (int)((227 * 1024) / (smem + 1024));
  if (per_sm > 2048 / (warps * 32)) per_sm = 2048 / (warps * 32);
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)n_sm * per_sm;
  if (grid > n_seq) grid = n_seq;
  kern<<<(unsigned)grid, warps * 32, smem, st>>>(qkv, att, T, n_seq, n_buf);
  return count_launch();
}
}  // namespace

int launch_feat_attn_f32(const float* qkv, float* att, long long n_seq, int T, cudaStream_t st) {
  return launch_feat_attn<float, float>(qkv, att, n_seq, T, st);
}
int launch_feat_attn_bf16(const uint16_t* qkv, uint16_t* att, long long n_seq, int T, cudaStream_t st) {
  if (n_seq <= 0) return MMPFN_OK;
  if (T <= 32) return launch_feat_attn_mma_t<2>(qkv, att, n_seq, T, st);
  if (T <= 64) return launch_feat_attn_mma_t<4>(qkv, att, n_seq, T, st);
  if (T <= 96) return launch_feat_attn_mma_t<6>(qkv, att, n_seq, T, st);
  if (T <= 144) return launch_feat_attn_mma_t<9>(qkv, att, n_seq, T, st);
  if (T <= 192) return launch_feat_attn_mma_t<12>(qkv, att, n_seq, T, st);
  return launch_feat_attn<uint16_t, uint16_t>(qkv, att, n_seq, T, st);   // CUDA-core fallback for very wide rows
}

// ---------------------------------------------------------------------------------------------
// Attention between items, fp32 flash kernel (parity mode).  CTA = 64 queries of one (plane, head);
// streams 64-key tiles; S = Q K^T and O += P V on FFMA with 4x8 / 4x4 register tiles.
// ---------------------------------------------------------------------------------------------
namespace {
constexpr int IQ = 64, IK = 64;

__global__ void __launch_bounds__(128) item_attn_f32_kernel(ItemAttnF32 p) {
  __shared__ __align__(16) float Qt[kD][IQ];       // [d][query]
  __shared__ __align__(16) float Kt[kD][IK];       // [d][key]
  __shared__ __align__(16) float Vs[IK][kD];       // [key][d]
  __shared__ __align__(16) float Pt[IK][IQ + 4];   // [key][query]
  const int plane = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * IQ;
  const int tid = threadIdx.x;
  const int ty = tid >> 3, tx = tid & 7;   // S tile: rows ty*4..+3, cols tx*8..+7 ; O tile: rows ty*4.., d tx*4..
  const int pb = plane / p.inner, pt = plane % p.inner;
  const float* qb = p.q + pb * p.q_outer + pt * p.q_inner + h * kD;
  const int hk = p.shared_kv ? 0 : h;
  const float* kb = p.k + pb * p.kv_outer + pt * p.kv_inner + hk * kD;
  const float* vb = p.v + pb * p.kv_outer + pt * p.kv_inner + hk * kD;
  // this entry's own counts: its keys past n_kv are never read, its query rows from n_q on are written as zeros
  const int n_q = p.q_len ? min(max(p.q_len[pb], 0), p.n_q) : p.n_q;
  const int n_kv = p.kv_len ? min(max(p.kv_len[pb], 1), p.n_kv) : p.n_kv;
  if (q0 >= n_q) {
    for (int i = tid; i < IQ * (kD / 4); i += 128) {
      const int r = q0 + (i >> 3), c4 = (i & 7) * 4;
      if (r < p.n_q)
        *reinterpret_cast<float4*>(p.out + pb * p.o_outer + pt * p.o_inner + (long long)r * p.o_row + h * kD + c4) =
            make_float4(0.f, 0.f, 0.f, 0.f);
    }
    return;
  }

  // Q tile -> Qt (transposed), pre-scaled by 1/sqrt(d)
  const float scale = 0.17677669529663687f;
  for (int i = tid; i < IQ * (kD / 4); i += 128) {
    const int r = i >> 3, c4 = (i & 7) * 4;
    float4 v = make_float4(0, 0, 0, 0);
    if (q0 + r < n_q) v = *reinterpret_cast<const float4*>(qb + (long long)(q0 + r) * p.q_row + c4);
    Qt[c4 + 0][r] = v.x * scale; Qt[c4 + 1][r] = v.y * scale; Qt[c4 + 2][r] = v.z * scale; Qt[c4 + 3][r] = v.w * scale;
  }
  float m[4], l[4], o[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m[i] = -INFINITY;
    l[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
  }

  for (int k0 = 0; k0 < n_kv; k0 += IK) {
    __syncthreads();   // previous tile fully consumed (also orders the Qt stores the first time)
    for (int i = tid; i < IK * (kD / 4); i += 128) {
      const int r = i >> 3, c4 = (i & 7) * 4;
      float4 kv = make_float4(0, 0, 0, 0), vv = kv;
      if (k0 + r < n_kv) {
        kv = *reinterpret_cast<const float4*>(kb + (long long)(k0 + r) * p.kv_row + c4);
        vv = *reinterpret_cast<const float4*>(vb + (long long)(k0 + r) * p.kv_row + c4);
      }
      Kt[c4 + 0][r] = kv.x; Kt[c4 + 1][r] = kv.y; Kt[c4 + 2][r] = kv.z; Kt[c4 + 3][r] = kv.w;
      *reinterpret_cast<float4*>(&Vs[r][c4]) = vv;
    }
    __syncthreads();
    float s[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) s[i][j] = 0.f;
#pragma unroll 8
    for (int d = 0; d < kD; ++d) {
      const float4 a = *reinterpret_cast<const float4*>(&Qt[d][ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Kt[d][tx * 8]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Kt[d][tx * 8 + 4]);
      const float av[4] = {a.x, a.y, a.z, a.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) s[i][j] = fmaf(av[i], bv[j], s[i][j]);
    }
    // mask the key tail, online softmax per row (8 lanes share a row)
    float alpha[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (k0 + tx * 8 + j >= n_kv) s[i][j] = -INFINITY;
        mx = fmaxf(mx, s[i][j]);
      }
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
      const float mn = fmaxf(m[i], mx);
      alpha[i] = expf(m[i] - mn);   // first tile: exp(-inf) = 0
      float rs = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[i][j] = expf(s[i][j] - mn);
        rs += s[i][j];
      }
      rs += __shfl_xor_sync(0xffffffffu, rs, 1);
      rs += __shfl_xor_sync(0xffffffffu, rs, 2);
      rs += __shfl_xor_sync(0xffffffffu, rs, 4);
      l[i] = l[i] * alpha[i] + rs;
      m[i] = mn;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      *reinterpret_cast<float4*>(&Pt[tx * 8 + j][ty * 4]) = make_float4(s[0][j], s[1][j], s[2][j], s[3][j]);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) o[i][j] *= alpha[i];
#pragma unroll 8
    for (int j = 0; j < IK; ++j) {
      const float4 pv = *reinterpret_cast<const float4*>(&Pt[j][ty * 4]);
      const float4 vv = *reinterpret_cast<const float4*>(&Vs[j][tx * 4]);
      const float pa[4] = {pv.x, pv.y, pv.z, pv.w};
      const float va[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) o[i][c] = fmaf(pa[i], va[c], o[i][c]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = q0 + ty * 4 + i;
    if (r >= p.n_q) continue;
    const float inv = 1.0f / l[i];
    float* dst = p.out + pb * p.o_outer + pt * p.o_inner + (long long)r * p.o_row + h * kD + tx * 4;
    *reinterpret_cast<float4*>(dst) = r < n_q ? make_float4(o[i][0] * inv, o[i][1] * inv, o[i][2] * inv, o[i][3] * inv)
                                              : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
}  // namespace

namespace {
__global__ void kv_extract_f32_kernel(const float* __restrict__ qkv, float* __restrict__ kv, int S, int T,
                                      long long n, const int* __restrict__ n_rows) {
  // one thread per (b, t, s, 64 floats): k (32) | v (32) of head 0
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i & 63);
  const long long r = i >> 6;           // (b*T + t)*S + s
  const long long s = r % S, bt = r / S;
  const long long t = bt % T, b = bt / T;
  if (n_rows && s >= n_rows[b]) {                 // a pad row of entry b: not read
    kv[i] = 0.f;
    return;
  }
  const float* src = qkv + ((b * S + s) * T + t) * (3 * kE) + (c < 32 ? kE + c : 2 * kE + (c - 32));
  kv[i] = *src;
}
}  // namespace

int launch_kv_extract_f32(const float* qkv, float* kv, int B, int S, int T, cudaStream_t st, const int* n_rows) {
  const long long n = (long long)B * T * S * 64;
  if (n <= 0) return MMPFN_OK;
  kv_extract_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(qkv, kv, S, T, n, n_rows);
  return count_launch();
}

int launch_item_attn_f32(const ItemAttnF32& p, cudaStream_t st) {
  if (p.planes <= 0 || p.n_q <= 0) return MMPFN_OK;
  if (p.n_kv <= 0) {
    set_error("item attention: empty key set");
    return MMPFN_EINVAL;
  }
  if (p.planes > 65535) {
    set_error("item attention: %d planes exceed grid.z", p.planes);
    return MMPFN_EUNSUPPORTED;
  }
  dim3 grid((p.n_q + IQ - 1) / IQ, kH, p.planes);
  item_attn_f32_kernel<<<grid, 128, 0, st>>>(p);
  return count_launch();
}

}  // namespace mmpfn
