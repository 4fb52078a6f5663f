// common.cuh — shared declarations for libmmpfn_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/mmpfn_b200.h"

namespace mmpfn {

// TabPFN-v2 classifier geometry (reference model/config.py:18-83); validated at every entry point.
constexpr int kE = 192;    // emsize
constexpr int kH = 6;      // heads
constexpr int kD = 32;     // d_k = d_v
constexpr int kHid = 768;  // MLP hidden
constexpr float kLnEps = 1e-5f;

extern std::atomic<int64_t> g_launches;
void set_error(const char* fmt, ...);
int check_geometry(const mmpfn_geometry* g);

inline int count_launch() {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  // cudaGetLastError, not Peek: the library links cudart statically and owns this per-thread error
  // state; a non-sticky launch failure must be reported once and cleared, not poison every later call
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("kernel launch failed: %s", cudaGetErrorString(e));
    return MMPFN_ECUDA;
  }
  return MMPFN_OK;
}

// Per-device facts: the library may be called on several devices of one process (one after another or from one
// host thread per GPU), so nothing about "the" device is cached in a plain static.
inline int current_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); return -1; }
  return d;
}
inline int device_sm_count() {
  static int n[64] = {0};
  const int d = current_device();
  if (d < 0 || d >= 64) return 148;
  if (!n[d]) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d) != cudaSuccess || v < 1) { cudaGetLastError(); v = 148; }
    n[d] = v;
  }
  return n[d];
}
// Opt a kernel in to `bytes` of dynamic shared memory, once per device and call site; a failure is reported here
// (MMPFN_ECUDA with a message) instead of surfacing later as an unexplained launch error.
#define MMPFN_OPT_IN_SMEM(kern, bytes)                                                                     \
  do {                                                                                                     \
    static unsigned long long _done = 0;                                                                   \
    const int _d = ::mmpfn::current_device();                                                              \
    if (_d < 0 || _d >= 64 || !((_done >> _d) & 1ull)) {                                                   \
      if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)) != cudaSuccess) { \
        ::mmpfn::set_error("cannot opt in to %d bytes of dynamic shared memory: %s", (int)(bytes),           \
                           cudaGetErrorString(cudaGetLastError()));                                        \
        return MMPFN_ECUDA;                                                                                \
      }                                                                                                    \
      if (_d >= 0 && _d < 64) _done |= 1ull << _d;                                                         \
    }                                                                                                      \
  } while (0)

#define MMPFN_TRY(expr)            \
  do {                             \
    int _rc = (expr);              \
    if (_rc != MMPFN_OK) return _rc; \
  } while (0)

__device__ __forceinline__ float gelu_exact(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float fast_exp2f(float x) {   // MUFU.EX2
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float bf16_bits_to_float(uint16_t b) { return __uint_as_float(uint32_t(b) << 16); }

// ---- fp32 building blocks (kernels_f32.cu) ---------------------------------------------------
enum { EPI_NONE = 0, EPI_GELU = 1, EPI_GLU_PAIR = 2, EPI_ADD_C = 3 };

struct SgemmParams {
  const float* A;      // [M][lda]
  const float* W;      // [N][ldw]
  const float* bias;   // [N] or null
  float* C;            // out
  int M, N, K, lda, ldw, ldc;
  // batching over blockIdx.z
  long long a_batch, w_batch, bias_batch, c_batch;
  int batches;
  // output row remap: out_row = (m / row_inner) * row_outer + (m % row_inner)
  int row_inner, row_outer;
};
int launch_sgemm(const SgemmParams& p, int epi, cudaStream_t st);

// y = LN(x (+res)) (*gamma + beta); writes fp32 and/or bf16.  width in {192, 384, 768}.
// x_stride: elements between consecutive input rows (0 = width).
int launch_layernorm(const float* x, const float* res, const float* gamma, const float* beta, long long rows,
                     int width, float* y_f32, uint16_t* y_bf16, cudaStream_t st, long long x_stride = 0);
// copy head-0 k|v of the item-attention qkv buffer [B][S][T][3E] into the fp32 context [B][T][S][2][kD]; with
// n_rows (device [B]) the rows s >= n_rows[b] are written as zeros instead
int launch_kv_extract_f32(const float* qkv, float* kv, int B, int S, int T, cudaStream_t st, const int* n_rows = nullptr);

// attention between features: qkv [rows = n_seq*T][3*kE] (q|k|v, head-major) -> att [rows][kE]
int launch_feat_attn_f32(const float* qkv, float* att, long long n_seq, int T, cudaStream_t st);
int launch_feat_attn_bf16(const uint16_t* qkv, uint16_t* att, long long n_seq, int T, cudaStream_t st);
// QKV projection + feature attention in one kernel (kernels_featfused.cu); T <= 64
bool feat_qkv_attn_supported(int T);
int launch_feat_qkv_attn(const uint16_t* x, const uint16_t* w_qkv, long long M, int T, uint16_t* att, cudaStream_t st);

// attention between items, fp32 flash kernel.  For plane p in [0, planes) and head h:
//   q row i  at  q  + plane_off(q)  + i*q_row  + h*kD          (n_q rows)
//   k row j  at  k  + plane_off(kv) + j*kv_row + (shared_kv ? 0 : h*kD)   (n_kv rows);  v likewise
//   out row i at out + plane_off(o) + i*o_row + h*kD
// plane p = (b, t) with b = p / inner, t = p % inner; offsets are b*X_outer + t*X_inner.
struct ItemAttnF32 {
  const float *q, *k, *v;
  float* out;
  long long q_outer, q_inner, q_row, kv_outer, kv_inner, kv_row, o_outer, o_inner, o_row;
  int planes, inner, n_q, n_kv, shared_kv;
  // per-entry counts (device int32 [planes / inner], or NULL): entry b attends over its first kv_len[b] keys, its
  // query rows q_len[b] .. n_q-1 are written as zeros; rows past an entry's counts are never read
  const int *q_len, *kv_len;
};
int launch_item_attn_f32(const ItemAttnF32& p, cudaStream_t st);

// ---- tcgen05 path (kernels_tc.cu) ------------------------------------------------------------
enum { TC_EPI_BF16 = 0, TC_EPI_GELU_BF16 = 1, TC_EPI_RESID_LN = 2, TC_EPI_QKV_ITEMS = 3, TC_EPI_GLU_PAIR_F32 = 4 };
struct TcGemm {
  const uint16_t* A;   // bf16 activations; FLAT: [M][K]; ITEMS: state [B][S][T][K]
  const uint16_t* W;   // bf16 [N][K]
  int M, N, K;         // FLAT: M rows.  ITEMS: M unused (B,S,T below)
  int items;           // 0 FLAT, 1 ITEMS (A tile = 128 rows s at fixed (b,t))
  int B, S, T;
  int epi;
  // TC_EPI_BF16 / TC_EPI_GELU_BF16
  uint16_t* out_bf16;  // [M][N]
  // TC_EPI_RESID_LN (N == kE): state_f32 (residual in, LN out, in place) + bf16 shadow
  float* resid_f32;
  uint16_t* ln_bf16;
  // TC_EPI_QKV_ITEMS: planes (b,t,h); q/k [plane][S_pad][kD], vt [plane][kD][S_pad]
  uint16_t *q_out, *k_out, *vt_out;
  int S_pad;
  // optional head-0 context for this layer: k0 [B][T][S_pad][kD], vt0 [B][T][kD][S_pad]
  uint16_t *k0_out, *vt0_out;
  // TC_EPI_GLU_PAIR_F32 (kernels_tc.cu only): columns (2c, 2c+1) = (value, gate) + bias -> out_f32[m][c] = value * sigmoid(gate)
  const float* bias;
  float* out_f32;      // [M][N/2]
};
int launch_tc_gemm(const TcGemm& p, cudaStream_t st);
// persistent variant for K = 192, N % 192 == 0 (kernels_rowgemm.cu): BF16 / RESID_LN / QKV_ITEMS epilogues
int launch_tc_rowgemm(const TcGemm& p, cudaStream_t st);

// Fused MLP sublayer (kernels_mlp.cu): state <- LN(state + W2 gelu(W1 state)), in place.
struct TcMlp {
  const uint16_t* state_b;   // bf16 shadow of the state [M][kE] (MMA operand)
  uint16_t* state_b_out;     // where the new bf16 shadow goes (may alias state_b)
  float* resid_f32;          // fp32 state [M][kE]: residual in, LayerNorm out
  const uint16_t* w1;        // [kHid][kE] bf16
  const uint16_t* w2;        // [kE][kHid] bf16
  int M;
};
int launch_tc_mlp(const TcMlp& p, cudaStream_t st);

struct TcItemAttn {
  const uint16_t* q;    // [planes_q = B*T*kH][Sq_pad][kD]
  const uint16_t* k;    // [planes_kv][Skv_pad][kD]
  const uint16_t* vt;   // [planes_kv][kD][Skv_pad]
  uint16_t* out;        // att, state layout [B][S][T][kE] bf16 (row (b,s,t), cols h*kD+d)
  int B, T, n_q, Sq_pad, n_kv, Skv_pad;
  int shared_kv;        // 1: kv planes are (b,t) (head 0 for all six q heads); 0: (b,t,h)
  // shared_kv only: where estimator b's planes live.  kv_slots = 0: dense, plane (b,t) at (b*T + t) planes from k / vt.
  // kv_slots = c > 0: the context sits in an all-gather buffer, c estimators back to back per rank chunk:
  // estimator b = (rank b / c, slot b % c), its plane t at  rank * kv_rank_stride + (slot*T + t) planes  (elements).
  int kv_slots;
  long long kv_rank_stride;
  // Row segments (row-sharded context build, dist.py "rows" mode): the n_kv keys are stored as ceil(n_kv /
  // kv_seg_rows) chunks of kv_seg_rows rows (a multiple of the 48-key tile, so that no tile straddles two chunks
  // and the tiles are exactly those of the unsegmented layout), kv_seg_stride elements apart; inside a chunk the
  // planes are laid out as usual with Skv_pad allocated rows.  0 = one contiguous row range.
  int kv_seg_rows;
  long long kv_seg_stride;
  // per-entry counts (device int32 [B], or NULL = n_q / n_kv for every entry): entry b attends over its first
  // kv_len[b] keys (1..n_kv); its output rows q_len[b] .. n_q-1 are written as zeros.  Key rows between an entry's
  // count and n_kv that its last tile covers must be zero (what the TMA out-of-bounds fill gives an entry run alone).
  const int* q_len;
  const int* kv_len;
};
int launch_tc_item_attn(const TcItemAttn& p, cudaStream_t st);

// ---- stem / tail (kernels_stem.cu) -----------------------------------------------------------
// Statistics block per estimator, indexed by COMPACTED slot c = g*fpg + j (encoders.py:102-130):
//   src[Fp] (source column stored as float, -1 = empty slot) | fill | lo | hi | mean | std | scale[G]
// An empty slot holds the statistics of the zero column the reference pads the group with.
struct TabStatsLayout {
  int Fp, G;
  __host__ __device__ int src() const { return 0; }
  __host__ __device__ int fill() const { return Fp; }
  __host__ __device__ int lo() const { return 2 * Fp; }
  __host__ __device__ int hi() const { return 3 * Fp; }
  __host__ __device__ int mean() const { return 4 * Fp; }
  __host__ __device__ int stdv() const { return 5 * Fp; }
  __host__ __device__ int scale() const { return 6 * Fp; }
  __host__ __device__ int total() const { return 6 * Fp + G; }
};
// n_rows / n_train_b (device [B], or NULL = S / n_train): entry b's statistics over its first n_rows[b] rows, of
// which the first n_train_b[b] are train rows
int launch_tab_fit(const float* x, int B, int S, int F, int fpg, int n_train, float n_sigma, float* stats,
                   cudaStream_t st, const int* n_rows = nullptr, const int* n_train_b = nullptr);
// img_off (device [B], elements, or NULL = b * img_bstride): where entry b's image tokens start;
// n_rows (device [B], or NULL = S): rows s >= n_rows[b] are written as zeros
int launch_stem_tokens(const mmpfn_geometry* g, const mmpfn_weights* w, const float* x, const float* stats,
                       const float* img_tok, const float* y, const float* y_mean, const uint64_t* y_mask,
                       const float* pos_emb, int B, int S, int F, int H_img, long long x_bstride, long long y_bstride,
                       long long img_bstride, float* state_f32, uint16_t* state_bf16, int32_t* nan_flag, cudaStream_t st,
                       const long long* img_off = nullptr, const int* n_rows = nullptr);
int launch_cap_attn(const float* kv, const float* q, int S, int n_kv, int Hc, float* out, cudaStream_t st);
int launch_cap_combine(const float* o, const float* ffn, const float* gamma, const float* beta, long long rows,
                       float* out, cudaStream_t st);
int launch_moe_gate_scale(const float* gate_logits, float* tok, int S, int Hm, cudaStream_t st);
int launch_proba_tail(const float* logits, const int32_t* perm, const float* prior, int n_est, int S, int n_out,
                      int n_classes, float temperature, int avg_before, float* proba, cudaStream_t st);

// ---- bar-distribution tail (kernels_tail.cu) ------------------------------------------------------------------
// task_logits NULL: one task, logits [n_est][S][K]; else the many-task form (row_offset, n_tasks; logits unused)
int launch_bar_tail(const float* logits, const float* const* task_logits, const int32_t* row_offset, int n_tasks,
                    int n_est, int S, int K, const int32_t* src_bucket, const float* src_share, const uint8_t* cancel,
                    const float* borders, float temperature, int avg_before, const float* quantiles, int n_q,
                    float* mean, float* median, float* mode, float* quant, float* log_prob, cudaStream_t st);

}  // namespace mmpfn
