// kernels_tail.cu — the bar-distribution tail of the regressor (mmpfn_bar_tail and its many-task form
// mmpfn_bar_tail_tasks, include/mmpfn_b200.h).
//
// One CTA per test row.  Per estimator: load the row's K logits (float4 when aligned), temperature and cancel
// mask, block max / sum -> p_e in shared memory, exclusive prefix sum of p_e in float64, then the translated
// bucket masses q_e[j] accumulated into acc[j] (or log q_e[j] for average_before_softmax).  At the end P, log P,
// the mean, the mode and one binary search per quantile over the float64 prefix sum of P.
//
// The prefix sums are float64 because a bucket mass is a difference of two of them: in fp32 a 1e-6 bucket far into
// a 5000-bucket row would keep only a digit or two.  p_e itself is fp32 (relative error ~1e-7 per bucket).
#include <math.h>

#include "common.cuh"

namespace mmpfn {
namespace {

constexpr int kTailMaxK = 8192;
constexpr int kTailMaxWarps = 16;   // blockDim <= 512

struct TailScratch {
  double d[kTailMaxWarps];
  float f[kTailMaxWarps];
  int i[kTailMaxWarps];
};

__host__ __device__ inline size_t tail_smem_bytes(int K) {
  return sizeof(double) * (size_t)(K + 1) + 2 * sizeof(float) * (size_t)K + sizeof(TailScratch);
}

__device__ __forceinline__ float block_max(float v, TailScratch* sc) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) sc->f[wid] = v;
  __syncthreads();
  float r = -INFINITY;
  for (int w = 0; w < nw; ++w) r = fmaxf(r, sc->f[w]);
  return r;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ double block_sum_d(double v, TailScratch* sc) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  v = warp_sum_d(v);
  __syncthreads();
  if (lane == 0) sc->d[wid] = v;
  __syncthreads();
  double r = 0.0;
  for (int w = 0; w < nw; ++w) r += sc->d[w];
  return r;
}

// out[0] = 0, out[k+1] = sum_{i<=k} x[i] (float64), k < K.  Each thread scans a contiguous chunk.
__device__ void block_exclusive_scan(const float* x, int K, double* out, TailScratch* sc) {
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5, nw = blockDim.x >> 5;
  const int chunk = (K + blockDim.x - 1) / blockDim.x;
  const int b = min(t * chunk, K), e = min(b + chunk, K);
  double local = 0.0;
  for (int k = b; k < e; ++k) local += (double)x[k];
  double incl = local;                                   // inclusive scan of the thread totals inside the warp
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  __syncthreads();
  if (lane == 31) sc->d[wid] = incl;
  __syncthreads();
  double run = incl - local;
  for (int w = 0; w < wid; ++w) run += sc->d[w];
  if (t == 0) out[0] = 0.0;
  for (int k = b; k < e; ++k) {
    run += (double)x[k];
    out[k + 1] = run;
  }
  (void)nw;
  __syncthreads();
}

// position of common border j within estimator e's buckets: C_e(j) = pre[i] + p[i] * s  (i in [0, K]; p[K] := 0)
__device__ __forceinline__ void border_pos(const int32_t* sb, const float* ss, int j, int K, int& i, float& s) {
  if (j == 0) { i = 0; s = 0.f; return; }            // C_e(0) = 0
  if (j == K) { i = K; s = 0.f; return; }            // C_e(K) = 1 (the row's own total)
  const int b = __ldg(sb + j);
  if (b < 0) { i = 0; s = 0.f; return; }
  if (b >= K) { i = K; s = 0.f; return; }
  i = b;
  s = __ldg(ss + j);
}

// kTasks = false: one task, logits [n_est][S][K] (mmpfn_bar_tail).  kTasks = true: row s belongs to the task tk with
// row_offset[tk] <= s < row_offset[tk + 1]; its logits for estimator e start at task_logits[tk * n_est + e] (row
// stride K) and its maps and borders at task tk's slices (mmpfn_bar_tail_tasks).  S is the total row count.
// The tasks-only parameters come last: the one-task form keeps its parameter offsets, 32 registers and SASS.
template <bool kTasks>
__global__ void __launch_bounds__(512) bar_tail_kernel(
    const float* __restrict__ logits, int n_est, int S, int K, const int32_t* __restrict__ src_bucket,
    const float* __restrict__ src_share, const uint8_t* __restrict__ cancel, const float* __restrict__ borders,
    float temperature, int avg_before, const float* __restrict__ quantiles, int n_q, float* __restrict__ mean,
    float* __restrict__ median, float* __restrict__ mode, float* __restrict__ quant, float* __restrict__ log_prob,
    const float* const* __restrict__ task_logits, const int32_t* __restrict__ row_offset, int n_tasks) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* pre = reinterpret_cast<double*>(smem_raw);                        // [K+1]
  float* p = reinterpret_cast<float*>(pre + K + 1);                         // [K]
  float* acc = p + K;                                                       // [K]
  TailScratch* sc = reinterpret_cast<TailScratch*>(acc + K);
  const int s = blockIdx.x, t = threadIdx.x, nt = blockDim.x;
  const bool vec4 = (K % 4) == 0;
  int tk = 0;
  long long row = s;                                   // the row within its task
  if constexpr (kTasks) {
    int lo = 0, hi = n_tasks - 1;                      // last task whose first row is <= s (skips empty tasks)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (__ldg(row_offset + mid) <= s) lo = mid; else hi = mid - 1;
    }
    tk = lo;
    row = s - __ldg(row_offset + tk);
    src_bucket += (long long)tk * n_est * (K + 1);
    src_share += (long long)tk * n_est * (K + 1);
    if (cancel) cancel += (long long)tk * n_est * K;
    borders += (long long)tk * (K + 1);
  }

  for (int j = t; j < K; j += nt) acc[j] = 0.f;
  for (int e = 0; e < n_est; ++e) {
    const float* lg = kTasks ? task_logits[(long long)tk * n_est + e] + row * K : logits + ((long long)e * S + s) * K;
    const uint8_t* cm = cancel ? cancel + (long long)e * K : nullptr;
    float mx = -INFINITY;
    if (vec4) {
      for (int k4 = t; k4 < K / 4; k4 += nt) {
        float4 v = __ldcs(reinterpret_cast<const float4*>(lg) + k4);      // streamed: read once
        float z[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (temperature != 1.0f) z[u] = z[u] / temperature;
          if (cm && cm[4 * k4 + u]) z[u] = -INFINITY;
          p[4 * k4 + u] = z[u];
          mx = fmaxf(mx, z[u]);
        }
      }
    } else {
      for (int k = t; k < K; k += nt) {
        float z = __ldcs(lg + k);
        if (temperature != 1.0f) z = z / temperature;
        if (cm && cm[k]) z = -INFINITY;
        p[k] = z;
        mx = fmaxf(mx, z);
      }
    }
    mx = block_max(mx, sc);
    double sum = 0.0;
    for (int k = t; k < K; k += nt) {
      const float ex = expf(p[k] - mx);
      p[k] = ex;
      sum += ex;
    }
    const float inv_sum = (float)(1.0 / block_sum_d(sum, sc));
    for (int k = t; k < K; k += nt) p[k] *= inv_sum;
    __syncthreads();
    block_exclusive_scan(p, K, pre, sc);
    const int32_t* sb = src_bucket + (long long)e * (K + 1);
    const float* ss = src_share + (long long)e * (K + 1);
    for (int j = t; j < K; j += nt) {
      int i0, i1;
      float s0, s1;
      border_pos(sb, ss, j, K, i0, s0);
      border_pos(sb, ss, j + 1, K, i1, s1);
      const double p0 = i0 < K ? (double)p[i0] : 0.0, p1 = i1 < K ? (double)p[i1] : 0.0;
      double q = (pre[i1] - pre[i0]) + p1 * (double)s1 - p0 * (double)s0;
      q = q > 0.0 ? q : 0.0;
      acc[j] += avg_before ? logf((float)q) : (float)q;
    }
    __syncthreads();                                   // p / pre are rewritten by the next estimator
  }

  // combined distribution P -> acc
  const float inv_n = 1.0f / (float)n_est;
  if (avg_before) {
    float m = -INFINITY;
    for (int j = t; j < K; j += nt) { acc[j] *= inv_n; m = fmaxf(m, acc[j]); }
    m = block_max(m, sc);
    double sum = 0.0;
    for (int j = t; j < K; j += nt) { const float ex = expf(acc[j] - m); acc[j] = ex; sum += ex; }
    const float inv = (float)(1.0 / block_sum_d(sum, sc));
    for (int j = t; j < K; j += nt) acc[j] *= inv;
  } else {
    for (int j = t; j < K; j += nt) acc[j] *= inv_n;
  }
  __syncthreads();
  if (log_prob) {
    float* lp = log_prob + (long long)s * K;
    for (int j = t; j < K; j += nt) __stcs(lp + j, logf(acc[j]));
  }
  const float sqrt_2_over_pi = 0.79788456080286535588f;
  if (mean) {
    double m = 0.0;
    for (int j = t; j < K; j += nt) {
      const float g0 = __ldg(borders + j), g1 = __ldg(borders + j + 1);
      float mj = 0.5f * (g0 + g1);
      if (j == 0) mj = g1 - (g1 - g0) * sqrt_2_over_pi;
      if (j == K - 1) mj = g0 + (g1 - g0) * sqrt_2_over_pi;
      m += (double)acc[j] * (double)mj;
    }
    m = block_sum_d(m, sc);
    if (t == 0) mean[s] = (float)m;
  }
  if (mode) {
    float best = -INFINITY;
    int bj = K;
    for (int j = t; j < K; j += nt) {                  // increasing j per thread: ties keep the lowest
      const float d = acc[j] / (__ldg(borders + j + 1) - __ldg(borders + j));
      if (d > best) { best = d; bj = j; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
      if (ob > best || (ob == best && oj < bj)) { best = ob; bj = oj; }
    }
    __syncthreads();
    if ((t & 31) == 0) { sc->f[t >> 5] = best; sc->i[t >> 5] = bj; }
    __syncthreads();
    if (t == 0) {
      for (int w = 1; w < nt / 32; ++w)
        if (sc->f[w] > best || (sc->f[w] == best && sc->i[w] < bj)) { best = sc->f[w]; bj = sc->i[w]; }
      if (bj >= K) bj = 0;                              // all-NaN row
      mode[s] = 0.5f * (__ldg(borders + bj) + __ldg(borders + bj + 1));
    }
  }
  if (median || quant) {
    block_exclusive_scan(acc, K, pre, sc);             // pre[j+1] = c_j
    const int n_all = (median ? 1 : 0) + (quant ? n_q : 0);
    for (int qi = t; qi < n_all; qi += nt) {
      const bool is_median = median && qi == 0;
      const int qk = median ? qi - 1 : qi;
      const double q = is_median ? 0.5 : (double)__ldg(quantiles + qk);
      int lo = 0, hi = K - 1;                          // first j with c_j >= q, clamped to K-1
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (pre[mid + 1] >= q) hi = mid; else lo = mid + 1;
      }
      const int j = lo;
      const double pj = (double)acc[j];
      double r = pj > 0.0 ? (q - pre[j]) / pj : 1.0;
      r = fmin(fmax(r, 0.0), 1.0);
      const double g0 = __ldg(borders + j), g1 = __ldg(borders + j + 1), w = g1 - g0;
      double v;
      if (j == 0) v = g1 - w * 1.41421356237309504880 * erfinv(1.0 - r);
      else if (j == K - 1) v = g0 + w * 1.41421356237309504880 * erfinv(r);
      else v = g0 + r * w;
      if (is_median) median[s] = (float)v;
      else quant[(long long)qk * S + s] = (float)v;
    }
  }
}

// one instantiation each: MMPFN_OPT_IN_SMEM keeps its "done" flag per expansion
template <bool kTasks>
int launch_tail(const float* logits, const float* const* task_logits, const int32_t* row_offset, int n_tasks,
                int n_est, int S, int K, const int32_t* src_bucket, const float* src_share, const uint8_t* cancel,
                const float* borders, float temperature, int avg_before, const float* quantiles, int n_q, float* mean,
                float* median, float* mode, float* quant, float* log_prob, cudaStream_t st) {
  MMPFN_OPT_IN_SMEM(bar_tail_kernel<kTasks>, tail_smem_bytes(kTailMaxK));
  const int threads = K <= 1024 ? 128 : 512;
  bar_tail_kernel<kTasks><<<S, threads, tail_smem_bytes(K), st>>>(
      logits, n_est, S, K, src_bucket, src_share, cancel, borders, temperature,
      avg_before, quantiles, n_q, mean, median, mode, quant, log_prob, task_logits, row_offset, n_tasks);
  return count_launch();
}

}  // namespace

int launch_bar_tail(const float* logits, const float* const* task_logits, const int32_t* row_offset, int n_tasks,
                    int n_est, int S, int K, const int32_t* src_bucket, const float* src_share, const uint8_t* cancel,
                    const float* borders, float temperature, int avg_before, const float* quantiles, int n_q,
                    float* mean, float* median, float* mode, float* quant, float* log_prob, cudaStream_t st) {
  if (K > kTailMaxK) {
    set_error("bar_tail: %d buckets exceed the %d the shared-memory layout holds", K, kTailMaxK);
    return MMPFN_EUNSUPPORTED;
  }
  return (task_logits ? launch_tail<true> : launch_tail<false>)(
      logits, task_logits, row_offset, n_tasks, n_est, S, K, src_bucket, src_share, cancel, borders, temperature,
      avg_before, quantiles, n_q, mean, median, mode, quant, log_prob, st);
}

}  // namespace mmpfn
