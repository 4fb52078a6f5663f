// kernels_stem.cu — tabular / label / image-token stem and the probability tail.
// All of it is row-count-bound elementwise or tiny-reduction work (HBM-bound): coalesced accesses
// along the embedding dimension, block reductions in fp64 for the column statistics.
#include <math_constants.h>

#include "common.cuh"

namespace mmpfn {

namespace {

__device__ __forceinline__ void st_bf16(uint16_t* p, float v) {
  __nv_bfloat16 b = __float2bfloat16_rn(v);
  *p = *reinterpret_cast<uint16_t*>(&b);
}
__device__ __forceinline__ float nan_max(float a, float b) {   // torch.maximum: NaN propagates
  return (isnan(a) || isnan(b)) ? CUDART_NAN_F : fmaxf(a, b);
}
__device__ __forceinline__ float nan_min(float a, float b) {
  return (isnan(a) || isnan(b)) ? CUDART_NAN_F : fminf(a, b);
}
__device__ __forceinline__ float soft_clip(float x, float lo, float hi) {   // encoders.py:160-161
  x = nan_max(-logf(1.0f + fabsf(x)) + lo, x);
  return nan_min(logf(1.0f + fabsf(x)) + hi, x);
}
__device__ __forceinline__ float fill_bad(float x, float fill) {            // encoders.py:488-491
  return (isnan(x) || isinf(x)) ? fill : x;
}
__device__ __forceinline__ float clip100(float v) {                         // torch.clip keeps NaN
  return isnan(v) ? v : fminf(fmaxf(v, -100.f), 100.f);
}

// block-wide sum of two doubles (256 threads); result broadcast to every thread
__device__ void block_sum2(double& a, double& b, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) { sh[warp] = a; sh[8 + warp] = b; }
  __syncthreads();
  a = 0; b = 0;
  for (int w = 0; w < 8; ++w) { a += sh[w]; b += sh[8 + w]; }
}

// block-wide "any thread saw a difference"
__device__ bool block_any(int pred, int* flag) {
  if (threadIdx.x == 0) *flag = 0;
  __syncthreads();
  if (pred) atomicOr(flag, 1);
  __syncthreads();
  const bool r = *flag != 0;
  __syncthreads();
  return r;
}

// NaN-aware statistics over the first n rows of value(i): encoders.py:17-34 (`torch_nanmean`:
// sum / max(count,1)) and :37-50 (`torch_nanstd`: mean = sum/count, sqrt(nansum((mean-x)^2)/(count-1))).
template <typename Fn>
__device__ void nan_mean_std(Fn value, int n, float& mean_clip, float& stdv, double* sh) {
  double s = 0, c = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = value(i);
    if (!isnan(v)) { s += (double)v; c += 1.0; }
  }
  block_sum2(s, c, sh);
  const float mean_f = (float)(s / c);                         // NaN when count == 0, as sum/num is
  mean_clip = (float)(s / fmax(c, 1.0));
  double q = 0, unused = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float d = mean_f - value(i);
    d *= d;
    if (!isnan(d)) q += (double)d;                             // nansum
  }
  block_sum2(q, unused, sh);
  stdv = (float)sqrt(q / (c - 1.0));
}

// One CTA per (group g, estimator b).  Reference: RemoveEmptyFeaturesEncoderStep (encoders.py:496-527),
// NanHandlingEncoderStep._fit (:453-461), InputNormalizationEncoderStep._fit (:702-735),
// VariableNumFeaturesEncoderStep._fit (:608-619).
// n_rows / n_train_b (or NULL): entry b's own row counts; its rows are the first n_rows[b] of its S-row block.
__global__ void __launch_bounds__(256) tab_fit_kernel(const float* __restrict__ x, int S_alloc, int F, int fpg,
                                                      int n_train_all, float n_sigma, float* __restrict__ stats_all,
                                                      int G, const int* __restrict__ n_rows,
                                                      const int* __restrict__ n_train_b) {
  __shared__ double sh[16];
  __shared__ int s_flag;
  const int b = blockIdx.y, g = blockIdx.x;
  const TabStatsLayout L{G * fpg, G};
  float* st = stats_all + (long long)b * L.total();
  const float* xb = x + (long long)b * S_alloc * F;
  const int S = n_rows ? n_rows[b] : S_alloc;
  const int n_train = n_train_b ? n_train_b[b] : n_train_all;

  // 1. which source columns of this group vary over ALL rows (encoders.py:515)
  int kept[8];
  int n_kept = 0;
  for (int j = 0; j < fpg; ++j) {
    const int col = g * fpg + j;
    if (col >= F) continue;                                    // zero padding column (transformer.py:630-648)
    const float x0 = xb[col];
    int diff = 0;
    for (int i = 1 + threadIdx.x; i < S; i += blockDim.x) diff |= !(xb[(long long)i * F + col] == x0);
    if (block_any(diff, &s_flag)) kept[n_kept++] = col;        // NaN != NaN, so a NaN column is "kept"
  }

  int n_used = 0;
  for (int j = 0; j < fpg; ++j) {
    const int slot = g * fpg + j;
    const int col = j < n_kept ? kept[j] : -1;                 // kept features first (encoders.py:113-126)
    float fill = 0.f, lo = 0.f, hi = 0.f, mean = 0.f, stdv = 1e-20f;
    bool slot_varies = false;
    if (col >= 0) {
      auto raw = [&](int i) { return xb[(long long)i * F + col]; };
      // 2. NaN-fill value: torch.nanmean over train rows (encoders.py:461) — NaN skipped, inf kept
      {
        double s = 0, c = 0;
        for (int i = threadIdx.x; i < n_train; i += blockDim.x) {
          const float v = raw(i);
          if (!isnan(v)) { s += (double)v; c += 1.0; }
        }
        block_sum2(s, c, sh);
        fill = (float)(s / c);
      }
      auto x1 = [&](int i) { return fill_bad(raw(i), fill); };
      // 3. two-pass n_sigma bounds (encoders.py:145-158); n_sigma <= 0 or inf = step switched off
      //    (InferenceConfig.remove_outliers False, model/config.py:43): bounds at -inf/+inf are a no-op
      if (n_sigma > 0.f && !isinf(n_sigma)) {
        float mu, sd;
        nan_mean_std(x1, n_train, mu, sd, sh);
        float cut = sd * n_sigma;
        const float lo1 = mu - cut, hi1 = mu + cut;
        auto x1m = [&](int i) { const float v = x1(i); return (v > hi1 || v < lo1) ? CUDART_NAN_F : v; };
        nan_mean_std(x1m, n_train, mu, sd, sh);
        cut = sd * n_sigma;
        lo = mu - cut;
        hi = mu + cut;
      } else {
        lo = -CUDART_INF_F;
        hi = CUDART_INF_F;
      }
      // 4. z-norm statistics of the soft-clipped train rows (encoders.py:81-88)
      const float lo2 = lo, hi2 = hi;
      auto x2 = [&](int i) { return soft_clip(x1(i), lo2, hi2); };
      nan_mean_std(x2, n_train, mean, stdv, sh);
      stdv += 1e-20f;
      if (n_train == 1) stdv = 1.0f;
      // 5. does the normalised column vary over ALL rows (encoders.py:615)
      const float m2 = mean, s2 = stdv;
      auto x3 = [&](int i) { return clip100((x2(i) - m2) / s2); };
      const float v0 = x3(0);
      int diff = 0;
      for (int i = 1 + threadIdx.x; i < S; i += blockDim.x) diff |= !(x3(i) == v0);
      slot_varies = block_any(diff, &s_flag);
    } else {
      // an empty slot is the zero column select_features pads the group with (encoders.py:113-126), and the steps
      // above see it as such: fill 0, bounds 0, z-norm mean 0 / std 1e-20 (n_train == 1: std 1 and, with the outlier
      // step on, NaN bounds from the NaN std of one row).  Its normalised values are 0, or NaN with NaN bounds; NaN
      // values count as varying (encoders.py:615)
      if (!(n_sigma > 0.f && !isinf(n_sigma))) {
        lo = -CUDART_INF_F;
        hi = CUDART_INF_F;
      } else if (n_train == 1) {
        lo = hi = CUDART_NAN_F;
      }
      if (n_train == 1) stdv = 1.0f;
      slot_varies = isnan(lo) && S > 1;
    }
    if (slot_varies) ++n_used;
    if (threadIdx.x == 0) {
      st[L.src() + slot] = (float)col;
      st[L.fill() + slot] = fill;
      st[L.lo() + slot] = lo;
      st[L.hi() + slot] = hi;
      st[L.mean() + slot] = mean;
      st[L.stdv() + slot] = stdv;
    }
  }
  if (threadIdx.x == 0) st[L.scale() + g] = sqrtf((float)fpg / (float)max(n_used, 1));   // encoders.py:639-644
}

// One CTA (192 threads = embedding dim) per (row s, estimator b): writes all T tokens of the row.
__global__ void __launch_bounds__(kE) stem_tokens_kernel(
    const float* __restrict__ x, const float* __restrict__ stats_all, const float* __restrict__ img_tok,
    const float* __restrict__ y, const float* __restrict__ y_mean, const uint64_t* __restrict__ y_mask,
    const float* __restrict__ pos_emb, const float* __restrict__ enc_w, const float* __restrict__ yenc_w,
    const float* __restrict__ yenc_b, int S, int F, int fpg, int G, int H_img, long long x_bstride,
    long long y_bstride, long long img_bstride, float* __restrict__ state, uint16_t* __restrict__ state_bf,
    int32_t* __restrict__ nan_flag, const long long* __restrict__ img_off, const int* __restrict__ n_rows) {
  const int e = threadIdx.x;
  const long long s = blockIdx.x;
  const int b = blockIdx.y;
  const int T = G + H_img + 1;
  const TabStatsLayout L{G * fpg, G};
  const float* st = stats_all ? stats_all + (long long)b * L.total() : nullptr;
  const long long row = (long long)b * S + s;
  float* out = state + row * T * kE;
  uint16_t* outb = state_bf ? state_bf + row * T * kE : nullptr;
  if (n_rows && s >= n_rows[b]) {          // a pad row of entry b: all zeros (no positional embedding, no NaN test)
    for (int t = 0; t < T; ++t) {
      out[(long long)t * kE + e] = 0.f;
      if (outb) outb[(long long)t * kE + e] = 0;
    }
    return;
  }
  bool bad = false;
  auto emit = [&](int t, float v) {
    out[(long long)t * kE + e] = v;
    if (outb) st_bf16(outb + (long long)t * kE + e, v);
    bad |= isnan(v);
  };
  // tabular groups: transform (encoders.py:480-493, :761-780, :639-655) + Linear(2*fpg -> E) (:422-425).
  // The per-cell transform (NaN/inf fill, soft clip with its logarithms, z-norm) is the same for all 192
  // embedding columns: one thread per cell computes (value, indicator) into shared memory, then every
  // thread only does the 2*fpg FMAs of its column.
  if (G > 0) {
    __shared__ float cell_v[1024], cell_i[1024];                 // G * fpg <= 1024 cells per row (checked on launch)
    for (int slot = e; slot < G * fpg; slot += kE) {
      const int col = (int)st[L.src() + slot];
      // an empty slot (col < 0) is a zero column with its own statistics (tab_fit_kernel): it transforms to 0, or to
      // NaN where those statistics are NaN
      const float raw = col >= 0 ? x[b * x_bstride + s * F + col] : 0.f;
      const float ind = isnan(raw) ? -2.0f : (isinf(raw) ? (raw > 0 ? 2.0f : 4.0f) : 0.0f);
      float t1 = fill_bad(raw, st[L.fill() + slot]);
      t1 = soft_clip(t1, st[L.lo() + slot], st[L.hi() + slot]);
      t1 = clip100((t1 - st[L.mean() + slot]) / st[L.stdv() + slot]);
      cell_v[slot] = t1 * st[L.scale() + slot / fpg];
      cell_i[slot] = ind;
    }
    __syncthreads();
    float we[8];
    for (int j = 0; j < 2 * fpg; ++j) we[j] = enc_w[e * 2 * fpg + j];
    for (int g = 0; g < G; ++g) {
      float acc = 0.f;
      for (int j = 0; j < fpg; ++j) {
        acc = fmaf(cell_v[g * fpg + j], we[j], acc);
        acc = fmaf(cell_i[g * fpg + j], we[fpg + j], acc);
      }
      emit(g, acc + pos_emb[g * kE + e]);
    }
  }
  // image / text tokens appended after the tabular ones (transformer.py:768, :1038)
  // (img_bstride = 0: one set of tokens shared by the B estimators of a task; otherwise one per batch entry)
  for (int h = 0; h < H_img; ++h)
    emit(G + h, img_tok[(img_off ? img_off[b] : b * img_bstride) + ((long long)s * H_img + h) * kE + e] +
                    pos_emb[(G + h) * kE + e]);
  // y token, last (encoders.py:480-493 indicator/fill, :961-964 ordinal rank, :422-425 Linear(2 -> E) + b)
  {
    float yy = y[b * y_bstride + s];
    const float ind = isnan(yy) ? -2.0f : 0.0f;
    if (isnan(yy)) yy = y_mean[b];
    const uint64_t mask = y_mask[b];
    float val = yy;                       // regression checkpoints (bit 63): the target value itself, no rank step
    if (!(mask >> 63)) {
      int rank = 0;
      for (int c = 0; c < 63; ++c) rank += (((mask >> c) & 1ull) && ((float)c < yy)) ? 1 : 0;
      val = (float)rank;
    }
    emit(T - 1, fmaf(val, yenc_w[e * 2], fmaf(ind, yenc_w[e * 2 + 1], yenc_b[e])));
  }
  if (bad) atomicOr(nan_flag, 1);
}

// CAP attention core (transformer.py:81-85, nn.MultiheadAttention with Hc heads): one CTA per
// (row s, head hh); k/v of that head staged in shared memory; one warp per learned query.
//   kv [S][n_kv][2E] (k | v, already projected), q [Hc][E] (already projected), out [S][Hc][E]
__global__ void __launch_bounds__(128) cap_attn_kernel(const float* __restrict__ kv, const float* __restrict__ q,
                                                       int n_kv, int Hc, float* __restrict__ out) {
  extern __shared__ float sm[];
  const int hd = kE / Hc, P = hd + 1;
  float* ks = sm;                  // [n_kv][hd+1]
  float* vs = ks + n_kv * P;       // [n_kv][hd+1]
  float* ps = vs + n_kv * P;       // [4][n_kv]
  const long long s = blockIdx.x;
  const int hh = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* base = kv + s * n_kv * (2 * kE) + hh * hd;
  for (int i = threadIdx.x; i < n_kv * hd; i += blockDim.x) {
    const int j = i / hd, d = i % hd;
    ks[j * P + d] = base[(long long)j * 2 * kE + d];
    vs[j * P + d] = base[(long long)j * 2 * kE + kE + d];
  }
  __syncthreads();
  const float scale = rsqrtf((float)hd);
  float* pw = ps + warp * n_kv;
  for (int qi = warp; qi < Hc; qi += 4) {
    const float* qv = q + qi * kE + hh * hd;
    float mx = -INFINITY;
    for (int j = lane; j < n_kv; j += 32) {
      float a = 0.f;
      for (int d = 0; d < hd; ++d) a = fmaf(qv[d], ks[j * P + d], a);
      a *= scale;
      pw[j] = a;
      mx = fmaxf(mx, a);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < n_kv; j += 32) {
      const float ev = expf(pw[j] - mx);
      pw[j] = ev;
      sum += ev;
    }
    sum = warp_sum(sum);
    __syncwarp();
    for (int d = lane; d < hd; d += 32) {
      float o = 0.f;
      for (int j = 0; j < n_kv; ++j) o = fmaf(pw[j], vs[j * P + d], o);
      out[(s * Hc + qi) * kE + hh * hd + d] = o / sum;
    }
    __syncwarp();
  }
}

// out = LN(o; gamma, beta) + ffn   (transformer.py:86), one warp per 192-wide row
__global__ void __launch_bounds__(256) cap_combine_kernel(const float* __restrict__ o, const float* __restrict__ ffn,
                                                          const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, long long rows,
                                                          float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  float v[6];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    v[i] = o[row * kE + lane + 32 * i];
    s += v[i];
  }
  const float mean = warp_sum(s) * (1.0f / kE);
  float qv = 0.f;
#pragma unroll
  for (int i = 0; i < 6; ++i) qv = fmaf(v[i] - mean, v[i] - mean, qv);
  const float rstd = rsqrtf(warp_sum(qv) * (1.0f / kE) + kLnEps);
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const int e = lane + 32 * i;
    out[row * kE + e] = fmaf((v[i] - mean) * rstd, gamma[e], beta[e]) + ffn[row * kE + e];
  }
}

// MoE (transformer.py:112-125): tok[s][h][:] *= softmax(gate_logits[s][:])[h]
__global__ void moe_gate_scale_kernel(const float* __restrict__ gate_logits, float* __restrict__ tok, int S,
                                      int Hm) {
  const long long s = blockIdx.x;
  float mx = -INFINITY;
  for (int h = 0; h < Hm; ++h) mx = fmaxf(mx, gate_logits[s * Hm + h]);
  float sum = 0.f;
  for (int h = 0; h < Hm; ++h) sum += expf(gate_logits[s * Hm + h] - mx);
  for (int i = threadIdx.x; i < Hm * kE; i += blockDim.x) {
    const int h = i / kE;
    tok[s * Hm * kE + i] *= expf(gate_logits[s * Hm + h] - mx) / sum;
  }
}

// Probability tail (classifier.py:544-576).  One thread per test row; classes <= 64.
__global__ void proba_tail_kernel(const float* __restrict__ logits, const int32_t* __restrict__ perm,
                                  const float* __restrict__ prior, int n_est, int S, int n_out, int n_classes,
                                  float temperature, int avg_before, float* __restrict__ proba) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  float acc[64];
  for (int c = 0; c < n_classes; ++c) acc[c] = 0.f;
  for (int e = 0; e < n_est; ++e) {
    const float* lg = logits + ((long long)e * S + s) * n_out;
    float v[64];
    for (int c = 0; c < n_classes; ++c) {
      const float z = lg[perm[e * n_classes + c]];
      v[c] = (temperature != 1.0f) ? z / temperature : z;
    }
    if (!avg_before) {
      float mx = -INFINITY;
      for (int c = 0; c < n_classes; ++c) mx = fmaxf(mx, v[c]);
      float sum = 0.f;
      for (int c = 0; c < n_classes; ++c) { v[c] = expf(v[c] - mx); sum += v[c]; }
      for (int c = 0; c < n_classes; ++c) v[c] /= sum;
    }
    for (int c = 0; c < n_classes; ++c) acc[c] += v[c];
  }
  for (int c = 0; c < n_classes; ++c) acc[c] /= (float)n_est;
  if (avg_before) {
    float mx = -INFINITY;
    for (int c = 0; c < n_classes; ++c) mx = fmaxf(mx, acc[c]);
    float sum = 0.f;
    for (int c = 0; c < n_classes; ++c) { acc[c] = expf(acc[c] - mx); sum += acc[c]; }
    for (int c = 0; c < n_classes; ++c) acc[c] /= sum;
  }
  if (prior) {                                                 // classifier.py:563-566
    float sum = 0.f;
    for (int c = 0; c < n_classes; ++c) { acc[c] *= prior[c]; sum += acc[c]; }
    for (int c = 0; c < n_classes; ++c) acc[c] /= sum;
  }
  float sum = 0.f;                                             // classifier.py:576
  for (int c = 0; c < n_classes; ++c) sum += acc[c];
  for (int c = 0; c < n_classes; ++c) proba[s * n_classes + c] = acc[c] / sum;
}
}  // namespace

int launch_tab_fit(const float* x, int B, int S, int F, int fpg, int n_train, float n_sigma, float* stats,
                   cudaStream_t st, const int* n_rows, const int* n_train_b) {
  const int G = (F + fpg - 1) / fpg;
  if (G <= 0 || B <= 0) return MMPFN_OK;
  if (fpg > 8) { set_error("features_per_group %d > 8", fpg); return MMPFN_EUNSUPPORTED; }
  tab_fit_kernel<<<dim3(G, B), 256, 0, st>>>(x, S, F, fpg, n_train, n_sigma, stats, G, n_rows, n_train_b);
  return count_launch();
}

int launch_stem_tokens(const mmpfn_geometry* g, const mmpfn_weights* w, const float* x, const float* stats,
                       const float* img_tok, const float* y, const float* y_mean, const uint64_t* y_mask,
                       const float* pos_emb, int B, int S, int F, int H_img, long long x_bstride, long long y_bstride,
                       long long img_bstride, float* state_f32, uint16_t* state_bf16, int32_t* nan_flag, cudaStream_t st,
                       const long long* img_off, const int* n_rows) {
  const int fpg = g->features_per_group;
  const int G = x ? (F + fpg - 1) / fpg : 0;
  if (fpg > 4) { set_error("features_per_group %d > 4", fpg); return MMPFN_EUNSUPPORTED; }
  if (G * fpg > 1024) { set_error("stem_tokens: %d feature cells per row exceed the 1024 the kernel stages", G * fpg); return MMPFN_EUNSUPPORTED; }
  stem_tokens_kernel<<<dim3(S, B), kE, 0, st>>>(x, stats, img_tok, y, y_mean, y_mask, pos_emb, w->enc_w, w->yenc_w,
                                               w->yenc_b, S, F, fpg, G, H_img, x_bstride, y_bstride, img_bstride, state_f32, state_bf16,
                                               nan_flag, img_off, n_rows);
  return count_launch();
}

int launch_cap_attn(const float* kv, const float* q, int S, int n_kv, int Hc, float* out, cudaStream_t st) {
  const int hd = kE / Hc;
  const size_t smem = (size_t)(2 * n_kv * (hd + 1) + 4 * n_kv) * sizeof(float);
  if (smem > 200 * 1024) {
    set_error("CAP: %d source tokens x head_dim %d exceed the shared-memory tile", n_kv, hd);
    return MMPFN_EUNSUPPORTED;
  }
  if (smem > 48 * 1024 &&
      cudaFuncSetAttribute(cap_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    set_error("CAP: cannot opt in to %zu bytes of shared memory: %s", smem, cudaGetErrorString(cudaGetLastError()));
    return MMPFN_ECUDA;
  }
  cap_attn_kernel<<<dim3(S, Hc), 128, smem, st>>>(kv, q, n_kv, Hc, out);
  return count_launch();
}

int launch_cap_combine(const float* o, const float* ffn, const float* gamma, const float* beta, long long rows,
                       float* out, cudaStream_t st) {
  cap_combine_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(o, ffn, gamma, beta, rows, out);
  return count_launch();
}

int launch_moe_gate_scale(const float* gate_logits, float* tok, int S, int Hm, cudaStream_t st) {
  moe_gate_scale_kernel<<<S, 256, 0, st>>>(gate_logits, tok, S, Hm);
  return count_launch();
}

int launch_proba_tail(const float* logits, const int32_t* perm, const float* prior, int n_est, int S, int n_out,
                      int n_classes, float temperature, int avg_before, float* proba, cudaStream_t st) {
  if (n_classes > 64 || n_classes > n_out) { set_error("proba tail: n_classes %d", n_classes); return MMPFN_EINVAL; }
  proba_tail_kernel<<<(S + 127) / 128, 128, 0, st>>>(logits, perm, prior, n_est, S, n_out, n_classes, temperature,
                                                    avg_before, proba);
  return count_launch();
}

}  // namespace mmpfn
