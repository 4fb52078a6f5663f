/*
 * mmpfn_b200.h — C ABI of libmmpfn_b200.so: the sm_100a implementation of MMPFN's in-context
 * inference hot path (TabPFN-v2 PerFeatureTransformer forward + image/text token stem).
 *
 * The reference is pure Python/PyTorch and has no FFI of its own; the boundary this library
 * replaces is the model call of the inference engine,
 *     mmpfn/models/mmpfn/inference.py:343-348   self.model(None, X_full, image_full, y_train, ...)
 * i.e. PerFeatureTransformer._forward (mmpfn/models/mmpfn/model/transformer.py:555-867), plus the
 * probability tail of MMPFNClassifier.predict_proba (mmpfn/models/mmpfn/classifier.py:544-576).
 * Each entry point below cites the reference lines whose work it performs.  INTEGRATION.md shows
 * the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host; buffers are owned by the
 *    caller (torch allocates them); nothing is allocated or freed inside the library;
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs no host
 *    synchronisation, and returns 0 on success or a negative MMPFN_E* code; mmpfn_last_error()
 *    returns a thread-local message for the last failure;
 *  - calls on different streams of one device may overlap (buffers of their own, one workspace per
 *    call in flight); tools/concurrency_probe.py runs every pair and chains of the layer kernels
 *    on two streams against their results alone;
 *  - there is NO CPU fallback: on a machine without an sm_100 device every compute entry point
 *    returns MMPFN_ENODEVICE;
 *  - tensors are dense, row-major, innermost dimension last, in the layouts stated per call;
 *  - `precision`: MMPFN_F32 (FFMA kernels, the 1e-5 parity mode), MMPFN_BF16 (tcgen05/TMEM/TMA
 *    kernels: bf16 MMA operands, fp32 accumulation, fp32 softmax/LayerNorm statistics and an fp32
 *    residual stream) or MMPFN_F16 (the same kernels with fp16 MMA operands: 3 more significand bits than
 *    bf16; every fp32 -> fp16 rounding saturates at +-65504 instead of overflowing to inf).  In MMPFN_F16 every
 *    argument or buffer whose name says bf16 (state_bf16, the K/V context, the layout comments below) holds
 *    fp16 values instead, in the same layout and size; the weights come from mmpfn_weights.layers_f16.  The stem
 *    has no fp16 form: the layer passes write the fp16 shadow of the fp32 state themselves.  The *_f16 building
 *    blocks below are the fp16 twins of the *_bf16 ones.
 */
#ifndef MMPFN_B200_H
#define MMPFN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMPFN_ABI_VERSION 2

enum { MMPFN_OK = 0, MMPFN_EINVAL = -1, MMPFN_ENODEVICE = -2, MMPFN_ECUDA = -3, MMPFN_EUNSUPPORTED = -4 };
enum { MMPFN_F32 = 0, MMPFN_BF16 = 1, MMPFN_F16 = 2 };
enum { MMPFN_MIXER_NONE = 0, MMPFN_MIXER_MGM = 1, MMPFN_MIXER_MGM_CAP = 2, MMPFN_MIXER_MOE = 3 };

/* Geometry of the checkpoint (reference model/config.py:18-83, model/loading.py:470-538).
 * Supported: emsize 192, nhead 6 (d_k 32), nhid 768, features_per_group 1 or 2. */
typedef struct mmpfn_geometry {
  int32_t emsize, nhead, nhid, nlayers, n_out, features_per_group;
  int32_t img_dim, mgm_heads, cap_heads, mixer_type;
} mmpfn_geometry;

/* Repacked weights (device pointers).  Layouts are produced by multimodalpfn_b200/weights.py from a
 * reference state_dict (SURVEY.md Appendix B).  All matrices are "W[N][K]" (output-major), so a
 * projection is out[n] = sum_k in[k] * W[n][k].
 *
 * layers_f32 / layers_bf16 / layers_f16: nlayers consecutive blocks of
 *     feat_wqkv [3*E][E] | feat_wout [E][E] | item_wqkv [3*E][E] | item_wout [E][E]
 *     | mlp_w1 [nhid][E] | mlp_w2 [E][nhid]
 * where wqkv rows are ordered (j in q,k,v; head; d) exactly like the reference `_w_qkv [3,H,D,E]`
 * (model/multi_head_attention.py:216-260) and wout[e][h*D+d] = reference `_w_out[h][d][e]`. */
typedef struct mmpfn_weights {
  const float*    layers_f32;
  const uint16_t* layers_bf16;      /* may be NULL when only MMPFN_F32 is used */
  const float* enc_w;               /* [E][2*fpg]   encoder.5.layer.weight (no bias) */
  const float* yenc_w;              /* [E][2]       y_encoder.2.layer.weight */
  const float* yenc_b;              /* [E] */
  const float* dec_w1;              /* [nhid][E]    decoder_dict.standard.0 */
  const float* dec_b1;              /* [nhid] */
  const float* dec_w2;              /* [n_out][nhid] decoder_dict.standard.2 */
  const float* dec_b2;              /* [n_out] */
  /* image / text stem; NULL when mixer_type == MMPFN_MIXER_NONE */
  const float* mgm_w1;              /* [Hm*img][img]  LN affine folded in; GLU halves interleaved:
                                       row h*img + 2*c = value c, row h*img + 2*c+1 = gate c
                                       (MoE: [Hm*img/2][img], plain order) */
  const float* mgm_b1;              /* [Hm*img]       (MoE: [Hm*img/2]) */
  const float* mgm_w2;              /* [Hm][E][img/2] */
  const float* mgm_b2;              /* [Hm][E] */
  const float* moe_gate_w;          /* [Hm][img]   MoE only */
  const float* moe_gate_b;          /* [Hm] */
  const float* cap_knorm_w;         /* [E] */
  const float* cap_knorm_b;         /* [E] */
  const float* cap_q;               /* [Hc][E]  in_proj_q(q_proj(q_norm(queries))) precomputed (row independent) */
  const float* cap_wkv;             /* [2*E][E] in_proj rows E..3E */
  const float* cap_bkv;             /* [2*E] */
  const float* cap_wo;              /* [E][E] */
  const float* cap_bo;              /* [E] */
  const float* cap_onorm_w;         /* [E] */
  const float* cap_onorm_b;         /* [E] */
  const float* cap_f1_w;            /* [2E][E] */
  const float* cap_f1_b;            /* [2E] */
  const float* cap_f2_w;            /* [E][2E] */
  const float* cap_f2_b;            /* [E] */
  /* optional bf16 copy of mgm_w1 (MGM / MGM+CAP): when set and mgm_heads >= 32, the MGM gated projection — the stem's
   * one large GEMM, M0 x (Hm*img) x img — runs on tcgen05 with bf16 operands and fp32 accumulation; NULL (or fewer
   * heads) keeps it on the fp32 FFMA path (the 1e-5 parity mode) */
  const uint16_t* mgm_w1_bf16;
  /* fp16 copy of the layer blocks, layout of layers_bf16; read only under MMPFN_F16 (appended: callers that never
   * pass MMPFN_F16 need not know the field) */
  const uint16_t* layers_f16;
} mmpfn_weights;

/* ---- introspection ------------------------------------------------------------------------- */
int         mmpfn_abi_version(void);
const char* mmpfn_last_error(void);
/* number of kernels this library has launched in the calling process (bench `gpu_launches`) */
int64_t     mmpfn_launch_count(void);
/* 1 if device `dev` is an sm_100 part this library can run on */
int         mmpfn_device_supported(int dev);

/* floats per layer block in mmpfn_weights.layers_* */
size_t mmpfn_layer_weight_elems(const mmpfn_geometry* g);

/* ---- stem ---------------------------------------------------------------------------------- */
/* Number of image tokens the mixer emits per row (transformer.py:294-301, :755-761). */
int mmpfn_image_tokens(const mmpfn_geometry* g, int n_tok);

/* size in floats of the statistics block mmpfn_stem_tab_fit writes for n_groups groups */
size_t mmpfn_tab_stats_elems(const mmpfn_geometry* g, int n_groups);

/* Tabular stem statistics — encoders.py:515 (constant-column mask over ALL rows),
 * :461 (NaN fill means, train rows), :133-162 (two-pass 12-sigma bounds), :53-99 (z-norm mean/std),
 * :615-619 (used-feature count).  x: [B][S][F] fp32 (NaN allowed); stats: [B][tab_stats_elems].
 * F is padded to a multiple of features_per_group internally (transformer.py:630-648). */
int mmpfn_stem_tab_fit(const mmpfn_geometry* g, const float* x, int B, int S, int F, int n_train,
                       float n_sigma, float* stats, void* stream);

/* Image/text mixer — transformer.py:33-48 (MGM), :60-88 (CAP), :91-128 (MoE).
 * img: [S][n_tok][img_dim] fp32 -> out: [S][H_img][E] fp32.  workspace: mmpfn_stem_image_ws_bytes. */
size_t mmpfn_stem_image_ws_bytes(const mmpfn_geometry* g, int S, int n_tok);
int mmpfn_stem_image(const mmpfn_geometry* g, const mmpfn_weights* w, const float* img, int S, int n_tok,
                     float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Token assembly — transformer.py:682-788: tabular groups (encoders.py:382-425 after the fitted
 * transforms), image tokens, + positional embedding on every non-y token, y token last
 * (encoders.py:428-493, :949-974; rows with NaN label are test rows).
 *   x       [B][.][F] or NULL: S rows per estimator starting at x, estimators x_bstride elements apart
 *           (so the train rows and the test rows of one [B][S_full][F] table embed separately)
 *   stats   [B][tab_stats_elems] or NULL
 *   img_tok [S][H_img][E] or NULL: batch entry b reads img_tok + b * img_bstride (elements); img_bstride = 0
 *           = one set shared by the B estimators of a task (inference.py:272), S*H_img*E = one per entry
 *           (independent tasks packed on the batch axis)
 *   y       [B][.]: S labels per estimator, y_bstride apart (NaN = unlabeled test row)
 *   y_mean  [B], y_present_mask [B] (bit c set iff class c occurs among the train labels, c <= 62; bit 63 set =
 *   regression checkpoint: no class-rank step, the target value itself is embedded, model/loading.py:387-388)
 *   pos_emb [T-1][E]
 *   state_f32 [B][S][T][E] out; state_bf16 same shape, may be NULL.
 * nan_flag (int32, device): set to 1 if any produced value is NaN (transformer.py:727-731, :790-796). */
int mmpfn_stem_tokens(const mmpfn_geometry* g, const mmpfn_weights* w, const float* x, const float* stats,
                      const float* img_tok, const float* y, const float* y_mean, const uint64_t* y_present_mask,
                      const float* pos_emb, int B, int S, int F, int H_img, long long x_bstride, long long y_bstride, long long img_bstride,
                      float* state_f32, uint16_t* state_bf16, int32_t* nan_flag, void* stream);

/* ---- the 12 layers ------------------------------------------------------------------------- */
/* Bytes of the K/V context of n_train rows: per layer, head-0 keys and values of the item
 * attention for every (estimator, token column) — the reference's "first head only" cache
 * (multi_head_attention.py:328-336, :467-470) with a layer axis in front. */
size_t mmpfn_kv_bytes(const mmpfn_geometry* g, int B, int n_train, int T, int precision);

/* Whole passes through the 12 layers (layer.py:272-457), every precision; state is updated in place.
 *  - Train pass: every row is a train row (self-attention over items, all heads, layer.py:363-372); writes the
 *    head-0 K/V context of segment i to kv[i] when kv[i] != NULL.
 *  - Test pass: the item attention reads the cached head-0 K/V of the n_train train rows for all six query heads
 *    (layer.py:346-358, multi_head_attention.py:436-445); every kv[i] is required.
 * A call takes a list of estimator groups ("segments": same row count S, own batch B_i and token count T_i).  Their
 * states are laid back to back in one buffer — segment i occupies B_i*S*T_i token rows of 192, in list order —
 * and kv[i] is segment i's context, mmpfn_kv_bytes(B_i, n_train, T_i, precision).  One segment {B, T} is the plain
 * pass over a [B][S][T][E] state.  bf16: the sublayers that work on the flat token axis (QKV and output projections
 * + LayerNorm, MLP) launch once for all segments, the attentions per segment; fp32: one segment after another.
 * Every segment's result is that of a call over that segment alone.  state_bf16 is unused (may be NULL) in
 * MMPFN_F32.  MMPFN_F16: the call first writes the fp16 shadow of state_f32 into state_bf16 (an fp16 buffer of the
 * same size), then runs as MMPFN_BF16 does with fp16 operands; the K/V context is fp16 in the bf16 layout.
 * n_rows / n_ctx: per-entry row counts (device int32, see "per-entry row counts" below), or NULL = every entry
 * uses all S rows (and all n_train context rows).  With counts, entry b's item attention (layer.py:341-379) runs
 * over its own rows only. */
#define MMPFN_MAX_SEGMENTS 8
typedef struct mmpfn_segment {
  int32_t B, T;
} mmpfn_segment;
size_t mmpfn_layers_ragged_ws_bytes(const mmpfn_geometry* g, const mmpfn_segment* segs, int n_seg, int S, int precision);
int mmpfn_layers_train_ragged(const mmpfn_geometry* g, const mmpfn_weights* w, float* state_f32, uint16_t* state_bf16,
                              const mmpfn_segment* segs, int n_seg, int S, const int32_t* n_rows, int precision,
                              void* const* kv, void* workspace, size_t workspace_bytes, void* stream);
int mmpfn_layers_test_ragged(const mmpfn_geometry* g, const mmpfn_weights* w, float* state_f32, uint16_t* state_bf16,
                             const mmpfn_segment* segs, int n_seg, int S, int n_train, const int32_t* n_rows,
                             const int32_t* n_ctx, int precision, void* const* kv, void* workspace,
                             size_t workspace_bytes, void* stream);

/* The same passes over a RANGE of layers and with the K/V context addressed explicitly: what the multi-GPU
 * engine (multimodalpfn_b200/dist.py) needs to all-gather layer l's K/V under layers l+1.. and to let the test
 * pass read the gather buffer where the blocks land.  Per segment and layer the context block is
 *     K0 [c][T][Np][32]  then  V0^T [c][T][32][Np]      (bf16, Np = n_train rounded up to 64)
 * with c estimators back to back.  Train pass (train != 0): c = B, block of layer l written at
 * kv + l * layer_stride.  Test pass: estimator b of the segment = (rank b / slots, slot b % slots) lives in the block at
 * kv + l * layer_stride + rank * rank_stride with c = slots.  layer_stride 0 = blocks of consecutive layers are
 * adjacent; slots 0 = all B estimators in one block (rank_stride unused): then this is the bf16 pass of
 * mmpfn_layers_train_ragged / _test_ragged without counts.  bf16 only (there is no precision argument).
 * Layers [layer_begin, layer_end) run; the state is carried in state_f32 / state_bf16 between calls. */
typedef struct mmpfn_kv_segment {
  int32_t B, T;
  void* kv;
  int64_t layer_stride;   /* bytes */
  int32_t slots;
  int32_t seg_rows;       /* > 0: row-sharded context (below); 0: off */
  int64_t rank_stride;    /* bytes */
  /* Row-sharded context build (SURVEY.md section 8(f) rank 2): the train rows of ONE estimator batch are split over the
   * ranks, seg_rows rows per rank (a multiple of 48: key tiles then never straddle two ranks and are exactly the
   * tiles of the unsharded layout — results are bit-identical).  Every rank runs the row-wise sublayers on its own
   * rows; for the item attention its rows' K / V^T planes are written into chunk `rank` of the caller's gather buffers
   *     kg  [n_ranks][B*T*6][Sp][32]      vtg [n_ranks][B*T*6][32][Sp]      (Sp = S rounded up to 64, bf16;
   *     gather_stride bytes between chunks; pad rows must hold finite values: zero the buffers once)
   * in phase 1, the caller all-gathers both buffers, and in phase 2 the rank's queries attend to all n_rows_total
   * keys.  The head-0 context block of the layer (at kv + l * layer_stride, layout as above with c = B) holds this
   * rank's rows only; gathered over the ranks (chunks rank_stride apart) it is what the TEST pass reads when its
   * segment has seg_rows > 0: estimator b's keys = chunks 0..n_ranks-1, seg_rows rows each. */
  void* kg;
  void* vtg;
  int64_t gather_stride;  /* bytes */
  int32_t rank, n_ranks;
  int32_t n_rows_total;
  int32_t reserved;
} mmpfn_kv_segment;
/* phase: 0 = whole layers; 1 = layer `layer_begin` up to and including the item-attention QKV projection;
 * 2 = the rest of that layer (phases 1 / 2 need layer_end == layer_begin + 1). */
int mmpfn_layers_run(const mmpfn_geometry* g, const mmpfn_weights* w, float* state_f32, uint16_t* state_bf16,
                     const mmpfn_kv_segment* segs, int n_seg, int S, int n_train, int train, int layer_begin,
                     int layer_end, int phase, void* workspace, size_t workspace_bytes, void* stream);

/* ---- per-entry row counts ("ragged" passes) ------------------------------------------------------------------
 * Independent tasks of different sizes share one pass.  A batch ENTRY is one (task, estimator) pair; a pass has a
 * row capacity S (train pass: S train rows; test pass: S test rows against n_train context rows) and entry b uses
 * its first n_rows[b] rows (test pass: attends to its first n_ctx[b] context rows).  The counts are device int32
 * arrays with one element per entry (over all segments, in list order); NULL = every entry uses all rows.
 *
 * Pad-row contract: the rows between an entry's count and the capacity must be ZERO when a kernel reads them.
 * mmpfn_stem_tokens_ragged writes them as zeros, and the layers keep them exactly zero (no biases; LayerNorm of a
 * zero row, GELU(0), attention over zero tokens are zero; the item attention writes zeros for pad queries), so the
 * K/V rows a pad row produces are the zeros the TMA out-of-bounds fill gives an entry run alone: every entry's result
 * is bit-identical to a pass over that entry alone. */

/* mmpfn_stem_tab_fit (encoders.py:515, :461, :133-162, :53-99, :615-619) per entry: entry b's rows are the first
 * n_rows[b] rows of its S-row block of x, train rows (n_train[b] of them) first; its statistics are those of a call
 * over that entry alone (the reductions run in the same order). */
int mmpfn_stem_tab_fit_ragged(const mmpfn_geometry* g, const float* x, int B, int S, int F, const int32_t* n_rows,
                              const int32_t* n_train, float n_sigma, float* stats, void* stream);
/* mmpfn_stem_tokens (transformer.py:682-788) per entry: rows s >= n_rows[b] of entry b are written as all zeros (no
 * positional embedding, never a NaN flag; n_rows NULL = all S rows).  img_offset [B] (int64, elements; required with img_tok): entry b's
 * [S][H_img][E] image tokens start at img_tok + img_offset[b] (estimators of one task share one set). */
int mmpfn_stem_tokens_ragged(const mmpfn_geometry* g, const mmpfn_weights* w, const float* x, const float* stats,
                             const float* img_tok, const float* y, const float* y_mean, const uint64_t* y_present_mask,
                             const float* pos_emb, int B, int S, int F, int H_img, long long x_bstride,
                             long long y_bstride, const int64_t* img_offset, const int32_t* n_rows, float* state_f32,
                             uint16_t* state_bf16, int32_t* nan_flag, void* stream);

/* ---- decoder + probability tail ------------------------------------------------------------ */
/* transformer.py:392-396, :850-853: logits[b][s][:] = W2 gelu(W1 state[b][s][T-1] + b1) + b2.
 * state [B][S][T][E] -> logits [B][S][n_out]; hidden scratch [B*S][nhid] fp32. */
int mmpfn_decode(const mmpfn_geometry* g, const mmpfn_weights* w, const float* state_f32, int B, int S, int T,
                 float* hidden_scratch, float* logits, void* stream);

/* classifier.py:544-576: per estimator (slice to n_classes and divide by temperature iff
 * temperature != 1) -> gather class_perm -> softmax -> mean over estimators (or mean then softmax)
 * -> optional class-prior balancing -> renormalise.  logits [n_est][S][n_out]; class_perm
 * [n_est][n_classes] int32; class_prior [n_classes] or NULL; proba [S][n_classes]. */
int mmpfn_proba_tail(const float* logits, const int32_t* class_perm, const float* class_prior, int n_est, int S,
                     int n_out, int n_classes, float temperature, int average_before_softmax, float* proba,
                     void* stream);

/* Bar-distribution tail of the regressor (the reference's regressor.py predict: translate_probs_across_borders +
 * FullSupportBarDistribution mean / icdf / mode), one CTA per test row; only the requested outputs leave the row.
 *   logits     [n_est][S][K]   per-estimator logits over K buckets (what the decoder writes)
 *   src_bucket [n_est][K+1]    int32: for common border g_j, the bucket i of estimator e's own borders f_e with
 *                              f_e[i] <= g_j < f_e[i+1]; -1 below f_e[0], K at or above f_e[K]
 *   src_share  [n_est][K+1]    (g_j - f_e[i]) / (f_e[i+1] - f_e[i]) clamped to [0, 1] (unused for i = -1, K)
 *   cancel     [n_est][K]      uint8, nonzero = that bucket's logit is -inf; may be NULL
 *   borders    [K+1]           common borders G in target units, increasing
 *   quantiles  [n_q]           in (0, 1)
 *   mean, median, mode [S]; quant [n_q][S]; log_prob [S][K].  Every output may be NULL (not computed).
 * Per row s:
 *  1. z_e = logits[e][s] / temperature (as is when temperature == 1); cancelled buckets -inf; p_e = softmax(z_e);
 *     P_e(i) = sum_{k<i} p_e[k].
 *  2. C_e(j) = 0 for i = -1, 1 for i = K, else P_e(i) + p_e[i] * src_share[e][j] (i = src_bucket[e][j]);
 *     C_e(0) = 0, C_e(K) = 1; q_e[j] = max(C_e(j+1) - C_e(j), 0): estimator e's piecewise-linear CDF at G.
 *  3. P = mean_e q_e (average_before_softmax = 0) or softmax(mean_e log q_e) (= 1); log_prob = log P.
 *  4. w_j = G_{j+1} - G_j.  mean = sum_j P_j m_j, m_j = (G_j + G_{j+1}) / 2 inside, half-normal tails outside:
 *     m_0 = G_1 - w_0 sqrt(2/pi), m_{K-1} = G_{K-1} + w_{K-1} sqrt(2/pi).
 *  5. quantile q: c_j = sum_{i<=j} P_i, j = first index with c_j >= q (clamped to K-1), r = (q - c_{j-1}) / P_j
 *     clamped to [0, 1]: G_j + r w_j inside, G_1 - w_0 sqrt(2) erfinv(1 - r) in the left tail,
 *     G_{K-1} + w_{K-1} sqrt(2) erfinv(r) in the right tail.  median = the quantile at 0.5.
 *  6. mode = midpoint of the bucket with the largest P_j / w_j (lowest j on ties).
 * Prefix sums run in float64 (a bucket mass is a difference of two).  2 <= K <= 8192 (MMPFN_EUNSUPPORTED beyond:
 * the row's working set lives in shared memory). */
int mmpfn_bar_tail(const float* logits, int n_est, int S, int K, const int32_t* src_bucket, const float* src_share,
                   const uint8_t* cancel, const float* borders, float temperature, int average_before_softmax,
                   const float* quantiles, int n_q, float* mean, float* median, float* mode, float* quant,
                   float* log_prob, void* stream);

/* mmpfn_bar_tail over the rows of many tasks in one launch, one CTA per global row; steps 1-6 per row exactly as
 * mmpfn_bar_tail, with task t's own maps and borders (each task's G is in its own target units):
 *   logits     [n_tasks * n_est]  device array of pointers: logits[t * n_est + e] points to row 0 of task t's rows
 *                                 for estimator e, rows K floats apart (the decoder's per-entry outputs, in place)
 *   row_offset [n_tasks + 1]      int32 on the device: task t owns global rows [row_offset[t], row_offset[t+1])
 *   src_bucket, src_share [n_tasks][n_est][K+1];  cancel [n_tasks][n_est][K] or NULL;  borders [n_tasks][K+1]
 *   mean, median, mode [S_total]; quant [n_q][S_total]; log_prob [S_total][K], indexed by global row; any may be NULL.
 * K, n_est, the temperature, the averaging mode and the quantiles are shared by all tasks.  Preconditions the call
 * cannot check without a host sync: row_offset[0] == 0, row_offset is nondecreasing (a task may own no rows) and
 * row_offset[n_tasks] == S_total.  MMPFN_EINVAL / MMPFN_EUNSUPPORTED as mmpfn_bar_tail. */
int mmpfn_bar_tail_tasks(const float* const* logits, int n_tasks, int n_est, const int32_t* row_offset, int S_total,
                         int K, const int32_t* src_bucket, const float* src_share, const uint8_t* cancel,
                         const float* borders, float temperature, int average_before_softmax, const float* quantiles,
                         int n_q, float* mean, float* median, float* mode, float* quant, float* log_prob,
                         void* stream);

/* ---- building blocks exported for unit tests and profiling ---------------------------------- */
/* y = LayerNorm(x (+ res)) over `width` (192 or 768), eps 1e-5, optional affine (layer.py:40-64). */
int mmpfn_layernorm(const float* x, const float* res, const float* gamma, const float* beta, int rows, int width,
                    float* y_f32, uint16_t* y_bf16, void* stream);
/* out[M][N] = epi(A[M][K] W[N][K]^T + bias); epi: 0 none, 1 exact GELU.  fp32 FFMA kernel. */
int mmpfn_linear_f32(const float* A, const float* W, const float* bias, int M, int N, int K, int epi, float* out,
                     void* stream);
/* Same contract on the tcgen05 path: A, W bf16; out bf16. */
int mmpfn_linear_bf16(const uint16_t* A, const uint16_t* W, int M, int N, int K, int epi, uint16_t* out,
                      void* stream);

/* An attention output projection with its residual + LayerNorm (multi_head_attention.py:513-517,
 * layer.py:437-455), one persistent tcgen05 kernel, in place:
 *   state_f32 [M][192] <- LayerNorm(state_f32 + A W^T),  state_bf16 <- bf16(state_f32);  A [M][192], W [192][192] bf16. */
int mmpfn_linear_ln_bf16(const uint16_t* A, const uint16_t* W, int M, float* state_f32, uint16_t* state_bf16,
                         void* stream);
/* fp16 twin: A, W, state_f16 fp16 */
int mmpfn_linear_ln_f16(const uint16_t* A, const uint16_t* W, int M, float* state_f32, uint16_t* state_f16,
                        void* stream);

/* The QKV projection of the attention across items (multi_head_attention.py:430-434) with its scatter into
 * the layouts the item-attention kernel reads: state [B][S][T][192] bf16, w_qkv [n_proj*192][192] bf16
 * (n_proj = 3: q|k|v, the train pass; 1: q only, the test pass) ->
 *   q, k [B*T*nhead][S_pad][32],  vt [B*T*nhead][32][S_pad],  and, when given, the head-0 context
 *   k0 [B*T][S_pad][32], vt0 [B*T][32][S_pad] (multi_head_attention.py:328-336).  S_pad % 64 == 0. */
int mmpfn_item_qkv_bf16(const uint16_t* state_bf16, const uint16_t* w_qkv, int B, int S, int T, int S_pad, int n_proj,
                        uint16_t* q, uint16_t* k, uint16_t* vt, uint16_t* k0, uint16_t* vt0, void* stream);
/* fp16 twin: every 16-bit buffer fp16 */
int mmpfn_item_qkv_f16(const uint16_t* state_f16, const uint16_t* w_qkv, int B, int S, int T, int S_pad, int n_proj,
                       uint16_t* q, uint16_t* k, uint16_t* vt, uint16_t* k0, uint16_t* vt0, void* stream);

/* The MLP sublayer alone (mlp.py:93-138 + layer.py:437-455), one fused tcgen05 kernel, in place:
 *   state_f32 [M][192] <- LayerNorm(state_f32 + W2 gelu(W1 state_bf16)),  state_bf16 <- bf16(state_f32)
 * w1 [768][192], w2 [192][768] bf16 (the reference's linear1.weight / linear2.weight). */
int mmpfn_mlp_bf16(float* state_f32, uint16_t* state_bf16, const uint16_t* w1, const uint16_t* w2, int M,
                   void* stream);
/* fp16 twin: state_f16, w1, w2 fp16 */
int mmpfn_mlp_f16(float* state_f32, uint16_t* state_f16, const uint16_t* w1, const uint16_t* w2, int M, void* stream);

/* Item-axis attention alone (layer.py:341-379), bf16 tcgen05 kernel, for unit tests and roofline timing.
 *   q  [B*T*nhead][Sq_pad][32]   k [planes_kv][Skv_pad][32]   vt [planes_kv][32][Skv_pad]   (bf16)
 *   planes_kv = B*T (shared_kv = 1: every query head reads head 0) or B*T*nhead (shared_kv = 0)
 *   out [B][n_q][T][nhead*32] bf16.  Sq_pad/Skv_pad are the allocated row counts (multiples of 8).
 * With shared_kv = 1 the six query heads of a column may be stacked on the tile row axis (fewer, fuller
 * tiles): the rows n_q .. Sq_pad-1 of every q plane are then read (their results are dropped) and should
 * hold finite values — mmpfn_item_qkv_bf16 writes zeros there. */
int mmpfn_item_attention_bf16(const uint16_t* q, const uint16_t* k, const uint16_t* vt, int B, int T, int n_q,
                              int Sq_pad, int n_kv, int Skv_pad, int shared_kv, uint16_t* out, void* stream);

/* The same with per-entry counts (entry b = plane column / T): entry b attends over its first kv_len[b] keys
 * (1..n_kv) and its output rows q_len[b] .. n_q-1 are zeros.  Key rows between kv_len[b] and n_kv must be zero. */
int mmpfn_item_attention_bf16_ragged(const uint16_t* q, const uint16_t* k, const uint16_t* vt, int B, int T, int n_q,
                                     int Sq_pad, int n_kv, int Skv_pad, int shared_kv, const int32_t* q_len,
                                     const int32_t* kv_len, uint16_t* out, void* stream);
/* fp16 twin of both (q, k, vt, out fp16): q_len / kv_len NULL = the plain form, both set = the per-entry form */
int mmpfn_item_attention_f16(const uint16_t* q, const uint16_t* k, const uint16_t* vt, int B, int T, int n_q,
                             int Sq_pad, int n_kv, int Skv_pad, int shared_kv, const int32_t* q_len,
                             const int32_t* kv_len, uint16_t* out, void* stream);
/* Item-axis attention of the fp32 parity mode (layer.py:341-379), for unit tests:
 *   q, out [B][n_q][T][nhead*32];  shared_kv = 0: k, v [B][n_kv][T][nhead*32];  shared_kv = 1 (every query head reads
 *   head 0, multi_head_attention.py:436-445): k, v [B][T][n_kv][32].
 * q_len / kv_len: per-entry counts as above, or NULL. */
int mmpfn_item_attention_f32(const float* q, const float* k, const float* v, int B, int T, int n_q, int n_kv,
                             int shared_kv, const int32_t* q_len, const int32_t* kv_len, float* out, void* stream);

/* Feature-axis attention alone (layer.py:332-339: per table row, 6 heads over the row's T tokens, d = 32), bf16
 * tensor-core kernel, for unit tests and HBM-roofline timing.
 *   qkv [n_rows*T][576] bf16 (q | k | v, head-major inside each third)  ->  att [n_rows*T][192] bf16 */
int mmpfn_feature_attention_bf16(const uint16_t* qkv, uint16_t* att, long long n_rows, int T, void* stream);
/* fp16 twin: qkv, att fp16 */
int mmpfn_feature_attention_f16(const uint16_t* qkv, uint16_t* att, long long n_rows, int T, void* stream);

/* QKV projection + feature-axis attention in ONE kernel (multi_head_attention.py:430-434 + layer.py:332-339 for the
 * feature axis): the [tokens][576] qkv block never leaves the SM.  What the bf16 layer passes run for T <= 64
 * (MMPFN_EUNSUPPORTED beyond); exported for unit tests (bit-identical to mmpfn_linear_bf16 +
 * mmpfn_feature_attention_bf16) and timing.
 *   x [n_rows*T][192] bf16, w_qkv [576][192] bf16  ->  att [n_rows*T][192] bf16 */
int mmpfn_feature_qkv_attention_bf16(const uint16_t* x, const uint16_t* w_qkv, long long n_rows, int T, uint16_t* att,
                                     void* stream);
/* fp16 twin: x, w_qkv, att fp16 */
int mmpfn_feature_qkv_attention_f16(const uint16_t* x, const uint16_t* w_qkv, long long n_rows, int T, uint16_t* att,
                                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MMPFN_B200_H */
