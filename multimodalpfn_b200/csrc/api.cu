// api.cu — the C ABI of libmmpfn_b200.so (include/mmpfn_b200.h): argument checking and the launch
// sequences of the stem, the 12 layers, the decoder and the probability tail.  No allocation, no
// host synchronisation; everything is enqueued on the caller's stream.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace mmpfn {

std::atomic<int64_t> g_launches{0};
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_geometry(const mmpfn_geometry* g) {
  if (!g) { set_error("null geometry"); return MMPFN_EINVAL; }
  if (g->emsize != kE || g->nhead != kH || g->nhid != kHid) {
    set_error("unsupported geometry: emsize %d nhead %d nhid %d (built for %d/%d/%d)", g->emsize, g->nhead, g->nhid,
              kE, kH, kHid);
    return MMPFN_EUNSUPPORTED;
  }
  if (g->features_per_group < 1 || g->features_per_group > 4 || g->nlayers < 1 || g->n_out < 1) {
    set_error("bad geometry: features_per_group %d nlayers %d n_out %d", g->features_per_group, g->nlayers, g->n_out);
    return MMPFN_EINVAL;
  }
  if (g->mixer_type != MMPFN_MIXER_NONE) {
    if (g->img_dim % 128 != 0 || g->mgm_heads < 1) { set_error("bad image stem geometry"); return MMPFN_EINVAL; }
    if (g->mixer_type == MMPFN_MIXER_MGM_CAP && (g->cap_heads < 1 || kE % g->cap_heads != 0)) {
      set_error("cap_heads %d must divide %d", g->cap_heads, kE);
      return MMPFN_EINVAL;
    }
  }
  return MMPFN_OK;
}

// the verdict is per device (0 unknown, 1 supported, 2 not): a process may use several
static int require_device() {
  static signed char ok[64] = {0};
  static int n_dev = -1;
  if (n_dev < 0) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); n = 0; }
    n_dev = n;
  }
  const int dev = n_dev > 0 ? current_device() : -1;
  if (dev >= 0 && dev < 64) {
    if (!ok[dev]) ok[dev] = mmpfn_device_supported(dev) ? 1 : 2;
    if (ok[dev] == 1) return MMPFN_OK;
  }
  set_error("no sm_100 CUDA device is current: libmmpfn_b200 holds sm_100a code only and has no CPU fallback");
  return MMPFN_ENODEVICE;
}

static SgemmParams gemm(const float* A, int lda, const float* W, int ldw, const float* bias, float* C, int ldc, int M,
                        int N, int K) {
  SgemmParams p{};
  p.A = A; p.W = W; p.bias = bias; p.C = C;
  p.M = M; p.N = N; p.K = K; p.lda = lda; p.ldw = ldw; p.ldc = ldc;
  p.batches = 1; p.row_inner = 1; p.row_outer = 1;
  return p;
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct LayerW {
  const float *fqkv, *fout, *iqkv, *iout, *w1, *w2;
  const uint16_t *fqkv_b, *fout_b, *iqkv_b, *iout_b, *w1_b, *w2_b;
};
static size_t layer_elems() { return (size_t)2 * (3 * kE * kE + kE * kE) + (size_t)2 * kHid * kE; }
static LayerW layer_w(const mmpfn_weights* w, int l) {
  LayerW r{};
  const size_t o0 = 0, o1 = o0 + 3 * kE * kE, o2 = o1 + kE * kE, o3 = o2 + 3 * kE * kE, o4 = o3 + kE * kE,
               o5 = o4 + (size_t)kHid * kE;
  const float* f = w->layers_f32 + l * layer_elems();
  r.fqkv = f + o0; r.fout = f + o1; r.iqkv = f + o2; r.iout = f + o3; r.w1 = f + o4; r.w2 = f + o5;
  if (w->layers_bf16) {
    const uint16_t* b = w->layers_bf16 + l * layer_elems();
    r.fqkv_b = b + o0; r.fout_b = b + o1; r.iqkv_b = b + o2; r.iout_b = b + o3; r.w1_b = b + o4; r.w2_b = b + o5;
  }
  return r;
}

static int kv_pad(int n) { return (n + 63) / 64 * 64; }

// K = 192 projections: the persistent kernel (kernels_rowgemm.cu).  In the tuning build (-DMMPFN_DEBUG)
// MMPFN_ROWGEMM=0 selects the one-tile-per-CTA kernel of kernels_tc.cu instead (A/B timing and bisecting);
// the product library reads no environment variable.
static int proj_gemm(const TcGemm& g, cudaStream_t st) {
#ifdef MMPFN_DEBUG
  static int persistent = -1;
  if (persistent < 0) {
    const char* e = getenv("MMPFN_ROWGEMM");
    persistent = e ? atoi(e) : 1;
  }
  if (!persistent) return launch_tc_gemm(g, st);
#endif
  return launch_tc_rowgemm(g, st);
}

// workspace carving for the layers
struct LayerWs {
  // fp32 mode
  float *qkv, *att, *hid, *tmp;
  // bf16 mode
  uint16_t *qkv_b, *att_b, *hid_b, *qi, *ki, *vti;
  size_t bytes;
};
static LayerWs carve(void* base, long long M, int B, int S, int T, int precision) {
  LayerWs w{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? (char*)base + off : nullptr;
    off += align_up(bytes, 1024);
    return (void*)p;
  };
  if (precision == MMPFN_F32) {
    w.qkv = (float*)take((size_t)M * 3 * kE * 4);
    w.att = (float*)take((size_t)M * kE * 4);
    w.hid = (float*)take((size_t)M * kHid * 4);
    w.tmp = (float*)take((size_t)M * kE * 4);
  } else {
    const size_t plane = (size_t)B * T * kH * kv_pad(S) * kD * 2;
    // qkv (features) and hid (MLP) are never live together: share one buffer
    w.hid_b = (uint16_t*)take((size_t)M * kHid * 2);
    w.qkv_b = w.hid_b;
    w.att_b = (uint16_t*)take((size_t)M * kE * 2);
    w.qi = (uint16_t*)take(plane);
    w.ki = (uint16_t*)take(plane);
    w.vti = (uint16_t*)take(plane);
  }
  w.bytes = off;
  return w;
}

}  // namespace mmpfn

using namespace mmpfn;

extern "C" {

int mmpfn_abi_version(void) { return MMPFN_ABI_VERSION; }
const char* mmpfn_last_error(void) { return g_err; }
int64_t mmpfn_launch_count(void) { return g_launches.load(); }

int mmpfn_device_supported(int dev) {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  // the library carries sm_100a SASS and no PTX: compute capability 10.0 exactly (an sm_103 part would pass a
  // "major == 10" test and then fail at the first launch)
  return (prop.major == 10 && prop.minor == 0) ? 1 : 0;
}

size_t mmpfn_layer_weight_elems(const mmpfn_geometry* g) {
  if (check_geometry(g) != MMPFN_OK) return 0;
  return layer_elems();
}

int mmpfn_image_tokens(const mmpfn_geometry* g, int n_tok) {
  switch (g->mixer_type) {
    case MMPFN_MIXER_MGM: return g->mgm_heads * n_tok;
    case MMPFN_MIXER_MGM_CAP: return g->cap_heads;
    case MMPFN_MIXER_MOE: return g->mgm_heads;
    default: return 0;
  }
}

size_t mmpfn_tab_stats_elems(const mmpfn_geometry* g, int n_groups) {
  TabStatsLayout L{n_groups * g->features_per_group, n_groups};
  return (size_t)L.total();
}

int mmpfn_stem_tab_fit(const mmpfn_geometry* g, const float* x, int B, int S, int F, int n_train, float n_sigma,
                       float* stats, void* stream) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  if (!x || !stats || B < 1 || S < 1 || F < 1 || n_train < 1 || n_train > S) {
    set_error("stem_tab_fit: bad arguments (B %d S %d F %d n_train %d)", B, S, F, n_train);
    return MMPFN_EINVAL;
  }
  return launch_tab_fit(x, B, S, F, g->features_per_group, n_train, n_sigma, stats, (cudaStream_t)stream);
}

int mmpfn_stem_tab_fit_ragged(const mmpfn_geometry* g, const float* x, int B, int S, int F, const int32_t* n_rows,
                              const int32_t* n_train, float n_sigma, float* stats, void* stream) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  if (!x || !stats || !n_rows || !n_train || B < 1 || S < 1 || F < 1) {
    set_error("stem_tab_fit_ragged: bad arguments (B %d S %d F %d)", B, S, F);
    return MMPFN_EINVAL;
  }
  return launch_tab_fit(x, B, S, F, g->features_per_group, 0, n_sigma, stats, (cudaStream_t)stream, n_rows, n_train);
}

// image stem scratch (floats)
struct ImgWs {
  float *xhat, *u, *src, *srcn, *kv, *o, *o2, *f1, *f2, *gl;
  uint16_t* xhat_b;     // bf16 copy of the normalised embeddings: A operand of the tcgen05 MGM GEMM
  size_t bytes;
};
static ImgWs carve_img(const mmpfn_geometry* g, void* base, int S, int n_tok) {
  ImgWs w{};
  size_t off = 0;
  auto take = [&](size_t elems) {
    char* p = base ? (char*)base + off : nullptr;
    off += align_up(elems * 4, 1024);
    return (float*)p;
  };
  const size_t I = g->img_dim, Hm = g->mgm_heads;
  if (g->mixer_type == MMPFN_MIXER_MOE) {
    w.xhat = take((size_t)S * I);
    w.u = take((size_t)S * Hm * (I / 2));
    w.gl = take((size_t)S * Hm);
  } else {
    const size_t M0 = (size_t)S * n_tok, n_kv = Hm * n_tok, Hc = g->cap_heads;
    w.xhat = take(M0 * I);
    w.xhat_b = (uint16_t*)take((M0 * I + 1) / 2);
    w.u = take(M0 * Hm * (I / 2));
    if (g->mixer_type == MMPFN_MIXER_MGM_CAP) {
      w.src = take((size_t)S * n_kv * kE);
      w.srcn = take((size_t)S * n_kv * kE);
      w.kv = take((size_t)S * n_kv * 2 * kE);
      w.o = take((size_t)S * Hc * kE);
      w.o2 = take((size_t)S * Hc * kE);
      w.f1 = take((size_t)S * Hc * 2 * kE);
      w.f2 = take((size_t)S * Hc * kE);
    }
  }
  w.bytes = off;
  return w;
}

size_t mmpfn_stem_image_ws_bytes(const mmpfn_geometry* g, int S, int n_tok) {
  if (check_geometry(g) != MMPFN_OK || g->mixer_type == MMPFN_MIXER_NONE) return 0;
  return carve_img(g, nullptr, S, n_tok).bytes;
}

int mmpfn_stem_image(const mmpfn_geometry* g, const mmpfn_weights* w, const float* img, int S, int n_tok, float* out,
                     void* workspace, size_t workspace_bytes, void* stream) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  cudaStream_t st = (cudaStream_t)stream;
  if (g->mixer_type == MMPFN_MIXER_NONE || !img || !out || S < 1 || n_tok < 1 || !w || !w->mgm_w1) {
    set_error("stem_image: bad arguments");
    return MMPFN_EINVAL;
  }
  ImgWs ws = carve_img(g, workspace, S, n_tok);
  if (!workspace || workspace_bytes < ws.bytes) {
    set_error("stem_image: workspace %zu < %zu bytes", workspace_bytes, ws.bytes);
    return MMPFN_EINVAL;
  }
  const int I = g->img_dim, Hm = g->mgm_heads, Ih = I / 2;
  if (I != 768) { set_error("stem_image: img_dim %d (built for 768)", I); return MMPFN_EUNSUPPORTED; }

  if (g->mixer_type == MMPFN_MIXER_MOE) {
    // transformer.py:109 uses the first token only
    MMPFN_TRY(launch_layernorm(img, nullptr, nullptr, nullptr, S, I, ws.xhat, nullptr, st, (long long)n_tok * I));
    MMPFN_TRY(launch_sgemm(gemm(ws.xhat, I, w->mgm_w1, I, w->mgm_b1, ws.u, Hm * Ih, S, Hm * Ih, I), EPI_GELU, st));
    SgemmParams p = gemm(ws.u, Hm * Ih, w->mgm_w2, Ih, w->mgm_b2, out, kE, S, kE, Ih);
    p.batches = Hm; p.a_batch = Ih; p.w_batch = (long long)kE * Ih; p.bias_batch = kE; p.c_batch = kE;
    p.row_inner = 1; p.row_outer = Hm;
    MMPFN_TRY(launch_sgemm(p, EPI_NONE, st));
    MMPFN_TRY(launch_sgemm(gemm(img, n_tok * I, w->moe_gate_w, I, w->moe_gate_b, ws.gl, Hm, S, Hm, I), EPI_NONE, st));
    return launch_moe_gate_scale(ws.gl, out, S, Hm, st);
  }

  const int M0 = S * n_tok, n_kv = Hm * n_tok;
  // MGM (transformer.py:33-48): LayerNorm statistics once, per-head affine folded into W1/b1
  if (w->mgm_w1_bf16 && Hm >= 32) {
    // bf16 mode, many MGM heads: the one large GEMM of the stem (M0 x Hm*768 x 768: 0.09 TFLOP per 300 rows at 256
    // heads) on tcgen05, bias + GLU in the epilogue, fp32 out; everything downstream of it stays fp32.  Below 32 heads
    // the FFMA GEMM takes < 0.1 ms per call and keeps the stem exact (measured: bf16 operands here cost 13 % of the
    // bf16 error budget at trained-like logit scales, tests/test_gpu_model.py stress_tiny)
    MMPFN_TRY(launch_layernorm(img, nullptr, nullptr, nullptr, M0, I, ws.xhat, ws.xhat_b, st));
    TcGemm t{};
    t.A = ws.xhat_b; t.W = w->mgm_w1_bf16; t.M = M0; t.N = Hm * I; t.K = I; t.epi = TC_EPI_GLU_PAIR_F32;
    t.bias = w->mgm_b1; t.out_f32 = ws.u;
    MMPFN_TRY(launch_tc_gemm(t, st));
  } else {
    MMPFN_TRY(launch_layernorm(img, nullptr, nullptr, nullptr, M0, I, ws.xhat, nullptr, st));
    MMPFN_TRY(launch_sgemm(gemm(ws.xhat, I, w->mgm_w1, I, w->mgm_b1, ws.u, Hm * Ih, M0, Hm * I, I), EPI_GLU_PAIR, st));
  }
  float* src = g->mixer_type == MMPFN_MIXER_MGM ? out : ws.src;
  {
    SgemmParams p = gemm(ws.u, Hm * Ih, w->mgm_w2, Ih, w->mgm_b2, src, kE, M0, kE, Ih);
    p.batches = Hm; p.a_batch = Ih; p.w_batch = (long long)kE * Ih; p.bias_batch = kE;
    p.c_batch = (long long)n_tok * kE;                          // head-major on the token axis
    p.row_inner = n_tok; p.row_outer = n_kv;
    MMPFN_TRY(launch_sgemm(p, EPI_NONE, st));
  }
  if (g->mixer_type == MMPFN_MIXER_MGM) return MMPFN_OK;

  // CAP (transformer.py:77-88)
  const int Hc = g->cap_heads;
  const long long Ms = (long long)S * n_kv, Mq = (long long)S * Hc;
  MMPFN_TRY(launch_layernorm(ws.src, nullptr, w->cap_knorm_w, w->cap_knorm_b, Ms, kE, ws.srcn, nullptr, st));
  MMPFN_TRY(launch_sgemm(gemm(ws.srcn, kE, w->cap_wkv, kE, w->cap_bkv, ws.kv, 2 * kE, (int)Ms, 2 * kE, kE), EPI_NONE, st));
  MMPFN_TRY(launch_cap_attn(ws.kv, w->cap_q, S, n_kv, Hc, ws.o, st));
  MMPFN_TRY(launch_sgemm(gemm(ws.o, kE, w->cap_wo, kE, w->cap_bo, ws.o2, kE, (int)Mq, kE, kE), EPI_NONE, st));
  MMPFN_TRY(launch_sgemm(gemm(ws.o2, kE, w->cap_f1_w, kE, w->cap_f1_b, ws.f1, 2 * kE, (int)Mq, 2 * kE, kE), EPI_GELU, st));
  MMPFN_TRY(launch_sgemm(gemm(ws.f1, 2 * kE, w->cap_f2_w, 2 * kE, w->cap_f2_b, ws.f2, kE, (int)Mq, kE, 2 * kE), EPI_NONE, st));
  return launch_cap_combine(ws.o2, ws.f2, w->cap_onorm_w, w->cap_onorm_b, Mq, out, st);
}

int mmpfn_stem_tokens(const mmpfn_geometry* g, const mmpfn_weights* w, const float* x, const float* stats,
                      const float* img_tok, const float* y, const float* y_mean, const uint64_t* y_present_mask,
                      const float* pos_emb, int B, int S, int F, int H_img, long long x_bstride, long long y_bstride,
                      long long img_bstride, float* state_f32, uint16_t* state_bf16, int32_t* nan_flag, void* stream) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  if (!w || !y || !y_mean || !y_present_mask || !pos_emb || !state_f32 || !nan_flag || B < 1 || S < 1 ||
      (x && (!stats || F < 1)) || (!x && !img_tok) || (img_tok && H_img < 1) || (!img_tok && H_img != 0) ||
      img_bstride < 0) {
    set_error("stem_tokens: bad arguments");
    return MMPFN_EINVAL;
  }
  return launch_stem_tokens(g, w, x, stats, img_tok, y, y_mean, y_present_mask, pos_emb, B, S, x ? F : 0, H_img,
                            x_bstride, y_bstride, img_bstride, state_f32, state_bf16, nan_flag, (cudaStream_t)stream);
}

int mmpfn_stem_tokens_ragged(const mmpfn_geometry* g, const mmpfn_weights* w, const float* x, const float* stats,
                             const float* img_tok, const float* y, const float* y_mean, const uint64_t* y_present_mask,
                             const float* pos_emb, int B, int S, int F, int H_img, long long x_bstride,
                             long long y_bstride, const int64_t* img_offset, const int32_t* n_rows, float* state_f32,
                             uint16_t* state_bf16, int32_t* nan_flag, void* stream) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  if (!w || !y || !y_mean || !y_present_mask || !pos_emb || !state_f32 || !nan_flag || B < 1 || S < 1 ||
      (x && (!stats || F < 1)) || (!x && !img_tok) || (img_tok && (H_img < 1 || !img_offset)) || (!img_tok && H_img != 0)) {
    set_error("stem_tokens_ragged: bad arguments");
    return MMPFN_EINVAL;
  }
  return launch_stem_tokens(g, w, x, stats, img_tok, y, y_mean, y_present_mask, pos_emb, B, S, x ? F : 0, H_img,
                            x_bstride, y_bstride, 0, state_f32, state_bf16, nan_flag, (cudaStream_t)stream,
                            (const long long*)img_offset, n_rows);
}

size_t mmpfn_layers_ws_bytes(const mmpfn_geometry* g, int B, int S, int T, int precision) {
  if (check_geometry(g) != MMPFN_OK) return 0;
  return carve(nullptr, (long long)B * S * T, B, S, T, precision).bytes;
}

size_t mmpfn_kv_bytes(const mmpfn_geometry* g, int B, int n_train, int T, int precision) {
  if (check_geometry(g) != MMPFN_OK) return 0;
  if (precision == MMPFN_F32) return (size_t)g->nlayers * B * T * n_train * 2 * kD * 4;
  return (size_t)g->nlayers * B * T * kv_pad(n_train) * 2 * kD * 2;
}

// One layer's two row-wise sublayers shared by the train and the test pass.
static int feature_attention(const LayerW& lw, float* state, uint16_t* state_b, long long M, long long n_seq, int T,
                             int precision, const LayerWs& ws, cudaStream_t st) {
  if (precision == MMPFN_F32) {
    MMPFN_TRY(launch_sgemm(gemm(state, kE, lw.fqkv, kE, nullptr, ws.qkv, 3 * kE, (int)M, 3 * kE, kE), EPI_NONE, st));
    MMPFN_TRY(launch_feat_attn_f32(ws.qkv, ws.att, n_seq, T, st));
    MMPFN_TRY(launch_sgemm(gemm(ws.att, kE, lw.fout, kE, nullptr, ws.tmp, kE, (int)M, kE, kE), EPI_NONE, st));
    return launch_layernorm(ws.tmp, state, nullptr, nullptr, M, kE, state, nullptr, st);
  }
  TcGemm a{};
  a.A = state_b; a.W = lw.fqkv_b; a.M = (int)M; a.N = 3 * kE; a.K = kE; a.epi = TC_EPI_BF16; a.out_bf16 = ws.qkv_b;
  MMPFN_TRY(proj_gemm(a, st));
  MMPFN_TRY(launch_feat_attn_bf16(ws.qkv_b, ws.att_b, n_seq, T, st));
  TcGemm o{};
  o.A = ws.att_b; o.W = lw.fout_b; o.M = (int)M; o.N = kE; o.K = kE; o.epi = TC_EPI_RESID_LN;
  o.resid_f32 = state; o.ln_bf16 = state_b;
  return proj_gemm(o, st);
}

static int mlp(const LayerW& lw, float* state, uint16_t* state_b, long long M, int precision, const LayerWs& ws,
               cudaStream_t st) {
  if (precision == MMPFN_F32) {
    MMPFN_TRY(launch_sgemm(gemm(state, kE, lw.w1, kE, nullptr, ws.hid, kHid, (int)M, kHid, kE), EPI_GELU, st));
    MMPFN_TRY(launch_sgemm(gemm(ws.hid, kHid, lw.w2, kHid, nullptr, ws.tmp, kE, (int)M, kE, kHid), EPI_NONE, st));
    return launch_layernorm(ws.tmp, state, nullptr, nullptr, M, kE, state, nullptr, st);
  }
#ifdef MMPFN_DEBUG
  // tuning build only: MMPFN_FUSED_MLP=0 takes the two-GEMM form (A/B timing and bisecting)
  static int fused = -1;
  if (fused < 0) {
    const char* e = getenv("MMPFN_FUSED_MLP");
    fused = e ? atoi(e) : 1;
  }
#else
  constexpr int fused = 1;
#endif
  if (fused) {
    TcMlp f{};
    f.state_b = state_b; f.state_b_out = state_b; f.resid_f32 = state; f.w1 = lw.w1_b; f.w2 = lw.w2_b; f.M = (int)M;
    return launch_tc_mlp(f, st);
  }
  TcGemm a{};
  a.A = state_b; a.W = lw.w1_b; a.M = (int)M; a.N = kHid; a.K = kE; a.epi = TC_EPI_GELU_BF16; a.out_bf16 = ws.hid_b;
  MMPFN_TRY(launch_tc_gemm(a, st));
  TcGemm o{};
  o.A = ws.hid_b; o.W = lw.w2_b; o.M = (int)M; o.N = kE; o.K = kHid; o.epi = TC_EPI_RESID_LN;
  o.resid_f32 = state; o.ln_bf16 = state_b;
  return launch_tc_gemm(o, st);
}

static int out_proj_ln(const LayerW& lw, float* state, uint16_t* state_b, long long M, int precision,
                       const LayerWs& ws, cudaStream_t st) {
  if (precision == MMPFN_F32) {
    MMPFN_TRY(launch_sgemm(gemm(ws.att, kE, lw.iout, kE, nullptr, ws.tmp, kE, (int)M, kE, kE), EPI_NONE, st));
    return launch_layernorm(ws.tmp, state, nullptr, nullptr, M, kE, state, nullptr, st);
  }
  TcGemm o{};
  o.A = ws.att_b; o.W = lw.iout_b; o.M = (int)M; o.N = kE; o.K = kE; o.epi = TC_EPI_RESID_LN;
  o.resid_f32 = state; o.ln_bf16 = state_b;
  return proj_gemm(o, st);
}

static int check_layers_args(const mmpfn_geometry* g, const mmpfn_weights* w, float* state, uint16_t* state_b, int B,
                             int S, int T, int precision, void* workspace, size_t workspace_bytes, LayerWs* ws) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  if (!w || !w->layers_f32 || !state || B < 1 || S < 1 || T < 2 ||
      (precision != MMPFN_F32 && precision != MMPFN_BF16)) {
    set_error("layers: bad arguments (B %d S %d T %d precision %d)", B, S, T, precision);
    return MMPFN_EINVAL;
  }
  if (precision == MMPFN_BF16 && (!state_b || !w->layers_bf16)) {
    set_error("layers: bf16 mode needs the bf16 state shadow and bf16 weights");
    return MMPFN_EINVAL;
  }
  // row counts are passed as int to the GEMM tiles
  if ((long long)B * S * T > 2147483647LL) { set_error("layers: too many tokens"); return MMPFN_EUNSUPPORTED; }
  *ws = carve(workspace, (long long)B * S * T, B, S, T, precision);
  if (!workspace || workspace_bytes < ws->bytes) {
    set_error("layers: workspace %zu < %zu bytes", workspace_bytes, ws->bytes);
    return MMPFN_EINVAL;
  }
  return MMPFN_OK;
}

static int layers_run(const mmpfn_geometry* g, const mmpfn_weights* w, float* state, uint16_t* state_b,
                      const mmpfn_kv_segment* ks, int n_seg, int S, int n_train, int train, int layer_begin,
                      int layer_end, int phase, void* workspace, size_t workspace_bytes, cudaStream_t st,
                      const int* n_rows = nullptr, const int* n_ctx = nullptr);

// The fp32 (parity mode) passes over one [B][S][T] state.  train != 0: self-attention over the S rows, head-0 K/V
// written to kv (may be NULL); else the S rows attend to the n_train rows of the context kv.  n_rows / n_ctx (device
// [B], or NULL = S / n_train): entry b's own row count in this pass and context rows of the test pass.
static int layers_f32(const mmpfn_geometry* g, const mmpfn_weights* w, float* state, int B, int S, int T, int n_train,
                      int train, void* kv, const int* n_rows, const int* n_ctx, const LayerWs& ws, cudaStream_t st) {
  const long long M = (long long)B * S * T;
  for (int l = 0; l < g->nlayers; ++l) {
    const LayerW lw = layer_w(w, l);
    MMPFN_TRY(feature_attention(lw, state, nullptr, M, (long long)B * S, T, MMPFN_F32, ws, st));
    ItemAttnF32 a{};
    a.out = ws.att;
    a.o_outer = (long long)S * T * kE; a.o_inner = kE; a.o_row = (long long)T * kE;
    a.planes = B * T; a.inner = T; a.n_q = S; a.q_len = n_rows;
    if (train) {
      MMPFN_TRY(launch_sgemm(gemm(state, kE, lw.iqkv, kE, nullptr, ws.qkv, 3 * kE, (int)M, 3 * kE, kE), EPI_NONE, st));
      if (kv) {
        float* kvl = (float*)kv + (size_t)l * B * T * S * 2 * kD;
        MMPFN_TRY(launch_kv_extract_f32(ws.qkv, kvl, B, S, T, st, n_rows));
      }
      a.q = ws.qkv; a.k = ws.qkv + kE; a.v = ws.qkv + 2 * kE;
      a.q_outer = (long long)S * T * 3 * kE; a.q_inner = 3 * kE; a.q_row = (long long)T * 3 * kE;
      a.kv_outer = a.q_outer; a.kv_inner = a.q_inner; a.kv_row = a.q_row;
      a.n_kv = S; a.shared_kv = 0; a.kv_len = n_rows;
    } else {
      // queries only (multi_head_attention.py:432-434); K/V come from the context
      MMPFN_TRY(launch_sgemm(gemm(state, kE, lw.iqkv, kE, nullptr, ws.qkv, kE, (int)M, kE, kE), EPI_NONE, st));
      const float* kvl = (const float*)kv + (size_t)l * B * T * n_train * 2 * kD;
      a.q = ws.qkv; a.k = kvl; a.v = kvl + kD;
      a.q_outer = (long long)S * T * kE; a.q_inner = kE; a.q_row = (long long)T * kE;
      a.kv_outer = (long long)T * n_train * 2 * kD; a.kv_inner = (long long)n_train * 2 * kD; a.kv_row = 2 * kD;
      a.n_kv = n_train; a.shared_kv = 1; a.kv_len = n_ctx;
    }
    MMPFN_TRY(launch_item_attn_f32(a, st));
    MMPFN_TRY(out_proj_ln(lw, state, nullptr, M, MMPFN_F32, ws, st));
    MMPFN_TRY(mlp(lw, state, nullptr, M, MMPFN_F32, ws, st));
  }
  return MMPFN_OK;
}

int mmpfn_layers_train(const mmpfn_geometry* g, const mmpfn_weights* w, float* state, uint16_t* state_b, int B, int S,
                       int T, int precision, void* kv, void* workspace, size_t workspace_bytes, void* stream) {
  LayerWs ws;
  MMPFN_TRY(check_layers_args(g, w, state, state_b, B, S, T, precision, workspace, workspace_bytes, &ws));
  cudaStream_t st = (cudaStream_t)stream;
  if (precision == MMPFN_BF16) {      // one segment of the general bf16 pass (same workspace layout)
    mmpfn_kv_segment k{};
    k.B = B; k.T = T; k.kv = kv;
    return layers_run(g, w, state, state_b, &k, 1, S, 0, 1, 0, g->nlayers, 0, workspace, workspace_bytes, st);
  }
  return layers_f32(g, w, state, B, S, T, 0, 1, kv, nullptr, nullptr, ws, st);
}

int mmpfn_layers_test(const mmpfn_geometry* g, const mmpfn_weights* w, float* state, uint16_t* state_b, int B, int S,
                      int T, int n_train, int precision, const void* kv, void* workspace, size_t workspace_bytes,
                      void* stream) {
  LayerWs ws;
  MMPFN_TRY(check_layers_args(g, w, state, state_b, B, S, T, precision, workspace, workspace_bytes, &ws));
  if (!kv || n_train < 1) { set_error("layers_test: needs the K/V context of the train rows"); return MMPFN_EINVAL; }
  cudaStream_t st = (cudaStream_t)stream;
  if (precision == MMPFN_BF16) {
    mmpfn_kv_segment k{};
    k.B = B; k.T = T; k.kv = const_cast<void*>(kv);
    return layers_run(g, w, state, state_b, &k, 1, S, n_train, 0, 0, g->nlayers, 0, workspace, workspace_bytes, st);
  }
  return layers_f32(g, w, state, B, S, T, n_train, 0, const_cast<void*>(kv), nullptr, nullptr, ws, st);
}

// ---- several estimator groups (segments) in one call -------------------------------------------------
// Segments differ in their token count T (and batch B) but share the row count S.  Their states sit back
// to back in ONE [M_total][192] buffer, so the sublayers that do not care about T — both QKV/output
// projections on the flat token axis and the MLP — run as ONE launch over all segments (longer grids:
// less tile-count rounding per launch, half the launches); only the two attentions and the item QKV
// scatter, whose tiling follows T, launch per segment.
struct SegWs {
  uint16_t *qi, *ki, *vti;
};
struct MultiWs {
  uint16_t *hid_b, *att_b;
  SegWs seg[MMPFN_MAX_SEGMENTS];
  size_t bytes;
};
static MultiWs carve_multi(void* base, const mmpfn_segment* segs, int n_seg, int S, long long M_total) {
  MultiWs w{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? (char*)base + off : nullptr;
    off += align_up(bytes, 1024);
    return (uint16_t*)p;
  };
  w.hid_b = take((size_t)M_total * kHid * 2);      // also the feature-attention qkv block (never live together)
  w.att_b = take((size_t)M_total * kE * 2);
  for (int i = 0; i < n_seg; ++i) {
    const size_t plane = (size_t)segs[i].B * segs[i].T * kH * kv_pad(S) * kD * 2;
    w.seg[i].qi = take(plane);
    w.seg[i].ki = take(plane);
    w.seg[i].vti = take(plane);
  }
  w.bytes = off;
  return w;
}
static int check_segments(const mmpfn_segment* segs, int n_seg, int S, long long* M_total) {
  if (!segs || n_seg < 1 || n_seg > MMPFN_MAX_SEGMENTS || S < 1) { set_error("layers_multi: bad segment list"); return MMPFN_EINVAL; }
  long long m = 0;
  for (int i = 0; i < n_seg; ++i) {
    if (segs[i].B < 1 || segs[i].T < 2) { set_error("layers_multi: bad segment %d (B %d T %d)", i, segs[i].B, segs[i].T); return MMPFN_EINVAL; }
    m += (long long)segs[i].B * S * segs[i].T;
  }
  if (m > 2147483647LL) { set_error("layers_multi: too many tokens"); return MMPFN_EUNSUPPORTED; }
  *M_total = m;
  return MMPFN_OK;
}

size_t mmpfn_layers_multi_ws_bytes(const mmpfn_geometry* g, const mmpfn_segment* segs, int n_seg, int S) {
  long long M = 0;
  if (check_geometry(g) != MMPFN_OK || check_segments(segs, n_seg, S, &M) != MMPFN_OK) return 0;
  return carve_multi(nullptr, segs, n_seg, S, M).bytes;
}

// One K/V context block per segment and layer: K0 [c][T][Np][32] then V0^T [c][T][32][Np] (bf16), c = the
// estimators stored back to back (train pass: c = B; test pass: c = slots, see mmpfn_kv_segment).
static size_t kv_block_elems(int c, int T, int n_pad) { return (size_t)2 * c * T * n_pad * kD; }

// train != 0: self-attention over the S rows, head-0 K/V written to segs[i].kv (may be NULL);
// train == 0: the S rows are test rows attending to the n_train rows' context segs[i].kv
// n_rows / n_ctx (device, one entry per estimator of every segment in list order, or NULL): per-entry row counts of
// this pass and context rows of the test pass (mmpfn_layers_*_ragged)
static int layers_run(const mmpfn_geometry* g, const mmpfn_weights* w, float* state, uint16_t* state_b,
                      const mmpfn_kv_segment* ks, int n_seg, int S, int n_train, int train, int layer_begin,
                      int layer_end, int phase, void* workspace, size_t workspace_bytes, cudaStream_t st,
                      const int* n_rows, const int* n_ctx) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  if (!ks || n_seg < 1 || n_seg > MMPFN_MAX_SEGMENTS) { set_error("layers_run: bad segment list"); return MMPFN_EINVAL; }
  mmpfn_segment segs[MMPFN_MAX_SEGMENTS];
  for (int i = 0; i < n_seg; ++i) { segs[i].B = ks[i].B; segs[i].T = ks[i].T; }
  long long M = 0;
  MMPFN_TRY(check_segments(segs, n_seg, S, &M));
  if (!w || !w->layers_f32 || !w->layers_bf16 || !state || !state_b) { set_error("layers_run: null argument (bf16 mode only)"); return MMPFN_EINVAL; }
  if (layer_begin < 0 || layer_end > g->nlayers || layer_begin >= layer_end) { set_error("layers_run: bad layer range [%d, %d)", layer_begin, layer_end); return MMPFN_EINVAL; }
  if (phase < 0 || phase > 2 || (phase != 0 && layer_end != layer_begin + 1)) { set_error("layers_run: phase %d needs a single layer", phase); return MMPFN_EINVAL; }
  for (int i = 0; i < n_seg; ++i) {
    const mmpfn_kv_segment& k = ks[i];
    if (train && k.seg_rows > 0 && (!k.kg || !k.vtg || k.n_ranks < 1 || k.rank < 0 || k.rank >= k.n_ranks || k.seg_rows % 48 != 0 ||
                                    S > k.seg_rows || k.n_rows_total < 1 || k.gather_stride % 16 != 0)) {
      set_error("layers_run: bad row-sharding description of segment %d", i);
      return MMPFN_EINVAL;
    }
  }
  if (!train) for (int i = 0; i < n_seg; ++i) if (!ks[i].kv || n_train < 1) { set_error("layers_run: the test pass needs every segment's context"); return MMPFN_EINVAL; }
  // row-sharded build: every rank lays its planes out for seg_rows rows (the last rank holds fewer), so that the
  // chunks of the gather buffers and of the gathered context have one plane stride
  int Sa = S;
  if (train) for (int i = 0; i < n_seg; ++i) if (ks[i].seg_rows > Sa) Sa = ks[i].seg_rows;
  MultiWs ws = carve_multi(workspace, segs, n_seg, Sa, M);
  if (!workspace || workspace_bytes < ws.bytes) { set_error("layers_run: workspace %zu < %zu bytes", workspace_bytes, ws.bytes); return MMPFN_EINVAL; }
  const int Sp = kv_pad(Sa), Np = kv_pad(n_train);
  LayerWs flat{};
  flat.hid_b = ws.hid_b; flat.qkv_b = ws.hid_b; flat.att_b = ws.att_b;
#ifdef MMPFN_DEBUG
  // tuning build only: MMPFN_FEAT_FUSED=0 takes the two-kernel form of the feature sublayer's first half
  static int feat_fused = -1;
  if (feat_fused < 0) {
    const char* e = getenv("MMPFN_FEAT_FUSED");
    feat_fused = e ? atoi(e) : 1;
  }
#else
  constexpr bool feat_fused = true;
#endif
  for (int l = layer_begin; l < layer_end; ++l) {
    const LayerW lw = layer_w(w, l);
    // features: QKV over all tokens, attention per segment (rows of T_i tokens), out-projection + LN over all
    if (phase != 2) {
      // rows of up to 64 tokens: projection and attention in one kernel (the qkv block stays on chip); wider rows:
      // the projection, then the attention.  Per segment either way.
      long long off = 0;
      for (int i = 0; i < n_seg; ++i) {
        const long long m = (long long)segs[i].B * S * segs[i].T;
        if (feat_fused && feat_qkv_attn_supported(segs[i].T)) {
          MMPFN_TRY(launch_feat_qkv_attn(state_b + off * kE, lw.fqkv_b, m, segs[i].T, ws.att_b + off * kE, st));
        } else {
          TcGemm a{};
          a.A = state_b + off * kE; a.W = lw.fqkv_b; a.M = (int)m; a.N = 3 * kE; a.K = kE; a.epi = TC_EPI_BF16;
          a.out_bf16 = ws.hid_b + off * 3 * kE;
          MMPFN_TRY(proj_gemm(a, st));
          MMPFN_TRY(launch_feat_attn_bf16(ws.hid_b + off * 3 * kE, ws.att_b + off * kE, (long long)segs[i].B * S, segs[i].T, st));
        }
        off += m;
      }
      TcGemm o{};
      o.A = ws.att_b; o.W = lw.fout_b; o.M = (int)M; o.N = kE; o.K = kE; o.epi = TC_EPI_RESID_LN;
      o.resid_f32 = state; o.ln_bf16 = state_b;
      MMPFN_TRY(proj_gemm(o, st));
    }
    // items: QKV scatter + attention per segment (tiles follow T_i), out-projection + LN over all
    {
      long long off = 0, entry = 0;
      for (int i = 0; i < n_seg; ++i) {
        const int B = segs[i].B, T = segs[i].T;
        TcGemm q{};
        q.A = state_b + off * kE; q.W = lw.iqkv_b; q.N = train ? 3 * kE : kE; q.K = kE; q.items = 1; q.B = B; q.S = S; q.T = T;
        q.epi = TC_EPI_QKV_ITEMS; q.q_out = ws.seg[i].qi; q.S_pad = Sp;
        TcItemAttn a{};
        a.q = ws.seg[i].qi; a.out = ws.att_b + off * kE; a.B = B; a.T = T; a.n_q = S; a.Sq_pad = Sp;
        a.q_len = n_rows ? n_rows + entry : nullptr;
        a.kv_len = train ? a.q_len : (n_ctx ? n_ctx + entry : nullptr);
        const bool rows_mode = train && ks[i].seg_rows > 0;
        if (rows_mode) {
          // row-sharded build: this rank's K / V^T planes go into its chunk of the gather buffers; after the
          // caller's all-gather the attention reads every chunk as one key range of n_rows_total rows
          uint16_t* kg = (uint16_t*)ks[i].kg;
          uint16_t* vg = (uint16_t*)ks[i].vtg;
          const size_t cs = (size_t)ks[i].gather_stride / 2;
          q.k_out = kg + cs * ks[i].rank; q.vt_out = vg + cs * ks[i].rank;
          if (ks[i].kv) {
            const size_t stride = ks[i].layer_stride > 0 ? (size_t)ks[i].layer_stride / 2 : kv_block_elems(B, T, Sp);
            uint16_t* kvl = (uint16_t*)ks[i].kv + (size_t)l * stride;
            q.k0_out = kvl;
            q.vt0_out = kvl + (size_t)B * T * Sp * kD;
          }
          a.k = kg; a.vt = vg; a.n_kv = ks[i].n_rows_total; a.Skv_pad = Sp; a.shared_kv = 0;
          a.kv_seg_rows = ks[i].seg_rows; a.kv_seg_stride = (long long)cs;
        } else if (train) {
          q.k_out = ws.seg[i].ki; q.vt_out = ws.seg[i].vti;
          if (ks[i].kv) {
            const size_t stride = ks[i].layer_stride > 0 ? (size_t)ks[i].layer_stride / 2 : kv_block_elems(B, T, Sp);
            uint16_t* kvl = (uint16_t*)ks[i].kv + (size_t)l * stride;
            q.k0_out = kvl;
            q.vt0_out = kvl + (size_t)B * T * Sp * kD;
          }
          a.k = ws.seg[i].ki; a.vt = ws.seg[i].vti; a.n_kv = S; a.Skv_pad = Sp; a.shared_kv = 0;
        } else {
          const int c = ks[i].slots > 0 ? ks[i].slots : B;
          const size_t stride = ks[i].layer_stride > 0 ? (size_t)ks[i].layer_stride / 2 : kv_block_elems(B, T, Np);
          const uint16_t* kvl = (const uint16_t*)ks[i].kv + (size_t)l * stride;
          a.k = kvl; a.vt = kvl + (size_t)c * T * Np * kD; a.n_kv = n_train; a.Skv_pad = Np; a.shared_kv = 1;
          a.kv_slots = ks[i].slots > 0 ? ks[i].slots : 0;
          a.kv_rank_stride = ks[i].rank_stride / 2;
          if (ks[i].seg_rows > 0) {
            // the context was built row-sharded: chunk r (rank_stride apart) holds rows [r * seg_rows, ...) of every
            // estimator, each chunk laid out K0 [B][T][Sp_loc][32] then V0^T [B][T][32][Sp_loc]
            const int Sl = kv_pad(ks[i].seg_rows);
            a.Skv_pad = Sl; a.vt = kvl + (size_t)B * T * Sl * kD; a.kv_slots = 0;
            a.kv_seg_rows = ks[i].seg_rows; a.kv_seg_stride = ks[i].rank_stride / 2;
          }
        }
        if (phase != 2) MMPFN_TRY(proj_gemm(q, st));
        if (phase != 1) MMPFN_TRY(launch_tc_item_attn(a, st));
        off += (long long)B * S * T;
        entry += B;
      }
      if (phase != 1) MMPFN_TRY(out_proj_ln(lw, state, state_b, M, MMPFN_BF16, flat, st));
    }
    if (phase != 1) MMPFN_TRY(mlp(lw, state, state_b, M, MMPFN_BF16, flat, st));
  }
  return MMPFN_OK;
}

static int layers_multi(const mmpfn_geometry* g, const mmpfn_weights* w, float* state, uint16_t* state_b,
                        const mmpfn_segment* segs, int n_seg, int S, int n_train, int train, void* const* kv,
                        void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (!segs || !kv || n_seg < 1 || n_seg > MMPFN_MAX_SEGMENTS || !g) { set_error("layers_multi: bad segment list"); return MMPFN_EINVAL; }
  mmpfn_kv_segment ks[MMPFN_MAX_SEGMENTS];
  for (int i = 0; i < n_seg; ++i) {
    ks[i] = mmpfn_kv_segment{};
    ks[i].B = segs[i].B; ks[i].T = segs[i].T; ks[i].kv = kv[i];
  }
  return layers_run(g, w, state, state_b, ks, n_seg, S, n_train, train, 0, g->nlayers, 0, workspace, workspace_bytes, st);
}

int mmpfn_layers_train_multi(const mmpfn_geometry* g, const mmpfn_weights* w, float* state_f32, uint16_t* state_bf16,
                             const mmpfn_segment* segs, int n_seg, int S, void* const* kv, void* workspace,
                             size_t workspace_bytes, void* stream) {
  return layers_multi(g, w, state_f32, state_bf16, segs, n_seg, S, 0, 1, kv, workspace, workspace_bytes, (cudaStream_t)stream);
}

int mmpfn_layers_test_multi(const mmpfn_geometry* g, const mmpfn_weights* w, float* state_f32, uint16_t* state_bf16,
                            const mmpfn_segment* segs, int n_seg, int S, int n_train, void* const* kv, void* workspace,
                            size_t workspace_bytes, void* stream) {
  return layers_multi(g, w, state_f32, state_bf16, segs, n_seg, S, n_train, 0, kv, workspace, workspace_bytes, (cudaStream_t)stream);
}

int mmpfn_layers_run(const mmpfn_geometry* g, const mmpfn_weights* w, float* state_f32, uint16_t* state_bf16,
                     const mmpfn_kv_segment* segs, int n_seg, int S, int n_train, int train, int layer_begin,
                     int layer_end, int phase, void* workspace, size_t workspace_bytes, void* stream) {
  return layers_run(g, w, state_f32, state_bf16, segs, n_seg, S, n_train, train, layer_begin, layer_end, phase, workspace,
                    workspace_bytes, (cudaStream_t)stream);
}

// ---- per-entry row counts ----------------------------------------------------------------------------
size_t mmpfn_layers_ragged_ws_bytes(const mmpfn_geometry* g, const mmpfn_segment* segs, int n_seg, int S, int precision) {
  long long M = 0;
  if (check_geometry(g) != MMPFN_OK || check_segments(segs, n_seg, S, &M) != MMPFN_OK) return 0;
  if (precision == MMPFN_BF16) return carve_multi(nullptr, segs, n_seg, S, M).bytes;
  if (precision != MMPFN_F32) return 0;
  long long m_max = 0;         // fp32: one segment after another
  for (int i = 0; i < n_seg; ++i) {
    const long long m = (long long)segs[i].B * S * segs[i].T;
    if (m > m_max) m_max = m;
  }
  return carve(nullptr, m_max, 1, S, 2, MMPFN_F32).bytes;
}

static int layers_ragged(const mmpfn_geometry* g, const mmpfn_weights* w, float* state, uint16_t* state_b,
                         const mmpfn_segment* segs, int n_seg, int S, int n_train, int train, const int* n_rows,
                         const int* n_ctx, int precision, void* const* kv, void* workspace, size_t workspace_bytes,
                         cudaStream_t st) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  long long M = 0;
  if (!kv) { set_error("layers_ragged: null context list"); return MMPFN_EINVAL; }
  MMPFN_TRY(check_segments(segs, n_seg, S, &M));
  if (!train && n_train < 1) { set_error("layers_ragged: the test pass needs n_train >= 1"); return MMPFN_EINVAL; }
  if (precision == MMPFN_BF16) {
    mmpfn_kv_segment ks[MMPFN_MAX_SEGMENTS];
    for (int i = 0; i < n_seg; ++i) {
      ks[i] = mmpfn_kv_segment{};
      ks[i].B = segs[i].B; ks[i].T = segs[i].T; ks[i].kv = kv[i];
    }
    return layers_run(g, w, state, state_b, ks, n_seg, S, n_train, train, 0, g->nlayers, 0, workspace, workspace_bytes,
                      st, n_rows, n_ctx);
  }
  if (precision != MMPFN_F32 || !w || !w->layers_f32 || !state) { set_error("layers_ragged: bad arguments"); return MMPFN_EINVAL; }
  if (workspace_bytes < mmpfn_layers_ragged_ws_bytes(g, segs, n_seg, S, precision) || !workspace) {
    set_error("layers_ragged: workspace %zu bytes too small", workspace_bytes);
    return MMPFN_EINVAL;
  }
  long long off = 0, entry = 0;
  for (int i = 0; i < n_seg; ++i) {
    const int B = segs[i].B, T = segs[i].T;
    if (!train && !kv[i]) { set_error("layers_ragged: the test pass needs every segment's context"); return MMPFN_EINVAL; }
    const LayerWs ws = carve(workspace, (long long)B * S * T, B, S, T, MMPFN_F32);
    MMPFN_TRY(layers_f32(g, w, state + off * kE, B, S, T, n_train, train, kv[i], n_rows ? n_rows + entry : nullptr,
                         n_ctx ? n_ctx + entry : nullptr, ws, st));
    off += (long long)B * S * T;
    entry += B;
  }
  return MMPFN_OK;
}

int mmpfn_layers_train_ragged(const mmpfn_geometry* g, const mmpfn_weights* w, float* state_f32, uint16_t* state_bf16,
                              const mmpfn_segment* segs, int n_seg, int S, const int32_t* n_rows, int precision,
                              void* const* kv, void* workspace, size_t workspace_bytes, void* stream) {
  return layers_ragged(g, w, state_f32, state_bf16, segs, n_seg, S, 0, 1, n_rows, nullptr, precision, kv, workspace,
                       workspace_bytes, (cudaStream_t)stream);
}

int mmpfn_layers_test_ragged(const mmpfn_geometry* g, const mmpfn_weights* w, float* state_f32, uint16_t* state_bf16,
                             const mmpfn_segment* segs, int n_seg, int S, int n_train, const int32_t* n_rows,
                             const int32_t* n_ctx, int precision, void* const* kv, void* workspace,
                             size_t workspace_bytes, void* stream) {
  return layers_ragged(g, w, state_f32, state_bf16, segs, n_seg, S, n_train, 0, n_rows, n_ctx, precision, kv, workspace,
                       workspace_bytes, (cudaStream_t)stream);
}

int mmpfn_decode(const mmpfn_geometry* g, const mmpfn_weights* w, const float* state, int B, int S, int T,
                 float* hidden_scratch, float* logits, void* stream) {
  MMPFN_TRY(check_geometry(g));
  MMPFN_TRY(require_device());
  if (!w || !state || !hidden_scratch || !logits || B < 1 || S < 1 || T < 1) {
    set_error("decode: bad arguments");
    return MMPFN_EINVAL;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int M = B * S;
  // rows = the y token (last) of every row: lda = T*E, base offset (T-1)*E
  MMPFN_TRY(launch_sgemm(gemm(state + (size_t)(T - 1) * kE, T * kE, w->dec_w1, kE, w->dec_b1, hidden_scratch, kHid, M,
                              kHid, kE), EPI_GELU, st));
  return launch_sgemm(gemm(hidden_scratch, kHid, w->dec_w2, kHid, w->dec_b2, logits, g->n_out, M, g->n_out, kHid),
                      EPI_NONE, st);
}

int mmpfn_proba_tail(const float* logits, const int32_t* class_perm, const float* class_prior, int n_est, int S,
                     int n_out, int n_classes, float temperature, int average_before_softmax, float* proba,
                     void* stream) {
  MMPFN_TRY(require_device());
  if (!logits || !class_perm || !proba || n_est < 1 || S < 1) { set_error("proba_tail: bad arguments"); return MMPFN_EINVAL; }
  return launch_proba_tail(logits, class_perm, class_prior, n_est, S, n_out, n_classes, temperature,
                           average_before_softmax, proba, (cudaStream_t)stream);
}

int mmpfn_bar_tail(const float* logits, int n_est, int S, int K, const int32_t* src_bucket, const float* src_share,
                   const uint8_t* cancel, const float* borders, float temperature, int average_before_softmax,
                   const float* quantiles, int n_q, float* mean, float* median, float* mode, float* quant,
                   float* log_prob, void* stream) {
  MMPFN_TRY(require_device());
  if (!logits || !src_bucket || !src_share || !borders || n_est < 1 || S < 1 || K < 2 || n_q < 0 ||
      !(temperature > 0.f) || (quant && (!quantiles || n_q < 1))) {
    set_error("bar_tail: bad arguments (n_est %d S %d K %d n_q %d temperature %g)", n_est, S, K, n_q, temperature);
    return MMPFN_EINVAL;
  }
  if (!mean && !median && !mode && !quant && !log_prob) return MMPFN_OK;
  return launch_bar_tail(logits, nullptr, nullptr, 1, n_est, S, K, src_bucket, src_share, cancel, borders, temperature,
                         average_before_softmax, quantiles, n_q, mean, median, mode, quant, log_prob,
                         (cudaStream_t)stream);
}

int mmpfn_bar_tail_tasks(const float* const* logits, int n_tasks, int n_est, const int32_t* row_offset, int S_total,
                         int K, const int32_t* src_bucket, const float* src_share, const uint8_t* cancel,
                         const float* borders, float temperature, int average_before_softmax, const float* quantiles,
                         int n_q, float* mean, float* median, float* mode, float* quant, float* log_prob,
                         void* stream) {
  MMPFN_TRY(require_device());
  if (!logits || !row_offset || !src_bucket || !src_share || !borders || n_tasks < 1 || n_est < 1 || S_total < 1 ||
      K < 2 || n_q < 0 || !(temperature > 0.f) || (quant && (!quantiles || n_q < 1))) {
    set_error("bar_tail_tasks: bad arguments (n_tasks %d n_est %d S_total %d K %d n_q %d temperature %g)", n_tasks,
              n_est, S_total, K, n_q, temperature);
    return MMPFN_EINVAL;
  }
  if (!mean && !median && !mode && !quant && !log_prob) return MMPFN_OK;
  return launch_bar_tail(nullptr, logits, row_offset, n_tasks, n_est, S_total, K, src_bucket, src_share, cancel,
                         borders, temperature, average_before_softmax, quantiles, n_q, mean, median, mode, quant,
                         log_prob, (cudaStream_t)stream);
}

int mmpfn_layernorm(const float* x, const float* res, const float* gamma, const float* beta, int rows, int width,
                    float* y_f32, uint16_t* y_bf16, void* stream) {
  MMPFN_TRY(require_device());
  if (!x || (!y_f32 && !y_bf16) || rows < 1 || ((gamma == nullptr) != (beta == nullptr))) {
    set_error("layernorm: bad arguments");
    return MMPFN_EINVAL;
  }
  return launch_layernorm(x, res, gamma, beta, rows, width, y_f32, y_bf16, (cudaStream_t)stream);
}

int mmpfn_linear_f32(const float* A, const float* W, const float* bias, int M, int N, int K, int epi, float* out,
                     void* stream) {
  MMPFN_TRY(require_device());
  if (!A || !W || !out || (epi != 0 && epi != 1)) { set_error("linear_f32: bad arguments"); return MMPFN_EINVAL; }
  return launch_sgemm(gemm(A, K, W, K, bias, out, N, M, N, K), epi, (cudaStream_t)stream);
}

int mmpfn_linear_bf16(const uint16_t* A, const uint16_t* W, int M, int N, int K, int epi, uint16_t* out,
                      void* stream) {
  MMPFN_TRY(require_device());
  if (!A || !W || !out || (epi != 0 && epi != 1)) { set_error("linear_bf16: bad arguments"); return MMPFN_EINVAL; }
  TcGemm a{};
  a.A = A; a.W = W; a.M = M; a.N = N; a.K = K; a.epi = epi == 1 ? TC_EPI_GELU_BF16 : TC_EPI_BF16; a.out_bf16 = out;
  if (epi == 0 && K == kE && N % kE == 0) return proj_gemm(a, (cudaStream_t)stream);
  return launch_tc_gemm(a, (cudaStream_t)stream);
}

int mmpfn_linear_ln_bf16(const uint16_t* A, const uint16_t* W, int M, float* state_f32, uint16_t* state_bf16,
                         void* stream) {
  MMPFN_TRY(require_device());
  if (!A || !W || !state_f32 || !state_bf16 || M < 1) { set_error("linear_ln_bf16: bad arguments"); return MMPFN_EINVAL; }
  TcGemm o{};
  o.A = A; o.W = W; o.M = M; o.N = kE; o.K = kE; o.epi = TC_EPI_RESID_LN; o.resid_f32 = state_f32; o.ln_bf16 = state_bf16;
  return proj_gemm(o, (cudaStream_t)stream);
}

int mmpfn_item_qkv_bf16(const uint16_t* state_bf16, const uint16_t* w_qkv, int B, int S, int T, int S_pad, int n_proj,
                        uint16_t* q, uint16_t* k, uint16_t* vt, uint16_t* k0, uint16_t* vt0, void* stream) {
  MMPFN_TRY(require_device());
  if (!state_bf16 || !w_qkv || !q || B < 1 || S < 1 || T < 1 || S_pad < S || S_pad % 64 || (n_proj != 1 && n_proj != 3) ||
      (n_proj == 3 && (!k || !vt))) {
    set_error("item_qkv_bf16: bad arguments");
    return MMPFN_EINVAL;
  }
  TcGemm g{};
  g.A = state_bf16; g.W = w_qkv; g.N = n_proj * kE; g.K = kE; g.items = 1; g.B = B; g.S = S; g.T = T;
  g.epi = TC_EPI_QKV_ITEMS; g.q_out = q; g.k_out = k; g.vt_out = vt; g.k0_out = k0; g.vt0_out = vt0; g.S_pad = S_pad;
  return proj_gemm(g, (cudaStream_t)stream);
}

int mmpfn_mlp_bf16(float* state_f32, uint16_t* state_bf16, const uint16_t* w1, const uint16_t* w2, int M,
                   void* stream) {
  MMPFN_TRY(require_device());
  if (!state_f32 || !state_bf16 || !w1 || !w2 || M < 1) { set_error("mlp_bf16: bad arguments"); return MMPFN_EINVAL; }
  TcMlp f{};
  f.state_b = state_bf16; f.state_b_out = state_bf16; f.resid_f32 = state_f32; f.w1 = w1; f.w2 = w2; f.M = M;
  return launch_tc_mlp(f, (cudaStream_t)stream);
}

int mmpfn_item_attention_bf16(const uint16_t* q, const uint16_t* k, const uint16_t* vt, int B, int T, int n_q,
                              int Sq_pad, int n_kv, int Skv_pad, int shared_kv, uint16_t* out, void* stream) {
  MMPFN_TRY(require_device());
  if (!q || !k || !vt || !out || B < 1 || T < 1 || n_q < 1 || n_kv < 1 || Sq_pad < n_q || Skv_pad < n_kv ||
      Sq_pad % 8 || Skv_pad % 8) {
    set_error("item_attention_bf16: bad arguments");
    return MMPFN_EINVAL;
  }
  TcItemAttn a{};
  a.q = q; a.k = k; a.vt = vt; a.out = out; a.B = B; a.T = T; a.n_q = n_q; a.Sq_pad = Sq_pad; a.n_kv = n_kv;
  a.Skv_pad = Skv_pad; a.shared_kv = shared_kv;
  return launch_tc_item_attn(a, (cudaStream_t)stream);
}

int mmpfn_item_attention_bf16_ragged(const uint16_t* q, const uint16_t* k, const uint16_t* vt, int B, int T, int n_q,
                                     int Sq_pad, int n_kv, int Skv_pad, int shared_kv, const int32_t* q_len,
                                     const int32_t* kv_len, uint16_t* out, void* stream) {
  MMPFN_TRY(require_device());
  if (!q || !k || !vt || !out || !q_len || !kv_len || B < 1 || T < 1 || n_q < 1 || n_kv < 1 || Sq_pad < n_q ||
      Skv_pad < n_kv || Sq_pad % 8 || Skv_pad % 8) {
    set_error("item_attention_bf16_ragged: bad arguments");
    return MMPFN_EINVAL;
  }
  TcItemAttn a{};
  a.q = q; a.k = k; a.vt = vt; a.out = out; a.B = B; a.T = T; a.n_q = n_q; a.Sq_pad = Sq_pad; a.n_kv = n_kv;
  a.Skv_pad = Skv_pad; a.shared_kv = shared_kv; a.q_len = q_len; a.kv_len = kv_len;
  return launch_tc_item_attn(a, (cudaStream_t)stream);
}

int mmpfn_item_attention_f32(const float* q, const float* k, const float* v, int B, int T, int n_q, int n_kv,
                             int shared_kv, const int32_t* q_len, const int32_t* kv_len, float* out, void* stream) {
  MMPFN_TRY(require_device());
  if (!q || !k || !v || !out || B < 1 || T < 1 || n_q < 1 || n_kv < 1) {
    set_error("item_attention_f32: bad arguments");
    return MMPFN_EINVAL;
  }
  ItemAttnF32 a{};
  a.q = q; a.k = k; a.v = v; a.out = out;
  a.q_outer = (long long)n_q * T * kE; a.q_inner = kE; a.q_row = (long long)T * kE;
  a.o_outer = a.q_outer; a.o_inner = kE; a.o_row = a.q_row;
  if (shared_kv) {
    a.kv_outer = (long long)T * n_kv * kD; a.kv_inner = (long long)n_kv * kD; a.kv_row = kD;
  } else {
    a.kv_outer = (long long)n_kv * T * kE; a.kv_inner = kE; a.kv_row = (long long)T * kE;
  }
  a.planes = B * T; a.inner = T; a.n_q = n_q; a.n_kv = n_kv; a.shared_kv = shared_kv ? 1 : 0;
  a.q_len = q_len; a.kv_len = kv_len;
  return launch_item_attn_f32(a, (cudaStream_t)stream);
}

int mmpfn_feature_attention_bf16(const uint16_t* qkv, uint16_t* att, long long n_rows, int T, void* stream) {
  MMPFN_TRY(require_device());
  if (!qkv || !att || n_rows < 1 || T < 1) { set_error("feature_attention_bf16: bad arguments"); return MMPFN_EINVAL; }
  return launch_feat_attn_bf16(qkv, att, n_rows, T, (cudaStream_t)stream);
}

int mmpfn_feature_qkv_attention_bf16(const uint16_t* x, const uint16_t* w_qkv, long long n_rows, int T, uint16_t* att,
                                     void* stream) {
  MMPFN_TRY(require_device());
  if (!x || !w_qkv || !att || n_rows < 1 || T < 2) { set_error("feature_qkv_attention: bad arguments"); return MMPFN_EINVAL; }
  return launch_feat_qkv_attn(x, w_qkv, n_rows * T, T, att, (cudaStream_t)stream);
}

}  // extern "C"
