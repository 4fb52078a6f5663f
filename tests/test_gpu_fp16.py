"""The fp16 inference precision (MMPFN_F16): the tensor-core layer kernels instantiated for fp16 operands, the layer
passes, the model and the estimators.

* Every fp16 kernel against a float64 restatement computed from the same fp16 operands, with the bounds of
  ``test_gpu_layer_kernels.py`` and the fp16 unit roundoff 2^-11 in place of bf16's 2^-8; on the same fp32 inputs each
  kernel's fp16 error must also be below its bf16 error (the operand format really switched).
* An fp32 result past fp16's range is stored as +-65504 (satfinite), never inf.
* The whole model against the golden vectors, fp16 and bf16 side by side: fp16 is gated at a quarter of the bf16 gate
  and at a third of bf16's own deviation wherever that deviation is large enough to say anything (> 1e-5).
* Ragged passes and packed tasks in fp16 are bit-identical to each entry / task alone; the estimators run in fp16.
"""
import numpy as np
import pytest
import torch

from multimodalpfn_b200 import _lib
from multimodalpfn_b200.model import B200PerFeatureTransformer
from oracle.make_golden import MODEL_CASES
from tests.cases import check_proba, load_golden, model_case, softmax_np, t
from tests.test_gpu_layer_kernels import (E, FEAT_T, KV_EDGES, PATTERNS, POLY, Q_EDGES, U32, V_OFFSETS,
                                          _assert_tail_untouched, _attn_bound, _attn_ref, _i32, _item_inputs, _ln_check,
                                          _ln_rows, _nan, _pad64, _pad8, _ratio, _stream, LN_M)

pytestmark = pytest.mark.gpu

UF16 = 2.0 ** -11         # fp16 unit roundoff (11 significant bits)
F16_MAX = 65504.0
# fp16 item attention: as ITEM_BF16 with P and the output rounded to fp16
ITEM_F16 = dict(p_round=UF16 + POLY, out_round=UF16, k_score=64)
# fp16 feature attention: as FEAT_BF16 with fp16 P and output
FEAT_F16 = dict(p_round=UF16 + 2.0 ** -21, out_round=UF16, k_score=64)
# the fused feature QKV + attention against attention over float64 q / k / v rounded to fp16: where the kernel's fp32
# accumulation and the float64 product fall on the two sides of an fp16 rounding boundary, the kernel's q, k or v
# element is one fp16 ulp away from the reference's — a score moves by up to 2^-11 sabs (k_score 2^13 ulps of fp32)
# and an output by up to 2^-11 of P|V| (a second UF16 in p_round)
FUSED_F16 = dict(p_round=2 * UF16 + 2.0 ** -21, out_round=UF16, k_score=64 + 2 ** 13)

RATIOS = {}


def _note(name, r):
    RATIOS[name] = max(RATIOS.get(name, 0.0), r)
    print(f"max err/bound {name}: {RATIOS[name]:.3f}")


def _h(x):
    """float64 values rounded to fp16 (and back): the operands the fp16 kernels receive."""
    return x.to(torch.float16).double()


# ---------------------------------------------------------------------------------------------------------------
# item attention
# ---------------------------------------------------------------------------------------------------------------
def _f16_planes(q, k, v, Sq_pad, Skv_pad, kv_fill):
    P, n_q, _ = q.shape
    Pk, n_kv, _ = k.shape
    qb = torch.randn(P, Sq_pad, 32).to(torch.float16)
    qb[:, :n_q] = q.to(torch.float16)
    kb = torch.full((Pk, Skv_pad, 32), kv_fill, dtype=torch.float16)
    kb[:, :n_kv] = k.to(torch.float16)
    vt = torch.full((Pk, 32, Skv_pad), kv_fill, dtype=torch.float16)
    vt[:, :, :n_kv] = v.transpose(1, 2).to(torch.float16)
    return qb.cuda(), kb.cuda(), vt.cuda()


def _check_item(out_bth, q, k, v, shared, n_q, n_kv, T, consts, name):
    kk = k.repeat_interleave(6, 0) if shared else k
    vv = v.repeat_interleave(6, 0) if shared else v
    ref, pva, sabs = _attn_ref(q.cuda(), kk.cuda(), vv.cuda())
    got = out_bth.reshape(n_q, T, 6, 32).permute(1, 2, 0, 3).reshape(T * 6, n_q, 32)
    r = _ratio(got, ref, _attn_bound(ref, pva, sabs, n_kv, **consts))
    _note(name, r)
    return r


@pytest.mark.parametrize("shared", [0, 1])
@pytest.mark.parametrize("n_kv", KV_EDGES)
def test_item_attention_f16_vs_float64(n_kv, shared):
    """As test_item_attention_bf16_vs_float64: every n_q of Q_EDGES, every score pattern (references that move on every
    tile, every other tile, never), V with and without offset; keys past n_kv are NaN."""
    lib = _lib.load()
    B, T = 1, 2
    planes, kv_planes = B * T * 6, (B * T if shared else B * T * 6)
    g = torch.Generator().manual_seed(5000 + 1000 * n_kv + shared)
    for i, pattern in enumerate(PATTERNS):
        for v_off in V_OFFSETS:
            q_counts = [Q_EDGES[(2 * i + int(v_off > 0)) % len(Q_EDGES)]] if n_kv == 2000 else Q_EDGES
            for n_q in q_counts:
                q, k, v = (_h(a) for a in _item_inputs(planes, kv_planes, n_q, n_kv, pattern, v_off, g))
                Sq_pad, Skv_pad = _pad8(n_q), _pad64(n_kv)
                qb, kb, vt = _f16_planes(q, k, v, Sq_pad, Skv_pad, float("nan"))
                out, buf = _nan((B, n_q, T, E), torch.float16)
                _lib.check(lib.mmpfn_item_attention_f16(qb.data_ptr(), kb.data_ptr(), vt.data_ptr(), B, T, n_q, Sq_pad,
                                                        n_kv, Skv_pad, shared, None, None, buf.data_ptr(), _stream()),
                           "item_attention_f16")
                torch.cuda.synchronize()
                _assert_tail_untouched(buf, out.numel())
                r = _check_item(out[0], q, k, v, shared, n_q, n_kv, T, ITEM_F16, "item_attention_f16")
                assert r <= 1.0, (pattern, v_off, n_q, r)


@pytest.mark.parametrize("shared", [0, 1])
def test_item_attention_f16_ragged_vs_float64(shared):
    """Per-entry key counts at every tile edge and query counts cycling through Q_EDGES in one launch; pad output rows
    exactly zero, key rows between an entry's count and the capacity zero, rows past the capacity NaN."""
    lib = _lib.load()
    kv_len = KV_EDGES
    B, T = len(kv_len), 1
    q_len = [Q_EDGES[b % len(Q_EDGES)] for b in range(B)]
    n_q, n_kv = max(q_len), max(kv_len)
    Sq_pad, Skv_pad = _pad8(n_q), _pad64(n_kv)
    per_q, per_kv = T * 6, (T if shared else T * 6)
    for pattern in ("random1", "up8.25", "up7.75"):
        for v_off in V_OFFSETS:
            g = torch.Generator().manual_seed(177 + shared)
            ents = [tuple(_h(a) for a in _item_inputs(per_q, per_kv, q_len[b], kv_len[b], pattern, v_off, g))
                    for b in range(B)]
            qb = torch.zeros(B * per_q, Sq_pad, 32, dtype=torch.float16)
            kb = torch.full((B * per_kv, Skv_pad, 32), float("nan"), dtype=torch.float16)
            vt = torch.full((B * per_kv, 32, Skv_pad), float("nan"), dtype=torch.float16)
            kb[:, :n_kv] = 0
            vt[:, :, :n_kv] = 0
            for b, (q, k, v) in enumerate(ents):
                qb[b * per_q:(b + 1) * per_q, :q_len[b]] = q.to(torch.float16)
                kb[b * per_kv:(b + 1) * per_kv, :kv_len[b]] = k.to(torch.float16)
                vt[b * per_kv:(b + 1) * per_kv, :, :kv_len[b]] = v.transpose(1, 2).to(torch.float16)
            qb, kb, vt = qb.cuda(), kb.cuda(), vt.cuda()
            out, buf = _nan((B, n_q, T, E), torch.float16)
            ql, kl = _i32(q_len), _i32(kv_len)
            _lib.check(lib.mmpfn_item_attention_f16(qb.data_ptr(), kb.data_ptr(), vt.data_ptr(), B, T, n_q, Sq_pad,
                                                    n_kv, Skv_pad, shared, ql.data_ptr(), kl.data_ptr(),
                                                    buf.data_ptr(), _stream()), "item_attention_f16 ragged")
            torch.cuda.synchronize()
            _assert_tail_untouched(buf, out.numel())
            for b, (q, k, v) in enumerate(ents):
                assert (out[b, q_len[b]:] == 0).all(), b
                r = _check_item(out[b, :q_len[b]], q, k, v, shared, q_len[b], kv_len[b], T, ITEM_F16,
                                "item_attention_f16_ragged")
                assert r <= 1.0, (pattern, v_off, b, q_len[b], kv_len[b], r)


# ---------------------------------------------------------------------------------------------------------------
# feature attention, stand-alone and fused with its QKV projection
# ---------------------------------------------------------------------------------------------------------------
def _feat_ref_ratio(att, qkv64, n_rows, T, consts):
    worst = 0.0
    xd = qkv64.view(n_rows, T, 3, 6, 32)
    step = max(1, 2 ** 27 // (36 * T * T))
    for r0 in range(0, n_rows, step):
        r1 = min(n_rows, r0 + step)
        q, k, v = (xd[r0:r1, :, j].permute(0, 2, 1, 3) for j in range(3))
        ref, pva, sabs = _attn_ref(q, k, v)
        got = att.view(n_rows, T, 6, 32)[r0:r1].permute(0, 2, 1, 3)
        worst = max(worst, _ratio(got, ref, _attn_bound(ref, pva, sabs, T, **consts)))
    return worst


@pytest.mark.parametrize("T", FEAT_T)
def test_feature_attention_f16_vs_float64(T):
    """Every register-tile size and the CUDA-core fallback above 192 tokens; scores at scales 1 and 8, V with and
    without offset."""
    lib = _lib.load()
    n_rows = 5 if T <= 192 else 2
    for scale in (1.0, 8.0):
        for v_off in V_OFFSETS:
            g = torch.Generator(device="cuda").manual_seed(T * 10 + int(scale) + int(v_off) + 7)
            x = torch.randn(n_rows * T, 3, 6, 32, device="cuda", generator=g)
            x[:, :2] *= scale ** 0.5
            x[:, 2] += v_off
            qkv = x.reshape(n_rows * T, 3 * E).to(torch.float16)
            att, buf = _nan((n_rows * T, E), torch.float16)
            _lib.check(lib.mmpfn_feature_attention_f16(qkv.data_ptr(), buf.data_ptr(), n_rows, T, _stream()),
                       "feature_attention_f16")
            torch.cuda.synchronize()
            _assert_tail_untouched(buf, att.numel())
            r = _feat_ref_ratio(att, qkv.double(), n_rows, T, FEAT_F16)
            _note("feature_attention_f16", r)
            assert r <= 1.0, (scale, v_off, r)


@pytest.mark.parametrize("T", [2, 15, 16, 17, 31, 32, 33, 63, 64])
def test_feature_qkv_attention_f16_vs_float64(T):
    """The fused kernel (rows of up to 64 tokens) against float64 attention over the qkv block projected from the same
    fp16 operands and rounded to fp16, as the kernel rounds it."""
    lib = _lib.load()
    n_rows = 3001 // T + 1
    for scale, v_off in ((1.0, 0.0), (4.0, 4.0)):
        g = torch.Generator(device="cuda").manual_seed(900 + T + int(scale))
        x = torch.randn(n_rows * T, E, device="cuda", generator=g).to(torch.float16)
        w = torch.randn(3 * E, E, device="cuda", generator=g) / E ** 0.5
        w[:2 * E] *= scale ** 0.5
        w = w.to(torch.float16)
        bias_v = torch.zeros(3 * E, dtype=torch.float64, device="cuda")
        att, buf = _nan((n_rows * T, E), torch.float16)
        if v_off:                    # V offset: one input column constant, its V weights carry the offset
            x[:, 0] = 1.0
            w[2 * E:, 0] = v_off
        _lib.check(lib.mmpfn_feature_qkv_attention_f16(x.data_ptr(), w.data_ptr(), n_rows, T, buf.data_ptr(),
                                                       _stream()), "feature_qkv_attention_f16")
        torch.cuda.synchronize()
        _assert_tail_untouched(buf, att.numel())
        qkv = _h(x.double() @ w.double().T + bias_v)
        r = _feat_ref_ratio(att, qkv, n_rows, T, FUSED_F16)
        _note("feature_qkv_attention_f16", r)
        assert r <= 1.0, (scale, v_off, r)


# ---------------------------------------------------------------------------------------------------------------
# item QKV scatter
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_proj", [1, 3])
@pytest.mark.parametrize("S", [1, 127, 129, 300])
def test_item_qkv_f16_vs_float64(S, n_proj):
    """q / k planes, the V^T planes and the head-0 context copies against the float64 projection of the same fp16
    operands: one fp16 rounding per element on top of the fp32 accumulation.  Pad rows S .. S_pad-1 of the q and k
    planes (and of the k0 copy) are zero; nothing is written past the buffers."""
    lib = _lib.load()
    B, T = 2, 3
    S_pad = _pad64(S)
    g = torch.Generator(device="cuda").manual_seed(S * 7 + n_proj)
    x = torch.randn(B, S, T, E, device="cuda", generator=g).to(torch.float16)
    w = (torch.randn(n_proj * E, E, device="cuda", generator=g) / E ** 0.5).to(torch.float16)
    P, P0 = B * T * 6, B * T
    q, qb = _nan((P, S_pad, 32), torch.float16)
    k, kb = _nan((P, S_pad, 32), torch.float16)
    vt, vb = _nan((P, 32, S_pad), torch.float16)
    k0, k0b = _nan((P0, S_pad, 32), torch.float16)
    vt0, vt0b = _nan((P0, 32, S_pad), torch.float16)
    three = n_proj == 3
    _lib.check(lib.mmpfn_item_qkv_f16(x.data_ptr(), w.data_ptr(), B, S, T, S_pad, n_proj, qb.data_ptr(),
                                      kb.data_ptr() if three else None, vb.data_ptr() if three else None,
                                      k0b.data_ptr() if three else None, vt0b.data_ptr() if three else None,
                                      _stream()), "item_qkv_f16")
    torch.cuda.synchronize()
    for view, buf in ((q, qb), (k, kb), (vt, vb), (k0, k0b), (vt0, vt0b)):
        _assert_tail_untouched(buf, view.numel())
    ref = x.double() @ w.double().T                                   # [B][S][T][n_proj*192]
    bound = UF16 * ref.abs() + 2 * E * U32 * (x.double().abs() @ w.double().abs().T) + 1e-7
    # [B][S][T][j][h][d] -> planes (b, t, h) [S][d]
    ref6 = ref.view(B, S, T, n_proj, 6, 32).permute(3, 0, 2, 4, 1, 5).reshape(n_proj, P, S, 32)
    bnd6 = bound.view(B, S, T, n_proj, 6, 32).permute(3, 0, 2, 4, 1, 5).reshape(n_proj, P, S, 32)
    worst = float(((q[:, :S].double() - ref6[0]).abs() / bnd6[0]).max())
    assert (q[:, S:] == 0).all(), "pad rows of the q planes must be zero"
    if three:
        worst = max(worst, float(((k[:, :S].double() - ref6[1]).abs() / bnd6[1]).max()))
        worst = max(worst, float(((vt[:, :, :S].double() - ref6[2].transpose(1, 2)).abs() / bnd6[2].transpose(1, 2)).max()))
        assert (k[:, S:] == 0).all(), "pad rows of the k planes must be zero"
        # head-0 context: exactly the head-0 planes
        k_h0 = k.view(B * T, 6, S_pad, 32)[:, 0]
        vt_h0 = vt.view(B * T, 6, 32, S_pad)[:, 0]
        assert torch.equal(k0, k_h0)
        assert torch.equal(vt0[:, :, :S], vt_h0[:, :, :S])
    _note("item_qkv_f16", worst)
    assert worst <= 1.0, worst


# ---------------------------------------------------------------------------------------------------------------
# LayerNorm epilogues
# ---------------------------------------------------------------------------------------------------------------
def test_linear_ln_f16_row_statistics():
    """As test_linear_ln_bf16_row_statistics (rows with |mean| up to 4096 x their std), fp16 operands and shadow."""
    lib = _lib.load()
    x, std, zero = _ln_rows(LN_M, E, seed=11)
    g = torch.Generator().manual_seed(12)
    a = (torch.randn(LN_M, E, generator=g, dtype=torch.float64) * std[:, None]).to(torch.float16)
    w = (torch.randn(E, E, generator=g) / E ** 0.5).to(torch.float16)
    st, ad, wd = x.cuda(), a.cuda(), w.cuda()
    sth, buf = _nan((LN_M, E), torch.float16)
    _lib.check(lib.mmpfn_linear_ln_f16(ad.data_ptr(), wd.data_ptr(), LN_M, st.data_ptr(), buf.data_ptr(), _stream()),
               "linear_ln_f16")
    torch.cuda.synchronize()
    _assert_tail_untouched(buf, sth.numel())
    pre = x.double().cuda() + a.double().cuda() @ w.double().cuda().T
    # fp16 shadow: one fp16 rounding of O(4) values (4 * 2^-11 = 0.002)
    r32, r16, worst = _ln_check(st, sth, pre, zero.cuda(), 2e-4, 0.004)
    _note("linear_ln_f16 fp32", r32)
    _note("linear_ln_f16 fp16", r16)
    assert r32 <= 1.0 and r16 <= 1.0, (r32, r16, worst)


def test_mlp_f16_row_statistics():
    """As test_mlp_bf16_row_statistics, fp16 operands, hidden activation and shadow.  The MMA input is scaled by
    2^-4 x the row's std (2^-8 in the bf16 test would put it among fp16's subnormals): the sublayer still adds only
    ~2 % of the row's spread, so the GELU form and the fp16 hidden activation stay below the fp32 base."""
    lib = _lib.load()
    x, std, zero = _ln_rows(LN_M, E, seed=13)
    g = torch.Generator().manual_seed(14)
    xh = (torch.randn(LN_M, E, generator=g, dtype=torch.float64) * std[:, None] / 16).to(torch.float16)
    w1 = (torch.randn(768, E, generator=g) / E ** 0.5).to(torch.float16)
    w2 = (torch.randn(E, 768, generator=g) / 768 ** 0.5).to(torch.float16)
    st, sth, w1d, w2d = x.cuda(), xh.cuda(), w1.cuda(), w2.cuda()
    _lib.check(lib.mmpfn_mlp_f16(st.data_ptr(), sth.data_ptr(), w1d.data_ptr(), w2d.data_ptr(), LN_M, _stream()),
               "mlp_f16")
    torch.cuda.synchronize()
    h = torch.nn.functional.gelu(xh.double().cuda() @ w1.double().cuda().T)
    pre = x.double().cuda() + h @ w2.double().cuda().T
    r32, r16, worst = _ln_check(st, sth, pre, zero.cuda(), 2e-4, 0.004)
    _note("mlp_f16 fp32", r32)
    _note("mlp_f16 fp16", r16)
    assert r32 <= 1.0 and r16 <= 1.0, (r32, r16, worst)


# ---------------------------------------------------------------------------------------------------------------
# the format really switched: on the same fp32 inputs the fp16 kernel is closer to float64 than the bf16 one
# ---------------------------------------------------------------------------------------------------------------
def _both(fn, *xs):
    """fn(format tag, 16-bit copies of xs) for bf16 and fp16 -> the two outputs as float64."""
    return [fn(tag, *(x.to(dt) for x in xs)).double() for tag, dt in (("bf16", torch.bfloat16), ("f16", torch.float16))]


def _cmp(name, outs, ref):
    eb, eh = (float((o - ref).abs().max()) for o in outs)
    print(f"{name}: max err bf16 {eb:.3e}  fp16 {eh:.3e}  ratio {eh / eb:.3f}")
    assert eh < eb, (name, eb, eh)


def test_f16_error_below_bf16():
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(2024)
    st = _stream()
    # item attention (train form, B = 1, T = 2, 300 queries, 500 keys)
    n_q, n_kv, T = 300, 500, 2
    q = torch.randn(12, n_q, 32, device="cuda", generator=g)
    k = torch.randn(12, n_kv, 32, device="cuda", generator=g)
    v = torch.randn(12, n_kv, 32, device="cuda", generator=g) + 1
    ref = _attn_ref(q, k, v)[0].view(T, 6, n_q, 32).permute(2, 0, 1, 3).reshape(1, n_q, T, E)

    def item(tag, q, k, v):
        Sq, Skv = _pad8(n_q), _pad64(n_kv)
        qp = torch.zeros(12, Sq, 32, dtype=q.dtype, device="cuda"); qp[:, :n_q] = q
        kp = torch.zeros(12, Skv, 32, dtype=q.dtype, device="cuda"); kp[:, :n_kv] = k
        vp = torch.zeros(12, 32, Skv, dtype=q.dtype, device="cuda"); vp[:, :, :n_kv] = v.transpose(1, 2)
        out = torch.empty(1, n_q, T, E, dtype=q.dtype, device="cuda")
        if tag == "bf16":
            rc = lib.mmpfn_item_attention_bf16(qp.data_ptr(), kp.data_ptr(), vp.data_ptr(), 1, T, n_q, Sq, n_kv, Skv, 0,
                                               out.data_ptr(), st)
        else:
            rc = lib.mmpfn_item_attention_f16(qp.data_ptr(), kp.data_ptr(), vp.data_ptr(), 1, T, n_q, Sq, n_kv, Skv, 0,
                                              None, None, out.data_ptr(), st)
        _lib.check(rc, "item attention " + tag)
        torch.cuda.synchronize()
        return out
    _cmp("item_attention", _both(item, q, k, v), ref)

    # feature attention (T = 20 and T = 100) and the fused QKV + feature attention (T = 20)
    for Tf in (20, 100):
        n_rows = 200
        qkv = torch.randn(n_rows * Tf, 3 * E, device="cuda", generator=g)
        xd = qkv.double().view(n_rows, Tf, 3, 6, 32)
        ref = _attn_ref(*(xd[:, :, j].permute(0, 2, 1, 3) for j in range(3)))[0].permute(0, 2, 1, 3).reshape(-1, E)

        def feat(tag, qkv):
            att = torch.empty(n_rows * Tf, E, dtype=qkv.dtype, device="cuda")
            fn = lib.mmpfn_feature_attention_bf16 if tag == "bf16" else lib.mmpfn_feature_attention_f16
            _lib.check(fn(qkv.data_ptr(), att.data_ptr(), n_rows, Tf, st), "feature attention " + tag)
            torch.cuda.synchronize()
            return att
        _cmp(f"feature_attention T={Tf}", _both(feat, qkv), ref)
    n_rows, Tf = 200, 20
    x = torch.randn(n_rows * Tf, E, device="cuda", generator=g)
    w = torch.randn(3 * E, E, device="cuda", generator=g) / E ** 0.5
    xd = (x.double() @ w.double().T).view(n_rows, Tf, 3, 6, 32)
    ref = _attn_ref(*(xd[:, :, j].permute(0, 2, 1, 3) for j in range(3)))[0].permute(0, 2, 1, 3).reshape(-1, E)

    def fused(tag, x, w):
        att = torch.empty(n_rows * Tf, E, dtype=x.dtype, device="cuda")
        fn = lib.mmpfn_feature_qkv_attention_bf16 if tag == "bf16" else lib.mmpfn_feature_qkv_attention_f16
        _lib.check(fn(x.data_ptr(), w.data_ptr(), n_rows, Tf, att.data_ptr(), st), "fused feature attention " + tag)
        torch.cuda.synchronize()
        return att
    _cmp("feature_qkv_attention", _both(fused, x, w), ref)

    # item QKV scatter (q planes)
    B, S, T = 1, 200, 2
    x = torch.randn(B, S, T, E, device="cuda", generator=g)
    w = torch.randn(E, E, device="cuda", generator=g) / E ** 0.5
    ref = (x.double() @ w.double().T).view(B, S, T, 6, 32).permute(0, 2, 3, 1, 4).reshape(B * T * 6, S, 32)

    def qkv_items(tag, x, w):
        qo = torch.zeros(B * T * 6, 256, 32, dtype=x.dtype, device="cuda")
        fn = lib.mmpfn_item_qkv_bf16 if tag == "bf16" else lib.mmpfn_item_qkv_f16
        _lib.check(fn(x.data_ptr(), w.data_ptr(), B, S, T, 256, 1, qo.data_ptr(), None, None, None, None, st),
                   "item qkv " + tag)
        torch.cuda.synchronize()
        return qo[:, :S]
    _cmp("item_qkv", _both(qkv_items, x, w), ref)

    # out-projection + LayerNorm and the fused MLP: the 16-bit shadow they write
    M = 5000
    state = torch.randn(M, E, device="cuda", generator=g)
    a = torch.randn(M, E, device="cuda", generator=g)
    w = torch.randn(E, E, device="cuda", generator=g) / E ** 0.5
    ref = torch.nn.functional.layer_norm(state.double() + a.double() @ w.double().T, (E,), eps=1e-5)

    def lin_ln(tag, a, w):
        s = state.clone()
        sh = torch.empty(M, E, dtype=a.dtype, device="cuda")
        fn = lib.mmpfn_linear_ln_bf16 if tag == "bf16" else lib.mmpfn_linear_ln_f16
        _lib.check(fn(a.data_ptr(), w.data_ptr(), M, s.data_ptr(), sh.data_ptr(), st), "linear_ln " + tag)
        torch.cuda.synchronize()
        return sh
    _cmp("linear_ln (shadow)", _both(lin_ln, a, w), ref)
    w1 = torch.randn(768, E, device="cuda", generator=g) / E ** 0.5
    w2 = torch.randn(E, 768, device="cuda", generator=g) / 768 ** 0.5
    ref = torch.nn.functional.layer_norm(
        state.double() + torch.nn.functional.gelu(state.double() @ w1.double().T) @ w2.double().T, (E,), eps=1e-5)

    def mlp(tag, s16, w1, w2):
        s = state.clone()
        fn = lib.mmpfn_mlp_bf16 if tag == "bf16" else lib.mmpfn_mlp_f16
        _lib.check(fn(s.data_ptr(), s16.data_ptr(), w1.data_ptr(), w2.data_ptr(), M, st), "mlp " + tag)
        torch.cuda.synchronize()
        return s
    _cmp("mlp (fp32 state)", _both(mlp, state, w1, w2), ref)


def test_f16_saturates_instead_of_inf():
    """Projections whose fp32 result is past fp16's range are stored as +-65504 (cvt.rn.satfinite), not inf."""
    lib = _lib.load()
    B, S, T = 1, 64, 2
    x = torch.full((B, S, T, E), 16.0, dtype=torch.float16, device="cuda")
    w = torch.full((E, E), 32.0, dtype=torch.float16, device="cuda")
    w[1::2] = -32.0                                   # 192 * 16 * 32 = 98304 > 65504, both signs
    q = torch.zeros(B * T * 6, S, 32, dtype=torch.float16, device="cuda")
    _lib.check(lib.mmpfn_item_qkv_f16(x.data_ptr(), w.data_ptr(), B, S, T, S, 1, q.data_ptr(), None, None, None, None,
                                      _stream()), "item_qkv_f16")
    torch.cuda.synchronize()
    assert torch.isfinite(q).all()
    vals = set(q.float().unique().tolist())
    assert vals == {F16_MAX, -F16_MAX}, vals


# ---------------------------------------------------------------------------------------------------------------
# the whole model against the golden vectors, fp16 and bf16 side by side
# ---------------------------------------------------------------------------------------------------------------
def _joint(model, X, img, y):
    out = model(None, None if X is None else torch.as_tensor(X)[:, None].cuda(),
                None if img is None else torch.as_tensor(img).cuda(), torch.as_tensor(y).cuda(),
                only_return_standard_out=True, categorical_inds=[], single_eval_pos=len(y))
    return out.squeeze(1).cpu().numpy()


def _cached(model, X, img, y, n_tr):
    ctx = model.fit_context(t(X[:n_tr]), None if img is None else t(img[:n_tr]), t(y))
    return model.predict_with_context(ctx, t(X[n_tr:]), None if img is None else t(img[n_tr:]))[0].cpu().numpy()


def _gate(name, form, dp16, dpbf, agree16):
    print(f"[{name} {form}] max|dp| fp16 {dp16:.3e}  bf16 {dpbf:.3e}  fp16/bf16 {dp16 / max(dpbf, 1e-30):.3f}  "
          f"fp16 argmax agreement {agree16:.2%}")
    if name == "stress_tiny":
        assert dp16 <= dpbf / 3 and agree16 == 1.0, (name, form, dp16, dpbf, agree16)
        return
    assert dp16 <= 5e-4, (name, form, dp16)
    if dpbf > 1e-5:
        assert dp16 <= dpbf / 3, (name, form, dp16, dpbf)


@pytest.mark.parametrize("form", ["joint", "cached"])
@pytest.mark.parametrize("name", list(MODEL_CASES))
def test_model_f16_vs_golden(name, form):
    geom, sd, X, img, y, n_tr = model_case(name)
    g = load_golden("model_" + name)
    key = "logits" if form == "joint" else "logits_cached"
    if key not in g:
        pytest.skip(f"the golden file of {name} has no {key}")
    if form == "cached" and X is None:
        pytest.skip("the cached form takes a table")
    pg = softmax_np(g[key][:, :3] / 0.9)
    dps, agree = {}, {}
    for precision in ("fp16", "bf16"):
        model = B200PerFeatureTransformer(sd, geom, precision=precision, seed=0)
        logits = _joint(model, X, img, y) if form == "joint" else _cached(model, X, img, y, n_tr)
        assert np.isfinite(logits).all()
        p = softmax_np(logits[:, :3] / 0.9)
        dps[precision] = float(np.abs(p - pg).max())
        agree[precision] = float((p.argmax(1) == pg.argmax(1)).mean())
    _gate(name, form, dps["fp16"], dps["bf16"], agree["fp16"])


def test_large_clf8_pad_ufes_f16():
    """configs[1] (8 estimators, PAD-UFES shape) through the engine's multi-group pass in fp16 against the real
    reference's fp32 probabilities: argmax agreement in full or the margin rule of check_proba, at a quarter of the
    bf16 gate."""
    from multimodalpfn_b200.engine import proba_from_logits
    from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
    g = load_golden("large_clf8_pad_ufes")
    geom = Geometry(mgm_heads=8, cap_heads=8)
    sd = make_state_dict(geom, seed=1)
    d = make_dataset("pad_ufes", 0)
    n_est, n_tr = int(g["n_estimators"]), len(d["y_train"])
    model = B200PerFeatureTransformer(sd, geom, precision="fp16", seed=0)
    img = torch.as_tensor(np.concatenate([d["img_train"], d["img_test"]])).cuda()
    by_f = {}
    for e in range(n_est):
        by_f.setdefault(g[f"X_full_{e}"].shape[1], []).append(e)
    tok = model.stem_image(img)
    groups = [(es, torch.as_tensor(np.stack([g[f"X_full_{e}"] for e in es])).cuda(),
               torch.as_tensor(np.stack([g[f"y_train_{e}"] for e in es])).cuda()) for _, es in sorted(by_f.items())]
    ctxs = model.fit_contexts([dict(X_train=Xb[:, :n_tr].contiguous(), y_train=yb, X_all=Xb,
                                    img_tok_train=tok[:n_tr].contiguous()) for _, Xb, yb in groups])
    outs = model.predict_with_contexts(ctxs, [Xb[:, n_tr:].contiguous() for _, Xb, _ in groups],
                                       img_tok_test=tok[n_tr:].contiguous())
    logits = [None] * n_est
    for (es, _, _), out in zip(groups, outs):
        for i, e in enumerate(es):
            logits[e] = out[i]
    proba = proba_from_logits(torch.stack(logits), [g[f"class_perm_{e}"] for e in range(n_est)],
                              n_classes=int(g["n_classes"]), class_counts=g["class_counts"])
    check_proba(proba, g["proba"], 5e-4, "clf8 fp16")


def test_classifier_torch_float16_vs_fp32():
    """MMPFNClassifier(inference_precision=torch.float16) on the PAD-UFES shape (8 estimators) against the same
    classifier in fp32: within a quarter of the bf16 gate, argmax agreement in full or the margin rule."""
    from multimodalpfn_b200.classifier import MMPFNClassifier
    from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
    geom = Geometry(mgm_heads=8, cap_heads=8)
    sd = make_state_dict(geom, seed=1)
    d = make_dataset("pad_ufes", 0)
    out = {}
    for p in (torch.float16, "fp32"):
        clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=8, cap_heads=8, features_per_group=2, n_estimators=8,
                              model_path=(sd, geom), device="cuda", inference_precision=p,
                              ignore_pretraining_limits=True, random_state=0)
        clf.fit(d["X_train"], d["img_train"], d["y_train"])
        assert clf.executor_.model.precision_name == ("fp16" if p is torch.float16 else "fp32")
        out[str(p)] = clf.predict_proba(d["X_test"], d["img_test"])
    check_proba(out[str(torch.float16)], out["fp32"], 5e-4, "classifier torch.float16 vs fp32")


# ---------------------------------------------------------------------------------------------------------------
# ragged passes and packed tasks, bit for bit
# ---------------------------------------------------------------------------------------------------------------
def test_ragged_pass_f16_equals_each_entry_alone():
    from tests.test_gpu_ragged import test_ragged_pass_equals_each_entry_alone as run
    run("fp16")


def test_ragged_regression_pass_f16_equals_each_entry_alone():
    from tests.test_gpu_regression_tasks import test_ragged_regression_pass_equals_each_entry_alone as run
    run("fp16")


def test_packed_tasks_f16_equal_one_by_one():
    from tests.test_gpu_tasks import test_packed_tasks_equal_one_by_one as run
    run("fp16")


def test_regression_tasks_f16_equal_one_by_one():
    from tests.test_gpu_regression_tasks import test_regression_tasks_equal_one_by_one as run
    run("fp16", 64, False)


# ---------------------------------------------------------------------------------------------------------------
# estimator surface
# ---------------------------------------------------------------------------------------------------------------
def test_regressor_f16_end_to_end_vs_oracle():
    from tests.test_gpu_regressor import test_regressor_end_to_end_vs_oracle as run
    run(64, "fp16")


def test_regressor_f16_fit_with_cache_equals_fit_preprocessors():
    from tests.test_gpu_regressor import _regression_data, _regressor
    d, y_tr, _ = _regression_data(1)
    outs = []
    for mode in ("fit_preprocessors", "fit_with_cache"):
        reg = _regressor(64, "fp16", fit_mode=mode).fit(d["X_train"], d["img_train"], y_tr)
        assert reg.model_.precision_name == "fp16"
        outs.append(reg.predict(d["X_test"], d["img_test"], output_type="full"))
    for k in ("mean", "median", "mode", "logits"):
        assert np.array_equal(outs[0][k], outs[1][k]), k
    assert np.array_equal(np.stack(outs[0]["quantiles"]), np.stack(outs[1]["quantiles"]))


def _f16_classifier(n_est=4):
    from multimodalpfn_b200.classifier import MMPFNClassifier
    from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
    geom = Geometry(mgm_heads=2, cap_heads=4)
    sd = make_state_dict(geom, seed=3)
    d = make_dataset("pad_ufes_small", 0)
    clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=2, cap_heads=4, features_per_group=2, n_estimators=n_est,
                          model_path=(sd, geom), device="cuda", inference_precision="fp16",
                          ignore_pretraining_limits=True, random_state=0)
    clf.fit(d["X_train"], d["img_train"], d["y_train"])
    return clf, d


def test_graph_replay_f16_equals_eager():
    from multimodalpfn_b200.preprocessing import transform_all
    clf, d = _f16_classifier()
    eng = clf.executor_
    for X, I in ((d["X_test"], d["img_test"]), (d["X_test"][:77], d["img_test"][:77])):
        staged = eng.stage(transform_all(clf.members_, X), I)
        a = eng.logits_graphed(staged).clone()
        b = eng.logits_staged(staged).clone()
        assert torch.isfinite(a).all() and torch.equal(a, b), X.shape


def test_classifier_f16_fit_with_cache_equals_fit_preprocessors():
    from multimodalpfn_b200.classifier import MMPFNClassifier
    from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
    geom = Geometry(mgm_heads=2, cap_heads=4)
    sd = make_state_dict(geom, seed=3)
    d = make_dataset("pad_ufes_small", 0)
    outs = []
    for mode in ("fit_preprocessors", "fit_with_cache"):
        clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=2, cap_heads=4, features_per_group=2, n_estimators=4,
                              model_path=(sd, geom), device="cuda", inference_precision="fp16", fit_mode=mode,
                              ignore_pretraining_limits=True, random_state=0)
        clf.fit(d["X_train"], d["img_train"], d["y_train"])
        outs.append(clf.predict_proba(d["X_test"], d["img_test"]))
    assert np.array_equal(outs[0], outs[1]), float(np.abs(outs[0] - outs[1]).max())


def test_sharded_engine_refuses_f16():
    from multimodalpfn_b200.dist import ShardedEngine
    clf, _ = _f16_classifier()
    with pytest.raises(ValueError, match="fp16"):
        ShardedEngine(clf.executor_, 0, 2, group="emulate")
    with pytest.raises(ValueError, match="bf16 only"):
        m = clf.executor_.model
        m.layers_run(None, None, [], 1, None, 0, 1)
