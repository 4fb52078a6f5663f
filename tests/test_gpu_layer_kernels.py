"""The kernels of the twelve layers, each against a float64 restatement of the same operation computed from the same
bf16 / fp32 operands the kernel received:

* ``mmpfn_item_attention_bf16`` / ``_bf16_ragged`` / ``_f32``: key counts at the edges of the 48-key tiles and of the
  64-key V^T blocks, query counts at the edges of the 128-row tiles, the shared head-0 K/V with the six heads stacked on
  the tile rows, and score ramps that move the lazy softmax reference (kernels_attn.cu: it only follows the running
  maximum when a tile's row sum exceeds 2^8) on every tile, every other tile, or never;
* ``mmpfn_feature_attention_bf16``: every register-tile size, the CUDA-core fallback above 192 tokens and its limit;
* the LayerNorm epilogues of ``mmpfn_linear_ln_bf16`` (out-projection) and ``mmpfn_mlp_bf16`` (fused MLP) on rows
  whose mean is large against their spread, with ``mmpfn_layernorm`` as the control.

Attention tolerances are per element and scale-aware: |out - ref| <= a * (P|V|) + b * |ref| + c, where P|V| is the
float64 softmax(S) @ |V| (see ``_attn_bound``).  Every attention case runs with zero-mean V and with V = 4 + randn: the
offset turns any error of the softmax normaliser (a key counted or dropped, a missed rescale) into an output shift of
about 4 x that key's weight, far outside the bound.  Output buffers are NaN before the call and have NaN elements past
their end, which must stay NaN.
"""
import math

import pytest
import torch

from multimodalpfn_b200 import _lib

pytestmark = pytest.mark.gpu

E = 192
PAD = 7                   # NaN elements past the end of every output buffer
EUNSUPPORTED = -4
U32 = 2.0 ** -24          # fp32 unit roundoff
UBF = 2.0 ** -8           # bf16 unit roundoff (8 significant bits)
POLY = 7.6e-5             # max relative error of the item attention's polynomial 2^x (kernels_attn.cu, poly_exp2_pair)
LOG2E = 1.0 / math.log(2.0)
V_OFFSETS = (0.0, 4.0)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _pad8(n):
    return (n + 7) // 8 * 8


def _pad64(n):
    return (n + 63) // 64 * 64


def _i32(a):
    return torch.tensor(a, dtype=torch.int32, device="cuda")


def _nan(shape, dtype):
    """A NaN buffer of `shape` with PAD NaN elements past its end: (the view, the whole buffer)."""
    n = math.prod(shape)
    buf = torch.full((n + PAD,), float("nan"), dtype=dtype, device="cuda")
    return buf[:n].view(*shape), buf


def _assert_tail_untouched(buf, n):
    assert torch.isnan(buf[n:].float()).all(), "a kernel wrote past the end of its output"


# ---------------------------------------------------------------------------------------------------------------
# attention: reference and bound
# ---------------------------------------------------------------------------------------------------------------
def _attn_ref(q, k, v):
    """float64 softmax(q k^T / sqrt 32) v over the last two axes, and P|V|, and per query row the largest
    sum_d |q_d k_d| / sqrt 32 over its keys (the magnitude the fp32 score and exponent arithmetic round at)."""
    q, k, v = q.double(), k.double(), v.double()
    p = torch.softmax(q @ k.transpose(-1, -2) / 32 ** 0.5, dim=-1)
    sabs = (q.abs() @ k.abs().transpose(-1, -2) / 32 ** 0.5).amax(-1, keepdim=True)
    return p @ v, p @ v.abs(), sabs


def _attn_bound(ref, pv_abs, sabs, n_kv, p_round, out_round, k_score):
    """Per-element bound on |out - ref| for an online-softmax attention.

    * The exponentials p_i = exp(s_i - m) have relative error e_p (p_round: the 2^x used, plus P rounded to bf16 before
      P V where the kernel does that); P V accumulates n_kv fp32 terms (n_kv * 2^-24 relative); the scores and the
      exponent arguments s*c - m*c are fp32 sums of products of size up to sabs, each rounding moves p by its absolute
      error (k_score ulps of sabs).  Numerator terms: at most (e_p + n_kv u + k_score u sabs) * sum_i P_i |v_i|.
    * The normaliser sum_i p_i has the same relative error from the 2^x, the accumulation and the exponent arguments
      (not the bf16 rounding: the row sum adds fp32 p), and the output is rounded once (out_round): * |ref|.
    """
    xerr = k_score * U32 * sabs
    a = p_round + n_kv * U32 + xerr
    b = out_round + POLY + n_kv * U32 + xerr
    return a * pv_abs + b * ref.abs() + 1e-6


def _ratio(out, ref, bound):
    out = out.double()
    assert torch.isfinite(out).all()
    return float(((out - ref).abs() / bound).max())


# bf16 item attention (kernels_attn.cu): P = 2^x by the polynomial (7.6e-5) or MUFU (~2^-22), rounded to bf16 before
# P V (2^-8); the output is rounded to bf16 (2^-8).  Scores: tensor-core fp32 sums of 32 exact bf16 products, then one
# FFMA2 x = s*c - m*c: 64 ulps of sabs covers the accumulation (rounding or truncating) and the scaling.
ITEM_BF16 = dict(p_round=UBF + POLY, out_round=UBF, k_score=64)
# fp32 item attention (kernels_f32.cu, flash FFMA kernel): expf (2 ulp), no rounding of P; fp32 output.
ITEM_F32 = dict(p_round=4 * U32, out_round=U32, k_score=64)
# bf16 feature attention (feat_attn_core.cuh): ex2.approx (2^-22), P rounded to bf16, bf16 output; the CUDA-core
# fallback (T > 192) rounds less (expf, fp32 P) and is held to the same bound.
FEAT_BF16 = dict(p_round=UBF + 2.0 ** -21, out_round=UBF, k_score=64)

RATIOS = {}               # largest err / bound per test (printed with -s)


def _note(name, r):
    RATIOS[name] = max(RATIOS.get(name, 0.0), r)
    print(f"max err/bound {name}: {RATIOS[name]:.3f}")


# ---------------------------------------------------------------------------------------------------------------
# item attention: inputs
# ---------------------------------------------------------------------------------------------------------------
KV_EDGES = [1, 47, 48, 49, 63, 64, 65, 95, 96, 97, 143, 144, 145, 2000]
Q_EDGES = [1, 127, 128, 129, 300]
PATTERNS = ["random1", "random16", "up7.75", "up8.25", "down"]


def _ramp_levels(n_kv, pattern, g):
    """Score of every key in log2 units.  Tile t of 48 keys holds one peak at t * step (ascending) or -t * step
    (descending); its other keys sit 20-21 log2 units lower, so a tile's row sum against the previous reference is
    2^(its rise) to within 2^-14.  Ascending by 8.25: the sum exceeds 2^8 on every tile (the reference moves every
    time); by 7.75: it stays below on odd tiles and exceeds it on even ones (a reference that did not move two tiles
    in a row)."""
    step = 8.25 if pattern in ("up8.25", "down") else 7.75
    sign = -1.0 if pattern == "down" else 1.0
    j = torch.arange(n_kv, dtype=torch.float64)
    t = torch.div(j, 48, rounding_mode="floor")
    peak = (t * 17 + 5) % 48                       # the peak's place inside its tile moves from tile to tile
    peak = torch.minimum(peak, (n_kv - 1 - t * 48))  # a partial last tile still has its peak
    lev = sign * t * step - 20.0 - torch.rand(n_kv, generator=g, dtype=torch.float64)
    is_peak = (j - t * 48) == peak
    lev[is_peak] = sign * t[is_peak] * step
    return lev


def _score_rows(n, n_kv, pattern, g, dims=32):
    """q [n][32], k [n_kv][32] (float64, already representable in bf16) whose scores q k^T / sqrt 32 follow `pattern`:
    q = (Q0, Q1, small noise), k_j = (a_j, b_j, small noise); a_j carries the level, b_j its bf16 rounding error, so
    the levels hold to ~2^-16 relative after the rounding of the operands to bf16."""
    if pattern.startswith("random"):
        scale = float(pattern[len("random"):])
        q = (torch.randn(n, dims, generator=g, dtype=torch.float64) * scale)
        k = (torch.randn(n_kv, dims, generator=g, dtype=torch.float64) * scale)
        return q.to(torch.bfloat16).double(), k.to(torch.bfloat16).double()
    s = _ramp_levels(n_kv, pattern, g) / LOG2E * 32 ** 0.5          # wanted q.k
    q0, q1 = 8.0, 1.0 / 32
    a = (s / q0).to(torch.bfloat16).double()
    b = ((s - q0 * a) / q1).to(torch.bfloat16).double()
    q = (torch.randn(n, dims, generator=g, dtype=torch.float64) * 0.01).to(torch.bfloat16).double()
    k = (torch.randn(n_kv, dims, generator=g, dtype=torch.float64) * 0.01).to(torch.bfloat16).double()
    q[:, 0], q[:, 1] = q0, q1
    k[:, 0], k[:, 1] = a, b
    return q, k


def _item_inputs(n_planes_q, n_planes_kv, n_q, n_kv, pattern, v_off, g):
    """Per q plane n_q query rows, per kv plane n_kv keys and values (float64, bf16-representable)."""
    q = torch.empty(n_planes_q, n_q, 32, dtype=torch.float64)
    k = torch.empty(n_planes_kv, n_kv, 32, dtype=torch.float64)
    per = n_planes_q // n_planes_kv
    for pk in range(n_planes_kv):
        qq, kk = _score_rows(per * n_q, n_kv, pattern, g)
        q[pk * per:(pk + 1) * per] = qq.view(per, n_q, 32)
        k[pk] = kk
    v = (v_off + torch.randn(n_planes_kv, n_kv, 32, generator=g, dtype=torch.float64)).to(torch.bfloat16).double()
    return q, k, v


def _bf16_planes(q, k, v, Sq_pad, Skv_pad, kv_fill):
    """The kernel's plane layouts: q [P][Sq_pad][32] (pad rows finite), k [Pkv][Skv_pad][32], vt [Pkv][32][Skv_pad]
    (rows past n_kv = kv_fill)."""
    P, n_q, _ = q.shape
    Pk, n_kv, _ = k.shape
    qb = torch.randn(P, Sq_pad, 32).to(torch.bfloat16)
    qb[:, :n_q] = q.to(torch.bfloat16)
    kb = torch.full((Pk, Skv_pad, 32), kv_fill, dtype=torch.bfloat16)
    kb[:, :n_kv] = k.to(torch.bfloat16)
    vt = torch.full((Pk, 32, Skv_pad), kv_fill, dtype=torch.bfloat16)
    vt[:, :, :n_kv] = v.transpose(1, 2).to(torch.bfloat16)
    return qb.cuda(), kb.cuda(), vt.cuda()


def _check_item(out_bth, q, k, v, shared, n_q, n_kv, T, consts, name):
    """out [n_q][T][192] of one entry (b) against the reference of its planes q [T*6][n_q][32], k/v [T or T*6][n_kv]."""
    kk = k.repeat_interleave(6, 0) if shared else k
    vv = v.repeat_interleave(6, 0) if shared else v
    ref, pva, sabs = _attn_ref(q.cuda(), kk.cuda(), vv.cuda())
    got = out_bth.reshape(n_q, T, 6, 32).permute(1, 2, 0, 3).reshape(T * 6, n_q, 32)
    r = _ratio(got, ref, _attn_bound(ref, pva, sabs, n_kv, **consts))
    _note(name, r)
    return r


@pytest.mark.parametrize("shared", [0, 1])
@pytest.mark.parametrize("n_kv", KV_EDGES)
def test_item_attention_bf16_vs_float64(n_kv, shared):
    """Every n_q of Q_EDGES (Sq_pad = n_q rounded up to 8: with shared K/V the six heads are stacked on the tile rows
    for n_q 1, 129 and 300, not for 127 / 128), every score pattern, V with and without offset.  Keys past n_kv are
    NaN: the tensor maps end at n_kv and never fetch them."""
    lib = _lib.load()
    B, T = 1, 2
    planes, kv_planes = B * T * 6, (B * T if shared else B * T * 6)
    g = torch.Generator().manual_seed(1000 * n_kv + shared)
    for i, pattern in enumerate(PATTERNS):
        for v_off in V_OFFSETS:
            # 2000 keys: one query count per (pattern, offset), the five in turn
            q_counts = [Q_EDGES[(2 * i + int(v_off > 0)) % len(Q_EDGES)]] if n_kv == 2000 else Q_EDGES
            for n_q in q_counts:
                q, k, v = _item_inputs(planes, kv_planes, n_q, n_kv, pattern, v_off, g)
                Sq_pad, Skv_pad = _pad8(n_q), _pad64(n_kv)
                qb, kb, vt = _bf16_planes(q, k, v, Sq_pad, Skv_pad, float("nan"))
                out, buf = _nan((B, n_q, T, E), torch.bfloat16)
                _lib.check(lib.mmpfn_item_attention_bf16(qb.data_ptr(), kb.data_ptr(), vt.data_ptr(), B, T, n_q,
                                                         Sq_pad, n_kv, Skv_pad, shared, buf.data_ptr(), _stream()),
                           "item_attention_bf16")
                torch.cuda.synchronize()
                _assert_tail_untouched(buf, out.numel())
                r = _check_item(out[0], q, k, v, shared, n_q, n_kv, T, ITEM_BF16, "item_attention_bf16")
                assert r <= 1.0, (pattern, v_off, n_q, r)


@pytest.mark.parametrize("shared", [0, 1])
def test_item_attention_bf16_ragged_vs_float64(shared):
    """Per-entry key counts at every tile edge in one launch (capacity n_kv = 2000), query counts cycling through
    Q_EDGES (capacity 300): every entry against its own float64 reference, its pad output rows exactly zero.  Key rows
    between an entry's count and the capacity are zero (the pad-row contract), rows past the capacity NaN."""
    lib = _lib.load()
    kv_len = KV_EDGES
    B, T = len(kv_len), 1
    q_len = [Q_EDGES[b % len(Q_EDGES)] for b in range(B)]
    n_q, n_kv = max(q_len), max(kv_len)
    Sq_pad, Skv_pad = _pad8(n_q), _pad64(n_kv)
    per_q, per_kv = T * 6, (T if shared else T * 6)
    for pattern in ("random1", "up8.25", "up7.75"):
        for v_off in V_OFFSETS:
            g = torch.Generator().manual_seed(77 + shared)
            ents = [_item_inputs(per_q, per_kv, q_len[b], kv_len[b], pattern, v_off, g) for b in range(B)]
            qb = torch.zeros(B * per_q, Sq_pad, 32, dtype=torch.bfloat16)
            kb = torch.full((B * per_kv, Skv_pad, 32), float("nan"), dtype=torch.bfloat16)
            vt = torch.full((B * per_kv, 32, Skv_pad), float("nan"), dtype=torch.bfloat16)
            kb[:, :n_kv] = 0
            vt[:, :, :n_kv] = 0
            for b, (q, k, v) in enumerate(ents):
                qb[b * per_q:(b + 1) * per_q, :q_len[b]] = q.to(torch.bfloat16)
                kb[b * per_kv:(b + 1) * per_kv, :kv_len[b]] = k.to(torch.bfloat16)
                vt[b * per_kv:(b + 1) * per_kv, :, :kv_len[b]] = v.transpose(1, 2).to(torch.bfloat16)
            qb, kb, vt = qb.cuda(), kb.cuda(), vt.cuda()
            out, buf = _nan((B, n_q, T, E), torch.bfloat16)
            ql, kl = _i32(q_len), _i32(kv_len)
            _lib.check(lib.mmpfn_item_attention_bf16_ragged(qb.data_ptr(), kb.data_ptr(), vt.data_ptr(), B, T, n_q,
                                                            Sq_pad, n_kv, Skv_pad, shared, ql.data_ptr(), kl.data_ptr(),
                                                            buf.data_ptr(), _stream()), "item_attention_bf16_ragged")
            torch.cuda.synchronize()
            _assert_tail_untouched(buf, out.numel())
            for b, (q, k, v) in enumerate(ents):
                assert (out[b, q_len[b]:] == 0).all(), b
                r = _check_item(out[b, :q_len[b]], q, k, v, shared, q_len[b], kv_len[b], T, ITEM_BF16,
                                "item_attention_bf16_ragged")
                assert r <= 1.0, (pattern, v_off, b, q_len[b], kv_len[b], r)


@pytest.mark.parametrize("shared", [0, 1])
@pytest.mark.parametrize("n_kv", [1, 47, 63, 64, 65, 127, 128, 129, 2000])
def test_item_attention_f32_vs_float64(n_kv, shared):
    """The fp32 flash kernel (64-key tiles) at its tile edges, random scores at scales 1 and 16 and the ramps; rows of
    q, k, v past the counts are NaN (never read)."""
    lib = _lib.load()
    B, T = 1, 2
    g = torch.Generator().manual_seed(3000 + n_kv * 2 + shared)
    for i, pattern in enumerate(PATTERNS):
        for v_off in V_OFFSETS:
            n_q = Q_EDGES[(2 * i + int(v_off > 0)) % len(Q_EDGES)]
            q, k, v = _item_inputs(T * 6, T if shared else T * 6, n_q, n_kv, pattern, v_off, g)
            qd = q.view(T, 6, n_q, 32).permute(2, 0, 1, 3).reshape(1, n_q, T, E).float().cuda()
            if shared:                                                     # [B][T][n_kv][32]
                kd, vd = k.view(1, T, n_kv, 32).float().cuda(), v.view(1, T, n_kv, 32).float().cuda()
            else:                                                          # [B][n_kv][T][192]
                kd = k.view(T, 6, n_kv, 32).permute(2, 0, 1, 3).reshape(1, n_kv, T, E).float().cuda()
                vd = v.view(T, 6, n_kv, 32).permute(2, 0, 1, 3).reshape(1, n_kv, T, E).float().cuda()
            out, buf = _nan((B, n_q, T, E), torch.float32)
            _lib.check(lib.mmpfn_item_attention_f32(qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), B, T, n_q, n_kv,
                                                    shared, None, None, buf.data_ptr(), _stream()), "item_attention_f32")
            torch.cuda.synchronize()
            _assert_tail_untouched(buf, out.numel())
            r = _check_item(out[0], q, k, v, shared, n_q, n_kv, T, ITEM_F32, "item_attention_f32")
            assert r <= 1.0, (pattern, v_off, n_q, r)


# ---------------------------------------------------------------------------------------------------------------
# feature attention
# ---------------------------------------------------------------------------------------------------------------
FEAT_T = [2, 15, 16, 17, 31, 32, 33, 64, 65, 80, 81, 96, 97, 144, 145, 192, 193, 300, 497]


def _feat_case(lib, n_rows, T, scale, v_off, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n_rows * T, 3, 6, 32, device="cuda", generator=g)
    x[:, :2] *= scale ** 0.5                                          # q k^T / sqrt 32 has standard deviation `scale`
    x[:, 2] += v_off
    qkv = x.reshape(n_rows * T, 3 * E).to(torch.bfloat16)
    att, buf = _nan((n_rows * T, E), torch.bfloat16)
    _lib.check(lib.mmpfn_feature_attention_bf16(qkv.data_ptr(), buf.data_ptr(), n_rows, T, _stream()), "feat_attn")
    torch.cuda.synchronize()
    _assert_tail_untouched(buf, att.numel())
    xd = qkv.view(n_rows, T, 3, 6, 32)
    worst = 0.0
    for r0 in range(0, n_rows, max(1, 2 ** 27 // (36 * T * T))):      # float64 scores in chunks of ~1 GB
        r1 = min(n_rows, r0 + max(1, 2 ** 27 // (36 * T * T)))
        q, k, v = (xd[r0:r1, :, j].permute(0, 2, 1, 3) for j in range(3))   # [rows, h, T, d]
        ref, pva, sabs = _attn_ref(q, k, v)
        got = att.view(n_rows, T, 6, 32)[r0:r1].permute(0, 2, 1, 3)
        worst = max(worst, _ratio(got, ref, _attn_bound(ref, pva, sabs, T, **FEAT_BF16)))
    _note("feature_attention_bf16", worst)
    return worst


@pytest.mark.parametrize("T", FEAT_T)
def test_feature_attention_bf16_vs_float64(T):
    """Every register-tile size (KT 2/4/6/9/12: T 32/64/96/144/192 and one past each), the one-/two-buffer switch at
    80/96 padded tokens, and the CUDA-core fallback (193-497 tokens); scores at scales 1 and 8, V with and without
    offset."""
    lib = _lib.load()
    n_rows = 5 if T <= 192 else 2
    for scale in (1.0, 8.0):
        for v_off in V_OFFSETS:
            r = _feat_case(lib, n_rows, T, scale, v_off, seed=T * 10 + int(scale) + int(v_off))
            assert r <= 1.0, (scale, v_off, r)


@pytest.mark.parametrize("n_rows,T", [(30000, 20), (4000, 90)])
def test_feature_attention_bf16_many_rows(n_rows, T):
    """Enough rows that every CTA walks several of them (the double-buffered row loop)."""
    lib = _lib.load()
    for scale, v_off in ((1.0, 4.0), (8.0, 0.0)):
        r = _feat_case(lib, n_rows, T, scale, v_off, seed=n_rows + T)
        assert r <= 1.0, (scale, v_off, r)


def test_feature_attention_bf16_rejects_498_tokens():
    """The fallback keeps a row's q, k, v and scores in shared memory: 200 KB ends at 497 tokens."""
    lib = _lib.load()
    qkv = torch.zeros(498, 3 * E, dtype=torch.bfloat16, device="cuda")
    att = torch.zeros(498, E, dtype=torch.bfloat16, device="cuda")
    assert lib.mmpfn_feature_attention_bf16(qkv.data_ptr(), att.data_ptr(), 1, 498, _stream()) == EUNSUPPORTED


# ---------------------------------------------------------------------------------------------------------------
# LayerNorm epilogues
# ---------------------------------------------------------------------------------------------------------------
LN_MEANS = [0.0, 1.0, -1.0, 16.0, -16.0, 256.0, -256.0, 4096.0, -4096.0]
LN_STDS = [1.0, 1e-2, 1e-3]
LN_CELLS = [(m, s) for m in LN_MEANS for s in LN_STDS] + [None]       # None: a row of exact zeros
LN_M = 62101              # a partial last tile of 128 rows, and persistent CTAs that wrap around the SMs
# fp32 rounding of a = state + acc moves a by up to 2^-24 |mean|, and the row mean the kernel subtracts carries a few
# more such roundings (a shift near the mean plus a sum of 192 shifted values; the fp32 layernorm_kernel: a plain sum):
# 32 ulps of |mean| bound them, and the error of (a - mean) is divided by the row's std.
LN_K = 32


def _ln_rows(M, width, seed):
    """fp32 rows mean + std * randn cycling through LN_CELLS, the cell's std per row (0 for zero rows)."""
    g = torch.Generator().manual_seed(seed)
    mean = torch.tensor([c[0] if c else 0.0 for c in LN_CELLS], dtype=torch.float64)
    std = torch.tensor([c[1] if c else 0.0 for c in LN_CELLS], dtype=torch.float64)
    idx = torch.arange(M) % len(LN_CELLS)
    x = mean[idx, None] + std[idx, None] * torch.randn(M, width, generator=g, dtype=torch.float64)
    return x.float(), std[idx], idx == len(LN_CELLS) - 1


def _ln_check(y32, ybf, pre, zero, base32, basebf):
    """y = LN(pre) (no affine, eps 1e-5) per row against float64, with a per-row term for the rounding of pre."""
    ref = torch.nn.functional.layer_norm(pre, (pre.shape[1],), None, None, 1e-5)
    mu = pre.mean(1, keepdim=True)
    sd = (pre.var(1, unbiased=False, keepdim=True) + 1e-5).sqrt()
    extra = LN_K * U32 * mu.abs() / sd
    e32 = (y32.double() - ref).abs()
    r32 = float((e32 / (base32 + extra)).max())
    rbf = None
    if ybf is not None:
        rbf = float(((ybf.double() - ref).abs() / (basebf + extra)).max())
        assert (ybf[zero] == 0).all()
    assert torch.isfinite(y32).all()
    assert (y32[zero] == 0).all(), "a zero row must normalise to exact zeros (pad-row contract)"
    worst = int((e32 / (base32 + extra)).amax(1).argmax())
    return r32, rbf, (float(mu[worst]), float(sd[worst]), float(e32[worst].max()))


def test_linear_ln_bf16_row_statistics():
    """state <- LN(state + A W^T) on rows whose mean is up to 4096 x their std: the epilogue's variance must be taken
    about the mean (a one-pass sq/n - mean^2 loses it with the square of mean/std).  A rows are scaled by the row's
    std so the sum keeps the cell's mean/std; zero rows have zero A rows."""
    lib = _lib.load()
    x, std, zero = _ln_rows(LN_M, E, seed=1)
    g = torch.Generator().manual_seed(2)
    a = (torch.randn(LN_M, E, generator=g, dtype=torch.float64) * std[:, None]).to(torch.bfloat16)
    w = (torch.randn(E, E, generator=g) / E ** 0.5).to(torch.bfloat16)
    st, ad, wd = x.cuda(), a.cuda(), w.cuda()
    stb, buf = _nan((LN_M, E), torch.bfloat16)
    _lib.check(lib.mmpfn_linear_ln_bf16(ad.data_ptr(), wd.data_ptr(), LN_M, st.data_ptr(), buf.data_ptr(), _stream()),
               "linear_ln")
    torch.cuda.synchronize()
    _assert_tail_untouched(buf, stb.numel())
    pre = x.double().cuda() + a.double().cuda() @ w.double().cuda().T
    # fp32: exact bf16 products summed in fp32 (2e-4 of O(1) outputs, as test_out_projection_layernorm_tcgen05);
    # bf16 shadow: one bf16 rounding of O(4) values
    r32, rbf, worst = _ln_check(st, stb, pre, zero.cuda(), 2e-4, 0.03)
    _note("linear_ln_bf16 fp32", r32)
    _note("linear_ln_bf16 bf16", rbf)
    assert r32 <= 1.0 and rbf <= 1.0, (r32, rbf, worst)


def test_mlp_bf16_row_statistics():
    """state <- LN(state + W2 gelu(W1 state_bf16)) on the same rows.  state_bf16 is independent of state_f32 (the API
    takes both) and scaled by 2^-8 x the row's std: the sublayer adds ~1e-3 of the row's spread, so the kernel's
    tanh-form GELU and bf16 hidden activation (~1e-2 of the sublayer output) stay far below the fp32 base and the
    test sees the epilogue alone."""
    lib = _lib.load()
    x, std, zero = _ln_rows(LN_M, E, seed=3)
    g = torch.Generator().manual_seed(4)
    xb = (torch.randn(LN_M, E, generator=g, dtype=torch.float64) * std[:, None] / 256).to(torch.bfloat16)
    w1 = (torch.randn(768, E, generator=g) / E ** 0.5).to(torch.bfloat16)
    w2 = (torch.randn(E, 768, generator=g) / 768 ** 0.5).to(torch.bfloat16)
    st, stb, w1d, w2d = x.cuda(), xb.cuda(), w1.cuda(), w2.cuda()    # held: the kernel runs after the call returns
    _lib.check(lib.mmpfn_mlp_bf16(st.data_ptr(), stb.data_ptr(), w1d.data_ptr(), w2d.data_ptr(), LN_M, _stream()), "mlp")
    torch.cuda.synchronize()
    h = torch.nn.functional.gelu(xb.double().cuda() @ w1.double().cuda().T)
    pre = x.double().cuda() + h @ w2.double().cuda().T
    r32, rbf, worst = _ln_check(st, stb, pre, zero.cuda(), 2e-4, 0.03)
    _note("mlp_bf16 fp32", r32)
    _note("mlp_bf16 bf16", rbf)
    assert r32 <= 1.0 and rbf <= 1.0, (r32, rbf, worst)


@pytest.mark.parametrize("width", [192, 384, 768])
def test_layernorm_row_statistics(width):
    """Control: the fp32 layernorm_kernel centres before squaring and meets the same per-row bound (its input is
    the fp32 row itself: the ratio term covers the summation of the mean)."""
    lib = _lib.load()
    x, _, zero = _ln_rows(4097, width, seed=width)
    xd = x.cuda()
    y, buf = _nan((4097, width), torch.float32)
    yb, bufb = _nan((4097, width), torch.bfloat16)
    _lib.check(lib.mmpfn_layernorm(xd.data_ptr(), None, None, None, 4097, width, buf.data_ptr(), bufb.data_ptr(),
                                   _stream()), "layernorm")
    torch.cuda.synchronize()
    _assert_tail_untouched(buf, y.numel())
    _assert_tail_untouched(bufb, yb.numel())
    # fp32 base as test_layernorm (5e-6: fp32 vs fp64 on O(4) outputs); bf16: one rounding of O(4) values
    r32, rbf, worst = _ln_check(y, yb, xd.double(), zero.cuda(), 5e-6, 0.03)
    _note(f"layernorm{width} fp32", r32)
    assert r32 <= 1.0 and rbf <= 1.0, (r32, rbf, worst)
