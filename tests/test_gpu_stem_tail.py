"""The kernels at the two ends of the forward, each against a float64 restatement of the same operation:

* ``mmpfn_stem_tab_fit`` (tab_fit_kernel) against ``oracle.forward_ref.stem_tab_fit``;
* ``mmpfn_stem_tokens`` (stem_tokens_kernel) against ``stem_tab_apply`` + positional embedding + image tokens +
  ``stem_y_apply`` on the kernel's own statistics;
* ``mmpfn_stem_image`` (MGM, tcgen05 GLU GEMM, cap_attn / cap_combine, MoE gate) against ``stem_image``;
* ``mmpfn_decode`` (two sgemm launches reading the y token at stride T*192) against ``decode``;
* ``mmpfn_proba_tail`` (proba_tail_kernel, through ``engine.proba_device``) against ``oracle.proba_tail`` restated
  in float64.

A whole-model check is weak for these kernels: 12 post-LN layers renormalise every token, so a stem error of a few
percent can pass it.  Every output buffer here is NaN before the call and has a few NaN elements past its end:
what the kernel writes must be finite wherever the reference is, and the elements past the end stay NaN.
"""
import math

import numpy as np
import pytest
import torch

from multimodalpfn_b200 import _lib
from multimodalpfn_b200.engine import proba_device
from multimodalpfn_b200.model import B200PerFeatureTransformer
from multimodalpfn_b200.synth import Geometry, make_state_dict
from oracle import forward_ref as R

pytestmark = pytest.mark.gpu

E = 192
PAD = 7               # NaN elements past the end of every output buffer
EINVAL, EUNSUPPORTED = -1, -4
U32 = 2.0 ** -24      # fp32 unit roundoff


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _nan_buffer(n, dtype=torch.float32):
    """n elements + PAD past the end, all NaN."""
    return torch.full((n + PAD,), float("nan"), dtype=dtype, device="cuda")


def _assert_tail_untouched(buf, n):
    assert torch.isnan(buf[n:].float()).all(), "a kernel wrote past the end of its output"


def _sd64(sd):
    return {k: torch.as_tensor(v, dtype=torch.float64) for k, v in sd.items()}


_MODELS = {}


def _model(precision="fp32", **geom_kw):
    """One model per geometry (nlayers 1: only the stem / decoder weights matter here)."""
    key = (precision, tuple(sorted(geom_kw.items())))
    if key not in _MODELS:
        regression = geom_kw.pop("regression", False)
        geom = Geometry(nlayers=1, **geom_kw)
        sd = make_state_dict(geom, seed=7, regression=regression)
        if regression:
            sd = {k: v for k, v in sd.items() if not k.startswith("criterion.")}
        _MODELS[key] = (B200PerFeatureTransformer(sd, geom, precision=precision), sd, geom)
    return _MODELS[key]


def _assert_close(got, ref, tol, what):
    """|got - ref| <= tol elementwise where ref is finite; got NaN exactly where ref is NaN."""
    got, ref = got.double().cpu(), ref.double().cpu()
    tol = torch.as_tensor(tol, dtype=torch.float64).expand_as(ref)
    nan_ref = torch.isnan(ref)
    assert torch.equal(torch.isnan(got), nan_ref), f"{what}: NaN pattern differs ({int((torch.isnan(got) != nan_ref).sum())} elements)"
    inf_ref = torch.isinf(ref)
    assert torch.equal(got[inf_ref], ref[inf_ref]), f"{what}: infinities differ"
    fin = ~(nan_ref | inf_ref)
    assert torch.isfinite(got[fin]).all(), f"{what}: not finite where the reference is"
    err = (got[fin] - ref[fin]).abs()
    bad = err > tol[fin]
    assert not bad.any(), f"{what}: {int(bad.sum())} elements off, worst {float((err - tol[fin]).max()):.3e} over tolerance"


# =============================================================================================================
# tabular statistics: mmpfn_stem_tab_fit
# =============================================================================================================
# column kinds; c is a dyadic constant, so a sum of its copies is exact in fp32 and fp64 alike and the constant
# tests do not depend on the accumulation order
C = 2.5


def _column(kind, S, n_train, rng):
    x = (rng.standard_normal(S) * 3.0 + 1.0).astype(np.float32)
    if kind == "normal":
        pass
    elif kind == "int":                                   # few levels: ties
        x = rng.integers(0, 4, S).astype(np.float32)
    elif kind == "outliers":                              # far outside 12 sigma: masked in the first pass, soft-clipped
        x[rng.choice(n_train, size=min(2, n_train), replace=False)] = np.float32(1e5)
        if S > n_train:
            x[n_train] = np.float32(-1e5)
    elif kind == "nan_some":                              # row 0 observed: a finite fill even at n_train == 1
        x[1:][rng.random(S - 1) < 0.15] = np.nan
    elif kind == "const":                                 # constant over all rows: dropped
        x[:] = C
    elif kind == "const_train":                           # constant over the train rows, varies in the test rows
        x[:n_train] = C
    elif kind == "const_nan":                             # its only variation is NaN cells: kept, not "used"
        x[:] = C
        x[rng.random(S) < 0.3] = np.nan
        x[0] = np.nan
    elif kind == "all_nan":                               # kept (NaN != NaN); NaN fill, NaN tokens
        x[:] = np.nan
    elif kind == "nan_train":                             # NaN in every train row, observed in the test rows
        x[:n_train] = np.nan
    elif kind == "inf_test":                              # +-inf only in test rows: indicators 2 / 4, filled
        if S > n_train + 1:
            x[n_train] = np.inf
            x[n_train + 1] = -np.inf
    elif kind == "inf_train":                             # +inf in a train row: the fill keeps inf (torch.nanmean)
        x[0] = np.inf
    else:
        raise KeyError(kind)
    return x


def _table(kinds, B, S, n_train, seed):
    rng = np.random.default_rng(seed)
    return np.stack([np.stack([_column(k, S, n_train, rng) for k in kinds], axis=1) for _ in range(B)])


def _tab_fit_raw(model, X, n_train, n_sigma):
    """mmpfn_stem_tab_fit into a NaN buffer -> (stats [B, n], buffer)."""
    B, S, F = X.shape
    G = model._n_groups(F)
    n = model.lib.mmpfn_tab_stats_elems(model._g, G)
    buf = _nan_buffer(B * n)
    rc = model.lib.mmpfn_stem_tab_fit(model._g, X.data_ptr(), B, S, F, n_train, float(n_sigma), buf.data_ptr(), _stream())
    _lib.check(rc, "mmpfn_stem_tab_fit")
    torch.cuda.synchronize()
    _assert_tail_untouched(buf, B * n)
    return buf[:B * n].view(B, n).cpu(), G


def _split_stats(st, G, fpg):
    """TabStatsLayout (csrc/common.cuh): src | fill | lo | hi | mean | std per compacted slot g*fpg + j, scale per g."""
    Fp = G * fpg
    f = [st[i * Fp:(i + 1) * Fp].view(G, fpg) for i in range(6)]
    return dict(src=f[0], fill=f[1], lo=f[2], hi=f[3], mean=f[4], std=f[5], scale=st[6 * Fp:6 * Fp + G])


TAB_CASES = [
    # fpg, F, S, n_train, n_sigma, kinds (column c of each group cycles through them)
    (1, 7, 300, 200, 12.0, ["normal", "int", "outliers", "nan_some", "const", "const_train", "const_nan"]),
    (2, 7, 300, 200, 12.0, ["normal", "const", "const_nan", "nan_some", "outliers", "const_train", "int"]),
    (2, 8, 300, 200, math.inf, ["normal", "const", "const_nan", "const_train", "outliers", "int", "nan_some", "normal"]),
    (3, 9, 129, 100, 12.0, ["const", "const_nan", "normal", "all_nan", "nan_train", "inf_test", "const_train", "const",
                            "int"]),
    (3, 10, 129, 100, math.inf, ["const", "const_nan", "normal", "all_nan", "nan_train", "inf_test", "const_train",
                                 "const", "int", "inf_train"]),
    (4, 13, 257, 256, 12.0, ["inf_train", "normal", "outliers", "const_nan", "const", "const", "nan_some", "int",
                             "const_train", "normal", "all_nan", "normal", "nan_train"]),
    (4, 12, 257, 256, math.inf, ["const", "normal", "const", "const", "const_nan", "const", "const_train", "const",
                                 "outliers", "nan_some", "int", "normal"]),
    # n_train == 1: std forced to 1; with the outlier step on, its statistics are NaN
    (2, 5, 40, 1, 12.0, ["normal", "const_train", "int", "nan_some", "const"]),
    (2, 5, 40, 1, math.inf, ["normal", "const_train", "int", "nan_some", "const"]),
    (1, 3, 1, 1, 12.0, ["normal", "int", "nan_some"]),
    # long columns: the fp64 block reductions over tens of thousands of rows
    (2, 5, 50_000, 40_000, 12.0, ["outliers", "nan_some", "normal", "const_train", "const_nan"]),
    (3, 4, 70_001, 69_000, math.inf, ["normal", "outliers", "nan_some", "int"]),
]


def _ref_fit(X, n_train, fpg, n_sigma):
    """The oracle on one estimator's table: float64 for the values, fp32 for the discrete outcomes (which columns
    are kept, how many slots are used): fp32 is the arithmetic of the reference."""
    x64 = R.group_features(torch.from_numpy(X).double(), fpg)
    x32 = R.group_features(torch.from_numpy(X), fpg)
    return R.stem_tab_fit(x64, n_train, n_sigma=n_sigma), R.stem_tab_fit(x32, n_train, n_sigma=n_sigma)


@pytest.mark.parametrize("fpg,F,S,n_train,n_sigma,kinds", TAB_CASES)
def test_stem_tab_fit_vs_oracle(fpg, F, S, n_train, n_sigma, kinds):
    """Every field of the statistics block against the float64 oracle.  At n_sigma = inf the reference has no
    outlier step (bounds -inf / +inf, the kernel's branch); the oracle follows it there."""
    kinds = (kinds * F)[:F]
    B = 2
    model, _, _ = _model(features_per_group=fpg, mixer_type="none")
    X = _table(kinds, B, S, n_train, seed=F * 1000 + S + fpg)
    stats, G = _tab_fit_raw(model, torch.from_numpy(X).cuda(), n_train, n_sigma)
    for b in range(B):
        got = _split_stats(stats[b], G, fpg)
        r64, r32 = _ref_fit(X[b], n_train, fpg, n_sigma)
        # discrete outcomes, exactly: the source column of every compacted slot (kept columns first, in order) ...
        src = torch.full((G, fpg), -1.0)
        for g in range(G):
            kept = [g * fpg + j for j in range(fpg) if bool(r32["sel"][g, j])]
            src[g, :len(kept)] = torch.tensor(kept, dtype=torch.float32)
        assert torch.equal(got["src"], src), (got["src"], src)
        assert torch.equal(r64["sel"], r32["sel"])
        # ... and the used-slot count behind scale = sqrt(fpg / used)
        used = torch.round(fpg / got["scale"].double() ** 2)
        assert torch.equal(used, r32["used"].double()), (used, r32["used"])
        # sqrtf of the fp32 quotient of two small integers: two fp32 roundings
        ref_scale = torch.sqrt(fpg / r32["used"].double())
        _assert_close(got["scale"], ref_scale, 2 * U32 * ref_scale, "scale")
        # every slot, the empty ones included: an empty slot is the zero column the reference pads the group with, and
        # has that column's statistics (with n_train == 1 and the outlier step on, NaN bounds, and it counts as used)
        # fill: an fp64 sum rounded once to fp32
        _assert_close(got["fill"], r64["fill"], 2 * U32 * r64["fill"].abs(), "fill")
        # lo / hi = mu -+ n_sigma sd: mu and sd are fp64 sums of fp32 terms ((mean_f - x)^2 rounded in fp32 before the
        # fp64 sum), each within a few 2^-24 of its value; scale = the larger bound
        bscale = torch.maximum(r64["lo"].abs(), r64["hi"].abs())
        for k in ("lo", "hi"):
            _assert_close(got[k], r64[k], 16 * U32 * bscale, k)
        # z-norm statistics of the soft-clipped column: the same reductions over values exact in fp32 inside the
        # bounds (the soft clip returns x itself) and within 2 ulps (logf) outside
        _assert_close(got["mean"], r64["mean"], 16 * U32 * (r64["mean"].abs() + r64["std"].abs()), "mean")
        _assert_close(got["std"], r64["std"], 16 * U32 * r64["std"].abs(), "std")


# =============================================================================================================
# token assembly: mmpfn_stem_tokens
# =============================================================================================================
def _stats_dict(st, G, fpg):
    """The kernel's statistics block as the oracle's dict (float64): sel from the source columns, used such that
    sqrt(fpg / used) is the kernel's own scale."""
    s = _split_stats(st, G, fpg)
    sel = torch.zeros(G, fpg, dtype=torch.bool)
    for g in range(G):
        for j in range(fpg):
            c = int(s["src"][g, j])
            if c >= 0:
                sel[g, c - g * fpg] = True
    d = {k: s[k].double() for k in ("fill", "lo", "hi", "mean", "std")}
    d["sel"] = sel
    d["used"] = fpg / s["scale"].double() ** 2
    return d


def _embed_raw(model, X, stats, img_tok, y, y_mean, y_mask, pos, *, B, S, F, x_bstride, y_bstride):
    """model.embed into NaN buffers with PAD elements past their ends -> (state, state_bf16, nan_flag)."""
    G = model._n_groups(F) if X is not None else 0
    H = 0 if img_tok is None else img_tok.shape[-2]
    n = B * S * (G + H + 1) * E
    buf = _nan_buffer(n)
    buf_b = _nan_buffer(n, torch.bfloat16)
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    shape = (B, S, G + H + 1, E)
    model.embed(X, stats, img_tok, y, y_mean, y_mask, pos, B=B, S=S, F=F, x_bstride=x_bstride, y_bstride=y_bstride,
                nan_flag=flag, out=(buf[:n].view(shape), buf_b[:n].view(shape)))
    torch.cuda.synchronize()
    _assert_tail_untouched(buf, n)
    _assert_tail_untouched(buf_b, n)
    return buf[:n].view(shape), buf_b[:n].view(shape), int(flag.item())


def _ref_tokens(sd, X_rows, st_b, img_b, yy, y_mean_b, uniq, pos, fpg, regression):
    """float64 reference of one estimator's tokens [S, T, E] and a bound on the magnitude of each token's terms."""
    sd64 = _sd64(sd)
    pos64 = pos.double().cpu()
    toks, mags = [], []
    if X_rows is not None:
        xg = R.group_features(torch.from_numpy(X_rows).double(), fpg)
        cells = R.stem_tab_apply(xg, st_b, torch.eye(2 * fpg, dtype=torch.float64))      # [S, G, 2 fpg]: (x4 | ind)
        w = sd64["encoder.5.layer.weight"]
        toks.append(cells @ w.T)
        mags.append(cells.abs() @ w.abs().T)
    if img_b is not None:
        toks.append(img_b.double().cpu())
        mags.append(img_b.double().cpu().abs())
    G_H = sum(t.shape[1] for t in toks)
    tok = torch.cat(toks, dim=1) + pos64[None, :G_H]
    mag = torch.cat(mags, dim=1) + pos64[None, :G_H].abs()
    w_y, b_y, reg = R.y_encoder_weights(sd64)
    assert reg == regression
    st_y = dict(mean=torch.tensor(float(y_mean_b), dtype=torch.float64), uniq=uniq)
    ty = R.stem_y_apply(yy, st_y, w_y, b_y, regression)
    vi = R.stem_y_apply(yy, st_y, torch.eye(2, dtype=torch.float64), torch.zeros(2, dtype=torch.float64), regression)
    my = vi.abs() @ w_y.abs().T + b_y.abs()
    return torch.cat([tok, ty[:, None]], dim=1), torch.cat([mag, my[:, None]], dim=1)


def _check_tokens(state, state_b, flag, refs):
    """state against the references; bf16 shadow = the fp32 state rounded to bf16, bit for bit; nan_flag set iff a
    NaN token was written."""
    for b, (ref, mag) in enumerate(refs):
        # at most 2 fpg + 2 fp32 roundings (fmaf chain, + pos) of terms bounded by mag, and the fp32 cell transform
        # (fill, soft clip, (x - mean) / std, * scale: a few 2^-24 of |x4| each) from the same statistics: 2e-6 of mag
        _assert_close(state[b], ref, 2e-6 * mag + 1e-30, f"tokens of entry {b}")
    f32 = state.cpu()
    bf = state_b.cpu()
    nan = torch.isnan(f32)
    assert torch.equal(torch.isnan(bf.float()), nan)
    assert torch.equal(bf[~nan].view(torch.int16), f32[~nan].to(torch.bfloat16).view(torch.int16))
    assert flag == int(nan.any()), (flag, int(nan.sum()))


TOKEN_CASES = [
    # fpg, F, n_train, n_test, n_sigma, kinds, H_img (0: no image tokens; -H: one set per entry)
    (2, 7, 150, 60, 12.0, ["normal", "const_train", "inf_test", "const_nan", "outliers", "int", "nan_some"], 0),
    (1, 5, 90, 37, math.inf, ["normal", "inf_test", "const_train", "const_nan", "const"], 3),
    (3, 8, 64, 65, 12.0, ["const", "nan_some", "normal", "inf_test", "const_train", "int", "outliers", "const_nan"], -2),
    (4, 9, 33, 20, 12.0, ["normal", "const_nan", "inf_test", "const", "const_train", "int", "normal", "outliers",
                          "nan_some"], 0),
    (4, 6, 33, 20, math.inf, ["normal", "int", "inf_test", "const_nan", "const_train", "outliers"], 1),
    # n_train == 1: finite without the outlier step; NaN tokens (and the flag) with it, also in the last group, whose
    # only column is constant (both of its slots empty: zero columns with NaN bounds)
    (2, 5, 1, 9, math.inf, ["normal", "int", "const_train", "nan_some", "const"], 0),
    (2, 5, 1, 9, 12.0, ["normal", "int", "const_train", "nan_some", "const"], 0),
    # a column NaN in every row: NaN tokens in its group only
    (2, 6, 40, 10, 12.0, ["normal", "all_nan", "int", "normal", "nan_train", "normal"], 0),
]


@pytest.mark.parametrize("fpg,F,n_train,n_test,n_sigma,kinds,H_img", TOKEN_CASES)
def test_stem_tokens_vs_oracle(fpg, F, n_train, n_test, n_sigma, kinds, H_img):
    """Train rows and test rows of B = 3 estimators embedded separately out of one [B, S, F] table (x_bstride
    S * F > rows * F), per-entry labels with classes {0, 2, 5} (the presence mask has gaps), NaN test labels replaced
    by the label mean and ranked, image tokens shared or per entry; tokens from the kernel's own statistics."""
    kinds = (kinds * F)[:F]
    B, S = 3, n_train + n_test
    model, sd, _ = _model("bf16", features_per_group=fpg, mixer_type="none")
    X = _table(kinds, B, S, n_train, seed=17 * F + S)
    Xd = torch.from_numpy(X).cuda()
    stats, G = _tab_fit_raw(model, Xd, n_train, n_sigma)
    stats_d = stats.cuda()
    rng = np.random.default_rng(S)
    y_tr = rng.choice([0, 2, 5], size=(B, n_train)).astype(np.float32)
    y_tr[:, :3] = [0, 2, 5][:n_train]
    uniq = [torch.from_numpy(np.unique(y_tr[b])).double() for b in range(B)]
    y_mean, y_mask = model.label_stats(torch.from_numpy(y_tr).cuda())
    assert [int(m) for m in y_mask.cpu()] == [sum(1 << int(c) for c in u) for u in uniq]
    gen = torch.Generator().manual_seed(S)
    H = abs(H_img)
    img = None
    if H_img > 0:
        img = torch.randn(S, H, E, generator=gen)
    elif H_img < 0:
        img = torch.randn(B, S, H, E, generator=gen)
    pos = torch.randn(G + H, E, generator=gen).cuda()
    y_nan = torch.full((1, n_test), float("nan"), device="cuda")
    for part, rows, n, y_dev, y_bstride in (("train", slice(0, n_train), n_train, torch.from_numpy(y_tr).cuda(), n_train),
                                            ("test", slice(n_train, S), n_test, y_nan, 0)):
        img_part = None if img is None else (img[rows] if img.dim() == 3 else img[:, rows]).contiguous()
        state, state_b, flag = _embed_raw(
            model, Xd[:, rows], stats_d, None if img_part is None else img_part.cuda(), y_dev, y_mean, y_mask, pos,
            B=B, S=n, F=F, x_bstride=S * F, y_bstride=y_bstride)
        refs = []
        for b in range(B):
            yy = torch.from_numpy(y_tr[b]).double() if part == "train" else torch.full((n,), math.nan, dtype=torch.float64)
            img_b = None if img_part is None else (img_part if img_part.dim() == 3 else img_part[b])
            refs.append(_ref_tokens(sd, X[b, rows], _stats_dict(stats[b], G, fpg), img_b, yy, y_mean[b].item(),
                                    uniq[b], pos, fpg, False))
        _check_tokens(state, state_b, flag, refs)
        # NaN tokens in exactly the two cases that give them: n_train == 1 with the outlier step on (NaN bounds), and
        # a column NaN in every row (NaN fill)
        nan_expected = (n_train == 1 and not math.isinf(n_sigma)) or "all_nan" in kinds or \
            (part == "train" and "nan_train" in kinds)
        assert flag == int(nan_expected)


def test_stem_tokens_regression_target_and_image_only():
    """Bit 63 of the mask: the target value itself (no rank step) with the label mean for NaN rows, on a regression
    checkpoint; and image tokens without a table."""
    model, sd, _ = _model("bf16", features_per_group=2, mixer_type="none", regression=True)
    B, S, H = 2, 45, 4
    gen = torch.Generator().manual_seed(5)
    y = (torch.randn(B, S, generator=gen) * 4 + 1.5)
    y[:, 30:] = float("nan")
    y_mean = y[:, :30].mean(dim=1).contiguous().cuda()
    y_mask = torch.full((B,), model.REGRESSION_MASK, dtype=torch.int64, device="cuda")
    img = torch.randn(S, H, E, generator=gen)
    pos = torch.randn(H, E, generator=gen).cuda()
    state, state_b, flag = _embed_raw(model, None, None, img.cuda(), y.cuda(), y_mean, y_mask, pos, B=B, S=S, F=0,
                                      x_bstride=0, y_bstride=S)
    refs = [_ref_tokens(sd, None, None, img, y[b].double(), y_mean[b].item(), None, pos, 2, True)
            for b in range(B)]
    _check_tokens(state, state_b, flag, refs)
    assert flag == 0


@pytest.mark.parametrize("fpg,F,ok", [(1, 1024, True), (1, 1025, False), (4, 1021, True), (4, 1025, False)])
def test_stem_tokens_cell_limit(fpg, F, ok):
    """The kernel stages G * fpg <= 1024 cells of a row in shared memory: 1024 is embedded (and checked against the
    reference), 1025 or more is refused with MMPFN_EUNSUPPORTED before any launch."""
    model, sd, _ = _model("bf16", features_per_group=fpg, mixer_type="none")
    B, n_train, S = 1, 5, 7
    X = _table(["normal", "int", "nan_some", "inf_test"] * (F // 4 + 1), B, S, n_train, seed=F)[:, :, :F].copy()
    Xd = torch.from_numpy(X).cuda()
    stats, G = _tab_fit_raw(model, Xd, n_train, 12.0)
    y = torch.tensor([[0.0, 1.0, 1.0, 0.0, 1.0, math.nan, math.nan]], device="cuda")
    y_mean, y_mask = model.label_stats(y[:, :n_train])
    pos = torch.randn(G, E, generator=torch.Generator().manual_seed(F)).cuda()
    if not ok:
        with pytest.raises(RuntimeError, match="EUNSUPPORTED"):
            _embed_raw(model, Xd, stats.cuda(), None, y, y_mean, y_mask, pos, B=B, S=S, F=F, x_bstride=S * F,
                       y_bstride=S)
        return
    state, state_b, flag = _embed_raw(model, Xd, stats.cuda(), None, y, y_mean, y_mask, pos, B=B, S=S, F=F,
                                      x_bstride=S * F, y_bstride=S)
    ref = _ref_tokens(sd, X[0], _stats_dict(stats[0], G, fpg), None, y[0].double().cpu(), y_mean[0].item(),
                      torch.tensor([0.0, 1.0], dtype=torch.float64), pos, fpg, False)
    _check_tokens(state, state_b, flag, [ref])
    assert flag == 0


# =============================================================================================================
# image / text stem: mmpfn_stem_image
# =============================================================================================================
def _stem_image_raw(model, img):
    """mmpfn_stem_image into a NaN buffer, with a NaN-filled workspace -> (rc, out [S, H, E] or None)."""
    S, n_tok, _ = img.shape
    H = model.n_image_tokens(n_tok)
    n = S * H * E
    out = _nan_buffer(n)
    nbytes = model.lib.mmpfn_stem_image_ws_bytes(model._g, S, n_tok)
    ws = torch.full(((nbytes + 3) // 4,), float("nan"), device="cuda")
    rc = model.lib.mmpfn_stem_image(model._g, model._w, img.data_ptr(), S, n_tok, out.data_ptr(), ws.data_ptr(),
                                    nbytes, _stream())
    torch.cuda.synchronize()
    if rc != 0:
        return rc, None
    _assert_tail_untouched(out, n)
    return rc, out[:n].view(S, H, E)


def _cap_smem(mgm, n_tok, cap):
    """bytes of dynamic shared memory cap_attn_kernel takes (launch_cap_attn)."""
    n_kv, hd = mgm * n_tok, E // cap
    return (2 * n_kv * (hd + 1) + 4 * n_kv) * 4


IMAGE_CASES = [
    # mixer, mgm_heads, cap_heads, n_tok, rows
    ("MGM+CAP", 1, 1, 1, 37),
    ("MGM+CAP", 1, 3, 3, 20),
    ("MGM+CAP", 31, 24, 1, 17),
    ("MGM+CAP", 32, 1, 1, 16),          # CAP over 32 sources at head dim 192: 49 920 B, above 48 KB (opt-in path)
    ("MGM+CAP", 8, 1, 8, 9),            # 64 sources: 99 840 B
    ("MGM+CAP", 1, 1, 131, 3),          # 131 sources: 204 360 B, the largest geometry accepted
    ("MGM+CAP", 64, 64, 1, 12),         # head dim 3
    ("MGM+CAP", 64, 24, 1, 13),
    ("MGM+CAP", 32, 3, 3, 5),           # 96 sources at head dim 64: 51 456 B
    ("MGM", 1, 0, 1, 29),
    ("MGM", 31, 0, 3, 7),               # head-major token layout over several tokens
    ("MGM", 32, 0, 8, 4),
    ("MGM", 64, 0, 1, 30),
    ("MoE", 1, 0, 1, 25),
    ("MoE", 31, 0, 3, 11),              # only the first token is read
    ("MoE", 64, 0, 8, 16),
]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("mixer,mgm,cap,n_tok,rows", IMAGE_CASES)
def test_stem_image_vs_oracle(mixer, mgm, cap, n_tok, rows, precision):
    """MGM (transformer.py:33-48), MGM+CAP (:60-88), MoE (:91-128) against the float64 oracle.  In bf16 mode the MGM
    gated projection runs on tcgen05 from 32 MGM heads on (MoE never does)."""
    model, sd, geom = _model(precision, mixer_type=mixer, mgm_heads=mgm, cap_heads=cap or 8)
    if mixer == "MGM+CAP":
        assert (_cap_smem(mgm, n_tok, cap) > 48 * 1024) == ((mgm, cap, n_tok) in ((32, 1, 1), (8, 1, 8), (1, 1, 131), (32, 3, 3)))
    img = torch.randn(rows, n_tok, 768, generator=torch.Generator().manual_seed(mgm * 100 + n_tok + rows))
    rc, out = _stem_image_raw(model, img.cuda())
    assert rc == 0, model.lib.mmpfn_last_error()
    ref = R.stem_image(img.double(), _sd64(sd), geom)
    assert tuple(out.shape) == tuple(ref.shape)
    scale = max(1.0, float(ref.abs().max()))
    if precision == "bf16" and mixer != "MoE" and mgm >= 32:
        # bf16 operands of the 768-deep gated projection (relative 2^-9 each, fp32 accumulation), then LayerNorms and
        # fp32 GEMMs downstream: the 0.03-of-scale budget of test_image_stem_bf16_vs_fp32
        tol = 0.03 * scale
    else:
        # fp32 FFMA GEMMs of depth <= 768 and fp32 LayerNorm / softmax statistics, the LayerNorms (k_norm, out_norm)
        # rescaling their inputs' rounding to O(1): 2e-5 of scale, the fp32 stem budget of the golden state test
        tol = 2e-5 * scale
    _assert_close(out.cpu(), ref, tol, f"{mixer} {mgm}/{cap} x{n_tok} {precision}")


@pytest.mark.parametrize("mgm,n_tok", [(1, 132), (64, 3)])
def test_stem_image_refuses_cap_tile_above_200k(mgm, n_tok):
    """CAP at head dim 192 over more than 131 sources needs more than 200 KB of shared memory: refused."""
    assert _cap_smem(mgm, n_tok, 1) > 200 * 1024
    model, _, _ = _model("fp32", mixer_type="MGM+CAP", mgm_heads=mgm, cap_heads=1)
    img = torch.randn(2, n_tok, 768, device="cuda")
    rc, _ = _stem_image_raw(model, img)
    assert rc == EUNSUPPORTED, rc
    assert b"shared-memory" in model.lib.mmpfn_last_error()


# =============================================================================================================
# decoder: mmpfn_decode
# =============================================================================================================
@pytest.mark.parametrize("n_out,B,S,T", [(10, 1, 1, 1), (10, 3, 77, 2), (64, 2, 129, 17), (64, 1, 300, 40),
                                         (1000, 2, 65, 5), (1000, 1, 257, 1), (5000, 3, 41, 11), (5000, 1, 300, 39)])
def test_decode_vs_oracle(n_out, B, S, T):
    """logits = W2 gelu(W1 state[:, :, T-1] + b1) + b2 (transformer.py:392-396): every token but the y token is
    NaN, so a read of any other token shows; n_out 5000 is the regressor's bucket count (not a multiple of the
    64-column tile)."""
    model, sd, _ = _model("fp32", n_out=n_out, mixer_type="none")
    state = torch.full((B, S, T, E), float("nan"))
    y_tok = torch.randn(B, S, E, generator=torch.Generator().manual_seed(n_out + S + T))
    state[:, :, T - 1] = y_tok
    state = state.cuda()
    hid = _nan_buffer(B * S * model.geom.nhid)
    out = _nan_buffer(B * S * n_out)
    _lib.check(model.lib.mmpfn_decode(model._g, model._w, state.data_ptr(), B, S, T, hid.data_ptr(), out.data_ptr(),
                                      _stream()), "mmpfn_decode")
    torch.cuda.synchronize()
    _assert_tail_untouched(out, B * S * n_out)
    got = out[:B * S * n_out].view(B, S, n_out).cpu()
    assert torch.isfinite(got).all()
    ref = R.decode(y_tok.double(), _sd64(sd))
    # fp32 accumulation over K = 192 (|W1| <= 192^-0.5, O(1) state) then K = 768 (|W2| <= 768^-0.5, O(1) hidden):
    # the 2e-5 of test_linear_f32 for one such product
    _assert_close(got, ref, 2e-5, f"decode n_out {n_out}")


# =============================================================================================================
# probability tail: mmpfn_proba_tail through engine.proba_device
# =============================================================================================================
def _proba_ref(logits, perms, n_classes, temperature, avg_before, class_counts):
    """oracle.proba_tail (classifier.py:544-576) in float64, line by line, including the quirk that the
    [:n_classes] slice happens only when the temperature is not 1.  The temperature is the fp32 value the C ABI
    takes (and the one an fp32 tensor is divided by)."""
    outs = []
    t32 = float(np.float32(temperature))
    for lg, perm in zip(logits.double(), perms):
        if temperature != 1:
            lg = lg[:, :n_classes] / t32
        if perm is not None:
            lg = lg[..., torch.as_tensor(perm, dtype=torch.long)]
        outs.append(lg)
    if avg_before:
        out = torch.softmax(torch.stack(outs).mean(0), dim=1)
    else:
        out = torch.stack([torch.softmax(o, dim=1) for o in outs]).mean(0)
    if class_counts is not None:
        cc = torch.as_tensor(class_counts, dtype=torch.float64)
        out = out * (cc / cc.sum())
        out = out / out.sum(-1, keepdim=True)
    return out / out.sum(1, keepdim=True)


def _proba_raw(logits, perms, *, n_classes, temperature, avg_before, class_counts):
    """engine.proba_device, and mmpfn_proba_tail with the same arguments into a NaN buffer with PAD elements past its
    end: the two must agree bit for bit -> proba [S, width] (CPU)."""
    n_est, S, n_out = logits.shape
    got = proba_device(logits, perms, n_classes=n_classes, softmax_temperature=temperature,
                       average_before_softmax=avg_before, balance_probabilities=class_counts is not None,
                       class_counts=class_counts)
    width = n_out if (temperature == 1 and all(p is None for p in perms)) else n_classes
    perm = np.stack([np.arange(width) if p is None else np.asarray(p) for p in perms]).astype(np.int32)
    perm = torch.from_numpy(perm).cuda()
    prior = None
    if class_counts is not None:
        cc = np.asarray(class_counts, dtype=np.float64)
        prior = torch.from_numpy((cc / cc.sum()).astype(np.float32)).cuda()
    out = _nan_buffer(S * width)
    _lib.check(_lib.load().mmpfn_proba_tail(logits.data_ptr(), perm.data_ptr(), None if prior is None else prior.data_ptr(),
                                            n_est, S, n_out, width, temperature, int(avg_before), out.data_ptr(),
                                            _stream()), "mmpfn_proba_tail")
    torch.cuda.synchronize()
    _assert_tail_untouched(out, S * width)
    raw = out[:S * width].view(S, width)
    assert got.shape == raw.shape and torch.equal(got, raw)
    return got.cpu()


PROBA_CASES = [
    # n_est, S, n_out, n_classes, permuted
    (1, 1, 10, 2, False),
    (3, 333, 10, 3, True),
    (8, 1000, 10, 10, True),
    (4, 517, 64, 10, False),
    (2, 129, 64, 64, True),
    (5, 77, 64, 33, True),
    (8, 100_003, 10, 10, True),
]


@pytest.mark.parametrize("temperature", [0.9, 1.0])
@pytest.mark.parametrize("avg_before", [False, True])
@pytest.mark.parametrize("n_est,S,n_out,n_classes,permuted", PROBA_CASES)
def test_proba_tail_vs_oracle(n_est, S, n_out, n_classes, permuted, temperature, avg_before):
    """Logits up to +-80 (exp of 80 / 0.9 overflows fp32 without the max shift), 1 to 8 estimators, up to 64 classes,
    with and without class permutations, both temperatures (at 1 without permutations every one of the n_out logits
    enters the softmax), both averaging modes, with and without balanced priors."""
    gen = torch.Generator().manual_seed(n_est * 1000 + S + n_out + n_classes)
    logits = (torch.rand(n_est, S, n_out, generator=gen) * 160 - 80)
    logits[:, 0] = 80.0                                        # a row of equal extreme logits
    rng = np.random.default_rng(S + n_classes)
    perms = [rng.permutation(n_classes) if permuted else None for _ in range(n_est)]
    width = n_out if (temperature == 1 and not permuted) else n_classes
    counts = rng.integers(1, 50, size=width)
    for class_counts in (None, counts):
        got = _proba_raw(logits.cuda(), perms, n_classes=n_classes, temperature=temperature, avg_before=avg_before,
                         class_counts=class_counts)
        ref = _proba_ref(logits, perms, n_classes, temperature, avg_before, class_counts)
        assert got.shape == ref.shape
        if S <= 1000:
            # the restatement is the oracle's: the fp32 oracle agrees with it to fp32 rounding at these logit scales
            # (a slice, permutation or prior applied differently would be off by O(1 / n_classes))
            ora = R.proba_tail(list(logits), perms, n_classes, softmax_temperature=temperature,
                               average_before_softmax=avg_before, balance_probabilities=class_counts is not None,
                               class_counts=class_counts)
            assert np.abs(ora - ref.numpy()).max() < 1e-3
        # z / T in fp32 (|z/T| <= 89) carries 2^-24 * 89 of absolute error, the estimator sum (partial sums up to
        # n_est * 89, then / n_est) up to n_est times that, and - max up to twice that: an exponent off by at most
        # (n_est + 3) * 2^-24 * 89, which each probability carries twice (numerator and normaliser) as relative error;
        # exp, the sums, the prior and the renormalisations add a few 2^-24 inside that margin
        rel = 2 * (n_est + 3) * U32 * 89.0
        _assert_close(got, ref, rel * ref + 1e-30, "proba")
        assert torch.allclose(got.double().sum(1), torch.ones(S, dtype=torch.float64), atol=1e-5)


def test_proba_tail_refusals():
    """More than 64 classes, or more classes than logits per row: MMPFN_EINVAL, nothing written."""
    lib = _lib.load()
    logits = torch.zeros(1, 5, 70, device="cuda")
    perm = torch.arange(70, dtype=torch.int32, device="cuda")
    out = _nan_buffer(5 * 70)
    for n_out, n_classes in ((70, 65), (10, 11)):
        rc = lib.mmpfn_proba_tail(logits.data_ptr(), perm.data_ptr(), None, 1, 5, n_out, n_classes, 0.9, 0,
                                  out.data_ptr(), _stream())
        assert rc == EINVAL, rc
        assert b"n_classes" in lib.mmpfn_last_error()
    torch.cuda.synchronize()
    assert torch.isnan(out).all()
    # at 64 classes the kernel runs (its per-row arrays hold 64)
    rc = lib.mmpfn_proba_tail(logits.data_ptr(), perm.data_ptr(), None, 1, 5, 70, 64, 0.9, 0, out.data_ptr(), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.allclose(out[:5 * 64], torch.full((5 * 64,), 1 / 64, device="cuda"))
    _assert_tail_untouched(out, 5 * 64)


def test_proba_device_refuses_priors_of_other_width():
    """Temperature 1 without permutations keeps all n_out columns; class counts for n_classes of them do not
    broadcast (the reference fails there too), and the kernel would read past the end of the prior."""
    logits = torch.zeros(2, 4, 10, device="cuda")
    with pytest.raises(ValueError, match="class counts"):
        proba_device(logits, [None, None], n_classes=3, softmax_temperature=1.0, balance_probabilities=True,
                     class_counts=[3, 4, 5])
