"""CPU checks of the regressor: the border maps, the float64 oracle of the bar-distribution tail, and the refusals of
``MMPFNRegressor`` that need no device."""
import warnings

import numpy as np
import pytest
import torch
from scipy.stats import halfnorm
from sklearn.preprocessing import PowerTransformer

from multimodalpfn_b200.regressor import MMPFNRegressor, border_map, member_borders
from multimodalpfn_b200.synth import Geometry, make_state_dict
from oracle import bar_distribution as O
from oracle import ref_compat


def _g(K, seed=0):
    rng = np.random.default_rng(seed)
    return np.cumsum(np.concatenate([[-3.0], rng.uniform(0.05, 1.0, K)]))


def _power(seed=0, n=300):
    rng = np.random.default_rng(seed)
    y = rng.lognormal(0.0, 0.8, n)
    y_z = (y - y.mean()) / y.std()
    return PowerTransformer(method="yeo-johnson", standardize=True).fit(y_z[:, None])


def _translate_direct(p, f, g):
    """Estimator CDF at the common borders by direct float64 interpolation of its piecewise-linear CDF."""
    cdf_f = np.concatenate([[0.0], np.cumsum(p)])
    C = np.interp(g, f, cdf_f, left=0.0, right=1.0)
    C[0], C[-1] = 0.0, 1.0
    return np.maximum(np.diff(C), 0.0)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_border_map_matches_direct_cdf(seed):
    rng = np.random.default_rng(seed)
    K = 50
    g = _g(K, seed)
    f = np.sort(g * rng.uniform(0.5, 1.5) + rng.normal(0, 0.5) + rng.normal(0, 0.05, K + 1))
    b, s = border_map(f, g)
    ob, os_ = O.border_map(f, g)
    np.testing.assert_array_equal(b, ob)
    np.testing.assert_allclose(s, os_, atol=1e-7)
    logits = rng.normal(0, 2, (4, K))
    q = O.translate(logits, b, s.astype(np.float64))
    p = np.exp(logits - logits.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    for r in range(4):
        np.testing.assert_allclose(q[r], _translate_direct(p[r], f, g), atol=1e-6)
    np.testing.assert_allclose(q.sum(1), 1.0, atol=1e-12)


def test_identity_translation():
    K = 40
    g = _g(K)
    b, s = border_map(g, g)
    np.testing.assert_array_equal(b[:K], np.arange(K))
    assert b[K] == K and np.all(s == 0)
    logits = np.random.default_rng(3).normal(0, 1, (5, K))
    p = np.exp(logits - logits.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    np.testing.assert_allclose(O.translate(logits, b, s), p, rtol=1e-12, atol=1e-15)
    f, cancel = member_borders(None, g)
    assert np.array_equal(f, g) and not cancel.any()


def test_cancel_rule_on_non_finite_borders():
    pt = _power(0)
    # wide borders: the inverse Yeo-Johnson transform leaves its domain on one side
    g = np.linspace(-40.0, 40.0, 65)
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        raw = pt.inverse_transform(g[:, None]).ravel()
    assert not np.all(np.isfinite(raw)), "this transform should produce non-finite borders"
    f, cancel = member_borders(pt, g)
    assert np.all(np.isfinite(f)) and np.all(np.diff(f) >= 0)
    of, ocancel = O.member_borders(raw)
    np.testing.assert_array_equal(f, of)
    np.testing.assert_array_equal(cancel, ocancel)
    bad = ~np.isfinite(raw)
    assert np.all(cancel[bad[:-1] | bad[1:]])
    assert np.all(cancel == ~(np.diff(f) > 0) | bad[:-1] | bad[1:])
    # cancelled buckets carry no mass
    b, s = border_map(f, g)
    logits = np.random.default_rng(1).normal(0, 1, (3, 64))
    z = np.where(cancel[None], -np.inf, logits)
    p = np.exp(z - z.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    assert np.all(p[:, cancel] == 0)
    q = O.translate(logits, b, s, cancel)
    np.testing.assert_allclose(q.sum(1), 1.0, atol=1e-12)


def test_one_bucket_distribution_mean():
    K = 10
    G = _g(K)
    for j in (1, 4, K - 2):
        P = np.zeros((1, K))
        P[0, j] = 1.0
        assert O.mean(P, G)[0] == pytest.approx(0.5 * (G[j] + G[j + 1]))
        assert O.mode(P, G)[0] == pytest.approx(0.5 * (G[j] + G[j + 1]))
        assert O.quantile(P, G, 0.5)[0] == pytest.approx(0.5 * (G[j] + G[j + 1]))


def test_quantiles_monotone():
    rng = np.random.default_rng(4)
    K = 100
    G = _g(K, 4)
    P = rng.dirichlet(np.full(K, 0.3), size=20)
    qs = np.linspace(0.001, 0.999, 200)
    vals = np.stack([O.quantile(P, G, q) for q in qs])
    assert np.all(np.diff(vals, axis=0) >= -1e-12)


def test_symmetric_distribution_median_at_centre():
    K = 21
    G = np.linspace(-5, 5, K + 1) + 2.0
    w = np.exp(-0.5 * np.linspace(-2, 2, K) ** 2)
    P = (w / w.sum())[None]
    assert O.quantile(P, G, 0.5)[0] == pytest.approx(2.0, abs=1e-12)
    assert O.mean(P, G)[0] == pytest.approx(2.0, abs=1e-12)
    lo, hi = O.quantile(P, G, 0.2)[0], O.quantile(P, G, 0.8)[0]
    assert lo - 2.0 == pytest.approx(2.0 - hi, abs=1e-12)


def test_tail_quantiles_are_half_normal():
    K = 8
    G = _g(K, 5)
    P = np.full((1, K), 1.0 / K)
    w0, wl = G[1] - G[0], G[K] - G[K - 1]
    for q in (0.01, 0.05, 0.1):
        r = q / P[0, 0]
        assert O.quantile(P, G, q)[0] == pytest.approx(G[1] - halfnorm.ppf(1 - r, scale=w0), rel=1e-10)
    for q in (0.9, 0.95, 0.99):
        r = (q - (K - 1) / K) / P[0, -1]
        assert O.quantile(P, G, q)[0] == pytest.approx(G[K - 1] + halfnorm.ppf(r, scale=wl), rel=1e-10)
    assert O.mean(P, G)[0] == pytest.approx(np.mean(O.bucket_means(G)))
    assert O.bucket_means(G)[0] == pytest.approx(G[1] - halfnorm.mean(scale=w0))


def test_average_before_softmax_zero_bucket():
    q1 = np.array([[0.5, 0.5, 0.0]])
    q2 = np.array([[0.2, 0.3, 0.5]])
    P = O.combine([q1, q2], average_before_softmax=True)
    assert P[0, 2] == 0 and P.sum() == pytest.approx(1.0)
    np.testing.assert_allclose(O.combine([q1, q2]), [[0.35, 0.4, 0.25]])


# ---- constructor and fit validation (no device needed: the checks run before the model is built) -------------
def _reg_ckpt(n_out=16, regression=True):
    geom = Geometry(mgm_heads=2, cap_heads=4, n_out=n_out)
    return make_state_dict(geom, seed=3, regression=regression), geom


def test_regressor_params_round_trip():
    r = MMPFNRegressor(n_estimators=3, softmax_temperature=1.0)
    p = r.get_params()
    assert p["n_estimators"] == 3 and p["softmax_temperature"] == 1.0 and p["average_before_softmax"] is False
    for k in ("mixer_type", "mgm_heads", "cap_heads", "features_per_group", "model_path", "device",
              "ignore_pretraining_limits", "inference_precision", "fit_mode", "random_state", "inference_config"):
        assert k in p


@pytest.mark.parametrize("y, msg", [([1.0, np.nan, 2.0], "NaN or infinite"), ([1.0, np.inf, 2.0], "NaN or infinite"),
                                    ([2.0, 2.0, 2.0], "zero spread")])
def test_fit_refuses_bad_targets(y, msg):
    X = np.zeros((3, 2), np.float32)
    with pytest.raises(ValueError, match=msg):
        MMPFNRegressor(model_path=_reg_ckpt()).fit(X, None, y)


def test_fit_refuses_classification_checkpoint():
    X = np.random.default_rng(0).normal(size=(5, 2)).astype(np.float32)
    with pytest.raises(ValueError, match="classification checkpoint"):
        MMPFNRegressor(model_path=_reg_ckpt(regression=False)).fit(X, None, np.arange(5.0))


def test_fit_refuses_missing_or_bad_borders():
    X = np.random.default_rng(0).normal(size=(5, 2)).astype(np.float32)
    sd, geom = _reg_ckpt()
    sd2 = dict(sd)
    del sd2["criterion.borders"]
    with pytest.raises(ValueError, match="criterion.borders"):
        MMPFNRegressor(model_path=(sd2, geom)).fit(X, None, np.arange(5.0))
    sd3 = dict(sd, **{"criterion.borders": sd["criterion.borders"][::-1].copy()})
    with pytest.raises(ValueError, match="increasing"):
        MMPFNRegressor(model_path=(sd3, geom)).fit(X, None, np.arange(5.0))
    with pytest.raises(ValueError, match="model_path"):
        MMPFNRegressor().fit(X, None, np.arange(5.0))


def test_load_borders_from_checkpoint(tmp_path):
    from multimodalpfn_b200.synth import make_checkpoint_config
    from multimodalpfn_b200.weights import load_borders, load_checkpoint
    sd, geom = _reg_ckpt()
    path = tmp_path / "reg.ckpt"
    torch.save({"state_dict": {k: torch.as_tensor(v) for k, v in sd.items()},
                "config": make_checkpoint_config(geom, regression=True)}, path)
    np.testing.assert_array_equal(load_borders(path), sd["criterion.borders"].astype(np.float64))
    sd_loaded, geom_loaded = load_checkpoint(path, mgm_heads=2, cap_heads=4)
    assert "criterion.borders" not in sd_loaded and geom_loaded.n_out == 16
    sdc, geomc = _reg_ckpt(regression=False)
    torch.save({"state_dict": {k: torch.as_tensor(v) for k, v in sdc.items()},
                "config": make_checkpoint_config(geomc)}, tmp_path / "clf.ckpt")
    with pytest.raises(ValueError, match="criterion.borders"):
        load_borders(tmp_path / "clf.ckpt")


def test_fit_refuses_bad_options():
    X = np.random.default_rng(0).normal(size=(5, 2)).astype(np.float32)
    with pytest.raises(ValueError, match="fit_mode"):
        MMPFNRegressor(model_path=_reg_ckpt(), fit_mode="nope").fit(X, None, np.arange(5.0))
    with pytest.raises(ValueError, match="REGRESSION_Y_PREPROCESS_TRANSFORMS"):
        MMPFNRegressor(model_path=_reg_ckpt(),
                       inference_config={"REGRESSION_Y_PREPROCESS_TRANSFORMS": ("log",)}).fit(X, None, np.arange(5.0))
    with pytest.raises(ValueError, match="different numbers of rows"):
        MMPFNRegressor(model_path=_reg_ckpt()).fit(X, None, np.arange(4.0))


# ---- the oracle against the reference's own bar distribution (skips unless the reference is installed) -------
@pytest.mark.skipif(not ref_compat.reference_available(), reason="reference package not installed")
def test_oracle_matches_reference_bar_distribution():
    ref_compat.install()
    from mmpfn.models.mmpfn.model.bar_distribution import FullSupportBarDistribution
    from mmpfn.models.mmpfn.regressor import translate_probs_across_borders
    rng = np.random.default_rng(7)
    K = 64
    g = _g(K, 7)
    f, cancel = member_borders(_power(7), g)
    logits = rng.normal(0, 2, (6, K))
    z = np.where(cancel[None], -np.inf, logits)
    b, s = O.border_map(f, g)
    ours = O.translate(logits, b, s, cancel)
    theirs = translate_probs_across_borders(torch.as_tensor(z), frm=torch.as_tensor(f),
                                            to=torch.as_tensor(g)).numpy()
    np.testing.assert_allclose(ours, theirs, atol=1e-9)
    P = rng.dirichlet(np.full(K, 0.5), size=6)
    crit = FullSupportBarDistribution(torch.as_tensor(g))
    lp = torch.as_tensor(np.log(P))
    np.testing.assert_allclose(O.mean(P, g), crit.mean(lp).numpy(), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(O.mode(P, g), crit.mode(lp).numpy(), rtol=1e-9, atol=1e-9)
    for q in (0.05, 0.5, 0.95):
        np.testing.assert_allclose(O.quantile(P, g, q), crit.icdf(lp, q).numpy(), rtol=1e-7, atol=1e-7)
