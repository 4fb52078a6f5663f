"""GPU checks of the regressor: ``mmpfn_bar_tail`` against the float64 oracle (oracle/bar_distribution.py) on seeded
logits, and ``MMPFNRegressor`` end to end against the oracle applied to the same engine logits.

Tolerances: log P within 1e-4 where P >= 1e-6; mean, median, mode and quantiles within 1e-4 of the inner border span
G[K-1] - G[1].  With average_before_softmax, log P is compared only on buckets where every estimator's mass is at
least 1e-12: below that the geometric mean is set by float64 rounding in the oracle and the kernel alike."""
import numpy as np
import pytest
import torch
from sklearn.preprocessing import PowerTransformer

from multimodalpfn_b200 import _lib
from multimodalpfn_b200.preprocessing import transform_all
from multimodalpfn_b200.regressor import MMPFNRegressor, bar_tail_device, border_map, member_borders
from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
from oracle import bar_distribution as O

pytestmark = pytest.mark.gpu

LP_TOL = 1e-4
VAL_TOL = 1e-4
QS = (0.05, 0.1, 0.25, 0.5, 0.75, 0.9, 0.95)
ALL = ("mean", "median", "mode", "quantiles", "log_prob")


def _std_borders(K):
    return np.asarray(make_state_dict(Geometry(mgm_heads=1, cap_heads=1, n_out=K, nlayers=1), seed=0,
                                      regression=True)["criterion.borders"], dtype=np.float64)


def _maps(K, n_est, seed):
    """Border maps of real power transforms (every other member) plus a random cancel mask on some members."""
    rng = np.random.default_rng(seed)
    g = _std_borders(K)
    buckets, shares, cancels = [], [], []
    for e in range(n_est):
        tf = None
        if e % 2 == 1:
            y = rng.lognormal(0.0, rng.uniform(0.3, 1.2), 400)
            y_z = (y - y.mean()) / y.std()
            tf = PowerTransformer(method="yeo-johnson", standardize=True).fit(y_z[:, None])
        f, cancel = member_borders(tf, g)
        if e % 3 == 2:
            cancel = cancel | (rng.random(K) < 0.03)
        b, s = border_map(f, g)
        buckets.append(b)
        shares.append(s)
        cancels.append(cancel)
    G = g * rng.uniform(0.5, 3.0) + rng.normal()
    return np.stack(buckets), np.stack(shares), np.stack(cancels), G


def _oracle(logits, b, s, cancel, G, temperature, avg):
    return O.bar_tail(logits.astype(np.float64), b, s.astype(np.float64), cancel, G, temperature=temperature,
                      average_before_softmax=avg, quantiles=QS)


def _check(got, ref, G, what=""):
    span = float(G[-2] - G[1])
    if "log_prob" in got:
        lp = got["log_prob"]
        big = ref["P"] >= 1e-6
        ok = ref["conditioned"]
        err = float(np.abs(lp[big & ok] - ref["log_prob"][big & ok]).max())
        assert err <= LP_TOL, (what, "log_prob", err)
        assert np.all(np.exp(lp[~big & ok]) <= 2e-6), (what, "small buckets")
    for k in ("mean", "median", "quantiles"):
        if k in got:
            err = float(np.abs(got[k] - ref[k]).max()) / span
            assert err <= VAL_TOL, (what, k, err)
    if "mode" in got:
        bad = np.abs(got["mode"] - ref["mode"]) > VAL_TOL * span
        if bad.any():                   # a near tie of two bucket densities may resolve either way in fp32
            dens = ref["P"] / np.diff(G)[None]
            mid = 0.5 * (G[:-1] + G[1:])
            j = np.argmin(np.abs(mid[None] - got["mode"][:, None]), axis=1)
            rows = np.nonzero(bad)[0]
            assert np.all(dens[rows, j[rows]] >= dens[rows].max(1) * (1 - 1e-5)), (what, "mode")


def _run(logits, b, s, cancel, G, temperature, avg, outputs=ALL):
    dev = torch.device("cuda")
    out = bar_tail_device(torch.as_tensor(logits, device=dev), torch.as_tensor(b, device=dev),
                          torch.as_tensor(s, device=dev),
                          None if cancel is None else torch.as_tensor(cancel.astype(np.uint8), device=dev),
                          torch.as_tensor(G.astype(np.float32), device=dev), softmax_temperature=temperature,
                          average_before_softmax=avg, quantiles=torch.tensor(QS, dtype=torch.float32, device=dev),
                          outputs=outputs)
    return {k: v.cpu().numpy() for k, v in out.items()}


SHAPES = [(64, 1, 1), (64, 3, 2000), (64, 8, 777), (5000, 1, 64), (5000, 3, 200), (5000, 8, 120)]


@pytest.mark.parametrize("K,n_est,S", SHAPES)
@pytest.mark.parametrize("temperature", [1.0, 0.9])
@pytest.mark.parametrize("avg", [False, True])
def test_bar_tail_vs_oracle(K, n_est, S, temperature, avg):
    seed = K + 10 * n_est + S
    rng = np.random.default_rng(seed)
    b, s, cancel, G = _maps(K, n_est, seed)
    logits = (rng.normal(0, 2.5, (n_est, S, K)) + np.linspace(-3, 3, K)[None, None] ** 2 * -0.5).astype(np.float32)
    got = _run(logits, b, s, cancel, G, temperature, avg)
    ref = _oracle(logits, b, s, cancel, G, temperature, avg)
    _check(got, ref, G, f"K{K} n{n_est} S{S} t{temperature} avg{avg}")


def test_outputs_alone_equal_together_and_null_untouched():
    K, n_est, S = 64, 3, 300
    rng = np.random.default_rng(5)
    b, s, cancel, G = _maps(K, n_est, 5)
    logits = rng.normal(0, 2, (n_est, S, K)).astype(np.float32)
    together = _run(logits, b, s, cancel, G, 0.9, False)
    lib = _lib.load()
    dev = torch.device("cuda")
    lg = torch.as_tensor(logits, device=dev)
    bd, sd = torch.as_tensor(b, device=dev), torch.as_tensor(s, device=dev)
    cd = torch.as_tensor(cancel.astype(np.uint8), device=dev)
    Gd = torch.as_tensor(G.astype(np.float32), device=dev)
    qd = torch.tensor(QS, dtype=torch.float32, device=dev)
    shapes = dict(mean=(S,), median=(S,), mode=(S,), quantiles=(len(QS), S), log_prob=(S, K))
    for name in ALL:
        bufs = {k: torch.full(shapes[k], 7.0, device=dev) for k in ALL}
        ptrs = [bufs[k].data_ptr() if k == name else None for k in ALL]
        _lib.check(lib.mmpfn_bar_tail(lg.data_ptr(), n_est, S, K, bd.data_ptr(), sd.data_ptr(), cd.data_ptr(),
                                      Gd.data_ptr(), 0.9, 0, qd.data_ptr(), len(QS), *ptrs,
                                      torch.cuda.current_stream().cuda_stream), "mmpfn_bar_tail")
        torch.cuda.synchronize()
        for k in ALL:
            v = bufs[k].cpu().numpy()
            if k == name:
                assert np.array_equal(v, together[k]), name
            else:
                assert np.all(v == 7.0), (name, k)


def test_bar_tail_refusals():
    lib = _lib.load()
    dev = torch.device("cuda")
    K = 8193
    lg = torch.zeros((1, 1, K), device=dev)
    b = torch.zeros((1, K + 1), dtype=torch.int32, device=dev)
    s = torch.zeros((1, K + 1), device=dev)
    G = torch.arange(K + 1, dtype=torch.float32, device=dev)
    mean = torch.zeros(1, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    args = (None, G.data_ptr(), 0.9, 0, None, 0, mean.data_ptr(), None, None, None, None, st)
    assert lib.mmpfn_bar_tail(lg.data_ptr(), 1, 1, K, b.data_ptr(), s.data_ptr(), *args) == -4     # EUNSUPPORTED
    assert b"8192" in lib.mmpfn_last_error()
    assert lib.mmpfn_bar_tail(lg.data_ptr(), 1, 1, 1, b.data_ptr(), s.data_ptr(), None, G.data_ptr(), 0.9, 0, None,
                              0, mean.data_ptr(), None, None, None, None, st) == -1                  # K < 2
    assert lib.mmpfn_bar_tail(lg.data_ptr(), 1, 1, 64, b.data_ptr(), s.data_ptr(), None, G.data_ptr(), 0.9, 0, None,
                              0, None, None, None, mean.data_ptr(), None, st) == -1                  # quant w/o levels
    assert lib.mmpfn_bar_tail(lg.data_ptr(), 1, 1, 64, b.data_ptr(), s.data_ptr(), None, G.data_ptr(), 0.0, 0, None,
                              0, mean.data_ptr(), None, None, None, None, st) == -1                  # temperature 0


# ---- the regressor end to end ---------------------------------------------------------------------------------
def _regression_data(seed=0):
    d = make_dataset("pad_ufes_small", seed)
    rng = np.random.default_rng(seed + 100)
    X = np.concatenate([d["X_train"], d["X_test"]])
    Xz = np.nan_to_num(X)
    Xz = (Xz - Xz.mean(0)) / (Xz.std(0) + 1e-6)
    img = np.concatenate([d["img_train"], d["img_test"]])
    y = np.exp(0.3 * (Xz @ rng.normal(0, 0.4, X.shape[1]) + img[:, 0, :8].sum(1) * 0.2)) * 10 + rng.normal(0, 0.5, len(X))
    n = len(d["X_train"])
    return d, y[:n].astype(np.float32), y[n:]


def _regressor(n_out, precision, fit_mode="fit_preprocessors", n_estimators=4, **kw):
    geom = Geometry(mgm_heads=2, cap_heads=4, n_out=n_out)
    sd = make_state_dict(geom, seed=9, regression=True)
    return MMPFNRegressor(mgm_heads=2, cap_heads=4, n_estimators=n_estimators, model_path=(sd, geom), device="cuda",
                          inference_precision=precision, fit_mode=fit_mode, random_state=0, **kw)


def _oracle_of(reg, X_test, img_test):
    logits = reg.executor_.logits(transform_all(reg.members_, X_test), img_test).cpu().numpy()
    cancel = None if reg._cancel is None else reg._cancel.cpu().numpy().astype(bool)
    qs = np.round(np.arange(1, 10) * 0.1, 1)
    ref = O.bar_tail(logits.astype(np.float64), reg._src_bucket.cpu().numpy(),
                     reg._src_share.cpu().numpy().astype(np.float64), cancel, reg.target_borders_,
                     temperature=reg.softmax_temperature, average_before_softmax=reg.average_before_softmax,
                     quantiles=qs)
    return ref


@pytest.mark.parametrize("n_out", [64, 5000])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_regressor_end_to_end_vs_oracle(n_out, precision):
    d, y_tr, _ = _regression_data(0)
    reg = _regressor(n_out, precision).fit(d["X_train"], d["img_train"], y_tr)
    assert any(t is not None for t in reg.target_transforms_) and any(t is None for t in reg.target_transforms_)
    ref = _oracle_of(reg, d["X_test"], d["img_test"])
    G = reg.target_borders_
    full = reg.predict(d["X_test"], d["img_test"], output_type="full")
    assert set(full) == {"mean", "median", "mode", "quantiles", "logits", "borders"}
    assert full["logits"].shape == (len(d["X_test"]), n_out) and full["logits"].dtype == np.float32
    np.testing.assert_allclose(full["borders"], G.astype(np.float32))
    _check(dict(mean=full["mean"], median=full["median"], mode=full["mode"], quantiles=np.stack(full["quantiles"]),
                log_prob=full["logits"]), ref, G, f"full {n_out} {precision}")
    main = reg.predict(d["X_test"], d["img_test"], output_type="main")
    assert set(main) == {"mean", "median", "mode", "quantiles"} and len(main["quantiles"]) == 9
    _check(dict(mean=main["mean"], median=main["median"], mode=main["mode"], quantiles=np.stack(main["quantiles"])),
           ref, G, f"main {n_out} {precision}")
    for k in ("mean", "median", "mode"):
        v = reg.predict(d["X_test"], d["img_test"], output_type=k)
        assert v.dtype == np.float32 and v.shape == (len(d["X_test"]),)
        np.testing.assert_array_equal(v, main[k])
    q = reg.predict(d["X_test"], d["img_test"], output_type="quantiles", quantiles=[0.5, 0.9])
    np.testing.assert_array_equal(q[0], main["median"])
    np.testing.assert_array_equal(q[1], main["quantiles"][8])
    assert np.all(np.diff(np.stack(main["quantiles"]), axis=0) >= 0)


def test_fit_with_cache_equals_fit_preprocessors():
    d, y_tr, _ = _regression_data(1)
    outs = []
    for mode in ("fit_preprocessors", "fit_with_cache"):
        reg = _regressor(64, "bf16", fit_mode=mode).fit(d["X_train"], d["img_train"], y_tr)
        outs.append(reg.predict(d["X_test"], d["img_test"], output_type="full"))
    for k in ("mean", "median", "mode", "logits"):
        assert np.array_equal(outs[0][k], outs[1][k]), k
    assert np.array_equal(np.stack(outs[0]["quantiles"]), np.stack(outs[1]["quantiles"]))


def test_image_only_and_average_before_softmax():
    d, y_tr, _ = _regression_data(2)
    reg = _regressor(64, "fp32", average_before_softmax=True, softmax_temperature=1.0)
    reg.fit(None, d["img_train"], y_tr)
    ref = _oracle_of(reg, None, d["img_test"])
    main = reg.predict(None, d["img_test"], output_type="main")
    _check(dict(mean=main["mean"], median=main["median"], mode=main["mode"], quantiles=np.stack(main["quantiles"])),
           ref, reg.target_borders_, "image only")


def test_regressor_refusals():
    d, y_tr, _ = _regression_data(0)
    reg = _regressor(64, "bf16")
    with pytest.raises(ValueError, match="classification checkpoint"):
        geom = Geometry(mgm_heads=2, cap_heads=4)
        MMPFNRegressor(mgm_heads=2, cap_heads=4, model_path=(make_state_dict(geom, seed=1), geom),
                       device="cuda").fit(d["X_train"], d["img_train"], y_tr)
    with pytest.raises(ValueError, match="NaN or infinite"):
        reg.fit(d["X_train"], d["img_train"], np.where(np.arange(len(y_tr)) == 3, np.nan, y_tr))
    with pytest.raises(ValueError, match="zero spread"):
        reg.fit(d["X_train"], d["img_train"], np.ones_like(y_tr))
    reg.fit(d["X_train"], d["img_train"], y_tr)
    with pytest.raises(ValueError, match="output_type"):
        reg.predict(d["X_test"], d["img_test"], output_type="proba")
    with pytest.raises(ValueError, match="between 0 and 1"):
        reg.predict(d["X_test"], d["img_test"], output_type="quantiles", quantiles=[0.0, 0.5])
    with pytest.raises(ValueError, match="features"):
        reg.predict(d["X_test"][:, :5], d["img_test"])
