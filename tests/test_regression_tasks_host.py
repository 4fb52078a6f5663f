"""Host side of packed regression tasks: the shared per-dataset preparation (``prepare_regression``) is deterministic,
and the refusals of ``predict_regression_tasks`` that come before any device work."""
from types import SimpleNamespace

import numpy as np
import pytest

from multimodalpfn_b200.regressor import MMPFNRegressor, check_borders, prepare_regression
from multimodalpfn_b200.synth import Geometry, make_state_dict
from multimodalpfn_b200.tasks import predict_regression_tasks


def _borders(K=64):
    geom = Geometry(mgm_heads=1, cap_heads=1, n_out=K, nlayers=1)
    return make_state_dict(geom, seed=0, regression=True)["criterion.borders"]


def _data(seed=0, n=120, F=6):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, F)).astype(np.float32)
    X[::5, 2] = np.nan
    y = np.exp(0.5 * X[:, 0] + rng.normal(0, 0.4, n)) * 4 + 1
    return X, y


def _stand_in(regression=True, n_out=64):
    """What predict_regression_tasks reads of a model before its first device call."""
    return SimpleNamespace(w=SimpleNamespace(regression=regression), geom=SimpleNamespace(n_out=n_out), device=None)


def _tasks(n=3):
    out = []
    for i in range(n):
        X, y = _data(i)
        out.append(dict(X_train=X[:100], X_test=X[100:], y_train=y[:100], img_train=None, img_test=None))
    return out


@pytest.mark.parametrize("with_table", [True, False])
def test_prepare_regression_is_deterministic(with_table):
    g = check_borders(_borders(), 64)
    X, y = _data(3)
    X = X if with_table else None
    a = prepare_regression(X, y, g, n_estimators=5, random_state=7)
    b = prepare_regression(X, y, g, n_estimators=5, random_state=7)
    for k in ("src_bucket", "src_share", "cancel", "target_borders"):
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k
    assert a["src_bucket"].shape == (5, 65) and a["src_bucket"].dtype == np.int32
    assert a["src_share"].dtype == np.float32 and a["cancel"].shape == (5, 64) and a["cancel"].dtype == bool
    assert a["y_mean"] == b["y_mean"] and a["y_std"] == b["y_std"]
    assert [t is None for t in a["transforms"]] == [True, False, True, False, True]
    for ta, tb in zip(a["tables"], b["tables"]):
        assert ta["class_perm"] is None and tb["class_perm"] is None
        assert ta["y_train"].dtype == np.float32 and np.array_equal(ta["y_train"], tb["y_train"])
        if with_table:
            assert np.array_equal(ta["X_train"], tb["X_train"], equal_nan=True)
        else:
            assert ta["X_train"] is None and tb["X_train"] is None
    np.testing.assert_allclose(a["target_borders"], g * a["y_std"] + a["y_mean"], rtol=0, atol=0)


def test_check_borders_refusals():
    g = np.asarray(_borders(), dtype=np.float64)
    assert np.array_equal(check_borders(g, 64), g)
    for bad in (g[:-1], g[::-1], np.where(np.arange(65) == 9, np.nan, g), np.where(np.arange(65) == 0, -np.inf, g)):
        with pytest.raises(ValueError, match="65 finite increasing"):
            check_borders(bad, 64)
    with pytest.raises(ValueError, match="without criterion.borders"):
        check_borders(None, 64)


def test_prepare_regression_target_refusals():
    g = check_borders(_borders(), 64)
    X, y = _data()
    with pytest.raises(ValueError, match="NaN or infinite"):
        prepare_regression(X, np.where(np.arange(len(y)) == 4, np.nan, y), g, n_estimators=2)
    with pytest.raises(ValueError, match="zero spread"):
        prepare_regression(X, np.full(len(y), 2.5), g, n_estimators=2)
    with pytest.raises(ValueError, match="1-dimensional"):
        prepare_regression(X, y[:, None], g, n_estimators=2)


def test_tasks_host_refusals():
    g = _borders()
    tasks = _tasks()
    with pytest.raises(ValueError, match="classification checkpoint"):
        predict_regression_tasks(_stand_in(regression=False), g, tasks)
    with pytest.raises(ValueError, match="65 finite increasing"):
        predict_regression_tasks(_stand_in(), g[:-1], tasks)
    with pytest.raises(ValueError, match="64 finite increasing"):
        predict_regression_tasks(_stand_in(n_out=63), g, tasks)
    with pytest.raises(ValueError, match="at most 8192"):
        predict_regression_tasks(_stand_in(n_out=8193), np.linspace(-4, 4, 8194), tasks)
    bad = [dict(t) for t in tasks]
    bad[1]["y_train"] = np.where(np.arange(100) == 7, np.nan, bad[1]["y_train"])
    with pytest.raises(ValueError, match="task 1: y holds NaN or infinite"):
        predict_regression_tasks(_stand_in(), g, bad)
    bad = [dict(t) for t in tasks]
    bad[2]["y_train"] = np.ones(100)
    with pytest.raises(ValueError, match="task 2: y has zero spread"):
        predict_regression_tasks(_stand_in(), g, bad)
    with pytest.raises(ValueError, match="quantiles must lie"):
        predict_regression_tasks(_stand_in(), g, tasks, output_type="quantiles", quantiles=[0.5, 1.0])


def test_regressor_refuses_classification_state_dict():
    geom = Geometry(mgm_heads=1, cap_heads=1, nlayers=1)
    reg = MMPFNRegressor(mgm_heads=1, cap_heads=1, model_path=(make_state_dict(geom, seed=0), geom))
    with pytest.raises(ValueError, match="classification checkpoint"):
        reg._checkpoint()
