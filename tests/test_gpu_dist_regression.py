"""GPU checks of regression on the multi-GPU engine with emulated ranks (``ShardedEngine(..., group="emulate")``: one
device plays every rank, so the K/V addressing of every ownership mode, the row-sharded build, the test-row chunking
and the output gather run on a single B200).  ``MMPFNRegressor.predict(..., sharded=...)`` must return exactly what
the unsharded ``predict`` returns; the classifier's probabilities through the estimator emulation must equal
``predict_proba`` exactly."""
import numpy as np
import pytest
import torch

from multimodalpfn_b200.classifier import MMPFNClassifier
from multimodalpfn_b200.dist import ShardedEngine
from multimodalpfn_b200.preprocessing import transform_all
from multimodalpfn_b200.regressor import MMPFNRegressor
from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict

pytestmark = pytest.mark.gpu

K = 5000


def _data(name, seed=0):
    d = make_dataset(name, seed)
    rng = np.random.default_rng(seed + 100)
    X = np.nan_to_num(np.concatenate([d["X_train"], d["X_test"]]))
    X = (X - X.mean(0)) / (X.std(0) + 1e-6)
    img = np.concatenate([d["img_train"], d["img_test"]])
    y = np.exp(0.3 * (X @ rng.normal(0, 0.4, X.shape[1]) + img[:, 0, :8].sum(1) * 0.2)) * 10 \
        + rng.normal(0, 0.5, len(X))
    return d, y[:len(d["X_train"])].astype(np.float32)


def _regressor(d, y, precision, n_estimators):
    geom = Geometry(mgm_heads=2, cap_heads=4, n_out=K)
    sd = make_state_dict(geom, seed=9, regression=True)
    return MMPFNRegressor(mgm_heads=2, cap_heads=4, n_estimators=n_estimators, model_path=(sd, geom), device="cuda",
                          inference_precision=precision, random_state=0,
                          ignore_pretraining_limits=True).fit(d["X_train"], d["img_train"], y)


def _assert_same(got, ref, what):
    assert set(got) == set(ref), what
    for k in ref:
        a, b = (np.stack(got[k]), np.stack(ref[k])) if k == "quantiles" else (got[k], ref[k])
        assert a.shape == b.shape and a.dtype == b.dtype, (what, k)
        assert np.array_equal(a, b), (what, k, float(np.nanmax(np.abs(a - b))))


def _check(reg, d, world, shard="estimators", modes=None):
    sh = ShardedEngine(reg.executor_, 0, world, group="emulate", shard=shard)
    for output_type in ("main", "full"):
        ref = reg.predict(d["X_test"], d["img_test"], output_type=output_type)
        got = reg.predict(d["X_test"], d["img_test"], output_type=output_type, sharded=sh)
        _assert_same(got, ref, (world, shard, sh.exchange, output_type))
    if modes is not None:
        assert sh.exchange["mode"] in modes, sh.exchange
    return sh


# n_estimators 1 -> one group of 1 (broadcast at 2 and 4 ranks); 2 -> groups 1 + 1 (one_each at 2 ranks, broadcast at
# 4); 8 -> groups 4 + 4 (split at 2 and 4 ranks).  fp32 always runs the broadcast mode.
@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("n_est", [1, 2, 8])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_sharded_regression_estimators_emulated(precision, n_est, world):
    d, y = _data("pad_ufes_small", n_est)
    reg = _regressor(d, y, precision, n_est)
    expect = {(1, 2): "broadcast", (1, 4): "broadcast", (2, 2): "one_each", (2, 4): "broadcast", (8, 2): "split",
              (8, 4): "split"}[(n_est, world)] if precision == "bf16" else "broadcast"
    _check(reg, d, world, modes=(expect,))


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_regression_power_transform_and_cancelled_buckets(world):
    """Members with the power target transform, and buckets cancelled on some members (the tail sets their logits to
    -inf), through estimator ownership and row sharding."""
    d, y = _data("small_task", 3)
    reg = _regressor(d, y, "bf16", 8)
    assert any(t is not None for t in reg.target_transforms_)
    rng = np.random.default_rng(world)
    cancel = np.zeros((8, K), dtype=bool) if reg._cancel is None else reg._cancel.cpu().numpy().astype(bool)
    cancel[1::3] |= rng.random((len(cancel[1::3]), K)) < 0.03
    reg._cancel = torch.from_numpy(cancel.astype(np.uint8)).cuda()
    _check(reg, d, world, modes=("split",))
    _check(reg, d, world, shard="rows")


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("n_est", [1, 2])
def test_sharded_regression_rows_emulated_ragged(world, n_est):
    """800 train rows: 432 + 368 rows on 2 ranks, 240 + 240 + 240 + 80 on 4; 200 test rows."""
    d, y = _data("small_task", 0)
    reg = _regressor(d, y, "bf16", n_est)
    sh = _check(reg, d, world, shard="rows", modes=("rows",))
    assert (world - 1) * sh.seg_rows < len(d["X_train"]) < world * sh.seg_rows


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("n_est", [2, 8])
def test_classifier_estimators_emulated_equals_predict_proba(world, n_est):
    geom = Geometry(mgm_heads=2, cap_heads=4)
    d = make_dataset("pad_ufes_small", 0)
    clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=2, cap_heads=4, n_estimators=n_est,
                          model_path=(make_state_dict(geom, seed=1), geom), device="cuda", inference_precision="bf16",
                          ignore_pretraining_limits=True, random_state=0).fit(d["X_train"], d["img_train"], d["y_train"])
    ref = clf.predict_proba(d["X_test"], d["img_test"])
    sh = ShardedEngine(clf.executor_, 0, world, group="emulate")
    n = len(d["X_test"])
    rows = sh.test_rows(n)
    logits = sh.logits(transform_all(clf.members_, d["X_test"][rows]), d["img_test"][rows])
    p = sh.proba_gathered(logits, [m.class_perm for m in clf.members_], n_classes=clf.n_classes_,
                          softmax_temperature=clf.softmax_temperature)[:n].cpu().numpy()
    got = p / p.sum(axis=1, keepdims=True)
    assert sh.exchange["mode"] in ("split", "one_each", "broadcast")
    assert np.array_equal(got, ref), float(np.abs(got - ref).max())
