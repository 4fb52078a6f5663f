"""world-2 / -4 gloo tests (CPU) of regression on the multi-GPU engine (multimodalpfn_b200/dist.py):
``MMPFNRegressor.predict(..., sharded=ShardedEngine)`` in all three estimator-ownership modes and in the row-sharded
mode returns what the unsharded ``predict`` returns, in test-row order, with unequal test chunks; only the requested
outputs are all-gathered, ``log_prob`` only for "full".  The model is the arithmetic stand-in of test_dist_gloo.py with
a decoder whose bucket logits depend on the row, and the bar tail is the float64 oracle (oracle/bar_distribution.py),
so only the plumbing is tested; tests/test_gpu_dist_regression.py checks the kernels on a B200."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from multimodalpfn_b200 import dist as D
from multimodalpfn_b200 import regressor as R
from multimodalpfn_b200.dist import ShardedEngine
from multimodalpfn_b200.engine import B200InferenceEngine
from oracle import bar_distribution as O
from tests.test_dist_gloo import FakeModel, _make_engine

K = 24
N_FEATURES = 5


class FakeRegressionModel(FakeModel):
    """The stand-in with K bucket logits per row: a bump whose centre follows the row's final state."""

    def decode(self, state):
        centre = torch.tanh(state[:, :, -1, :1] * 0.05 + state.mean((2, 3))[..., None] * 0.01) * 2.5
        return -2.0 * (torch.linspace(-3.0, 3.0, K)[None, None] - centre) ** 2


def fake_bar_tail(logits, src_bucket, src_share, cancel, borders, *, softmax_temperature, average_before_softmax,
                  quantiles=None, outputs=("mean",)):
    """``regressor.bar_tail_device`` on the CPU, through the float64 oracle; same arguments and result layout."""
    qs = () if quantiles is None else [float(q) for q in quantiles]
    ref = O.bar_tail(logits.double().numpy(), src_bucket.numpy(), src_share.double().numpy(),
                     None if cancel is None else cancel.numpy().astype(bool), borders.double().numpy(),
                     temperature=softmax_temperature, average_before_softmax=average_before_softmax, quantiles=qs)
    return {k: torch.from_numpy(np.ascontiguousarray(ref[k], dtype=np.float32)) for k in outputs}


def _make_regressor(n_est, n_train, n_test=7):
    rng = np.random.default_rng(0)
    X = rng.standard_normal((n_train + n_test, N_FEATURES)).astype(np.float32)
    img = rng.standard_normal((n_train + n_test, 1, 8)).astype(np.float32)
    y = X @ rng.normal(0, 1, N_FEATURES) + rng.normal(0, 0.1, n_train + n_test)
    prep = R.prepare_regression(X[:n_train], y[:n_train], np.linspace(-3, 3, K + 1), n_estimators=n_est)
    reg = R.MMPFNRegressor(n_estimators=n_est)
    reg.n_features_in_ = N_FEATURES
    reg.members_ = prep["members"]
    reg.target_borders_ = prep["target_borders"]
    reg.model_ = FakeRegressionModel()
    reg._src_bucket = torch.from_numpy(prep["src_bucket"])
    reg._src_share = torch.from_numpy(prep["src_share"])
    cancel = prep["cancel"].copy()
    cancel[:, 3] = True                                       # a cancelled bucket, so the cancel mask travels too
    reg._cancel = torch.from_numpy(cancel.astype(np.uint8))
    reg._borders_dev = torch.from_numpy(reg.target_borders_.astype(np.float32))
    reg.executor_ = B200InferenceEngine(reg.model_, prep["tables"], img[:n_train])
    eng = reg.executor_
    # the unsharded predict replays a CUDA graph by default; the stand-in runs on the CPU
    eng.logits = lambda X_tests, image_test: B200InferenceEngine.logits(eng, X_tests, image_test, graph=False)
    return reg, X[n_train:], img[n_train:]


OUTPUT_TYPES = ("main", "full", "mean", "quantiles")


def _compare(got, ref, output_type):
    """-> max |got - ref| over every array of a ``predict`` result (same structure required)."""
    if isinstance(ref, dict):
        assert set(got) == set(ref), (sorted(got), sorted(ref))
        return max(_compare(got[k], ref[k], output_type) for k in ref)
    if isinstance(ref, list):
        assert len(got) == len(ref)
        return max(_compare(a, b, output_type) for a, b in zip(got, ref))
    assert got.shape == ref.shape and got.dtype == ref.dtype, (got.shape, ref.shape)
    return float(np.abs(np.where(got == ref, 0.0, got - ref)).max())          # (cancelled buckets: -inf on both)


def _check_predict(reg, X, img, sh, tol):
    """Sharded vs unsharded ``predict`` for every output type, and the all-gathers the sharded call made."""
    world = sh.world
    n = len(X)
    rows = n if sh.emulate else -(-n // world)
    ref_mean = reg.predict(X, img, output_type="mean")
    assert len(np.unique(ref_mean)) == n                      # distinct rows: a misplaced row cannot go unseen
    calls = []
    real_gather = D.all_gather_rows
    D.all_gather_rows = lambda x, group=None: calls.append(tuple(x.shape)) or real_gather(x, group)
    try:
        for output_type in OUTPUT_TYPES:
            ref = reg.predict(X, img, output_type=output_type)
            del calls[:]
            got = reg.predict(X, img, output_type=output_type, sharded=sh)
            err = _compare(got, ref, output_type)
            assert err <= tol, (output_type, err)
            width = {"main": 3 + 9, "full": 3 + 9, "mean": 1, "quantiles": 9}[output_type]     # 9 default quantiles
            expect = [] if sh.emulate else [(rows, width)] + ([(rows, K)] if output_type == "full" else [])
            assert calls == expect, (output_type, calls, expect)
    finally:
        D.all_gather_rows = real_gather


def _worker(rank, world, port, q, n_est, shard, n_train):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    R.bar_tail_device = fake_bar_tail
    try:
        reg, X, img = _make_regressor(n_est, n_train)
        sh = ShardedEngine(reg.executor_, rank, world, shard=shard)
        try:
            _check_predict(reg, X, img, sh, tol=2e-3)
            q.put((rank, "ok", sh.exchange["mode"]))
        except AssertionError as e:
            q.put((rank, f"failed: {e!r}", sh.exchange and sh.exchange["mode"]))
    finally:
        dist.destroy_process_group()


def _run(world, n_est, shard="estimators", n_train=40):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, n_est, shard, n_train)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=240) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


@pytest.mark.parametrize("world,n_est,shard,n_train,mode", [
    (2, 4, "estimators", 40, "split"),          # groups of 2 + 2 estimators: one of each group per rank
    (4, 4, "estimators", 40, "one_each"),       # 2 + 2 estimators on 4 ranks
    (2, 3, "estimators", 40, "broadcast"),      # 1 + 2 estimators on 2 ranks
    (2, 3, "rows", 100, "rows"),                # 96 + 4 train rows
    (4, 1, "rows", 190, "rows"),                # 48 + 48 + 48 + 46 train rows of one estimator
])
def test_sharded_regression_gloo(world, n_est, shard, n_train, mode):
    """7 test rows: chunks of 4 + 3 rows on 2 ranks, 2 + 2 + 2 + 1 on 4 (the short chunks are padded)."""
    res = _run(world, n_est, shard, n_train)
    assert all(r[1] == "ok" for r in res), res
    assert all(r[2] == mode for r in res), res


@pytest.mark.parametrize("world,n_est,shard,n_train,mode", [
    (2, 4, "estimators", 40, "split"),
    (4, 8, "estimators", 40, "split"),
    (2, 2, "estimators", 40, "one_each"),
    (4, 4, "estimators", 40, "one_each"),
    (3, 4, "estimators", 40, "broadcast"),
    (3, 2, "rows", 200, "rows"),
])
def test_sharded_regression_emulated_in_process(world, n_est, shard, n_train, mode, monkeypatch):
    """All ranks in this process (``group="emulate"``): their builds in turn, then the chunks of all ranks; the
    gathers move nothing."""
    monkeypatch.setattr(R, "bar_tail_device", fake_bar_tail)
    reg, X, img = _make_regressor(n_est, n_train)
    sh = ShardedEngine(reg.executor_, 0, world, group="emulate", shard=shard)
    _check_predict(reg, X, img, sh, tol=2e-3)
    assert sh.exchange["mode"] == mode


@pytest.mark.parametrize("world,n_a,n_b,mode", [
    (2, 4, 4, "split"), (4, 4, 4, "split"), (2, 2, 2, "split"), (4, 2, 2, "one_each"), (2, 1, 1, "one_each"),
    (2, 3, 2, "broadcast"), (4, 3, 2, "broadcast"),
])
def test_estimator_modes_emulated_logits(world, n_a, n_b, mode):
    """The estimator-ownership emulation on the classifier's stand-in engine: the same logits as unsharded."""
    eng, X_tests, img_test = _make_engine(0, n_a, n_b)
    ref = eng.logits(X_tests, img_test, graph=False)
    sh = ShardedEngine(eng, 0, world, group="emulate")
    got = sh.logits(X_tests, img_test)
    assert sh.exchange["mode"] == mode
    assert torch.allclose(got, ref, rtol=0, atol=1e-4), float((got - ref).abs().max())


def test_test_rows_chunking():
    eng, _, _ = _make_engine(0, 1, 0)
    for n in (1, 2, 5, 7, 8, 13):
        for world in (1, 2, 3, 4, 8):
            c = -(-n // world)
            parts = [ShardedEngine(eng, r, world).test_rows(n) for r in range(world)]
            assert all(len(p) == c for p in parts)
            whole = np.concatenate(parts)
            assert np.array_equal(whole[:n], np.arange(n))
            assert np.all(whole[n:] == n - 1)                   # padding repeats the last row
            assert np.array_equal(ShardedEngine(eng, 0, world, group="emulate").test_rows(n), whole)
    with pytest.raises(ValueError, match="no test rows"):
        ShardedEngine(eng, 0, 2).test_rows(0)
