"""The pass planner of the many-tasks path (multimodalpfn_b200/tasks.py): which (task, estimator) entries share a
pass.  Host logic only."""
import numpy as np

from multimodalpfn_b200.model import entry_counts
from multimodalpfn_b200.tasks import MAX_PAD_FRACTION, MAX_SEGMENTS, TOKEN_BUDGET, plan_passes


def _mixed(seed=0, n_tasks=64, n_est=8):
    rng = np.random.default_rng(seed)
    shapes = []
    for _ in range(n_tasks):
        n_tr, n_te, T = int(rng.integers(100, 2001)), int(rng.integers(20, 401)), int(rng.integers(4, 40))
        shapes += [(n_tr, n_te, T + int(rng.integers(0, 2))) for _ in range(n_est)]
    return shapes


def _check(shapes, passes, budget=TOKEN_BUDGET):
    seen = sorted(i for p in passes for i in p)
    assert seen == list(range(len(shapes)))                       # every entry in exactly one pass
    for p in passes:
        Ts = {shapes[i][2] for i in p}
        assert len(Ts) <= MAX_SEGMENTS
        S_tr, S_te = max(shapes[i][0] for i in p), max(shapes[i][1] for i in p)
        tokens = sum((S_tr + S_te) * shapes[i][2] for i in p)
        useful = sum((shapes[i][0] + shapes[i][1]) * shapes[i][2] for i in p)
        assert tokens - useful <= MAX_PAD_FRACTION * tokens
        assert tokens <= budget or len(p) == 1


def test_mixed_entries():
    shapes = _mixed()
    passes = plan_passes(shapes)
    _check(shapes, passes)
    assert len(passes) < len(shapes) // 4                         # it does pack


def test_small_budget_holds():
    shapes = _mixed(1, n_tasks=16)
    passes = plan_passes(shapes, token_budget=200_000)
    _check(shapes, passes, budget=200_000)
    one = plan_passes([(50_000, 10_000, 30)])                     # larger than the budget alone: its own pass
    assert one == [[0]]


def test_equal_tasks_pad_nothing():
    shapes = [(800, 200, 26)] * 256
    passes = plan_passes(shapes)
    _check(shapes, passes)
    for p in passes:
        n_tr = [shapes[i][0] for i in p]
        n_te = [shapes[i][1] for i in p]
        assert entry_counts(n_tr, max(n_tr)) is None and entry_counts(n_te, max(n_te)) is None
    assert entry_counts([5, 4], 5).tolist() == [5, 4]


def test_many_token_counts_need_several_passes():
    shapes = [(100, 10, T) for T in range(3, 3 + 2 * MAX_SEGMENTS + 1)]
    passes = plan_passes(shapes)
    _check(shapes, passes)
    assert len(passes) >= 3
