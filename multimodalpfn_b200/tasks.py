"""Many independent small tasks packed per launch (BASELINE.json configs[4], SURVEY.md section 8e).

The reference has a batch axis in the transformer (``x [S, B, F]``, state ``[B, S, T, E]``,
``layer.py:284-285``) but its engines always pass ``B = 1`` (``inference.py:305``) and the CAP stem
hard-codes it (``transformer.py:78-79``): 256 small datasets mean 256 x n_estimators sequential
forwards there.  Here the batch axis of every kernel carries *entries*, one per (task, estimator)
pair, and tasks of ANY sizes share launches:

* ``plan_passes`` splits the entries into passes.  A pass has the row capacity of its largest entry
  (train rows and test rows); the other entries' rows up to it are pad rows.  Entries are sorted by
  row count and a pass is closed before it would hold more than ``MAX_SEGMENTS`` distinct token
  counts T, more than ``token_budget`` tokens, or a padded share of its tokens above
  ``MAX_PAD_FRACTION``.  Tasks of equal shape pad nothing: their passes pass no count arrays.
* ``B200PerFeatureTransformer.forward_ragged`` runs one train pass and one test pass per pass
  (entries of equal T form one segment); the kernels keep every pad row exactly zero, so each
  entry's arithmetic is that of a forward over the entry alone (include/mmpfn_b200.h).
* The image stem runs once per embedding-token count over the rows of all its tasks.

Tasks are independent until the end, so a multi-GPU run just deals them out round-robin and gathers
the probabilities — no collective on the data path.

The result for every task is what ``MMPFNClassifier(n_estimators=..., random_state=...)`` returns
for that task alone (same members, same reference-equivalent joint forward); the packing only
changes which rows share a kernel launch.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np
import torch
from sklearn.preprocessing import LabelEncoder

from .engine import estimator_groups, proba_from_logits
from .model import B200PerFeatureTransformer
from .preprocessing import RECIPES, fit_transform_all, make_members, transform_all
from .regressor import bar_tail_tasks_device, check_borders, format_result, output_request, prepare_regression

__all__ = ["predict_proba_tasks", "predict_regression_tasks", "plan_passes", "shard_tasks", "gather_task_results"]

MAX_SEGMENTS = 8              # distinct token counts per pass (MMPFN_MAX_SEGMENTS)
MAX_PAD_FRACTION = 0.25       # padded tokens of a pass over all its tokens
TOKEN_BUDGET = 1 << 21        # train + test tokens per pass (~10 GB of state and bf16 workspace)


def plan_passes(shapes: Sequence[tuple], *, token_budget: int = TOKEN_BUDGET) -> list:
    """Split entries of shapes ``(n_train, n_test, T)`` into passes -> [[entry index]].

    A pass's tokens are ``(S_train + S_test) * sum T`` (its capacities times its entries' token counts).  Entries
    are taken in descending row count; an entry joins the open pass unless that pass would then hold more than
    ``MAX_SEGMENTS`` distinct T, more than ``token_budget`` tokens, or more than ``MAX_PAD_FRACTION`` of its tokens
    on pad rows; then it opens the next pass (alone, an entry pads nothing, whatever its size)."""
    order = sorted(range(len(shapes)), key=lambda i: (-shapes[i][0], -shapes[i][1], shapes[i][2], i))
    passes, cur = [], []
    S_tr = S_te = sum_T = useful = 0
    Ts = set()
    for i in order:
        n_tr, n_te, T = (int(v) for v in shapes[i])
        if cur:
            s_tr, s_te, s_T = max(S_tr, n_tr), max(S_te, n_te), sum_T + T
            tokens = (s_tr + s_te) * s_T
            if (len(Ts | {T}) <= MAX_SEGMENTS and tokens <= token_budget
                    and tokens - (useful + (n_tr + n_te) * T) <= MAX_PAD_FRACTION * tokens):
                cur.append(i)
                S_tr, S_te, sum_T = s_tr, s_te, s_T
                useful += (n_tr + n_te) * T
                Ts.add(T)
                continue
            passes.append(cur)
        cur = [i]
        S_tr, S_te, sum_T, useful, Ts = n_tr, n_te, T, (n_tr + n_te) * T, {T}
    if cur:
        passes.append(cur)
    return passes


def shard_tasks(n_tasks: int, rank: int, world: int) -> list:
    """Indices of the tasks rank ``rank`` owns (round-robin)."""
    return list(range(rank, n_tasks, world))


def gather_task_results(local: dict, n_tasks: int) -> list:
    """All-gather ``{task index: proba}`` dictionaries over the default process group -> list in task order."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return [local.get(i) for i in range(n_tasks)]
    parts = [None] * dist.get_world_size()
    dist.all_gather_object(parts, local)
    merged = {}
    for p in parts:
        merged.update(p)
    return [merged.get(i) for i in range(n_tasks)]


def _prepare(task: dict, n_estimators: int, random_state, recipes):
    X = None if task.get("X_train") is None else np.asarray(task["X_train"], dtype=np.float32)
    Xte = None if task.get("X_test") is None else np.asarray(task["X_test"], dtype=np.float32)
    y = np.asarray(task["y_train"])
    enc = LabelEncoder()
    yi = enc.fit_transform(y)
    n_cls = len(enc.classes_)
    _, counts = np.unique(y, return_counts=True)
    rng = np.random.default_rng(random_state if isinstance(random_state, (int, np.integer)) else None)
    members = make_members(n_estimators, 0 if X is None else X.shape[1], n_cls, rng, recipes=tuple(recipes))
    train = fit_transform_all(members, X, yi)
    test = transform_all(members, Xte)

    itr, ite = _images(task)
    n_te = len(Xte) if Xte is not None else len(ite)
    return dict(members=members, train=train, test=test, img_train=itr, img_test=ite, n_classes=n_cls, counts=counts,
                classes=enc.classes_, n_train=len(y), n_test=n_te)


def _prepare_all(indices, prepare, n_jobs):
    import os
    from concurrent.futures import ThreadPoolExecutor
    workers = (os.cpu_count() or 1) if n_jobs in (-1, None) else max(1, int(n_jobs))
    workers = min(workers, max(1, len(indices)))
    if workers > 1:
        with ThreadPoolExecutor(workers) as pool:
            return dict(zip(indices, pool.map(prepare, indices)))
    return {i: prepare(i) for i in indices}


def _task_logits(model: B200PerFeatureTransformer, prepared: dict, indices, n_estimators: int, y_means=None) -> dict:
    """The device part shared by the task functions: one image-stem pass per embedding-token count, the planned
    ragged passes -> ``{task index: [logits [n_test, n_out] per estimator]}`` (views into the passes' decoder
    outputs).  ``y_means``: ``{task index: [label mean per estimator]}`` (one-element device tensors) or None."""
    dev = model.device
    # one image-stem pass per embedding-token count over the rows of all its tasks
    tok_of = {}
    by_ntok = {}
    for i in indices:
        if prepared[i]["img_train"] is not None:
            by_ntok.setdefault(prepared[i]["img_train"].shape[1], []).append(i)
    for n_tok, idx in by_ntok.items():
        img_all = np.concatenate([np.concatenate([prepared[i]["img_train"], prepared[i]["img_test"]]) for i in idx])
        tok = model.stem_image(torch.from_numpy(img_all).to(dev))
        row = 0
        for i in idx:
            tok_of[i] = (tok, row, n_tok)
            row += prepared[i]["n_train"] + prepared[i]["n_test"]
    entries, owner = [], []
    for i in indices:
        pr = prepared[i]
        tok, row, n_tok = tok_of.get(i, (None, 0, 0))
        for e in range(n_estimators):
            X = pr["train"][e][0]
            # the stem statistics see train and test rows (the reference's joint forward, encoders.py:515, :615)
            X_all = None if X is None else np.concatenate([X, pr["test"][e]]).astype(np.float32, copy=False)
            entries.append(dict(X=X_all, y=pr["train"][e][1], n_train=pr["n_train"], n_test=pr["n_test"], tok=tok,
                                tok_row=row, n_tok=n_tok, y_mean=None if y_means is None else y_means[i][e]))
            owner.append((i, e))
    shapes = [(en["n_train"], en["n_test"],
               model.entry_tokens(None if en["X"] is None else en["X"].shape[1], en["n_tok"])) for en in entries]
    logits = {i: [None] * n_estimators for i in indices}
    for ps in plan_passes(shapes):
        for k, lg in zip(ps, model.forward_ragged([entries[k] for k in ps])):
            i, e = owner[k]
            logits[i][e] = lg
    return logits


def predict_proba_tasks(model: B200PerFeatureTransformer, tasks: Sequence[dict], *, n_estimators: int = 4,
                        random_state=0, softmax_temperature: float = 0.9, average_before_softmax: bool = False,
                        balance_probabilities: bool = False, recipes=RECIPES, indices: Optional[Sequence[int]] = None,
                        n_jobs: int = 1, timings: Optional[dict] = None):
    """``tasks``: dicts with ``X_train, img_train, y_train, X_test, img_test`` (tables or embeddings may be
    ``None`` like in ``MMPFNClassifier.fit``).  Returns ``{task index: float32 [Nte, n_classes]}`` for the
    tasks in ``indices`` (default: all).  Tasks of any shapes share launches (``plan_passes``).  The per-task host work
    (fitting the members' quantile / SVD transforms) can run in ``n_jobs`` threads (it is mostly GIL-bound
    sklearn glue: 16 threads measured slower than 1); ``timings`` (a dict) receives
    the seconds spent in ``host_prepare`` and ``device``."""
    import time
    indices = list(range(len(tasks))) if indices is None else list(indices)
    dev = model.device
    t0 = time.perf_counter()
    prepared = _prepare_all(indices, lambda i: _prepare(tasks[i], n_estimators, random_state, recipes), n_jobs)
    t1 = time.perf_counter()
    logits = _task_logits(model, prepared, indices, n_estimators)
    out = {}
    for i in indices:
        pr = prepared[i]
        out[i] = proba_from_logits(torch.stack(logits[i]), [m.class_perm for m in pr["members"]],
                                   n_classes=pr["n_classes"], class_counts=pr["counts"],
                                   softmax_temperature=softmax_temperature,
                                   average_before_softmax=average_before_softmax,
                                   balance_probabilities=balance_probabilities)
    if timings is not None:
        torch.cuda.synchronize(dev)
        timings["host_prepare"] = t1 - t0
        timings["device"] = time.perf_counter() - t1
    return out


def _images(task: dict):
    def img(a):
        if a is None:
            return None
        a = np.asarray(a, dtype=np.float32)
        return a[:, None] if a.ndim == 2 else a
    return img(task.get("img_train")), img(task.get("img_test"))


def _prepare_regression_task(i: int, task: dict, g: np.ndarray, n_estimators: int, random_state) -> dict:
    """``MMPFNRegressor.fit``'s host work for task ``i`` (``prepare_regression``) plus its test tables."""
    X = None if task.get("X_train") is None else np.asarray(task["X_train"], dtype=np.float32)
    Xte = None if task.get("X_test") is None else np.asarray(task["X_test"], dtype=np.float32)
    itr, ite = _images(task)
    if X is None and itr is None:
        raise ValueError(f"task {i}: needs a table X_train, an embedding img_train, or both")
    try:
        prep = prepare_regression(X, task["y_train"], g, n_estimators=n_estimators, random_state=random_state)
    except ValueError as exc:
        raise ValueError(f"task {i}: {exc}") from exc
    n_te = len(Xte) if Xte is not None else len(ite)
    prep.update(train=[(t["X_train"], t["y_train"]) for t in prep["tables"]], test=transform_all(prep["members"], Xte),
                img_train=itr, img_test=ite, n_train=len(prep["tables"][0]["y_train"]), n_test=n_te)
    return prep


def predict_regression_tasks(model: B200PerFeatureTransformer, borders, tasks: Sequence[dict], *,
                             n_estimators: int = 4, random_state=0, softmax_temperature: float = 0.9,
                             average_before_softmax: bool = False, output_type: str = "mean", quantiles=None,
                             indices: Optional[Sequence[int]] = None, n_jobs: int = 1,
                             timings: Optional[dict] = None) -> dict:
    """Many regression tasks in shared passes and ONE bar-distribution tail launch.

    ``model``: a regression checkpoint's ``B200PerFeatureTransformer``; ``borders``: that checkpoint's
    ``criterion.borders`` (``weights.load_borders``; the model does not hold them).  ``tasks``: the dicts of
    ``predict_proba_tasks`` with float ``y_train``.  Returns ``{task index: result}`` for the tasks in ``indices``
    (default: all), each exactly what ``MMPFNRegressor(n_estimators=..., random_state=...).fit(...).predict(...,
    output_type=..., quantiles=...)`` returns for that task alone when the regressor's model is built like ``model``
    (its seed ``int(random_state)``, ``outlier_std`` 12): arrays, a list of quantile arrays, or the "main" / "full"
    dicts with the task's own log P and borders G.

    Each task's host work (``prepare_regression``: target checks, transforms, members, border maps) runs in
    ``n_jobs`` threads.  The label mean of each entry is taken over the estimator groups the regressor's engine
    forms (``estimator_groups``), so the target token matches in every bit.  Every pass's logits stay on the device
    until the tail: sum over tasks of n_estimators * n_test * K * 4 bytes (about 1 GB for 32 tasks x 8 estimators x
    200 test rows x 5000 buckets).  ``timings`` (a dict) receives the seconds of ``host_prepare``, ``device`` (to
    the host copies inclusive) and ``tail`` (the tail launch alone, CUDA events)."""
    import time
    if not getattr(model.w, "regression", False):
        raise ValueError("model holds a classification checkpoint; use predict_proba_tasks")
    g = check_borders(borders, model.geom.n_out)
    K = len(g) - 1
    if K > 8192:
        raise ValueError(f"{K} buckets: the bar-distribution tail supports at most 8192")
    want, qs = output_request(output_type, quantiles)
    indices = list(range(len(tasks))) if indices is None else list(indices)
    dev = model.device
    t0 = time.perf_counter()
    prepared = _prepare_all(indices, lambda i: _prepare_regression_task(i, tasks[i], g, n_estimators, random_state),
                            n_jobs)
    t1 = time.perf_counter()
    y_means = {}
    for i in indices:
        tables = prepared[i]["tables"]
        y_means[i] = [None] * n_estimators
        for _, idx in estimator_groups(tables):
            ytr = torch.from_numpy(np.stack([np.asarray(tables[e]["y_train"], dtype=np.float32) for e in idx])).to(dev)
            y_mean, _ = model.label_stats(ytr)
            for k, e in enumerate(idx):
                y_means[i][e] = y_mean[k:k + 1]
    logits = _task_logits(model, prepared, indices, n_estimators, y_means)
    to_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)       # noqa: E731
    cancel = np.stack([prepared[i]["cancel"] for i in indices])
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)] if timings is not None else None
    args = (to_dev(np.stack([prepared[i]["src_bucket"] for i in indices])),
            to_dev(np.stack([prepared[i]["src_share"] for i in indices])),
            to_dev(cancel.astype(np.uint8)) if cancel.any() else None,
            to_dev(np.stack([prepared[i]["target_borders"] for i in indices]).astype(np.float32)))
    q_dev = to_dev(qs.astype(np.float32)) if "quantiles" in want else None
    if ev is not None:
        ev[0].record()
    out = bar_tail_tasks_device([logits[i] for i in indices], *args, softmax_temperature=softmax_temperature,
                                average_before_softmax=average_before_softmax, quantiles=q_dev, outputs=want)
    if ev is not None:
        ev[1].record()
    ro = out.pop("row_offset")
    host = {k: v.cpu().numpy() for k, v in out.items()}
    res = {}
    for n, i in enumerate(indices):
        r0, r1 = int(ro[n]), int(ro[n + 1])
        part = {k: np.array(v[..., r0:r1] if k == "quantiles" else v[r0:r1]) for k, v in host.items()}
        res[i] = format_result(part, output_type, prepared[i]["target_borders"])
    if timings is not None:
        torch.cuda.synchronize(dev)
        timings["host_prepare"] = t1 - t0
        timings["device"] = time.perf_counter() - t1
        timings["tail"] = ev[0].elapsed_time(ev[1]) / 1e3
    return res
