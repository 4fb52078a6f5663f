"""Shared builders for the golden cases: regenerate the seeded inputs/weights a fixture was
made from (``oracle/make_golden.py``) without touching the reference."""
import os

import numpy as np
import torch

from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
from oracle.make_golden import CLF_CASES, MODEL_CASES, case_state_dict, case_targets, mutate_inputs

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    if "X_cols" in g:                                   # tables stored by pack_tables
        cols = g.pop("X_cols")
        for k in [k for k in g if k.startswith("X_col_index_")]:
            g["X_full_" + k[len("X_col_index_"):]] = cols[:, g.pop(k)]
    return g


def pack_tables(out):
    """Replaces the ``X_full_<e>`` tables of a golden dict by the pool of their distinct columns (``X_cols``) and one
    column index per table (``X_col_index_<e>``): the estimators' tables share most of their columns, and stored
    whole the 8-estimator PAD-UFES tables take more than 1 MB.  ``load_golden`` restores them bit for bit."""
    pool, where = [], {}
    for k in [k for k in out if k.startswith("X_full_")]:
        X = out.pop(k)
        idx = []
        for j in range(X.shape[1]):
            key = X[:, j].tobytes()
            if key not in where:
                where[key] = len(pool)
                pool.append(X[:, j])
            idx.append(where[key])
        out["X_col_index_" + k[len("X_full_"):]] = np.asarray(idx, np.int16)
    out["X_cols"] = np.stack(pool, 1)
    return out


def model_case(name):
    """-> geom, state_dict(np), X_full(np|None), img_full(np|None), y_train(np f32), n_train"""
    gkw, ds, wseed, mut = MODEL_CASES[name]
    geom = Geometry(**{k: v for k, v in gkw.items() if v is not None or k == "cap_heads"})
    sd, _ = case_state_dict(geom, wseed, mut)
    sd = {k: v for k, v in sd.items() if not k.startswith("criterion.")}      # (bar-distribution borders: host side)
    d = make_dataset(ds, 0)
    X = np.concatenate([d["X_train"], d["X_test"]])
    img = np.concatenate([d["img_train"], d["img_test"]])
    X, img = mutate_inputs(mut, X, img)
    y = case_targets(mut, d, X)
    return geom, sd, X, img, y, len(y)


def clf_case(name):
    ds, n_est, kw = CLF_CASES[name]
    geom = Geometry(mgm_heads=2, cap_heads=4)
    sd = make_state_dict(geom, seed=11)
    d = make_dataset(ds, 0)
    return geom, sd, d, n_est, kw


def t(x):
    return None if x is None else torch.as_tensor(x)


# ---- large-config cases (oracle/make_golden_large.py) ---------------------------------------------------
CTX10K_GEOM = Geometry(mgm_heads=8, cap_heads=8)
CTX10K_WSEED = 1
CTX10K_N_TEST = 256
CTX10K_KV_ROWS = np.arange(0, 10_000, 625)          # 16 train rows whose cached K/V are kept


def ctx10k_inputs():
    """BASELINE configs[2] shape (10 000 train rows, 64 features, [N,2,768] image+text embeddings) for ONE
    estimator: a 65th uniform column stands where the reference's fingerprint feature would
    (model/preprocessing.py:476-523) so that F'=65 -> T=42 (SURVEY.md section 8(d)); 256 seeded test rows."""
    d = make_dataset("img_text_10k", 0)
    rng = np.random.default_rng(42)
    pick = np.sort(rng.choice(len(d["y_test"]), CTX10K_N_TEST, replace=False))
    fp_tr = rng.random((len(d["y_train"]), 1), dtype=np.float32)
    fp_te = rng.random((len(d["y_test"]), 1), dtype=np.float32)
    return dict(X_train=np.concatenate([d["X_train"], fp_tr], 1), img_train=d["img_train"],
                y_train=d["y_train"].astype(np.float32),
                X_test=np.concatenate([d["X_test"], fp_te], 1)[pick], img_test=d["img_test"][pick],
                X_test_all=np.concatenate([d["X_test"], fp_te], 1), img_test_all=d["img_test"], pick=pick,
                n_classes=d["n_classes"])


LAYER50K_GEOM = Geometry(mgm_heads=2, cap_heads=4, nlayers=1)
LAYER50K_WSEED = 3
LAYER50K_SSEED = 9
# g1: the reference's own initialisation law (near-uniform softmax over the 50 000 keys); g3: qkv weights x3, i.e.
# scores x9 (spread over tens of log2 units: a sharp softmax, the running reference of the bf16 kernel moves)
LAYER50K_GAINS = {"g1": 1.0, "g3": 3.0}
LAYER50K_SHAPE = (50_000, 128, 3)                   # train rows, test rows, tokens
LAYER50K_ROWS = np.concatenate([np.arange(0, 50_000, 50_000 // 64)[:64], 50_000 + np.arange(0, 128, 2)])


def layer_state(S, T, seed):
    """A LayerNorm-scaled token state [S, T, 192] (what a layer sees between sublayers)."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((S, T, 192)).astype(np.float32)
    x -= x.mean(-1, keepdims=True)
    x /= x.std(-1, keepdims=True)
    return x


def softmax_np(z):
    z = z - z.max(-1, keepdims=True)
    e = np.exp(z)
    return e / e.sum(-1, keepdims=True)


def check_proba(p, pr, tol, what):
    """BASELINE.json north_star gate: max |dp| <= tol, and argmax agreement reported in full — every
    disagreeing row must be one the tolerance cannot decide (reference top-2 margin below twice the
    measured deviation).  Returns (max |dp|, agreement)."""
    dp = float(np.abs(p - pr).max())
    flips = np.nonzero(p.argmax(-1) != pr.argmax(-1))[0]
    srt = np.sort(pr, -1)
    margin = srt[..., -1] - srt[..., -2]
    agree = 1.0 - len(flips) / p.shape[0]
    print(f"[{what}] max|dp| {dp:.3e} (tol {tol:g}); argmax agreement {agree:.4%}; "
          f"undecided rows (reference margin): {[(int(i), float(margin[i])) for i in flips[:8]]}")
    assert dp <= tol, (what, dp)
    assert all(margin[i] <= 2 * dp for i in flips), (what, [(int(i), float(margin[i])) for i in flips])
    return dp, agree
