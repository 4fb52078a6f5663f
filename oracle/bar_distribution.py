"""ORACLE (test infrastructure): float64 numpy restatement of the regressor's bar-distribution tail.

Steps 1-6 of ``mmpfn_bar_tail`` (include/mmpfn_b200.h) and the border-map construction of
``multimodalpfn_b200/regressor.py``, written independently of both, loop-free over rows.  The product package never
imports this module.
"""
from __future__ import annotations

import numpy as np
from scipy.special import erfinv

SQRT2 = np.sqrt(2.0)
SQRT_2_OVER_PI = np.sqrt(2.0 / np.pi)


def border_map(f, g):
    """(src_bucket int64 [K+1], src_share float64 [K+1]) of the common borders g within the borders f."""
    f = np.asarray(f, dtype=np.float64)
    g = np.asarray(g, dtype=np.float64)
    K = len(f) - 1
    bucket = np.empty(len(g), dtype=np.int64)
    share = np.zeros(len(g))
    for j, gj in enumerate(g):
        if gj < f[0]:
            bucket[j] = -1
        elif gj >= f[K]:
            bucket[j] = K
        else:
            i = int(np.nonzero(f <= gj)[0].max())       # f[i] <= g_j < f[i+1]
            bucket[j] = i
            share[j] = min(max((gj - f[i]) / (f[i + 1] - f[i]), 0.0), 1.0)
    return bucket, share


def member_borders(f):
    """Estimator borders as mapped back (may hold non-finite values) -> (borders with every non-finite value
    replaced by the nearest finite one, cancel [K] bool: buckets of zero or non-finite width)."""
    f = np.asarray(f, dtype=np.float64)
    ok = np.isfinite(f)
    idx = np.nonzero(ok)[0]
    out = f.copy()
    for k in np.nonzero(~ok)[0]:
        out[k] = f[idx[np.argmin(np.abs(idx - k))]]
    w = f[1:] - f[:-1]
    cancel = ~np.isfinite(w) | (out[1:] - out[:-1] <= 0)
    return out, cancel


def translate(logits, bucket, share, cancel=None, temperature=1.0):
    """Steps 1-2 for one estimator: logits [S, K] -> q [S, K] on the common borders."""
    z = np.asarray(logits, dtype=np.float64)
    if temperature != 1:
        z = z / temperature
    if cancel is not None:
        z = np.where(np.asarray(cancel, dtype=bool)[None], -np.inf, z)
    z = z - z.max(axis=1, keepdims=True)
    p = np.exp(z)
    p /= p.sum(axis=1, keepdims=True)
    S, K = p.shape
    pre = np.concatenate([np.zeros((S, 1)), np.cumsum(p, axis=1)], axis=1)      # P(i), i = 0..K
    C = np.empty((S, K + 1))
    for j in range(K + 1):
        i = bucket[j]
        if i < 0:
            C[:, j] = 0.0
        elif i >= K:
            C[:, j] = 1.0
        else:
            C[:, j] = pre[:, i] + p[:, i] * share[j]
    C[:, 0] = 0.0
    C[:, K] = 1.0
    return np.maximum(C[:, 1:] - C[:, :-1], 0.0)


def combine(qs, average_before_softmax=False):
    """Step 3: [n_est] x [S, K] -> P [S, K]."""
    qs = np.stack(qs)
    if not average_before_softmax:
        return qs.mean(axis=0)
    with np.errstate(divide="ignore"):
        lq = np.log(qs).mean(axis=0)
    lq = lq - lq.max(axis=1, keepdims=True)
    e = np.exp(lq)
    return e / e.sum(axis=1, keepdims=True)


def bucket_means(G):
    G = np.asarray(G, dtype=np.float64)
    w = np.diff(G)
    m = 0.5 * (G[:-1] + G[1:])
    m[0] = G[1] - w[0] * SQRT_2_OVER_PI
    m[-1] = G[-2] + w[-1] * SQRT_2_OVER_PI
    return m


def mean(P, G):
    return P @ bucket_means(G)


def quantile(P, G, q):
    """Step 5 at one level q in (0, 1) -> [S]."""
    G = np.asarray(G, dtype=np.float64)
    S, K = P.shape
    w = np.diff(G)
    c = np.cumsum(P, axis=1)
    j = np.minimum((c < q).sum(axis=1), K - 1)           # first index with c_j >= q
    rows = np.arange(S)
    prev = np.where(j > 0, c[rows, np.maximum(j - 1, 0)], 0.0)
    pj = P[rows, j]
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(pj > 0, (q - prev) / pj, 1.0)
    r = np.clip(r, 0.0, 1.0)
    out = G[j] + r * w[j]
    out = np.where(j == 0, G[1] - w[0] * SQRT2 * erfinv(1.0 - r), out)
    out = np.where(j == K - 1, G[K - 1] + w[K - 1] * SQRT2 * erfinv(r), out)
    return out


def mode(P, G):
    G = np.asarray(G, dtype=np.float64)
    j = np.argmax(P / np.diff(G)[None], axis=1)           # first maximum: ties go to the lowest j
    return 0.5 * (G[j] + G[j + 1])


def bar_tail(logits, buckets, shares, cancels, G, *, temperature=1.0, average_before_softmax=False,
             quantiles=()):
    """The whole tail: logits [n_est, S, K] -> dict(log_prob, mean, median, mode, quantiles [n_q, S])."""
    qs = [translate(logits[e], buckets[e], shares[e], None if cancels is None else cancels[e], temperature)
          for e in range(len(logits))]
    P = combine(qs, average_before_softmax)
    with np.errstate(divide="ignore"):
        lp = np.log(P)
    # average_before_softmax: a bucket where some estimator's mass is within float64 rounding of zero (a difference
    # of two CDF values near 1) has a geometric mean set by that rounding; "conditioned" marks the other buckets
    conditioned = np.min(np.stack(qs), axis=0) >= 1e-12 if average_before_softmax else np.ones(P.shape, dtype=bool)
    return dict(P=P, log_prob=lp, conditioned=conditioned, mean=mean(P, G), median=quantile(P, G, 0.5), mode=mode(P, G),
                quantiles=np.stack([quantile(P, G, q) for q in quantiles]) if len(quantiles) else np.zeros((0, len(P))))
