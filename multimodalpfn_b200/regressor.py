"""``MMPFNRegressor`` — the reference regressor's estimator surface on top of the sm_100a path: the classifier's
constructor keywords (``classifier.py`` here) plus ``fit(X, image, y)`` and
``predict(X, image_test, *, output_type="mean", quantiles=None)``.

The regression checkpoint's decoder emits logits over K buckets of a bar distribution whose borders g (the
checkpoint's ``criterion.borders``) live on the standardised target y_z = (y - mean) / std.  Each ensemble member
sees its own transform T_e of y_z (none, or a Yeo-Johnson power transform: the structure of TabPFN-v2's
``(None, "safepower")``), so its buckets are f_e = T_e^-1(g) on the y_z axis.  ``fit`` computes, once, where every
common border g_j falls within f_e (``border_map``); ``predict`` runs the forward and then ``mmpfn_bar_tail``
(include/mmpfn_b200.h, where the tail's semantics are stated), which translates every member onto g, combines the
members and reduces each test row to the requested outputs on the device, over the borders G = g * std + mean.
Only those outputs are copied to the host.
"""
from __future__ import annotations

import warnings
from typing import Optional

import numpy as np
import torch
from sklearn.base import BaseEstimator, RegressorMixin
from sklearn.utils.validation import check_is_fitted

from . import _lib
from .classifier import MAX_NUMBER_OF_FEATURES, MAX_NUMBER_OF_SAMPLES, MMPFNClassifier
from .engine import B200InferenceEngine
from .model import B200PerFeatureTransformer
from .preprocessing import RECIPES, fit_transform_all, make_members, transform_all
from .weights import load_borders, load_checkpoint

__all__ = ["MMPFNRegressor", "border_map", "member_borders", "bar_tail_device", "bar_tail_tasks_device",
           "check_borders", "prepare_regression"]

OUTPUT_TYPES = ("mean", "median", "mode", "quantiles", "main", "full")
TARGET_TRANSFORMS = (None, "power")
DEFAULT_QUANTILES = tuple(np.round(np.arange(1, 10) * 0.1, 1))


def border_map(f, g):
    """Where the common borders g [K+1] fall within the borders f [K+1] (both nondecreasing, finite) ->
    (src_bucket int32 [K+1], src_share float32 [K+1]): bucket i with f[i] <= g_j < f[i+1] (-1 below f[0], K at or
    above f[K]) and (g_j - f[i]) / (f[i+1] - f[i]) clamped to [0, 1].  Computed in float64."""
    f = np.asarray(f, dtype=np.float64)
    g = np.asarray(g, dtype=np.float64)
    K = len(f) - 1
    bucket = np.searchsorted(f, g, side="right") - 1            # last i with f[i] <= g_j
    share = np.zeros(len(g))
    inner = (bucket >= 0) & (bucket < K)
    i = bucket[inner]
    share[inner] = np.clip((g[inner] - f[i]) / (f[i + 1] - f[i]), 0.0, 1.0)
    return bucket.astype(np.int32), share.astype(np.float32)


def member_borders(transform, g):
    """A member's borders on the y_z axis: f = T^-1(g) in float64 (g itself for no transform).  Non-finite borders
    (the inverse power transform leaves its domain far out in the tails) are replaced by the nearest finite one;
    -> (f [K+1], cancel bool [K]: buckets of zero or non-finite width, whose logits the tail sets to -inf)."""
    g = np.asarray(g, dtype=np.float64)
    if transform is None:
        return g.copy(), np.zeros(len(g) - 1, dtype=bool)
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)          # sklearn warns about the NaN this handles
        f = np.asarray(transform.inverse_transform(g[:, None]), dtype=np.float64).ravel()
    ok = np.isfinite(f)
    if ok.sum() < 2:
        raise ValueError("the target transform maps fewer than two borders to finite values")
    fin = np.nonzero(ok)[0]
    bad = np.nonzero(~ok)[0]
    if len(bad):
        pos = np.clip(np.searchsorted(fin, bad), 1, len(fin) - 1)
        left, right = fin[pos - 1], fin[pos]
        f[bad] = f[np.where(bad - left <= right - bad, left, right)]
    with np.errstate(invalid="ignore"):
        cancel = ~(ok[:-1] & ok[1:]) | ~(np.diff(f) > 0)
    return f, cancel


TAIL_OUTPUTS = ("mean", "median", "mode", "quantiles", "log_prob")


def _bar_tail(entry, lead_args, S: int, K: int, src_bucket, src_share, cancel, borders, *, softmax_temperature,
              average_before_softmax, quantiles, outputs, dev) -> dict:
    """One tail call: ``entry(*lead_args, K, maps, borders, ..., outputs, stream)`` with the requested outputs
    allocated on ``dev`` (S rows) -> dict of device tensors."""
    unknown = set(outputs) - set(TAIL_OUTPUTS)
    if unknown:
        raise ValueError(f"unknown tail outputs {sorted(unknown)}")
    n_q = 0 if quantiles is None else int(quantiles.numel())
    if "quantiles" in outputs and n_q < 1:
        raise ValueError("the quantiles output needs at least one quantile")
    shapes = dict(mean=(S,), median=(S,), mode=(S,), quantiles=(n_q, S), log_prob=(S, K))
    out = {k: torch.empty(shapes[k], dtype=torch.float32, device=dev) for k in outputs}
    ptrs = [out[k].data_ptr() if k in out else None for k in TAIL_OUTPUTS]
    _lib.check(entry(*lead_args, K, src_bucket.data_ptr(), src_share.data_ptr(),
                     None if cancel is None else cancel.data_ptr(), borders.data_ptr(), float(softmax_temperature),
                     int(average_before_softmax), None if quantiles is None else quantiles.data_ptr(), n_q, *ptrs,
                     torch.cuda.current_stream(dev).cuda_stream), entry.__name__)
    return out


def bar_tail_device(logits: torch.Tensor, src_bucket: torch.Tensor, src_share: torch.Tensor,
                    cancel: Optional[torch.Tensor], borders: torch.Tensor, *, softmax_temperature: float,
                    average_before_softmax: bool, quantiles: Optional[torch.Tensor] = None,
                    outputs=("mean",)) -> dict:
    """``mmpfn_bar_tail`` on the current stream: logits [n_est, S, K] fp32 (device) -> dict of device tensors for the
    requested ``outputs`` among "mean", "median", "mode" ([S]), "quantiles" ([n_q, S]) and "log_prob" ([S, K])."""
    logits = logits.to(torch.float32).contiguous()
    n_est, S, K = logits.shape
    return _bar_tail(_lib.load().mmpfn_bar_tail, (logits.data_ptr(), n_est, S), S, K, src_bucket, src_share, cancel,
                     borders, softmax_temperature=softmax_temperature, average_before_softmax=average_before_softmax,
                     quantiles=quantiles, outputs=outputs, dev=logits.device)


def bar_tail_tasks_device(logits, src_bucket: torch.Tensor, src_share: torch.Tensor, cancel: Optional[torch.Tensor],
                          borders: torch.Tensor, *, softmax_temperature: float, average_before_softmax: bool,
                          quantiles: Optional[torch.Tensor] = None, outputs=("mean",)) -> dict:
    """``mmpfn_bar_tail_tasks`` on the current stream, one launch for all tasks: ``logits[t][e]`` fp32 device tensors
    [n_test_t, K] with rows K floats apart (read in place; all tasks have the same number of estimators), maps
    [n_tasks, n_est, K+1], cancel [n_tasks, n_est, K] or None, borders [n_tasks, K+1] -> dict of device tensors over
    the tasks' rows in task order ([S_total], [n_q, S_total], [S_total, K]) and "row_offset" (int32 [n_tasks + 1], on
    the host)."""
    n_est = len(logits[0])
    K = int(logits[0][0].shape[1])
    for lt in logits:
        if len(lt) != n_est:
            raise ValueError("every task needs the same number of estimators")
        for lg in lt:
            if lg.dtype != torch.float32 or lg.dim() != 2 or lg.shape[1] != K or lg.stride(1) != 1 \
                    or (lg.shape[0] > 1 and lg.stride(0) != K) or lg.shape[0] != lt[0].shape[0]:
                raise ValueError("task logits must be fp32 [n_test, K] with rows K floats apart")
    dev = logits[0][0].device
    row_offset = np.concatenate([[0], np.cumsum([lt[0].shape[0] for lt in logits])]).astype(np.int32)
    S_total = int(row_offset[-1])
    ptrs = torch.tensor([lg.data_ptr() for lt in logits for lg in lt], dtype=torch.int64).to(dev)
    ro = torch.from_numpy(row_offset).to(dev)
    out = _bar_tail(_lib.load().mmpfn_bar_tail_tasks, (ptrs.data_ptr(), len(logits), n_est, ro.data_ptr(), S_total),
                    S_total, K, src_bucket, src_share, cancel, borders, softmax_temperature=softmax_temperature,
                    average_before_softmax=average_before_softmax, quantiles=quantiles, outputs=outputs, dev=dev)
    out["row_offset"] = row_offset
    return out


def check_borders(borders, n_out: int) -> np.ndarray:
    """A regression checkpoint's ``criterion.borders`` -> g float64 [n_out + 1]; refuses anything but n_out + 1 finite
    increasing values."""
    if borders is None:
        raise ValueError("regression checkpoint without criterion.borders")
    g = np.asarray(borders.cpu() if isinstance(borders, torch.Tensor) else borders, dtype=np.float64).ravel()
    if len(g) != n_out + 1 or not np.all(np.isfinite(g)) or not np.all(np.diff(g) > 0):
        raise ValueError(f"criterion.borders must be {n_out + 1} finite increasing values")
    return g


def target_transforms(y_z: np.ndarray, n_estimators: int, inference_config: Optional[dict] = None) -> list:
    """One target transform per estimator (None or a fitted Yeo-Johnson ``PowerTransformer``), alternating through
    ``REGRESSION_Y_PREPROCESS_TRANSFORMS`` (default: none, power)."""
    from sklearn.preprocessing import PowerTransformer
    kinds = tuple((inference_config or {}).get("REGRESSION_Y_PREPROCESS_TRANSFORMS", TARGET_TRANSFORMS))
    if not kinds or any(k not in TARGET_TRANSFORMS for k in kinds):
        raise ValueError(f"REGRESSION_Y_PREPROCESS_TRANSFORMS entries must be among {TARGET_TRANSFORMS}")
    power = None
    out = []
    for e in range(n_estimators):
        if kinds[e % len(kinds)] == "power":
            if power is None:
                power = PowerTransformer(method="yeo-johnson", standardize=True).fit(y_z[:, None])
            out.append(power)
        else:
            out.append(None)
    return out


def prepare_regression(X: Optional[np.ndarray], y, g: np.ndarray, *, n_estimators: int, random_state=0,
                       inference_config: Optional[dict] = None) -> dict:
    """The per-dataset host work of a regression fit: target checks, standardisation, the members and their target
    transforms, the preprocessed train tables and the border maps.  ``X``: float32 [Ntr, F] or None; ``g``: the
    checkpoint's borders (``check_borders``).  -> dict with ``y_mean``, ``y_std``, ``transforms``, ``members``
    (``EnsembleMember``), ``tables`` (the engine's member dicts: ``X_train``, ``y_train``, ``class_perm``),
    ``src_bucket`` (int32 [n_est, K+1]), ``src_share`` (float32 [n_est, K+1]), ``cancel`` (bool [n_est, K]) and
    ``target_borders`` (G = g * std + mean, float64 [K+1])."""
    y = np.asarray(y, dtype=np.float64)
    if y.ndim != 1 or len(y) < 2:
        raise ValueError("y must be a 1-dimensional target with at least two rows")
    if not np.all(np.isfinite(y)):
        raise ValueError("y holds NaN or infinite targets")
    mu, sd_y = float(y.mean()), float(y.std())
    if not sd_y > 0:
        raise ValueError("y has zero spread: every target is the same value")
    y_std = sd_y + 1e-20
    y_z = (y - mu) / y_std
    transforms = target_transforms(y_z, n_estimators, inference_config)
    icfg = inference_config or {}
    rng = np.random.default_rng(random_state if isinstance(random_state, (int, np.integer)) else None)
    members = make_members(n_estimators, 0 if X is None else X.shape[1], 0, rng,
                           recipes=tuple(icfg.get("PREPROCESS_TRANSFORMS", RECIPES)),
                           fingerprint=icfg.get("FINGERPRINT_FEATURE", True),
                           feature_shift=icfg.get("FEATURE_SHIFT_METHOD", "shuffle") is not None,
                           class_shift=False)
    tables, buckets, shares, cancels = [], [], [], []
    for (Xt, _), tf in zip(fit_transform_all(members, X, y_z), transforms):
        y_e = y_z if tf is None else tf.transform(y_z[:, None]).ravel()
        tables.append(dict(X_train=Xt, y_train=y_e.astype(np.float32), class_perm=None))
        f, cancel = member_borders(tf, g)
        b, s = border_map(f, g)
        buckets.append(b)
        shares.append(s)
        cancels.append(cancel)
    return dict(y_mean=mu, y_std=y_std, transforms=transforms, members=members, tables=tables,
                src_bucket=np.stack(buckets), src_share=np.stack(shares), cancel=np.stack(cancels),
                target_borders=g * y_std + mu)


def output_request(output_type: str, quantiles=None):
    """``predict``'s ``output_type`` / ``quantiles`` -> (tail outputs to compute, quantile levels float64)."""
    if output_type not in OUTPUT_TYPES:
        raise ValueError(f"output_type must be one of {OUTPUT_TYPES}, got {output_type!r}")
    qs = np.asarray(DEFAULT_QUANTILES if quantiles is None else quantiles, dtype=np.float64).ravel()
    if len(qs) < 1 or not np.all((qs > 0) & (qs < 1)):
        raise ValueError("quantiles must lie strictly between 0 and 1")
    want = {"mean": ("mean",), "median": ("median",), "mode": ("mode",), "quantiles": ("quantiles",),
            "main": ("mean", "median", "mode", "quantiles"),
            "full": ("mean", "median", "mode", "quantiles", "log_prob")}[output_type]
    return want, qs


def format_result(host: dict, output_type: str, target_borders: np.ndarray):
    """Host copies of the tail outputs -> what ``predict(output_type=...)`` returns."""
    if output_type in ("mean", "median", "mode"):
        return host[output_type]
    quant = list(host["quantiles"])
    if output_type == "quantiles":
        return quant
    res = dict(mean=host["mean"], median=host["median"], mode=host["mode"], quantiles=quant)
    if output_type == "full":
        res["logits"] = host["log_prob"]
        res["borders"] = target_borders.astype(np.float32)
    return res


class MMPFNRegressor(RegressorMixin, BaseEstimator):
    def __init__(self, *, mixer_type: str = "MGM+CAP", mgm_heads: int = 8, cap_heads: Optional[int] = 8,
                 features_per_group: int = 2, n_estimators: int = 8, softmax_temperature: float = 0.9,
                 average_before_softmax: bool = False, model_path="auto", device="auto",
                 ignore_pretraining_limits: bool = False, inference_precision="auto",
                 fit_mode: str = "fit_preprocessors", random_state=0, inference_config: Optional[dict] = None):
        self.mixer_type = mixer_type
        self.mgm_heads = mgm_heads
        self.cap_heads = cap_heads
        self.features_per_group = features_per_group
        self.n_estimators = n_estimators
        self.softmax_temperature = softmax_temperature
        self.average_before_softmax = average_before_softmax
        self.model_path = model_path
        self.device = device
        self.ignore_pretraining_limits = ignore_pretraining_limits
        self.inference_precision = inference_precision
        self.fit_mode = fit_mode
        self.random_state = random_state
        self.inference_config = inference_config

    # the device, precision and table handling are the classifier's
    _precision = MMPFNClassifier._precision
    _device = MMPFNClassifier._device
    _to_numeric = MMPFNClassifier._to_numeric

    def _checkpoint(self):
        """-> (state_dict, geometry, borders g float64 [n_out + 1]) of a regression checkpoint; needs no device."""
        if isinstance(self.model_path, tuple):
            sd, geom = self.model_path
            borders = sd.get("criterion.borders")
        elif self.model_path in ("auto", None) or isinstance(self.model_path, B200PerFeatureTransformer):
            raise ValueError("model_path must point to a {'state_dict','config'} regression checkpoint "
                             "(or be a state_dict/geometry tuple): the regressor needs its criterion.borders")
        else:
            sd, geom = load_checkpoint(self.model_path, mixer_type=self.mixer_type, mgm_heads=self.mgm_heads,
                                       cap_heads=self.cap_heads, features_per_group=self.features_per_group)
            borders = load_borders(self.model_path) if "y_encoder.2.layer.weight" not in sd else None
        if "y_encoder.2.layer.weight" in sd:        # the class-rank y-encoder (weights.PackedWeights.regression)
            raise ValueError("model_path holds a classification checkpoint; use MMPFNClassifier")
        return sd, geom, check_borders(borders, geom.n_out)

    def fit(self, X, image, y):
        if self.fit_mode not in ("fit_preprocessors", "fit_with_cache", "low_memory"):
            raise ValueError(f"unknown fit_mode {self.fit_mode!r}")
        if int(self.n_estimators) < 1:
            raise ValueError("n_estimators must be at least 1")
        n_rows = len(np.asarray(y))
        if X is not None:
            X = self._to_numeric(X, fit=True)
            if X.shape[0] != n_rows:
                raise ValueError("X and y have different numbers of rows")
            if not self.ignore_pretraining_limits and (X.shape[0] > MAX_NUMBER_OF_SAMPLES
                                                       or X.shape[1] > MAX_NUMBER_OF_FEATURES):
                raise ValueError("dataset exceeds the pre-training limits; pass ignore_pretraining_limits=True")
            self.n_features_in_ = X.shape[1]
        if image is not None:
            image = np.asarray(image, dtype=np.float32)
            if image.ndim == 2:
                image = image[:, None]
            if len(image) != n_rows:
                raise ValueError("image and y have different numbers of rows")
        if X is None and image is None:
            raise ValueError("fit needs a table X, an embedding image, or both")
        sd, geom, g = self._checkpoint()
        prep = prepare_regression(X, y, g, n_estimators=self.n_estimators, random_state=self.random_state,
                                  inference_config=self.inference_config)
        self.y_train_mean_, self.y_train_std_ = prep["y_mean"], prep["y_std"]
        self.target_transforms_ = prep["transforms"]
        self.members_ = prep["members"]
        seed = int(self.random_state) if isinstance(self.random_state, (int, np.integer)) else 0
        outlier = (self.inference_config or {}).get("OUTLIER_REMOVAL_STD", "auto")
        outlier = 12.0 if outlier == "auto" else outlier
        self.model_ = B200PerFeatureTransformer(sd, geom, device=self._device(), precision=self._precision(),
                                                seed=seed, outlier_std=outlier)
        dev = self.model_.device
        self.borders_ = g                                                   # standardised-target borders
        self.target_borders_ = prep["target_borders"]                       # G, in target units
        self._src_bucket = torch.from_numpy(prep["src_bucket"]).to(dev)
        self._src_share = torch.from_numpy(prep["src_share"]).to(dev)
        self._cancel = (torch.from_numpy(prep["cancel"].astype(np.uint8)).to(dev) if prep["cancel"].any() else None)
        self._borders_dev = torch.from_numpy(self.target_borders_.astype(np.float32)).to(dev)
        self.executor_ = B200InferenceEngine(self.model_, prep["tables"], image,
                                             cache_context=(self.fit_mode == "fit_with_cache"))
        return self

    def predict(self, X, image_test, *, output_type: str = "mean", quantiles=None):
        """float32 numpy per test row: "mean" / "median" / "mode" -> [Nte]; "quantiles" -> a list with one [Nte]
        array per quantile (default 0.1, 0.2, ..., 0.9); "main" -> dict of those four; "full" -> "main" plus
        "logits" (log P, [Nte, K]) and "borders" (G, [K + 1])."""
        check_is_fitted(self, "executor_")
        want, qs = output_request(output_type, quantiles)
        Xn = None if X is None else self._to_numeric(X, fit=False)
        X_tests = transform_all(self.members_, Xn)
        if image_test is not None:
            image_test = np.asarray(image_test, dtype=np.float32)
            if image_test.ndim == 2:
                image_test = image_test[:, None]
        logits = self.executor_.logits(X_tests, image_test)
        q_dev = torch.from_numpy(qs.astype(np.float32)).to(self.model_.device) if "quantiles" in want else None
        out = bar_tail_device(logits, self._src_bucket, self._src_share, self._cancel, self._borders_dev,
                              softmax_temperature=self.softmax_temperature,
                              average_before_softmax=self.average_before_softmax, quantiles=q_dev, outputs=want)
        host = {k: v.cpu().numpy() for k, v in out.items()}
        self.executor_.check_nan()
        return format_result(host, output_type, self.target_borders_)
