"""``MMPFNClassifier`` — the reference's estimator surface (``classifier.py:112-137, 364-576``) on
top of the sm_100a path.  Same constructor keywords, ``fit(X, image, y)``,
``predict_proba(X, image_test)`` and ``predict(X, X_image)``; probabilities are float32, one
column per class seen in ``fit``, rows summing to one.

What differs from the reference is confined to the CPU stage in front of the hot path (see
``preprocessing.py`` here) and to scheduling: all estimators run in one batched forward per
feature count, weights stay on the device, and ``fit_mode="fit_with_cache"`` keeps the train
rows' K/V context from ``fit`` (in the reference that mode does not carry images,
SURVEY.md gotcha 5).
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch
from sklearn.base import BaseEstimator, ClassifierMixin
from sklearn.preprocessing import LabelEncoder, OrdinalEncoder
from sklearn.utils.validation import check_is_fitted

from .engine import B200InferenceEngine, proba_from_logits
from .model import B200PerFeatureTransformer
from .preprocessing import RECIPES, fit_transform_all, make_members, transform_all
from .weights import load_checkpoint

__all__ = ["MMPFNClassifier"]

MAX_NUMBER_OF_CLASSES = 10        # constants.py:34-211 (ModelInterfaceConfig)
MAX_NUMBER_OF_SAMPLES = 10_000
MAX_NUMBER_OF_FEATURES = 500


def precision_name(p) -> str:
    """The layer precision ("fp32", "bf16" or "fp16") an ``inference_precision`` value selects."""
    if p in ("auto", "autocast", torch.bfloat16, "bf16", "bfloat16"):
        return "bf16"          # the reference autocasts on CUDA (base.py:126-165); bf16 here, SURVEY gotcha 4
    if p in (torch.float32, "fp32", "float32"):
        return "fp32"
    if p in (torch.float16, "fp16", "float16"):
        return "fp16"          # the reference's own CUDA autocast type (inference.py:339): 3 more bits than bf16
    raise ValueError(f"unsupported inference_precision {p!r} (fp32, fp16, or bf16/auto)")


class MMPFNClassifier(ClassifierMixin, BaseEstimator):
    def __init__(self, *, mixer_type: str = "MGM+CAP", mgm_heads: int = 8, cap_heads: Optional[int] = 8,
                 features_per_group: int = 2, n_estimators: int = 4, categorical_features_indices=None,
                 softmax_temperature: float = 0.9, balance_probabilities: bool = False,
                 average_before_softmax: bool = False, model_path="auto", device="auto",
                 ignore_pretraining_limits: bool = False, inference_precision="auto",
                 fit_mode: str = "fit_preprocessors", memory_saving_mode="auto", random_state=0, n_jobs: int = -1,
                 inference_config: Optional[dict] = None):
        self.mixer_type = mixer_type
        self.mgm_heads = mgm_heads
        self.cap_heads = cap_heads
        self.features_per_group = features_per_group
        self.n_estimators = n_estimators
        self.categorical_features_indices = categorical_features_indices
        self.softmax_temperature = softmax_temperature
        self.balance_probabilities = balance_probabilities
        self.average_before_softmax = average_before_softmax
        self.model_path = model_path
        self.device = device
        self.ignore_pretraining_limits = ignore_pretraining_limits
        self.inference_precision = inference_precision
        self.fit_mode = fit_mode
        self.memory_saving_mode = memory_saving_mode
        self.random_state = random_state
        self.n_jobs = n_jobs
        self.inference_config = inference_config

    # -------------------------------------------------------------------------------------
    def _precision(self) -> str:
        return precision_name(self.inference_precision)

    def _device(self) -> torch.device:
        if self.device in ("auto", "cuda"):
            if not torch.cuda.is_available():
                raise RuntimeError("no CUDA device: this build has no CPU path (BASELINE.json north_star)")
            return torch.device("cuda", torch.cuda.current_device())
        dev = torch.device(self.device)
        if dev.type != "cuda":
            raise RuntimeError("device must be a CUDA device: this build has no CPU path")
        return dev

    def _load_model(self) -> B200PerFeatureTransformer:
        if isinstance(self.model_path, B200PerFeatureTransformer):
            return self.model_path
        if self.model_path in ("auto", None):
            # the reference ships no checkpoint and has downloads disabled (base.py:84)
            raise ValueError("model_path must point to a {'state_dict','config'} checkpoint "
                             "(or be a state_dict/geometry tuple)")
        if isinstance(self.model_path, tuple):
            sd, geom = self.model_path
        else:
            sd, geom = load_checkpoint(self.model_path, mixer_type=self.mixer_type, mgm_heads=self.mgm_heads,
                                       cap_heads=self.cap_heads, features_per_group=self.features_per_group)
        seed = int(self.random_state) if isinstance(self.random_state, (int, np.integer)) else 0
        icfg = self.inference_config or {}
        outlier = icfg.get("OUTLIER_REMOVAL_STD", "auto")
        outlier = 12.0 if outlier == "auto" else outlier        # constants.py:181
        return B200PerFeatureTransformer(sd, geom, device=self._device(), precision=self._precision(), seed=seed,
                                         outlier_std=outlier)

    def fit(self, X, image, y):
        """classifier.py:364-502."""
        if self.fit_mode not in ("fit_preprocessors", "fit_with_cache", "low_memory"):
            raise ValueError(f"unknown fit_mode {self.fit_mode!r}")
        rng = np.random.default_rng(self.random_state if isinstance(self.random_state, (int, np.integer)) else None)
        self.model_ = self._load_model()
        y = np.asarray(y)
        if X is not None:
            X = self._to_numeric(X, fit=True)
            if X.shape[0] != len(y):
                raise ValueError("X and y have different numbers of rows")
            if not self.ignore_pretraining_limits and (X.shape[0] > MAX_NUMBER_OF_SAMPLES
                                                       or X.shape[1] > MAX_NUMBER_OF_FEATURES):
                raise ValueError("dataset exceeds the pre-training limits; pass ignore_pretraining_limits=True")
            self.n_features_in_ = X.shape[1]
        _, counts = np.unique(y, return_counts=True)
        self.class_counts_ = counts
        self.label_encoder_ = LabelEncoder()
        yi = self.label_encoder_.fit_transform(y)
        self.classes_ = self.label_encoder_.classes_
        self.n_classes_ = len(self.classes_)
        if self.n_classes_ > MAX_NUMBER_OF_CLASSES:
            raise ValueError(f"Number of classes {self.n_classes_} exceeds the maximal number of classes supported")
        if image is not None:
            image = np.asarray(image, dtype=np.float32)
            if image.ndim == 2:
                image = image[:, None]
            if len(image) != len(y):
                raise ValueError("image and y have different numbers of rows")
        icfg = self.inference_config or {}
        recipes = icfg.get("PREPROCESS_TRANSFORMS", RECIPES)
        self.members_ = make_members(self.n_estimators, 0 if X is None else X.shape[1], self.n_classes_, rng,
                                     recipes=tuple(recipes), fingerprint=icfg.get("FINGERPRINT_FEATURE", True),
                                     feature_shift=icfg.get("FEATURE_SHIFT_METHOD", "shuffle") is not None,
                                     class_shift=icfg.get("CLASS_SHIFT_METHOD", "shuffle") is not None)
        members = [dict(X_train=Xt, y_train=yt, class_perm=m.class_perm)
                   for m, (Xt, yt) in zip(self.members_, fit_transform_all(self.members_, X, yi))]
        self.executor_ = B200InferenceEngine(self.model_, members, image,
                                             cache_context=(self.fit_mode == "fit_with_cache"))
        return self

    def _to_numeric(self, X, fit: bool) -> np.ndarray:
        """Ordinal-encode non-numeric columns (classifier.py:443-449)."""
        try:
            import pandas as pd
            if isinstance(X, pd.DataFrame):
                obj = [c for c in X.columns if not pd.api.types.is_numeric_dtype(X[c])]
                if obj:
                    X = X.copy()
                    if fit:
                        self.preprocessor_ = OrdinalEncoder(handle_unknown="use_encoded_value", unknown_value=np.nan)
                        self.obj_cols_ = obj
                        X[obj] = self.preprocessor_.fit_transform(X[obj].astype(str))
                    else:
                        X[self.obj_cols_] = self.preprocessor_.transform(X[self.obj_cols_].astype(str))
                X = X.to_numpy(dtype=np.float32)
        except ImportError:  # pragma: no cover
            pass
        X = np.asarray(X, dtype=np.float32)
        if X.ndim != 2:
            raise ValueError("X must be 2-dimensional")
        if not fit and X.shape[1] != self.n_features_in_:
            raise ValueError(f"X has {X.shape[1]} features, expected {self.n_features_in_}")
        return X

    def predict_proba(self, X, image_test):
        """classifier.py:517-576."""
        check_is_fitted(self, "executor_")
        Xn = None if X is None else self._to_numeric(X, fit=False)
        X_tests = transform_all(self.members_, Xn)
        if image_test is not None:
            image_test = np.asarray(image_test, dtype=np.float32)
            if image_test.ndim == 2:
                image_test = image_test[:, None]
        logits = self.executor_.logits(X_tests, image_test)
        proba = proba_from_logits(logits, [m.class_perm for m in self.members_], n_classes=self.n_classes_,
                                  class_counts=self.class_counts_, softmax_temperature=self.softmax_temperature,
                                  average_before_softmax=self.average_before_softmax,
                                  balance_probabilities=self.balance_probabilities)
        self.executor_.check_nan()      # transformer.py:727-731, :790-796 (one flag read after the D2H copy)
        return proba

    def predict(self, X, X_image):
        proba = self.predict_proba(X, X_image)
        return self.label_encoder_.inverse_transform(np.argmax(proba, axis=1))
