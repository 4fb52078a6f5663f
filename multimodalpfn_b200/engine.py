"""Inference engine: the caller of the hot path, mirroring the reference's
``InferenceEngineCachePreprocessing`` (``inference.py:204-351``) and the probability tail of
``MMPFNClassifier.predict_proba`` (``classifier.py:544-576``).

Differences from the reference, all result-neutral:
* estimators that share a preprocessed feature count run as ONE batched forward (the reference
  loops over them serially, ``inference.py:294-349``) and share the image/text stem, which does not
  depend on the estimator (``inference.py:272, 311-314``);
* weights stay resident on the device (the reference moves the model host<->device on every
  ``predict_proba``, ``inference.py:291, 351``);
* ``fit_mode="fit_with_cache"`` keeps the per-layer K/V context of the train rows from ``fit`` so
  that ``predict_proba`` runs the test rows only.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from .model import B200PerFeatureTransformer, TrainContext

__all__ = ["proba_device", "proba_from_logits", "estimator_groups", "B200InferenceEngine"]


def proba_device(logits: torch.Tensor, class_perms: Sequence[Optional[np.ndarray]], *, n_classes: int,
                 class_counts=None, softmax_temperature: float = 0.9, average_before_softmax: bool = False,
                 balance_probabilities: bool = False) -> torch.Tensor:
    """classifier.py:544-566 on the device: logits [n_est, Nte, n_out] -> float32 [Nte, n_classes] (device tensor,
    not yet renormalised on the host).

    Quirk mirrored from the reference: the ``[:, :n_classes]`` slice lives inside
    ``if softmax_temperature != 1`` (classifier.py:544-547); with temperature 1 and no class
    permutation all ``n_out`` logits enter the softmax.
    """
    lib = _lib.load()
    logits = logits.to(torch.float32).contiguous()
    n_est, S, n_out = logits.shape
    width = n_classes
    if softmax_temperature == 1 and all(p is None for p in class_perms):
        width = n_out
    perm = np.stack([np.arange(width) if p is None else np.asarray(p)[:width] for p in class_perms]).astype(np.int32)
    if perm.shape[1] != width:
        raise ValueError("class permutation length does not match the number of classes")
    dev = logits.device
    perm_d = torch.from_numpy(perm).to(dev)
    prior_d = None
    if balance_probabilities:
        cc = np.asarray(class_counts, dtype=np.float64)
        if cc.shape != (width,):
            # the reference's out * cc/cc.sum() (classifier.py:563-566) fails to broadcast; the kernel would read
            # past the end of the prior
            raise ValueError(f"{cc.size} class counts for {width} probability columns")
        prior_d = torch.from_numpy((cc / cc.sum()).astype(np.float32)).to(dev)
    proba = torch.empty((S, width), dtype=torch.float32, device=dev)
    _lib.check(lib.mmpfn_proba_tail(logits.data_ptr(), perm_d.data_ptr(), None if prior_d is None else prior_d.data_ptr(),
                                    n_est, S, n_out, width, float(softmax_temperature), int(average_before_softmax),
                                    proba.data_ptr(), torch.cuda.current_stream(dev).cuda_stream), "mmpfn_proba_tail")
    return proba


def proba_from_logits(logits: torch.Tensor, class_perms: Sequence[Optional[np.ndarray]], **kw) -> np.ndarray:
    """``proba_device`` + the D2H copy + the host renormalisation of classifier.py:568-576 -> float32 numpy."""
    out = proba_device(logits, class_perms, **kw).cpu().numpy()
    return out / out.sum(axis=1, keepdims=True)      # classifier.py:576 (after the D2H copy, like the reference)


def estimator_groups(members) -> list:
    """Estimators grouped by preprocessed width (-1: no table), widths ascending -> [(F, [member index])]: one
    batched forward per group, whose label statistics are taken over the group's [len(idx), Ntr] block."""
    groups = {}
    for i, m in enumerate(members):
        F = -1 if m["X_train"] is None else m["X_train"].shape[1]
        groups.setdefault(F, []).append(i)
    return sorted(groups.items())


class B200InferenceEngine:
    """Holds the per-estimator preprocessed training tables and runs all estimators per call.

    ``members``: list of dicts with keys ``X_train`` (np [Ntr, F'] float32 or None), ``y_train``
    (np [Ntr], permuted class ids), ``transform`` (callable: raw test table -> np [Nte, F']) and
    ``class_perm`` (np or None) — what the reference keeps per ``EnsembleConfig``
    (``inference.py:217-222``).
    """

    def __init__(self, model: B200PerFeatureTransformer, members, image_train: Optional[np.ndarray], *,
                 cache_context: bool = False):
        self.model = model
        self.members = list(members)
        self.image_train = None if image_train is None else np.asarray(image_train, dtype=np.float32)
        self.cache_context = cache_context
        dev = model.device
        self.groups = []
        for F, idx in estimator_groups(self.members):
            Xtr = None
            if F >= 0:
                Xtr = torch.from_numpy(np.stack([np.asarray(self.members[i]["X_train"], dtype=np.float32)
                                                 for i in idx])).to(dev)
            ytr = torch.from_numpy(np.stack([np.asarray(self.members[i]["y_train"], dtype=np.float32)
                                             for i in idx])).to(dev)
            # label statistics need a host sync (unique labels): once here, not per call
            self.groups.append(dict(F=F, idx=idx, X_train=Xtr, y_train=ytr, ctx=None,
                                    label_stats=model.label_stats(ytr)))
        self.img_train_dev = None if self.image_train is None else torch.from_numpy(self.image_train).to(dev)
        self._img_tok_train = None
        self.nan_flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self._graphs = {}                      # input shapes -> (graph, static inputs, static output, scratch epoch)
        self.max_graphs = 4                    # least recently used beyond that are dropped (each holds a private pool)
        self._pinned_bufs = {}
        self.multi_group = True                # False: one pass per group (tests compare the two, bit for bit)
        self._stage_event = None
        self._side = None                      # side stream of the test-row image stem
        self.launches_per_call = None
        if cache_context:
            self._build_contexts()

    def train_image_tokens(self):
        """Image/text tokens of the TRAIN rows: the MGM/CAP stem works row by row and the train embeddings never
        change between calls (inference.py:272 keeps them as they are), so they are projected once — the
        reference recomputes them inside every forward (transformer.py:755-761)."""
        if self.img_train_dev is not None and self._img_tok_train is None:
            self._img_tok_train = self.model.stem_image(self.img_train_dev)
        return self._img_tok_train

    def _build_contexts(self):
        self.train_image_tokens()
        for g in self.groups:
            g["ctx"] = self.model.fit_context(g["X_train"], None, g["y_train"], img_tok_train=self._img_tok_train,
                                              label_stats=g["label_stats"])
            if self.img_train_dev is not None:
                g["ctx"].n_tok = self.img_train_dev.shape[1]

    def _pinned(self, key, shape):
        """A persistent page-locked host buffer per input: the H2D copies of a call are asynchronous
        DMA transfers from pinned memory, not staged pageable copies."""
        buf = self._pinned_bufs.get(key)
        if buf is None or tuple(buf.shape) != tuple(shape):
            # (the CPU stand-in model of the gloo tests has no driver to pin memory with)
            buf = torch.empty(tuple(shape), dtype=torch.float32, pin_memory=self.model.device.type == "cuda")
            self._pinned_bufs[key] = buf
        return buf

    def stage(self, X_test_per_member: Sequence[Optional[np.ndarray]], image_test: Optional[np.ndarray], *,
              image_dev: Optional[torch.Tensor] = None):
        """Host -> device copies of one call's inputs (the per-step H2D traffic): the preprocessed test
        table of every estimator and the test embeddings, through pinned host buffers.  ``image_dev``: the test
        embeddings already on the device (several engines of one call share one upload)."""
        dev = self.model.device
        if self._stage_event is not None:
            self._stage_event.synchronize()        # the previous call's DMA has left the pinned buffers
        img_test_dev = None
        if image_dev is not None and self.img_train_dev is not None:
            img_test_dev = image_dev
        elif image_test is not None and self.img_train_dev is not None:        # inference.py:311-316
            img = np.asarray(image_test, dtype=np.float32)
            if img.ndim == 2:
                img = img[:, None]
            pin = self._pinned("img", img.shape)
            pin.numpy()[...] = img
            img_test_dev = pin.to(dev, non_blocking=True)
        Xte = []
        for gi, g in enumerate(self.groups):
            if g["F"] >= 0:
                first = np.asarray(X_test_per_member[g["idx"][0]])
                pin = self._pinned(("x", gi), (len(g["idx"]),) + first.shape)
                dst = pin.numpy()
                for k, i in enumerate(g["idx"]):
                    dst[k] = X_test_per_member[i]
                Xte.append(pin.to(dev, non_blocking=True))
            else:
                Xte.append(None)
        if dev.type == "cuda":
            self._stage_event = torch.cuda.Event()
            self._stage_event.record(torch.cuda.current_stream(dev))
        return dict(X_test=Xte, img_test=img_test_dev)

    def logits_staged(self, staged) -> torch.Tensor:
        """The device-resident part of one call -> [n_est, Nte, n_out], estimator order as given to
        the constructor."""
        m = self.model
        out = [None] * len(self.members)
        img_test_dev = staged["img_test"]
        flag = self.nan_flag
        flag.zero_()
        # several groups with tables, bf16: one batched pass over all of them (flat sublayers launch once)
        multi = (1 < len(self.groups) <= 8 and getattr(m, "precision", None) == _lib.BF16 and hasattr(m, "fit_contexts")
                 and all(g["F"] >= 0 for g in self.groups) and self.multi_group)
        if self.cache_context and multi:
            tok_test = m.stem_image(img_test_dev) if img_test_dev is not None else None
            lgs = m.predict_with_contexts([g["ctx"] for g in self.groups], staged["X_test"], img_tok_test=tok_test,
                                          nan_flag=flag)
            for g, lg in zip(self.groups, lgs):
                for k, i in enumerate(g["idx"]):
                    out[i] = lg[k]
        elif multi:
            tok_tr = tok_te = None
            join = None
            if img_test_dev is not None:
                tok_tr = self.train_image_tokens()
                # the image/text stem of the TEST rows (a dozen small, latency-bound launches) does not depend on the
                # context build: it runs on a side stream beside the train pass and joins before the test pass
                # (only the FFMA stem: from 32 MGM heads its gated projection is a TMA / tcgen05 kernel, and layer-type
                # kernels of two streams must not overlap, include/mmpfn_b200.h)
                if m.geom.mgm_heads < 32:
                    dev = m.device
                    main = torch.cuda.current_stream(dev)
                    if self._side is None:
                        self._side = torch.cuda.Stream(device=dev)
                    self._side.wait_stream(main)
                    with torch.cuda.stream(self._side):
                        tok_te = m.stem_image(img_test_dev)
                        join = torch.cuda.Event()
                        join.record(self._side)
                    if not torch.cuda.is_current_stream_capturing():
                        tok_te.record_stream(main)
                else:
                    tok_te = m.stem_image(img_test_dev)
            specs = [dict(X_train=g["X_train"], y_train=g["y_train"], X_all=torch.cat([g["X_train"], Xte], dim=1),
                          img_tok_train=tok_tr, label_stats=g["label_stats"])
                     for g, Xte in zip(self.groups, staged["X_test"])]
            ctxs = m.fit_contexts(specs, nan_flag=flag)
            if join is not None:
                torch.cuda.current_stream(m.device).wait_event(join)
            lgs = m.predict_with_contexts(ctxs, staged["X_test"], img_tok_test=tok_te, nan_flag=flag)
            for g, lg in zip(self.groups, lgs):
                for k, i in enumerate(g["idx"]):
                    out[i] = lg[k]
        elif self.cache_context:
            tok_test = m.stem_image(img_test_dev) if img_test_dev is not None else None
            for g, Xte in zip(self.groups, staged["X_test"]):
                lg = m.predict_with_context(g["ctx"], Xte, None, img_tok_test=tok_test, check=False, nan_flag=flag)
                for k, i in enumerate(g["idx"]):
                    out[i] = lg[k]
        else:
            # reference-equivalent: the train context is rebuilt inside every call (inference.py:302-348)
            tok_tr = tok_te = None
            if img_test_dev is not None:
                tok_tr, tok_te = self.train_image_tokens(), m.stem_image(img_test_dev)
            for g, Xte in zip(self.groups, staged["X_test"]):
                X_full = None if Xte is None else torch.cat([g["X_train"], Xte], dim=1)
                ctx = m.fit_context(g["X_train"], None, g["y_train"], X_all=X_full, img_tok_train=tok_tr, check=False,
                                    label_stats=g["label_stats"], nan_flag=flag)
                lg = m.predict_with_context(ctx, Xte, None, img_tok_test=tok_te, check=False, nan_flag=flag)
                for k, i in enumerate(g["idx"]):
                    out[i] = lg[k]
        return torch.stack(out)

    def check_nan(self):
        """One host sync: raises like the reference does when the stem produced NaN."""
        self.model._check_nan(self.nan_flag)

    # ---- CUDA-graph replay of the device-resident step ------------------------------------------
    def logits_graphed(self, staged) -> torch.Tensor:
        """Replays ``logits_staged`` as one CUDA graph (launch-latency bound otherwise: ~400 kernels
        per call).  ``staged`` is copied into static input buffers; the returned tensor is the
        graph's static output (valid until the next call)."""
        key = (tuple(None if x is None else tuple(x.shape) for x in staged["X_test"]),
               None if staged["img_test"] is None else tuple(staged["img_test"].shape))
        ent = self._graphs.get(key)
        epoch = getattr(self.model, "scratch_epoch", 0)
        if ent is not None and ent[3] != epoch:
            # a scratch buffer of the model was replaced since the capture (a larger batch, another engine or
            # predict_proba_tasks on the same model): every captured graph points into freed storage
            self._graphs.clear()
            ent = None
        if ent is None:
            static = dict(X_test=[None if x is None else x.clone() for x in staged["X_test"]],
                          img_test=None if staged["img_test"] is None else staged["img_test"].clone())
            side = torch.cuda.Stream(device=self.model.device)
            side.wait_stream(torch.cuda.current_stream(self.model.device))
            with torch.cuda.stream(side):
                for _ in range(2):                     # warm-up: sizes every scratch buffer, fills caches
                    self.logits_staged(static)
            torch.cuda.current_stream(self.model.device).wait_stream(side)
            torch.cuda.synchronize(self.model.device)
            graph = torch.cuda.CUDAGraph()
            l0 = _lib.launch_count()
            with torch.cuda.graph(graph):
                out = self.logits_staged(static)
            self.launches_per_call = _lib.launch_count() - l0
            # the warm-up may itself have grown the scratch buffers: graphs captured earlier are stale then
            epoch_now = getattr(self.model, "scratch_epoch", 0)
            if epoch_now != epoch:
                self._graphs.clear()
            ent = (graph, static, out, epoch_now)
            self._graphs[key] = ent
            while len(self._graphs) > self.max_graphs:
                self._graphs.pop(next(iter(self._graphs)))
        else:
            self._graphs[key] = self._graphs.pop(key)          # most recently used last
        graph, static, out, _ = ent
        for dst, src in zip(static["X_test"], staged["X_test"]):
            if dst is not None:
                dst.copy_(src, non_blocking=True)
        if static["img_test"] is not None:
            static["img_test"].copy_(staged["img_test"], non_blocking=True)
        graph.replay()
        return out

    def logits(self, X_test_per_member: Sequence[Optional[np.ndarray]], image_test: Optional[np.ndarray], *,
               graph: bool = True, image_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
        staged = self.stage(X_test_per_member, image_test, image_dev=image_dev)
        out = self.logits_graphed(staged) if graph else self.logits_staged(staged)
        return out
