"""Plug-in mode: keep the reference's own ``MMPFNClassifier`` in charge (validation, ordinal
encoding, ``EnsembleConfig`` generation, numpy/sklearn preprocessing) and swap only the object its
engine calls at ``inference.py:343-348`` for ``B200PerFeatureTransformer``.

    import multimodalpfn_b200.plugin as plugin
    plugin.install(precision="bf16")          # after `mmpfn` is importable; "fp16" (the reference's own CUDA
                                              # autocast type, closer to fp32) and "fp32" work the same way
    clf = mmpfn.models.mmpfn.MMPFNClassifier(..., device="cuda").fit(X, img, y)
    clf.predict_proba(X_te, img_te)           # forward runs on libmmpfn_b200.so

The patch wraps ``create_inference_engine`` (``base.py:168-257``, called from
``classifier.py:485-500``): the engine the reference builds keeps its per-estimator preprocessors
and tables; its ``.model`` attribute is replaced.  Nothing under the reference tree is edited.
Needs the reference and an sm_100 GPU in the same process: ``tests/test_gpu_plugin.py`` runs it on the
GPU box against the unmodified reference snapshot ``oracle/snapshot_ref.py`` ships there (real
``MMPFNClassifier``, real CUDA model, compared with the reference's own CPU and CUDA ``predict_proba``);
``tests/test_plugin_wiring.py`` checks the wiring on CPU with a recording stand-in for the CUDA model.
"""
from __future__ import annotations

import functools

from .synth import Geometry

_MIXERS = {"MGM": "MGM", "MGM+CAP": "MGM+CAP", "MoE": "MoE"}


def geometry_of(module) -> Geometry:
    """Read the geometry off a reference ``PerFeatureTransformer`` (``model/transformer.py:292-409``)."""
    mixer = getattr(module, "mixer_type", "MGM+CAP")
    mgm_heads = len(module.mgm.projs) if hasattr(module, "mgm") else (
        len(module.moe.experts) if hasattr(module, "moe") else 1)
    cap_heads = module.cap.queries.shape[0] if hasattr(module, "cap") else None
    dec = module.decoder_dict["standard"]
    return Geometry(emsize=module.ninp, nhead=module.nhead, nhid_factor=module.nhid // module.ninp,
                    nlayers=len(module.transformer_encoder.layers), n_out=dec[2].weight.shape[0],
                    features_per_group=module.features_per_group, img_dim=module.nhid, mgm_heads=mgm_heads,
                    cap_heads=cap_heads, mixer_type=_MIXERS[mixer])


def outlier_std_of(module):
    """``update_encoder_outlier_params`` (``utils.py:703-745``) stored it on the normalisation step."""
    for step in module.encoder:
        if "InputNormalizationEncoderStep" in str(step.__class__):
            return float(step.remove_outliers_sigma) if step.remove_outliers else None
    return None


def convert(module, *, device, precision="bf16", model_cls=None, pos_emb_device="cuda"):
    """reference nn.Module -> B200PerFeatureTransformer with the same weights and seed.

    ``pos_emb_device``: where the positional noise is drawn.  The reference draws it with a generator on
    the model's device (``transformer.py:887-892``), and torch's CPU and CUDA generators give different
    streams: "cuda" reproduces the reference running on the same GPU, "cpu" the reference on the host."""
    if model_cls is None:
        from .model import B200PerFeatureTransformer as model_cls
    sd = {k: v.detach().cpu() for k, v in module.state_dict().items()}
    return model_cls(sd, geometry_of(module), device=device, precision=precision, seed=module.seed,
                     outlier_std=outlier_std_of(module), pos_emb_device=pos_emb_device)


class B200PluginEngine:
    """Stands where the reference's ``InferenceEngineCachePreprocessing`` stands (``inference.py:204-351``),
    built FROM the engine the reference prepared: its fitted per-estimator preprocessors, preprocessed
    train tables, permuted labels, ensemble configs and train embeddings are taken as they are, so the
    tensors that reach the model are the reference's.  What changes is how ``iter_outputs``
    (``inference.py:282-351``) produces its logits: instead of a serial loop of B = 1 forwards that each wait
    for their host transform, the estimators run as a few batched CUDA passes (``engine.B200InferenceEngine``,
    one CUDA graph each) and the passes are PIPELINED with the host work — while the GPU runs the pass of one
    sub-batch, the host already transforms the test table for the next one with that estimator's own
    preprocessor (the reference's numpy/sklearn code, ~2-5 ms per estimator, GIL-bound).  ``(logits[Nte,
    n_out], config)`` is yielded per estimator in the reference's order — the rest of ``predict_proba``
    (``classifier.py:532-576``) is untouched.

    Sub-batches: estimators sharing a preprocessed width, ``stage_size`` at a time, cheapest recipe first (so
    that the GPU starts early).

    ``replay=True`` (default): the fitted preprocessors are also compiled into validation-free replays
    (``ref_transform.compile_preprocessor``: same arithmetic on the same fitted state, 5-7x cheaper per call).  The
    first table that arrives is transformed both ways, together with perturbed probe rows; only when every member's
    replay reproduces the reference's ``transform`` bit for bit are the replays used from then on — and since the
    host work then is a few milliseconds in all, the estimators run as ONE batched pass instead of the pipeline.
    A member whose preprocessor is not reproduced (``Unsupported`` step, any mismatch) keeps the whole engine on the
    reference's own ``transform`` calls."""

    def __init__(self, ref_engine, *, device, precision="bf16", pos_emb_device="cuda", model_cls=None,
                 cache_context=False, stage_size=2, replay=True):
        import numpy as np
        from .engine import B200InferenceEngine
        from . import ref_transform
        self.ref = ref_engine
        self.preprocessors = ref_engine.preprocessors
        self.ensemble_configs = ref_engine.ensemble_configs
        self.model = convert(ref_engine.model, device=device, precision=precision, model_cls=model_cls,
                             pos_emb_device=pos_emb_device)
        self.members = [dict(X_train=None if Xt is None else np.asarray(Xt, dtype=np.float32),
                             y_train=np.asarray(yt, dtype=np.float32), class_perm=None)
                        for Xt, yt in zip(ref_engine.X_trains, ref_engine.y_trains)]
        by_width = {}
        for i, m in enumerate(self.members):
            by_width.setdefault(-1 if m["X_train"] is None else m["X_train"].shape[1], []).append(i)
        self.stages = []
        for _, idx in sorted(by_width.items()):                     # fewer columns = the cheaper recipe first
            for a in range(0, len(idx), max(1, stage_size)):
                sub = idx[a:a + max(1, stage_size)]
                eng = B200InferenceEngine(self.model, [self.members[i] for i in sub], ref_engine.image_train,
                                          cache_context=cache_context)
                if self.stages:                                     # the train-row image tokens are the same for all
                    eng._img_tok_train = self.stages[0][1].train_image_tokens()
                self.stages.append((sub, eng))
        self._img_pin = None
        self._cache_context = cache_context
        # "unverified" -> "on" | "off" at the first table (see the class docstring); self.replay_note says why
        self.replay_state, self.replay_note, self._fast, self._all = "off", "disabled", None, None
        if replay:
            try:
                self._fast = [ref_transform.compile_preprocessor(p) for p in self.preprocessors]
                self.replay_state, self.replay_note = "unverified", "compiled, not yet compared with the reference"
            except ref_transform.Unsupported as exc:
                self.replay_note = f"not reproduced: {exc}"

    def _upload_image(self, image_test):
        import numpy as np
        import torch
        if image_test is None or self.ref.image_train is None:
            return None
        img = np.asarray(image_test, dtype=np.float32)
        if img.ndim == 2:
            img = img[:, None]
        if self._img_pin is None or tuple(self._img_pin.shape) != img.shape:
            self._img_pin = torch.empty(img.shape, dtype=torch.float32, pin_memory=self.model.device.type == "cuda")
        # (the previous call ended with a host sync — the NaN-flag read — so its DMA has left this buffer)
        self._img_pin.numpy()[...] = img
        return self._img_pin.to(self.model.device, non_blocking=True)

    def _verify_replay(self, X):
        import numpy as np
        from . import ref_transform
        from .engine import B200InferenceEngine
        probe = ref_transform.make_probe(X)
        for i, (pre, fast) in enumerate(zip(self.preprocessors, self._fast)):
            if self.members[i]["X_train"] is None:
                continue
            if not (ref_transform.verify(pre, fast, X) and ref_transform.verify(pre, fast, probe)):
                self.replay_state, self.replay_note = "off", f"replay of member {i} differs from the reference's transform"
                return
        # ... and through the memo that lets members share equal fitted nodes within one call
        fasts = [None if m["X_train"] is None else f for m, f in zip(self.members, self._fast)]
        for table in (X, probe):
            try:
                shared = ref_transform.replay_all(fasts, table)
                refs = [None if f is None else np.asarray(pre.transform(table).X) for pre, f in zip(self.preprocessors, fasts)]
            except Exception:
                continue                  # (a table the reference refuses: verified member by member above)
            if not all(a is None or (a.shape == b.shape and np.array_equal(a, b, equal_nan=True)) for a, b in zip(shared, refs)):
                self.replay_state, self.replay_note = "off", "shared replay differs from the reference's transform"
                return
        self._all = B200InferenceEngine(self.model, self.members, self.ref.image_train, cache_context=self._cache_context)
        self._all._img_tok_train = self.stages[0][1].train_image_tokens()
        self.replay_state, self.replay_note = "on", "bit-identical to the reference's transform on the first table and its probes"

    def iter_outputs(self, X, image_test, *, device=None, autocast=None):
        import numpy as np
        image_dev = self._upload_image(image_test)
        outs = [None] * len(self.members)
        if X is not None and self.replay_state == "unverified":
            self._verify_replay(X)
        if X is not None and self.replay_state == "on":
            from . import ref_transform
            X_tests = [None if t is None else np.asarray(t, dtype=np.float32) for t in ref_transform.replay_all(
                [None if m["X_train"] is None else f for m, f in zip(self.members, self._fast)], X)]
            lg = self._all.logits(X_tests, None, image_dev=image_dev)
            self._all.check_nan()
            for out, cfg in zip(lg, self.ensemble_configs):
                yield out, cfg
            return
        for sub, eng in self.stages:
            X_tests = [None if X is None or self.members[i]["X_train"] is None
                       else np.asarray(self.preprocessors[i].transform(X).X, dtype=np.float32) for i in sub]   # inference.py:303
            lg = eng.logits(X_tests, None, image_dev=image_dev)       # asynchronous: H2D + one CUDA-graph replay
            for k, i in enumerate(sub):
                outs[i] = lg[k]
        for _, eng in self.stages:
            eng.check_nan()                                           # transformer.py:790-796 (first host sync of the call)
        for lg, cfg in zip(outs, self.ensemble_configs):
            yield lg, cfg


def install(precision: str = "bf16", model_cls=None, pos_emb_device: str = "cuda", mode: str = "engine",
            replay: bool = True):
    """Patch ``create_inference_engine`` where the reference's estimators look it up
    (``mmpfn.models.mmpfn.classifier`` and ``.regressor``: ``MMPFNRegressor`` runs the same forward with a
    bar-distribution head, regressor.py:577-730); returns an ``uninstall()``.

    ``mode="model"``: the reference's engine keeps its serial per-estimator loop and only its ``.model`` is
    swapped (one B = 1 CUDA forward per estimator).  ``mode="engine"`` (default): the engine object itself is
    replaced by ``B200PluginEngine`` (all estimators in one batched pass) — what SURVEY.md section 7 step 1(i)
    describes.  Both leave every line of the reference's ``fit`` / ``predict_proba`` in charge; ``replay=False`` also
    keeps the reference's own per-member ``transform`` calls at predict time (``B200PluginEngine`` docstring).

    ``precision``: the layer precision of the swapped-in model — "bf16" (default), "fp16" (fp16 tensor-core operands:
    the type the reference itself autocasts to on CUDA, about 1/8 of bf16's distance from fp32) or "fp32" (the
    1e-5 parity mode); torch dtypes and the estimators' ``inference_precision`` spellings are accepted too."""
    from .classifier import precision_name
    precision = precision_name(precision)
    import mmpfn.models.mmpfn.classifier as C
    import mmpfn.models.mmpfn.regressor as R

    orig = C.create_inference_engine
    if getattr(orig, "_mmpfn_b200", False):
        return lambda: None
    orig_r = R.create_inference_engine

    def wrap(fn):
        @functools.wraps(fn)
        def create_inference_engine(**kw):
            engine = fn(**kw)
            dev = kw["device_"]
            if getattr(dev, "type", str(dev)) == "cuda" and hasattr(engine, "model"):
                if mode == "engine" and hasattr(engine, "preprocessors") and hasattr(engine, "X_trains"):
                    return B200PluginEngine(engine, device=dev, precision=precision, pos_emb_device=pos_emb_device,
                                            model_cls=model_cls, replay=replay)
                engine.model = convert(engine.model, device=dev, precision=precision, model_cls=model_cls,
                                       pos_emb_device=pos_emb_device)
            return engine
        create_inference_engine._mmpfn_b200 = True
        return create_inference_engine

    C.create_inference_engine = wrap(orig)
    R.create_inference_engine = wrap(orig_r)

    def uninstall():
        C.create_inference_engine = orig
        R.create_inference_engine = orig_r
    return uninstall
