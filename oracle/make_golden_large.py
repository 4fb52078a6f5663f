"""ORACLE support: golden vectors at BASELINE.json's LARGE configs, produced by the REAL reference.

    PYTHONHASHSEED=0 python -m oracle.make_golden_large [case ...]

The reference's own CPU path materialises the ``[batch, q, k, heads]`` attention logits
(``model/multi_head_attention.py:718-729``) and runs a T^2 diagnostic loop
(``model/transformer.py:809-813``), so the 10k/50k-row shapes are only reachable with the
reference's own memory knob (``reset_save_peak_mem_factor``, ``model/memory.py:78-97``), the
diagnostic block removed (``ref_compat.without_diagnostic_loop``: every other line of ``_forward``
stays the reference's) and, because test rows are independent of one another
(``model/layer.py:346-358``; SURVEY.md section 8(e)), a SAMPLE of the test rows.  Inputs and weights are
regenerated from seeds at test time (``multimodalpfn_b200.synth``, ``tests/cases.py``); only the
reference's outputs are stored.

Cases
* ``ctx10k``  — configs[2] shape: 10 000 train rows, 64 features + fingerprint-like column
  (F'=65 -> T=42 with MGM8+CAP8), [N,2,768] image+text embeddings, ONE estimator: the reference's own
  cached form (``cache_trainset_representation``; equal to the joint forward, ``model_*.npz`` hold both):
  train call -> per-layer head-0 K/V cache (layers 0 and 11 kept for 16 rows), then logits of 256
  sampled test rows.
* ``layer50k`` — the 50 000-key axis of configs[3]: ONE ``PerFeatureEncoderLayer`` (the loaded reference
  module) on a [50 000 + 128 rows, T=3] state, at the reference's own qkv initialisation (``g1``) and with
  scores nine times larger (``g3``, a sharp softmax), queries chunked through the reference's own
  ``MultiHeadAttention`` (x = a chunk of rows, x_kv = all train rows) — checked here against
  ``layer.forward`` at a small shape first.
* ``tasks4``  — configs[4]: four independent 800/200-row tasks, model-level logits each.
* ``clf8``    — configs[1] in full: the reference ``MMPFNClassifier`` with 8 estimators on the PAD-UFES
  shape; boundary tensors, per-estimator logits, probabilities.
* ``bf16ref`` — the reference's OWN autocast-bf16 deviation from its fp32 (same fp32-drawn positional
  embeddings injected; SURVEY.md gotchas 8, 9) on the cases the bf16 tests gate.
"""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from multimodalpfn_b200.synth import Geometry, make_checkpoint_config, make_dataset, make_state_dict  # noqa: E402
from oracle import ref_compat  # noqa: E402
from tests import cases  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _load(geom, seed, **kw):
    sd = make_state_dict(geom, seed=seed, **kw)
    model, _ = ref_compat.load_reference_model(
        sd, make_checkpoint_config(geom), mixer_type=geom.mixer_type, mgm_heads=geom.mgm_heads,
        cap_heads=geom.cap_heads, features_per_group=geom.features_per_group, model_seed=0)
    return model, sd


def _call(model, x, img, y, sep):
    with torch.inference_mode():
        return model(None, None if x is None else torch.as_tensor(x)[:, None],
                     None if img is None else torch.as_tensor(img), None if y is None else torch.as_tensor(y),
                     only_return_standard_out=True, categorical_inds=[], single_eval_pos=sep)


# ---------------------------------------------------------------------------------------------------
def run_ctx10k():
    c = cases.ctx10k_inputs()
    geom = cases.CTX10K_GEOM
    model, _ = _load(geom, cases.CTX10K_WSEED)
    n_tr = len(c["y_train"])
    T = (c["X_train"].shape[1] + 1) // 2 + geom.cap_heads + 1
    model.reset_save_peak_mem_factor(T)            # one token column per chunk: 10k x 10k x 6 logits = 2.4 GB
    model.cache_trainset_representation = True
    t0 = time.time()
    with ref_compat.without_diagnostic_loop():
        _call(model, c["X_train"], c["img_train"], c["y_train"], n_tr)
        print(f"ctx10k: train call {time.time() - t0:.0f} s", flush=True)
        layers = model.transformer_encoder.layers
        kv = [l.self_attn_between_items._kv_cache.squeeze(-2) for l in layers]      # [T, Ntr, 2, 32]
        rows = cases.CTX10K_KV_ROWS
        out = dict(kv_l0=kv[0][:, rows].numpy().copy(), kv_l11=kv[-1][:, rows].numpy().copy())
        model.reset_save_peak_mem_factor(None)
        lg = _call(model, c["X_test"], c["img_test"], None, None).squeeze(1).numpy()
    out["logits"] = lg
    model.empty_trainset_representation_cache()
    np.savez_compressed(os.path.join(OUT, "large_ctx10k.npz"), **out)
    print(f"ctx10k: logits {lg.shape}, T={T}, {time.time() - t0:.0f} s total", flush=True)


# ---------------------------------------------------------------------------------------------------
def ref_layer_chunked(layer, state, n_train, q_chunk):
    """``PerFeatureEncoderLayer.forward`` (model/layer.py:272-457) with the item attention's QUERIES
    chunked: the same three sublayers and LayerNorms, each one the loaded reference module; a chunk of
    query rows against x_kv = all train rows is the reference's own cross-attention call form
    (layer.py:346-358 uses it for the test rows)."""
    st = state.clone()
    st = layer.self_attn_between_features(st, add_input=True, allow_inplace=True)           # layer.py:332-339
    st = layer.layer_norms[0](st, allow_inplace=True)
    S = st.shape[1]
    src = st[:, :n_train].transpose(1, 2)
    new = torch.empty_like(st)
    a = 0
    while a < S:
        b = min(a + q_chunk, S if a >= n_train else n_train)
        x = st[:, a:b].transpose(1, 2).clone()
        if a < n_train:      # layer.py:363-372 (train rows: all six heads' own K/V)
            o = layer.self_attn_between_items(x, src, add_input=True, allow_inplace=True)
        else:                # layer.py:346-358 (test rows: head-0 K/V for every query head)
            o = layer.self_attn_between_items(x, src, add_input=True, allow_inplace=True, reuse_first_head_kv=True)
        new[:, a:b] = o.transpose(1, 2)
        a = b
    st = layer.layer_norms[1](new, allow_inplace=True)
    st = layer.mlp(st, add_input=True, allow_inplace=True)                                   # layer.py:410-424
    return layer.layer_norms[2](st, allow_inplace=True)


def run_layer50k(which=None):
    for name in ([which] if which else list(cases.LAYER50K_GAINS)):
        _run_layer50k(name)


def _run_layer50k(name):
    geom = cases.LAYER50K_GEOM
    model, _ = _load(geom, cases.LAYER50K_WSEED, qkv_gain=cases.LAYER50K_GAINS[name])
    layer = model.transformer_encoder.layers[0]
    with torch.inference_mode():
        # harness == layer.forward at a small shape (bit for bit)
        small = torch.as_tensor(cases.layer_state(300, 3, seed=5))[None]
        want = layer(small.clone(), single_eval_pos=200)
        got = ref_layer_chunked(layer, small, 200, q_chunk=64)
        err = (want - got).abs().max().item()
        assert err <= 1e-6, err
        print(f"layer50k: chunked harness vs layer.forward at 200+100 rows: {err:.1e}", flush=True)
        n_tr, n_te, T = cases.LAYER50K_SHAPE
        state = torch.as_tensor(cases.layer_state(n_tr + n_te, T, seed=cases.LAYER50K_SSEED))[None]
        t0 = time.time()
        out = ref_layer_chunked(layer, state, n_tr, q_chunk=1024)[0]
    rows = cases.LAYER50K_ROWS
    np.savez_compressed(os.path.join(OUT, f"large_layer50k_{name}.npz"), out_rows=out[rows].numpy().copy())
    print(f"layer50k {name}: {time.time() - t0:.0f} s", flush=True)


# ---------------------------------------------------------------------------------------------------
def run_tasks4():
    geom = Geometry(mgm_heads=8, cap_heads=8)
    model, _ = _load(geom, 1)
    outs = []
    with ref_compat.without_diagnostic_loop():
        for k in range(4):
            d = make_dataset("small_task", k)
            X = np.concatenate([d["X_train"], d["X_test"]])
            img = np.concatenate([d["img_train"], d["img_test"]])
            outs.append(_call(model, X, img, d["y_train"].astype(np.float32), len(d["y_train"])).squeeze(1).numpy())
    np.savez_compressed(os.path.join(OUT, "large_tasks4.npz"), logits=np.stack(outs))
    print("tasks4:", np.stack(outs).shape, flush=True)


# ---------------------------------------------------------------------------------------------------
def run_clf8():
    geom = Geometry(mgm_heads=8, cap_heads=8)
    sd = make_state_dict(geom, seed=1)
    ref_compat.install()
    path = os.path.join("/tmp", f"mmpfn_b200_clf8_{os.getpid()}.ckpt")
    torch.save({"state_dict": {k: torch.as_tensor(v) for k, v in sd.items()}, "config": make_checkpoint_config(geom)}, path)
    from mmpfn.models.mmpfn import MMPFNClassifier
    from mmpfn.models.mmpfn.model.transformer import PerFeatureTransformer
    d = make_dataset("pad_ufes", 0)
    clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=8, cap_heads=8, features_per_group=2, n_estimators=8,
                          model_path=path, device="cpu", ignore_pretraining_limits=True, random_state=0)
    clf.fit(d["X_train"], d["img_train"], d["y_train"])
    rec = []
    t0 = time.time()
    with ref_compat.without_diagnostic_loop():
        inner = PerFeatureTransformer._forward

        def spy(self, x, image, y, **k):
            xin, yin = x.clone(), y.clone()
            o = inner(self, x, image, y, **k)
            rec.append((xin[:, 0].numpy().copy(), yin.numpy().copy(), o.squeeze(1).numpy().copy()))
            return o
        PerFeatureTransformer._forward = spy
        proba = clf.predict_proba(d["X_test"], d["img_test"])
    out = dict(proba=proba, n_estimators=8, n_classes=clf.n_classes_, class_counts=clf.class_counts_)
    for e, ((x, y, lg), cfg) in enumerate(zip(rec, clf.executor_.ensemble_configs)):
        out[f"X_full_{e}"] = x.astype(np.float32)
        out[f"y_train_{e}"] = y.astype(np.float32)
        out[f"logits_{e}"] = lg
        out[f"class_perm_{e}"] = (np.arange(clf.n_classes_) if cfg.class_permutation is None
                                  else np.asarray(cfg.class_permutation))
    np.savez_compressed(os.path.join(OUT, "large_clf8_pad_ufes.npz"), **cases.pack_tables(out))
    print(f"clf8: proba {proba.shape}, F' {[r[0].shape[1] for r in rec]}, {time.time() - t0:.0f} s", flush=True)


# ---------------------------------------------------------------------------------------------------
class _fp32_randn:
    """Positional noise drawn in fp32 whatever dtype autocast hands ``add_embeddings``
    (``model/transformer.py:926-931``; SURVEY.md gotcha 8: a 16-bit ``randn`` is a different stream)."""

    def __enter__(self):
        self._orig = torch.randn

        def randn(*a, dtype=None, **k):
            t = self._orig(*a, dtype=torch.float32, **k)
            return t if dtype is None else t.to(dtype)
        torch.randn = randn

    def __exit__(self, *a):
        torch.randn = self._orig


def run_bf16ref():
    """fp32 vs autocast-bf16 logits of the reference itself on the cases whose bf16 parity is gated."""
    from oracle.make_golden import MODEL_CASES, mutate_inputs
    out = {}
    todo = [("stress_tiny", None), ("mgmcap_tiny", None), ("mgmcap_8x8_small", None)]
    for name, _ in todo:
        gkw, ds, wseed, mut = MODEL_CASES[name]
        geom = Geometry(**{k: v for k, v in gkw.items() if v is not None or k == "cap_heads"})
        extra = dict(residual_std=0.2, decoder_gain=20.0) if mut == "stress" else {}
        model, _ = _load(geom, wseed, **extra)
        d = make_dataset(ds, 0)
        X = np.concatenate([d["X_train"], d["X_test"]])
        img = np.concatenate([d["img_train"], d["img_test"]])
        X, img = mutate_inputs(mut, X, img)
        y = d["y_train"].astype(np.float32)
        with ref_compat.without_diagnostic_loop(), _fp32_randn():
            f32 = _call(model, X, img, y, len(y)).squeeze(1).float().numpy()
            with torch.autocast("cpu", dtype=torch.bfloat16):
                b16 = _call(model, X, img, y, len(y)).squeeze(1).float().numpy()
        out[name + "_bf16"] = b16
        n_cls = d["n_classes"]

        def proba(z):
            z = z[:, :n_cls] / 0.9
            e = np.exp(z - z.max(1, keepdims=True))
            return e / e.sum(1, keepdims=True)
        dp = np.abs(proba(b16) - proba(f32)).max()
        agree = (proba(b16).argmax(1) == proba(f32).argmax(1)).mean()
        out[name + "_dp"] = dp
        out[name + "_argmax_agree"] = agree
        print(f"bf16ref {name}: reference autocast-bf16 vs its fp32: max|dp| {dp:.3e}, argmax agreement {agree:.4f}", flush=True)
    np.savez_compressed(os.path.join(OUT, "ref_bf16_autocast.npz"), **out)


CASES = dict(tasks4=run_tasks4, bf16ref=run_bf16ref, clf8=run_clf8, layer50k=run_layer50k,
             layer50k_g1=lambda: run_layer50k("g1"), layer50k_g3=lambda: run_layer50k("g3"), ctx10k=run_ctx10k)


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(int(os.environ.get("MMPFN_GOLDEN_THREADS", "8")))
    assert os.environ.get("PYTHONHASHSEED") == "0", "run with PYTHONHASHSEED=0 (SURVEY.md gotcha 3)"
    for name in (sys.argv[1:] or list(CASES)):
        CASES[name]()


if __name__ == "__main__":
    main()
