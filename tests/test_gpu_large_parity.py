"""GPU parity at BASELINE.json's LARGE configs against vectors the REAL reference produced
(``oracle/make_golden_large.py`` -> ``tests/golden/large_*.npz``): 10 000-row context (configs[2]),
the 50 000-key item-attention axis (configs[3]), packed small tasks (configs[4]) and the full
8-estimator PAD-UFES classifier run (configs[1]).

Tolerances (BASELINE.json north_star): max-abs probability difference <= 1e-5 in fp32, <= 2e-3 in
bf16; argmax agreement is reported in full and every disagreeing row must be one the tolerance cannot
decide (reference top-2 margin below twice the measured deviation) — for these near-uniform random-init
posteriors the reference's OWN autocast-bf16 run flips 4 % of the rows (``ref_bf16_autocast.npz``)."""
import numpy as np
import pytest
import torch

from multimodalpfn_b200 import _lib
from multimodalpfn_b200.model import B200PerFeatureTransformer
from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
from tests import cases
from tests.cases import check_proba, load_golden, softmax_np, t

pytestmark = pytest.mark.gpu

P_TOL = {"fp32": 1e-5, "bf16": 2e-3}


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_ctx10k_vs_reference(precision):
    """configs[2] shape, one estimator (T = 42): context of 10 000 train rows, logits of 256 sampled test
    rows and the head-0 K/V of layers 0 / 11 against the reference's own cached forward."""
    c = cases.ctx10k_inputs()
    g = load_golden("large_ctx10k")
    geom = cases.CTX10K_GEOM
    sd = make_state_dict(geom, seed=cases.CTX10K_WSEED)
    model = B200PerFeatureTransformer(sd, geom, precision=precision, seed=0)
    ctx = model.fit_context(t(c["X_train"]), t(c["img_train"]), t(c["y_train"]))
    assert ctx.T == 42
    logits = model.predict_with_context(ctx, t(c["X_test"]), t(c["img_test"]))[0].cpu().numpy()
    n_cls = c["n_classes"]
    check_proba(softmax_np(logits[:, :n_cls] / 0.9), softmax_np(g["logits"][:, :n_cls] / 0.9), P_TOL[precision],
                f"ctx10k {precision}")
    rows = torch.as_tensor(cases.CTX10K_KV_ROWS)
    n_tr, L = ctx.n_train, geom.nlayers
    if precision == "fp32":
        kv = ctx.kv.view(torch.float32).view(L, 1, ctx.T, n_tr, 2, 32)
        k0, k11 = kv[0, 0][:, rows].cpu().numpy(), kv[-1, 0][:, rows].cpu().numpy()
        assert np.abs(k0 - g["kv_l0"]).max() < 2e-5
        assert np.abs(k11 - g["kv_l11"]).max() < 2e-4
        assert np.abs(logits - g["logits"]).max() < 2e-4
    else:
        Np = (n_tr + 63) // 64 * 64                      # per layer: K0 [T][Np][32] then V0^T [T][32][Np], bf16
        kv = ctx.kv.view(torch.bfloat16).view(L, 2, ctx.T * Np * 32)
        for li, key in ((0, "kv_l0"), (L - 1, "kv_l11")):
            k = kv[li, 0].view(ctx.T, Np, 32)[:, rows].float().cpu().numpy()
            v = kv[li, 1].view(ctx.T, 32, Np)[:, :, rows].permute(0, 2, 1).float().cpu().numpy()
            ref = g[key]                                 # [T, rows, 2, 32]
            assert np.abs(k - ref[:, :, 0]).max() < 0.06 and np.abs(v - ref[:, :, 1]).max() < 0.06, (li,)


@pytest.mark.parametrize("gain", ["g1", "g3"])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_layer50k_pass_vs_reference(precision, gain):
    """The 50 000-key axis of configs[3]: ONE layer (feature attention, item attention with 50 000 train
    rows as keys, MLP) on a [50 128 rows, T = 3] state; 64 train rows and 64 test rows of the output against
    the reference's own ``PerFeatureEncoderLayer`` modules (1042 key tiles accumulate per query).
    ``g1``: the reference's initialisation law.  ``g3``: scores nine times larger — a sharp softmax whose running
    reference moves; there bf16 OPERANDS alone (q, k rounded to 8 bits: |score| ~ 30 -> +-0.1 in the exponent)
    bound what any bf16 attention can reach, so bf16 is held to a loose bound and the kernel itself is checked
    against same-operand arithmetic in ``test_item_attention_50k_keys_sharp``."""
    geom = cases.LAYER50K_GEOM
    sd = make_state_dict(geom, seed=cases.LAYER50K_WSEED, qkv_gain=cases.LAYER50K_GAINS[gain])
    g = load_golden("large_layer50k_" + gain)
    n_tr, n_te, T = cases.LAYER50K_SHAPE
    model = B200PerFeatureTransformer(sd, geom, precision=precision, seed=0)
    state = torch.as_tensor(cases.layer_state(n_tr + n_te, T, seed=cases.LAYER50K_SSEED)).cuda()
    tr = state[None, :n_tr].contiguous()
    te = state[None, n_tr:].contiguous()
    bf = precision == "bf16"
    tr_b = tr.to(torch.bfloat16) if bf else None
    te_b = te.to(torch.bfloat16) if bf else None
    kv = model.alloc_kv(1, n_tr, T)
    model.layers(tr, tr_b, [(1, T)], n_tr, [kv])
    model.layers(te, te_b, [(1, T)], n_te, [kv], n_train=n_tr)
    out = torch.cat([tr[0], te[0]]).cpu().numpy()[cases.LAYER50K_ROWS]
    err = np.abs(out - g["out_rows"])
    print(f"[layer50k {gain} {precision}] max|err| train rows {err[:64].max():.3e}, test rows {err[64:].max():.3e}, "
          f"mean {err.mean():.2e} (LayerNorm-ed values, |x| up to {np.abs(g['out_rows']).max():.1f})")
    assert np.isfinite(out).all()
    tol = 2e-4 if not bf else (0.05 if gain == "g1" else 0.6)
    assert err.max() < tol, err.max()


def test_item_attention_50k_keys_sharp():
    """The bf16 item-attention kernel over 50 000 keys with scores spread over +-60 log2 units (the running
    reference moves, exponentials saturate against a stale reference and tiles are repeated), against fp32 torch
    on the SAME bf16 operands: what is left is the kernel's own error (P rounded to bf16, polynomial 2^x)."""
    lib = _lib.load()
    B, T, n_q, n_kv, scale = 1, 1, 256, 50_000, 3.0
    planes = B * T * 6
    qpad, kpad = 256, (n_kv + 63) // 64 * 64
    gen = torch.Generator().manual_seed(50)
    q = (torch.randn(planes, qpad, 32, generator=gen) * scale).cuda().to(torch.bfloat16)
    k = (torch.randn(planes, kpad, 32, generator=gen) * scale).cuda().to(torch.bfloat16)
    vt = torch.randn(planes, 32, kpad, generator=gen).cuda().to(torch.bfloat16)
    out = torch.full((B, n_q, T, 192), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.mmpfn_item_attention_bf16(q.data_ptr(), k.data_ptr(), vt.data_ptr(), B, T, n_q, qpad, n_kv, kpad, 0,
                                             out.data_ptr(), torch.cuda.current_stream().cuda_stream), "item_attention")
    torch.cuda.synchronize()
    err = 0.0
    for h in range(6):
        ref = torch.softmax(q[h, :n_q].float() @ k[h, :n_kv].float().T / 32 ** 0.5, dim=-1) @ vt[h, :, :n_kv].float().T
        err = max(err, float((out[0, :, 0, h * 32:(h + 1) * 32].float() - ref).abs().max()))
    print(f"[item attention, 50k keys, sharp] max|err| vs same-operand fp32: {err:.3e}")
    assert err < 0.03, err


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_packed_tasks_vs_reference(precision):
    """configs[4]: four independent 800/200-row tasks packed on the batch axis of every launch, each
    against the reference's model-level logits for that task alone."""
    g = load_golden("large_tasks4")
    geom = Geometry(mgm_heads=8, cap_heads=8)
    sd = make_state_dict(geom, seed=1)
    model = B200PerFeatureTransformer(sd, geom, precision=precision, seed=0)
    ds = [make_dataset("small_task", k) for k in range(4)]
    n_tr = len(ds[0]["y_train"])
    Xtr = torch.as_tensor(np.stack([d["X_train"] for d in ds])).cuda()
    Xte = torch.as_tensor(np.stack([d["X_test"] for d in ds])).cuda()
    ytr = torch.as_tensor(np.stack([d["y_train"].astype(np.float32) for d in ds])).cuda()
    img = torch.as_tensor(np.concatenate([np.concatenate([d["img_train"], d["img_test"]]) for d in ds])).cuda()
    tok = model.stem_image(img)
    tok = tok.view(4, -1, tok.shape[1], tok.shape[2])
    ctx = model.fit_context(Xtr, None, ytr, X_all=torch.cat([Xtr, Xte], 1), img_tok_train=tok[:, :n_tr].contiguous())
    lg = model.predict_with_context(ctx, Xte, None, img_tok_test=tok[:, n_tr:].contiguous()).cpu().numpy()
    for k in range(4):
        n_cls = ds[k]["n_classes"]
        check_proba(softmax_np(lg[k][:, :n_cls] / 0.9), softmax_np(g["logits"][k][:, :n_cls] / 0.9), P_TOL[precision],
                    f"task {k} {precision}")
        if precision == "fp32":
            assert np.abs(lg[k] - g["logits"][k]).max() < 5e-5


@pytest.mark.parametrize("path", ["multi_group", "per_group"])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_clf8_pad_ufes_vs_reference(precision, path):
    """configs[1] in full: the tensors that crossed the model boundary of the reference's 8-estimator
    ``MMPFNClassifier`` run on the PAD-UFES shape (its own preprocessing: 4 x F'=36 -> T=27, 4 x F'=22 ->
    T=20), through the multi-group pass bench.py times and through one pass per group; per-estimator logits
    (fp32) and the final probabilities against the reference's."""
    from multimodalpfn_b200.engine import proba_from_logits
    g = load_golden("large_clf8_pad_ufes")
    geom = Geometry(mgm_heads=8, cap_heads=8)
    sd = make_state_dict(geom, seed=1)
    d = make_dataset("pad_ufes", 0)
    n_est, n_tr = int(g["n_estimators"]), len(d["y_train"])
    model = B200PerFeatureTransformer(sd, geom, precision=precision, seed=0)
    img = torch.as_tensor(np.concatenate([d["img_train"], d["img_test"]])).cuda()
    by_f = {}
    for e in range(n_est):
        by_f.setdefault(g[f"X_full_{e}"].shape[1], []).append(e)
    assert sorted(by_f) == [22, 36]
    logits = [None] * n_est
    groups = []
    for F, es in sorted(by_f.items()):
        Xb = torch.as_tensor(np.stack([g[f"X_full_{e}"] for e in es])).cuda()
        yb = torch.as_tensor(np.stack([g[f"y_train_{e}"] for e in es])).cuda()
        groups.append((es, Xb, yb))
    if path == "multi_group":
        tok = model.stem_image(img)
        specs = [dict(X_train=Xb[:, :n_tr].contiguous(), y_train=yb, X_all=Xb, img_tok_train=tok[:n_tr].contiguous())
                 for _, Xb, yb in groups]
        ctxs = model.fit_contexts(specs)
        outs = model.predict_with_contexts(ctxs, [Xb[:, n_tr:].contiguous() for _, Xb, _ in groups],
                                           img_tok_test=tok[n_tr:].contiguous())
    else:
        outs = [model.forward_batch(Xb, img, yb) for _, Xb, yb in groups]
    for (es, _, _), out in zip(groups, outs):
        for i, e in enumerate(es):
            logits[e] = out[i]
    if precision == "fp32":
        for e in range(n_est):
            assert np.abs(logits[e].cpu().numpy() - g[f"logits_{e}"]).max() < 5e-5
    proba = proba_from_logits(torch.stack(logits), [g[f"class_perm_{e}"] for e in range(n_est)],
                              n_classes=int(g["n_classes"]), class_counts=g["class_counts"])
    check_proba(proba, g["proba"], P_TOL[precision], f"clf8 {precision} {path}")
    assert np.allclose(proba.sum(1), 1.0, atol=1e-6)
