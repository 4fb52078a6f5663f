"""Tasks of different sizes in one pass: per-entry row counts in the item attention (both precisions), the stem
statistics, the token assembly and the layer passes give every entry exactly what a run over that entry alone gives,
and the pad rows stay zero (include/mmpfn_b200.h, "ragged" passes)."""

import numpy as np
import pytest
import torch

from multimodalpfn_b200 import _lib
from multimodalpfn_b200.classifier import MMPFNClassifier
from multimodalpfn_b200.model import B200PerFeatureTransformer
from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
from multimodalpfn_b200.tasks import predict_proba_tasks

pytestmark = pytest.mark.gpu

KV_COUNTS = [1, 47, 48, 49, 130]      # one key, around the 48-key tile, several tiles
Q_COUNTS = [200, 1, 129, 77, 200]
CAP = 200


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _i32(a):
    return torch.tensor(a, dtype=torch.int32, device="cuda")


def _pad8(n):
    return (n + 7) // 8 * 8


def _bf16_inputs(shared, T, Sq_pad, Skv_pad, seed):
    B = len(KV_COUNTS)
    g = torch.Generator().manual_seed(seed)
    planes, kv_planes = B * T * 6, (B * T if shared else B * T * 6)
    q = torch.randn(planes, Sq_pad, 32, generator=g).cuda().to(torch.bfloat16)
    k = torch.randn(kv_planes, Skv_pad, 32, generator=g).cuda().to(torch.bfloat16)
    vt = torch.randn(kv_planes, 32, Skv_pad, generator=g).cuda().to(torch.bfloat16)
    for b in range(B):       # rows past an entry's counts are zero, as the layers keep them
        q[b * 6 * T:(b + 1) * 6 * T, Q_COUNTS[b]:] = 0
        per_kv = T if shared else 6 * T
        k[b * per_kv:(b + 1) * per_kv, KV_COUNTS[b]:] = 0
        vt[b * per_kv:(b + 1) * per_kv, :, KV_COUNTS[b]:] = 0
    return q, k, vt


@pytest.mark.parametrize("shared", [0, 1])
def test_item_attention_bf16_per_entry_counts(shared):
    """Train form (own K/V per head) and test form (head-0 K/V shared by the six heads, stacked on the tile rows when
    that saves tiles: Sq_pad = 200 gives 10 tiles of 128 instead of 12)."""
    lib = _lib.load()
    B, T = len(KV_COUNTS), 2
    Sq_pad = CAP if shared else 256
    Skv_pad = 256
    q, k, vt = _bf16_inputs(shared, T, Sq_pad, Skv_pad, seed=17 + shared)
    out = torch.full((B, CAP, T, 192), float("nan"), dtype=torch.bfloat16, device="cuda")
    q_len, kv_len = _i32(Q_COUNTS), _i32(KV_COUNTS)       # held: the kernel reads them after the call returns
    _lib.check(lib.mmpfn_item_attention_bf16_ragged(q.data_ptr(), k.data_ptr(), vt.data_ptr(), B, T, CAP, Sq_pad, CAP,
                                                    Skv_pad, shared, q_len.data_ptr(), kv_len.data_ptr(),
                                                    out.data_ptr(), _stream()),
               "item_attention_bf16_ragged")
    per_kv = T if shared else 6 * T
    err = 0.0
    for b in range(B):
        nq, nkv = Q_COUNTS[b], KV_COUNTS[b]
        qp, kp = _pad8(nq), (nkv + 63) // 64 * 64
        qa = q[b * 6 * T:(b + 1) * 6 * T, :qp].contiguous()
        ka = torch.zeros(per_kv, kp, 32, dtype=torch.bfloat16, device="cuda")
        va = torch.zeros(per_kv, 32, kp, dtype=torch.bfloat16, device="cuda")
        ka[:, :nkv] = k[b * per_kv:(b + 1) * per_kv, :nkv]
        va[:, :, :nkv] = vt[b * per_kv:(b + 1) * per_kv, :, :nkv]
        alone = torch.full((1, nq, T, 192), float("nan"), dtype=torch.bfloat16, device="cuda")
        _lib.check(lib.mmpfn_item_attention_bf16(qa.data_ptr(), ka.data_ptr(), va.data_ptr(), 1, T, nq, qp, nkv, kp,
                                                 shared, alone.data_ptr(), _stream()), "item_attention_bf16")
        torch.cuda.synchronize()
        assert torch.equal(out[b, :nq], alone[0]), (b, nq, nkv)
        assert torch.equal(out[b, nq:], torch.zeros_like(out[b, nq:])), b
        for t in range(T):
            for h in range(6):
                kvp = t if shared else t * 6 + h
                ref = torch.softmax(qa[t * 6 + h, :nq].float() @ ka[kvp, :nkv].float().T / 32 ** 0.5, dim=-1) \
                    @ va[kvp, :, :nkv].float().T
                err = max(err, float((out[b, :nq, t, h * 32:(h + 1) * 32].float() - ref).abs().max()))
    assert err < 0.03, err


@pytest.mark.parametrize("shared", [0, 1])
def test_item_attention_f32_per_entry_counts(shared):
    lib = _lib.load()
    B, T = len(KV_COUNTS), 2
    g = torch.Generator().manual_seed(5 + shared)
    q = torch.randn(B, CAP, T, 192, generator=g).cuda()
    kv_shape = (B, T, CAP, 32) if shared else (B, CAP, T, 192)
    k, v = torch.randn(*kv_shape, generator=g).cuda(), torch.randn(*kv_shape, generator=g).cuda()
    for b in range(B):       # never read: poison
        q[b, Q_COUNTS[b]:] = float("nan")
        if shared:
            k[b, :, KV_COUNTS[b]:] = float("nan")
            v[b, :, KV_COUNTS[b]:] = float("nan")
        else:
            k[b, KV_COUNTS[b]:] = float("nan")
            v[b, KV_COUNTS[b]:] = float("nan")
    out = torch.full((B, CAP, T, 192), float("nan"), device="cuda")
    q_len, kv_len = _i32(Q_COUNTS), _i32(KV_COUNTS)       # held: the kernel reads them after the call returns
    _lib.check(lib.mmpfn_item_attention_f32(q.data_ptr(), k.data_ptr(), v.data_ptr(), B, T, CAP, CAP, shared,
                                            q_len.data_ptr(), kv_len.data_ptr(), out.data_ptr(), _stream()),
               "item_attention_f32")
    for b in range(B):
        nq, nkv = Q_COUNTS[b], KV_COUNTS[b]
        qa = q[b:b + 1, :nq].contiguous()
        ka = (k[b:b + 1, :, :nkv] if shared else k[b:b + 1, :nkv]).contiguous()
        va = (v[b:b + 1, :, :nkv] if shared else v[b:b + 1, :nkv]).contiguous()
        alone = torch.full((1, nq, T, 192), float("nan"), device="cuda")
        _lib.check(lib.mmpfn_item_attention_f32(qa.data_ptr(), ka.data_ptr(), va.data_ptr(), 1, T, nq, nkv, shared,
                                                None, None, alone.data_ptr(), _stream()), "item_attention_f32")
        torch.cuda.synchronize()
        assert torch.equal(out[b, :nq], alone[0]), (b, nq, nkv)
        assert torch.equal(out[b, nq:], torch.zeros_like(out[b, nq:])), b
        for t in range(T):
            for h in range(6):
                kk = ka[0, t] if shared else ka[0, :, t, h * 32:(h + 1) * 32]
                vv = va[0, t] if shared else va[0, :, t, h * 32:(h + 1) * 32]
                ref = torch.softmax(qa[0, :, t, h * 32:(h + 1) * 32].double() @ kk.double().T / 32 ** 0.5, -1) @ vv.double()
                assert torch.allclose(alone[0, :, t, h * 32:(h + 1) * 32].double(), ref, atol=1e-5), (b, t, h)


def _model(precision, seed=5):
    geom = Geometry(mgm_heads=2, cap_heads=4)
    return B200PerFeatureTransformer(make_state_dict(geom, seed=seed), geom, precision=precision, seed=0), geom


def test_tab_fit_per_entry_equals_alone():
    model, _ = _model("bf16")
    rng = np.random.default_rng(3)
    rows, trains, S, F = [300, 31, 1, 200, 2], [250, 30, 1, 100, 1], 300, 7
    X = rng.standard_normal((len(rows), S, F)).astype(np.float32)
    X[:, :, 2] = 4.0                              # constant column
    X[:, ::3, 4] = np.nan                         # NaN cells
    X[1, :, 5] = np.nan                           # an all-NaN column
    X[:, 0, 6] = 1e6                              # an outlier
    for b, n in enumerate(rows):
        X[b, n:] = 0.0
    Xd = torch.from_numpy(X).cuda()
    got = model._stem_tab_fit_ragged(Xd, _i32(rows), _i32(trains))
    for b, (n, ntr) in enumerate(zip(rows, trains)):
        alone = model.stem_tab_fit(Xd[b:b + 1, :n].contiguous(), ntr)
        assert torch.equal(got[b:b + 1].nan_to_num(123.0), alone.nan_to_num(123.0)), b


def _entries(model, rng):
    """Entries of three token counts (no table / 5 / 13 features, with and without image tokens) and ragged rows."""
    spec = [(None, 1, 61, 7), (5, 0, 200, 33), (5, 0, 97, 1), (13, 1, 130, 40), (13, 1, 47, 12), (13, 0, 150, 9)]
    img_rows = sum(ntr + nte for F, ni, ntr, nte in spec if ni)
    tok = model.stem_image(torch.from_numpy(rng.standard_normal((img_rows, 1, 768)).astype(np.float32)).cuda())
    out, row = [], 0
    for F, ni, ntr, nte in spec:
        X = None if F is None else rng.standard_normal((ntr + nte, F)).astype(np.float32)
        if X is not None:
            X[::4, 1] = np.nan
        y = rng.integers(0, 3, ntr)
        y[:3] = [0, 1, 2]
        out.append(dict(X=X, y=y, n_train=ntr, n_test=nte, tok=tok if ni else None, tok_row=row, n_tok=ni))
        row += (ntr + nte) if ni else 0
    return out


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_ragged_pass_equals_each_entry_alone(precision):
    model, _ = _model(precision)
    entries = _entries(model, np.random.default_rng(11))
    assert len({model.entry_tokens(None if e["X"] is None else e["X"].shape[1], e["n_tok"]) for e in entries}) >= 3
    states = []
    got = model.forward_ragged(entries, final_states=states)
    for j, e in enumerate(entries):
        ntr = e["n_train"]
        X_all = None if e["X"] is None else torch.from_numpy(e["X"])[None].cuda()
        tok_tr = tok_te = None
        if e["tok"] is not None:
            tok_tr = e["tok"][e["tok_row"]:e["tok_row"] + ntr].contiguous()
            tok_te = e["tok"][e["tok_row"] + ntr:e["tok_row"] + ntr + e["n_test"]].contiguous()
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        y = torch.from_numpy(e["y"].astype(np.float32))[None].cuda()
        ctx = model.fit_context(None if X_all is None else X_all[:, :ntr].contiguous(), None, y, X_all=X_all,
                                img_tok_train=tok_tr, check=False, nan_flag=flag)
        alone = model.predict_with_context(ctx, None if X_all is None else X_all[:, ntr:].contiguous(), None,
                                           img_tok_test=tok_te, nan_flag=flag)
        assert torch.equal(got[j], alone[0]), (precision, j, float((got[j] - alone[0]).abs().max()))
    # the pad rows of every entry are exactly zero after the 12 layers, train and test pass
    assert len(states) >= 6
    n_seg = len(states) // 2
    for phase, part in (("n_train", states[:n_seg]), ("n_test", states[n_seg:])):
        for v, js in part:
            for k, j in enumerate(js):
                pad = v[k, entries[j][phase]:]
                assert torch.equal(pad, torch.zeros_like(pad)), (phase, j)


def _mixed_tasks():
    """Twelve seeded tasks cut from synth datasets: 30..900 train rows, one task with a single test row, 5..40
    features with NaN columns, one embedding, two (image + text), none, and one task with embeddings only."""
    rng = np.random.default_rng(2024)
    base = make_dataset("small_task", 7)                # 800 + 200 rows, 32 features, one embedding
    X = np.concatenate([base["X_train"], base["X_test"]])
    X = np.concatenate([X, X[:, :8] * 0.5 + 1.0], axis=1)      # 40 columns
    img = np.concatenate([base["img_train"], base["img_test"]])
    y = np.concatenate([base["y_train"], base["y_test"]])
    spec = [  # n_train, n_test, n_features, embeddings (0, 1, 2 = image + text, -1 = embeddings only)
        (30, 11, 5, 1), (47, 1, 6, 0), (61, 20, 9, 2), (96, 40, 12, 1), (130, 13, 17, -1), (200, 50, 21, 0),
        (257, 64, 25, 1), (333, 30, 29, 2), (401, 99, 33, 1), (577, 123, 37, 0), (750, 150, 40, 1), (900, 7, 40, 2)]
    tasks = []
    for n_tr, n_te, F, ne in spec:
        rows = rng.permutation(len(X))[:n_tr + n_te]
        cols = rng.permutation(X.shape[1])[:F]
        Xt = X[rows][:, cols].copy()
        Xt[rng.random(len(rows)) < 0.2, 0] = np.nan           # a column with NaN cells
        yt = y[rows].copy()
        yt[:3] = [0, 1, 2]
        if ne == 0:
            it = None
        elif ne == 2:
            it = np.stack([img[rows, 0], img[rng.permutation(len(X))[:len(rows)], 0]], axis=1)
        else:
            it = img[rows]
        tasks.append(dict(X_train=None if ne == -1 else Xt[:n_tr], X_test=None if ne == -1 else Xt[n_tr:],
                          y_train=yt[:n_tr], img_train=None if it is None else it[:n_tr],
                          img_test=None if it is None else it[n_tr:]))
    return tasks


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_mixed_tasks_equal_one_by_one(precision):
    tasks = _mixed_tasks()
    # more than MMPFN_MAX_SEGMENTS token counts (before the members' preprocessing): several passes
    assert len({(t["X_train"] is None and -1 or (t["X_train"].shape[1] + 1) // 2, t["img_train"] is None)
                for t in tasks}) > 8
    model, _ = _model(precision)
    packed = predict_proba_tasks(model, tasks, n_estimators=4, random_state=0)
    assert sorted(packed) == list(range(len(tasks)))
    for i, t in enumerate(tasks):
        clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=2, cap_heads=4, features_per_group=2, n_estimators=4,
                              model_path=model, device="cuda", inference_precision=precision,
                              ignore_pretraining_limits=True, random_state=0)
        clf.fit(t["X_train"], t["img_train"], t["y_train"])
        one = clf.predict_proba(t["X_test"], t["img_test"])
        assert packed[i].shape == one.shape
        assert np.array_equal(packed[i], one), (precision, i, np.abs(packed[i] - one).max())
