"""Packed regression tasks: ``mmpfn_bar_tail_tasks`` against ``mmpfn_bar_tail`` run on each task alone (bit for bit)
and the float64 oracle, regression entries in ragged passes against a forward over each entry alone, and
``predict_regression_tasks`` against one ``MMPFNRegressor`` per task (bit for bit)."""
import numpy as np
import pytest
import torch

from multimodalpfn_b200 import _lib
from multimodalpfn_b200.model import B200PerFeatureTransformer
from multimodalpfn_b200.regressor import MMPFNRegressor, bar_tail_device, bar_tail_tasks_device
from multimodalpfn_b200.synth import Geometry, make_state_dict
from multimodalpfn_b200.tasks import predict_regression_tasks
from tests.test_gpu_ragged import _mixed_tasks
from tests.test_gpu_regressor import ALL, QS, SHAPES, _check, _maps, _oracle

pytestmark = pytest.mark.gpu

ROWS = [1, 7, 64, 300, 33]
PAD = (5, 3)                    # NaN rows before and after each task's slice of its allocation


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _tasks_inputs(K, n_est, seed, rows=ROWS, with_cancel=True):
    """Per task: logits in their own NaN-padded allocation, border maps, cancel masks (odd tasks none) and G."""
    rng = np.random.default_rng(seed)
    out = []
    for t, S in enumerate(rows):
        b, s, cancel, G = _maps(K, n_est, seed + 7 * t)
        if t % 2 == 1 or not with_cancel:
            cancel = np.zeros_like(cancel)
        lg = (rng.normal(0, 2.5, (n_est, S, K)) - 0.5 * np.linspace(-3, 3, K)[None, None] ** 2).astype(np.float32)
        buf = torch.full((n_est, PAD[0] + S + PAD[1], K), float("nan"), device="cuda")
        buf[:, PAD[0]:PAD[0] + S] = torch.from_numpy(lg).cuda()
        out.append(dict(logits=lg, buf=buf, b=b, s=s, cancel=cancel, G=G, S=S))
    return out


def _dev(a, dtype=None):
    return torch.as_tensor(np.ascontiguousarray(a), device="cuda", dtype=dtype)


def _run_tasks(tasks, temperature, avg, null_cancel, outputs=ALL):
    views = [[tk["buf"][e, PAD[0]:PAD[0] + tk["S"]] for e in range(tk["buf"].shape[0])] for tk in tasks]
    cancel = None if null_cancel else _dev(np.stack([tk["cancel"] for tk in tasks]).astype(np.uint8))
    out = bar_tail_tasks_device(views, _dev(np.stack([tk["b"] for tk in tasks])),
                                _dev(np.stack([tk["s"] for tk in tasks])), cancel,
                                _dev(np.stack([tk["G"] for tk in tasks]).astype(np.float32)),
                                softmax_temperature=temperature, average_before_softmax=avg,
                                quantiles=torch.tensor(QS, dtype=torch.float32, device="cuda"), outputs=outputs)
    ro = out.pop("row_offset")
    return {k: v.cpu().numpy() for k, v in out.items()}, ro


def _run_one(tk, temperature, avg, null_cancel, outputs=ALL):
    lg = tk["buf"][:, PAD[0]:PAD[0] + tk["S"]].contiguous()
    out = bar_tail_device(lg, _dev(tk["b"]), _dev(tk["s"]), None if null_cancel else _dev(tk["cancel"].astype(np.uint8)),
                          _dev(tk["G"].astype(np.float32)), softmax_temperature=temperature,
                          average_before_softmax=avg, quantiles=torch.tensor(QS, dtype=torch.float32, device="cuda"),
                          outputs=outputs)
    return {k: v.cpu().numpy() for k, v in out.items()}


def _same(a, b):
    """Bit for bit (NaN payloads and signed zeros included)."""
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _slice(got, r0, r1):
    return {k: (v[:, r0:r1] if k == "quantiles" else v[r0:r1]) for k, v in got.items()}


@pytest.mark.parametrize("K,n_est", [(64, 1), (64, 3), (64, 8), (5000, 1), (5000, 3), (5000, 8)])
@pytest.mark.parametrize("temperature", [1.0, 0.9])
@pytest.mark.parametrize("avg", [False, True])
def test_tail_tasks_equal_each_task_alone(K, n_est, temperature, avg):
    null_cancel = n_est == 1            # one estimator: no power transform, no cancelled bucket -> the NULL case
    tasks = _tasks_inputs(K, n_est, K + n_est, with_cancel=not null_cancel)
    got, ro = _run_tasks(tasks, temperature, avg, null_cancel)
    assert list(ro) == list(np.concatenate([[0], np.cumsum(ROWS)]))
    for t, tk in enumerate(tasks):
        part = _slice(got, ro[t], ro[t + 1])
        one = _run_one(tk, temperature, avg, null_cancel)
        for k in ALL:
            assert _same(part[k], one[k]), (t, k)
        # the oracle on the borders the kernel reads (fp32): at 5000 buckets the fp32 bucket widths differ from the
        # float64 ones by ~1e-4 relative, more than the near-tie tolerance of the mode check
        G32 = tk["G"].astype(np.float32).astype(np.float64)
        ref = _oracle(tk["logits"], tk["b"], tk["s"], None if null_cancel else tk["cancel"], G32, temperature, avg)
        _check(part, ref, G32, f"task {t} K{K} n{n_est} t{temperature} avg{avg}")


@pytest.mark.parametrize("K,n_est,S", SHAPES)
@pytest.mark.parametrize("avg", [False, True])
def test_one_task_equals_bar_tail(K, n_est, S, avg):
    tk = _tasks_inputs(K, n_est, 3 * K + S, rows=[S])[0]
    got, _ = _run_tasks([tk], 0.9, avg, False)
    one = _run_one(tk, 0.9, avg, False)
    for k in ALL:
        assert _same(got[k], one[k]), k


def test_tasks_outputs_alone_equal_together_and_null_untouched():
    K, n_est = 64, 3
    tasks = _tasks_inputs(K, n_est, 41, rows=[20, 1, 57])
    together, ro = _run_tasks(tasks, 0.9, False, False)
    S = int(ro[-1])
    lib = _lib.load()
    ptrs = _dev(np.array([tk["buf"][e, PAD[0]].data_ptr() for tk in tasks for e in range(n_est)], dtype=np.int64))
    ro_d = _dev(ro)
    bd, sd = _dev(np.stack([tk["b"] for tk in tasks])), _dev(np.stack([tk["s"] for tk in tasks]))
    cd = _dev(np.stack([tk["cancel"] for tk in tasks]).astype(np.uint8))
    Gd = _dev(np.stack([tk["G"] for tk in tasks]).astype(np.float32))
    qd = torch.tensor(QS, dtype=torch.float32, device="cuda")
    shapes = dict(mean=(S,), median=(S,), mode=(S,), quantiles=(len(QS), S), log_prob=(S, K))
    for name in ALL:
        bufs = {k: torch.full(shapes[k], 7.0, device="cuda") for k in ALL}
        outs = [bufs[k].data_ptr() if k == name else None for k in ALL]
        _lib.check(lib.mmpfn_bar_tail_tasks(ptrs.data_ptr(), len(tasks), n_est, ro_d.data_ptr(), S, K, bd.data_ptr(),
                                            sd.data_ptr(), cd.data_ptr(), Gd.data_ptr(), 0.9, 0, qd.data_ptr(), len(QS),
                                            *outs, _stream()), "mmpfn_bar_tail_tasks")
        torch.cuda.synchronize()
        for k in ALL:
            v = bufs[k].cpu().numpy()
            if k == name:
                assert _same(v, together[k]), name
            else:
                assert np.all(v == 7.0), (name, k)


def test_tail_tasks_refusals():
    lib = _lib.load()
    K = 64
    lg = torch.zeros((2, K), device="cuda")
    ptrs = _dev(np.array([lg.data_ptr()], dtype=np.int64))
    ro = _dev(np.array([0, 2], dtype=np.int32))
    b = torch.zeros((1, 8194), dtype=torch.int32, device="cuda")
    s = torch.zeros((1, 8194), device="cuda")
    G = torch.arange(8194, dtype=torch.float32, device="cuda")
    mean = torch.zeros(2, device="cuda")
    q = torch.tensor([0.5], device="cuda")

    def call(**kw):
        a = dict(logits=ptrs.data_ptr(), n_tasks=1, n_est=1, row_offset=ro.data_ptr(), S_total=2, K=K,
                 src_bucket=b.data_ptr(), src_share=s.data_ptr(), cancel=None, borders=G.data_ptr(), temperature=0.9,
                 avg=0, quantiles=q.data_ptr(), n_q=1, mean=mean.data_ptr(), median=None, mode=None, quant=None,
                 log_prob=None)
        a.update(kw)
        return lib.mmpfn_bar_tail_tasks(*a.values(), _stream())

    assert call() == 0
    for bad in (dict(logits=None), dict(row_offset=None), dict(src_bucket=None), dict(src_share=None),
                dict(borders=None), dict(n_tasks=0), dict(n_est=0), dict(S_total=0), dict(K=1),
                dict(temperature=0.0), dict(temperature=-1.0), dict(quant=mean.data_ptr(), quantiles=None),
                dict(quant=mean.data_ptr(), n_q=0)):
        assert call(**bad) == -1, bad                                                     # EINVAL
    big = torch.zeros((2, 8193), device="cuda")
    big_ptrs = _dev(np.array([big.data_ptr()], dtype=np.int64))
    assert call(logits=big_ptrs.data_ptr(), K=8193) == -4                                # EUNSUPPORTED
    assert b"8192" in lib.mmpfn_last_error()
    torch.cuda.synchronize()


# ---- regression entries in ragged passes ------------------------------------------------------------------------
def _reg_model(precision, n_out=64, seed=9):
    geom = Geometry(mgm_heads=2, cap_heads=4, n_out=n_out)
    sd = make_state_dict(geom, seed=seed, regression=True)
    return sd, geom, B200PerFeatureTransformer(sd, geom, device="cuda", precision=precision, seed=0, outlier_std=12.0)


def _reg_entries(model, rng):
    """Entries of three token counts (no table / 5 / 13 features, with and without image tokens), ragged rows and
    float targets; every other entry carries its label mean."""
    spec = [(None, 1, 61, 7), (5, 0, 200, 33), (5, 0, 97, 1), (13, 1, 130, 40), (13, 1, 47, 12), (13, 0, 150, 9)]
    img_rows = sum(ntr + nte for F, ni, ntr, nte in spec if ni)
    tok = model.stem_image(torch.from_numpy(rng.standard_normal((img_rows, 1, 768)).astype(np.float32)).cuda())
    out, row = [], 0
    for k, (F, ni, ntr, nte) in enumerate(spec):
        X = None if F is None else rng.standard_normal((ntr + nte, F)).astype(np.float32)
        if X is not None:
            X[::4, 1] = np.nan
        y = (np.exp(rng.normal(0, 0.8, ntr)) * 3.0 - 2.0).astype(np.float32)
        y_mean = model.label_stats(torch.from_numpy(y)[None].cuda())[0] if k % 2 else None
        out.append(dict(X=X, y=y, n_train=ntr, n_test=nte, tok=tok if ni else None, tok_row=row, n_tok=ni,
                        y_mean=y_mean))
        row += (ntr + nte) if ni else 0
    return out


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_ragged_regression_pass_equals_each_entry_alone(precision):
    _, _, model = _reg_model(precision)
    entries = _reg_entries(model, np.random.default_rng(12))
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
        y = torch.from_numpy(e["y"])[None].cuda()
        ctx = model.fit_context(None if X_all is None else X_all[:, :ntr].contiguous(), None, y, X_all=X_all,
                                img_tok_train=tok_tr, check=False, nan_flag=flag)
        alone = model.predict_with_context(ctx, None if X_all is None else X_all[:, ntr:].contiguous(), None,
                                           img_tok_test=tok_te, nan_flag=flag)
        assert got[j].shape == (e["n_test"], 64)
        assert torch.equal(got[j], alone[0]), (precision, j, float((got[j] - alone[0]).abs().max()))
    assert len(states) >= 6
    n_seg = len(states) // 2
    for phase, part in (("n_train", states[:n_seg]), ("n_test", states[n_seg:])):
        for v, js in part:
            for k, j in enumerate(js):
                pad = v[k, entries[j][phase]:]
                assert torch.equal(pad, torch.zeros_like(pad)), (phase, j)


# ---- predict_regression_tasks end to end --------------------------------------------------------------------------
def _regression_tasks():
    """The twelve mixed tasks with skewed continuous targets (lognormal-like, as the regressor tests use)."""
    rng = np.random.default_rng(77)
    tasks = _mixed_tasks()
    for t in tasks:
        n = len(t["y_train"])
        if t["X_train"] is not None:
            Xz = np.nan_to_num(t["X_train"])
            Xz = (Xz - Xz.mean(0)) / (Xz.std(0) + 1e-6)
            lin = Xz @ rng.normal(0, 0.4, Xz.shape[1])
        else:
            lin = t["img_train"][:, 0, :8].sum(1)
        t["y_train"] = (np.exp(0.3 * lin + rng.normal(0, 0.3, n)) * 10 + rng.normal(0, 0.5, n)).astype(np.float32)
    return tasks


def _one_by_one(sd, geom, tasks, precision, indices, **kw):
    out = {}
    for i in indices:
        t = tasks[i]
        reg = MMPFNRegressor(mgm_heads=2, cap_heads=4, n_estimators=4, model_path=(sd, geom), device="cuda",
                             inference_precision=precision, random_state=0, ignore_pretraining_limits=True,
                             average_before_softmax=kw.get("average_before_softmax", False))
        reg.fit(t["X_train"], t["img_train"], t["y_train"])
        out[i] = reg.predict(t["X_test"], t["img_test"], output_type="full")
    return out


def _assert_full_equal(a, b, what):
    assert set(a) == set(b) == {"mean", "median", "mode", "quantiles", "logits", "borders"}, what
    for k in ("mean", "median", "mode", "logits", "borders"):
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, (what, k)
        assert np.array_equal(a[k], b[k]), (what, k, float(np.nanmax(np.abs(a[k] - b[k]))))
    assert len(a["quantiles"]) == len(b["quantiles"])
    assert np.array_equal(np.stack(a["quantiles"]), np.stack(b["quantiles"])), (what, "quantiles")


@pytest.mark.parametrize("precision,K,avg", [("fp32", 64, False), ("bf16", 64, False), ("fp32", 5000, False),
                                             ("bf16", 5000, False), ("bf16", 64, True), ("fp32", 5000, True)])
def test_regression_tasks_equal_one_by_one(precision, K, avg):
    tasks = _regression_tasks()
    # more than MMPFN_MAX_SEGMENTS token counts (before the members' preprocessing): several passes
    assert len({(t["X_train"] is None and -1 or (t["X_train"].shape[1] + 1) // 2, t["img_train"] is None)
                for t in tasks}) > 8
    sd, geom, model = _reg_model(precision, n_out=K)
    packed = predict_regression_tasks(model, sd["criterion.borders"], tasks, n_estimators=4, random_state=0,
                                      average_before_softmax=avg, output_type="full")
    assert sorted(packed) == list(range(len(tasks)))
    one = _one_by_one(sd, geom, tasks, precision, range(len(tasks)), average_before_softmax=avg)
    for i in range(len(tasks)):
        _assert_full_equal(packed[i], one[i], (precision, K, avg, i))


def test_regression_tasks_indices_and_output_types():
    tasks = _regression_tasks()
    sd, _, model = _reg_model("bf16")
    g = sd["criterion.borders"]
    full = predict_regression_tasks(model, g, tasks, output_type="full")
    sub = predict_regression_tasks(model, g, tasks, output_type="full", indices=[9, 2, 5], n_jobs=3)
    assert sorted(sub) == [2, 5, 9]
    for i in sub:
        _assert_full_equal(sub[i], full[i], i)
    mean = predict_regression_tasks(model, g, tasks, output_type="mean")
    quant = predict_regression_tasks(model, g, tasks, output_type="quantiles", quantiles=[0.5, 0.9, 0.25])
    main = predict_regression_tasks(model, g, tasks, output_type="main")
    for i, t in enumerate(tasks):
        n = len(t["X_test"] if t["X_test"] is not None else t["img_test"])
        assert isinstance(mean[i], np.ndarray) and mean[i].dtype == np.float32 and mean[i].shape == (n,)
        assert np.array_equal(mean[i], full[i]["mean"])
        assert isinstance(quant[i], list) and len(quant[i]) == 3
        assert all(q.dtype == np.float32 and q.shape == (n,) for q in quant[i])
        assert np.array_equal(quant[i][0], full[i]["median"])
        assert np.array_equal(quant[i][1], full[i]["quantiles"][8])
        assert set(main[i]) == {"mean", "median", "mode", "quantiles"} and len(main[i]["quantiles"]) == 9
        for k in ("mean", "median", "mode"):
            assert main[i][k].dtype == np.float32 and np.array_equal(main[i][k], full[i][k])
        assert full[i]["logits"].shape == (n, 64) and full[i]["borders"].shape == (65,)


def test_regression_tasks_refusals():
    tasks = _regression_tasks()[:4]
    sd, _, model = _reg_model("bf16")
    g = np.asarray(sd["criterion.borders"])
    geom_c = Geometry(mgm_heads=2, cap_heads=4)
    clf = B200PerFeatureTransformer(make_state_dict(geom_c, seed=1), geom_c, device="cuda", precision="bf16", seed=0)
    with pytest.raises(ValueError, match="classification checkpoint"):
        predict_regression_tasks(clf, g, tasks)
    with pytest.raises(ValueError, match="65 finite increasing"):
        predict_regression_tasks(model, g[:-1], tasks)
    with pytest.raises(ValueError, match="65 finite increasing"):
        predict_regression_tasks(model, g[::-1], tasks)
    _, _, big = _reg_model("bf16", n_out=8193)
    with pytest.raises(ValueError, match="8192"):
        predict_regression_tasks(big, np.linspace(-5, 5, 8194), tasks)
    bad = [dict(t) for t in tasks]
    bad[3]["y_train"] = np.where(np.arange(len(bad[3]["y_train"])) == 2, np.inf, bad[3]["y_train"])
    with pytest.raises(ValueError, match="task 3: .*NaN or infinite"):
        predict_regression_tasks(model, g, bad)
    bad = [dict(t) for t in tasks]
    bad[2]["y_train"] = np.full(len(bad[2]["y_train"]), 4.0)
    with pytest.raises(ValueError, match="task 2: .*zero spread"):
        predict_regression_tasks(model, g, bad)
    with pytest.raises(ValueError, match="output_type"):
        predict_regression_tasks(model, g, tasks, output_type="proba")
