"""Many regression tasks on one GPU: predict_regression_tasks over all tasks at once ("packed") against one
MMPFNRegressor per task ("one regressor per task"), run alternately in the same process, on two seeded workloads:
  (a) BASELINE.json configs[4] per GPU: 32 equal tasks (800 train + 200 test rows, 32 features, one embedding);
  (b) 64 tasks of different sizes cut as in tools/ragged_tasks_bench.py: 100-2000 train rows, 20-400 test rows, 4-64
      features, three quarters of them with one embedding.
Continuous skewed targets (exp of a linear function of the standardised table, plus noise), a synthetic bf16
checkpoint with 5000 buckets, 8 estimators, output_type "main" (mean, median, mode, nine quantiles).
One JSON line per (workload, mode, repetition): tasks/s, test rows/s, wall ms, host ms (packed: prepare_regression
of every task; per task: each regressor's fit, which also builds its model from the state dict), device-phase ms
(packed: stems, passes, tail and host copies; per task: the sum of the predict calls, their host-side test
transforms included), tail ms (packed: the one mmpfn_bar_tail_tasks call, its pointer-table upload included; per task:
the sum of the mmpfn_bar_tail calls; CUDA events), the padded share of the pass tokens, whether the means equal the
packed run's bit for bit, the card and its power limit.
usage: python tools/regression_tasks_bench.py [--workload a|b] [--reps N] [--tag NAME]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from multimodalpfn_b200 import regressor as R  # noqa: E402
from multimodalpfn_b200.model import B200PerFeatureTransformer  # noqa: E402
from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict  # noqa: E402
from multimodalpfn_b200.tasks import predict_regression_tasks  # noqa: E402

N_EST = 8
K = 5000

ap = argparse.ArgumentParser()
ap.add_argument("--workload", choices=["a", "b"], default="a")
ap.add_argument("--reps", type=int, default=2)
ap.add_argument("--tag", default="")
args = ap.parse_args()


def continuous_target(X, img, rng):
    Xz = np.nan_to_num(X)
    Xz = (Xz - Xz.mean(0)) / (Xz.std(0) + 1e-6)
    lin = Xz @ rng.normal(0, 0.4, X.shape[1]) + (0 if img is None else img[:, 0, :8].sum(1) * 0.2)
    return (np.exp(0.3 * lin) * 10 + rng.normal(0, 0.5, len(X))).astype(np.float32)


def workload_a():
    rng = np.random.default_rng(4)
    tasks = []
    for k in range(32):
        d = make_dataset("small_task", k)
        n = len(d["X_train"])
        y = continuous_target(np.concatenate([d["X_train"], d["X_test"]]),
                              np.concatenate([d["img_train"], d["img_test"]]), rng)
        tasks.append(dict(X_train=d["X_train"], img_train=d["img_train"], y_train=y[:n], X_test=d["X_test"],
                          img_test=d["img_test"]))
    return tasks


def workload_b():
    rng = np.random.default_rng(64)
    d = make_dataset("img_text_10k", 1)
    X = np.concatenate([d["X_train"], d["X_test"]])
    img = np.concatenate([d["img_train"], d["img_test"]])[:, :1]
    y = continuous_target(X, img, np.random.default_rng(65))
    tasks = []
    for k in range(64):
        n_tr, n_te, F = int(rng.integers(100, 2001)), int(rng.integers(20, 401)), int(rng.integers(4, 65))
        rows = rng.permutation(len(X))[:n_tr + n_te]
        cols = rng.permutation(X.shape[1])[:F]
        Xt, it = X[rows][:, cols], (img[rows] if k % 4 != 3 else None)
        tasks.append(dict(X_train=Xt[:n_tr], X_test=Xt[n_tr:], y_train=y[rows[:n_tr]],
                          img_train=None if it is None else it[:n_tr], img_test=None if it is None else it[n_tr:]))
    return tasks


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        q = ""
    return q or torch.cuda.get_device_name(0)


geom = Geometry(mgm_heads=8, cap_heads=8, n_out=K)
sd = make_state_dict(geom, seed=1, regression=True)
model = B200PerFeatureTransformer(sd, geom, precision="bf16", seed=0, outlier_std=12.0)
tasks = workload_a() if args.workload == "a" else workload_b()
rows = sum(len(t["X_test"]) if t["X_test"] is not None else len(t["img_test"]) for t in tasks)

pad = {"tokens": 0, "useful": 0}
_inner = model.forward_ragged


def _recording(entries, **kw):
    Ts = [model.entry_tokens(None if e["X"] is None else e["X"].shape[1], e["n_tok"]) for e in entries]
    S = max(e["n_train"] for e in entries) + max(e["n_test"] for e in entries)
    pad["tokens"] += S * sum(Ts)
    pad["useful"] += sum((e["n_train"] + e["n_test"]) * T for e, T in zip(entries, Ts))
    return _inner(entries, **kw)


model.forward_ragged = _recording

# CUDA events around every one-task tail call of the regressors
tail_events = []
_tail = R.bar_tail_device


def _timed_tail(*a, **kw):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    out = _tail(*a, **kw)
    ev[1].record()
    tail_events.append(ev)
    return out


R.bar_tail_device = _timed_tail

name = card()
ref = None
for rep in range(args.reps + 1):                       # repetition 0 warms every shape up and is not reported
    for mode in ("packed", "one regressor per task"):
        pad["tokens"] = pad["useful"] = 0
        tail_events.clear()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tm = {"host_prepare": 0.0, "device": 0.0, "tail": 0.0}
        if mode == "packed":
            out = predict_regression_tasks(model, sd["criterion.borders"], tasks, n_estimators=N_EST, random_state=0,
                                           output_type="main", timings=tm)
        else:
            out = {}
            for i, t in enumerate(tasks):
                a = time.perf_counter()
                reg = R.MMPFNRegressor(mgm_heads=8, cap_heads=8, n_estimators=N_EST, model_path=(sd, geom),
                                       device="cuda", inference_precision="bf16", random_state=0,
                                       ignore_pretraining_limits=True).fit(t["X_train"], t["img_train"], t["y_train"])
                torch.cuda.synchronize()
                b = time.perf_counter()
                out[i] = reg.predict(t["X_test"], t["img_test"], output_type="main")
                torch.cuda.synchronize()
                tm["host_prepare"] += b - a
                tm["device"] += time.perf_counter() - b
            tm["tail"] = sum(e[0].elapsed_time(e[1]) for e in tail_events) / 1e3
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if mode == "packed":
            ref = out
        if rep == 0:
            continue
        same = all(np.array_equal(out[i]["mean"], ref[i]["mean"]) for i in out)
        print(json.dumps(dict(
            tag=args.tag, workload=args.workload, mode=mode, rep=rep, n_tasks=len(tasks), n_estimators=N_EST,
            buckets=K, test_rows=rows, tasks_per_s=round(len(tasks) / dt, 2), test_rows_per_s=round(rows / dt),
            wall_ms=round(dt * 1e3, 1), host_ms=round(tm["host_prepare"] * 1e3, 1),
            device_phase_ms=round(tm["device"] * 1e3, 1), tail_ms=round(tm["tail"] * 1e3, 3),
            padded_token_fraction=(round(1 - pad["useful"] / pad["tokens"], 4) if pad["tokens"] else None),
            mean_equal_to_packed=same, card=name)), flush=True)
