"""Many tasks on one GPU: predict_proba_tasks over all tasks at once ("packed") against one task at a time, on two
seeded workloads:
  (a) BASELINE.json configs[4] per GPU: 32 equal tasks (800 train + 200 test rows, 32 features, one embedding);
  (b) 64 tasks of different sizes: 100-2000 train rows, 20-400 test rows, 4-64 features, three quarters of them with
      one embedding (rows and columns cut from synth's img_text_10k).
8 estimators each.  One JSON line per (workload, mode, repetition): tasks/s, test rows/s, wall ms, host ms (fitting
the members' transforms on the host), device-phase ms (stem + layers + tail up to a synchronise, host launch work
included), library launches per call, the padded share of the pass tokens, the card and its power limit.
usage: python tools/ragged_tasks_bench.py [--root TREE] [--workload a|b] [--reps N] [--tag NAME]
(--root: the repository tree to import, so that an exported older commit can be measured by the same script)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--workload", choices=["a", "b"], default="a")
ap.add_argument("--reps", type=int, default=2)
ap.add_argument("--tag", default="")
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from multimodalpfn_b200 import _lib  # noqa: E402
from multimodalpfn_b200.model import B200PerFeatureTransformer  # noqa: E402
from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict  # noqa: E402
from multimodalpfn_b200.tasks import predict_proba_tasks  # noqa: E402

N_EST = 8


def workload_a():
    tasks = []
    for k in range(32):
        d = make_dataset("small_task", k)
        tasks.append(dict(X_train=d["X_train"], img_train=d["img_train"], y_train=d["y_train"], X_test=d["X_test"],
                          img_test=d["img_test"]))
    return tasks


def workload_b():
    rng = np.random.default_rng(64)
    d = make_dataset("img_text_10k", 1)
    X = np.concatenate([d["X_train"], d["X_test"]])
    img = np.concatenate([d["img_train"], d["img_test"]])[:, :1]
    y = np.concatenate([d["y_train"], d["y_test"]])
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


geom = Geometry(mgm_heads=8, cap_heads=8)
model = B200PerFeatureTransformer(make_state_dict(geom, seed=1), geom, precision="bf16", seed=0)
tasks = workload_a() if args.workload == "a" else workload_b()
rows = sum(len(t["X_test"]) if t["X_test"] is not None else len(t["img_test"]) for t in tasks)

# the padded share of the pass tokens (forward_ragged exists from the ragged passes on)
pad = {"tokens": 0, "useful": 0}
if hasattr(model, "forward_ragged"):
    _inner = model.forward_ragged

    def _recording(entries, **kw):
        Ts = [model.entry_tokens(None if e["X"] is None else e["X"].shape[1], e["n_tok"]) for e in entries]
        S = max(e["n_train"] for e in entries) + max(e["n_test"] for e in entries)
        pad["tokens"] += S * sum(Ts)
        pad["useful"] += sum((e["n_train"] + e["n_test"]) * T for e, T in zip(entries, Ts))
        return _inner(entries, **kw)
    model.forward_ragged = _recording

name = card()
outs = {}
for rep in range(args.reps + 1):                       # repetition 0 warms every shape up and is not reported
    for mode in ("packed", "one task at a time"):
        pad["tokens"] = pad["useful"] = 0
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        t0 = time.perf_counter()
        tm = {"host_prepare": 0.0, "device": 0.0}
        if mode == "packed":
            out = predict_proba_tasks(model, tasks, n_estimators=N_EST, random_state=0, timings=tm)
        else:
            out = {}
            for i, t in enumerate(tasks):
                t1 = {}
                out[i] = predict_proba_tasks(model, [t], n_estimators=N_EST, random_state=0, timings=t1)[0]
                tm = {k: tm[k] + t1[k] for k in tm}
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        launches = _lib.launch_count() - l0
        outs.setdefault(mode, out)
        if rep == 0:
            continue
        same = all(np.array_equal(out[i], outs["packed"][i]) for i in out)
        digest = hashlib.sha256(b"".join(np.ascontiguousarray(out[i]).tobytes() for i in sorted(out))).hexdigest()[:16]
        print(json.dumps(dict(
            tag=args.tag, workload=args.workload, mode=mode, rep=rep, n_tasks=len(tasks), n_estimators=N_EST,
            tasks_per_s=round(len(tasks) / dt, 2), test_rows_per_s=round(rows / dt), wall_ms=round(dt * 1e3, 1),
            host_ms=round(tm["host_prepare"] * 1e3, 1), device_phase_ms=round(tm["device"] * 1e3, 1),
            launches_per_call=launches,
            padded_token_fraction=(round(1 - pad["useful"] / pad["tokens"], 4) if pad["tokens"] else None),
            equal_to_packed=same, proba_sha256=digest, card=name)), flush=True)
