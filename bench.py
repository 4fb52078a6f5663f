#!/usr/bin/env python
"""bench.py — test rows/s of MMPFN ``predict_proba`` on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload at N=1 (BASELINE.json configs[1]): PAD-UFES-20 shape — 2000 train / 300 test rows,
21 tabular features + one 768-d image embedding per row, 8 estimators, bf16, random-init
TabPFN-v2 weights (12 layers, emsize 192) with MGM(8)+CAP(8) image stem.  One *step* = one
reference-equivalent ``predict_proba`` pass: the train context is rebuilt inside the call exactly
like the reference does (inference.py:302-348), then the 300 test rows are classified.

* ``value``  — rows/s with every input already resident in HBM (device-timed, CUDA events).
* ``e2e``    — rows/s through ``MMPFNClassifier.predict_proba`` with HOST buffers: per-estimator
  host preprocessing, H2D of the test table + test embeddings, D2H of the probabilities.
* ``roofline`` — the dominant kernel (item-axis attention, tcgen05) timed alone at the workload's
  shape against the measured bf16 tensor peak (MEASURED_PEAKS.json).
* ``cpu_baseline`` — the oracle port (oracle/forward_ref.py, fp32 torch on all host cores) on a
  bounded sample of the same workload, scaled by the algorithmic FLOP ratio.

With N>1 (torchrun, one rank per GPU) every rank classifies its own 300-row test chunk
(weak scaling); the train context is built once per estimator on its owner rank and the K/V context is
all-gathered over NCCL layer by layer under the build (multimodalpfn_b200/dist.py); the probabilities of all ranks
are all-gathered inside the timed step.  ``strong_scaling`` times a fixed total of 2400 test rows beside it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

E, NH, DK, HID, L = 192, 6, 32, 768, 12
N_EST = 8
WORKLOAD = "pad_ufes"


# --------------------------------------------------------------------------------------------
# algorithmic FLOP model (BASELINE.md section 4), 2 FLOP per MAC
# --------------------------------------------------------------------------------------------
def flops_estimator(n_tr, n_te, T, layers=L):
    S = n_tr + n_te
    feat = S * (8 * T * E * E + 4 * T * T * E)
    item = 8 * n_tr * T * E * E + 4 * T * n_tr * n_tr * E + 4 * n_te * T * E * E + 4 * T * n_te * n_tr * E
    mlp = 16 * S * T * E * E
    return layers * (feat + item + mlp)


def flops_item_attention(n_q, n_kv, T, B):
    return 4.0 * B * T * NH * n_q * n_kv * DK


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], burst=d["bf16_tflops"], sustained=d["bf16_tflops_sustained"], src="measured",
                    sm_max_mhz=d.get("sm_max_mhz", 1965.0))
    return dict(hbm=6650.0, burst=1590.0, sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([c.strip() for c in out.stdout.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# --------------------------------------------------------------------------------------------
# CPU arm: the oracle port on a bounded sample
# --------------------------------------------------------------------------------------------
def cpu_sample(n_layers_sample: int, which: str = "quantile_svd"):
    """Times the oracle on ONE estimator of the workload truncated to ``n_layers_sample`` of the 12
    (identical-cost) layers, all host threads; returns (seconds, flops of the sample, T)."""
    import torch
    from multimodalpfn_b200.preprocessing import make_members
    from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
    from oracle import forward_ref as R

    torch.set_num_threads(os.cpu_count() or 1)
    d = make_dataset(WORKLOAD, 0)
    geom = Geometry(mgm_heads=8, cap_heads=8, nlayers=n_layers_sample)
    sd_full = make_state_dict(Geometry(mgm_heads=8, cap_heads=8), seed=1)
    tsd = R.as_torch_state_dict(sd_full)
    members = make_members(N_EST, d["X_train"].shape[1], d["n_classes"], np.random.default_rng(0))
    m = [mm for mm in members if mm.recipe == which][0]
    Xtr, ytr = m.fit_transform(d["X_train"], d["y_train"])
    Xte = m.transform(d["X_test"])
    X = torch.as_tensor(np.concatenate([Xtr, Xte]))
    img = torch.as_tensor(np.concatenate([d["img_train"], d["img_test"]]))
    y = torch.as_tensor(ytr)
    T = (X.shape[1] + 1) // 2 + 8 + 1
    t0 = time.perf_counter()
    with torch.inference_mode():
        R.forward_joint(X, img, y, tsd, geom, seed=0)
    dt = time.perf_counter() - t0
    n_tr, n_te = len(ytr), Xte.shape[0]
    return dt, flops_estimator(n_tr, n_te, T, layers=n_layers_sample), T


def full_flops():
    from multimodalpfn_b200.synth import DATASETS
    n_tr, n_te = DATASETS[WORKLOAD][:2]
    return (N_EST // 2) * (flops_estimator(n_tr, n_te, 27) + flops_estimator(n_tr, n_te, 20)), n_tr, n_te


def _reference_classifier(device, n_estimators, **kw):
    """The UNMODIFIED reference ``MMPFNClassifier`` (``/root/reference`` here, the ``oracle/_ref`` snapshot on the
    GPU box) on the bench workload with the bench weights; returns (fitted classifier, dataset)."""
    import torch
    from multimodalpfn_b200.synth import Geometry, make_checkpoint_config, make_dataset, make_state_dict
    from oracle import ref_compat
    ref_compat.install()
    from mmpfn.models.mmpfn import MMPFNClassifier as RefClassifier
    geom = Geometry(mgm_heads=8, cap_heads=8)
    path = os.path.join("/tmp", f"mmpfn_b200_bench_{os.getpid()}.ckpt")
    if not os.path.exists(path):
        sd = make_state_dict(geom, seed=1)
        torch.save({"state_dict": {k: torch.as_tensor(v) for k, v in sd.items()},
                    "config": make_checkpoint_config(geom)}, path)
    d = make_dataset(WORKLOAD, 0)
    clf = RefClassifier(mixer_type="MGM+CAP", mgm_heads=8, cap_heads=8, features_per_group=2,
                        n_estimators=n_estimators, model_path=path, device=device, ignore_pretraining_limits=True,
                        random_state=0, **kw)
    clf.fit(d["X_train"], d["img_train"], d["y_train"])
    return clf, d


def _token_counts(clf):
    return sorted({(np.asarray(x).shape[1] + 1) // 2 + 8 + 1 for x in clf.executor_.X_trains}, reverse=True)


def reference_cpu_sample(steps, warmup):
    """Times the reference's own ``predict_proba`` (``classifier.py:517-576``, unmodified, diagnostic loop
    ``transformer.py:809-813`` included) on the host cores.  The estimators are a serial loop in the reference
    (``inference.py:294-349``) and its default ensemble alternates two preprocessing recipes, so a call with
    n_estimators=2 is exactly one quarter of the 8-estimator workload: one T=27 and one T=20 forward over the
    full 2000 train / 300 test rows.  Returns (seconds per 2-estimator call [list], token counts, n_test)."""
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    clf, d = _reference_classifier("cpu", 2)
    Ts = _token_counts(clf)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        p = clf.predict_proba(d["X_test"], d["img_test"])
        dt = time.perf_counter() - t0
        assert p.shape[0] == len(d["y_test"]) and np.allclose(p.sum(1), 1.0, atol=1e-5)
        if i >= warmup:
            times.append(dt)
    return times, Ts, len(d["y_test"])


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, all host cores.  One step = one
    ``predict_proba`` call of the unmodified reference with 2 of the 8 estimators (see
    ``reference_cpu_sample``); ``ms_per_step`` is the time actually spent per step, ``value`` = test rows /
    (4 x that); exactly ``--steps`` steps are timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_compat
    from multimodalpfn_b200.synth import DATASETS
    n_tr, n_te = DATASETS[WORKLOAD][:2]
    cores = os.cpu_count() or 1
    if ref_compat.reference_available():
        times, Ts, n_te = reference_cpu_sample(args.steps, min(args.warmup, 1))
        step_s = float(np.mean(times))
        value = n_te / (step_s * (N_EST / 2))
        kind = "reference"
        sample = (f"unmodified reference MMPFNClassifier.predict_proba (oracle/_ref snapshot), device=cpu fp32, "
                  f"{cores} threads, 2 of {N_EST} estimators per step (one of each preprocessing recipe, T={Ts}; "
                  f"the reference loops estimators serially), full {n_tr} train / {n_te} test rows, diagnostic loop "
                  f"included; value = {n_te} rows / ({N_EST // 2} x measured step)")
    else:                                            # no reference snapshot on this box: the oracle port
        total, n_tr, n_te = full_flops()
        t1, f1, _ = cpu_sample(1)
        layers = int(max(1, min(L, (150.0 / max(args.steps + args.warmup, 1)) // max(t1, 1e-3))))
        times = []
        for _ in range(args.steps):
            dt, fl, T = cpu_sample(layers)
            times.append(dt)
        step_s = float(np.mean(times))
        value = n_te / (step_s * total / fl)
        kind = "port"
        sample = f"oracle port: 1 of {N_EST} estimators (T=27), {layers} of {L} layers per step, scaled by algorithmic FLOPs"
    line = {
        "impl": "reference", "metric": "test rows/sec predict_proba", "value": value, "unit": "rows/s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": min(args.warmup, 1),
        "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{WORKLOAD}: {n_tr} train / {n_te} test rows, 21 feats + 768-d image emb, "
                               f"{N_EST} estimators, reference-equivalent (context rebuilt per call)",
                   "step": sample},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def gpu_reference_leg(steps=3):
    """The like-for-like GPU baseline (SURVEY.md section 8(d)): the UNMODIFIED reference on device="cuda" of the same
    B200 — torch eager, cuBLAS, ``F.scaled_dot_product_attention`` — full 8-estimator ``predict_proba`` with host
    inputs, under its default autocast (fp16) and in fp32, with the diagnostic loop (``transformer.py:809-813``:
    T^2 GEMMs + host syncs per forward) as shipped and removed.  None of this repo's kernels run here."""
    import torch
    from oracle import ref_compat
    out = {}
    for prec_name, prec in (("autocast_fp16", "auto"), ("fp32", torch.float32)):
        clf, d = _reference_classifier("cuda", N_EST, inference_precision=prec)
        n_te = len(d["y_test"])
        for diag in ("as_shipped", "diagnostic_loop_removed"):
            ctx = ref_compat.without_diagnostic_loop() if diag != "as_shipped" else None
            if ctx:
                ctx.__enter__()
            try:
                clf.predict_proba(d["X_test"], d["img_test"])
                torch.cuda.synchronize()
                ts = []
                for _ in range(steps):
                    t0 = time.perf_counter()
                    clf.predict_proba(d["X_test"], d["img_test"])
                    torch.cuda.synchronize()
                    ts.append(time.perf_counter() - t0)
            finally:
                if ctx:
                    ctx.__exit__(None, None, None)
            out[f"{prec_name}_{diag}"] = {"value": n_te / float(np.mean(ts)), "unit": "rows/s",
                                          "ms_per_step": float(np.mean(ts)) * 1e3}
        del clf
    out["note"] = ("unmodified reference MMPFNClassifier.predict_proba on device=cuda of this B200, 8 estimators, host "
                   "inputs, wall clock around the call (it ends with a D2H copy), mean of %d calls after one warm-up" % steps)
    return out


def plugin_e2e(args, dev_index, flush, precision):
    """End to end through the REFERENCE's own ``MMPFNClassifier.predict_proba`` with this repo's engine plugged in
    (``multimodalpfn_b200.plugin``, engine mode): the reference's validation, per-estimator numpy/sklearn transform
    and probability tail on the host, H2D of the preprocessed test tables + test embeddings, one batched CUDA pass,
    D2H of the probabilities."""
    import torch
    from multimodalpfn_b200 import plugin
    from oracle import ref_compat
    ref_compat.install()
    uninstall = plugin.install(precision=precision, pos_emb_device="cuda", mode="engine")
    try:
        clf, d = _reference_classifier(f"cuda:{dev_index}", N_EST)
    finally:
        uninstall()
    assert isinstance(clf.executor_, plugin.B200PluginEngine)
    for _ in range(3):
        p = clf.predict_proba(d["X_test"], d["img_test"])
    torch.cuda.synchronize()
    ts = []
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p = clf.predict_proba(d["X_test"], d["img_test"])
        ts.append(time.perf_counter() - t0)
    n_te = len(d["y_test"])
    widths = [0 if x is None else np.asarray(x).shape[1] for x in clf.executor_.ref.X_trains]
    h2d = sum(n_te * w * 4 for w in widths) + d["img_test"].nbytes
    return {"value": n_te / float(np.mean(ts)), "unit": "rows/s", "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(p.nbytes), "ms_per_step": float(np.mean(ts)) * 1e3,
            "api": "reference MMPFNClassifier.predict_proba + multimodalpfn_b200.plugin (engine mode)",
            "host_preprocessing": "the reference's fitted per-member transformers, "
                                  + ("replayed without sklearn's per-call validation (multimodalpfn_b200/ref_transform.py): "
                                     if clf.executor_.replay_state == "on" else "the reference's own transform calls: ")
                                  + clf.executor_.replay_note,
            "T": _token_counts(type("E", (), {"executor_": clf.executor_.ref})())}, p


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from multimodalpfn_b200 import _lib
    from multimodalpfn_b200.classifier import MMPFNClassifier
    from multimodalpfn_b200.engine import proba_from_logits
    from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    peaks = load_peaks()
    geom = Geometry(mgm_heads=8, cap_heads=8)
    sd = make_state_dict(geom, seed=1)
    d = make_dataset(WORKLOAD, 0)
    n_tr, n_te = len(d["y_train"]), len(d["y_test"])
    # weak scaling: rank r classifies its own copy-sized chunk of test rows (distinct rows per rank)
    rng = np.random.default_rng(100 + rank)
    X_test = d["X_test"] if rank == 0 else d["X_test"][rng.permutation(n_te)]
    img_test = d["img_test"] if rank == 0 else rng.standard_normal(d["img_test"].shape).astype(np.float32)

    clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=8, cap_heads=8, features_per_group=2, n_estimators=N_EST,
                          model_path=(sd, geom), device=f"cuda:{local}", inference_precision=args.precision,
                          ignore_pretraining_limits=True, random_state=0)
    clf.fit(d["X_train"], d["img_train"], d["y_train"])
    eng = clf.executor_
    if world > 1:
        from multimodalpfn_b200.dist import ShardedEngine
        eng = ShardedEngine(eng, rank, world)
        clf.executor_ = eng
    Ts = sorted({(g["F"] + 1) // 2 + 8 + 1 for g in eng.groups}, reverse=True)

    # ---- device-resident step -------------------------------------------------------------------
    from multimodalpfn_b200.preprocessing import transform_all
    X_tests_host = transform_all(clf.members_, X_test)
    staged = eng.stage(X_tests_host, img_test)
    perms = [m.class_perm for m in clf.members_]

    use_graph = world == 1 and not args.no_graph

    gathered = {}

    def step_device(st=None):
        st = staged if st is None else st
        lg = eng.logits_graphed(st) if use_graph else eng.logits_staged(st)
        if world > 1:
            # the tail on the device and the all-gather of every rank's probabilities belong to the step
            gathered["p"] = eng.proba_gathered(lg, perms, n_classes=clf.n_classes_)
        return lg

    # ---- roofline of the dominant kernel: item-axis attention (train rows, T=27 group), and the row-wise kernels,
    # each timed ALONE before the step loop heats the GPU (the peak they are held against is the burst figure)
    roof = extra = None
    if rank == 0 and not args.profile:
        roof = roofline_item_attention(torch, _lib, dev, n_tr, Ts[0], N_EST // 2, peaks)
        extra = kernel_breakdown(torch, _lib, dev, n_tr + n_te, Ts[0], N_EST // 2, peaks)
        torch.cuda.empty_cache()

    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    sync_all()
    l0 = _lib.launch_count()
    evs = []
    with ClockSampler(local) as clocks:
        sync_all()
        t_wall0 = time.perf_counter()
        for _ in range(args.steps):
            flush.zero_()                              # L2 flush between timed iterations (not timed)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            lg = step_device()
            b.record()
            evs.append((a, b))
        sync_all()
        t_wall = time.perf_counter() - t_wall0
    launches = (_lib.launch_count() - l0) // max(args.steps, 1)
    if use_graph:
        launches = eng.launches_per_call      # kernels inside the replayed CUDA graph
    ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    if world > 1:
        tms = torch.tensor([ms], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    value = world * n_te / (ms * 1e-3)
    proba_dev = proba_from_logits(lg, perms, n_classes=clf.n_classes_)
    assert np.allclose(proba_dev.sum(1), 1.0, atol=1e-5)
    if args.dump_outputs and rank == 0:
        # with N > 1 the step ends with every rank's probabilities all-gathered: that array is the step's result
        dump_outputs(args.dump_outputs, logits=lg.float().cpu().numpy(),
                     proba=gathered["p"].float().cpu().numpy() if world > 1 else proba_dev)
    strong = None
    if world > 1:
        pg = gathered["p"]
        assert pg.shape[0] == world * n_te
        assert torch.allclose(pg[rank * n_te:(rank + 1) * n_te].cpu(), torch.as_tensor(proba_dev), atol=1e-5)
        # strong scaling beside the weak line: a FIXED total of 2400 test rows split over the ranks
        total_rows = 2400
        per = total_rows // world
        reps = (total_rows + n_te - 1) // n_te
        Xs = np.concatenate([d["X_test"]] * reps)[rank * per:(rank + 1) * per]
        Is = np.concatenate([d["img_test"]] * reps)[rank * per:(rank + 1) * per]
        staged_s = eng.stage(transform_all(clf.members_, Xs), Is)
        for _ in range(3):
            step_device(staged_s)
        sync_all()
        evs2 = []
        for _ in range(args.steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step_device(staged_s)
            b.record()
            evs2.append((a, b))
        sync_all()
        tms = torch.tensor([float(np.mean([a.elapsed_time(b) for a, b in evs2]))], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        strong = {"value": per * world / (float(tms.item()) * 1e-3), "unit": "rows/s", "ms_per_step": float(tms.item()),
                  "total_test_rows": per * world, "rows_per_rank": per, "scaling": "strong"}
        staged = eng.stage(X_tests_host, img_test)
    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": ms, "gpu_launches": int(launches)}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- end-to-end step through the public API, host buffers ----------------------------------
    for _ in range(max(1, min(args.warmup, 3))):
        clf.predict_proba(X_test, img_test)
    sync_all()
    e2e_times = []
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p = clf.predict_proba(X_test, img_test)       # ends with the D2H copy of the probabilities
        e2e_times.append(time.perf_counter() - t0)
    e2e_s = float(np.mean(e2e_times))
    if world > 1:
        te = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s = float(te.item())
    h2d = sum(x.nbytes for x in X_tests_host) + img_test.nbytes
    d2h = p.nbytes

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- second variant (SURVEY 8(d)): context kept from fit (fit_mode="fit_with_cache") ----------
    cached = None
    if world == 1:
        clf_c = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=8, cap_heads=8, features_per_group=2,
                                n_estimators=N_EST, model_path=(sd, geom), device=f"cuda:{local}",
                                inference_precision=args.precision, ignore_pretraining_limits=True, random_state=0,
                                fit_mode="fit_with_cache")
        clf_c.fit(d["X_train"], d["img_train"], d["y_train"])
        staged_c = clf_c.executor_.stage(X_tests_host, img_test)
        for _ in range(3):
            clf_c.executor_.logits_graphed(staged_c)
        torch.cuda.synchronize()
        evc = []
        for _ in range(args.steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            clf_c.executor_.logits_graphed(staged_c)
            b.record()
            evc.append((a, b))
        torch.cuda.synchronize()
        msc = float(np.mean([a.elapsed_time(b) for a, b in evc]))
        for _ in range(2):
            clf_c.predict_proba(X_test, img_test)
        e2e_c = []
        for _ in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pc = clf_c.predict_proba(X_test, img_test)
            e2e_c.append(time.perf_counter() - t0)
        e2ec = float(np.mean(e2e_c))
        cached = {"value": n_te / (msc * 1e-3), "unit": "rows/s", "ms_per_step": msc,
                  "e2e": {"value": n_te / e2ec, "unit": "rows/s", "ms_per_step": e2ec * 1e3},
                  "max_abs_dp_vs_rebuilt": float(np.abs(pc - p).max()),
                  "note": "train-row K/V context built once in fit; predict_proba runs the 300 test rows only "
                          "(not the headline: the reference rebuilds the context in every call)"}
        del clf_c

    # ---- plug-in end to end: the reference's own predict_proba with this engine behind it ----------
    from oracle import ref_compat
    have_ref = ref_compat.reference_available()
    e2e_standalone = {"value": world * n_te / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": int(h2d),
                      "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_s * 1e3,
                      "api": "multimodalpfn_b200.MMPFNClassifier.predict_proba (own host preprocessing, not the "
                             "reference's recipes)"}
    e2e_main, gpu_ref, plug_dp = e2e_standalone, None, None
    if world == 1 and have_ref:
        e2e_main, p_plug = plugin_e2e(args, local, flush, args.precision)
        if args.gpu_reference:
            gpu_ref = gpu_reference_leg()

    # ---- CPU baseline on the host cores (bounded sample) ----------------------------------------
    total, _, _ = full_flops()
    cpu = None
    if args.cpu_baseline:
        if have_ref:
            times, Tref, _ = reference_cpu_sample(1, 0)
            cpu = {"value": n_te / (times[0] * (N_EST / 2)), "unit": "rows/s", "cores": os.cpu_count() or 1,
                   "kind": "reference",
                   "sample": f"unmodified reference predict_proba (oracle/_ref), device=cpu fp32, 2 of {N_EST} estimators "
                             f"(T={Tref}) in one call, {times[0]:.1f} s measured; value = {n_te} rows / ({N_EST // 2} x that)"}
        else:
            t1, f1, _ = cpu_sample(1)
            layers = int(max(1, min(L, 20.0 // max(t1, 1e-3))))
            dt, fl, _ = cpu_sample(layers)
            cpu = {"value": n_te / (dt * total / fl), "unit": "rows/s", "cores": os.cpu_count() or 1, "kind": "port",
                   "sample": f"oracle (fp32 torch CPU) on 1 of {N_EST} estimators (T=27), {layers} of {L} layers, "
                             f"{dt:.1f} s measured, scaled by algorithmic FLOPs"}

    line = {
        "metric": "test rows/sec predict_proba", "value": value, "unit": "rows/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": {"workload": f"{WORKLOAD}: {n_tr} train / {n_te} test rows per GPU, 21 feats + 768-d image emb, "
                               f"{N_EST} estimators (T={Ts}), MGM8+CAP8, 12 layers, emsize 192, random-init weights; "
                               "reference-equivalent: train context rebuilt inside every call",
                   "l2": "flushed between timed iterations (384 MB memset)",
                   "launch": "one CUDA graph replay per step" if use_graph else "eager launches",
                   "algorithmic_tflop_per_step": total / 1e12},
        "achieved_tflops": total / (ms * 1e-3) / 1e12 if world == 1 else None,
        "e2e": e2e_main,
        "e2e_standalone": e2e_standalone,
        "gpu_reference": gpu_ref,
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": roof,
        "kernels": extra,
        "cpu_baseline": cpu,
        "cached_context": cached,
        "strong_scaling": strong,
        "exchange": getattr(eng, "exchange", None),
        "wall_ms_per_step_incl_flush": t_wall * 1e3 / max(args.steps, 1),
        "peaks": peaks,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(dirname, **arrays):
    """Writes each array as ``dirname/<name>.npy`` in float32, so that the outputs of two builds can be compared."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def _time_kernel(torch, fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def roofline_item_attention(torch, _lib, dev, n_tr, T, B, peaks):
    """The item-axis attention kernel alone at the workload's train-row shape (B estimators x T
    token columns x 6 heads, n_q = n_kv = Ntr, d = 32): 20 launches back to back, CUDA events on the
    launching stream.  Q/K/V^T planes (3 x 83 MB at T=27, B=4) do not fit what one wave of CTAs
    touches but fit L2; the kernel is compute bound — and, at d = 32, bound by the exponentials
    (128 tensor FLOP per ex2) long before the tensor pipe: the second bound is reported next to it."""
    lib = _lib.load()
    pad = (n_tr + 63) // 64 * 64
    planes = B * T * NH
    g = torch.Generator(device=dev).manual_seed(0)
    q = torch.randn(planes, pad, DK, device=dev, generator=g).to(torch.bfloat16)
    k = torch.randn(planes, pad, DK, device=dev, generator=g).to(torch.bfloat16)
    vt = torch.randn(planes, DK, pad, device=dev, generator=g).to(torch.bfloat16)
    out = torch.empty(B, n_tr, T, E, device=dev, dtype=torch.bfloat16)
    st = torch.cuda.current_stream().cuda_stream

    def run():
        _lib.check(lib.mmpfn_item_attention_bf16(q.data_ptr(), k.data_ptr(), vt.data_ptr(), B, T, n_tr, pad, n_tr, pad,
                                                 0, out.data_ptr(), st), "item_attention")
    ms = _time_kernel(torch, run)
    fl = flops_item_attention(n_tr, n_tr, T, B)
    ach = fl / (ms * 1e-3) / 1e12
    # DRAM traffic of one launch of this shape from the committed ncu --set full capture (profiles/)
    traffic, src = None, None
    cands = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_attention_ncu.json"))
    tp = os.path.join(ROOT, "profiles", cands[-1]) if cands else ""
    if tp and os.path.exists(tp):
        with open(tp) as f:
            t = json.load(f)
        if t.get("shape") == {"B": B, "T": T, "n_q": n_tr, "n_kv": n_tr}:
            traffic, src = t["dram_bytes_read"] + t["dram_bytes_write"], t["source"]
    sm_clk = peaks.get("sm_max_mhz", 1965.0) * 1e6
    xu = 16.0 * 148 * sm_clk * 4 * DK / 1e12        # 16 ex2/clk/SM (measured, tools/ubench.cu), 4*d FLOP per score
    return {"kernel": "tc_item_attn_kernel", "bound": "tensor", "achieved": ach, "peak": peaks["burst"],
            "unit": "TFLOP/s", "frac": ach / peaks["burst"], "traffic": traffic, "traffic_source": src,
            "ms_per_launch": ms, "flops_per_launch": fl,
            "algorithmic_bytes_per_launch": 2.0 * (3 * planes * n_tr * DK + B * n_tr * T * E),
            "peak_source": f"{peaks['src']} bf16 burst (kernel timed alone)",
            "exp_bound": {"tflops": xu, "frac": ach / xu,
                          "note": "d=32: one ex2 per 128 tensor FLOP; MUFU issues 16 ex2/clk/SM, so 595 TFLOP/s at "
                                  "1965 MHz is this kernel's ceiling unless exponentials move to the FMA pipe"}}


def kernel_breakdown(torch, _lib, dev, S, T, B, peaks):
    """Isolated timings of the row-wise kernels of one layer (B estimators, S rows, T tokens) against the
    HBM roofline: algorithmic bytes = every operand read or written once."""
    lib = _lib.load()
    M = B * S * T
    st = torch.cuda.current_stream().cuda_stream
    res = {}
    g = torch.Generator(device=dev).manual_seed(1)
    A = torch.randn(M, E, device=dev, generator=g).to(torch.bfloat16)

    def entry(ms, flops, nbytes, **kw):
        d = {"ms": ms, "gbs": nbytes / ms / 1e6, "frac_hbm": nbytes / ms / 1e6 / peaks["hbm"], "bytes": nbytes}
        if flops:
            d.update(tflops=flops / ms / 1e9, frac_tensor=flops / ms / 1e9 / peaks["burst"])
        d.update(kw)
        return d

    # feature sublayer, first half: QKV projection + attention between the T tokens of a table row in ONE kernel
    # (tcgen05 projection, mma.sync attention on the q/k/v block in shared memory): reads x, writes [M][192].
    # Bound by the legacy mma.sync rate of the attention items (profiles/r02_feature_fused_knockouts.txt), not by HBM;
    # the two kernels it replaces (timed below for reference) move 4x the bytes.
    W = (torch.randn(3 * E, E, device=dev, generator=g) / E ** 0.5).to(torch.bfloat16)
    att = torch.empty(M, E, device=dev, dtype=torch.bfloat16)
    ms = _time_kernel(torch, lambda: _lib.check(
        lib.mmpfn_feature_qkv_attention_bf16(A.data_ptr(), W.data_ptr(), B * S, T, att.data_ptr(), st), "feat_fused"))
    res["feature_qkv_attention_fused"] = entry(ms, 2.0 * M * 3 * E * E + 4.0 * M * T * E, 2.0 * (M * E + 3 * E * E + M * E),
                                               M=M, T=T, on_path=True)
    O = torch.empty(M, 3 * E, device=dev, dtype=torch.bfloat16)
    ms = _time_kernel(torch, lambda: _lib.check(
        lib.mmpfn_linear_bf16(A.data_ptr(), W.data_ptr(), M, 3 * E, E, 0, O.data_ptr(), st), "qkv"))
    res["qkv_proj"] = entry(ms, 2.0 * M * 3 * E * E, 2.0 * (M * E + 3 * E * E + M * 3 * E), M=M, N=3 * E, K=E,
                            on_path="rows wider than 64 tokens only")
    ms = _time_kernel(torch, lambda: _lib.check(
        lib.mmpfn_feature_attention_bf16(O.data_ptr(), att.data_ptr(), B * S, T, st), "feat_attn"))
    res["feature_attention"] = entry(ms, 4.0 * M * T * E, 2.0 * (M * 3 * E + M * E), M=M, T=T,
                                     on_path="rows wider than 64 tokens only")
    del O, att
    # item-attention QKV projection + scatter into q/k/v^T planes (+ head-0 context): [B][S][T] tiles by 4-D TMA
    Sp = (S + 63) // 64 * 64
    P = B * T * NH
    qkv = [torch.empty(P * Sp * DK, device=dev, dtype=torch.bfloat16) for _ in range(3)]
    ctx = [torch.empty(B * T * Sp * DK, device=dev, dtype=torch.bfloat16) for _ in range(2)]
    ms = _time_kernel(torch, lambda: _lib.check(
        lib.mmpfn_item_qkv_bf16(A.data_ptr(), W.data_ptr(), B, S, T, Sp, 3, qkv[0].data_ptr(), qkv[1].data_ptr(),
                                qkv[2].data_ptr(), ctx[0].data_ptr(), ctx[1].data_ptr(), st), "item_qkv"))
    res["item_qkv_scatter"] = entry(ms, 2.0 * M * 3 * E * E, 2.0 * (M * E + 3 * E * E + M * 3 * E + 2 * B * T * S * DK), M=M)
    del qkv, ctx
    # attention output projection + residual + LayerNorm: state fp32 in/out, bf16 shadow out
    x = torch.randn(M, E, device=dev, generator=g)
    xb = torch.empty(M, E, device=dev, dtype=torch.bfloat16)
    Wo = (torch.randn(E, E, device=dev, generator=g) / E ** 0.5).to(torch.bfloat16)
    ms = _time_kernel(torch, lambda: _lib.check(
        lib.mmpfn_linear_ln_bf16(A.data_ptr(), Wo.data_ptr(), M, x.data_ptr(), xb.data_ptr(), st), "out_ln"))
    res["out_proj_residual_layernorm"] = entry(ms, 2.0 * M * E * E, M * E * (2 + 4 + 4 + 2) + 2.0 * E * E, M=M)
    # fused MLP sublayer (GEMM -> GELU -> GEMM -> residual + LayerNorm)
    w1 = (torch.randn(HID, E, device=dev, generator=g) / E ** 0.5).to(torch.bfloat16)
    w2 = (torch.randn(E, HID, device=dev, generator=g) / HID ** 0.5).to(torch.bfloat16)
    xb.copy_(x)
    ms = _time_kernel(torch, lambda: _lib.check(
        lib.mmpfn_mlp_bf16(x.data_ptr(), xb.data_ptr(), w1.data_ptr(), w2.data_ptr(), M, st), "mlp"))
    res["mlp_fused"] = entry(ms, 4.0 * M * E * HID, M * E * (2 + 4 + 4 + 2) + 4.0 * E * HID, M=M)
    # LayerNorm (+residual) stand-alone (stem / fp32 path): the plain bandwidth reference point
    r = torch.randn(M, E, device=dev, generator=g)
    y = torch.empty_like(x)
    ms = _time_kernel(torch, lambda: _lib.check(
        lib.mmpfn_layernorm(x.data_ptr(), r.data_ptr(), None, None, M, E, y.data_ptr(), xb.data_ptr(), st), "layernorm"))
    res["layernorm_residual"] = entry(ms, 0, M * E * (4 + 4 + 4 + 2))
    res["note"] = (f"M = {M} tokens (B={B} estimators x S={S} rows x T={T}); working sets of 0.4-0.7 GB exceed the "
                   "126 MB L2, timed back to back (20 launches)")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-gpu-reference", dest="gpu_reference", action="store_false",
                    help="skip the reference-on-CUDA baseline leg")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--profile", action="store_true",
                    help="for ncu: 1 warm-up + K device-resident steps only (no e2e / roofline / CPU legs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's per-estimator logits (rank 0) and the test rows' "
                         "probabilities (all ranks) as DIR/logits.npy and DIR/proba.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours only")
    if args.impl == "ours" and not args.profile:
        args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
