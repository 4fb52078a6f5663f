"""bf16 against fp16 layer precision on bench.py's workload, in one process.

The workload is BASELINE.json configs[1] (PAD-UFES-20 shape: 2000 train / 300 test rows, 8 estimators, MGM+CAP 8/8):
the reference-equivalent device step of ``MMPFNClassifier`` (one CUDA-graph replay of ``executor_.logits_graphed``),
timed between CUDA events with the L2 overwritten (384 MB memset, not timed) before every step.  The two precisions
alternate step by step so that clocks, temperature and co-tenants affect both alike.  The same runs at the 64/24
MGM/CAP geometry, where the bf16 stem's MGM GEMM runs on tcgen05 and the fp16 stem's on the FFMA path.

Accuracy: each precision's max |dp| against the real reference's fp32 probabilities of ``large_clf8_pad_ufes``
(tests/golden), through the same multi-group pass.  The card's name and power limit are read in the same run.

    python tools/precision_bench.py --steps 30 --warmup 5 [--out profiles/r03_precision_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

PRECISIONS = ("bf16", "fp16")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as exc:          # the timing stands without it; say so
        return {"name": None, "error": str(exc)}


def dp_vs_reference(precision):
    import torch
    from multimodalpfn_b200.engine import proba_from_logits
    from multimodalpfn_b200.model import B200PerFeatureTransformer
    from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
    from tests.cases import load_golden
    g = load_golden("large_clf8_pad_ufes")
    geom = Geometry(mgm_heads=8, cap_heads=8)
    d = make_dataset("pad_ufes", 0)
    n_est, n_tr = int(g["n_estimators"]), len(d["y_train"])
    model = B200PerFeatureTransformer(make_state_dict(geom, seed=1), geom, precision=precision, seed=0)
    tok = model.stem_image(torch.as_tensor(np.concatenate([d["img_train"], d["img_test"]])).cuda())
    by_f = {}
    for e in range(n_est):
        by_f.setdefault(g[f"X_full_{e}"].shape[1], []).append(e)
    groups = [(es, torch.as_tensor(np.stack([g[f"X_full_{e}"] for e in es])).cuda(),
               torch.as_tensor(np.stack([g[f"y_train_{e}"] for e in es])).cuda()) for _, es in sorted(by_f.items())]
    ctxs = model.fit_contexts([dict(X_train=Xb[:, :n_tr].contiguous(), y_train=yb, X_all=Xb,
                                    img_tok_train=tok[:n_tr].contiguous()) for _, Xb, yb in groups])
    outs = model.predict_with_contexts(ctxs, [Xb[:, n_tr:].contiguous() for _, Xb, _ in groups],
                                       img_tok_test=tok[n_tr:].contiguous())
    logits = [None] * n_est
    for (es, _, _), out in zip(groups, outs):
        for i, e in enumerate(es):
            logits[e] = out[i]
    p = proba_from_logits(torch.stack(logits), [g[f"class_perm_{e}"] for e in range(n_est)],
                          n_classes=int(g["n_classes"]), class_counts=g["class_counts"])
    pr = g["proba"]
    return {"max_abs_dp": float(np.abs(p - pr).max()), "argmax_agreement": float((p.argmax(1) == pr.argmax(1)).mean())}


def timed_pair(mgm_heads, cap_heads, steps, warmup):
    """ms per step of each precision, alternating, on the configs[1] workload at the given MGM / CAP head counts."""
    import torch
    from multimodalpfn_b200.classifier import MMPFNClassifier
    from multimodalpfn_b200.preprocessing import transform_all
    from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict
    geom = Geometry(mgm_heads=mgm_heads, cap_heads=cap_heads)
    sd = make_state_dict(geom, seed=1)
    d = make_dataset("pad_ufes", 0)
    runs = {}
    for p in PRECISIONS:
        clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=mgm_heads, cap_heads=cap_heads, features_per_group=2,
                              n_estimators=8, model_path=(sd, geom), device="cuda", inference_precision=p,
                              ignore_pretraining_limits=True, random_state=0)
        clf.fit(d["X_train"], d["img_train"], d["y_train"])
        eng = clf.executor_
        staged = eng.stage(transform_all(clf.members_, d["X_test"]), d["img_test"])
        for _ in range(warmup):
            eng.logits_graphed(staged)
        runs[p] = (eng, staged)
    torch.cuda.synchronize()
    flush = torch.empty(384 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    evs = {p: [] for p in PRECISIONS}
    for i in range(steps):
        for p in (PRECISIONS if i % 2 == 0 else PRECISIONS[::-1]):
            eng, staged = runs[p]
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.logits_graphed(staged)
            b.record()
            evs[p].append((a, b))
    torch.cuda.synchronize()
    out = {}
    for p in PRECISIONS:
        ms = np.array([a.elapsed_time(b) for a, b in evs[p]])
        out[p] = {"ms_median": float(np.median(ms)), "ms_min": float(ms.min()), "ms_max": float(ms.max()),
                  "ms_p10": float(np.percentile(ms, 10)), "ms_p90": float(np.percentile(ms, 90))}
    out["fp16_over_bf16_median"] = out["fp16"]["ms_median"] / out["bf16"]["ms_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("precision_bench needs a CUDA device: there is no CPU measurement")
    res = {"card": card(), "workload": "configs[1]: PAD-UFES-20 shape, 2000 train / 300 test rows, 8 estimators, "
                                      "one CUDA-graph replay of the device step per timed step, L2 flushed between steps",
           "steps": args.steps, "warmup": args.warmup}
    res["configs1_mgm8_cap8"] = timed_pair(8, 8, args.steps, args.warmup)
    torch.cuda.empty_cache()
    res["mgm64_cap24"] = timed_pair(64, 24, args.steps, args.warmup)
    torch.cuda.empty_cache()
    res["dp_vs_reference_fp32_large_clf8_pad_ufes"] = {p: dp_vs_reference(p) for p in PRECISIONS}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
