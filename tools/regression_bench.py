"""Regressor timing: the bar-distribution tail kernel alone, MMPFNRegressor.predict end to end split into forward,
decoder and tail, and the float64 host oracle of the tail for scale.

* Tail kernel: n_est = 8, K = 5000 buckets, S = 300 / 10 000 / 50 000 test rows, with and without the log P output
  (mean, median, mode and nine quantiles always).  CUDA events around single launches; a 512 MB buffer is
  overwritten between launches so that no launch reads logits left in the 126 MB L2 by the previous one.  GB/s from
  the byte model n_est*S*K*4 read (+ S*K*4 written with log P), against the HBM bandwidth of a device-to-device copy
  of 4 GB measured in the same run.
* predict: the PAD-UFES shape (2 000 train rows, 300 test rows, 21 columns, one embedding), 8 estimators, a synthetic
  5000-bucket regression checkpoint, bf16, both fit modes.  "forward" = engine logits (CUDA graph) minus the
  decoder, "decoder" = mmpfn_decode timed alone on the same [8, 300] rows, "tail" = mmpfn_bar_tail.
* host oracle: oracle/bar_distribution.py on the S = 300 logits, float64 numpy on the host cores.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from multimodalpfn_b200.preprocessing import transform_all  # noqa: E402
from multimodalpfn_b200.regressor import MMPFNRegressor, bar_tail_device, border_map, member_borders  # noqa: E402
from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict  # noqa: E402
from oracle import bar_distribution as O  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="300,10000,50000")
ap.add_argument("--reps", type=int, default=20)
args = ap.parse_args()

K, N_EST = 5000, 8
QS = torch.tensor(np.round(np.arange(1, 10) * 0.1, 1), dtype=torch.float32)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        q = ""
    return q or torch.cuda.get_device_name(0)


def timed(fn, reps, flush=None):
    """Median ms of single calls, each between CUDA events, L2 overwritten before each."""
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
print(f"card: {card()}")
flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

# HBM bandwidth of a plain device-to-device copy (read + write)
src = torch.empty(1 << 30, dtype=torch.float32, device=dev)
dst = torch.empty_like(src)
dst.copy_(src)
ms, _ = timed(lambda: dst.copy_(src), 10)
hbm = 2 * src.numel() * 4 / ms / 1e6
print(f"copy 4 GB device-to-device: {ms:.3f} ms -> {hbm:.0f} GB/s (read + write)")
del src, dst

g = np.asarray(make_state_dict(Geometry(mgm_heads=1, cap_heads=1, n_out=K, nlayers=1), seed=0,
                               regression=True)["criterion.borders"], dtype=np.float64)
rng = np.random.default_rng(0)
bks, shs, cns = [], [], []
y = rng.lognormal(0.0, 0.8, 2000)
y_z = (y - y.mean()) / y.std()
from sklearn.preprocessing import PowerTransformer  # noqa: E402
pt = PowerTransformer(method="yeo-johnson", standardize=True).fit(y_z[:, None])
for e in range(N_EST):
    f, c = member_borders(pt if e % 2 else None, g)
    b, s = border_map(f, g)
    bks.append(b), shs.append(s), cns.append(c)
bd = torch.from_numpy(np.stack(bks)).to(dev)
sd = torch.from_numpy(np.stack(shs)).to(dev)
cd = torch.from_numpy(np.stack(cns).astype(np.uint8)).to(dev) if np.any(cns) else None
G = g * 3.0 + 10.0
Gd = torch.from_numpy(G.astype(np.float32)).to(dev)
qd = QS.to(dev)

print(f"\n== tail kernel alone: n_est {N_EST}, K {K}, outputs mean/median/mode/9 quantiles (+ log P) ==")
logits300 = None
for S in [int(x) for x in args.sizes.split(",")]:
    lg = torch.randn((N_EST, S, K), device=dev) * 2.0
    if S == 300:
        logits300 = lg.cpu().numpy()
    for with_lp in (False, True):
        outs = ("mean", "median", "mode", "quantiles") + (("log_prob",) if with_lp else ())
        run = lambda: bar_tail_device(lg, bd, sd, cd, Gd, softmax_temperature=0.9, average_before_softmax=False,  # noqa: E731
                                      quantiles=qd, outputs=outs)
        run()
        torch.cuda.synchronize()
        ms, mn = timed(run, args.reps, flush)
        nbytes = N_EST * S * K * 4 + (S * K * 4 if with_lp else 0)
        print(f"S {S:6d}  log_prob {int(with_lp)}: median {ms:8.3f} ms (min {mn:.3f})  {nbytes / 1e9:6.3f} GB  "
              f"{nbytes / ms / 1e6:6.0f} GB/s = {nbytes / ms / 1e6 / hbm * 100:5.1f} % of the measured copy bandwidth")
    del lg
    torch.cuda.empty_cache()

if logits300 is not None:
    t0 = time.perf_counter()
    O.bar_tail(logits300.astype(np.float64), np.stack(bks), np.stack(shs).astype(np.float64), np.stack(cns), G,
               temperature=0.9, quantiles=tuple(QS.tolist()))
    print(f"\nhost oracle (float64 numpy, {os.cpu_count()} host cores), S 300: {(time.perf_counter() - t0) * 1e3:.0f} ms")

print(f"\n== MMPFNRegressor.predict: PAD-UFES shape, {N_EST} estimators, K {K}, bf16 ==")
d = make_dataset("pad_ufes", 0)
yv = np.exp(0.1 * np.nan_to_num(d["X_train"])[:, -3] / 15.0) + rng.normal(0, 0.1, len(d["X_train"]))
geom = Geometry(n_out=K)
sdict = make_state_dict(geom, seed=9, regression=True)
for mode in ("fit_preprocessors", "fit_with_cache"):
    reg = MMPFNRegressor(n_estimators=N_EST, model_path=(sdict, geom), device="cuda", inference_precision="bf16",
                         fit_mode=mode, random_state=0).fit(d["X_train"], d["img_train"], yv)
    for _ in range(3):
        reg.predict(d["X_test"], d["img_test"], output_type="main")
    torch.cuda.synchronize()
    walls = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        reg.predict(d["X_test"], d["img_test"], output_type="main")
        torch.cuda.synchronize()
        walls.append((time.perf_counter() - t0) * 1e3)
    X_tests = transform_all(reg.members_, d["X_test"])
    eng = reg.executor_
    staged = eng.stage(X_tests, d["img_test"])
    fwd_ms, _ = timed(lambda: eng.logits_graphed(staged), args.reps)
    state = torch.randn((N_EST, len(d["X_test"]), 2, 192), device=dev)
    dec_ms, _ = timed(lambda: reg.model_.decode(state), args.reps)
    lg = eng.logits_graphed(staged)
    tail_ms, _ = timed(lambda: bar_tail_device(lg, reg._src_bucket, reg._src_share, reg._cancel, reg._borders_dev,
                                               softmax_temperature=0.9, average_before_softmax=False, quantiles=qd,
                                               outputs=("mean", "median", "mode", "quantiles")), args.reps)
    print(f"{mode:18s}: predict wall median {np.median(walls):7.2f} ms | device: forward {fwd_ms - dec_ms:7.2f} ms, "
          f"decoder {dec_ms:6.2f} ms, tail {tail_ms:6.3f} ms")
print(f"\ncard (again): {card()}")
