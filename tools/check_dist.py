"""torchrun --nproc-per-node N tools/check_dist.py [--regression] — sharded engine (per-layer K/V all-gather over NCCL,
test pass reading the gather buffer in place) vs the unsharded engine on every rank's own test chunk: bit-identical
logits.  ``--regression``: ``MMPFNRegressor.predict(..., sharded=ShardedEngine)`` (every rank passes the whole test
table, runs its own chunk and gets the gathered result) vs the unsharded ``predict`` on every rank, "main" and "full"
outputs, estimator ownership (bf16, and fp32, which runs the broadcast mode) and row sharding (bf16): bit-identical."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
from multimodalpfn_b200.classifier import MMPFNClassifier
from multimodalpfn_b200.dist import ShardedEngine
from multimodalpfn_b200.engine import proba_from_logits
from multimodalpfn_b200.synth import Geometry, make_dataset, make_state_dict

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))


def regression():
    from multimodalpfn_b200.regressor import MMPFNRegressor
    geom = Geometry(mgm_heads=2, cap_heads=4, n_out=5000)
    sd = make_state_dict(geom, seed=9, regression=True)
    big = ("pad_ufes", 8) if world <= 4 else ("img_text_10k", 2)       # enough train rows for 48-row tiles per rank
    cases = [("pad_ufes_small", 8, "estimators", "bf16"), ("pad_ufes_small", 8, "estimators", "fp32"),
             ("pad_ufes_small", 3, "estimators", "bf16"), big + ("rows", "bf16"), (big[0], 1, "rows", "bf16")]
    for name, n_est, shard, precision in cases:
        d = make_dataset(name, 0)
        rng = np.random.default_rng(7)                                  # the same test table on every rank
        X = np.nan_to_num(np.concatenate([d["X_train"], d["X_test"]]))
        X = (X - X.mean(0)) / (X.std(0) + 1e-6)
        img = np.concatenate([d["img_train"], d["img_test"]])
        y = np.exp(0.3 * (X @ rng.normal(0, 0.4, X.shape[1]) + img[:, 0, :8].sum(1) * 0.2)) * 10
        y = (y + rng.normal(0, 0.5, len(y)))[:len(d["X_train"])]
        n_te = 117                                                       # unequal chunks at 2, 4 and 8 ranks
        Xte, img_te = d["X_test"][:n_te], d["img_test"][:n_te]
        reg = MMPFNRegressor(mgm_heads=2, cap_heads=4, n_estimators=n_est, model_path=(sd, geom), device=f"cuda:{local}",
                             inference_precision=precision, ignore_pretraining_limits=True,
                             random_state=0).fit(d["X_train"], d["img_train"], y)
        sh = ShardedEngine(reg.executor_, rank, world, shard=shard)
        for output_type in ("main", "full"):
            ref = reg.predict(Xte, img_te, output_type=output_type)
            got = reg.predict(Xte, img_te, output_type=output_type, sharded=sh)
            err, same = 0.0, set(got) == set(ref)
            for k in ref:
                a, b = np.asarray(got[k]), np.asarray(ref[k])
                same = same and a.shape == b.shape and np.array_equal(a, b)
                if a.shape == b.shape:
                    err = max(err, float(np.nanmax(np.abs(np.where(a == b, 0, a - b)))))
            print(f"rank {rank}/{world} regression {name} {n_est} estimator(s) {shard} {precision} {output_type} "
                  f"mode={sh.exchange['mode']}: {n_te} test rows, sharded == unsharded bit for bit: {same} "
                  f"(max |diff| = {err:.3e})", flush=True)
            assert same, (name, n_est, shard, precision, output_type, err)
        del reg, sh
        torch.cuda.empty_cache()


if "--regression" in sys.argv[1:]:
    regression()
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0)

geom = Geometry(mgm_heads=2, cap_heads=4)
sd = make_state_dict(geom, seed=1)
d = make_dataset("pad_ufes_small", 0)
rng = np.random.default_rng(5 + rank)
Xte = d["X_test"][rng.permutation(len(d["X_test"]))]
img = rng.standard_normal(d["img_test"].shape).astype(np.float32)
for precision in ("bf16", "fp32"):
    clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=2, cap_heads=4, n_estimators=8, model_path=(sd, geom),
                          device=f"cuda:{local}", inference_precision=precision, ignore_pretraining_limits=True,
                          random_state=0).fit(d["X_train"], d["img_train"], d["y_train"])
    X_tests = [m.transform(Xte) for m in clf.members_]
    ref = clf.executor_.logits(X_tests, img, graph=False).clone()
    sh = ShardedEngine(clf.executor_, rank, world)
    got = sh.logits(X_tests, img).clone()
    got2 = sh.logits(X_tests, img)                    # second call: the gather buffer is reused
    err = (got - ref).abs().max().item()
    perms = [m.class_perm for m in clf.members_]
    p = torch.as_tensor(proba_from_logits(got, perms, n_classes=clf.n_classes_)).cuda()
    allp = sh.proba_gathered(got, perms, n_classes=clf.n_classes_)
    ok = allp.shape[0] == world * p.shape[0] and torch.allclose(allp[rank * p.shape[0]:(rank + 1) * p.shape[0]], p, atol=1e-6)
    print(f"rank {rank}/{world} {precision} mode={sh.plan.mode}: max |sharded - unsharded| logits = {err:.3e}; "
          f"repeat equal = {bool(torch.equal(got, got2))}; gather ok = {bool(ok)}; exchange = {sh.exchange}", flush=True)
    assert err == 0.0 if sh.plan.mode != "broadcast" and precision == "bf16" else err < 1e-4, err
    assert ok and torch.equal(got, got2)

# ---- train rows sharded over the ranks (shard="rows"): bit-identical to the unsharded engine as well ----------------
name, n_est = ("pad_ufes", 8) if world <= 4 else ("img_text_10k", 2)
d = make_dataset(name, 0)
n_te = 120
Xte = d["X_test"][rng.permutation(len(d["X_test"]))[:n_te]]
img = rng.standard_normal((n_te,) + d["img_test"].shape[1:]).astype(np.float32)
for n_members in (n_est, 1):
    clf = MMPFNClassifier(mixer_type="MGM+CAP", mgm_heads=2, cap_heads=4, n_estimators=n_members, model_path=(sd, geom),
                          device=f"cuda:{local}", inference_precision="bf16", ignore_pretraining_limits=True,
                          random_state=0).fit(d["X_train"], d["img_train"], d["y_train"])
    X_tests = [m.transform(Xte) for m in clf.members_]
    ref = clf.executor_.logits(X_tests, img, graph=False).clone()
    sh = ShardedEngine(clf.executor_, rank, world, shard="rows")
    got = sh.logits(X_tests, img).clone()
    got2 = sh.logits(X_tests, img)
    err = (got - ref).abs().max().item()
    print(f"rank {rank}/{world} rows mode, {name}, {n_members} estimator(s), {sh.seg_rows} rows per rank: "
          f"max |sharded - unsharded| logits = {err:.3e}; repeat equal = {bool(torch.equal(got, got2))}; "
          f"exchange = {sh.exchange}", flush=True)
    assert err == 0.0 and torch.equal(got, got2), err
    del clf, sh
    torch.cuda.empty_cache()
dist.barrier()
dist.destroy_process_group()
