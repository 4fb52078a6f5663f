"""world_size-2 / -4 gloo tests (CPU) of the multi-GPU host logic in multimodalpfn_b200/dist.py: estimator
ownership, the layout of the per-layer all-gather buffer (``KvPlan``), that every estimator's K/V block of every
layer arrives where the test pass reads it, and that the sharded engine returns what the unsharded engine returns
for each rank's test chunk.  The CUDA model is replaced by an arithmetic stand-in with the same host interface
(embed / layers_run / decode; fit_contexts / predict_with_contexts built from the same arithmetic), so only the
plumbing is tested."""
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from multimodalpfn_b200.dist import KvPlan, ShardedEngine, all_gather_rows, local_members, owner_of
from multimodalpfn_b200.model import TrainContext

L, E = 3, 4


def test_ownership_partition():
    for world in (1, 2, 4, 8):
        members = list(range(8))
        seen = []
        for r in range(world):
            seen += [members[k] for k in local_members(members, r, world)]
        assert sorted(seen) == members
        assert all(owner_of(i, world) < world for i in members)
    assert local_members([1, 3, 5, 7], 1, 2) == [0, 1, 2, 3]
    assert local_members([1, 3, 5, 7], 0, 2) == []


def test_kv_plan_layouts():
    shapes = [(4, 27), (4, 20)]
    for world, mode in ((1, "split"), (2, "split"), (4, "split"), (8, "one_each"), (3, "broadcast"), (16, "broadcast")):
        plan = KvPlan(shapes, 2000, world)
        assert plan.mode == mode, (world, plan.mode)
        if mode == "broadcast":
            continue
        assert plan.chunk % 1024 == 0
        seen = {}
        for r in range(world):
            for gi, pos in plan.owned(r):
                for b in pos:
                    assert plan.locate(gi, b)[0] == r
                    seen[(gi, b)] = r
        assert sorted(seen) == [(gi, b) for gi in range(2) for b in range(4)]          # every estimator built once
        # blocks of one rank chunk do not overlap and fit
        for r in range(world):
            spans = sorted((plan.groups[gi].offset, plan.groups[gi].offset + plan.groups[gi].block) for gi, _ in plan.owned(r))
            assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:])) and spans[-1][1] <= plan.chunk
    p8 = KvPlan(shapes, 2000, 8)
    assert [g.rank0 for g in p8.groups] == [0, 4] and p8.chunk >= 2 * 27 * 2048 * 32 * 2 - 1024 * 0


class FakeLib:
    def mmpfn_tab_stats_elems(self, g, G):
        return 6 * 2 * G + G

    def mmpfn_kv_bytes(self, g, B, n_tr, T, precision):
        return L * B * T * 8


class FakeModel:
    """Same host interface as B200PerFeatureTransformer, arithmetic instead of kernels.  A layer of the train pass
    stores, per estimator and token column, the row sum of its state (float64) as that layer's "K/V block" and then
    moves the state on; a layer of the test pass adds what it finds in the context to the test state."""
    device = torch.device("cpu")
    precision = 1
    lib = FakeLib()
    _g = None
    geom = types.SimpleNamespace(nlayers=L, emsize=E)

    def _n_groups(self, F):
        return (F + 1) // 2

    def n_image_tokens(self, n_tok):
        return 3

    def stem_image(self, img):
        return img[:, :, :E].mean(1, keepdim=True).repeat(1, 3, 1)          # [S, 3, E]

    def positional_embeddings(self, n):
        return torch.arange(n, dtype=torch.float32)

    @staticmethod
    def label_stats(y):
        return y.mean(1), y.sum(1).to(torch.int64)

    def _check_nan(self, flag):
        assert int(flag.item()) == 0

    def stem_tab_fit(self, X, n_train):
        B, S, F = X.shape
        G = self._n_groups(F)
        return X[:, :n_train].mean(1).repeat(1, 7)[:, : 6 * 2 * G + G].contiguous()

    def _group_buffers(self, shapes):
        total = sum(b * s * t for b, s, t in shapes)
        st = torch.zeros((total, E), dtype=torch.float32)
        stb = torch.zeros((total, E), dtype=torch.float32)
        views, off = [], 0
        for b, s, t in shapes:
            n = b * s * t
            views.append((st[off:off + n].view(b, s, t, E), stb[off:off + n].view(b, s, t, E)))
            off += n
        return st, stb, views

    def embed(self, X, stats, img_tok, y, y_mean, y_mask, pos_emb, *, B, S, F, x_bstride, y_bstride, nan_flag, out=None):
        G = self._n_groups(F)
        T = G + img_tok.shape[-2] + 1
        state = out[0] if out is not None else torch.zeros((B, S, T, E))
        base = X.sum(2)[:, :, None] + stats.sum(1)[:, None, None] + torch.arange(T, dtype=torch.float32)[None, None]
        state[:] = (base + img_tok.sum((1, 2))[None, :, None] + y_mean[:, None, None])[..., None]
        yy = torch.nan_to_num(y, nan=-1.0)
        state[:, :, T - 1, :] += yy.expand(B, S)[..., None]
        return state, None

    def layers_run(self, state, state_b, segs, S, n_train, l0, l1, phase=0, ws_key=""):
        off = 0
        for sg in segs:
            B, T = sg["B"], sg["T"]
            st = state[off:off + B * S * T].view(B, S, T, E)
            off += B * S * T
            rows = sg.get("bufs")                       # row-sharded mode (dist.py "rows"): buffers by rank
            flat = None if rows is not None else sg["kv_buffer"].view(-1)
            for l in range(l0, l1):
                if n_train is None and rows is not None:
                    # train rows sharded: phase 1 leaves this rank's partial row sum in its gather chunk and its
                    # context block; phase 2 (after the caller's all-gather) moves the state on with the total
                    r = sg["rank"]
                    if phase != 2:
                        part = st[..., 0].sum(1).double()
                        rows["kg"][r][:B * T * 8].view(torch.float64).view(B, T)[:] = part
                        rows["ctx"][r, l][:B * T * 8].view(torch.float64).view(B, T)[:] = part + (l if r == 0 else 0)
                    if phase != 1:
                        tot = sum(rows["kg"][k][:B * T * 8].view(torch.float64).view(B, T) for k in range(sg["n_ranks"]))
                        st.mul_(0.5).add_(1.0).add_((tot.float() * 1e-4)[:, None, :, None])
                elif n_train is None:                   # train: write this layer's block [B][T] float64
                    a = sg["kv_offset"] + l * (sg["layer_stride"] or B * T * 8)
                    tot = st[..., 0].sum(1).double()
                    flat[a:a + B * T * 8].view(torch.float64).view(B, T)[:] = tot + l
                    st.mul_(0.5).add_(1.0).add_((tot.float() * 1e-4)[:, None, :, None])
                elif rows is not None:                  # test against a row-sharded context: the chunks add up
                    for b in range(B):
                        ctx = sum(rows["ctx"][k, l][b * T * 8:(b + 1) * T * 8].view(torch.float64) for k in range(sg["n_ranks"]))
                        st[b] = st[b] * 0.5 + (ctx.float() * 1e-3)[None, :, None]
                else:                                   # test: read estimator b at (rank, slot)
                    c = sg["slots"] or B
                    for b in range(B):
                        a = sg["kv_offset"] + l * (sg["layer_stride"] or B * T * 8) + (b // c) * sg["rank_stride"] + (b % c) * T * 8
                        ctx = flat[a:a + T * 8].view(torch.float64)
                        st[b] = st[b] * 0.5 + (ctx.float() * 1e-3)[None, :, None]

    def decode(self, state):
        return state[:, :, -1, :1].repeat(1, 1, 10) + state.mean((2, 3))[..., None]

    # ---- the unsharded engine's entry points, from the same arithmetic -------------------------------------
    def fit_contexts(self, specs, *, nan_flag=None):
        ctxs = []
        for sp in specs:
            X_train, X_all, img_tok_train = sp["X_train"], sp.get("X_all"), sp["img_tok_train"]
            B, n_tr, F = X_train.shape
            stats = self.stem_tab_fit(X_all if X_all is not None else X_train, n_tr)
            y_mean, y_mask = sp["label_stats"] if sp.get("label_stats") is not None else self.label_stats(sp["y_train"])
            T = self._n_groups(F) + img_tok_train.shape[1] + 1
            st, _, views = self._group_buffers([(B, n_tr, T)])
            self.embed(X_train, stats, img_tok_train, sp["y_train"], y_mean, y_mask, None, B=B, S=n_tr, F=F, x_bstride=0,
                       y_bstride=0, nan_flag=None, out=views[0])
            kv = torch.zeros(L * B * T * 8, dtype=torch.uint8)
            self.layers_run(st, None, [dict(B=B, T=T, kv=kv, layer_stride=0, slots=0, rank_stride=0, kv_buffer=kv,
                                            kv_offset=0)], n_tr, None, 0, L)
            ctxs.append(TrainContext(B=B, n_train=n_tr, F=F, T=T, kv=kv, tab_stats=stats, y_mean=y_mean, y_mask=y_mask,
                                     pos_emb=None, precision=1))
        return ctxs

    def merge_kv(self, parts, B, n_train, T):
        out = torch.zeros(L * B * T * 8, dtype=torch.uint8)
        for kv, pos in parts:
            out.view(torch.float64).view(L, B, T)[:, pos] = kv.view(torch.float64).view(L, len(pos), T)
        return out

    def predict_with_contexts(self, ctxs, X_tests, *, img_tok_test=None, nan_flag=None):
        logits = []
        for ctx, X_test in zip(ctxs, X_tests):
            B, n_te, F = X_test.shape
            st, _, views = self._group_buffers([(B, n_te, ctx.T)])
            y_nan = torch.full((1, n_te), float("nan"))
            self.embed(X_test, ctx.tab_stats, img_tok_test, y_nan, ctx.y_mean, ctx.y_mask, None, B=B, S=n_te, F=F,
                       x_bstride=0, y_bstride=0, nan_flag=None, out=views[0])
            self.layers_run(st, None, [dict(B=B, T=ctx.T, kv=ctx.kv, layer_stride=0, slots=0, rank_stride=0,
                                            kv_buffer=ctx.kv, kv_offset=0)], n_te, ctx.n_train, 0, L)
            logits.append(self.decode(views[0][0]))
        return logits


def _make_engine(rank_seed, n_a=4, n_b=4, n_train=20):
    from multimodalpfn_b200.engine import B200InferenceEngine
    rng = np.random.default_rng(0)
    members = []
    for e in range(n_a + n_b):
        F = 6 if e < n_a else 4
        members.append(dict(X_train=rng.standard_normal((n_train, F)).astype(np.float32),
                            y_train=rng.integers(0, 3, n_train).astype(np.float32), class_perm=None))
    img_train = rng.standard_normal((n_train, 1, 8)).astype(np.float32)
    eng = B200InferenceEngine(FakeModel(), members, img_train)
    rng2 = np.random.default_rng(10 + rank_seed)
    X_tests = [rng2.standard_normal((5, m["X_train"].shape[1])).astype(np.float32) for m in members]
    img_test = rng2.standard_normal((5, 1, 8)).astype(np.float32)
    return eng, X_tests, img_test


def _worker(rank, world, port, q, n_a, n_b, shard="estimators", n_train=20):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        eng, X_tests, img_test = _make_engine(rank, n_a, n_b, n_train)
        ref = eng.logits(X_tests, img_test, graph=False)          # unsharded, this rank's chunk
        sh = ShardedEngine(eng, rank, world, shard=shard)
        got = sh.logits(X_tests, img_test)
        got2 = sh.logits(X_tests, img_test)                       # the gather buffer is reused across calls
        ok = bool(torch.allclose(got, ref, rtol=0, atol=1e-4)) and bool(torch.equal(got, got2))
        rows = all_gather_rows(got[0, :, :3].contiguous())
        ok2 = rows.shape == (world * 5, 3) and torch.equal(rows[rank * 5:(rank + 1) * 5], got[0, :, :3])
        owned = sorted(i for s in sh.subs if s.owner == rank for i in s.members)
        q.put((rank, ok, ok2, owned, sh.exchange["mode"], float((got - ref).abs().max())))
    finally:
        dist.destroy_process_group()


def _run(world, n_a=4, n_b=4, shard="estimators", n_train=20):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, n_a, n_b, shard, n_train)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def test_sharded_engine_world2_split():
    res = _run(2)
    assert all(r[1] and r[2] for r in res), res
    assert all(r[4] == "split" for r in res)
    assert sorted(res[0][3] + res[1][3]) == list(range(8))
    assert res[0][3] == [0, 1, 4, 5] and res[1][3] == [2, 3, 6, 7]       # two consecutive estimators of each group


def test_sharded_engine_world4_one_each():
    res = _run(4, n_a=2, n_b=2)                                           # 4 estimators on 4 ranks: one each
    assert all(r[1] and r[2] for r in res), res
    assert all(r[4] == "one_each" for r in res)
    assert [r[3] for r in res] == [[2], [3], [0], [1]]          # groups in feature-count order: F=4 (members 2, 3) first


def test_sharded_engine_world4_split():
    res = _run(4)                                                         # 4 + 4 estimators on 4 ranks: one of each group per rank
    assert all(r[1] and r[2] for r in res), res
    assert all(r[4] == "split" for r in res)
    assert [r[3] for r in res] == [[0, 4], [1, 5], [2, 6], [3, 7]]


def test_sharded_engine_world2_broadcast_fallback():
    res = _run(2, n_a=3, n_b=2)                                           # 3 + 2 estimators on 2 ranks: round-robin + broadcast
    assert all(r[1] and r[2] for r in res), res
    assert all(r[4] == "broadcast" for r in res)
    assert sorted(res[0][3] + res[1][3]) == list(range(5))


def test_sharded_engine_world2_rows():
    """Train rows split over the ranks (96 + 4 of 100 rows: the last rank's segment is ragged)."""
    res = _run(2, n_a=2, n_b=1, shard="rows", n_train=100)
    assert all(r[1] and r[2] for r in res), res
    assert all(r[4] == "rows" for r in res)


def test_sharded_engine_world4_rows_single_estimator():
    res = _run(4, n_a=1, n_b=0, shard="rows", n_train=190)            # 48 + 48 + 48 + 46 rows of ONE estimator
    assert all(r[1] and r[2] for r in res), res


def test_rows_mode_rejects_short_tables():
    eng, _, _ = _make_engine(0, 1, 0, n_train=96)
    with pytest.raises(ValueError, match="too few"):
        ShardedEngine(eng, 0, 4, shard="rows")


@pytest.mark.parametrize("world", [2, 3])
def test_rows_mode_emulated_in_process(world):
    """All ranks' row shares one after the other in this process (no process group): same logits as unsharded."""
    eng, X_tests, img_test = _make_engine(0, 2, 1, n_train=250)
    ref = eng.logits(X_tests, img_test, graph=False)
    sh = ShardedEngine(eng, 0, world, group="emulate", shard="rows")
    got = sh.logits(X_tests, img_test)
    assert torch.allclose(got, ref, rtol=0, atol=1e-4), float((got - ref).abs().max())
