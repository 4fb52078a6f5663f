"""Multi-GPU partitioning of the hot path on one NVLink/NVSwitch box (SURVEY.md section 8(e)).

One process per GPU (``torch.distributed``, backend ``nccl``; ``gloo`` in the CPU tests).  The
path shards along its two independent axes:

* **ensemble estimators** — the train context of an estimator (the 12-layer head-0 K/V of its train
  rows) is built once, on the rank that owns it;
* **test rows** — every rank classifies its own chunk of test rows against ALL estimators.

The one real exchange step sits between the two.  Per layer ``l`` the K/V blocks the ranks have just
written are **all-gathered** (``all_gather_into_tensor``, in place: every rank builds its block at its
own offset of the gather buffer) on a communication stream, as soon as the owner's layer ``l`` has run:
the transfer of layer ``l`` overlaps layers ``l+1 .. 11`` of the context build and only the last one is
exposed.  The buffer is laid out so that the test pass reads it where it lands — ``[layer][rank][group:
K[slots][T][Np][32], V^T[slots][T][32][Np]]`` addressed by a 5-D TMA tensor map (estimator ``b`` of a
group = (rank, slot)) — so nothing is re-gathered or merged.  The per-rank probabilities (classifier) or the
requested bar-distribution outputs (regressor) are all-gathered at the end.  Nothing else crosses GPUs.

Test rows: rank r runs rows [r * c, (r + 1) * c) of the table, c = ceil(Nte / W) (``ShardedEngine.test_rows``); a short
or empty last chunk repeats the table's last row, so that every rank's outputs have the same shape for the all-gather,
and the gathered rows past Nte are dropped.

Ownership (``KvPlan``): with W ranks and groups of B_g estimators (one group per preprocessed feature
count),
* W divides every B_g  -> every rank owns B_g / W consecutive estimators of EVERY group (W = 1, 2, 4 at
  the 4 + 4 estimators of the default ensemble), all rank chunks are equally full;
* W == sum of B_g      -> one estimator per rank, the groups take consecutive rank ranges (W = 8), chunks
  are padded to the largest group's block;
* anything else        -> the estimators are dealt round-robin and every context is broadcast from its owner
  after the build (``_logits_broadcast``, the round-1 path: no overlap, merged on arrival).

The stem statistics of every estimator are cheap (one column-reduction launch per group) and are computed
by every rank for itself from the train rows plus ITS test chunk (``encoders.py:515, 615`` look at all rows
of the call; after preprocessing no train column is constant, so every chunk gives the same mask — SURVEY.md
section 8(e) caveat).
"""
from __future__ import annotations

import dataclasses
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

__all__ = ["owner_of", "local_members", "broadcast_bundle", "all_gather_rows", "KvPlan", "ShardedEngine"]


def owner_of(member: int, world: int) -> int:
    return member % world


def local_members(members: List[int], rank: int, world: int) -> List[int]:
    """Positions (within ``members``) of the estimators this rank owns (round-robin dealing)."""
    return [k for k, i in enumerate(members) if owner_of(i, world) == rank]


def broadcast_bundle(tensors: Optional[List[torch.Tensor]], shapes: List[Tuple[torch.Size, torch.dtype]], src: int,
                     device, group=None) -> List[torch.Tensor]:
    """Broadcast a list of tensors from ``src``; non-owners allocate from ``shapes``."""
    out = []
    for k, (shape, dtype) in enumerate(shapes):
        t = tensors[k].contiguous() if tensors is not None else torch.empty(shape, dtype=dtype, device=device)
        dist.broadcast(t, src=src, group=group)
        out.append(t)
    return out


def all_gather_rows(x: torch.Tensor, group=None) -> torch.Tensor:
    """[rows, c] per rank (same shape on every rank) -> [world*rows, c], rank-major (one ncclAllGather)."""
    world = dist.get_world_size(group)
    out = torch.empty((world * x.shape[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, x.contiguous(), group=group)
    return out


@dataclasses.dataclass
class GroupPlan:
    B: int                 # estimators of the group
    T: int                 # tokens per row
    slots: int             # estimators of the group stored back to back in one rank chunk
    rank0: int             # first rank holding estimators of this group
    n_ranks: int           # ranks holding them (B == slots * n_ranks)
    offset: int            # byte offset of the group's block inside a rank chunk
    block: int             # bytes of the block: K[slots][T][Np][32] + V^T[slots][T][32][Np]


class KvPlan:
    """Where every estimator's per-layer K/V lives in the gather buffer ``[L][W][chunk]`` (bytes)."""

    def __init__(self, group_shapes: List[Tuple[int, int]], n_train: int, world: int, *, elem_bytes: int = 2,
                 d: int = 32, pad: int = 64):
        self.world = world
        self.n_pad = (n_train + pad - 1) // pad * pad
        self.slab = lambda T: 2 * T * self.n_pad * d * elem_bytes           # K + V^T of ONE estimator
        Bs = [b for b, _ in group_shapes]
        self.groups: List[GroupPlan] = []
        if all(b % world == 0 for b in Bs):
            self.mode = "split"
            off = 0
            for b, t in group_shapes:
                c = b // world
                self.groups.append(GroupPlan(b, t, c, 0, world, off, c * self.slab(t)))
                off += c * self.slab(t)
            self.chunk = off
        elif sum(Bs) == world:
            self.mode = "one_each"
            r0 = 0
            for b, t in group_shapes:
                self.groups.append(GroupPlan(b, t, 1, r0, b, 0, self.slab(t)))
                r0 += b
            self.chunk = max(g.block for g in self.groups)
        else:
            self.mode = "broadcast"
            self.chunk = 0
        self.chunk = (self.chunk + 1023) // 1024 * 1024

    def owned(self, rank: int) -> List[Tuple[int, List[int]]]:
        """[(group index, positions of the group's batch this rank builds)]"""
        out = []
        for gi, g in enumerate(self.groups):
            if g.rank0 <= rank < g.rank0 + g.n_ranks:
                r = rank - g.rank0
                out.append((gi, list(range(r * g.slots, (r + 1) * g.slots))))
        return out

    def locate(self, gi: int, b: int) -> Tuple[int, int]:
        """estimator ``b`` of group ``gi`` -> (rank, slot)"""
        g = self.groups[gi]
        return g.rank0 + b // g.slots, b % g.slots


class ShardedEngine:
    """Wraps a ``B200InferenceEngine``: contexts are built by their owner ranks and all-gathered layer by
    layer under the build; every rank runs its own test rows against all of them."""

    def __init__(self, engine, rank: int, world: int, group=None, shard: str = "estimators"):
        """``shard="estimators"`` (default): every estimator's context is built by one owner rank (module docstring).
        ``shard="rows"``: the TRAIN ROWS of every estimator are split over the ranks (``_logits_rows``) — the mode for
        fewer estimators than GPUs, where a single estimator's 50 000-row self-attention would otherwise run on one
        GPU (SURVEY.md section 8(f) rank 2).  ``group="emulate"``: this process plays all ``world`` ranks on one device,
        without any collective (tests of the addressing on a single GPU).  With ``shard="rows"`` the shares of all ranks
        run one after the other; with estimator ownership every rank's owned build runs in turn into its offset of the
        gather buffer (which then holds every rank's block, as after the all-gathers), or, in the broadcast mode, every
        owner's contexts are built in turn and merged.  Then the staged test rows run, which for ``test_rows`` are the
        chunks of all ranks, and the gathers of ``proba_gathered`` / ``regression_gathered`` have nothing to move."""
        self.engine = engine
        self.shard = shard
        self.model = engine.model
        self.rank, self.world, self.group = rank, world, group
        self.emulate = group == "emulate"
        self.groups = engine.groups
        self.members = engine.members
        m = self.model
        if getattr(m, "precision", None) == 2:        # _lib.F16
            raise ValueError("ShardedEngine does not run fp16 models (the multi-GPU layer entry point is bf16 only); "
                             "build the model with precision='bf16' or 'fp32'")
        n_tr = engine.groups[0]["y_train"].shape[1]
        H_img = 0
        if engine.img_train_dev is not None:
            H_img = m.n_image_tokens(engine.img_train_dev.shape[1])
        self.Ts = [(m._n_groups(g["F"]) if g["F"] >= 0 else 0) + H_img + 1 for g in engine.groups]
        tabular = all(g["F"] >= 0 for g in engine.groups) and getattr(m, "precision", None) == 1 \
            and hasattr(m, "layers_run") and len(engine.groups) <= 8
        self.plan = KvPlan([(len(g["idx"]), t) for g, t in zip(engine.groups, self.Ts)], n_tr, world)
        if not tabular:
            self.plan.mode = "broadcast"
        self.subs = []        # (group, owner, positions, member ids): who builds what
        if self.plan.mode == "broadcast":
            for gi, g in enumerate(engine.groups):
                for r in range(world):
                    pos = local_members(g["idx"], r, world)
                    if pos:
                        self.subs.append(_Sub(gi, r, pos, [g["idx"][k] for k in pos]))
        else:
            for r in range(world):
                for gi, pos in self.plan.owned(r):
                    self.subs.append(_Sub(gi, r, pos, [engine.groups[gi]["idx"][k] for k in pos]))
        self._gather = None
        self._comm = None
        self._rows = None          # buffers of the row-sharded mode
        self._side = None          # side stream: stem + embedding of the test rows beside the context build
        self.exchange = None       # filled per call: bytes gathered, for the bench line
        if shard == "rows":
            if not tabular:
                raise ValueError("row sharding needs the bf16 path and tabular estimator groups")
            # rows per rank: a multiple of the 48-key attention tile, so that key tiles never straddle two ranks and
            # are exactly the tiles of the unsharded layout (bit-identical results)
            self.seg_rows = -(-(-(-n_tr // world)) // 48) * 48
            if (world - 1) * self.seg_rows >= n_tr:
                raise ValueError(f"{n_tr} train rows are too few to shard over {world} ranks in tiles of 48")

    # ------------------------------------------------------------------------------------------------
    def stage(self, X_test_per_member, image_test):
        return self.engine.stage(X_test_per_member, image_test)

    def test_rows(self, n_test: int) -> np.ndarray:
        """Row indices (into a table of ``n_test`` test rows) that this rank runs: rows [r * c, (r + 1) * c) with
        c = ceil(n_test / W), a short or empty chunk padded by repeating row ``n_test - 1``.  Test rows are independent
        and a repeated row cannot change the stem's "column varies over all rows" test, so the padding changes no real
        row's result.  ``group="emulate"``: the chunks of all ranks, rank-major."""
        if n_test < 1:
            raise ValueError("no test rows")
        c = -(-n_test // self.world)
        ranks = range(self.world) if self.emulate else [self.rank]
        return np.concatenate([np.minimum(np.arange(r * c, (r + 1) * c), n_test - 1) for r in ranks])

    def _gather_rows(self, x: torch.Tensor) -> torch.Tensor:
        """``all_gather_rows``; emulated, this process already holds the rows of every rank."""
        return x if self.emulate else all_gather_rows(x, self.group)

    def _buffers(self):
        m = self.model
        if self._gather is None:
            L = m.geom.nlayers
            self._gather = torch.empty((L, self.world, self.plan.chunk), dtype=torch.uint8, device=m.device)
            if m.device.type == "cuda":
                self._comm = torch.cuda.Stream(device=m.device)
        return self._gather

    def logits_staged(self, staged) -> torch.Tensor:
        if self.shard == "rows":
            return self._logits_rows(staged)
        if self.plan.mode == "broadcast":
            return self._logits_broadcast(staged)
        eng, m, plan = self.engine, self.model, self.plan
        dev = m.device
        cuda = dev.type == "cuda"
        eng.nan_flag.zero_()
        flag = eng.nan_flag
        G = self._buffers()
        L = m.geom.nlayers
        n_tr = eng.groups[0]["y_train"].shape[1]
        tok_tr = eng.train_image_tokens() if staged["img_test"] is not None else None
        # stem statistics of every estimator from the train rows + this rank's test chunk (cheap, no exchange)
        stats = [m.stem_tab_fit(torch.cat([g["X_train"], Xte], dim=1), n_tr)
                 for g, Xte in zip(eng.groups, staged["X_test"])]
        # The image/text stem and the token embedding of this rank's TEST rows (a dozen small launches) do not depend
        # on the context build: they run on a side stream beside it and join before the first test layer.
        n_te = staged["X_test"][0].shape[1]

        def embed_test_rows():
            tok_te = m.stem_image(staged["img_test"]) if staged["img_test"] is not None else None
            y_nan = torch.full((1, n_te), float("nan"), dtype=torch.float32, device=dev)
            bufs = m._group_buffers([(len(g["idx"]), n_te, t) for g, t in zip(eng.groups, self.Ts)])
            for gi, (g, v) in enumerate(zip(eng.groups, bufs[2])):
                ls = g["label_stats"]
                m.embed(staged["X_test"][gi], stats[gi], tok_te, y_nan, ls[0], ls[1], m.positional_embeddings(self.Ts[gi] - 1),
                        B=len(g["idx"]), S=n_te, F=g["F"], x_bstride=n_te * g["F"], y_bstride=0, nan_flag=flag, out=v)
            return bufs
        test_ready = None
        # (from 32 MGM heads the stem has a TMA / tcgen05 kernel: keep it in line; emulated ranks run in line too)
        if cuda and m.geom.mgm_heads < 32 and not self.emulate:
            main = torch.cuda.current_stream(dev)
            if self._side is None:
                self._side = torch.cuda.Stream(device=dev)
            self._side.wait_stream(main)
            with torch.cuda.stream(self._side):
                st2, stb2, views2 = embed_test_rows()
                test_ready = torch.cuda.Event()
                test_ready.record(self._side)
            for tns in (st2, stb2):
                tns.record_stream(main)
        else:
            st2, stb2, views2 = embed_test_rows()
        # ---- 1. context build of the estimators this rank owns, all-gather of layer l under layers l+1.. -------
        # (``group="emulate"``: the owned builds of all ranks, each into its own offset of the gather buffer)
        builds = []
        for rk in (range(self.world) if self.emulate else [self.rank]):
            owned = plan.owned(rk)
            shapes = [(len(pos), n_tr, self.Ts[gi]) for gi, pos in owned]
            st, stb, views = m._group_buffers(shapes)
            segs = []
            for (gi, pos), v in zip(owned, views):
                g, gp = eng.groups[gi], plan.groups[gi]
                # the label statistics of the whole group, never of this rank's estimators (float targets: DESIGN.md
                # section 6, label-mean rule)
                ls = g["label_stats"]
                sel = slice(pos[0], pos[-1] + 1)
                m.embed(g["X_train"][sel].contiguous(), stats[gi][sel].contiguous(), tok_tr, g["y_train"][sel].contiguous(),
                        ls[0][sel].contiguous(), ls[1][sel].contiguous(), m.positional_embeddings(self.Ts[gi] - 1),
                        B=len(pos), S=n_tr, F=g["F"], x_bstride=n_tr * g["F"], y_bstride=n_tr, nan_flag=flag, out=v)
                segs.append(dict(B=len(pos), T=self.Ts[gi], kv=G[0, rk, gp.offset:gp.offset + gp.block],
                                 layer_stride=self.world * plan.chunk, slots=0, rank_stride=0,
                                 kv_buffer=G, kv_offset=rk * plan.chunk + gp.offset))
            builds.append((st, stb, segs))
        # this rank's test rows against every estimator read the gathered buffer in place (5-D tensor maps)
        tsegs = []
        for gi, g in enumerate(eng.groups):
            gp = plan.groups[gi]
            tsegs.append(dict(B=len(g["idx"]), T=self.Ts[gi], kv=G[0, gp.rank0, gp.offset:gp.offset + gp.block],
                              layer_stride=self.world * plan.chunk, slots=gp.slots, rank_stride=plan.chunk,
                              kv_buffer=G, kv_offset=gp.rank0 * plan.chunk + gp.offset))
        # Three streams: the build of layer l (main), its all-gather (communication stream, under the build of layers
        # l+1..), and — as soon as layer l of every estimator has landed — layer l of the TEST rows (side stream, under
        # the build of layer l+1: at few estimators per rank both passes are made of short launches that leave SMs idle in
        # their tails).  The launches are issued in this order, so every stream finds its work in dependency order.
        interleave = cuda and test_ready is not None
        landed = []
        for l in range(L):
            for st, stb, segs in builds:
                if segs:
                    m.layers_run(st, stb, segs, n_tr, None, l, l + 1)
            if self.emulate:
                continue
            if cuda:
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(dev))
                with torch.cuda.stream(self._comm):
                    self._comm.wait_event(ev)
                    dist.all_gather_into_tensor(G[l].view(-1), G[l, self.rank], group=self.group)
                    done = torch.cuda.Event()
                    done.record(self._comm)
                landed.append(done)
                if interleave:
                    with torch.cuda.stream(self._side):
                        self._side.wait_event(done)
                        m.layers_run(st2, stb2, tsegs, n_te, n_tr, l, l + 1, ws_key="_test")
            else:
                dist.all_gather_into_tensor(G[l].view(-1), G[l, self.rank].clone(), group=self.group)
        self.exchange = {"collective": None, "mode": plan.mode} if self.emulate else \
            {"collective": "all_gather_into_tensor", "calls_per_step": L,
             "bytes_received_per_rank": int(L * (self.world - 1) * plan.chunk), "mode": plan.mode}
        if interleave:
            torch.cuda.current_stream(dev).wait_stream(self._side)
        else:
            for l in range(L):
                if cuda and not self.emulate:
                    torch.cuda.current_stream(dev).wait_event(landed[l])
                m.layers_run(st2, stb2, tsegs, n_te, n_tr, l, l + 1)
        out = [None] * len(self.members)
        for g, v in zip(eng.groups, views2):
            lg = m.decode(v[0])
            for k, i in enumerate(g["idx"]):
                out[i] = lg[k]
        return torch.stack(out)

    # ------------------------------------------------------------------------------------------------
    def _logits_rows(self, staged) -> torch.Tensor:
        """Row-sharded context build.  Rank r holds train rows [r * seg_rows, (r+1) * seg_rows) of EVERY estimator and
        runs the row-wise sublayers (feature attention, projections, MLP, LayerNorms) on them alone.  For the item
        attention each rank writes its rows' K / V^T planes into its chunk of two gather buffers, the buffers are
        all-gathered (two ``all_gather_into_tensor`` per layer, in place), and the rank's query rows attend to all
        keys through row-segmented tensor maps: no all-to-all, the state never leaves its rank.  The head-0 K/V blocks
        every rank kept for its rows are all-gathered once after the last layer into the context the test pass reads
        (again as row segments).  Work per rank: 1/W of everything; bit-identical to the unsharded engine."""
        eng, m = self.engine, self.model
        dev = m.device
        W, r, L = self.world, self.rank, m.geom.nlayers
        eng.nan_flag.zero_()
        flag = eng.nan_flag
        n_tr = eng.groups[0]["y_train"].shape[1]
        seg = self.seg_rows
        Sp = (seg + 63) // 64 * 64
        if self._rows is None:
            bufs = []
            for g, T in zip(eng.groups, self.Ts):
                B = len(g["idx"])
                chunk = B * T * 6 * Sp * 32 * 2                 # K (or V^T) planes of one rank's rows
                block = 2 * B * T * Sp * 32 * 2                 # head-0 K0 + V0^T of one layer, one rank's rows
                bufs.append(dict(kg=torch.zeros((W, chunk), dtype=torch.uint8, device=dev),
                                 vtg=torch.zeros((W, chunk), dtype=torch.uint8, device=dev),
                                 ctx=torch.zeros((W, L, block), dtype=torch.uint8, device=dev), chunk=chunk, block=block))
            self._rows = bufs
        bufs = self._rows
        tok_tr = tok_te = None
        if staged["img_test"] is not None:
            tok_tr, tok_te = eng.train_image_tokens(), m.stem_image(staged["img_test"])
        stats = [m.stem_tab_fit(torch.cat([g["X_train"], Xte], dim=1), n_tr)
                 for g, Xte in zip(eng.groups, staged["X_test"])]
        # ---- context build on this rank's rows of every estimator ---------------------------------------------
        # (``group="emulate"``: all W ranks' shares one after the other on this device, no collective — the
        # single-GPU test of the segment addressing)
        emulate = self.group == "emulate"
        shares = []
        for rk in (range(W) if emulate else [r]):
            lo, hi = rk * seg, min((rk + 1) * seg, n_tr)
            S_loc = hi - lo
            st, stb, views = m._group_buffers([(len(g["idx"]), S_loc, T) for g, T in zip(eng.groups, self.Ts)])
            segs = []
            for gi, (g, v) in enumerate(zip(eng.groups, views)):
                ls, b = g["label_stats"], bufs[gi]
                m.embed(g["X_train"][:, lo:hi].contiguous(), stats[gi], None if tok_tr is None else tok_tr[lo:hi].contiguous(),
                        g["y_train"][:, lo:hi].contiguous(), ls[0], ls[1], m.positional_embeddings(self.Ts[gi] - 1),
                        B=len(g["idx"]), S=S_loc, F=g["F"], x_bstride=S_loc * g["F"], y_bstride=S_loc, nan_flag=flag, out=v)
                segs.append(dict(B=len(g["idx"]), T=self.Ts[gi], kv=b["ctx"][rk, 0], layer_stride=b["block"], seg_rows=seg,
                                 kg=b["kg"], vtg=b["vtg"], gather_stride=b["chunk"], rank=rk, n_ranks=W, n_rows_total=n_tr,
                                 bufs=b))
            shares.append((st, stb, segs, S_loc, dict(ws_key=f"_share{rk}") if emulate else {}))
        nbytes = 0

        def gather(t):
            if not emulate:
                flat = t.view(W, -1)
                dist.all_gather_into_tensor(flat.view(-1), flat[r] if dev.type == "cuda" else flat[r].clone(), group=self.group)
            return (W - 1) * (t.numel() // W)
        if dev.type == "cuda" and not emulate and len(bufs) > 1:
            # several estimator groups: group by group, with the all-gathers on a communication stream — the planes
            # of group g travel while group g+1 runs its row-wise sublayers and while earlier groups attend
            if self._comm is None:
                self._comm = torch.cuda.Stream(device=dev)
            main = torch.cuda.current_stream(dev)
            st, stb, segs, S_loc, _ = shares[0]
            parts, off = [], 0
            for sg in segs:
                n = sg["B"] * S_loc * sg["T"]
                parts.append((st[off:off + n], stb[off:off + n]))
                off += n
            for l in range(L):
                landed = []
                for gi, (sg, (ps, pb)) in enumerate(zip(segs, parts)):
                    m.layers_run(ps, pb, [sg], S_loc, None, l, l + 1, phase=1, ws_key=f"_group{gi}")
                    ev = torch.cuda.Event()
                    ev.record(main)
                    with torch.cuda.stream(self._comm):
                        self._comm.wait_event(ev)
                        nbytes += gather(bufs[gi]["kg"]) + gather(bufs[gi]["vtg"])
                        done = torch.cuda.Event()
                        done.record(self._comm)
                    landed.append(done)
                for gi, (sg, (ps, pb)) in enumerate(zip(segs, parts)):
                    main.wait_event(landed[gi])
                    m.layers_run(ps, pb, [sg], S_loc, None, l, l + 1, phase=2, ws_key=f"_group{gi}")
        else:
            for l in range(L):
                for st, stb, segs, S_loc, kw in shares:
                    m.layers_run(st, stb, segs, S_loc, None, l, l + 1, phase=1, **kw)
                for b in bufs:
                    nbytes += gather(b["kg"]) + gather(b["vtg"])
                for st, stb, segs, S_loc, kw in shares:
                    m.layers_run(st, stb, segs, S_loc, None, l, l + 1, phase=2, **kw)
        for b in bufs:
            nbytes += gather(b["ctx"])
        self.exchange = {"collective": "all_gather_into_tensor", "calls_per_step": 2 * L * len(bufs) + len(bufs),
                         "bytes_received_per_rank": int(nbytes), "mode": "rows", "rows_per_rank": seg}
        # ---- this rank's test rows against every estimator's gathered context ------------------------------------
        n_te = staged["X_test"][0].shape[1]
        y_nan = torch.full((1, n_te), float("nan"), dtype=torch.float32, device=dev)
        st2, stb2, views2 = m._group_buffers([(len(g["idx"]), n_te, T) for g, T in zip(eng.groups, self.Ts)])
        tsegs = []
        for gi, (g, v) in enumerate(zip(eng.groups, views2)):
            ls, b = g["label_stats"], bufs[gi]
            m.embed(staged["X_test"][gi], stats[gi], tok_te, y_nan, ls[0], ls[1], m.positional_embeddings(self.Ts[gi] - 1),
                    B=len(g["idx"]), S=n_te, F=g["F"], x_bstride=n_te * g["F"], y_bstride=0, nan_flag=flag, out=v)
            tsegs.append(dict(B=len(g["idx"]), T=self.Ts[gi], kv=b["ctx"][0, 0], layer_stride=b["block"], seg_rows=seg,
                              rank_stride=L * b["block"], bufs=b, n_ranks=W))
        m.layers_run(st2, stb2, tsegs, n_te, n_tr, 0, L)
        out = [None] * len(self.members)
        for g, v in zip(eng.groups, views2):
            lg = m.decode(v[0])
            for k, i in enumerate(g["idx"]):
                out[i] = lg[k]
        return torch.stack(out)

    # ------------------------------------------------------------------------------------------------
    def proba_gathered(self, logits: torch.Tensor, class_perms, *, n_classes: int, softmax_temperature: float = 0.9):
        """The tail on the device (classifier.py:544-561) and the all-gather of every rank's probabilities:
        [Nte_local, n_classes] per rank -> [W * Nte_local, n_classes] on every rank (device tensor)."""
        from .engine import proba_device
        p = proba_device(logits, class_perms, n_classes=n_classes, softmax_temperature=softmax_temperature)
        return self._gather_rows(p)

    def regression_gathered(self, logits: torch.Tensor, src_bucket, src_share, cancel, borders, *,
                            softmax_temperature: float, average_before_softmax: bool, quantiles=None,
                            outputs=("mean",), n_rows: Optional[int] = None) -> dict:
        """The regressor's bar-distribution tail (``regressor.bar_tail_device``) on this rank's logits
        [n_est, rows_r, K] and the all-gather of the requested outputs; the logits never leave the rank.  "mean",
        "median", "mode" and "quantiles" travel as one [rows_r, 3 + n_q] block (one collective), "log_prob"
        ([rows_r, K]) as a second one, only when it is requested.  -> dict of device tensors over the rows of all ranks
        in test-row order, on every rank: [rows], [n_q, rows], [rows, K]; ``n_rows`` drops the padding rows of the last
        chunk (``test_rows``)."""
        from .regressor import bar_tail_device
        out = bar_tail_device(logits, src_bucket, src_share, cancel, borders, softmax_temperature=softmax_temperature,
                              average_before_softmax=average_before_softmax, quantiles=quantiles, outputs=outputs)
        keep = slice(None) if n_rows is None else slice(0, n_rows)
        scalars = [k for k in ("mean", "median", "mode") if k in out]
        cols = [out[k][:, None] for k in scalars] + ([out["quantiles"].t()] if "quantiles" in out else [])
        res = {}
        if cols:
            block = self._gather_rows(torch.cat(cols, dim=1))[keep]
            for j, k in enumerate(scalars):
                res[k] = block[:, j].contiguous()
            if "quantiles" in out:
                res["quantiles"] = block[:, len(scalars):].t().contiguous()
        if "log_prob" in out:
            res["log_prob"] = self._gather_rows(out["log_prob"])[keep]
        return res

    def logits(self, X_test_per_member, image_test, *, graph: bool = False) -> torch.Tensor:
        return self.logits_staged(self.stage(X_test_per_member, image_test))

    def check_nan(self):
        self.engine.check_nan()

    # ------------------------------------------------------------------------------------------------
    def _logits_broadcast(self, staged) -> torch.Tensor:
        """Ownership that does not fit the gather layout (see the module docstring): every context is built by
        its owner and broadcast afterwards, then merged per group."""
        from .model import TrainContext
        eng, m = self.engine, self.model
        dev = m.device
        eng.nan_flag.zero_()
        tok_tr = tok_te = None
        if staged["img_test"] is not None:
            tok_tr, tok_te = eng.train_image_tokens(), m.stem_image(staged["img_test"])
        mine: Dict[int, TrainContext] = {}
        for rk in (range(self.world) if self.emulate else [self.rank]):      # emulated: every owner in turn
            owned = [si for si, sub in enumerate(self.subs) if sub.owner == rk]
            specs = []
            for si in owned:
                sub = self.subs[si]
                g = eng.groups[sub.group]
                Xtr = None if g["X_train"] is None else g["X_train"][sub.pos].contiguous()
                Xte = staged["X_test"][sub.group]
                Xte = None if Xte is None else Xte[sub.pos].contiguous()
                ls = g["label_stats"]
                specs.append(dict(X_train=Xtr, y_train=g["y_train"][sub.pos].contiguous(),
                                  X_all=None if Xte is None else torch.cat([Xtr, Xte], dim=1), img_tok_train=tok_tr,
                                  label_stats=(ls[0][sub.pos].contiguous(), ls[1][sub.pos].contiguous())))
            if specs:
                mine.update(zip(owned, m.fit_contexts(specs, nan_flag=eng.nan_flag)))
        ctxs: Dict[int, TrainContext] = {}
        for si, sub in enumerate(self.subs):
            g = eng.groups[sub.group]
            B, n_tr = len(sub.pos), g["y_train"].shape[1]
            F = max(g["F"], 0)
            G_ = m._n_groups(F) if g["F"] >= 0 else 0
            T = G_ + (0 if tok_tr is None else tok_tr.shape[1]) + 1
            n_stats = m.lib.mmpfn_tab_stats_elems(m._g, G_) if G_ else 0
            shapes = [((m.lib.mmpfn_kv_bytes(m._g, B, n_tr, T, m.precision),), torch.uint8),
                      ((B,), torch.float32), ((B,), torch.int64)]
            if G_:
                shapes.append(((B, n_stats), torch.float32))
            src = None
            if si in mine:
                c = mine[si]
                src = [c.kv, c.y_mean, c.y_mask] + ([c.tab_stats] if G_ else [])
            got = src if self.emulate else broadcast_bundle(src, shapes, sub.owner, dev, self.group)
            ctxs[si] = TrainContext(B=B, n_train=n_tr, F=F, T=T, kv=got[0], tab_stats=got[3] if G_ else None,
                                    y_mean=got[1], y_mask=got[2], pos_emb=m.positional_embeddings(T - 1),
                                    precision=m.precision)
        merged = []
        for gi, g in enumerate(eng.groups):
            subs = [(si, sub) for si, sub in enumerate(self.subs) if sub.group == gi]
            if len(subs) == 1:
                ctx = ctxs[subs[0][0]]
            else:
                Bg = len(g["idx"])
                c0 = ctxs[subs[0][0]]
                y_mean = torch.empty(Bg, dtype=c0.y_mean.dtype, device=dev)
                y_mask = torch.empty(Bg, dtype=c0.y_mask.dtype, device=dev)
                stats = None if c0.tab_stats is None else torch.empty((Bg,) + tuple(c0.tab_stats.shape[1:]),
                                                                      dtype=c0.tab_stats.dtype, device=dev)
                for si, sub in subs:
                    c = ctxs[si]
                    y_mean[sub.pos] = c.y_mean
                    y_mask[sub.pos] = c.y_mask
                    if stats is not None:
                        stats[sub.pos] = c.tab_stats
                kv = m.merge_kv([(ctxs[si].kv, sub.pos) for si, sub in subs], Bg, c0.n_train, c0.T)
                ctx = TrainContext(B=Bg, n_train=c0.n_train, F=c0.F, T=c0.T, kv=kv, tab_stats=stats,
                                   y_mean=y_mean, y_mask=y_mask, pos_emb=c0.pos_emb, precision=m.precision)
            merged.append(ctx)
        lgs = m.predict_with_contexts(merged, staged["X_test"], img_tok_test=tok_te, nan_flag=eng.nan_flag)
        out = [None] * len(self.members)
        for g, lg in zip(eng.groups, lgs):
            for k, i in enumerate(g["idx"]):
                out[i] = lg[k]
        self.exchange = {"collective": None if self.emulate else "broadcast", "mode": "broadcast"}
        return torch.stack(out)


@dataclasses.dataclass
class _Sub:
    group: int            # index into engine.groups
    owner: int
    pos: List[int]        # positions inside the group's batch
    members: List[int]    # estimator ids
