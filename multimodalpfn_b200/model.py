"""``B200PerFeatureTransformer`` — host-side mirror of the reference's ``PerFeatureTransformer``
(``model/transformer.py:182-867``) for inference, running entirely on libmmpfn_b200.so.

It is callable exactly like the module the reference's engine holds
(``inference.py:343-348``)::

    logits = model(None, X_full, image_full, y_train, only_return_standard_out=True,
                   categorical_inds=cat_ix, single_eval_pos=len(y_train))      # [Nte, 1, n_out]

and additionally exposes what the reference cannot do: a batch axis over ensemble estimators
(``forward_batch``) and an explicit train-context / test-rows split (``fit_context`` /
``predict_with_context``), which is the reference's own KV-cache mode
(``multi_head_attention.py:328-336``, ``layer.py:346-372``) made first class.

There is no PyTorch compute on this path: torch only allocates device buffers, provides the CUDA
stream, and draws the positional-embedding noise with its generator (the reference's RNG
semantics, ``transformer.py:421-424, 925-933``, cannot be reproduced otherwise).
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from typing import Optional

import numpy as np
import torch

from . import _lib
from .synth import Geometry
from .weights import PackedWeights

__all__ = ["B200PerFeatureTransformer", "TrainContext", "entry_counts"]


def entry_counts(counts, capacity: int):
    """Per-entry row counts of a pass (int32), or None when every entry fills the capacity: such a pass passes no
    count arrays, i.e. runs the kernels of the equal-shape passes."""
    counts = np.asarray(counts, dtype=np.int32)
    return None if bool((counts == capacity).all()) else counts


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


@dataclasses.dataclass
class TrainContext:
    """Everything the test rows need from the train rows (SURVEY.md Appendix A, "KV-cache form")."""
    B: int
    n_train: int
    F: int
    T: int
    n_tok: int
    kv: torch.Tensor                      # per-layer head-0 K/V of the item attention (layout: include/mmpfn_b200.h)
    tab_stats: Optional[torch.Tensor]     # [B, stats_elems]
    y_mean: torch.Tensor                  # [B]
    y_mask: torch.Tensor                  # [B] uint64 as int64
    pos_emb: torch.Tensor                 # [T-1, E]
    precision: int
    train_out: Optional[torch.Tensor] = None   # [B, Ntr, E]: y-token of the train rows after the last layer (on request)


class B200PerFeatureTransformer:
    def __init__(self, state_dict, geom: Geometry, *, device=None, precision: str = "bf16", seed: int = 0,
                 outlier_std: Optional[float] = 12.0, pos_emb_device: str = "cpu"):
        self.lib = _lib.load()
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else None
        if device is None or torch.device(device).type != "cuda":
            raise RuntimeError("B200PerFeatureTransformer needs a CUDA device (sm_100); there is no CPU path")
        self.device = torch.device(device)
        if not self.lib.mmpfn_device_supported(self.device.index or 0):
            raise RuntimeError(f"{torch.cuda.get_device_name(self.device)} is not an sm_100 device")
        self.geom = geom
        self.precision_name = precision
        self.precision = {"fp32": _lib.F32, "bf16": _lib.BF16}[precision]
        self.seed = seed
        # reference: classifier.py:396-406 switches the outlier step on with sigma 12; a model used
        # without that call keeps InferenceConfig.remove_outliers = False (model/config.py:43).
        self.outlier_std = outlier_std
        self.pos_emb_device = pos_emb_device
        with torch.cuda.device(self.device):
            self.w = PackedWeights(state_dict, geom, self.device, with_bf16=True, stem_bf16=(precision == "bf16"))
        self._g = C.byref(self.w.c_geom)
        self._w = C.byref(self.w.c_weights)
        self._w_test = C.byref(self.w.c_weights_test)      # second query set of two_sets_of_queries checkpoints
        self._cached_ctx = None                            # the reference's model-level train-set cache
        self._pos_cache = {}
        self._buf = {}
        # bumped whenever a shared scratch buffer is replaced (and its old storage freed): CUDA graphs captured
        # before hold raw pointers into the old storage and must not be replayed (engine.logits_graphed checks)
        self.scratch_epoch = 0
        # attributes the reference's engine / loader touch (SURVEY.md section 8(b))
        self.ninp = geom.emsize
        self.features_per_group = geom.features_per_group
        self.cache_trainset_representation = False
        # model/memory.py:185-189 counts len(model.transformer_encoder.layers)
        self.transformer_encoder = type("LayerStackShim", (), {"layers": [None] * geom.nlayers})()

    # ------------------------------------------------------------------ nn.Module duck-typing
    def to(self, *a, **k):
        return self

    def type(self, *a, **k):
        return self

    def cpu(self):
        return self

    def eval(self):
        return self

    def parameters(self):
        return iter(self.w._t.values())

    def reset_save_peak_mem_factor(self, factor=None):
        return None

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _scratch(self, name: str, nbytes: int) -> torch.Tensor:
        t = self._buf.get(name)
        if t is None or t.numel() < nbytes:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError(f"scratch buffer {name!r} would grow during CUDA-graph capture: warm up first")
            t = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=self.device)
            if name in self._buf:
                self.scratch_epoch += 1
            self._buf[name] = t
        return t

    def n_image_tokens(self, n_tok: int) -> int:
        return int(self.lib.mmpfn_image_tokens(self._g, n_tok)) if n_tok > 0 else 0

    def positional_embeddings(self, n_feature_tokens: int) -> torch.Tensor:
        """transformer.py:421-424, :925-933 — a fresh generator per forward (seeded iff seed != 0)
        draws randn((T-1, E/4)) in fp32; Linear(E/4 -> E) applied on the host (48x192, negligible)."""
        key = n_feature_tokens
        if key not in self._pos_cache:
            gen = torch.Generator(device=self.pos_emb_device)
            if self.seed:
                gen.manual_seed(self.seed)
            z = torch.randn((n_feature_tokens, self.geom.emsize // 4), generator=gen, device=self.pos_emb_device,
                            dtype=torch.float32).cpu()
            emb = z @ self.w.pe_w.T + self.w.pe_b
            self._pos_cache[key] = emb.to(self.device).contiguous()
        return self._pos_cache[key]

    # ------------------------------------------------------------------ stem
    def stem_image(self, img: torch.Tensor) -> torch.Tensor:
        """[S, n_tok, img_dim] fp32 -> [S, H_img, E] fp32 (transformer.py:755-761)."""
        img = img.to(self.device, torch.float32).contiguous()
        S, n_tok, I = img.shape
        if I != self.geom.img_dim:
            raise ValueError(f"embedding width {I} != {self.geom.img_dim}")
        H_img = self.n_image_tokens(n_tok)
        out = torch.empty((S, H_img, self.geom.emsize), dtype=torch.float32, device=self.device)
        nbytes = self.lib.mmpfn_stem_image_ws_bytes(self._g, S, n_tok)
        ws = self._scratch("img", nbytes)
        _lib.check(self.lib.mmpfn_stem_image(self._g, self._w, img.data_ptr(), S, n_tok, out.data_ptr(),
                                             ws.data_ptr(), nbytes, self._stream()), "mmpfn_stem_image")
        return out

    def _n_groups(self, F: int) -> int:
        fpg = self.geom.features_per_group
        return (F + fpg - 1) // fpg

    def stem_tab_fit(self, X: torch.Tensor, n_train: int) -> torch.Tensor:
        """X [B, S, F] fp32 -> statistics [B, stats_elems] (encoders.py:453-461, :508-515, :608-619, :702-735)."""
        B, S, F = X.shape
        G = self._n_groups(F)
        n = self.lib.mmpfn_tab_stats_elems(self._g, G)
        stats = torch.empty((B, n), dtype=torch.float32, device=self.device)
        sigma = float(self.outlier_std) if self.outlier_std is not None else float("inf")
        _lib.check(self.lib.mmpfn_stem_tab_fit(self._g, X.data_ptr(), B, S, F, n_train, sigma, stats.data_ptr(),
                                               self._stream()), "mmpfn_stem_tab_fit")
        return stats

    REGRESSION_MASK = -(1 << 63)        # bit 63 of the presence mask: "embed the target value itself"

    def label_stats(self, y_train: torch.Tensor):
        """y_train [B, Ntr] -> (mean [B], presence bitmask [B]).
        Classification (class ids as floats): encoders.py:461 (nanmean for the test-row fill) and :954-958 (unique
        train labels, for the ordinal rank).  Regression checkpoints: the mean only — no rank step exists
        (model/loading.py:387-388) and bit 63 of the mask tells the stem kernel so."""
        if getattr(self.w, "regression", False):
            mask = torch.full((y_train.shape[0],), self.REGRESSION_MASK, dtype=torch.int64, device=y_train.device)
            return y_train.to(torch.float32).mean(dim=1).contiguous(), mask
        yl = y_train.to(torch.int64)
        if not torch.equal(yl.to(y_train.dtype), y_train) or int(yl.min()) < 0 or int(yl.max()) > 62:
            raise ValueError("labels must be integer class ids in [0, 62]")
        mask = torch.zeros(y_train.shape[0], dtype=torch.int64, device=y_train.device)
        one = torch.ones_like(yl)
        bits = torch.bitwise_left_shift(one, yl)
        for b in range(y_train.shape[0]):
            mask[b] = torch.unique(bits[b]).sum()
        return y_train.to(torch.float32).mean(dim=1).contiguous(), mask

    def embed(self, X, stats, img_tok, y, y_mean, y_mask, pos_emb, *, B, S, F, x_bstride, y_bstride, nan_flag, out=None):
        """Token assembly -> (state_f32 [B,S,T,E], state_bf16 or None)."""
        G = self._n_groups(F) if X is not None else 0
        # img_tok [S, H, E]: shared by the B entries; [B, S, H, E]: one set per entry (packed tasks)
        H_img = 0 if img_tok is None else img_tok.shape[-2]
        img_bstride = 0
        if img_tok is not None and img_tok.dim() == 4:
            if img_tok.shape[0] != B or img_tok.shape[1] != S:
                raise ValueError("per-entry image tokens must be [B, S, H, E]")
            img_tok = img_tok.contiguous()
            img_bstride = img_tok.shape[1] * img_tok.shape[2] * img_tok.shape[3]
        T = G + H_img + 1
        E = self.geom.emsize
        if out is not None:          # views into a buffer shared by several estimator groups (layers_*_multi)
            state, state_b = out
            assert tuple(state.shape) == (B, S, T, E) and state.is_contiguous()
        else:
            state = torch.empty((B, S, T, E), dtype=torch.float32, device=self.device)
            state_b = torch.empty((B, S, T, E), dtype=torch.bfloat16, device=self.device) \
                if self.precision == _lib.BF16 else None
        _lib.check(self.lib.mmpfn_stem_tokens(
            self._g, self._w, _ptr(X), _ptr(stats), _ptr(img_tok), y.data_ptr(), y_mean.data_ptr(),
            y_mask.data_ptr(), pos_emb.data_ptr(), B, S, F if X is not None else 0, H_img, x_bstride, y_bstride,
            img_bstride, state.data_ptr(), _ptr(state_b), nan_flag.data_ptr(), self._stream()), "mmpfn_stem_tokens")
        return state, state_b

    # ------------------------------------------------------------------ layers / decoder
    def layers_train(self, state, state_b, kv: Optional[torch.Tensor]):
        B, S, T, _ = state.shape
        nbytes = self.lib.mmpfn_layers_ws_bytes(self._g, B, S, T, self.precision)
        ws = self._scratch("layers", nbytes)
        _lib.check(self.lib.mmpfn_layers_train(self._g, self._w, state.data_ptr(), _ptr(state_b), B, S, T,
                                               self.precision, _ptr(kv), ws.data_ptr(), nbytes, self._stream()),
                   "mmpfn_layers_train")

    def layers_test(self, state, state_b, kv: torch.Tensor, n_train: int):
        B, S, T, _ = state.shape
        nbytes = self.lib.mmpfn_layers_ws_bytes(self._g, B, S, T, self.precision)
        ws = self._scratch("layers", nbytes)
        _lib.check(self.lib.mmpfn_layers_test(self._g, self._w_test, state.data_ptr(), _ptr(state_b), B, S, T, n_train,
                                              self.precision, kv.data_ptr(), ws.data_ptr(), nbytes, self._stream()),
                   "mmpfn_layers_test")

    def _layers_multi(self, state, state_b, segs, S: int, kvs, n_train: Optional[int]):
        """``state`` / ``state_b``: flat [M_total, E] buffers holding the segments' [B_i, S, T_i, E] states back
        to back; ``segs``: [(B_i, T_i)]; ``kvs``: one context tensor per segment."""
        n = len(segs)
        arr = (_lib.Segment * n)(*[_lib.Segment(int(b), int(t)) for b, t in segs])
        kvp = (C.c_void_p * n)(*[kv.data_ptr() for kv in kvs])
        nbytes = self.lib.mmpfn_layers_multi_ws_bytes(self._g, arr, n, S)
        ws = self._scratch("layers", nbytes)
        if n_train is None:
            _lib.check(self.lib.mmpfn_layers_train_multi(self._g, self._w, state.data_ptr(), state_b.data_ptr(), arr, n, S,
                                                         kvp, ws.data_ptr(), nbytes, self._stream()),
                       "mmpfn_layers_train_multi")
        else:
            _lib.check(self.lib.mmpfn_layers_test_multi(self._g, self._w_test, state.data_ptr(), state_b.data_ptr(), arr, n, S,
                                                        n_train, kvp, ws.data_ptr(), nbytes, self._stream()),
                       "mmpfn_layers_test_multi")

    def layers_run(self, state, state_b, segs, S: int, n_train: Optional[int], layer_begin: int, layer_end: int,
                   phase: int = 0, ws_key: str = ""):
        """Layers ``[layer_begin, layer_end)`` over segment states held back to back in ``state`` / ``state_b``
        (``_group_buffers``), with the K/V context of every segment addressed explicitly (``mmpfn_layers_run``).
        ``segs``: dicts ``B, T, kv`` (uint8 tensor view starting at the segment's block of layer 0),
        ``layer_stride`` / ``rank_stride`` (bytes) and ``slots``.  ``n_train=None``: train pass (writes the K/V),
        else test pass against ``n_train`` context rows.  ``phase`` 1 leaves the queries in the workspace for
        ``phase`` 2: callers that interleave several states between the two name a workspace each (``ws_key``)."""
        n = len(segs)
        def seg(s):
            k = _lib.KvSegment()
            k.B, k.T, k.kv = int(s["B"]), int(s["T"]), s["kv"].data_ptr()
            k.layer_stride, k.slots, k.rank_stride = int(s.get("layer_stride", 0)), int(s.get("slots", 0)), int(s.get("rank_stride", 0))
            k.seg_rows = int(s.get("seg_rows", 0))
            if s.get("kg") is not None:        # row-sharded context build (dist.py "rows" mode; include/mmpfn_b200.h)
                k.kg, k.vtg = s["kg"].data_ptr(), s["vtg"].data_ptr()
                k.gather_stride, k.rank, k.n_ranks = int(s["gather_stride"]), int(s["rank"]), int(s["n_ranks"])
                k.n_rows_total = int(s["n_rows_total"])
            return k
        arr = (_lib.KvSegment * n)(*[seg(s) for s in segs])
        plain = (_lib.Segment * n)(*[_lib.Segment(int(s["B"]), int(s["T"])) for s in segs])
        S_alloc = max([S] + [int(s.get("seg_rows", 0)) for s in segs]) if n_train is None else S
        nbytes = self.lib.mmpfn_layers_multi_ws_bytes(self._g, plain, n, S_alloc)
        ws = self._scratch("layers" + ws_key, nbytes)
        _lib.check(self.lib.mmpfn_layers_run(self._g, self._w if n_train is None else self._w_test, state.data_ptr(),
                                             state_b.data_ptr(), arr, n, S,
                                             0 if n_train is None else int(n_train), 1 if n_train is None else 0,
                                             int(layer_begin), int(layer_end), int(phase), ws.data_ptr(), nbytes,
                                             self._stream()),
                   "mmpfn_layers_run")

    def alloc_kv(self, B: int, n_train: int, T: int) -> torch.Tensor:
        nbytes = self.lib.mmpfn_kv_bytes(self._g, B, n_train, T, self.precision)
        # not zero-filled: the bf16 layout pads the row axis to a multiple of 64, but every reader goes through a
        # TMA tensor map whose extent is the true row count (pad rows are never fetched: out-of-bounds zero fill)
        return torch.empty(nbytes, dtype=torch.uint8, device=self.device)

    def merge_kv(self, parts, B: int, n_train: int, T: int) -> torch.Tensor:
        """Assemble the K/V context of a batch of B estimators from contexts built for subsets of it
        (``parts``: [(kv, positions within the batch)]) — the layer axis is outermost in the context
        layout, so every subset lands as L strided slabs (one device copy per subset)."""
        L = self.geom.nlayers
        out = torch.empty(self.lib.mmpfn_kv_bytes(self._g, B, n_train, T, self.precision), dtype=torch.uint8,
                          device=self.device)
        if self.precision == _lib.BF16:       # per layer: K0 [B][T][Sp][32] then V0^T [B][T][32][Sp]
            per_b = out.numel() // (L * 2 * B)
            dst = out.view(L, 2, B, per_b)
            for kv, pos in parts:
                dst[:, :, pos] = kv.view(L, 2, len(pos), per_b)
        else:                                  # per layer: [B][T][n][2][32] fp32
            per_b = out.numel() // (L * B)
            dst = out.view(L, B, per_b)
            for kv, pos in parts:
                dst[:, pos] = kv.view(L, len(pos), per_b)
        return out

    def decode(self, state: torch.Tensor) -> torch.Tensor:
        """[B,S,T,E] -> logits [B,S,n_out] (transformer.py:850-853)."""
        B, S, T, _ = state.shape
        hid = self._scratch("dec", B * S * self.geom.nhid * 4)
        logits = torch.empty((B, S, self.geom.n_out), dtype=torch.float32, device=self.device)
        _lib.check(self.lib.mmpfn_decode(self._g, self._w, state.data_ptr(), B, S, T, hid.data_ptr(),
                                         logits.data_ptr(), self._stream()), "mmpfn_decode")
        return logits

    # ------------------------------------------------------------------ whole forwards
    def _prep(self, X, img):
        if X is not None:
            X = X.to(self.device, torch.float32)
            if X.dim() == 2:
                X = X[None]
            X = X.contiguous()
        if img is not None:
            img = img.to(self.device, torch.float32)
            if img.dim() == 2:
                img = img[:, None]
            img = img.contiguous()
        return X, img

    def _check_nan(self, flag: torch.Tensor):
        if int(flag.item()) != 0:
            # transformer.py:727-731, :790-796
            raise ValueError("There should be no NaNs in the encoded x and y. Check that you do not feed NaNs "
                             "or use a NaN-handling encoder (an all-NaN column or inf in a train column).")

    def fit_context(self, X_train, img_train, y_train, *, X_all=None, img_tok_train=None, check=True,
                    label_stats=None, nan_flag=None, keep_train_out=False) -> TrainContext:
        """Run the train rows through the stem and the 12 layers once; keep the K/V context.

        X_train [B, Ntr, F] (or [Ntr, F]) / img_train [Ntr, n_tok, img_dim] / y_train [B, Ntr].
        ``X_all`` ([B, S, F], train rows first): when given, the "constant column" tests of the stem
        see all S rows, which is what the reference's joint forward does (encoders.py:515, :615).
        """
        with torch.cuda.device(self.device):
            X_train, img_train = self._prep(X_train, img_train)
            y_train = y_train.to(self.device, torch.float32)
            if y_train.dim() == 1:
                y_train = y_train[None]
            y_train = y_train.contiguous()
            B, n_train = y_train.shape
            F = 0 if X_train is None else X_train.shape[2]
            n_tok = 0 if img_train is None else img_train.shape[1]
            if X_train is None and img_train is None and img_tok_train is None:
                raise ValueError("need tabular features, image embeddings, or both")
            stats = None
            if X_train is not None:
                if X_all is not None:
                    X_all, _ = self._prep(X_all, None)
                    stats = self.stem_tab_fit(X_all, n_train)
                else:
                    stats = self.stem_tab_fit(X_train, n_train)
            if img_tok_train is None and img_train is not None:
                img_tok_train = self.stem_image(img_train)
            # label statistics involve a host sync: callers that replay a CUDA graph pass them in
            y_mean, y_mask = label_stats if label_stats is not None else self.label_stats(y_train)
            G = self._n_groups(F) if X_train is not None else 0
            H_img = 0 if img_tok_train is None else img_tok_train.shape[-2]
            T = G + H_img + 1
            pos = self.positional_embeddings(T - 1)
            flag = nan_flag if nan_flag is not None else torch.zeros(1, dtype=torch.int32, device=self.device)
            state, state_b = self.embed(X_train, stats, img_tok_train, y_train, y_mean, y_mask, pos, B=B, S=n_train,
                                        F=F, x_bstride=n_train * F, y_bstride=n_train, nan_flag=flag)
            kv = self.alloc_kv(B, n_train, T)
            self.layers_train(state, state_b, kv)
            if check:
                self._check_nan(flag)
            return TrainContext(B=B, n_train=n_train, F=F, T=T, n_tok=n_tok, kv=kv, tab_stats=stats, y_mean=y_mean,
                                y_mask=y_mask, pos_emb=pos, precision=self.precision,
                                train_out=state[:, :, T - 1].clone() if keep_train_out else None)

    def predict_with_context(self, ctx: TrainContext, X_test, img_test, *, img_tok_test=None, check=True,
                             nan_flag=None, return_embeddings=False):
        """Test rows only -> logits [B, Nte, n_out] (with ``return_embeddings``: also the y-token of the test
        rows after the last layer, [B, Nte, E] — the reference's ``test_embeddings``, transformer.py:862-866)."""
        with torch.cuda.device(self.device):
            X_test, img_test = self._prep(X_test, img_test)
            if img_tok_test is None and img_test is not None:
                img_tok_test = self.stem_image(img_test)
            n_test = X_test.shape[1] if X_test is not None else img_tok_test.shape[-3]
            if X_test is not None and (X_test.shape[0] != ctx.B or X_test.shape[2] != ctx.F):
                raise ValueError(f"test table {tuple(X_test.shape)} does not match the context (B {ctx.B}, F {ctx.F})")
            y_nan = torch.full((1, n_test), float("nan"), dtype=torch.float32, device=self.device)
            flag = nan_flag if nan_flag is not None else torch.zeros(1, dtype=torch.int32, device=self.device)
            state, state_b = self.embed(X_test, ctx.tab_stats, img_tok_test, y_nan, ctx.y_mean, ctx.y_mask, ctx.pos_emb,
                                        B=ctx.B, S=n_test, F=ctx.F, x_bstride=n_test * ctx.F, y_bstride=0,
                                        nan_flag=flag)
            if state.shape[2] != ctx.T:
                raise ValueError("test rows produce a different number of tokens than the context")
            self.layers_test(state, state_b, ctx.kv, ctx.n_train)
            logits = self.decode(state)
            if check:
                self._check_nan(flag)
            if return_embeddings:
                return logits, state[:, :, ctx.T - 1].clone()
            return logits

    # ---- several estimator groups at once (bf16): one launch per flat sublayer for all of them ----------
    def _group_buffers(self, shapes, with_bf16: bool = True):
        """One fp32 + one bf16 buffer for states of the given [(B, S, T)] shapes, and the per-group views."""
        E = self.geom.emsize
        total = sum(b * s * t for b, s, t in shapes)
        st = torch.empty((total, E), dtype=torch.float32, device=self.device)
        stb = torch.empty((total, E), dtype=torch.bfloat16, device=self.device) if with_bf16 else None
        views, off = [], 0
        for b, s, t in shapes:
            n = b * s * t
            views.append((st[off:off + n].view(b, s, t, E), None if stb is None else stb[off:off + n].view(b, s, t, E)))
            off += n
        return st, stb, views

    # ---- entries of different sizes in one pass (tasks.py) ------------------------------------------------
    def entry_tokens(self, F: Optional[int], n_tok: int) -> int:
        """Token count T of an entry with ``F`` preprocessed features (None: no table) and ``n_tok`` embeddings."""
        return (0 if F is None else self._n_groups(F)) + self.n_image_tokens(n_tok) + 1

    def forward_ragged(self, entries, *, final_states: Optional[list] = None):
        """One train pass and one test pass over batch entries of any sizes -> [logits [n_test, n_out]] in entry order.

        An entry is one (task, estimator) pair: a dict with ``X`` (float32 [n_train + n_test, F], train rows first, or
        None), ``y`` (class ids [n_train], or float targets for a regression checkpoint), ``n_train``, ``n_test`` and
        ``tok`` / ``tok_row`` / ``n_tok`` (image tokens [rows, H, E] from ``stem_image`` of ``n_tok`` embeddings per
        row and the row of the entry's first train row in it, or ``tok`` None), and optionally ``y_mean`` (a float32
        device tensor of one element: the label mean to use, as ``fit_context(label_stats=...)`` takes it).  Without
        it the mean is that of the entry's own labels; for float targets torch's mean of a [k, n] block can change in
        the last bit with k, so callers that must match a forward over a group of entries pass the group's means.
        The pass
        has the row capacity of its largest entry; the other entries' rows up to it are pad rows, kept exactly zero
        (include/mmpfn_b200.h, "ragged" passes), so every entry's logits are bit-identical to ``fit_context`` +
        ``predict_with_context`` over that entry alone (the stem statistics see its train and test rows).  Entries of
        equal T form one segment (at most ``MMPFN_MAX_SEGMENTS``); a pass whose entries all have the capacity passes
        no count arrays, i.e. runs the kernels of the equal-shape passes.  ``final_states`` (a list) receives, for the
        train pass and then the test pass, ``(state [B_i, S, T_i, E], [entry index])`` per segment after the layers."""
        regression = getattr(self.w, "regression", False)
        dev = self.device
        T_of = [self.entry_tokens(None if e["X"] is None else e["X"].shape[1],
                                  0 if e["tok"] is None else e["n_tok"]) for e in entries]
        seg_T = list(dict.fromkeys(sorted(T_of)))
        if len(seg_T) > _lib.MAX_SEGMENTS:
            raise ValueError(f"{len(seg_T)} token counts in one pass (at most {_lib.MAX_SEGMENTS})")
        # pass order: segments by T; inside a segment, blocks of one (feature count, embedding) kind
        def block_key(j):
            e = entries[j]
            return (-1 if e["X"] is None else e["X"].shape[1], -1 if e["tok"] is None else id(e["tok"]))
        order = sorted(range(len(entries)), key=lambda j: (T_of[j], block_key(j)))
        segs = [(T, [j for j in order if T_of[j] == T]) for T in seg_T]
        n_tr = np.array([entries[j]["n_train"] for j in order], dtype=np.int32)
        n_te = np.array([entries[j]["n_test"] for j in order], dtype=np.int32)
        S_tr, S_te = int(n_tr.max()), int(n_te.max())
        c_tr, c_te = entry_counts(n_tr, S_tr), entry_counts(n_te, S_te)
        c_all = entry_counts(n_tr + n_te, S_tr + S_te)
        dev_i32 = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)
        d_tr, d_te = dev_i32(c_tr), dev_i32(c_te)
        pos_in_pass = {j: k for k, j in enumerate(order)}
        with torch.cuda.device(dev):
            # stem statistics: one call per feature count over the entries' train + test rows
            Sa = S_tr + S_te
            stats_of = {}
            X_all = {}
            by_F = {}
            for j in order:
                if entries[j]["X"] is not None:
                    by_F.setdefault(entries[j]["X"].shape[1], []).append(j)
            for F, js in by_F.items():
                xa = np.zeros((len(js), Sa, F), dtype=np.float32)
                for k, j in enumerate(js):
                    xa[k, :len(entries[j]["X"])] = entries[j]["X"]
                xa = torch.from_numpy(xa).to(dev)
                if c_all is None:
                    stats = self.stem_tab_fit(xa, S_tr)
                else:
                    idx = np.array([pos_in_pass[j] for j in js])
                    stats = self._stem_tab_fit_ragged(xa, dev_i32(n_tr[idx] + n_te[idx]), dev_i32(n_tr[idx]))
                for k, j in enumerate(js):
                    stats_of[j] = (stats, k)
                    X_all[j] = (xa, k)
            # label statistics per entry on its own labels: the mean of class ids over a [k, n] block is exact, so
            # entries of equal n share a block; float targets are averaged one entry per block (the presence mask
            # is exact integer work)
            y_mean = torch.empty(len(order), dtype=torch.float32, device=dev)
            by_n, given = {}, []
            for k, j in enumerate(order):
                if entries[j].get("y_mean") is not None:
                    given.append(k)
                else:
                    by_n.setdefault((entries[j]["n_train"], k if regression else -1), []).append(k)
            if given:
                y_mean[torch.tensor(given, device=dev)] = torch.cat([entries[order[k]]["y_mean"].reshape(1)
                                                                     for k in given])
            ys = [np.asarray(entries[j]["y"]) for j in order]
            for ks in by_n.values():
                y_blk = torch.from_numpy(np.stack([ys[k] for k in ks]).astype(np.float32)).to(dev)
                y_mean[torch.tensor(ks, device=dev)] = y_blk.mean(dim=1)
            if regression:
                y_mask = torch.full((len(order),), self.REGRESSION_MASK, dtype=torch.int64, device=dev)
            else:
                masks = []
                for y in ys:
                    yl = y.astype(np.int64)
                    if not np.array_equal(yl, y) or yl.min() < 0 or yl.max() > 62:
                        raise ValueError("labels must be integer class ids in [0, 62]")
                    masks.append(int(np.bitwise_or.reduce(np.left_shift(np.int64(1), np.unique(yl)))))
                y_mask = torch.tensor(masks, dtype=torch.int64, device=dev)
            y_tr = np.zeros((len(order), S_tr), dtype=np.float32)
            for k, y in enumerate(ys):
                y_tr[k, :len(y)] = y
            y_tr = torch.from_numpy(y_tr).to(dev)
            y_nan = torch.full((S_te,), float("nan"), dtype=torch.float32, device=dev)
            flag = torch.zeros(1, dtype=torch.int32, device=dev)
            bf16 = self.precision == _lib.BF16
            shapes = [(len(js), T) for T, js in segs]
            kvs = [self.alloc_kv(b, S_tr, T) for b, T in shapes]
            logits = [None] * len(entries)
            for train in (True, False):
                S = S_tr if train else S_te
                st, stb, views = self._group_buffers([(b, S, T) for b, T in shapes], with_bf16=bf16)
                k0 = 0
                for (T, js), (v, vb) in zip(segs, views):
                    pos = self.positional_embeddings(T - 1)
                    i0 = 0
                    while i0 < len(js):          # blocks: entries of one feature count and one embedding kind
                        i1 = i0 + 1
                        while i1 < len(js) and block_key(js[i1]) == block_key(js[i0]):
                            i1 += 1
                        blk = js[i0:i1]
                        self._embed_block([entries[j] for j in blk], blk, stats_of, X_all, train, S_tr, S_te,
                                          y_tr[k0 + i0:k0 + i1], y_nan, y_mean[k0 + i0:k0 + i1],
                                          y_mask[k0 + i0:k0 + i1], pos, v[i0:i1], None if vb is None else vb[i0:i1],
                                          (d_tr if train else d_te), k0 + i0, flag)
                        i0 = i1
                    k0 += len(js)
                seg_arr = (_lib.Segment * len(shapes))(*[_lib.Segment(b, T) for b, T in shapes])
                kvp = (C.c_void_p * len(kvs))(*[kv.data_ptr() for kv in kvs])
                nbytes = self.lib.mmpfn_layers_ragged_ws_bytes(self._g, seg_arr, len(shapes), S, self.precision)
                ws = self._scratch("layers", nbytes)
                if train:
                    _lib.check(self.lib.mmpfn_layers_train_ragged(
                        self._g, self._w, st.data_ptr(), _ptr(stb), seg_arr, len(shapes), S, _ptr(d_tr),
                        self.precision, kvp, ws.data_ptr(), nbytes, self._stream()), "mmpfn_layers_train_ragged")
                    if final_states is not None:
                        final_states.extend(zip([v for v, _ in views], [js for _, js in segs]))
                else:
                    _lib.check(self.lib.mmpfn_layers_test_ragged(
                        self._g, self._w_test, st.data_ptr(), _ptr(stb), seg_arr, len(shapes), S, S_tr, _ptr(d_te),
                        _ptr(d_tr), self.precision, kvp, ws.data_ptr(), nbytes, self._stream()),
                        "mmpfn_layers_test_ragged")
                    for (T, js), (v, _) in zip(segs, views):
                        lg = self.decode(v)
                        if final_states is not None:
                            final_states.append((v, js))
                        for k, j in enumerate(js):
                            logits[j] = lg[k, :entries[j]["n_test"]]
                del st, stb, views
            self._check_nan(flag)
            return logits

    def _stem_tab_fit_ragged(self, X, n_rows, n_train):
        B, S, F = X.shape
        n = self.lib.mmpfn_tab_stats_elems(self._g, self._n_groups(F))
        stats = torch.empty((B, n), dtype=torch.float32, device=self.device)
        sigma = float(self.outlier_std) if self.outlier_std is not None else float("inf")
        _lib.check(self.lib.mmpfn_stem_tab_fit_ragged(self._g, X.data_ptr(), B, S, F, n_rows.data_ptr(),
                                                      n_train.data_ptr(), sigma, stats.data_ptr(), self._stream()),
                   "mmpfn_stem_tab_fit_ragged")
        return stats

    def _embed_block(self, ents, js, stats_of, X_all, train, S_tr, S_te, y_tr, y_nan, y_mean, y_mask, pos, out,
                     out_b, counts, k0, flag):
        """Token assembly of one block (same feature count and embeddings) of a ragged pass into its views."""
        dev, B = self.device, len(ents)
        S = S_tr if train else S_te
        x = stats = None
        F = 0
        if ents[0]["X"] is not None:
            xa, _ = X_all[js[0]]
            F = xa.shape[2]
            rows = torch.tensor([X_all[j][1] for j in js], device=dev)
            stats = stats_of[js[0]][0][rows].contiguous()
            if train:
                x = xa[rows].contiguous()                     # train rows first: rows [0, n_train) of each block
                x_bstride = x.shape[1] * F
            else:
                xt = np.zeros((B, S_te, F), dtype=np.float32)
                for k, e in enumerate(ents):
                    xt[k, :e["n_test"]] = e["X"][e["n_train"]:]
                x = torch.from_numpy(xt).to(dev)
                x_bstride = S_te * F
        else:
            x_bstride = 0
        tok = ents[0]["tok"]
        H = 0 if tok is None else tok.shape[1]
        off = None
        if tok is not None:
            off = torch.tensor([(e["tok_row"] + (0 if train else e["n_train"])) * H * tok.shape[2] for e in ents],
                               dtype=torch.int64, device=dev)
        cnt = None if counts is None else counts[k0:k0 + B]
        _lib.check(self.lib.mmpfn_stem_tokens_ragged(
            self._g, self._w, _ptr(x), _ptr(stats), _ptr(tok), y_tr.data_ptr() if train else y_nan.data_ptr(),
            y_mean.data_ptr(), y_mask.data_ptr(), pos.data_ptr(), B, S, F, H, x_bstride, S_tr if train else 0,
            _ptr(off), _ptr(cnt), out.data_ptr(), _ptr(out_b), flag.data_ptr(), self._stream()),
            "mmpfn_stem_tokens_ragged")

    def fit_contexts(self, specs, *, nan_flag=None):
        """``fit_context`` for several estimator groups that share the train rows (same n_train) — specs:
        dicts with ``X_train [B, Ntr, F]``, ``y_train [B, Ntr]``, optional ``X_all``, ``img_tok_train``,
        ``label_stats``.  Same results as one ``fit_context`` per group; the layers run as
        ``mmpfn_layers_train_multi``."""
        assert self.precision == _lib.BF16
        with torch.cuda.device(self.device):
            flag = nan_flag if nan_flag is not None else torch.zeros(1, dtype=torch.int32, device=self.device)
            prep = []
            for sp in specs:
                X_train, _ = self._prep(sp["X_train"], None)
                y_train = sp["y_train"].to(self.device, torch.float32).contiguous()
                B, n_train = y_train.shape
                F = X_train.shape[2]
                X_all = sp.get("X_all")
                if X_all is not None:
                    X_all, _ = self._prep(X_all, None)
                stats = self.stem_tab_fit(X_all if X_all is not None else X_train, n_train)
                tok = sp.get("img_tok_train")
                y_mean, y_mask = sp["label_stats"] if sp.get("label_stats") is not None else self.label_stats(y_train)
                T = self._n_groups(F) + (0 if tok is None else tok.shape[-2]) + 1
                prep.append(dict(X=X_train, y=y_train, B=B, n_train=n_train, F=F, stats=stats, tok=tok, y_mean=y_mean,
                                 y_mask=y_mask, T=T, pos=self.positional_embeddings(T - 1)))
            n_train = prep[0]["n_train"]
            assert all(p["n_train"] == n_train for p in prep)
            st, stb, views = self._group_buffers([(p["B"], n_train, p["T"]) for p in prep])
            for p, v in zip(prep, views):
                self.embed(p["X"], p["stats"], p["tok"], p["y"], p["y_mean"], p["y_mask"], p["pos"], B=p["B"], S=n_train,
                           F=p["F"], x_bstride=n_train * p["F"], y_bstride=n_train, nan_flag=flag, out=v)
            kvs = [self.alloc_kv(p["B"], n_train, p["T"]) for p in prep]
            self._layers_multi(st, stb, [(p["B"], p["T"]) for p in prep], n_train, kvs, None)
            return [TrainContext(B=p["B"], n_train=n_train, F=p["F"], T=p["T"], n_tok=0, kv=kv, tab_stats=p["stats"],
                                 y_mean=p["y_mean"], y_mask=p["y_mask"], pos_emb=p["pos"], precision=self.precision)
                    for p, kv in zip(prep, kvs)]

    def predict_with_contexts(self, ctxs, X_tests, *, img_tok_test=None, nan_flag=None):
        """``predict_with_context`` for several groups at once (same test rows) -> [logits [B_i, Nte, n_out]]."""
        assert self.precision == _lib.BF16
        with torch.cuda.device(self.device):
            flag = nan_flag if nan_flag is not None else torch.zeros(1, dtype=torch.int32, device=self.device)
            Xs = [self._prep(X, None)[0] for X in X_tests]
            n_test = Xs[0].shape[1]
            y_nan = torch.full((1, n_test), float("nan"), dtype=torch.float32, device=self.device)
            st, stb, views = self._group_buffers([(c.B, n_test, c.T) for c in ctxs])
            for c, X, v in zip(ctxs, Xs, views):
                if X.shape[0] != c.B or X.shape[2] != c.F or X.shape[1] != n_test:
                    raise ValueError("test tables do not match their contexts")
                self.embed(X, c.tab_stats, img_tok_test, y_nan, c.y_mean, c.y_mask, c.pos_emb, B=c.B, S=n_test, F=c.F,
                           x_bstride=n_test * c.F, y_bstride=0, nan_flag=flag, out=v)
            self._layers_multi(st, stb, [(c.B, c.T) for c in ctxs], n_test, [c.kv for c in ctxs], ctxs[0].n_train)
            return [self.decode(v[0]) for v in views]

    def forward_batch(self, X_full, img_full, y_train, *, check=True, return_embeddings=False):
        """Reference-equivalent joint forward for B estimators sharing the image embeddings:
        X_full [B, S, F] (train rows first), img_full [S, n_tok, img_dim], y_train [B, Ntr]
        -> logits [B, Nte, n_out].  Identical to ``_forward`` (transformer.py:555-867) because train
        rows never attend to test rows (layer.py:346-372); the stem statistics see all S rows."""
        with torch.cuda.device(self.device):
            X_full, img_full = self._prep(X_full, img_full)
            y_train = y_train.to(self.device, torch.float32)
            if y_train.dim() == 1:
                y_train = y_train[None]
            n_train = y_train.shape[1]
            S = X_full.shape[1] if X_full is not None else img_full.shape[0]
            if not 0 < n_train < S:
                raise ValueError("single_eval_pos must split the rows into train and test")
            img_tok = self.stem_image(img_full) if img_full is not None else None
            X_tr = None if X_full is None else X_full[:, :n_train].contiguous()
            X_te = None if X_full is None else X_full[:, n_train:].contiguous()
            # ONE flag for train and test rows: the reference raises on NaN anywhere in the embedded input
            # (transformer.py:790-796)
            flag = torch.zeros(1, dtype=torch.int32, device=self.device)
            ctx = self.fit_context(X_tr, None, y_train, X_all=X_full,
                                   img_tok_train=None if img_tok is None else img_tok[:n_train].contiguous(),
                                   check=False, nan_flag=flag, keep_train_out=return_embeddings)
            if img_full is not None:
                ctx.n_tok = img_full.shape[1]
            out = self.predict_with_context(ctx, X_te, None,
                                            img_tok_test=None if img_tok is None else img_tok[n_train:].contiguous(),
                                            check=check, nan_flag=flag, return_embeddings=return_embeddings)
            if return_embeddings:
                return out[0], ctx.train_out, out[1]
            return out

    def empty_trainset_representation_cache(self):
        """transformer.py:999-1001"""
        self._cached_ctx = None

    def __call__(self, *args, only_return_standard_out: bool = True, categorical_inds=None,
                 single_eval_pos: Optional[int] = None, **kwargs):
        """The reference's 4-positional-argument inference call (transformer.py:540-543):
        ``model(style, x [S,1,F], image [S,n_tok,768], y [Ntr]) -> [Nte, 1, n_out]``.

        With ``cache_trainset_representation`` set (the reference's model-level cache,
        multi_head_attention.py:328-336, layer.py:305-309): a call with ``y`` and ``single_eval_pos`` builds and
        KEEPS the train context (rows past ``single_eval_pos``, if any, are classified against it); a call with
        ``y=None, single_eval_pos=None`` classifies its rows against the kept context.
        ``only_return_standard_out=False`` returns the reference's dictionary (transformer.py:855-867):
        ``standard`` plus ``train_embeddings`` / ``test_embeddings`` (the y-token after the last layer)."""
        if kwargs:
            raise AssertionError(f"unsupported keyword arguments: {sorted(kwargs)}")        # transformer.py:515-516
        if len(args) != 4:
            raise ValueError("Unrecognized input. Please follow the doc string.")          # transformer.py:545
        style, x, image, y = args
        assert style is None                                                               # transformer.py:592
        if x is not None:
            if x.dim() != 3 or x.shape[1] != 1:
                raise ValueError("x must be [S, 1, F] (the engine passes batch size 1, inference.py:305)")
            x = x[:, 0]
        if image is not None and image.dim() > 3:
            image = torch.movedim(image, 0, 1)[0]                                           # transformer.py:586-588
        want_emb = not only_return_standard_out

        def pack(logits, train_emb, test_emb):
            std = logits[0][:, None, :]
            if not want_emb:
                return std
            return {"standard": std, "train_embeddings": train_emb[0][:, None, :], "test_embeddings": test_emb[0][:, None, :]}

        if self.cache_trainset_representation and not single_eval_pos:                      # transformer.py:593-595
            assert y is None
            if self._cached_ctx is None:
                raise AssertionError("the train-set representation cache is empty")         # layer.py:307
            out = self.predict_with_context(self._cached_ctx, None if x is None else x[None], image,
                                            return_embeddings=want_emb)
            if want_emb:
                empty = out[1].new_zeros((1, 0, out[1].shape[-1]))
                return pack(out[0], empty, out[1])
            return pack(out, None, None)
        assert y is not None and single_eval_pos                                            # transformer.py:597-598
        y = y.reshape(-1)
        if y.shape[0] != single_eval_pos:
            raise AssertionError("For main y, y must not be given for target time steps")   # transformer.py:695-698
        n_train = int(single_eval_pos)
        S = x.shape[0] if x is not None else image.shape[0]
        if self.cache_trainset_representation:
            # the cached form: the stem statistics come from the rows of THIS call (encoders.py:368-371)
            with torch.cuda.device(self.device):
                Xd, imgd = self._prep(None if x is None else x[None], image)
                ctx = self.fit_context(None if Xd is None else Xd[:, :n_train].contiguous(),
                                       None if imgd is None else imgd[:n_train].contiguous(), y[None], X_all=Xd,
                                       keep_train_out=want_emb)
                self._cached_ctx = ctx
                if S > n_train:
                    out = self.predict_with_context(ctx, None if Xd is None else Xd[:, n_train:].contiguous(),
                                                    None if imgd is None else imgd[n_train:].contiguous(),
                                                    return_embeddings=want_emb)
                    return pack(out[0], ctx.train_out, out[1]) if want_emb else pack(out, None, None)
                empty_l = torch.zeros((1, 0, self.geom.n_out), dtype=torch.float32, device=self.device)
                empty_e = torch.zeros((1, 0, self.geom.emsize), dtype=torch.float32, device=self.device)
                return pack(empty_l, ctx.train_out, empty_e)
        out = self.forward_batch(None if x is None else x[None], image, y[None], return_embeddings=want_emb)
        return pack(*out) if want_emb else pack(out, None, None)
