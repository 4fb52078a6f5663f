"""Repack a reference state_dict (SURVEY.md Appendix B; reference ``model/loading.py:401-542``)
into the device layouts ``include/mmpfn_b200.h`` documents.

Host-side algebra done once at load time (float64, then rounded to fp32):
* the per-head LayerNorm affine of MGM (``model/transformer.py:38-39``) is folded into the first
  linear layer, W' = W diag(gamma), b' = b + W beta, so that the 768-wide normalisation runs once
  for all heads; the GLU halves (``nn.GLU``, ``:40``) are interleaved row-wise so that a GEMM
  epilogue sees (value, gate) in adjacent columns;
* CAP's learned queries are row independent (``model/transformer.py:81``): q_norm, q_proj and the
  query third of ``mha.in_proj`` are applied here.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .synth import Geometry

__all__ = ["PackedWeights", "load_checkpoint", "load_borders"]


def _np(v) -> np.ndarray:
    if isinstance(v, torch.Tensor):
        v = v.detach().cpu().numpy()
    return np.asarray(v)


def _ln64(x, g, b, eps=1e-5):
    mu = x.mean(-1, keepdims=True)
    var = ((x - mu) ** 2).mean(-1, keepdims=True)
    return (x - mu) / np.sqrt(var + eps) * g + b


class PackedWeights:
    """Device-resident weights + the ctypes structs the C ABI takes."""

    def __init__(self, state_dict, geom: Geometry, device: torch.device, *, with_bf16: bool = True,
                 stem_bf16: bool = True, with_f16: bool = False):
        sd = {k: _np(v).astype(np.float64) for k, v in state_dict.items()}
        self.geom = geom
        self.device = torch.device(device)
        E, H, D, Hid, L = geom.emsize, geom.nhead, geom.d_k, geom.nhid, geom.nlayers
        # Checkpoints with ``two_sets_of_queries`` (multi_head_attention.py:216-260) carry, for the item attention,
        # ``_w_q [2,H,D,E]`` + ``_w_kv [2,H,D,E]`` instead of ``_w_qkv [3,H,D,E]``: query set 0 serves the train rows
        # and set 1 the test rows (layer.py:357, ``use_second_set_of_queries``).  The train pass and the test pass are
        # separate launches here, so the second set simply is the test pass's copy of the layer block.
        def qkv_of(prefix, q_set):
            if prefix + "._w_qkv" in sd:
                w = sd[prefix + "._w_qkv"]
            else:
                wq, wkv = sd[prefix + "._w_q"], sd[prefix + "._w_kv"]
                assert wq.shape[1:] == (H, D, E) and wkv.shape == (2, H, D, E), (wq.shape, wkv.shape)
                w = np.stack([wq[min(q_set, wq.shape[0] - 1)], wkv[0], wkv[1]])
            assert w.shape == (3, H, D, E), w.shape
            return w.reshape(3 * H * D, E)

        self.two_sets_of_queries = any(k.endswith("self_attn_between_items._w_q") and v.shape[0] == 2 for k, v in sd.items())

        def layer_blocks(q_set):
            blocks = []
            for l in range(L):
                p = f"transformer_encoder.layers.{l}."
                for att in ("self_attn_between_features", "self_attn_between_items"):
                    blocks.append(qkv_of(p + att, q_set if att == "self_attn_between_items" else 0))
                    blocks.append(sd[p + att + "._w_out"].reshape(H * D, E).T)       # [e][h*D+d]
                blocks.append(sd[p + "mlp.linear1.weight"])
                blocks.append(sd[p + "mlp.linear2.weight"])
            return np.concatenate([np.ascontiguousarray(b).reshape(-1) for b in blocks]).astype(np.float32)

        layers = layer_blocks(0)
        self._t = {}
        self._t["layers_f32"] = torch.from_numpy(layers).to(self.device)
        # 16-bit copies of the layer blocks for the tensor-core layers: bf16 (MMPFN_BF16) and / or fp16 (MMPFN_F16)
        half = [(sfx, dt) for sfx, dt, on in (("bf16", torch.bfloat16, with_bf16), ("f16", torch.float16, with_f16)) if on]
        for sfx, dt in half:
            self._t["layers_" + sfx] = self._t["layers_f32"].to(dt)
        if self.two_sets_of_queries:
            self._t["layers_test_f32"] = torch.from_numpy(layer_blocks(1)).to(self.device)
            for sfx, dt in half:
                self._t["layers_test_" + sfx] = self._t["layers_test_f32"].to(dt)

        def put(name, arr):
            self._t[name] = torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float32)).to(self.device)

        put("enc_w", sd["encoder.5.layer.weight"])
        # regression checkpoints (max_num_classes = 0): the y-encoder has no class-rank step, its Linear is step 1
        # (model/loading.py:374-398); the target value itself is embedded
        self.regression = "y_encoder.2.layer.weight" not in sd
        ykey = "y_encoder.1.layer." if self.regression else "y_encoder.2.layer."
        put("yenc_w", sd[ykey + "weight"])
        put("yenc_b", sd[ykey + "bias"])
        put("dec_w1", sd["decoder_dict.standard.0.weight"])
        put("dec_b1", sd["decoder_dict.standard.0.bias"])
        put("dec_w2", sd["decoder_dict.standard.2.weight"])
        put("dec_b2", sd["decoder_dict.standard.2.bias"])
        # positional-embedding projection stays on the host (torch RNG semantics, transformer.py:925-933)
        self.pe_w = torch.from_numpy(sd["feature_positional_embedding_embeddings.weight"].astype(np.float32))
        self.pe_b = torch.from_numpy(sd["feature_positional_embedding_embeddings.bias"].astype(np.float32))

        I = geom.img_dim
        if geom.mixer_type in ("MGM", "MGM+CAP"):
            w1s, b1s, w2s, b2s = [], [], [], []
            for h in range(geom.mgm_heads):
                p = f"mgm.projs.{h}."
                g_, be = sd[p + "0.weight"], sd[p + "0.bias"]
                W1, b1 = sd[p + "1.weight"], sd[p + "1.bias"]
                W1f = W1 * g_[None, :]
                b1f = b1 + W1 @ be
                inter = np.empty_like(W1f)
                inter[0::2] = W1f[: I // 2]
                inter[1::2] = W1f[I // 2:]
                bint = np.empty_like(b1f)
                bint[0::2] = b1f[: I // 2]
                bint[1::2] = b1f[I // 2:]
                w1s.append(inter)
                b1s.append(bint)
                w2s.append(sd[p + "4.weight"])
                b2s.append(sd[p + "4.bias"])
            put("mgm_w1", np.concatenate(w1s, 0))
            put("mgm_b1", np.concatenate(b1s, 0))
            put("mgm_w2", np.stack(w2s, 0))
            put("mgm_b2", np.stack(b2s, 0))
            if with_bf16 and stem_bf16:
                # operand of the tcgen05 MGM GEMM (bf16 mode only; the fp32 mode keeps the FFMA path for the 1e-5 gate)
                self._t["mgm_w1_bf16"] = self._t["mgm_w1"].to(torch.bfloat16)
        if geom.mixer_type == "MoE":
            w1s, b1s, w2s, b2s = [], [], [], []
            for h in range(geom.mgm_heads):
                p = f"moe.experts.{h}."
                g_, be = sd[p + "0.weight"], sd[p + "0.bias"]
                W1, b1 = sd[p + "1.weight"], sd[p + "1.bias"]
                w1s.append(W1 * g_[None, :])
                b1s.append(b1 + W1 @ be)
                w2s.append(sd[p + "4.weight"])
                b2s.append(sd[p + "4.bias"])
            put("mgm_w1", np.concatenate(w1s, 0))
            put("mgm_b1", np.concatenate(b1s, 0))
            put("mgm_w2", np.stack(w2s, 0))
            put("mgm_b2", np.stack(b2s, 0))
            put("moe_gate_w", sd["moe.gate.weight"])
            put("moe_gate_b", sd["moe.gate.bias"])
        if geom.mixer_type == "MGM+CAP":
            Wi, bi = sd["cap.mha.in_proj_weight"], sd["cap.mha.in_proj_bias"]
            q0 = _ln64(sd["cap.queries"], sd["cap.q_norm.weight"], sd["cap.q_norm.bias"]) @ sd["cap.q_proj.weight"].T
            put("cap_q", q0 @ Wi[:E].T + bi[:E])
            put("cap_wkv", Wi[E:])
            put("cap_bkv", bi[E:])
            put("cap_knorm_w", sd["cap.k_norm.weight"])
            put("cap_knorm_b", sd["cap.k_norm.bias"])
            put("cap_wo", sd["cap.mha.out_proj.weight"])
            put("cap_bo", sd["cap.mha.out_proj.bias"])
            put("cap_onorm_w", sd["cap.out_norm.weight"])
            put("cap_onorm_b", sd["cap.out_norm.bias"])
            put("cap_f1_w", sd["cap.ffn.0.weight"])
            put("cap_f1_b", sd["cap.ffn.0.bias"])
            put("cap_f2_w", sd["cap.ffn.3.weight"])
            put("cap_f2_b", sd["cap.ffn.3.bias"])

        self.c_geom = _lib.Geometry(E, H, Hid, L, geom.n_out, geom.features_per_group, I, geom.mgm_heads,
                                    geom.cap_heads or 0, _lib.MIXER[geom.mixer_type])
        self.c_weights = _lib.Weights()
        for name in _lib.WEIGHT_FIELDS:
            t = self._t.get(name)
            setattr(self.c_weights, name, None if t is None else t.data_ptr())
        # the weights the TEST pass uses: the same struct unless the checkpoint has a second set of item queries
        self.c_weights_test = self.c_weights
        if self.two_sets_of_queries:
            self.c_weights_test = _lib.Weights()
            for name in _lib.WEIGHT_FIELDS:
                t = self._t.get({"layers_f32": "layers_test_f32", "layers_bf16": "layers_test_bf16",
                                 "layers_f16": "layers_test_f16"}.get(name, name))
                setattr(self.c_weights_test, name, None if t is None else t.data_ptr())
        expected = _lib.load().mmpfn_layer_weight_elems(C.byref(self.c_geom)) * L
        if expected != layers.size:
            raise RuntimeError(f"layer weight block mismatch: packed {layers.size}, library expects {expected}")

    def tensor(self, name):
        return self._t[name]

    def n_params(self) -> int:
        return sum(t.numel() for k, t in self._t.items() if not k.endswith(("_bf16", "_f16")))


def geometry_from_checkpoint(config: dict, state_dict, *, mixer_type, mgm_heads, cap_heads,
                             features_per_group=None) -> Geometry:
    """Geometry from a reference ``.ckpt`` config (``model/config.py:18-83``) + the ctor kwargs the
    reference takes outside the checkpoint (``classifier.py:112-137``)."""
    n_out = int(_np(state_dict["decoder_dict.standard.2.weight"]).shape[0])
    img_dim = int(config.get("emsize", 192)) * int(config.get("nhid_factor", 4))   # transformer.py:295-301
    return Geometry(emsize=int(config.get("emsize", 192)), nhead=int(config.get("nhead", 6)),
                    nhid_factor=int(config.get("nhid_factor", 4)), nlayers=int(config.get("nlayers", 12)),
                    n_out=n_out,
                    features_per_group=int(features_per_group or config.get("features_per_group", 2)),
                    img_dim=img_dim, mgm_heads=int(mgm_heads), cap_heads=cap_heads, mixer_type=mixer_type)


def load_checkpoint(path, *, mixer_type="MGM+CAP", mgm_heads=8, cap_heads=8, features_per_group=None):
    """Read the reference checkpoint format ``{"state_dict", "config"}`` (``model/loading.py:427-444``)."""
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    sd = ckpt["state_dict"]
    sd = {k: v for k, v in sd.items() if not k.startswith("criterion.")}      # bar-distribution borders: host side
    geom = geometry_from_checkpoint(ckpt.get("config", {}), sd, mixer_type=mixer_type, mgm_heads=mgm_heads,
                                    cap_heads=cap_heads, features_per_group=features_per_group)
    return sd, geom


def load_borders(path) -> np.ndarray:
    """The bar-distribution borders ``criterion.borders`` [n_out + 1] of a regression checkpoint (float64, over the
    standardised target); ValueError when the checkpoint has none."""
    sd = torch.load(path, map_location="cpu", weights_only=False)["state_dict"]
    if "criterion.borders" not in sd:
        raise ValueError("checkpoint has no criterion.borders (not a regression checkpoint)")
    return _np(sd["criterion.borders"]).astype(np.float64).ravel()
