"""ctypes binding of libmmpfn_b200.so (include/mmpfn_b200.h).

There is no fallback of any kind: if the shared library is missing or a call fails, a
``RuntimeError`` is raised with the library's own message.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

c_void_p, c_int, c_float, c_size_t, c_int64, c_ll = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_int64, C.c_longlong

F32, BF16, F16 = 0, 1, 2
MAX_SEGMENTS = 8          # MMPFN_MAX_SEGMENTS
MIXER = {"none": 0, "MGM": 1, "MGM+CAP": 2, "MoE": 3}
ERRORS = {-1: "EINVAL", -2: "ENODEVICE", -3: "ECUDA", -4: "EUNSUPPORTED"}


class Geometry(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("emsize", "nhead", "nhid", "nlayers", "n_out", "features_per_group",
                                         "img_dim", "mgm_heads", "cap_heads", "mixer_type")]


WEIGHT_FIELDS = ("layers_f32", "layers_bf16", "enc_w", "yenc_w", "yenc_b", "dec_w1", "dec_b1", "dec_w2", "dec_b2",
                 "mgm_w1", "mgm_b1", "mgm_w2", "mgm_b2", "moe_gate_w", "moe_gate_b", "cap_knorm_w", "cap_knorm_b",
                 "cap_q", "cap_wkv", "cap_bkv", "cap_wo", "cap_bo", "cap_onorm_w", "cap_onorm_b", "cap_f1_w",
                 "cap_f1_b", "cap_f2_w", "cap_f2_b", "mgm_w1_bf16", "layers_f16")


class Weights(C.Structure):
    _fields_ = [(n, c_void_p) for n in WEIGHT_FIELDS]


class Segment(C.Structure):
    _fields_ = [("B", C.c_int32), ("T", C.c_int32)]


class KvSegment(C.Structure):
    """mmpfn_kv_segment (include/mmpfn_b200.h)"""
    _fields_ = [("B", C.c_int32), ("T", C.c_int32), ("kv", C.c_void_p), ("layer_stride", C.c_int64),
                ("slots", C.c_int32), ("seg_rows", C.c_int32), ("rank_stride", C.c_int64),
                ("kg", C.c_void_p), ("vtg", C.c_void_p), ("gather_stride", C.c_int64), ("rank", C.c_int32),
                ("n_ranks", C.c_int32), ("n_rows_total", C.c_int32), ("reserved", C.c_int32)]


PG, PW = C.POINTER(Geometry), C.POINTER(Weights)
PS, PVP = C.POINTER(Segment), C.POINTER(C.c_void_p)
PKS = C.POINTER(KvSegment)

# name -> (restype, argtypes): exactly the entry points include/mmpfn_b200.h declares
SIGNATURES = {
    "mmpfn_abi_version": (c_int, []),
    "mmpfn_last_error": (C.c_char_p, []),
    "mmpfn_launch_count": (c_int64, []),
    "mmpfn_device_supported": (c_int, [c_int]),
    "mmpfn_layer_weight_elems": (c_size_t, [PG]),
    "mmpfn_image_tokens": (c_int, [PG, c_int]),
    "mmpfn_tab_stats_elems": (c_size_t, [PG, c_int]),
    "mmpfn_stem_tab_fit": (c_int, [PG, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "mmpfn_stem_image_ws_bytes": (c_size_t, [PG, c_int, c_int]),
    "mmpfn_stem_image": (c_int, [PG, PW, c_void_p, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "mmpfn_stem_tokens": (c_int, [PG, PW, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int, c_int, c_ll, c_ll, c_ll, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mmpfn_kv_bytes": (c_size_t, [PG, c_int, c_int, c_int, c_int]),
    "mmpfn_layers_run": (c_int, [PG, PW, c_void_p, c_void_p, PKS, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                 c_void_p, c_size_t, c_void_p]),
    "mmpfn_decode": (c_int, [PG, PW, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "mmpfn_proba_tail": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p,
                                 c_void_p]),
    "mmpfn_bar_tail": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int,
                               c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mmpfn_bar_tail_tasks": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_float, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p]),
    "mmpfn_layernorm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "mmpfn_linear_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "mmpfn_linear_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "mmpfn_item_qkv_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p]),
    "mmpfn_linear_ln_bf16": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "mmpfn_mlp_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "mmpfn_feature_attention_bf16": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_void_p]),
    "mmpfn_feature_qkv_attention_bf16": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_void_p, c_void_p]),
    "mmpfn_item_attention_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                          c_int, c_void_p, c_void_p]),
    "mmpfn_stem_tab_fit_ragged": (c_int, [PG, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p,
                                          c_void_p]),
    "mmpfn_stem_tokens_ragged": (c_int, [PG, PW, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_int, c_int, c_int, c_int, c_ll, c_ll, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p]),
    "mmpfn_layers_ragged_ws_bytes": (c_size_t, [PG, PS, c_int, c_int, c_int]),
    "mmpfn_layers_train_ragged": (c_int, [PG, PW, c_void_p, c_void_p, PS, c_int, c_int, c_void_p, c_int, PVP, c_void_p,
                                          c_size_t, c_void_p]),
    "mmpfn_layers_test_ragged": (c_int, [PG, PW, c_void_p, c_void_p, PS, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                         PVP, c_void_p, c_size_t, c_void_p]),
    "mmpfn_item_attention_bf16_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                                 c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mmpfn_linear_ln_f16": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "mmpfn_item_qkv_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p]),
    "mmpfn_mlp_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "mmpfn_item_attention_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                         c_void_p, c_void_p, c_void_p, c_void_p]),
    "mmpfn_feature_attention_f16": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_void_p]),
    "mmpfn_feature_qkv_attention_f16": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_void_p, c_void_p]),
    "mmpfn_item_attention_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                         c_void_p, c_void_p, c_void_p]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """Load the shared library (compiling it in-tree if it is absent or stale and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if build_if_missing and not _build.is_current():
        try:
            _build.build()
        except Exception as exc:  # no nvcc on this machine: use the shipped .so if there is one
            if not os.path.exists(path):
                raise RuntimeError(f"libmmpfn_b200.so is missing and could not be built: {exc}") from exc
            import warnings
            warnings.warn(f"{os.path.basename(path)} is older than its sources and could not be rebuilt ({exc}); "
                          "loading the stale library", RuntimeWarning, stacklevel=2)
    if not os.path.exists(path):
        raise RuntimeError(f"{path} not found — run `python -m multimodalpfn_b200.build`; there is no fallback path")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError here = header and library out of sync
        fn.restype = res
        fn.argtypes = args
    if lib.mmpfn_abi_version() != 2:
        raise RuntimeError("libmmpfn_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().mmpfn_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed ({ERRORS.get(rc, rc)}): {msg}")


def launch_count() -> int:
    return int(load().mmpfn_launch_count())
