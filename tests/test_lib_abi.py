"""CPU-side checks of the C-ABI boundary: the library builds, loads, exports every symbol the
header declares, and refuses to compute without an sm_100 device (no CPU fallback)."""
import ctypes
import os
import re

import pytest
import torch

from multimodalpfn_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "mmpfn_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mmpfn_[a-z0-9_]+)\s*\(", src)))


def test_header_and_binding_agree():
    syms = header_symbols()
    assert len(syms) >= 18
    assert set(syms) == set(_lib.SIGNATURES), set(syms) ^ set(_lib.SIGNATURES)


def test_library_matches_header():
    _lib.load()
    lib = ctypes.CDLL(_lib.lib_path())
    for s in header_symbols():
        assert hasattr(lib, s), s
    assert _lib.load().mmpfn_abi_version() == 2


def test_struct_layouts():
    assert ctypes.sizeof(_lib.Geometry) == 40
    assert ctypes.sizeof(_lib.Weights) == 8 * len(_lib.WEIGHT_FIELDS)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_compute_calls_refuse_without_device():
    lib = _lib.load()
    rc = lib.mmpfn_layernorm(None, None, None, None, 1, 192, None, None, None)
    assert rc == -2  # MMPFN_ENODEVICE
    assert b"no CPU fallback" in lib.mmpfn_last_error()
    g = _lib.Geometry(192, 6, 768, 12, 10, 2, 768, 8, 8, 2)
    segs = (_lib.Segment * 1)(_lib.Segment(1, 5))
    kv = (ctypes.c_void_p * 1)(None)
    assert lib.mmpfn_layers_train_ragged(ctypes.byref(g), None, None, None, segs, 1, 10, None, 1, kv, None, 0,
                                         None) == -2
    assert lib.mmpfn_item_qkv_bf16(None, None, 1, 1, 2, 64, 3, None, None, None, None, None, None) == -2
    from multimodalpfn_b200.model import B200PerFeatureTransformer
    from multimodalpfn_b200.synth import Geometry
    with pytest.raises(RuntimeError):
        B200PerFeatureTransformer({}, Geometry())


def test_size_queries_need_no_device():
    lib = _lib.load()
    g = _lib.Geometry(192, 6, 768, 12, 10, 2, 768, 8, 8, 2)
    assert lib.mmpfn_layer_weight_elems(ctypes.byref(g)) == 2 * (3 * 192 * 192 + 192 * 192) + 2 * 768 * 192
    assert lib.mmpfn_image_tokens(ctypes.byref(g), 3) == 8
    assert lib.mmpfn_tab_stats_elems(ctypes.byref(g), 11) == 6 * 22 + 11
    assert lib.mmpfn_kv_bytes(ctypes.byref(g), 2, 100, 20, 0) == 12 * 2 * 20 * 100 * 64 * 4
    assert lib.mmpfn_kv_bytes(ctypes.byref(g), 2, 100, 20, 1) == 12 * 2 * 20 * 128 * 64 * 2
    one = (_lib.Segment * 1)(_lib.Segment(1, 20))
    assert lib.mmpfn_layers_ragged_ws_bytes(ctypes.byref(g), one, 1, 100, 0) > 0
    segs = (_lib.Segment * 2)(_lib.Segment(4, 27), _lib.Segment(4, 20))
    M = 4 * 100 * 27 + 4 * 100 * 20
    planes = 3 * 4 * (27 + 20) * 6 * 128 * 32 * 2
    assert lib.mmpfn_layers_ragged_ws_bytes(ctypes.byref(g), segs, 2, 100, 1) >= M * 768 * 2 + M * 192 * 2 + planes
    assert lib.mmpfn_layers_ragged_ws_bytes(ctypes.byref(g), segs, 9, 100, 1) == 0     # more than MMPFN_MAX_SEGMENTS
