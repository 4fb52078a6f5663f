"""The fp16 precision on the host side, without a GPU: precision parsing of the estimators and the plug-in, the new
ABI symbols, and the fp16 weight copy."""
import ctypes as C

import numpy as np
import pytest
import torch

from multimodalpfn_b200 import _lib
from multimodalpfn_b200.classifier import MMPFNClassifier, precision_name
from multimodalpfn_b200.regressor import MMPFNRegressor

F16_SYMBOLS = ["mmpfn_item_attention_f16", "mmpfn_item_qkv_f16", "mmpfn_feature_attention_f16",
               "mmpfn_feature_qkv_attention_f16", "mmpfn_linear_ln_f16", "mmpfn_mlp_f16"]


@pytest.mark.parametrize("value,name", [(torch.float16, "fp16"), ("fp16", "fp16"), ("float16", "fp16"),
                                        ("auto", "bf16"), ("autocast", "bf16"), (torch.bfloat16, "bf16"),
                                        ("bf16", "bf16"), ("bfloat16", "bf16"), (torch.float32, "fp32"),
                                        ("fp32", "fp32"), ("float32", "fp32")])
def test_precision_parsing(value, name):
    assert precision_name(value) == name
    assert MMPFNClassifier(inference_precision=value)._precision() == name
    assert MMPFNRegressor(inference_precision=value)._precision() == name


@pytest.mark.parametrize("value", ["fp8", torch.float64, "half-ish", None])
def test_precision_parsing_rejects(value):
    with pytest.raises(ValueError):
        precision_name(value)
    with pytest.raises(ValueError):
        MMPFNClassifier(inference_precision=value)._precision()


def test_default_is_still_bf16():
    assert MMPFNClassifier()._precision() == "bf16"
    assert MMPFNRegressor()._precision() == "bf16"


def test_plugin_install_parses_precision(monkeypatch):
    """plugin.install normalises the precision before it patches anything: fp16 spellings give "fp16", "auto" stays
    bf16, an unknown one raises."""
    import sys
    import types

    from multimodalpfn_b200 import plugin
    seen = []

    def fake_factory(**kw):
        return types.SimpleNamespace(model="ref-model")
    mods = {}
    for name in ("mmpfn", "mmpfn.models", "mmpfn.models.mmpfn", "mmpfn.models.mmpfn.classifier",
                 "mmpfn.models.mmpfn.regressor"):
        mods[name] = types.ModuleType(name)
    mods["mmpfn.models.mmpfn.classifier"].create_inference_engine = fake_factory
    mods["mmpfn.models.mmpfn.regressor"].create_inference_engine = fake_factory
    for name, m in mods.items():
        monkeypatch.setitem(sys.modules, name, m)
    mods["mmpfn"].models = mods["mmpfn.models"]
    mods["mmpfn.models"].mmpfn = mods["mmpfn.models.mmpfn"]
    mods["mmpfn.models.mmpfn"].classifier = mods["mmpfn.models.mmpfn.classifier"]
    mods["mmpfn.models.mmpfn"].regressor = mods["mmpfn.models.mmpfn.regressor"]
    monkeypatch.setattr(plugin, "convert", lambda m, *, device, precision, model_cls, pos_emb_device="cuda":
                        seen.append(precision) or "b200-model")
    for value, name in ((torch.float16, "fp16"), ("fp16", "fp16"), ("auto", "bf16"), ("fp32", "fp32")):
        uninstall = plugin.install(precision=value, mode="model")
        eng = mods["mmpfn.models.mmpfn.classifier"].create_inference_engine(device_=torch.device("cuda"))
        assert eng.model == "b200-model"
        assert seen[-1] == name
        uninstall()
    with pytest.raises(ValueError):
        plugin.install(precision="fp8")


def test_f16_symbols_bound():
    assert _lib.F16 == 2
    assert "layers_f16" in _lib.WEIGHT_FIELDS and _lib.WEIGHT_FIELDS[-1] == "layers_f16"
    lib = _lib.load()
    for s in F16_SYMBOLS:
        assert s in _lib.SIGNATURES
        assert getattr(lib, s).argtypes == _lib.SIGNATURES[s][1]
    # the fp16 pass sizes its workspace and K/V context like the bf16 pass
    from multimodalpfn_b200.synth import Geometry
    g = Geometry(mgm_heads=2, cap_heads=4)
    cg = _lib.Geometry(g.emsize, g.nhead, g.nhid, g.nlayers, g.n_out, g.features_per_group, g.img_dim, g.mgm_heads,
                       g.cap_heads, _lib.MIXER[g.mixer_type])
    segs = (_lib.Segment * 2)(_lib.Segment(4, 12), _lib.Segment(3, 20))
    for S in (1, 300):
        assert lib.mmpfn_layers_ragged_ws_bytes(C.byref(cg), segs, 2, S, _lib.F16) == \
            lib.mmpfn_layers_ragged_ws_bytes(C.byref(cg), segs, 2, S, _lib.BF16) > 0
        assert lib.mmpfn_kv_bytes(C.byref(cg), 4, S, 12, _lib.F16) == lib.mmpfn_kv_bytes(C.byref(cg), 4, S, 12, _lib.BF16)


def test_f16_entry_points_need_a_device():
    """No CPU fallback: without an sm_100 device the fp16 building blocks return MMPFN_ENODEVICE like the others."""
    if torch.cuda.is_available():
        pytest.skip("this machine has a GPU")
    lib = _lib.load()
    assert lib.mmpfn_mlp_f16(None, None, None, None, 1, None) == -2
    assert lib.mmpfn_feature_attention_f16(None, None, 1, 2, None) == -2


def test_packed_weights_f16_holds_no_bf16_copy():
    """PackedWeights for an fp16 model: fp16 copies of the layer blocks (the second query set too), no bf16 copy
    anywhere, and the struct points layers_f16 at them (on the CPU device: the packing needs no GPU)."""
    from multimodalpfn_b200.synth import Geometry, make_state_dict
    from multimodalpfn_b200.weights import PackedWeights
    geom = Geometry(mgm_heads=2, cap_heads=4)
    sd = make_state_dict(geom, seed=0)
    # a two_sets_of_queries checkpoint: _w_q [2,H,D,E] + _w_kv [2,H,D,E] for the item attention
    for l in range(geom.nlayers):
        p = f"transformer_encoder.layers.{l}.self_attn_between_items."
        w = sd.pop(p + "_w_qkv")
        sd[p + "_w_q"] = np.stack([w[0], w[0] * 0.5])
        sd[p + "_w_kv"] = w[1:]
    w = PackedWeights(sd, geom, torch.device("cpu"), with_bf16=False, stem_bf16=False, with_f16=True)
    assert w.two_sets_of_queries
    names = set(w._t)
    assert {"layers_f16", "layers_test_f16"} <= names
    assert not any(n.endswith("_bf16") for n in names), names
    assert w.tensor("layers_f16").dtype == torch.float16
    assert w.c_weights.layers_f16 == w.tensor("layers_f16").data_ptr()
    assert w.c_weights_test.layers_f16 == w.tensor("layers_test_f16").data_ptr()
    assert not w.c_weights.layers_bf16 and not w.c_weights.mgm_w1_bf16
    np.testing.assert_array_equal(w.tensor("layers_f16").float().numpy(),
                                  w.tensor("layers_f32").to(torch.float16).float().numpy())
    # the default (bf16) packing is unchanged: no fp16 copy
    wb = PackedWeights(sd, geom, torch.device("cpu"))
    assert "layers_f16" not in wb._t and "layers_bf16" in wb._t and not wb.c_weights.layers_f16
