"""GPU parity of the building blocks exported through the C ABI (LayerNorm, fp32 linear, tcgen05
linear) and of single layers against the oracle.  Each check compares with plain fp32 torch /
the oracle on the same seeded inputs; tolerances are written next to each assert."""
import ctypes as C

import numpy as np
import pytest
import torch

from multimodalpfn_b200 import _lib
from multimodalpfn_b200.synth import Geometry, make_state_dict

pytestmark = pytest.mark.gpu


def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("width", [192, 768])
@pytest.mark.parametrize("rows", [1, 77, 4097])
def test_layernorm(width, rows):
    lib = _lib.load()
    g = torch.Generator().manual_seed(rows + width)
    x = (torch.randn(rows, width, generator=g) * 3 + 0.5).cuda()
    r = torch.randn(rows, width, generator=g).cuda()
    gam = torch.randn(width, generator=g).cuda()
    bet = torch.randn(width, generator=g).cuda()
    y = torch.empty_like(x)
    yb = torch.empty(rows, width, dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.mmpfn_layernorm(x.data_ptr(), r.data_ptr(), gam.data_ptr(), bet.data_ptr(), rows, width,
                                   y.data_ptr(), yb.data_ptr(), _stream()), "layernorm")
    ref = torch.nn.functional.layer_norm((x + r).double(), (width,), gam.double(), bet.double(), 1e-5)
    assert (y.double() - ref).abs().max().item() < 5e-6          # fp32 vs fp64 reference
    assert (yb.double() - ref).abs().max().item() < 0.05          # bf16 rounding of O(4) values
    y2 = torch.empty_like(x)
    _lib.check(lib.mmpfn_layernorm(x.data_ptr(), None, None, None, rows, width, y2.data_ptr(), None, _stream()), "ln")
    ref2 = torch.nn.functional.layer_norm(x.double(), (width,), None, None, 1e-5)
    assert (y2.double() - ref2).abs().max().item() < 5e-6


@pytest.mark.parametrize("M,N,K,epi", [(1, 10, 768, 0), (300, 768, 192, 1), (1000, 576, 192, 0), (129, 192, 768, 0),
                                       (2300, 384, 192, 0)])
def test_linear_f32(M, N, K, epi):
    lib = _lib.load()
    g = torch.Generator().manual_seed(M * 7 + N)
    A = torch.randn(M, K, generator=g).cuda()
    W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
    b = torch.randn(N, generator=g).cuda()
    out = torch.empty(M, N, device="cuda")
    _lib.check(lib.mmpfn_linear_f32(A.data_ptr(), W.data_ptr(), b.data_ptr(), M, N, K, epi, out.data_ptr(), _stream()),
               "linear_f32")
    ref = A.double() @ W.double().T + b.double()
    if epi == 1:
        ref = torch.nn.functional.gelu(ref)
    assert (out.double() - ref).abs().max().item() < 2e-5         # fp32 accumulation over K <= 768


@pytest.mark.parametrize("M,N,K,epi", [(128, 192, 192, 0), (300, 576, 192, 0), (1000, 768, 192, 1), (129, 192, 768, 0),
                                       (62100, 576, 192, 0), (5, 768, 768, 1)])
def test_linear_bf16_tcgen05(M, N, K, epi):
    lib = _lib.load()
    g = torch.Generator().manual_seed(M * 3 + N + K)
    A = torch.randn(M, K, generator=g).cuda().to(torch.bfloat16)
    W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda().to(torch.bfloat16)
    out = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.mmpfn_linear_bf16(A.data_ptr(), W.data_ptr(), M, N, K, epi, out.data_ptr(), _stream()),
               "linear_bf16")
    torch.cuda.synchronize()
    ref = A.double() @ W.double().T                                # exact product of the bf16 operands
    if epi == 1:
        ref = torch.nn.functional.gelu(ref)
    err = (out.double() - ref).abs().max().item()
    assert not torch.isnan(out).any()
    assert err < 0.04, err                                          # bf16 output rounding of O(4) values


@pytest.mark.parametrize("M", [1, 128, 300, 20000, 62101])
def test_fused_mlp_tcgen05(M):
    """state <- LN(state + W2 gelu(W1 state)) (mlp.py:93-138, layer.py:437-455) in one kernel vs fp64 torch
    on the same bf16 operands.  The hidden activation is rounded to bf16 inside the kernel and the
    GELU is the tanh-form erf (kernels_mlp.cu): tolerance 0.03 on O(1) LayerNorm outputs."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(M)
    x = torch.randn(M, 192, generator=g).cuda()
    xb = x.to(torch.bfloat16)
    w1 = (torch.randn(768, 192, generator=g) / 192 ** 0.5).cuda().to(torch.bfloat16)
    w2 = (torch.randn(192, 768, generator=g) / 768 ** 0.5).cuda().to(torch.bfloat16)
    st, stb = x.clone(), xb.clone()
    _lib.check(lib.mmpfn_mlp_bf16(st.data_ptr(), stb.data_ptr(), w1.data_ptr(), w2.data_ptr(), M, _stream()), "mlp")
    torch.cuda.synchronize()
    h = torch.nn.functional.gelu(xb.double() @ w1.double().T)
    ref = torch.nn.functional.layer_norm(x.double() + h @ w2.double().T, (192,), None, None, 1e-5)
    e1 = (st.double() - ref).abs().max().item()
    e2 = (stb.double() - ref).abs().max().item()
    assert not torch.isnan(st).any()
    assert e1 < 0.03 and e2 < 0.05, (e1, e2)


@pytest.mark.parametrize("M", [1, 127, 128, 300, 18945, 62101])
def test_out_projection_layernorm_tcgen05(M):
    """state <- LN(state + A W^T) (multi_head_attention.py:513-517 + layer.py:437-455): the persistent
    tcgen05 kernel (resident W, TMA-staged fp32 residual ring) vs fp64 torch on the same bf16 operands."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + 11)
    x = torch.randn(M, 192, generator=g).cuda()
    a = torch.randn(M, 192, generator=g).cuda().to(torch.bfloat16)
    w = (torch.randn(192, 192, generator=g) / 192 ** 0.5).cuda().to(torch.bfloat16)
    st, stb = x.clone(), torch.full((M, 192), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.mmpfn_linear_ln_bf16(a.data_ptr(), w.data_ptr(), M, st.data_ptr(), stb.data_ptr(), _stream()),
               "linear_ln")
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(x.double() + a.double() @ w.double().T, (192,), None, None, 1e-5)
    e1 = (st.double() - ref).abs().max().item()
    e2 = (stb.double() - ref).abs().max().item()
    assert not torch.isnan(st).any() and not torch.isnan(stb.float()).any()
    assert e1 < 2e-4 and e2 < 0.03, (e1, e2)        # fp32 accumulation; bf16 rounding of O(4) values


@pytest.mark.parametrize("n_q,n_kv,shared,scale", [(128, 48, 0, 1.0), (333, 1999, 0, 1.0), (300, 2000, 1, 1.0),
                                                   (257, 1000, 0, 4.0), (200, 1500, 1, 8.0), (130, 700, 0, 16.0),
                                                   (1, 1, 0, 1.0), (5, 49, 1, 2.0)])
def test_item_attention_tcgen05(n_q, n_kv, shared, scale):
    """softmax(q k^T / sqrt 32) v across items (layer.py:341-379) on tcgen05 vs torch fp32 on the same bf16
    operands; ragged sizes, the shared head-0 K/V of the test pass (multi_head_attention.py:436-445), and
    score scales at which the running maximum moves often and exponentials overflow against a stale
    reference (scale 16: |score| ~ 1000)."""
    lib = _lib.load()
    B, T = 2, 3
    planes, kv_planes = B * T * 6, (B * T if shared else B * T * 6)
    qpad, kpad = (n_q + 63) // 64 * 64, (n_kv + 63) // 64 * 64
    g = torch.Generator().manual_seed(n_q * 31 + n_kv)
    q = (torch.randn(planes, qpad, 32, generator=g) * scale).cuda().to(torch.bfloat16)
    k = (torch.randn(kv_planes, kpad, 32, generator=g) * scale).cuda().to(torch.bfloat16)
    vt = torch.randn(kv_planes, 32, kpad, generator=g).cuda().to(torch.bfloat16)
    # the pad rows of the K / V^T planes are never fetched (the tensor maps end at n_kv: out-of-bounds zero fill),
    # so the context buffers need no memset: poison them
    k[:, n_kv:] = float("nan")
    vt[:, :, n_kv:] = float("nan")
    out = torch.full((B, n_q, T, 192), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.mmpfn_item_attention_bf16(q.data_ptr(), k.data_ptr(), vt.data_ptr(), B, T, n_q, qpad, n_kv, kpad,
                                             shared, out.data_ptr(), _stream()), "item_attention")
    torch.cuda.synchronize()
    assert not torch.isnan(out.float()).any()
    err = 0.0
    for plane in range(planes):
        bt, h = divmod(plane, 6)
        b, t = divmod(bt, T)
        kp = bt if shared else plane
        ref = torch.softmax(q[plane, :n_q].float() @ k[kp, :n_kv].float().T / 32 ** 0.5, dim=-1) @ vt[kp, :, :n_kv].float().T
        err = max(err, float((out[b, :, t, h * 32:(h + 1) * 32].float() - ref).abs().max()))
    # P is rounded to bf16 (2^-9 relative) before P V, the output to bf16: O(1) values -> ~1e-2 worst case
    assert err < 0.03, err


@pytest.mark.parametrize("B,S,T,n_proj", [(1, 128, 3, 3), (2, 333, 5, 3), (1, 2000, 2, 3), (2, 300, 4, 1), (1, 1, 2, 3)])
def test_item_qkv_scatter_tcgen05(B, S, T, n_proj):
    """QKV projection across items + scatter into the attention kernel's plane layouts (q/k row-major,
    v transposed, head-0 context copies) vs torch on the same bf16 operands."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(B * 1000 + S + T)
    x = torch.randn(B, S, T, 192, generator=g).cuda().to(torch.bfloat16)
    w = (torch.randn(n_proj * 192, 192, generator=g) / 192 ** 0.5).cuda().to(torch.bfloat16)
    Sp = (S + 63) // 64 * 64
    P = B * T * 6
    q = torch.zeros(P, Sp, 32, dtype=torch.bfloat16, device="cuda")
    k = torch.zeros(P, Sp, 32, dtype=torch.bfloat16, device="cuda")
    vt = torch.zeros(P, 32, Sp, dtype=torch.bfloat16, device="cuda")
    k0 = torch.zeros(B * T, Sp, 32, dtype=torch.bfloat16, device="cuda")
    vt0 = torch.zeros(B * T, 32, Sp, dtype=torch.bfloat16, device="cuda")
    full = n_proj == 3
    _lib.check(lib.mmpfn_item_qkv_bf16(x.data_ptr(), w.data_ptr(), B, S, T, Sp, n_proj, q.data_ptr(),
                                       k.data_ptr() if full else None, vt.data_ptr() if full else None,
                                       k0.data_ptr() if full else None, vt0.data_ptr() if full else None, _stream()),
               "item_qkv")
    torch.cuda.synchronize()
    ref = (x.double() @ w.double().T).reshape(B, S, T, n_proj, 6, 32)       # [b, s, t, j, h, d]
    rq = ref[:, :, :, 0].permute(0, 2, 3, 1, 4).reshape(P, S, 32)             # [(b t h), s, d]
    assert (q[:, :S].double() - rq).abs().max().item() < 0.04
    assert (q[:, S:] == 0).all()                                              # rows past S are never written
    if full:
        rk = ref[:, :, :, 1].permute(0, 2, 3, 1, 4).reshape(P, S, 32)
        rv = ref[:, :, :, 2].permute(0, 2, 3, 4, 1).reshape(P, 32, S)         # [(b t h), d, s]
        assert (k[:, :S].double() - rk).abs().max().item() < 0.04
        assert (vt[:, :, :S].double() - rv).abs().max().item() < 0.04
        assert (vt[:, :, S:] == 0).all() and (k[:, S:] == 0).all()
        assert torch.equal(k0, k.reshape(B * T, 6, Sp, 32)[:, 0]) and torch.equal(vt0, vt.reshape(B * T, 6, 32, Sp)[:, 0])


@pytest.mark.parametrize("n_rows,T", [(1, 1), (7, 3), (300, 20), (515, 27), (64, 42), (33, 90), (9, 127)])
def test_feature_attention_bf16(n_rows, T):
    """softmax(q k^T / sqrt 32) v over the T tokens of every table row, 6 heads (layer.py:332-339), mma.sync kernel
    vs torch fp32 on the same bf16 operands; token counts of every BASELINE config (20/27, 42/90, up to 127)."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(n_rows * 131 + T)
    qkv = torch.randn(n_rows * T, 576, generator=g).cuda().to(torch.bfloat16)
    att = torch.full((n_rows * T, 192), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.mmpfn_feature_attention_bf16(qkv.data_ptr(), att.data_ptr(), n_rows, T, _stream()), "feat_attn")
    torch.cuda.synchronize()
    x = qkv.float().view(n_rows, T, 3, 6, 32)
    q, k, v = (x[:, :, j].permute(0, 2, 1, 3) for j in range(3))              # [rows, h, T, d]
    ref = (torch.softmax(q @ k.transpose(-1, -2) / 32 ** 0.5, dim=-1) @ v).permute(0, 2, 1, 3).reshape(n_rows * T, 192)
    assert not torch.isnan(att.float()).any()
    assert (att.float() - ref).abs().max().item() < 0.03      # P and the output rounded to bf16, O(1) values


@pytest.mark.parametrize("n_rows,T", [(1, 2), (5, 3), (7, 16), (301, 20), (2000, 27), (333, 32), (9200, 27), (100, 33), (640, 42), (77, 50),
                                      (9, 64)])
def test_feature_qkv_attention_fused(n_rows, T):
    """QKV projection + feature attention in one kernel (csrc/kernels_featfused.cu) against the two-kernel form
    (persistent tcgen05 projection, then the mma.sync attention) on the same operands: the same MMAs in the same
    order and the same attention core, so the outputs must be EQUAL; pad rows of the destination stay untouched."""
    lib = _lib.load()
    g = torch.Generator().manual_seed(n_rows * 7 + T)
    M = n_rows * T
    x = torch.randn(M, 192, generator=g).cuda().to(torch.bfloat16)
    w = (torch.randn(576, 192, generator=g) * 0.1).cuda().to(torch.bfloat16)
    qkv = torch.empty(M, 576, dtype=torch.bfloat16, device="cuda")
    ref = torch.empty(M, 192, dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.mmpfn_linear_bf16(x.data_ptr(), w.data_ptr(), M, 576, 192, 0, qkv.data_ptr(), _stream()), "linear")
    _lib.check(lib.mmpfn_feature_attention_bf16(qkv.data_ptr(), ref.data_ptr(), n_rows, T, _stream()), "feat_attn")
    got = torch.full((M + 3, 192), float("nan"), dtype=torch.bfloat16, device="cuda")
    _lib.check(lib.mmpfn_feature_qkv_attention_bf16(x.data_ptr(), w.data_ptr(), n_rows, T, got.data_ptr(), _stream()), "fused")
    torch.cuda.synchronize()
    assert torch.isnan(got[M:].float()).all()
    assert not torch.isnan(got[:M].float()).any()
    assert torch.equal(got[:M], ref), float((got[:M].float() - ref.float()).abs().max())


def test_feature_qkv_attention_fused_rejects_wide_rows():
    lib = _lib.load()
    x = torch.zeros(130, 192, dtype=torch.bfloat16, device="cuda")
    w = torch.zeros(576, 192, dtype=torch.bfloat16, device="cuda")
    out = torch.zeros(130, 192, dtype=torch.bfloat16, device="cuda")
    assert lib.mmpfn_feature_qkv_attention_bf16(x.data_ptr(), w.data_ptr(), 2, 65, out.data_ptr(), _stream()) == -4      # MMPFN_EUNSUPPORTED


@pytest.mark.parametrize("mgm,cap,rows,n_tok", [(2, 4, 77, 1), (8, 8, 300, 2), (64, 24, 130, 1)])
def test_image_stem_bf16_vs_fp32(mgm, cap, rows, n_tok):
    """MGM + CAP stem (transformer.py:33-88): the bf16 mode (gated projection on tcgen05, bf16 operands) against the
    fp32 mode of the same library (FFMA, itself held to 2e-5 of the reference by test_stem_state_vs_golden), at the
    default head counts and at the authors' 64 / 24 geometry (CAP head_dim 8)."""
    from multimodalpfn_b200.model import B200PerFeatureTransformer
    geom = Geometry(nlayers=1, mgm_heads=mgm, cap_heads=cap)
    sd = make_state_dict(geom, seed=4)
    img = torch.randn(rows, n_tok, 768, generator=torch.Generator().manual_seed(rows)).cuda()
    a = B200PerFeatureTransformer(sd, geom, precision="fp32").stem_image(img)
    b = B200PerFeatureTransformer(sd, geom, precision="bf16").stem_image(img)
    assert tuple(a.shape) == (rows, cap, 192) and torch.isfinite(b).all()
    err = float((a - b).abs().max())
    # below 32 MGM heads both modes take the FFMA path (identical); above, bf16 operand rounding and nothing else
    assert (err == 0.0) if mgm < 32 else (0 < err < 0.03 * max(1.0, float(a.abs().max()))), err


def _one_layer_model(precision, seed=3):
    from multimodalpfn_b200.model import B200PerFeatureTransformer
    geom = Geometry(nlayers=1, mgm_heads=2, cap_heads=4)
    sd = make_state_dict(geom, seed=seed)
    return B200PerFeatureTransformer(sd, geom, precision=precision), sd, geom


@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("bf16", 0.06)])
@pytest.mark.parametrize("B,S,T,n_test", [(1, 200, 7, 60), (2, 333, 12, 130), (1, 1100, 5, 257), (1, 40, 120, 9),
                                          (1, 24, 200, 7)])
def test_single_layer_pass_vs_oracle(precision, tol, B, S, T, n_test):
    """The train pass (writes the K/V context) then the test pass on random O(1) states vs the
    oracle's layer_forward (layer.py:272-457).  T = 120 and 200: the fp32 feature attention past 48 KB of shared
    memory (its opt-in starts at 120 tokens); the bf16 pass takes the CUDA-core feature attention above 192."""
    from oracle import forward_ref as R
    model, sd, geom = _one_layer_model(precision)
    tsd = R.as_torch_state_dict(sd)
    g = torch.Generator().manual_seed(B * 100 + S + T)
    tr = torch.randn(B, S, T, 192, generator=g)
    te = torch.randn(B, n_test, T, 192, generator=g)
    st = tr.cuda().contiguous()
    stb = st.to(torch.bfloat16) if precision == "bf16" else None
    kv = model.alloc_kv(B, S, T)
    model.layers(st, stb, [(B, T)], S, [kv])
    se = te.cuda().contiguous()
    seb = se.to(torch.bfloat16) if precision == "bf16" else None
    model.layers(se, seb, [(B, T)], n_test, [kv], n_train=S)
    torch.cuda.synchronize()
    for b in range(B):
        ref_tr, kvr = R.layer_forward(tr[b], S, tsd, 0, want_kv=True)
        ref_te, _ = R.layer_forward(te[b], 0, tsd, 0, kv_in=kvr)
        e1 = (st[b].cpu() - ref_tr).abs().max().item()
        e2 = (se[b].cpu() - ref_te).abs().max().item()
        assert e1 < tol and e2 < tol, (e1, e2)
        if precision == "bf16":
            assert (stb[b].float().cpu() - ref_tr).abs().max().item() < tol + 0.03


@pytest.mark.parametrize("seed", list(range(10)))
def test_single_layer_pass_random_shapes(seed):
    """Train + test pass at random ragged shapes (1-700 rows, 2-140 tokens, 1-3 estimators): tiles
    that are mostly padding, key sets shorter than one 48-key tile, token counts that switch the feature
    attention between its register-tile sizes — bf16 path vs the oracle's layer_forward."""
    from oracle import forward_ref as R
    rng = np.random.default_rng(1000 + seed)
    B = int(rng.integers(1, 4))
    S = int(rng.choice([1, 2, 37, 47, 48, 49, 127, 128, 129, 300, 511, 700]))
    T = int(rng.choice([2, 3, 9, 16, 17, 33, 65, 100, 140]))
    n_test = int(rng.choice([1, 5, 44, 128, 131, 300]))
    if B * S * T > 60000:
        B = 1
    model, sd, geom = _one_layer_model("bf16", seed=seed)
    tsd = R.as_torch_state_dict(sd)
    g = torch.Generator().manual_seed(seed)
    tr = torch.randn(B, S, T, 192, generator=g)
    te = torch.randn(B, n_test, T, 192, generator=g)
    st, se = tr.cuda().contiguous(), te.cuda().contiguous()
    stb, seb = st.to(torch.bfloat16), se.to(torch.bfloat16)
    kv = model.alloc_kv(B, S, T)
    model.layers(st, stb, [(B, T)], S, [kv])
    model.layers(se, seb, [(B, T)], n_test, [kv], n_train=S)
    torch.cuda.synchronize()
    assert torch.isfinite(st).all() and torch.isfinite(se).all()
    for b in range(B):
        ref_tr, kvr = R.layer_forward(tr[b], S, tsd, 0, want_kv=True)
        ref_te, _ = R.layer_forward(te[b], 0, tsd, 0, kv_in=kvr)
        e1 = (st[b].cpu() - ref_tr).abs().max().item()
        e2 = (se[b].cpu() - ref_te).abs().max().item()
        assert e1 < 0.06 and e2 < 0.06, (B, S, T, n_test, e1, e2)
        assert (stb[b].float().cpu() - ref_tr).abs().max().item() < 0.09


def test_layer_kernels_on_two_streams():
    """Every pair of layer kernels, and layer-like chains of six launches, on two streams at once (buffers of their
    own) against the same kernels run alone: bit-identical.  Regression test of the residual-ring release order of
    the LayerNorm epilogues (csrc/kernels_mlp.cu, kernels_rowgemm.cu): released before the ld.shared data had
    arrived, a few rows per launch went wrong under a co-running load — never alone."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "concurrency_probe.py")], capture_output=True,
                         text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "pairs that differ: []" in out.stdout, out.stdout[-3000:]
    assert "DIFFERS" not in out.stdout, out.stdout[-3000:]
    assert "chains of six launches per stream" in out.stdout
