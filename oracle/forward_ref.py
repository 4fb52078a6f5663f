"""ORACLE (test infrastructure, never shipped): CPU restatement of the MMPFN in-context forward.

This file is the checker for the CUDA path.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import it; the product package
``multimodalpfn_b200`` never does.

It restates, in plain fp32 torch on the CPU, what the reference computes between
``InferenceEngineCachePreprocessing.iter_outputs`` (reference ``inference.py:343-348``) and the
probability tail of ``MMPFNClassifier.predict_proba`` (``classifier.py:544-576``), from the
weights alone.  It is PINNED: ``oracle/make_golden.py`` runs the real reference
(``/root/reference``) on seeded inputs and stores its outputs under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks this restatement against those vectors.

Every function cites the reference lines it follows (paths relative to
``/root/reference/mmpfn/models/mmpfn/``).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

LN_EPS = 1e-5


def as_torch_state_dict(sd):
    return {k: torch.as_tensor(v, dtype=torch.float32) for k, v in sd.items()}


# ---------------------------------------------------------------------------------------------
# helpers: NaN-aware statistics (model/encoders.py:17-50)
# ---------------------------------------------------------------------------------------------
def _nanmean_clip(x):
    """encoders.py:17-34 (`torch_nanmean`): sum of non-NaN / max(count, 1)."""
    m = torch.isnan(x)
    num = (~m).sum(0).to(x.dtype)
    val = torch.where(m, torch.zeros_like(x), x).sum(0)
    return val / num.clip(min=1.0)


def _nanstd(x):
    """encoders.py:37-50 (`torch_nanstd`): unbiased, NaN ignored, mean = sum/count."""
    m = torch.isnan(x)
    num = (~m).sum(0).to(x.dtype)
    val = torch.where(m, torch.zeros_like(x), x).sum(0)
    mean = val / num
    return torch.sqrt(torch.nansum(torch.square(mean[None] - x), dim=0) / (num - 1))


# ---------------------------------------------------------------------------------------------
# tabular stem (a2) — model/loading.py:308-371 builds the step list
# ---------------------------------------------------------------------------------------------
def stem_tab_fit(xg, n_train, *, n_sigma=12.0):
    """Statistics the x-stem keeps between a train call and a test call.

    xg: [S, G, fpg] raw grouped features (NaN allowed).  Returns a dict.
    The "constant column" tests look at ALL rows given (encoders.py:515, :615); the other
    statistics use the first n_train rows (encoders.py:461, :710).
    n_sigma None or inf: no outlier step (InferenceConfig.remove_outliers False, model/config.py:43, leaves it
    out of the step list, model/loading.py:308-371); the bounds are -inf / +inf, which the soft clip passes through.
    """
    S = xg.shape[0]
    sel = (xg[1:] == xg[0]).sum(0) != (S - 1)                       # encoders.py:515
    xc = _compact(xg, sel)
    fill = torch.nanmean(xc[:n_train], dim=0)                       # encoders.py:461
    x1 = _nan_fill(xc, fill)
    d = x1[:n_train]
    if n_sigma is None or math.isinf(n_sigma):
        # inf * sd would give NaN bounds wherever sd is 0 or NaN (a constant column, n_train == 1)
        lo, hi = torch.full_like(fill, -math.inf), torch.full_like(fill, math.inf)
    else:
        mu, sd_ = _nanmean_clip(d), _nanstd(d)                      # encoders.py:148-150
        lo, hi = mu - n_sigma * sd_, mu + n_sigma * sd_
        d2 = d.clone()
        d2[torch.logical_or(d2 > hi, d2 < lo)] = float("nan")       # encoders.py:152
        mu, sd_ = _nanmean_clip(d2), _nanstd(d2)
        lo, hi = mu - n_sigma * sd_, mu + n_sigma * sd_             # encoders.py:157-158
    x2 = _soft_clip(x1, lo, hi)
    mean = _nanmean_clip(x2[:n_train])                              # encoders.py:81-82
    std = _nanstd(x2[:n_train]) + 1e-20
    if n_train == 1:
        std = torch.ones_like(std)                                  # encoders.py:87-88
    x3 = torch.clip((x2 - mean) / std, -100, 100)
    sel2 = (x3[1:] == x3[0]).sum(0) != (S - 1)                      # encoders.py:615
    used = sel2.sum(-1).clip(min=1)                                 # encoders.py:616-619
    return dict(sel=sel, fill=fill, lo=lo, hi=hi, mean=mean, std=std, used=used)


def _compact(xg, sel):
    """encoders.py:102-130 (`select_features`): kept features first, zeros after, per group.
    (With a single group the reference shrinks the feature axis instead and re-pads it at
    encoders.py:648-654; the values are the same.)"""
    out = torch.zeros_like(xg)
    for g in range(xg.shape[1]):
        kept = xg[:, g, sel[g]]
        out[:, g, : kept.shape[1]] = kept
    return out


def _nan_fill(x, fill):
    bad = torch.logical_or(torch.isnan(x), torch.isinf(x))          # encoders.py:488-491
    return torch.where(bad, fill[None].expand_as(x), x)


def _soft_clip(x, lo, hi):
    x = torch.maximum(-torch.log(1 + torch.abs(x)) + lo, x)         # encoders.py:160
    return torch.minimum(torch.log(1 + torch.abs(x)) + hi, x)      # encoders.py:161


def stem_tab_apply(xg, st, w_enc):
    """Transform rows with fitted statistics and embed: [S,G,fpg] -> [S,G,E]."""
    fpg = xg.shape[-1]
    xc = _compact(xg, st["sel"])
    ind = (torch.isnan(xc) * -2.0
           + torch.logical_and(torch.isinf(xc), xc > 0) * 2.0
           + torch.logical_and(torch.isinf(xc), xc < 0) * 4.0).to(xc.dtype)   # encoders.py:480-486
    x1 = _nan_fill(xc, st["fill"])
    x2 = _soft_clip(x1, st["lo"], st["hi"])
    x3 = torch.clip((x2 - st["mean"]) / st["std"], -100, 100)       # encoders.py:92-95
    x4 = x3 * torch.sqrt(fpg / st["used"].to(x3.dtype))[None, :, None]   # encoders.py:639-644
    return torch.cat([x4, ind], dim=-1) @ w_enc.T                   # encoders.py:422-425


def group_features(X, fpg):
    """transformer.py:630-657: zero-pad F' to a multiple of fpg, reshape to [S,G,fpg]."""
    S, Fp = X.shape
    pad = (-Fp) % fpg
    if pad:
        X = torch.cat([X, torch.zeros(S, pad, dtype=X.dtype)], dim=1)
    return X.reshape(S, -1, fpg)


# ---------------------------------------------------------------------------------------------
# y stem (a3) — model/loading.py:374-398, encoders.py:453-493, :949-974
# ---------------------------------------------------------------------------------------------
def y_encoder_weights(sd):
    """(weight, bias, regression): the classification y-encoder is NaN handling -> class rank -> Linear (step 2),
    the regression one has no rank step, so its Linear is step 1 (model/loading.py:374-398)."""
    if "y_encoder.2.layer.weight" in sd:
        return sd["y_encoder.2.layer.weight"], sd["y_encoder.2.layer.bias"], False
    return sd["y_encoder.1.layer.weight"], sd["y_encoder.1.layer.bias"], True


def stem_y(y_train, n_rows, w_y, b_y, regression=False):
    """[Ntr] labels -> [n_rows, E]; rows past Ntr are the NaN-padded test rows
    (transformer.py:682-718)."""
    n_tr = y_train.shape[0]
    yy = torch.cat([y_train.to(torch.float32), torch.full((n_rows - n_tr,), float("nan"))])
    return stem_y_apply(yy, stem_y_fit(y_train), w_y, b_y, regression)


def stem_y_fit(y_train):
    y_train = y_train.to(torch.float32)
    return dict(mean=torch.nanmean(y_train), uniq=torch.unique(y_train))


def stem_y_apply(yy, st, w_y, b_y, regression=False):
    ind = torch.isnan(yy) * -2.0
    yy = torch.where(torch.isnan(yy), st["mean"], yy)
    if not regression:
        yy = (yy[:, None] > st["uniq"][None]).sum(-1).to(yy.dtype)         # class rank, encoders.py:961-964
    return torch.stack([yy, ind.to(yy.dtype)], dim=-1) @ w_y.T + b_y


# ---------------------------------------------------------------------------------------------
# image / text stem (a4-a6)
# ---------------------------------------------------------------------------------------------
def stem_image(img, sd, geom):
    """[S, n_tok, 768] -> [S, H_img, E].  transformer.py:33-48 (MGM), :60-88 (CAP),
    :91-128 (MoE)."""
    E = geom.emsize
    if geom.mixer_type == "MoE":
        x = img[:, 0]                                               # transformer.py:109
        gate = F.softmax(x @ sd["moe.gate.weight"].T + sd["moe.gate.bias"], dim=-1)
        n_exp = geom.mgm_heads
        top_k = max(geom.mgm_heads, geom.cap_heads or 0)            # transformer.py:301
        if top_k < n_exp:                                           # never true, kept for fidelity
            _, idx = torch.topk(gate, top_k, dim=-1)
            mask = torch.zeros_like(gate).scatter_(1, idx, 1.0)
            gate = gate * mask
            gate = gate / (gate.sum(-1, keepdim=True) + 1e-9)
        outs = []
        for h in range(n_exp):
            p = f"moe.experts.{h}."
            t = F.layer_norm(x, (x.shape[-1],), sd[p + "0.weight"], sd[p + "0.bias"], LN_EPS)
            t = F.gelu(t @ sd[p + "1.weight"].T + sd[p + "1.bias"])
            t = t @ sd[p + "4.weight"].T + sd[p + "4.bias"]
            outs.append(gate[:, h:h + 1] * t)
        return torch.stack(outs, dim=1)
    outs = []
    for h in range(geom.mgm_heads):
        p = f"mgm.projs.{h}."
        t = F.layer_norm(img, (img.shape[-1],), sd[p + "0.weight"], sd[p + "0.bias"], LN_EPS)
        t = t @ sd[p + "1.weight"].T + sd[p + "1.bias"]
        half = t.shape[-1] // 2
        t = t[..., :half] * torch.sigmoid(t[..., half:])            # nn.GLU
        outs.append(t @ sd[p + "4.weight"].T + sd[p + "4.bias"])
    src = torch.cat(outs, dim=-2)                                   # head-major on the token axis
    if geom.mixer_type == "MGM":
        return src
    # --- CAP ---
    C = geom.cap_heads
    hd = E // C
    src = F.layer_norm(src, (E,), sd["cap.k_norm.weight"], sd["cap.k_norm.bias"], LN_EPS)
    q0 = F.layer_norm(sd["cap.queries"], (E,), sd["cap.q_norm.weight"], sd["cap.q_norm.bias"], LN_EPS)
    q0 = q0 @ sd["cap.q_proj.weight"].T
    Wi, bi = sd["cap.mha.in_proj_weight"], sd["cap.mha.in_proj_bias"]
    q = q0 @ Wi[:E].T + bi[:E]                                      # [C, E]
    k = src @ Wi[E:2 * E].T + bi[E:2 * E]                           # [S, n_kv, E]
    v = src @ Wi[2 * E:].T + bi[2 * E:]
    S, n_kv, _ = k.shape
    qh = q.reshape(C, C, hd).permute(1, 0, 2)                       # [head, query, hd]
    kh = k.reshape(S, n_kv, C, hd).permute(0, 2, 1, 3)              # [S, head, n_kv, hd]
    vh = v.reshape(S, n_kv, C, hd).permute(0, 2, 1, 3)
    att = torch.softmax(torch.einsum("hqd,shkd->shqk", qh, kh) / math.sqrt(hd), dim=-1)
    o = torch.einsum("shqk,shkd->shqd", att, vh).permute(0, 2, 1, 3).reshape(S, C, E)
    o = o @ sd["cap.mha.out_proj.weight"].T + sd["cap.mha.out_proj.bias"]
    ffn = F.gelu(o @ sd["cap.ffn.0.weight"].T + sd["cap.ffn.0.bias"])
    ffn = ffn @ sd["cap.ffn.3.weight"].T + sd["cap.ffn.3.bias"]
    return F.layer_norm(o, (E,), sd["cap.out_norm.weight"], sd["cap.out_norm.bias"], LN_EPS) + ffn


def positional_embeddings(n_feature_tokens, sd, geom, seed, device="cpu"):
    """transformer.py:421-424, :925-933: fresh generator per forward, seeded iff seed != 0;
    randn((T-1, E//4)) in fp32 then the 48->192 linear."""
    gen = torch.Generator(device=device)
    if seed:
        gen.manual_seed(seed)
    z = torch.randn((n_feature_tokens, geom.emsize // 4), generator=gen, device=device,
                    dtype=torch.float32).cpu()
    return (z @ sd["feature_positional_embedding_embeddings.weight"].T
            + sd["feature_positional_embedding_embeddings.bias"])


# ---------------------------------------------------------------------------------------------
# the 12 layers (a9-a12)
# ---------------------------------------------------------------------------------------------
def _ln(x):
    return F.layer_norm(x, (x.shape[-1],), None, None, LN_EPS)      # layer.py:40-64, no affine


def _attend(q, k, v):
    """q [..., Lq, H, D], k/v [..., Lk, H, D] -> [..., Lq, H, D]; softmax(q k^T / sqrt(D)) v
    (multi_head_attention.py:693-729)."""
    D = q.shape[-1]
    logits = torch.einsum("...qhd,...khd->...hqk", q, k) / math.sqrt(D)
    p = torch.softmax(logits, dim=-1)
    return torch.einsum("...hqk,...khd->...qhd", p, v)


def _attend_chunked(q, k, v, chunk=2048):
    outs = [_attend(q[..., i:i + chunk, :, :], k, v) for i in range(0, q.shape[-3], chunk)]
    return torch.cat(outs, dim=-3)


def layer_forward(state, n_train, sd, l, *, kv_in=None, want_kv=False):
    """One PerFeatureEncoderLayer (layer.py:272-457) on state [S, T, E].

    Rows [:n_train] are train rows (self-attention over items, all heads); rows [n_train:]
    are test rows: their item attention reads head-0 K/V of the train rows
    (layer.py:346-358, multi_head_attention.py:436-445), taken from ``kv_in`` ([T, Ntr, 2, D])
    when given (the reference's cached path, multi_head_attention.py:328-336).
    Returns (state, kv) with kv = head-0 K/V of this layer's train rows if want_kv.
    """
    p = f"transformer_encoder.layers.{l}."
    S, T, E = state.shape
    # --- attention between features (per row) ---
    Wf, Of = sd[p + "self_attn_between_features._w_qkv"], sd[p + "self_attn_between_features._w_out"]
    qkv = torch.einsum("ste,jhde->stjhd", state, Wf)                # multi_head_attention.py:430
    a = _attend(qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2])           # over tokens
    state = _ln(state + torch.einsum("sthd,hde->ste", a, Of))       # :513-517, memory.py:99-100
    # --- attention between items (per token column) ---
    Oi = sd[p + "self_attn_between_items._w_out"]
    if p + "self_attn_between_items._w_qkv" in sd:
        Wi = sd[p + "self_attn_between_items._w_qkv"]
        Wq_test = Wi[0]
    else:
        # two_sets_of_queries checkpoints (multi_head_attention.py:216-260, :418-419): query set 0 for the train
        # rows, set 1 for the test rows (layer.py:357), keys / values from _w_kv
        wq, wkv = sd[p + "self_attn_between_items._w_q"], sd[p + "self_attn_between_items._w_kv"]
        Wi = torch.stack([wq[0], wkv[0], wkv[1]])
        Wq_test = wq[wq.shape[0] - 1]
    xt = state.transpose(0, 1)                                      # [T, S, E]
    tr, te = xt[:, :n_train], xt[:, n_train:]
    outs, kv = [], None
    if n_train > 0:
        qkv = torch.einsum("tse,jhde->tsjhd", tr, Wi)
        outs.append(_attend_chunked(qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]))
        kv0 = qkv[:, :, 1:, 0]                                      # [T, Ntr, 2, D] head 0
        if want_kv:
            kv = kv0.clone()
    else:
        kv0 = kv_in
    if te.shape[1] > 0:
        H = Wi.shape[1]
        q = torch.einsum("tse,hde->tshd", te, Wq_test)
        k0 = kv0[:, :, 0][:, :, None].expand(-1, -1, H, -1)         # all q-heads share head 0
        v0 = kv0[:, :, 1][:, :, None].expand(-1, -1, H, -1)
        outs.append(_attend_chunked(q, k0, v0))
    a = torch.cat(outs, dim=1)                                      # [T, S, H, D]
    xt = xt + torch.einsum("tshd,hde->tse", a, Oi)
    state = _ln(xt.transpose(0, 1))
    # --- MLP (mlp.py:93-104) ---
    h = F.gelu(state @ sd[p + "mlp.linear1.weight"].T)
    state = _ln(state + h @ sd[p + "mlp.linear2.weight"].T)
    return state, kv


def decode(state_y, sd):
    """transformer.py:392-396, :850-853: decoder on the y token of the test rows."""
    h = F.gelu(state_y @ sd["decoder_dict.standard.0.weight"].T + sd["decoder_dict.standard.0.bias"])
    return h @ sd["decoder_dict.standard.2.weight"].T + sd["decoder_dict.standard.2.bias"]


# ---------------------------------------------------------------------------------------------
# whole forward
# ---------------------------------------------------------------------------------------------
def embed_rows(X, img, yy_embedded, tab_stats, embs, sd, geom):
    """Token assembly (transformer.py:740-788): tabular groups, image tokens, + pos-emb on all
    non-y tokens, y token last."""
    toks = []
    if X is not None:
        toks.append(stem_tab_apply(group_features(X, geom.features_per_group), tab_stats,
                                   sd["encoder.5.layer.weight"]))
    if img is not None:
        toks.append(stem_image(img, sd, geom))
    x = torch.cat(toks, dim=1)
    x = x + embs[None]
    return torch.cat([x, yy_embedded[:, None]], dim=1)


def forward_joint(X_full, img_full, y_train, sd, geom, *, seed=0, n_sigma=12.0, return_state=False):
    """Reference `_forward` (transformer.py:555-867) for x [S,F'] / image [S,n_tok,768] /
    y [Ntr] -> logits [Nte, n_out].  X_full or img_full may be None."""
    n_train = y_train.shape[0]
    S = X_full.shape[0] if X_full is not None else img_full.shape[0]
    tab_stats = None
    if X_full is not None:
        tab_stats = stem_tab_fit(group_features(X_full.to(torch.float32), geom.features_per_group),
                                 n_train, n_sigma=n_sigma)
    ey = stem_y(y_train, S, *y_encoder_weights(sd))
    n_feat_tok = (0 if X_full is None else -(-X_full.shape[1] // geom.features_per_group)) + \
        (0 if img_full is None else n_image_tokens(img_full.shape[1], geom))
    embs = positional_embeddings(n_feat_tok, sd, geom, seed)
    state = embed_rows(None if X_full is None else X_full.to(torch.float32), img_full, ey,
                       tab_stats, embs, sd, geom)
    for l in range(geom.nlayers):
        state, _ = layer_forward(state, n_train, sd, l)
    logits = decode(state[n_train:, -1], sd)
    return (logits, state) if return_state else logits


def n_image_tokens(n_tok, geom):
    if geom.mixer_type == "MGM+CAP":
        return geom.cap_heads
    if geom.mixer_type == "MGM":
        return n_tok * geom.mgm_heads
    return geom.mgm_heads  # MoE


def forward_fit_context(X_train, img_train, y_train, sd, geom, *, seed=0, n_sigma=12.0):
    """Cached-context form (the reference's model-level cache path, SURVEY.md gotcha 5 /
    Appendix C 3b): run the train rows once, keep stem statistics, pos-emb and per-layer head-0
    K/V of the item attention."""
    n_train = y_train.shape[0]
    tab_stats = None
    if X_train is not None:
        tab_stats = stem_tab_fit(group_features(X_train.to(torch.float32), geom.features_per_group),
                                 n_train, n_sigma=n_sigma)
    yst = stem_y_fit(y_train)
    ey = stem_y_apply(y_train.to(torch.float32), yst, *y_encoder_weights(sd))
    n_feat_tok = (0 if X_train is None else -(-X_train.shape[1] // geom.features_per_group)) + \
        (0 if img_train is None else n_image_tokens(img_train.shape[1], geom))
    embs = positional_embeddings(n_feat_tok, sd, geom, seed)
    state = embed_rows(None if X_train is None else X_train.to(torch.float32), img_train, ey,
                       tab_stats, embs, sd, geom)
    kvs = []
    for l in range(geom.nlayers):
        state, kv = layer_forward(state, n_train, sd, l, want_kv=True)
        kvs.append(kv)
    return dict(tab_stats=tab_stats, y_stats=yst, embs=embs, kv=kvs, n_train=n_train)


def forward_with_context(X_test, img_test, ctx, sd, geom):
    """Test rows only, against a cached context -> logits [Nte, n_out]."""
    n_te = X_test.shape[0] if X_test is not None else img_test.shape[0]
    ey = stem_y_apply(torch.full((n_te,), float("nan")), ctx["y_stats"], *y_encoder_weights(sd))
    state = embed_rows(None if X_test is None else X_test.to(torch.float32), img_test, ey,
                       ctx["tab_stats"], ctx["embs"], sd, geom)
    for l in range(geom.nlayers):
        state, _ = layer_forward(state, 0, sd, l, kv_in=ctx["kv"][l])
    return decode(state[:, -1], sd)


def proba_tail(logits_list, class_perms, n_classes, *, softmax_temperature=0.9,
               average_before_softmax=False, balance_probabilities=False, class_counts=None):
    """classifier.py:544-576.  logits_list: per-estimator [Nte, n_out]; class_perms: per-estimator
    permutation (or None).  Mirrors the quirk that the [:n_classes] slice only happens when the
    temperature is not 1 (classifier.py:544-547)."""
    outs = []
    for lg, perm in zip(logits_list, class_perms):
        if softmax_temperature != 1:
            lg = lg[:, :n_classes].float() / softmax_temperature
        if perm is not None:
            lg = lg[..., torch.as_tensor(perm, dtype=torch.long)]
        outs.append(lg)
    if average_before_softmax:
        out = torch.softmax(torch.stack(outs).mean(0), dim=1)
    else:
        out = torch.stack([torch.softmax(o, dim=1) for o in outs]).mean(0)
    if balance_probabilities:
        cc = torch.as_tensor(class_counts, dtype=torch.float32)
        out = out * (cc / cc.sum())
        out = out / out.sum(-1, keepdim=True)
    out = out.float().numpy()
    return out / out.sum(axis=1, keepdims=True)
