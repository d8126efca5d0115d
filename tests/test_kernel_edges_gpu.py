"""The engine at the shape edges its kernels dispatch on, against float64 references.

`tests/test_engine_gpu.py` pins the engine at the tuned shapes.  This file runs the branches those shapes never reach:
partial 32-column blocks and one-column n-tiles of the score passes, rows split over several n-tiles per chunk, single
M-tile launches, 9-row fine windows, corner windows of unequal fine grids, and the match wire format on one GPU.
Every comparison is against a float64 restatement of the reference below (`oracle/loftr_oracle.py` rounds every
intermediate to float32, so it stays the reference for the match-list semantics only).  The coarse-matching and
transformer inputs have logits of O(1): a padded row or column that leaked into a normaliser would then move it by far
more than the tolerances (asserted per case).  `test_float64_references_match_float32_oracle` pins the restatements
themselves against the oracle and the golden vectors and runs without a GPU.

Tolerances are the suite's: transformer 2e-4 absolute, `mconf` rtol 1e-3, `conf_matrix` rtol 2e-3, keypoints 1e-3 px at
stage level."""
import math

import numpy as np
import pytest
import torch

import util
import weights as WTS
from cases import CASES, CM_CASES, build_cfg, build_cm_inputs
from oracle import loftr_oracle as O

gpu = pytest.mark.gpu
DEV = "cuda:0"
F64 = np.float64


def _t(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    return t if dtype is None else t.to(dtype)


# ================================================================================================ float64 references
# Restatements of the reference in float64; file:line citations are relative to the reference root, as in the oracle.
def _softmax_f64(x, axis):
    e = np.exp(x - x.max(axis=axis, keepdims=True))
    return e / e.sum(axis=axis, keepdims=True)


def _lse_f64(x, axis):
    m = x.max(axis=axis, keepdims=True)
    return (m + np.log(np.exp(x - m).sum(axis=axis, keepdims=True))).squeeze(axis)


def log_optimal_transport_f64(scores, alpha, iters):
    """third_party/SuperGluePretrainedNetwork/models/superglue.py:141-170 -> log assignment [b, m+1, n+1]."""
    b, m, n = scores.shape
    couplings = np.full((b, m + 1, n + 1), float(alpha), F64)                  # :156-160
    couplings[:, :m, :n] = scores
    norm = -math.log(m + n)                                                    # :162
    log_mu = np.concatenate([np.full(m, norm), [math.log(n) + norm]])          # :163
    log_nu = np.concatenate([np.full(n, norm), [math.log(m) + norm]])          # :164
    u, v = np.zeros((b, m + 1)), np.zeros((b, n + 1))
    for _ in range(iters):                                                     # :144-148
        u = log_mu[None] - _lse_f64(couplings + v[:, None, :], 2)
        v = log_nu[None] - _lse_f64(couplings + u[:, :, None], 1)
    return couplings + u[:, :, None] + v[:, None, :] - norm                    # :148,169


def similarity_f64(f0, f1, cfg, m0=None, m1=None):
    """The masked similarity CoarseMatching.forward normalises (coarse_matching.py:103-125).  m0/m1: bool [N,L]/[N,S]."""
    c = f0.shape[-1]
    sim = (f0.astype(F64) / math.sqrt(c)) @ (f1.astype(F64) / math.sqrt(c)).transpose(0, 2, 1)   # :106-109, :119
    if cfg["match_type"] == "dual_softmax":
        sim = sim / cfg["dsmax_temperature"]                                   # :110
    if m0 is not None:
        sim[~(m0[:, :, None] & m1[:, None, :])] = -1e9                         # :111-114, :122-125
    return sim


def conf_matrix_f64(f0, f1, cfg, m0=None, m1=None, bin_score=None):
    """CoarseMatching.forward up to conf_matrix (coarse_matching.py:103-143) in float64."""
    sim = similarity_f64(f0, f1, cfg, m0, m1)
    if cfg["match_type"] == "dual_softmax":
        return _softmax_f64(sim, 1) * _softmax_f64(sim, 2)                    # :115
    assign = np.exp(log_optimal_transport_f64(sim, bin_score, cfg["skh_iters"]))   # :126-128
    conf = assign[:, :-1, :-1].copy()
    if cfg.get("skh_prefilter", False):                                        # :132-136
        L, S = conf.shape[1:]
        conf[np.broadcast_to((assign.argmax(axis=2) == S)[:, :-1, None], conf.shape)] = 0
        conf[np.broadcast_to((assign.argmax(axis=1) == L)[:, None, :-1], conf.shape)] = 0
    return conf


def top2_f64(conf):
    """The two largest confidences of every row and every column (the near-tie statistics of util.compare_matches)."""
    row = -np.sort(-conf, axis=2)[:, :, :2]
    col = -np.sort(-conf, axis=1)[:, :2, :].transpose(0, 2, 1)
    return {"row_top2_f64": row, "col_top2_f64": col}


def _elu1(x):
    return np.where(x > 0, x, np.expm1(np.minimum(x, 0))) + 1.0                # linear_attention.py:10-11


def linear_attention_f64(q, k, v, q_mask=None, kv_mask=None, eps=1e-6):
    """LinearAttention.forward (linear_attention.py:20-47).  q [N,L,H,D], k/v [N,S,H,D]."""
    Q, K = _elu1(q), _elu1(k)
    if q_mask is not None:
        Q = Q * q_mask[:, :, None, None]
    if kv_mask is not None:
        K = K * kv_mask[:, :, None, None]
        v = v * kv_mask[:, :, None, None]
    s = v.shape[1]
    v = v / s                                                                  # :41-42
    KV = np.einsum("nshd,nshv->nhdv", K, v)                                    # :43
    Z = 1.0 / (np.einsum("nlhd,nhd->nlh", Q, K.sum(axis=1)) + eps)             # :44
    return np.einsum("nlhd,nhdv->nlhv", Q, KV) * Z[..., None] * s              # :45


def layer_norm_f64(x, g, b, eps=1e-5):
    mu = x.mean(axis=-1, keepdims=True)
    d = x - mu
    return d / np.sqrt((d * d).mean(axis=-1, keepdims=True) + eps) * g + b


def encoder_layer_f64(x, source, w, nhead, x_mask=None, source_mask=None):
    """LoFTREncoderLayer.forward (transformer.py:35-58)."""
    w = {k: v.astype(F64) for k, v in w.items()}
    bs, _, c = x.shape
    q = (x @ w["q_proj.weight"].T).reshape(bs, -1, nhead, c // nhead)           # :47
    k = (source @ w["k_proj.weight"].T).reshape(bs, -1, nhead, c // nhead)      # :48
    v = (source @ w["v_proj.weight"].T).reshape(bs, -1, nhead, c // nhead)      # :49
    msg = linear_attention_f64(q, k, v, x_mask, source_mask).reshape(bs, -1, c) @ w["merge.weight"].T   # :50-51
    msg = layer_norm_f64(msg, w["norm1.weight"], w["norm1.bias"])             # :52
    h = np.maximum(np.concatenate([x, msg], axis=2) @ w["mlp.0.weight"].T, 0)  # :55
    msg = layer_norm_f64(h @ w["mlp.2.weight"].T, w["norm2.weight"], w["norm2.bias"])   # :56
    return x + msg                                                             # :58


def transformer_f64(feat0, feat1, layers, layer_names, nhead, mask0=None, mask1=None):
    """LocalFeatureTransformer.forward (transformer.py:80-101); a cross layer's feat1 sees the new feat0 (:96-97)."""
    feat0, feat1 = feat0.astype(F64), feat1.astype(F64)
    for w, name in zip(layers, layer_names):
        if name == "self":
            feat0 = encoder_layer_f64(feat0, feat0, w, nhead, mask0, mask0)
            feat1 = encoder_layer_f64(feat1, feat1, w, nhead, mask1, mask1)
        else:
            feat0 = encoder_layer_f64(feat0, feat1, w, nhead, mask0, mask1)
            feat1 = encoder_layer_f64(feat1, feat0, w, nhead, mask1, mask0)
    return feat0, feat1


def gather_windows_f64(feat_f, b_ids, idx, wc, W, stride):
    """F.unfold(kernel=W, stride, padding=W//2)[b_ids, idx] (fine_preprocess.py:40-47) as a direct gather:
    win[m, ky*W+kx, c] = feat_f[b, c, stride*y - W//2 + ky, stride*x - W//2 + kx], zero outside the map."""
    _, c, hf, wf = feat_f.shape
    out = np.zeros((len(b_ids), W * W, c), F64)
    cy, cx = idx // wc, idx % wc
    for ky in range(W):
        for kx in range(W):
            y, x = stride * cy - W // 2 + ky, stride * cx - W // 2 + kx
            ok = (y >= 0) & (y < hf) & (x >= 0) & (x < wf)
            out[ok, ky * W + kx] = feat_f[b_ids[ok], :, y[ok], x[ok]]
    return out


def fine_preprocess_f64(feat_f0, feat_f1, feat_c0, feat_c1, b_ids, i_ids, j_ids, w0c, w1c, W, stride, w):
    """FinePreprocess.forward with fine_concat_coarse_feat=True (fine_preprocess.py:29-59)."""
    w = {k: v.astype(F64) for k, v in w.items()}
    win = np.concatenate([gather_windows_f64(feat_f0, b_ids, i_ids, w0c, W, stride),
                          gather_windows_f64(feat_f1, b_ids, j_ids, w1c, W, stride)], 0)
    fc = np.concatenate([feat_c0[b_ids, i_ids], feat_c1[b_ids, j_ids]], 0).astype(F64)   # :50-51
    c_win = fc @ w["down_proj.weight"].T + w["down_proj.bias"]
    cat = np.concatenate([win, np.repeat(c_win[:, None, :], W * W, axis=1)], -1)         # :52-55
    merged = cat @ w["merge_feat.weight"].T + w["merge_feat.bias"]
    m = len(b_ids)
    return merged[:m], merged[m:]                                                         # :56


def fine_matching_f64(f0, f1, mkpts1_c, b_ids, scale, scale1=None):
    """FineMatching.forward + get_fine_match (fine_matching.py:15-74): softmax heat map of the window-0 centre against
    window 1, expectation and std over the normalised grid linspace(-1, 1, W)^2 (x along the window's second axis)."""
    m, ww, c = f0.shape
    W = int(round(math.sqrt(ww)))
    f0, f1 = f0.astype(F64), f1.astype(F64)
    sim = np.einsum("mc,mrc->mr", f0[:, ww // 2], f1)                         # :43-44
    heat = _softmax_f64(sim / math.sqrt(c), 1)                                 # :45-46
    lin = np.linspace(-1, 1, W)
    grid = np.stack([np.tile(lin, W), np.repeat(lin, W)], -1)                  # [WW, 2]  :50
    coords = heat @ grid                                                       # :49
    var = heat @ grid ** 2 - coords ** 2                                       # :53
    std = np.sqrt(np.clip(var, 1e-10, None)).sum(-1)                           # :54
    s1 = scale * scale1[b_ids].astype(F64) if scale1 is not None else scale    # :68
    return np.concatenate([coords, std[:, None]], -1), mkpts1_c + coords * (W // 2) * s1   # :57, :69


# ------------------------------------------------------------------------------------------------ shared helpers
def _layer_weights(tf):
    sd = {k: v.detach().cpu().numpy() for k, v in tf.state_dict().items()}
    return O.split_layers({"x." + k: v for k, v in sd.items()}, "x", len(tf.layers))


def _model(W=5, device="cpu"):
    """LoFTR with the deterministic weights of tests/golden/weights.py and fine window size W."""
    import loftr_b200
    cfg = build_cfg(CASES[0])
    cfg["fine_window_size"] = W
    model = loftr_b200.LoFTR(cfg).eval()
    state = WTS.make_state({k: tuple(v.shape) for k, v in model.state_dict().items()}, seed=0)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in state.items()})
    return model.to(device), cfg, state


def _grid_masks(n, hw, valid):
    m = np.zeros((n, *hw), bool)
    for b, (vh, vw) in enumerate(valid):
        m[b, :vh, :vw] = True
    return m


def _cm_cfg(case):
    cfg = build_cfg({"thr": 0.0, "border_rm": case.get("border_rm", 2), "match_type": case.get("match_type", "dual_softmax"),
                     "prefilter": case.get("prefilter", False)})["match_coarse"]
    cfg["skh_iters"] = case.get("skh_iters", 3)
    return cfg


# ================================================================================================ CPU: pin the references
def test_float64_references_match_float32_oracle():
    """Each float64 restatement above agrees with the float32 oracle (and with the reference's golden vectors) to
    float32 precision, so the GPU tests below compare against the reference and not against a private variant."""
    rs = np.random.RandomState(17)
    # coarse confidence: dual-softmax / Sinkhorn (+prefilter), masked and unmasked, against the oracle
    for mt, pf, masked in (("dual_softmax", False, False), ("dual_softmax", False, True), ("sinkhorn", False, False),
                           ("sinkhorn", True, True)):
        cfg = _cm_cfg({"match_type": mt, "prefilter": pf, "skh_iters": 3})
        f0 = (rs.standard_normal((2, 35, 256)) * 1.5).astype(np.float32)
        f1 = (rs.standard_normal((2, 40, 256)) * 1.5).astype(np.float32)
        f1[:, :30] = f0[:, 5:] + 0.3 * rs.standard_normal((2, 30, 256)).astype(np.float32)
        m0 = _grid_masks(2, (5, 7), [(5, 6), (4, 7)]).reshape(2, -1) if masked else None
        m1 = _grid_masks(2, (5, 8), [(4, 8), (5, 5)]).reshape(2, -1) if masked else None
        ref, _ = O.coarse_conf_matrix(f0, f1, cfg, m0, m1, bin_score=0.5)
        got = conf_matrix_f64(f0, f1, cfg, m0, m1, bin_score=0.5)
        np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-9, err_msg=f"{mt} prefilter={pf} masked={masked}")
        if mt == "dual_softmax":   # the near-tie statistics agree with util.near_tie_top2_f64 (also float64)
            t2 = top2_f64(got)
            for b in range(2):
                r, c = util.near_tie_top2_f64(f0[b], f1[b], cfg, None if m0 is None else m0[b],
                                              None if m1 is None else m1[b])
                np.testing.assert_allclose(t2["row_top2_f64"][b], r, rtol=1e-7, atol=1e-300)
                np.testing.assert_allclose(t2["col_top2_f64"][b], c, rtol=1e-7, atol=1e-300)
    # ... and against the reference's own conf_matrix (golden vectors of the stage-level cases)
    for case in CM_CASES:
        gold = util.load_golden(case["name"])
        inp = build_cm_inputs(case)
        cfg = build_cfg(case)["match_coarse"]
        m0 = inp["mask0"].reshape(case["n"], -1) if "mask0" in inp else None
        m1 = inp["mask1"].reshape(case["n"], -1) if "mask1" in inp else None
        got = conf_matrix_f64(inp["feat_c0"], inp["feat_c1"], cfg, m0, m1, case.get("bin_score", 1.0))
        ref = gold["conf_matrix"]
        if m0 is not None:   # fully padded cells: 1/(L*S) in the reference, 0 in the engine; not compared anywhere
            valid = m0[:, :, None] | m1[:, None, :]
            got, ref = got * valid, ref * valid
        np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-9, err_msg=case["name"])
    # transformer, masked (including an all-False source mask and a single valid source row)
    model, cfg, state = _model()
    for prefix, c, nl, (n, l, s) in (("loftr_coarse", 256, 8, (3, 11, 9)), ("loftr_fine", 128, 2, (4, 9, 9))):
        layers = O.split_layers(state, prefix, nl)
        names = cfg["coarse" if c == 256 else "fine"]["layer_names"]
        f0 = (rs.standard_normal((n, l, c)) * 0.5).astype(np.float32)
        f1 = (rs.standard_normal((n, s, c)) * 0.5).astype(np.float32)
        m0 = rs.uniform(size=(n, l)) > 0.3
        m1 = rs.uniform(size=(n, s)) > 0.3
        m1[0], m1[1], m1[1, 4] = False, False, True
        for mm0, mm1 in ((None, None), (m0, m1)):
            r0, r1 = O.local_feature_transformer(f0, f1, layers, names, 8, mm0, mm1)
            g0, g1 = transformer_f64(f0, f1, layers, names, 8, mm0, mm1)
            np.testing.assert_allclose(g0, r0, atol=2e-5, err_msg=prefix)
            np.testing.assert_allclose(g1, r1, atol=2e-5, err_msg=prefix)
    # fine level at W = 3 and 5 on unequal grids, with and without scale1
    fw = {k: state[f"fine_preprocess.{k}"] for k in ["down_proj.weight", "down_proj.bias", "merge_feat.weight",
                                                      "merge_feat.bias"]}
    (h0, w0), (h1, w1) = (3, 5), (4, 3)
    ff0 = rs.standard_normal((2, 128, 4 * h0, 4 * w0)).astype(np.float32)
    ff1 = rs.standard_normal((2, 128, 4 * h1, 4 * w1)).astype(np.float32)
    fc0 = rs.standard_normal((2, h0 * w0, 256)).astype(np.float32)
    fc1 = rs.standard_normal((2, h1 * w1, 256)).astype(np.float32)
    b_ids = np.array([0, 0, 1, 1, 1])
    i_ids, j_ids = np.array([0, 4, 10, 14, 7]), np.array([11, 2, 0, 9, 5])
    mk1 = rs.uniform(0, 40, (5, 2)).astype(np.float32)
    scale1 = rs.uniform(1, 2, (2, 2)).astype(np.float32)
    for W in (3, 5):
        r0, r1 = O.fine_preprocess(ff0, ff1, fc0, fc1, b_ids, i_ids, j_ids, w0, w1, W, 4, fw)
        g0, g1 = fine_preprocess_f64(ff0, ff1, fc0, fc1, b_ids, i_ids, j_ids, w0, w1, W, 4, fw)
        np.testing.assert_allclose(g0, r0, atol=2e-5)
        np.testing.assert_allclose(g1, r1, atol=2e-5)
        for s1 in (None, scale1):
            ro = O.fine_matching(r0, r1, mk1, mk1, b_ids, (8 * h0, 8 * w0), (4 * h0, 4 * w0), s1)
            e, k = fine_matching_f64(r0, r1, mk1, b_ids, 2.0, s1)
            np.testing.assert_allclose(e, ro["expec_f"], atol=2e-6)
            np.testing.assert_allclose(k, ro["mkpts1_f"], atol=1e-4)


# ================================================================================================ coarse matching
def _chunking(n, L, S, sms):
    """(chunks, tiles_per_chunk) of the score passes: pick_chunks + launch_gemm's re-derivation in csrc/engine.cu."""
    m_tiles, n_tiles = -(-L // 128), -(-S // 256)
    c = 1
    while n * m_tiles * c < 40 * sms and c < n_tiles:
        c += 1
    c = min(c, 32)
    tpc = -(-n_tiles // c)
    return -(-n_tiles // tpc), tpc


# L and S straddle the 32-column blocks (31 / 33), the 128-row tiles (127 / 128 / 129) and the 256-column n-tiles
# (255 / 256 / 257: S = 257 leaves a one-column last tile).  Grids with a side < 5 use border_rm 0, otherwise nothing
# could match.  "l6_s9000" gives a row 36 n-tiles: more than the 32 chunks, so every chunk sweeps two tiles.  In the
# masked cases one pair has a valid region of 2 * border_rm cells along one side (nothing survives the border removal)
# and one of 2 * border_rm + 1 (only the centre line survives).  With logits of O(1) the Sinkhorn prefilter sends every
# row to the dustbin, so the prefilter cases plant a few strong pairs (logit ~ 9) among O(1) rows.
CM_EDGE_CASES = [
    {"name": "ds_l15_s6", "n": 1, "hw0c": (3, 5), "hw1c": (2, 3), "border_rm": 0},
    {"name": "ds_l31_s33", "n": 3, "hw0c": (1, 31), "hw1c": (3, 11), "border_rm": 0},
    {"name": "ds_l33_s31", "n": 1, "hw0c": (3, 11), "hw1c": (1, 31), "border_rm": 0},
    {"name": "ds_l127_s129", "n": 5, "hw0c": (1, 127), "hw1c": (3, 43), "border_rm": 0},
    {"name": "ds_l128_s127", "n": 1, "hw0c": (8, 16), "hw1c": (1, 127), "border_rm": 0},
    {"name": "ds_l129_s128", "n": 3, "hw0c": (3, 43), "hw1c": (8, 16), "border_rm": 0},
    {"name": "ds_l256_s256", "n": 5, "hw0c": (16, 16), "hw1c": (16, 16)},
    {"name": "ds_l255_s257", "n": 3, "hw0c": (15, 17), "hw1c": (1, 257), "border_rm": 0},
    {"name": "ds_l257_s255", "n": 1, "hw0c": (1, 257), "hw1c": (5, 51), "border_rm": 0},
    {"name": "ds_l6_s9000", "n": 1, "hw0c": (2, 3), "hw1c": (90, 100), "border_rm": 0},
    {"name": "ds_masked_l255_s261", "n": 3, "hw0c": (15, 17), "hw1c": (9, 29),
     "valid0c": [(15, 17), (4, 17), (12, 10)], "valid1c": [(9, 20), (9, 29), (5, 25)]},
    {"name": "ot1_l129_s257", "n": 3, "hw0c": (3, 43), "hw1c": (1, 257), "border_rm": 0, "match_type": "sinkhorn",
     "skh_iters": 1},
    {"name": "ot3_l257_s127", "n": 1, "hw0c": (1, 257), "hw1c": (1, 127), "border_rm": 0, "match_type": "sinkhorn"},
    {"name": "ot1_pf_l31_s129", "n": 5, "hw0c": (1, 31), "hw1c": (3, 43), "border_rm": 0, "match_type": "sinkhorn",
     "skh_iters": 1, "prefilter": True},
    {"name": "ot3_pf_l255_s33", "n": 1, "hw0c": (15, 17), "hw1c": (3, 11), "border_rm": 0, "match_type": "sinkhorn",
     "prefilter": True},
    {"name": "ot3_pf_masked_l255_s261", "n": 3, "hw0c": (15, 17), "hw1c": (9, 29), "match_type": "sinkhorn",
     "prefilter": True, "valid0c": [(15, 17), (15, 4), (12, 10)], "valid1c": [(9, 20), (9, 29), (9, 25)]},
]


def _run_coarse(mod_cfg, f0, f1, hw0c, hw1c, m0g=None, m1g=None, bin_score=None):
    import loftr_b200.loftr as L
    mod = L.CoarseMatching(dict(mod_cfg, return_conf_matrix=True)).eval().to(DEV)
    if bin_score is not None:
        mod.bin_score.data = torch.tensor(float(bin_score), device=DEV)
    (h0, w0), (h1, w1) = hw0c, hw1c
    data = {"hw0_i": (h0 * 8, w0 * 8), "hw1_i": (h1 * 8, w1 * 8), "hw0_c": (h0, w0), "hw1_c": (h1, w1)}
    m0 = m1 = None
    if m0g is not None:
        data["mask0"], data["mask1"] = _t(m0g), _t(m1g)
        m0, m1 = data["mask0"].flatten(-2), data["mask1"].flatten(-2)
    mod(_t(f0), _t(f1), data, m0, m1)
    return data


@gpu
@pytest.mark.parametrize("case", CM_EDGE_CASES, ids=[c["name"] for c in CM_EDGE_CASES])
def test_coarse_matching_tile_edges_vs_fp64(case):
    sinkhorn = case.get("match_type") == "sinkhorn"
    # logits of O(1): dual-softmax sim = <f0, f1> / (C T), Sinkhorn sim = <f0, f1> / C
    inp = build_cm_inputs(dict(case, amp=1.0 if sinkhorn else 0.3, frac=0.6))
    f0, f1 = inp["feat_c0"], inp["feat_c1"]
    n, L, S = f0.shape[0], f0.shape[1], f1.shape[1]
    if case.get("prefilter"):
        rs = np.random.RandomState(3)
        k = max(2, min(L, S) // 8)
        for b in range(n):
            src, dst = rs.permutation(L)[:k], rs.permutation(S)[:k]
            f0[b, src] *= 3.0
            f1[b, dst] = f0[b, src]
    cfg = _cm_cfg(case)
    bin_score = 0.5 if sinkhorn else None
    m0 = inp["mask0"].reshape(n, -1) if "mask0" in inp else None
    m1 = inp["mask1"].reshape(n, -1) if "mask1" in inp else None
    sim = similarity_f64(f0, f1, cfg, m0, m1)
    live = sim > -1e8
    row_max = np.where(live, np.abs(sim), 0).max(2)[live.any(2)]
    assert (np.median(row_max) if case.get("prefilter") else row_max.max()) < 3.0, "the case is meant to have logits of O(1)"
    if not sinkhorn:
        # One logit-0 term leaked into a normaliser (zero-filled padding column of a partial 32-column block, or row of
        # a partial 128-row tile) must move that LSE by more than 1e-3, well above what mconf rtol 1e-3 resolves.
        pad_c, pad_r = (-S) % 32, (-L) % 128
        with np.errstate(invalid="ignore"):   # fully padded rows / columns have no normaliser: inf, filtered below
            row_lse = np.where(live.any(2), _lse_f64(np.where(live, sim, -np.inf), 2), np.inf)
            col_lse = np.where(live.any(1), _lse_f64(np.where(live, sim, -np.inf), 1), np.inf)
        if pad_c:
            assert np.log1p(pad_c * np.exp(-row_lse[np.isfinite(row_lse)])).min() > 1e-3
        if pad_r:
            assert np.log1p(pad_r * np.exp(-col_lse[np.isfinite(col_lse)])).min() > 1e-3
    if case["name"] == "ds_l6_s9000":
        chunks, tpc = _chunking(n, L, S, torch.cuda.get_device_properties(DEV).multi_processor_count)
        assert tpc > 1, (chunks, tpc)

    data = _run_coarse(cfg, f0, f1, case["hw0c"], case["hw1c"], inp.get("mask0"), inp.get("mask1"), bin_score)
    got = {k: data[k].cpu().numpy() for k in ["b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c"]}
    (h0, w0) = case["hw0c"]
    ref = O.coarse_matching(f0, f1, cfg, (h0 * 8, w0 * 8), case["hw0c"], case["hw1c"], inp.get("mask0"),
                            inp.get("mask1"), bin_score=bin_score)
    conf64 = conf_matrix_f64(f0, f1, cfg, m0, m1, bin_score)
    if sinkhorn:
        gold = top2_f64(conf64)
    else:
        t2 = [util.near_tie_top2_f64(f0[b], f1[b], cfg, None if m0 is None else m0[b], None if m1 is None else m1[b])
              for b in range(n)]
        gold = {"row_top2_f64": np.stack([r for r, _ in t2]), "col_top2_f64": np.stack([c for _, c in t2])}
    stats = util.compare_matches(got, ref, gold, conf_rtol=1e-3, px_tol=1e-3, min_overlap=0.995, label=case["name"])
    assert len(ref["b_ids"]) > 0 and stats["n"] > 0, f"{case['name']}: no matches to compare"
    # mconf against the float64 confidence of the engine's own (b, i, j)
    want = conf64[got["b_ids"], got["i_ids"], got["j_ids"]]
    rel = np.abs(got["mconf"] - want) / want
    stats["mconf_rel_vs_fp64"] = float(rel.max())
    assert rel.max() <= 1e-3, f"{case['name']}: mconf vs fp64 rel err {rel.max():.3e}"
    # conf_matrix everywhere except the fully padded cells (documented deviation, DESIGN.md §5)
    conf = data["conf_matrix"].cpu().numpy().astype(F64)
    want = conf64
    if m0 is not None:
        valid = m0[:, :, None] | m1[:, None, :]
        conf, want = conf * valid, want * valid
    err = np.abs(conf - want) / np.maximum(np.abs(want), 1e-300)
    stats["conf_matrix_rel_vs_fp64"] = float(err[want > 1e-30].max())
    np.testing.assert_allclose(conf, want, rtol=2e-3, atol=1e-12, err_msg=case["name"])
    if m0 is not None:   # a pair whose valid region is no wider than 2 * border_rm cells has nothing to match
        for b in range(n):
            (vh0, vw0), (vh1, vw1) = case["valid0c"][b], case["valid1c"][b]
            if min(vh0, vw0, vh1, vw1) <= 2 * cfg["border_rm"]:
                assert not (got["b_ids"] == b).any() and not (ref["b_ids"] == b).any(), f"pair {b} must have no match"
    util.record("edge_cm_" + case["name"], stats)


@gpu
def test_coarse_matching_exact_tie_picks_smallest_index():
    """DESIGN.md §5: exact floating-point ties pick the smallest index.  Columns j1 < j2 of f1 are identical and sit in
    the same 32-column block, so both run the same epilogue path and get bit-identical confidences; the reference's
    `mask.max(dim=2)` (coarse_matching.py:185) then returns j1."""
    rs = np.random.RandomState(31)
    n, hw, c = 2, (8, 16), 256
    f0 = (rs.standard_normal((n, 128, c)) * 0.3).astype(np.float32)
    f1 = (rs.standard_normal((n, 128, c)) * 0.3).astype(np.float32)
    i, j1, j2 = 3 * 16 + 7, 3 * 16 + 5, 3 * 16 + 9          # all interior cells (border_rm 2); j1, j2 in block 32..63
    for b in range(n):
        f1[b, j1] = f1[b, j2] = f0[b, i] * 1.5
    cfg = _cm_cfg({})
    data = _run_coarse(cfg, f0, f1, hw, hw)
    conf = data["conf_matrix"]
    assert torch.equal(conf[:, :, j1], conf[:, :, j2]), "identical columns must give bit-identical confidences"
    ref = O.coarse_matching(f0, f1, cfg, (64, 128), hw, hw)
    for b in range(n):
        assert ((ref["b_ids"] == b) & (ref["i_ids"] == i)).sum() == 1
        assert ref["j_ids"][(ref["b_ids"] == b) & (ref["i_ids"] == i)][0] == j1
        sel = (data["b_ids"] == b) & (data["i_ids"] == i)
        assert int(sel.sum()) == 1 and int(data["j_ids"][sel][0]) == j1, "the tie must resolve to the smaller index"
        assert not ((data["b_ids"] == b) & (data["j_ids"] == j2)).any()


# ================================================================================================ transformer
def _check_transformer(tf, cfg_tf, f0, f1, m0, m1, label):
    w = _layer_weights(tf)
    e0, e1 = transformer_f64(f0, f1, w, cfg_tf["layer_names"], cfg_tf["nhead"], m0, m1)
    g0, g1 = tf(_t(f0), _t(f1), None if m0 is None else _t(m0), None if m1 is None else _t(m1))
    stats = {}
    for g, e, side in ((g0, e0, "0"), (g1, e1, "1")):
        err = np.abs(g.cpu().numpy().astype(F64) - e).max()
        stats["max_abs_err_" + side] = float(err)
        assert err < 2e-4, f"{label}: transformer output {side} differs from fp64 by {err:.3e}"
    util.record("edge_tf_" + label, stats)


TF_COARSE = [(1, 1, 1), (3, 33, 7), (2, 64, 65), (1, 129, 257)]


@gpu
@pytest.mark.parametrize("nls", TF_COARSE + ["masked"], ids=[f"{n}x{l}x{s}" for n, l, s in TF_COARSE] + ["masked"])
def test_coarse_transformer_edges_vs_fp64(nls):
    """Coarse transformer at one-row groups, single k-block sources (S <= 64 clamps the K^T V split to 1), partial
    128-row tiles; low-amplitude inputs, so a zero-filled row leaking into sum(K) (elu(0) + 1 = 1) is visible."""
    model, cfg, _ = _model(device=DEV)
    rs = np.random.RandomState(5)
    m0 = m1 = None
    if nls == "masked":
        n, l, s = 3, 40, 70
        m0 = rs.uniform(size=(n, l)) > 0.25
        m1 = rs.uniform(size=(n, s)) > 0.25
        m1[0] = False                       # pair 0: no valid source row at all
        m1[1] = False
        m1[1, 37] = True                    # pair 1: a single valid source row
        m0[2, 0] = False
    else:
        n, l, s = nls
    f0 = (rs.standard_normal((n, l, 256)) * 0.3).astype(np.float32)
    f1 = (rs.standard_normal((n, s, 256)) * 0.3).astype(np.float32)
    _check_transformer(model.loftr_coarse, cfg["coarse"], f0, f1, m0, m1, f"coarse_{nls if isinstance(nls, str) else 'x'.join(map(str, nls))}")


@gpu
@pytest.mark.parametrize("W", [3, 5])
@pytest.mark.parametrize("windows", [1, 37, 3000])
def test_fine_transformer_windows_vs_fp64(W, windows):
    """Fine transformer over windows of W*W rows (9 or 25 tokens per group), from one window to several thousand."""
    model, cfg, _ = _model(W, DEV)
    rs = np.random.RandomState(6)
    ww = W * W
    f0 = (rs.standard_normal((windows, ww, 128)) * 0.3).astype(np.float32)
    f1 = (rs.standard_normal((windows, ww, 128)) * 0.3).astype(np.float32)
    _check_transformer(model.loftr_fine, cfg["fine"], f0, f1, None, None, f"fine_W{W}_{windows}")


# ================================================================================================ fine level
@gpu
@pytest.mark.parametrize("W", [3, 5])
@pytest.mark.parametrize("with_scale", [False, True], ids=["no_scale1", "scale1"])
def test_fine_level_corners_vs_fp64(W, with_scale):
    """FinePreprocess + FineMatching on unequal fine grids (hw0 != hw1): windows at all four corners of both maps (zero
    padding on every side), M = 1, both feature layouts (NCHW: scalar gather, NHWC: 8-channel vector gather)."""
    model, _, state = _model(W, DEV)
    rs = np.random.RandomState(8 + W)
    n, (h0c, w0c), (h1c, w1c), stride = 2, (6, 10), (9, 7), 4
    L, S = h0c * w0c, h1c * w1c
    ff0 = rs.standard_normal((n, 128, h0c * stride, w0c * stride)).astype(np.float32)
    ff1 = rs.standard_normal((n, 128, h1c * stride, w1c * stride)).astype(np.float32)
    fc0 = rs.standard_normal((n, L, 256)).astype(np.float32)
    fc1 = rs.standard_normal((n, S, 256)).astype(np.float32)
    corners0 = [0, w0c - 1, (h0c - 1) * w0c, L - 1]
    corners1 = [0, w1c - 1, (h1c - 1) * w1c, S - 1]
    sets = {"m1": (np.array([1]), np.array([L - 1]), np.array([0])),
            "corners": (np.array([0, 0, 0, 0, 1, 1, 1, 1, 1]), np.array(corners0 + corners0[::-1] + [23]),
                        np.array(corners1[1:] + corners1[:1] + corners1 + [30]))}
    fw = {k: state[f"fine_preprocess.{k}"] for k in ["down_proj.weight", "down_proj.bias", "merge_feat.weight",
                                                      "merge_feat.bias"]}
    scale1 = rs.uniform(1, 2.5, (n, 2)).astype(np.float32) if with_scale else None
    hw0_i, hw0_f, hw1_f = (h0c * 8, w0c * 8), (h0c * stride, w0c * stride), (h1c * stride, w1c * stride)
    for name, (b_ids, i_ids, j_ids) in sets.items():
        m = len(b_ids)
        e0, e1 = fine_preprocess_f64(ff0, ff1, fc0, fc1, b_ids, i_ids, j_ids, w0c, w1c, W, stride, fw)
        stats = {"M": m}
        for layout in ("nchw", "nhwc"):
            t0, t1 = _t(ff0), _t(ff1)
            if layout == "nhwc":
                t0, t1 = t0.contiguous(memory_format=torch.channels_last), t1.contiguous(memory_format=torch.channels_last)
            data = {"hw0_i": hw0_i, "hw0_c": (h0c, w0c), "hw1_c": (h1c, w1c), "hw0_f": hw0_f, "hw1_f": hw1_f,
                    "b_ids": _t(b_ids), "i_ids": _t(i_ids), "j_ids": _t(j_ids)}
            g0, g1 = model.fine_preprocess(t0, t1, _t(fc0), _t(fc1), data)
            assert g0.shape == (m, W * W, 128) and data["W"] == W
            for g, e, side in ((g0, e0, "0"), (g1, e1, "1")):
                err = np.abs(g.cpu().numpy().astype(F64) - e).max()
                stats[f"preprocess_{layout}_{side}_max_abs_err"] = float(err)
                assert err < 2e-4, f"{name} {layout}: window features {side} differ from fp64 by {err:.3e}"
        # fine matching on the fp32 image of the reference windows (isolates it from the preprocess error)
        x0, x1 = e0.astype(np.float32), e1.astype(np.float32)
        mk0 = rs.uniform(0, 80, (m, 2)).astype(np.float32)
        mk1 = rs.uniform(0, 80, (m, 2)).astype(np.float32)
        expec, kp1 = fine_matching_f64(x0, x1, mk1.astype(F64), b_ids, hw0_i[0] / hw0_f[0], scale1)
        data.update({"mkpts0_c": _t(mk0), "mkpts1_c": _t(mk1), "mconf": torch.ones(m, device=DEV)})
        if with_scale:
            data["scale0"], data["scale1"] = _t(scale1), _t(scale1)
        model.fine_matching(_t(x0), _t(x1), data)
        ge, gk = data["expec_f"].cpu().numpy(), data["mkpts1_f"].cpu().numpy()
        stats.update({"expec_max_abs_err": float(np.abs(ge - expec).max()), "mkpts1_f_max_px": float(np.abs(gk - kp1).max())})
        np.testing.assert_allclose(ge, expec, atol=2e-5, err_msg=name)
        np.testing.assert_allclose(gk, kp1, atol=1e-3, err_msg=name)
        assert np.abs(expec[:, :2]).max() > 0.05, "the heat maps are meant to be off-centre"
        util.record(f"edge_fine_W{W}_{'scale1' if with_scale else 'noscale'}_{name}", stats)


# ================================================================================================ match wire format
def _fake_matches(m, n_pairs, seed, device):
    g = torch.Generator().manual_seed(seed)
    d = {"mkpts0_f": torch.rand(m, 2, generator=g) * 640, "mkpts1_f": torch.rand(m, 2, generator=g) * 480,
         "mconf": torch.rand(m, generator=g),
         "m_bids": torch.sort(torch.randint(0, max(n_pairs, 1), (m,), generator=g)).values}
    return {k: v.to(device) for k, v in d.items()}


def _bits(t):
    return t.detach().cpu().contiguous().view(torch.int32)


@gpu
def test_match_wire_format_cuda_matches_cpu():
    """lb_pack_matches / lb_unpack_matches against the torch path of loftr_b200.parallel (the form the gloo test
    exercises), bit for bit: empty list, a list filling the capacity, a pair offset, and a world-3 gathered buffer."""
    from loftr_b200 import parallel
    cap = 64
    ranks = [(0, 0, 11), (cap, 3, 12), (17, 7, 13)]          # (count, pair offset, seed): empty / full / offset
    cpu_bufs, gpu_bufs = [], []
    for m, off, seed in ranks:
        dc, dg = _fake_matches(m, 4, seed, "cpu"), _fake_matches(m, 4, seed, DEV)
        bc, bg = parallel.pack_matches(dc, off, cap), parallel.pack_matches(dg, off, cap)
        assert bg.is_cuda and bg.shape == bc.shape == (1 + cap, 6)
        # row 0 and the payload rows are defined; rows past the count are not part of the format
        assert torch.equal(_bits(bg[:1 + m]), _bits(bc[:1 + m])), f"pack differs (count {m}, offset {off})"
        cpu_bufs.append(bc)
        gpu_bufs.append(bg)
        one_c, one_g = parallel.unpack_matches(bc.unsqueeze(0)), parallel.unpack_matches(bg.unsqueeze(0))
        assert one_g["counts"] == one_c["counts"] == [m]
        for k in ("mkpts0_f", "mkpts1_f", "mconf"):
            assert torch.equal(_bits(one_g[k]), _bits(one_c[k])), k
        assert torch.equal(one_g["m_bids"].cpu(), one_c["m_bids"]) and one_g["m_bids"].dtype == torch.int64
        assert torch.equal(one_c["m_bids"], dc["m_bids"] + off)
    allc = parallel.unpack_matches(torch.stack(cpu_bufs, 0))
    allg = parallel.unpack_matches(torch.stack(gpu_bufs, 0))
    assert allg["counts"] == allc["counts"] == [m for m, _, _ in ranks]
    total = sum(m for m, _, _ in ranks)
    for k in ("mkpts0_f", "mkpts1_f", "mconf"):
        assert allg[k].shape[0] == total
        assert torch.equal(_bits(allg[k]), _bits(allc[k])), k
    assert torch.equal(allg["m_bids"].cpu(), allc["m_bids"])
    want = torch.cat([_fake_matches(m, 4, seed, "cpu")["m_bids"] + off for m, off, seed in ranks])
    assert torch.equal(allc["m_bids"], want)
    util.record("edge_wire_format", {"world": 3, "capacity": cap, "total": total})
