"""Parity tests proper: the CUDA engine (through the C ABI) against the numpy oracle and against the
golden vectors of the reference.  Tolerances are BASELINE.json's: |dxy| < 0.5 px on keypoints, mconf
rtol 1e-3 (match sets compared by key with near-tie adjudication)."""
import ctypes as C

import numpy as np
import pytest
import torch

import util
from cases import BASELINE_CASES, CASES, CM_CASES, build_cfg, build_cm_inputs, build_inputs
from oracle import loftr_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
    return t if dtype is None else t.to(dtype)


# ------------------------------------------------------------------------------------------------ contraction core
# (batches, M, N, K[, "shared_b" | "wide"]).  Edge cases: M = 1 / 127 / 129 (one M-tile: single-CTA launch; a one-row
# second tile), N = 32 (128-column tiles), 160 (one partial 256-column tile), 288 (a 32-column second tile), K = 64 (one
# k-block) / 1024; "shared_b": batched A against ONE B (b_batch_stride = 0); "wide": magnitudes 1e-3 .. 1e3 with random
# signs, so the products of the `lo` planes carry real information.
_GEMM_EDGE = [(1, m, n, k) for m in (1, 127, 129) for n in (32, 160, 288) for k in (64, 1024)]


@pytest.mark.parametrize("shape", [(1, 128, 256, 64), (1, 300, 768, 256), (1, 1000, 128, 128), (2, 200, 512, 256),
                                   (1, 1200, 384, 128), (1, 77, 256, 512)] + _GEMM_EDGE +
                         [(3, 129, 288, 64, "shared_b"), (4, 1, 32, 1024, "shared_b"), (2, 300, 160, 256, "shared_b"),
                          (1, 129, 288, 1024, "wide"), (3, 127, 160, 512, "wide"), (2, 1, 288, 64, "wide")])
def test_gemm_split_matches_fp64(shape):
    from loftr_b200 import _lib
    from loftr_b200.loftr import split_planes, _stream
    b, m, n, k = shape[:4]
    kind = shape[4] if len(shape) > 4 else ""
    nb = 1 if kind == "shared_b" else b
    rs = np.random.RandomState(0)
    if kind == "wide":
        a = (10.0 ** rs.uniform(-3, 3, (b * m, k)) * rs.choice([-1, 1], (b * m, k))).astype(np.float32)
        w = (10.0 ** rs.uniform(-3, 3, (nb * n, k)) * rs.choice([-1, 1], (nb * n, k))).astype(np.float32)
    else:
        a = (rs.standard_normal((b * m, k)) * 3 + 1).astype(np.float32)
        w = (rs.standard_normal((nb * n, k)) * 3 + 1).astype(np.float32)
    ta, tw = _t(a), _t(w)
    ah, al = split_planes(ta)
    wh, wl = split_planes(tw)
    out = torch.empty(b * m, n, dtype=torch.float32, device=DEV)
    lib = _lib.load()
    _lib.check(lib.lb_gemm_split(ah.data_ptr(), al.data_ptr(), k, m * k, wh.data_ptr(), wl.data_ptr(), k,
                                 n * k if nb > 1 else 0, out.data_ptr(), n, m * n, b, m, n, k, _stream()))
    ref = np.einsum("bmk,bnk->bmn", a.reshape(b, m, k).astype(np.float64),
                    np.broadcast_to(w.reshape(nb, n, k), (b, n, k)).astype(np.float64))
    got = out.cpu().numpy().reshape(b, m, n)
    err = np.abs(got - ref).max() / np.abs(ref).max()
    util.record("gemm_split_" + "x".join(map(str, shape)), {"max_err_rel_to_max_ref": float(err)})
    assert err < 5e-6


# ------------------------------------------------------------------------------------------------ transformer
def _layer_weights(model_tf):
    names = ["q_proj.weight", "k_proj.weight", "v_proj.weight", "merge.weight", "mlp.0.weight", "mlp.2.weight",
             "norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"]
    sd = {k: v.detach().cpu().numpy() for k, v in model_tf.state_dict().items()}
    return [{k: sd[f"layers.{i}.{k}"] for k in names} for i in range(len(model_tf.layers))]


@pytest.mark.parametrize("cfgname", ["coarse_equal", "coarse_masked_unequal", "fine_windows"])
def test_transformer_matches_oracle(cfgname):
    case = CASES[0]
    model, cfg, _ = util.build_model(case, DEV)
    rs = np.random.RandomState(3)
    if cfgname == "fine_windows":
        tf, tcfg = model.loftr_fine, cfg["fine"]
        n, l, s, c = 37, 25, 25, 128
        m0 = m1 = None
    else:
        tf, tcfg = model.loftr_coarse, cfg["coarse"]
        c = 256
        if cfgname == "coarse_equal":
            n, l, s = 2, 300, 300
            m0 = m1 = None
        else:
            n, l, s = 2, 280, 200
            m0 = rs.uniform(size=(n, l)) > 0.2
            m1 = rs.uniform(size=(n, s)) > 0.3
    f0 = rs.standard_normal((n, l, c)).astype(np.float32)
    f1 = rs.standard_normal((n, s, c)).astype(np.float32)
    o0, o1 = O.local_feature_transformer(f0, f1, _layer_weights(tf), tcfg["layer_names"], tcfg["nhead"], m0, m1)
    g0, g1 = tf(_t(f0), _t(f1), None if m0 is None else _t(m0), None if m1 is None else _t(m1))
    for g, o in ((g0, o0), (g1, o1)):
        err = np.abs(g.cpu().numpy() - o).max()
        assert err < 2e-4, f"{cfgname}: transformer output differs by {err:.3e}"


# ------------------------------------------------------------------------------------------------ coarse matching
@pytest.mark.parametrize("case", CM_CASES, ids=[c["name"] for c in CM_CASES])
def test_coarse_matching_matches_reference_golden(case):
    import loftr_b200.loftr as L
    gold = util.load_golden(case["name"])
    cfg = build_cfg(case)["match_coarse"]
    cfg["return_conf_matrix"] = True
    inp = build_cm_inputs(case)
    mod = L.CoarseMatching(cfg).eval().to(DEV)
    if cfg["match_type"] == "sinkhorn":
        mod.bin_score.data = torch.tensor(float(case.get("bin_score", 1.0)), device=DEV)
    (h0, w0), (h1, w1) = case["hw0c"], case["hw1c"]
    data = {"hw0_i": (h0 * 8, w0 * 8), "hw1_i": (h1 * 8, w1 * 8), "hw0_c": (h0, w0), "hw1_c": (h1, w1)}
    m0 = m1 = None
    if "mask0" in inp:
        data["mask0"], data["mask1"] = _t(inp["mask0"]), _t(inp["mask1"])
        m0, m1 = data["mask0"].flatten(-2), data["mask1"].flatten(-2)
    mod(_t(inp["feat_c0"]), _t(inp["feat_c1"]), data, m0, m1)
    got = {k: data[k].cpu().numpy() for k in ["b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c"]}
    stats = util.compare_matches(got, gold, gold, conf_rtol=1e-3, px_tol=1e-3, min_overlap=1.0, label=case["name"])
    assert stats["n"] == len(gold["b_ids"])
    assert data["b_ids"].dtype == torch.int64 and data["mconf"].dtype == torch.float32
    # opt-in conf_matrix: identical to the reference's except on cells where both the row and the column are
    # padding (reference: 1/(L*S)-like constants, engine: 0 -- documented deviation, never matchable)
    conf = data["conf_matrix"].cpu().numpy()
    ref = gold["conf_matrix"]
    if "mask0" in inp:
        valid = inp["mask0"].reshape(ref.shape[0], -1)[:, :, None] | inp["mask1"].reshape(ref.shape[0], -1)[:, None, :]
        conf, ref = conf * valid, ref * valid
    np.testing.assert_allclose(conf, ref, rtol=2e-3, atol=1e-9)


def test_coarse_matching_full_size_vs_oracle():
    """640x480 grid (L = S = 4800, 38 row tiles, partial last tile), 2 pairs, dual-softmax, thr 0."""
    import loftr_b200.loftr as L
    rs = np.random.RandomState(5)
    n, h, w, c = 2, 60, 80, 256
    base = rs.standard_normal((n, h * w, c)).astype(np.float32)
    f0 = base * 1.2 + 3.0   # large common-mode part like the real features (SURVEY.md §7 hard part 1)
    perm = rs.permutation(h * w)
    f1 = (base[:, perm] * 1.2 + 3.0 + 0.3 * rs.standard_normal((n, h * w, c))).astype(np.float32)
    cfg = build_cfg({"thr": 0.0})["match_coarse"]
    out = O.coarse_matching(f0, f1, cfg, (480, 640), (h, w), (h, w))
    mod = L.CoarseMatching(cfg).eval()
    data = {"hw0_i": (480, 640), "hw1_i": (480, 640), "hw0_c": (h, w), "hw1_c": (h, w)}
    mod(_t(f0), _t(f1), data)
    got = {k: data[k].cpu().numpy() for k in ["b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c"]}
    assert len(out["b_ids"]) > 1000
    g64 = [util.near_tie_top2_f64(f0[b], f1[b], cfg) for b in range(n)]
    gold = {"row_top2_f64": np.stack([g[0] for g in g64]), "col_top2_f64": np.stack([g[1] for g in g64])}
    stats = util.compare_matches(got, out, gold, conf_rtol=1e-3, px_tol=1e-3, min_overlap=0.995, label="full")
    assert stats["n"] > 1000


# ------------------------------------------------------------------------------------------------ fine level
def test_fine_level_matches_oracle():
    case = CASES[0]
    model, cfg, state = util.build_model(case, DEV)
    rs = np.random.RandomState(9)
    n, hc, wc = 2, 12, 16
    hf, wf = hc * 4, wc * 4
    feat_f0 = rs.standard_normal((n, 128, hf, wf)).astype(np.float32)
    feat_f1 = rs.standard_normal((n, 128, hf, wf)).astype(np.float32)
    feat_c0 = rs.standard_normal((n, hc * wc, 256)).astype(np.float32)
    feat_c1 = rs.standard_normal((n, hc * wc, 256)).astype(np.float32)
    m = 50
    b_ids = np.sort(rs.randint(0, n, m)).astype(np.int64)
    i_ids = rs.randint(0, hc * wc, m).astype(np.int64)   # includes border cells -> zero padding of windows
    j_ids = rs.randint(0, hc * wc, m).astype(np.int64)
    i_ids[0], j_ids[0] = 0, hc * wc - 1
    fw = {k: state[f"fine_preprocess.{k}"] for k in ["down_proj.weight", "down_proj.bias", "merge_feat.weight",
                                                      "merge_feat.bias"]}
    o0, o1 = O.fine_preprocess(feat_f0, feat_f1, feat_c0, feat_c1, b_ids, i_ids, j_ids, wc, wc, 5, 4, fw)
    data = {"hw0_i": (hc * 8, wc * 8), "hw0_c": (hc, wc), "hw1_c": (hc, wc), "hw0_f": (hf, wf), "hw1_f": (hf, wf),
            "b_ids": _t(b_ids), "i_ids": _t(i_ids), "j_ids": _t(j_ids)}
    for layout in ("nchw", "nhwc"):
        tf0, tf1 = _t(feat_f0), _t(feat_f1)
        if layout == "nhwc":
            tf0, tf1 = tf0.contiguous(memory_format=torch.channels_last), tf1.contiguous(memory_format=torch.channels_last)
        g0, g1 = model.fine_preprocess(tf0, tf1, _t(feat_c0), _t(feat_c1), data)
        assert np.abs(g0.cpu().numpy() - o0).max() < 2e-4, layout
        assert np.abs(g1.cpu().numpy() - o1).max() < 2e-4, layout
    # fine matching on the oracle's transformer output
    mk0 = rs.uniform(0, 100, (m, 2)).astype(np.float32)
    mk1 = rs.uniform(0, 100, (m, 2)).astype(np.float32)
    scale1 = rs.uniform(1, 2, (n, 2)).astype(np.float32)
    of = O.fine_matching(o0, o1, mk0, mk1, b_ids, (hc * 8, wc * 8), (hf, wf), scale1)
    data.update({"mkpts0_c": _t(mk0), "mkpts1_c": _t(mk1), "scale0": _t(scale1), "scale1": _t(scale1),
                 "mconf": torch.ones(m, device=DEV)})
    model.fine_matching(_t(o0), _t(o1), data)
    np.testing.assert_allclose(data["expec_f"].cpu().numpy(), of["expec_f"], atol=2e-5)
    np.testing.assert_allclose(data["mkpts1_f"].cpu().numpy(), of["mkpts1_f"], atol=2e-4)
    assert data["mkpts0_f"] is data["mkpts0_c"]   # the reference aliases them (fine_matching.py:67)


# ------------------------------------------------------------------------------------------------ end to end
def _run_engine(case):
    model, cfg, state = util.build_model(case, DEV)
    inp = build_inputs(case)
    data = {k: _t(v) for k, v in inp.items()}
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    model.expose_coarse_features = True   # test tap: data['_feat_c0'/'_feat_c1']
    model(data)
    return model, data


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_end_to_end_matches_reference_golden(case):
    gold = util.load_golden(case["name"])
    _, data = _run_engine(case)
    for k in ["hw0_i", "hw1_i", "hw0_c", "hw1_c", "hw0_f", "hw1_f"]:
        assert tuple(data[k]) == tuple(gold[k])
    assert data["bs"] == case["n"] and data["W"] == 5
    got = {k: data[k].cpu().numpy() for k in ["b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c", "mkpts0_f",
                                              "mkpts1_f", "expec_f"]}
    np.testing.assert_allclose(data["_feat_c0"].cpu().numpy()[:, ::7, ::5], gold["feat_c0_s"], rtol=1e-3, atol=1e-3)
    np.testing.assert_allclose(data["_feat_c1"].cpu().numpy()[:, ::7, ::5], gold["feat_c1_s"], rtol=1e-3, atol=1e-3)
    stats = util.compare_matches(got, gold, gold, conf_rtol=1e-3, px_tol=0.5, min_overlap=0.995, label=case["name"])
    util.record("e2e_golden_" + case["name"], stats)
    m = len(gold["b_ids"])
    if m == 0:
        assert got["b_ids"].shape == (0,) and got["mkpts0_f"].shape == (0, 2) and got["expec_f"].shape == (0, 3)
        assert data["mkpts0_f"] is data["mkpts0_c"]
    else:
        assert stats["n"] >= m - max(1, int(0.005 * m))
    assert got["mkpts1_f"].dtype == np.float32 and data["m_bids"].dtype == torch.int64
    assert data["gt_mask"].dtype == torch.bool and data["gt_mask"].shape[0] == len(got["b_ids"])


_KEYS = ["b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c", "mkpts0_f", "mkpts1_f"]


def _engine_vs_oracle(case, label, min_matches, record_as=None, feat_tol=1e-3):
    """Engine (C ABI) vs the per-pair numpy oracle on the SAME backbone features, BASELINE.json tolerances:
    key overlap >= 99.5 %, every non-shared match an fp64 near-tie (dual-softmax), mconf rtol 1e-3, |dxy| < 0.5 px."""
    model, data = _run_engine(case)
    out, gold = util.oracle_forward_per_pair(case, backbone_device=DEV)
    got = {k: data[k].cpu().numpy() for k in _KEYS}
    assert len(out["b_ids"]) > min_matches, f"{label}: only {len(out['b_ids'])} oracle matches"
    stats = util.compare_matches(got, out, gold, conf_rtol=1e-3, px_tol=0.5, min_overlap=0.995, label=label)
    err = np.abs(data["_feat_c0"].cpu().numpy()[:, ::4] - out["feat_c0_s4"]).max()
    assert err < feat_tol, f"{label}: coarse transformer output differs by {err:.3e}"
    stats["feat_c0_max_abs_err"] = float(err)
    per_pair = np.bincount(got["b_ids"], minlength=case["n"])
    assert (per_pair > 0).all(), f"{label}: a pair of the batch produced no match: {per_pair}"
    util.record(record_as or label, stats)
    return data, out, stats


def test_end_to_end_640x480_vs_oracle():
    """Config 1 of BASELINE.json (single 640x480 pair, indoor_ds) at thr 0."""
    _engine_vs_oracle(BASELINE_CASES["full"], "640x480", 300, "e2e_640x480_ds_vs_oracle")


def test_batch8_640x480_ds_vs_oracle():
    """configs[1] EXACTLY as benchmarked: batch = 8 pairs 640x480, indoor_ds dual-softmax (the batch size
    changes the chunking / partial-merge layout of the score passes and the tile schedule of every GEMM)."""
    _engine_vs_oracle(BASELINE_CASES["b8"], "b8 640x480 ds", 8 * 300, "e2e_b8_640x480_ds_vs_oracle")


def test_batch8_640x480_default_thr_vs_oracle():
    """configs[1] at the cfg default thr = 0.2 (SURVEY.md §8(d) threshold caveat): with these weights no
    confidence reaches 0.2, so both sides must return the empty list through the M = 0 path."""
    case = BASELINE_CASES["b8thr"]
    model, data = _run_engine(case)
    out, _ = util.oracle_forward_per_pair(case, backbone_device=DEV, adjudicate=False)
    assert len(out["b_ids"]) == data["b_ids"].shape[0]
    if len(out["b_ids"]):
        got = {k: data[k].cpu().numpy() for k in _KEYS}
        util.compare_matches(got, out, None, conf_rtol=1e-3, px_tol=0.5, min_overlap=0.995, label="b8 thr0.2")
    else:
        assert data["mkpts0_f"].shape == (0, 2) and data["expec_f"].shape == (0, 3)


def test_batch8_640x480_sinkhorn_vs_oracle():
    """configs[4] EXACTLY as named: batch = 8 pairs 640x480, indoor_ot (Sinkhorn, 3 iterations)."""
    _engine_vs_oracle(BASELINE_CASES["b8ot"], "b8 640x480 ot", 8 * 300, "e2e_b8_640x480_sinkhorn_vs_oracle")


def test_outdoor_832_batch4_masked_vs_oracle():
    """configs[2] per-GPU shard: 4 pairs 832x832 (L = S = 10816) with MegaDepth-style padding masks (a different
    valid region per image) and scales."""
    case = BASELINE_CASES["out4"]
    data, out, _ = _engine_vs_oracle(case, "4x832 masked", 4 * 400, "e2e_4x832x832_masked_vs_oracle")
    b, i, j = (data[k].cpu().numpy() for k in ("b_ids", "i_ids", "j_ids"))
    for p in range(4):   # nothing may come from the padded area or its border  [coarse_matching.py:28-43]
        (vh0, vw0), (vh1, vw1) = case["valid0"][p], case["valid1"][p]
        sel = b == p
        assert (i[sel] // 104 < vh0 // 8 - 2).all() and (i[sel] % 104 < vw0 // 8 - 2).all()
        assert (j[sel] // 104 < vh1 // 8 - 2).all() and (j[sel] % 104 < vw1 // 8 - 2).all()


def test_no_cpu_fallback():
    import loftr_b200
    model = loftr_b200.LoFTR(loftr_b200.get_cfg("indoor_ds")).eval()
    with pytest.raises(RuntimeError):
        model({"image0": torch.rand(1, 1, 64, 64), "image1": torch.rand(1, 1, 64, 64)})


# ------------------------------------------------------------------------------------------------ BASELINE.json configs
def test_outdoor_832_masked_vs_oracle():
    """configs[2] shape: 832x832 (L = S = 10816), MegaDepth-style padding masks + scales, one pair."""
    data, out, _ = _engine_vs_oracle(BASELINE_CASES["outdoor"], "832 masked", 500, "e2e_832x832_masked_vs_oracle")
    i, j = data["i_ids"].cpu().numpy(), data["j_ids"].cpu().numpy()
    assert (i % 104 < 624 // 8 - 2).all() and (j // 104 < 640 // 8 - 2).all()


def test_sinkhorn_640x480_vs_oracle():
    """configs[4] shape: indoor_ot at 640x480 (one pair)."""
    _engine_vs_oracle(BASELINE_CASES["ot_full"], "ot 640x480", 300, "e2e_640x480_sinkhorn_vs_oracle")


@pytest.mark.parametrize("hw", [(240, 320), (720, 960), (960, 1280)])
def test_resolution_sweep_vs_oracle(hw):
    """configs[3]: token-count scaling, L = 1200 / 10800 / 19200 (4800 is test_end_to_end_640x480_vs_oracle).  The
    FULL match list is compared with the oracle at every size (the oracle's L x S temporaries are ~1.5 GB fp32 at
    1280x960; the fp64 adjudication statistics are evaluated row-blocked)."""
    h, w = hw
    case = BASELINE_CASES[f"sweep{h}"]
    _engine_vs_oracle(case, f"sweep {h}x{w}", (h // 8) * (w // 8) // 25, f"e2e_sweep_{h}x{w}_vs_oracle")


def test_large_batch_duplicate_pairs_agree():
    """Size-independent property at the largest sweep size (1280x960, L = 19200): the two copies of one pair
    inside a batch give bit-identical lists (no cross-pair leakage, schedule-independent reductions)."""
    case = {"name": "sweep", "n": 1, "hw0": (960, 1280), "hw1": (960, 1280), "thr": 0.0, "images": "smooth"}
    model, cfg, _ = util.build_model(case, DEV)
    inp = build_inputs(case)
    i0, i1 = _t(inp["image0"]), _t(inp["image1"])
    two = {"image0": torch.cat([i0, i0]), "image1": torch.cat([i1, i1])}
    model(two)
    nb = (two["m_bids"] == 0).sum().item()
    assert nb > 1000 and two["mconf"].shape[0] == 2 * nb
    for k in ("i_ids", "j_ids", "mconf", "mkpts1_f"):
        assert torch.equal(two[k][:nb], two[k][nb:]), k


# ------------------------------------------------------------------------------------------------ backbone on tensor cores
# Branches of run_conv / launch_conv the small and ragged shapes reach.  An output map of h x w pixels has
# ceil(h/8) * ceil(w/16) tiles of 8 x 16; one tile runs the single-CTA kernel (mode 0), two or more the CTA pair
# (mode 2).  A lateral (layer2_outconv: Cout 256 at 1/4, layer1_outconv: Cout 196 at 1/2) stages its x2 upsample source
# in shared memory (EpiConv<., 1, .>) only in mode 2, otherwise every thread gathers it (EpiConv<256|208, 2, true>).
#   shape         tiles 1/2, 1/4, 1/8     modes (1/2, 1/4, 1/8)   layer2_outconv   layer1_outconv   coarse grid
#   (2, 8, 8)     1, 1, 1                 0, 0, 0                 per-thread       per-thread       1 x 1
#   (2, 16, 32)   1, 1, 1                 0, 0, 0                 per-thread       per-thread       2 x 4
#   (3, 32, 64)   4, 1, 1                 2, 0, 0                 per-thread       staged           4 x 8
#   (1, 8, 256)   8, 4, 2                 2, 2, 2                 staged           staged           1 x 32
#   (1, 200, 40)  26, 7, 4                2, 2, 2                 staged           staged           25 x 5 (ragged tiles)
@pytest.mark.parametrize("shape", [(2, 96, 128), (1, 480, 640), (1, 136, 200), (2, 8, 8), (2, 16, 32), (3, 32, 64),
                                   (1, 8, 256), (1, 200, 40)])
def test_tensor_core_backbone_matches_torch(shape):
    """lb_backbone_forward (implicit-GEMM convolutions, folded BN, fused residual / FPN upsample-add) against the
    PyTorch ResNetFPN_8_2 forward in fp32 (TF32 off) with non-trivial BatchNorm statistics."""
    from loftr_b200.loftr import TensorCoreBackbone
    n, h, w = shape
    case = dict(CASES[0])
    model, _, _ = util.build_model(case, DEV)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    rs = np.random.RandomState(4)
    img = _t(rs.uniform(0, 1, (n, 1, h, w)).astype(np.float32))
    import copy
    with torch.no_grad():
        ref_c, ref_f = model.backbone(img)
        m64 = copy.deepcopy(model.backbone).double()
        ex_c, ex_f = m64(img.double())          # fp64 ground truth: both fp32 paths are judged against it
    tc = TensorCoreBackbone(model.backbone)
    got_c, got_f = tc(img)
    assert got_c.shape == (n, h // 8, w // 8, 256) and got_f.shape == (n, h // 2, w // 2, 128)
    for got, ref, ex, name in ((got_c, ref_c, ex_c, "coarse"), (got_f, ref_f, ex_f, "fine")):
        scale = ex.abs().max().item()
        err_ours = (got.permute(0, 3, 1, 2).double() - ex).abs().max().item()
        err_torch = (ref.double() - ex).abs().max().item()
        util.record(f"backbone_{name}_{n}x{h}x{w}", {"err_ours_vs_fp64": err_ours, "err_torch_fp32_vs_fp64": err_torch,
                                                      "scale": scale})
        # The tensor-core path is less accurate than cuDNN's fp32 FMA chain (measured ~4e-5 vs ~1.5e-6 of the
        # feature scale): tcgen05 accumulates in fp32 with truncation, once per MMA (K/16*3 adds per output), and
        # the bias compounds over the ~20 convolutions.  It stays well inside what the matcher tolerances need
        # (end-to-end mconf rel err 5e-4 < 1e-3, see parity_stats); bound it so regressions are caught.
        assert err_ours <= 1e-4 * scale, f"{name}: {err_ours:.3e} (torch fp32: {err_torch:.3e}, scale {scale:.3e})"


def test_coarse_matching_large_logit_spread():
    """Logits spanning hundreds of nats inside one 32x32 block: the shared-reference fast path of the LSE
    epilogue must detect the underflow risk and fall back to per-row / per-column references."""
    import loftr_b200.loftr as L
    rs = np.random.RandomState(21)
    n, h, w, c = 2, 20, 24, 256
    f0 = (rs.standard_normal((n, h * w, c)) * 3.0).astype(np.float32)
    f1 = (rs.standard_normal((n, h * w, c)) * 3.0).astype(np.float32)
    k = 200
    for b in range(n):
        src, dst = rs.permutation(h * w)[:k], rs.permutation(h * w)[:k]
        f1[b, dst] = f0[b, src] * rs.uniform(0.2, 1.5, (k, 1)).astype(np.float32)   # matched logits 18 .. 135
    f0[:, ::7] *= 0.02                                                                # some nearly featureless rows
    cfg = build_cfg({"thr": 0.2})["match_coarse"]
    out = O.coarse_matching(f0, f1, cfg, (h * 8, w * 8), (h, w), (h, w))
    sim = (f0[0] / 16) @ (f1[0] / 16).T / 0.1
    assert sim.max() - sim.min() > 150, "the case is meant to have a huge logit spread"
    mod = L.CoarseMatching(cfg).eval()
    data = {"hw0_i": (h * 8, w * 8), "hw1_i": (h * 8, w * 8), "hw0_c": (h, w), "hw1_c": (h, w)}
    mod(_t(f0), _t(f1), data)
    got = {kk: data[kk].cpu().numpy() for kk in ["b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c"]}
    assert len(out["b_ids"]) > 50
    stats = util.compare_matches(got, out, None, conf_rtol=1e-3, px_tol=1e-3, min_overlap=1.0, label="spread")
    util.record("cm_large_logit_spread", stats)


# ------------------------------------------------------------------------------------------------ host-object behaviour
def test_packed_caches_survive_copy_pickle_and_data_mutation():
    """ADVICE r1: after a forward the model must still deep-copy / pickle (the ctypes caches are not state), and
    `invalidate_packed()` must make `.data` writes visible to the kernels."""
    import copy
    import io
    case = dict(CASES[0])
    model, data = _run_engine(case)
    ref = {k: data[k].clone() for k in ("mconf", "mkpts1_f")}
    clone = copy.deepcopy(model)
    buf = io.BytesIO()
    torch.save(model, buf)
    buf.seek(0)
    loaded = torch.load(buf, weights_only=False)
    for m in (clone, loaded):
        d = {k: _t(v) for k, v in build_inputs(case).items()}
        m(d)
        assert torch.equal(d["mconf"], ref["mconf"]) and torch.equal(d["mkpts1_f"], ref["mkpts1_f"])
    # .data mutation is invisible to _version / data_ptr: stale until invalidate_packed()
    w = model.loftr_coarse.layers[0].merge.weight
    w.data.mul_(1.5)
    d1 = {k: _t(v) for k, v in build_inputs(case).items()}
    model(d1)
    model.invalidate_packed()
    d2 = {k: _t(v) for k, v in build_inputs(case).items()}
    model(d2)
    assert d2["mconf"].shape != ref["mconf"].shape or not torch.equal(d2["mconf"], ref["mconf"])
    # load_state_dict invalidates by itself
    model.load_state_dict(clone.state_dict())
    d3 = {k: _t(v) for k, v in build_inputs(case).items()}
    model(d3)
    assert torch.equal(d3["mconf"], ref["mconf"])
    assert "_feat_c0" in d3
    clone.expose_coarse_features = False
    d4 = {k: _t(v) for k, v in build_inputs(case).items()}
    clone(d4)
    assert "_feat_c0" not in d4 and "_feat_c1" not in d4
