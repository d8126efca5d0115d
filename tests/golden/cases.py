"""Golden-vector cases shared by make_golden.py (reference side) and the tests (oracle / CUDA side)."""
from __future__ import annotations

import copy

import numpy as np

import weights as W

_BASE = {
    "backbone_type": "ResNetFPN", "resolution": (8, 2), "fine_window_size": 5, "fine_concat_coarse_feat": True,
    "resnetfpn": {"initial_dim": 128, "block_dims": [128, 196, 256]},
    "coarse": {"d_model": 256, "d_ffn": 256, "nhead": 8, "layer_names": ["self", "cross"] * 4,
               "attention": "linear", "temp_bug_fix": True},
    "match_coarse": {"thr": 0.2, "border_rm": 2, "match_type": "dual_softmax", "dsmax_temperature": 0.1,
                     "skh_iters": 3, "skh_init_bin_score": 1.0, "skh_prefilter": False,
                     "train_coarse_percent": 0.2, "train_pad_num_gt_min": 200, "sparse_spvs": False},
    "fine": {"d_model": 128, "d_ffn": 128, "nhead": 8, "layer_names": ["self", "cross"], "attention": "linear"},
}

# Small shapes (the CPU reference and the numpy oracle both finish in seconds) covering every branch of
# the hot path: dual-softmax / sinkhorn (+prefilter), thresholds, padding masks + scales, unequal image
# sizes, the historical position-encoding variant, M == 0.
CASES = [
    {"name": "ds_thr0", "n": 2, "hw0": (96, 128), "hw1": (96, 128), "thr": 0.0, "images": "smooth",
     "keep": ("conf",)},
    {"name": "ds_thr_mid", "n": 2, "hw0": (96, 128), "hw1": (96, 128), "thr": 0.02, "images": "smooth"},
    {"name": "ds_empty", "n": 1, "hw0": (96, 128), "hw1": (96, 128), "thr": 0.97, "images": "rand"},
    {"name": "ds_masked_scaled", "n": 2, "hw0": (128, 128), "hw1": (128, 128), "thr": 0.0, "images": "smooth",
     "valid0": [(128, 96), (104, 128)], "valid1": [(112, 128), (128, 88)], "scales": True},
    {"name": "ds_unequal", "n": 1, "hw0": (96, 128), "hw1": (128, 104), "thr": 0.0, "images": "rand"},
    {"name": "ds_buggy_pe_border0", "n": 1, "hw0": (96, 128), "hw1": (96, 128), "thr": 0.0, "images": "smooth",
     "temp_bug_fix": False, "border_rm": 0},
    {"name": "ot_thr0", "n": 2, "hw0": (96, 128), "hw1": (96, 128), "thr": 0.0, "images": "smooth",
     "match_type": "sinkhorn", "keep": ("conf",)},
    {"name": "ot_prefilter", "n": 1, "hw0": (96, 128), "hw1": (96, 128), "thr": 0.0, "images": "smooth",
     "match_type": "sinkhorn", "prefilter": True, "bin_score": -3.0},
    {"name": "ot_masked", "n": 1, "hw0": (128, 128), "hw1": (128, 128), "thr": 0.0, "images": "smooth",
     "match_type": "sinkhorn", "valid0": [(128, 96)], "valid1": [(104, 128)], "scales": True},
]


def build_cfg(case):
    cfg = copy.deepcopy(_BASE)
    cfg["match_coarse"]["thr"] = case.get("thr", 0.2)
    cfg["match_coarse"]["match_type"] = case.get("match_type", "dual_softmax")
    cfg["match_coarse"]["skh_prefilter"] = case.get("prefilter", False)
    cfg["match_coarse"]["border_rm"] = case.get("border_rm", 2)
    cfg["coarse"]["temp_bug_fix"] = case.get("temp_bug_fix", True)
    return cfg


def build_inputs(case):
    """-> dict of numpy arrays with the reference's input keys."""
    n = case["n"]
    (h0, w0), (h1, w1) = case["hw0"], case["hw1"]
    seed = case.get("iseed", 1)
    if (h0, w0) == (h1, w1):
        mk = W.smooth_images if case.get("images") == "smooth" else W.make_images
        im0, im1 = mk(n, h0, w0, seed)
    else:
        im0, _ = W.make_images(n, h0, w0, seed)
        im1, _ = W.make_images(n, h1, w1, seed + 1)
    data = {"image0": im0, "image1": im1}
    if "valid0" in case:  # MegaDepth-style padding: zero the padded area, coarse-resolution bool masks
        m0 = np.zeros((n, h0 // 8, w0 // 8), bool)
        m1 = np.zeros((n, h1 // 8, w1 // 8), bool)
        for b in range(n):
            vh, vw = case["valid0"][b]
            m0[b, : vh // 8, : vw // 8] = True
            data["image0"][b, :, vh:, :] = 0
            data["image0"][b, :, :, vw:] = 0
            vh, vw = case["valid1"][b]
            m1[b, : vh // 8, : vw // 8] = True
            data["image1"][b, :, vh:, :] = 0
            data["image1"][b, :, :, vw:] = 0
        data["mask0"], data["mask1"] = m0, m1
    if case.get("scales"):
        rs = np.random.RandomState(7)
        data["scale0"] = rs.uniform(1.0, 2.5, (n, 2)).astype(np.float32)
        data["scale1"] = rs.uniform(1.0, 2.5, (n, 2)).astype(np.float32)
    return data


# Stage-level cases for CoarseMatching alone: synthetic features with planted correspondences, strong
# enough that the Sinkhorn prefilter keeps some rows and drops others and that thr=0.2 has real survivors.
CM_CASES = [
    {"name": "cm_ds_planted", "n": 2, "hw0c": (10, 14), "hw1c": (12, 12), "thr": 0.2, "amp": 1.6, "frac": 0.6},
    {"name": "cm_ot_planted", "n": 2, "hw0c": (10, 14), "hw1c": (12, 12), "thr": 0.2, "amp": 4.0, "frac": 0.6,
     "match_type": "sinkhorn", "bin_score": 2.0},
    {"name": "cm_ot_planted_prefilter", "n": 2, "hw0c": (10, 14), "hw1c": (12, 12), "thr": 0.05, "amp": 3.0,
     "frac": 0.6, "match_type": "sinkhorn", "prefilter": True, "bin_score": 6.0},
    {"name": "cm_ot_planted_prefilter_masked", "n": 2, "hw0c": (12, 12), "hw1c": (10, 14), "thr": 0.05, "amp": 3.0,
     "frac": 0.6, "match_type": "sinkhorn", "prefilter": True, "bin_score": 6.0,
     "valid0c": [(12, 9), (10, 12)], "valid1c": [(8, 14), (10, 11)]},
]


def build_cm_inputs(case, C=256):
    """-> feat_c0 [n, L, C], feat_c1 [n, S, C] float32, optional bool masks [n, h, w]."""
    rs = np.random.RandomState(case.get("iseed", 11))
    n = case["n"]
    (h0, w0), (h1, w1) = case["hw0c"], case["hw1c"]
    L, S = h0 * w0, h1 * w1
    f0 = (rs.standard_normal((n, L, C)) * case["amp"]).astype(np.float32)
    f1 = (rs.standard_normal((n, S, C)) * case["amp"]).astype(np.float32)
    k = int(min(L, S) * case["frac"])
    for b in range(n):
        src = rs.permutation(L)[:k]
        dst = rs.permutation(S)[:k]
        noise = rs.uniform(0.05, 0.6, (k, 1)).astype(np.float32)  # graded match strength
        f1[b, dst] = f0[b, src] + noise * rs.standard_normal((k, C)).astype(np.float32) * case["amp"]
    out = {"feat_c0": f0, "feat_c1": f1}
    if "valid0c" in case:
        m0 = np.zeros((n, h0, w0), bool)
        m1 = np.zeros((n, h1, w1), bool)
        for b in range(n):
            m0[b, : case["valid0c"][b][0], : case["valid0c"][b][1]] = True
            m1[b, : case["valid1c"][b][0], : case["valid1c"][b][1]] = True
        out["mask0"], out["mask1"] = m0, m1
    return out


# Full-size cases of the BASELINE.json configs (GPU parity tests `tests/test_engine_gpu.py`; their oracle outputs
# can be precomputed on CPU with tools/precompute_oracle.py into the git-ignored tests/_oracle_cache/).
BASELINE_CASES = {
    "full": {"name": "full", "n": 1, "hw0": (480, 640), "hw1": (480, 640), "thr": 0.0, "images": "smooth"},
    "b8": {"name": "b8", "n": 8, "hw0": (480, 640), "hw1": (480, 640), "thr": 0.0, "images": "smooth"},
    "b8thr": {"name": "b8thr", "n": 8, "hw0": (480, 640), "hw1": (480, 640), "thr": 0.2, "images": "smooth"},
    "b8ot": {"name": "b8ot", "n": 8, "hw0": (480, 640), "hw1": (480, 640), "thr": 0.0, "images": "smooth",
             "match_type": "sinkhorn"},
    "ot_full": {"name": "ot_full", "n": 1, "hw0": (480, 640), "hw1": (480, 640), "thr": 0.0, "images": "smooth",
                "match_type": "sinkhorn"},
    "outdoor": {"name": "outdoor", "n": 1, "hw0": (832, 832), "hw1": (832, 832), "thr": 0.0, "images": "smooth",
                "valid0": [(832, 624)], "valid1": [(640, 832)], "scales": True},
    "out4": {"name": "out4", "n": 4, "hw0": (832, 832), "hw1": (832, 832), "thr": 0.0, "images": "smooth",
             "valid0": [(832, 624), (832, 832), (560, 832), (704, 768)],
             "valid1": [(640, 832), (768, 832), (832, 832), (832, 616)], "scales": True},
    "sweep240": {"name": "sweep", "n": 1, "hw0": (240, 320), "hw1": (240, 320), "thr": 0.0, "images": "smooth"},
    "sweep720": {"name": "sweep", "n": 1, "hw0": (720, 960), "hw1": (720, 960), "thr": 0.0, "images": "smooth"},
    "sweep960": {"name": "sweep", "n": 1, "hw0": (960, 1280), "hw1": (960, 1280), "thr": 0.0, "images": "smooth"},
}
