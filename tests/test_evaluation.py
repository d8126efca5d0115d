"""Evaluation harness (SURVEY.md §8(f) rank 3) against golden vectors produced by the reference's own
src/utils/metrics.py (tests/golden/make_golden_metrics.py): the numpy oracle and the product module
`loftr_b200.evaluation` (host-side aggregation + OpenCV RANSAC on CPU; epipolar errors through the CUDA kernel)."""
import os

import numpy as np
import pytest
import torch

import util
from metrics_cases import AGG_CASE, make_scene_batch
from oracle import metrics_oracle as MO

GOLD = util.load_golden("metrics_scenes")
SCENES = (("a", 0, 3), ("b", 1, 2))


# ------------------------------------------------------------------------------------------------ oracle vs reference
@pytest.mark.parametrize("tag,seed,n", SCENES)
def test_oracle_epipolar_errors_match_reference(tag, seed, n):
    sc = make_scene_batch(seed, n)
    got = MO.symmetrical_epipolar_errors(sc["mkpts0_f"], sc["mkpts1_f"], sc["m_bids"], sc["T_0to1"], sc["K0"], sc["K1"])
    np.testing.assert_allclose(got, GOLD[f"{tag}_epi_errs"], rtol=2e-4, atol=1e-9)


@pytest.mark.parametrize("tag,seed,n", SCENES)
def test_oracle_and_product_pose_errors_match_reference(tag, seed, n):
    import cv2
    from loftr_b200 import evaluation as E
    sc = make_scene_batch(seed, n)
    for impl in ("oracle", "product"):
        cv2.setRNGSeed(0)
        R_errs, t_errs, n_inl = [], [], []
        if impl == "product":
            data = {k: torch.from_numpy(v) for k, v in sc.items()}
            E.compute_pose_errors(data, pixel_thr=0.5, conf=0.99999)
            R_errs, t_errs, n_inl = data["R_errs"], data["t_errs"], [int(i.sum()) for i in data["inliers"]]
        else:
            for b in range(n):
                sel = sc["m_bids"] == b
                R, t, inl = MO.estimate_pose(sc["mkpts0_f"][sel], sc["mkpts1_f"][sel], sc["K0"][b], sc["K1"][b], 0.5)
                te, re_ = MO.relative_pose_error(sc["T_0to1"][b], R, t)
                R_errs.append(re_), t_errs.append(te), n_inl.append(int(inl.sum()))
        # same OpenCV, same RNG seed, same call sequence -> the RANSAC result is reproduced exactly
        np.testing.assert_allclose(R_errs, GOLD[f"{tag}_R_errs"], rtol=1e-6, atol=1e-6, err_msg=impl)
        np.testing.assert_allclose(t_errs, GOLD[f"{tag}_t_errs"], rtol=1e-6, atol=1e-6, err_msg=impl)
        assert n_inl == list(GOLD[f"{tag}_n_inliers"]), impl
        assert max(R_errs) < 2.0 and max(t_errs) < 10.0     # and it is a sensible pose: 80 % inliers with 0.4 px noise


@pytest.mark.parametrize("tag,seed,n", SCENES)
def test_relative_pose_error_matches_reference(tag, seed, n):
    import cv2
    from loftr_b200 import evaluation as E
    sc = make_scene_batch(seed, n)
    rs = np.random.RandomState(seed + 10)
    for b in range(n):
        T = sc["T_0to1"][b].astype(np.float64)
        Rp, _ = cv2.Rodrigues(rs.standard_normal(3) * 0.05)
        R, t = Rp @ T[:3, :3], T[:3, 3] + 0.05 * rs.standard_normal(3)
        for fn in (MO.relative_pose_error, E.relative_pose_error):
            np.testing.assert_allclose(fn(T, R, t), GOLD[f"{tag}_rpe_{b}"], rtol=1e-9, atol=1e-9)
    # pure-rotation ground truth below the ignore threshold: translation error is defined as 0  [metrics.py:18-19]
    T = np.eye(4)
    T[:3, 3] = 1e-4
    assert E.relative_pose_error(T, np.eye(3), np.array([1.0, 0, 0]), ignore_gt_t_thr=1e-3)[0] == 0
    assert MO.relative_pose_error(T, np.eye(3), np.array([1.0, 0, 0]), ignore_gt_t_thr=1e-3)[0] == 0


def test_aggregation_matches_reference():
    from loftr_b200 import evaluation as E
    for mod in (MO, E):
        agg = mod.aggregate_metrics(AGG_CASE(), epi_err_thr=5e-4)
        assert set(agg) == {"auc@5", "auc@10", "auc@20", "prec@5e-04"}
        for k, v in agg.items():
            np.testing.assert_allclose(v, GOLD["agg_" + k], rtol=1e-12, err_msg=f"{mod.__name__} {k}")
        auc = mod.error_auc(np.asarray(AGG_CASE()["R_errs"]), [5, 10, 20])
        for k, v in auc.items():
            np.testing.assert_allclose(v, GOLD["aucR_" + k], rtol=1e-12)
    assert E.epidist_prec([np.array([]), np.array([1e-5, 1.0])], [5e-4]) == [0.25]       # an empty pair counts as 0
    assert E.error_auc([np.inf, np.inf])["auc@20"] == 0.0                                 # every pose failed


def test_pair_list_loader_reads_reference_layout(tmp_path):
    """The loader understands the `assets/scannet_test_1500` layout (name [P,4] uint16, rel_pose [P,12], one 3x3
    intrinsic per scene); the reference's real list (a copy in tests/golden/scannet_test_1500) is parsed as well."""
    from loftr_b200 import evaluation as E
    names = np.array([[707, 0, 15, 585], [708, 1, 45, 105]], np.uint16)
    rel = np.arange(24, dtype=np.float32).reshape(2, 12)
    np.savez(tmp_path / "test.npz", name=names, rel_pose=rel)
    K = np.array([[575.0, 0, 320], [0, 578, 240], [0, 0, 1]])
    np.savez(tmp_path / "intrinsics.npz", scene0707_00=K, scene0708_01=K * 2)
    pairs = E.load_scannet_pair_list(tmp_path / "test.npz", tmp_path / "intrinsics.npz")
    assert [p["scene_id"] for p in pairs] == ["scene0707_00", "scene0708_01"]
    assert pairs[0]["pair_names"] == ("scene0707_00/color/15.jpg", "scene0707_00/color/585.jpg")
    assert pairs[1]["pose_names"][1] == "scene0708_01/pose/105.txt"
    np.testing.assert_array_equal(pairs[1]["T_0to1_from_list"][:3], rel[1].reshape(3, 4))
    np.testing.assert_array_equal(pairs[1]["T_0to1_from_list"][3], [0, 0, 0, 1])
    np.testing.assert_array_equal(pairs[1]["K"], (K * 2).astype(np.float32))
    ref = os.path.join(util.GOLDEN, "scannet_test_1500")
    real = E.load_scannet_pair_list(os.path.join(ref, "test.npz"), os.path.join(ref, "intrinsics.npz"))
    assert len(real) == 1500 and real[0]["scene_id"] == "scene0707_00" and real[0]["K"].shape == (3, 3)


# ------------------------------------------------------------------------------------------------ CUDA kernel
@pytest.mark.gpu
@pytest.mark.parametrize("tag,seed,n", SCENES)
def test_epipolar_error_kernel_matches_reference(tag, seed, n):
    from loftr_b200 import evaluation as E
    sc = make_scene_batch(seed, n)
    data = {k: torch.from_numpy(v).cuda() for k, v in sc.items()}
    E.compute_symmetrical_epipolar_errors(data)
    got = data["epi_errs"].cpu().numpy()
    assert got.dtype == np.float32 and got.shape == GOLD[f"{tag}_epi_errs"].shape
    np.testing.assert_allclose(got, GOLD[f"{tag}_epi_errs"], rtol=2e-4, atol=1e-9)
    # empty match list and a batch whose last pair has no match
    empty = {"mkpts0_f": torch.zeros(0, 2).cuda(), "mkpts1_f": torch.zeros(0, 2).cuda(), "m_bids": torch.zeros(0, dtype=torch.int64).cuda(),
             "T_0to1": data["T_0to1"], "K0": data["K0"], "K1": data["K1"]}
    E.compute_symmetrical_epipolar_errors(empty)
    assert empty["epi_errs"].shape == (0,)


@pytest.mark.gpu
def test_evaluation_pipeline_on_matcher_output():
    """matcher(batch) -> epipolar errors -> RANSAC pose -> aggregation runs end to end on the engine's own outputs
    (synthetic images: the numbers are meaningless, the plumbing and key contract are what is checked)."""
    from cases import build_inputs
    from loftr_b200 import evaluation as E
    case = {"name": "ev", "n": 2, "hw0": (96, 128), "hw1": (96, 128), "thr": 0.0, "images": "smooth"}
    model, _, _ = util.build_model(case, "cuda:0")
    data = {k: torch.from_numpy(v).cuda() for k, v in build_inputs(case).items()}
    sc = make_scene_batch(3, 2)
    for k in ("T_0to1", "K0", "K1"):
        data[k] = torch.from_numpy(sc[k]).cuda()
    model(data)
    E.compute_symmetrical_epipolar_errors(data)
    E.compute_pose_errors(data, pixel_thr=0.5, conf=0.99999)
    assert data["epi_errs"].shape == data["mconf"].shape and len(data["R_errs"]) == 2 and len(data["inliers"]) == 2
    ref = MO.symmetrical_epipolar_errors(*(data[k].cpu().numpy() for k in ("mkpts0_f", "mkpts1_f", "m_bids", "T_0to1", "K0", "K1")))
    np.testing.assert_allclose(data["epi_errs"].cpu().numpy(), ref, rtol=5e-4, atol=1e-9)
    bids = data["m_bids"].cpu().numpy()
    metrics = {"identifiers": ["p0", "p1"], "R_errs": data["R_errs"], "t_errs": data["t_errs"],
               "epi_errs": [data["epi_errs"].cpu().numpy()[bids == b] for b in range(2)]}
    agg = E.aggregate_metrics(metrics)
    assert set(agg) == {"auc@5", "auc@10", "auc@20", "prec@5e-04"} and all(0.0 <= v <= 1.0 for v in agg.values())
