"""Generate the golden vectors that pin `oracle/loftr_oracle.py` (and, through it, the CUDA engine) to the
reference.  Runs ONLY in the authoring container: it imports the unmodified reference from /root/reference
(oracle/ref_import.py) and executes its forward on CPU in fp32.  Only OUTPUTS are stored; weights and
inputs are regenerated at test time from tests/golden/weights.py (frozen numpy RandomState streams).

    python tests/golden/make_golden.py            # rewrites tests/golden/*.npz
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from oracle import ref_import  # noqa: E402
import weights as W  # noqa: E402
from cases import CASES, CM_CASES, build_cfg, build_cm_inputs, build_inputs  # noqa: E402


def to_np(v):
    if isinstance(v, torch.Tensor):
        return v.detach().cpu().numpy()
    return np.asarray(v)


def run_case(ref, case):
    cfg = build_cfg(case)
    torch.manual_seed(0)
    model = ref.LoFTR(cfg).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    state = W.make_state(shapes, seed=case.get("wseed", 0))
    if "bin_score" in case:
        state["coarse_matching.bin_score"] = np.asarray(case["bin_score"], np.float32)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in state.items()})
    data = {k: torch.from_numpy(v) for k, v in build_inputs(case).items()}
    taps = {}

    def tap(name):
        def hook(_m, _inp, out):
            taps[name] = out
        return hook

    model.loftr_coarse.register_forward_hook(tap("coarse_tf"))
    model.fine_preprocess.register_forward_hook(tap("fine_pre"))
    model.loftr_fine.register_forward_hook(tap("fine_tf"))
    with torch.no_grad():
        model(data)
    out = {}
    for k in ["b_ids", "i_ids", "j_ids", "m_bids", "gt_mask", "mconf", "mkpts0_c", "mkpts1_c", "mkpts0_f", "mkpts1_f",
              "expec_f"]:
        out[k] = to_np(data[k])
    keep = case.get("keep", ())
    if "conf" in keep:
        out["conf_matrix"] = to_np(data["conf_matrix"])
    # strided samples of the big taps keep every fixture small but still position-sensitive
    out["feat_c0_s"], out["feat_c1_s"] = to_np(taps["coarse_tf"][0])[:, ::7, ::5], to_np(taps["coarse_tf"][1])[:, ::7, ::5]
    nfine = 6
    out["fine_pre0"], out["fine_pre1"] = to_np(taps["fine_pre"][0])[:nfine], to_np(taps["fine_pre"][1])[:nfine]
    if "fine_tf" in taps:
        out["fine_tf0"], out["fine_tf1"] = to_np(taps["fine_tf"][0])[:nfine], to_np(taps["fine_tf"][1])[:nfine]
    for k in ["hw0_i", "hw1_i", "hw0_c", "hw1_c", "hw0_f", "hw1_f"]:
        out[k] = np.asarray(tuple(data[k]), np.int64)
    # fp64 run of the same model for near-tie adjudication (SURVEY.md §7 hard part 2)
    m64 = ref.LoFTR(cfg).eval()
    m64.load_state_dict({k: torch.from_numpy(v) for k, v in state.items()})
    m64 = m64.double()
    d64 = {k: (torch.from_numpy(v).double() if v.dtype == np.float32 else torch.from_numpy(v))
           for k, v in build_inputs(case).items()}
    with torch.no_grad():
        m64(d64)
    c64 = d64["conf_matrix"]
    out["row_top2_f64"] = to_np(torch.topk(c64, 2, dim=2).values)   # [n, L, 2]
    out["col_top2_f64"] = to_np(torch.topk(c64, 2, dim=1).values.transpose(1, 2))  # [n, S, 2]
    out["b_ids_f64"], out["i_ids_f64"], out["j_ids_f64"] = to_np(d64["b_ids"]), to_np(d64["i_ids"]), to_np(d64["j_ids"])
    out["mconf_f64"], out["mkpts1_f_f64"] = to_np(d64["mconf"]), to_np(d64["mkpts1_f"])
    out["conf_max"] = np.asarray(float(data["conf_matrix"].max()))
    return out


def run_cm_case(ref, case):
    """CoarseMatching.forward alone on synthetic features (reference coarse_matching.py:87-148)."""
    from src.loftr.utils.coarse_matching import CoarseMatching
    cfg = build_cfg(case)["match_coarse"]
    inp = build_cm_inputs(case)
    outs = {}
    for tag, dt in (("", torch.float32), ("_f64", torch.float64)):
        mod = CoarseMatching(cfg).eval()
        if cfg["match_type"] == "sinkhorn":
            mod.bin_score.data = torch.tensor(float(case.get("bin_score", 1.0)))
        mod = mod.to(dt)
        (h0, w0), (h1, w1) = case["hw0c"], case["hw1c"]
        data = {"hw0_i": (h0 * 8, w0 * 8), "hw1_i": (h1 * 8, w1 * 8), "hw0_c": (h0, w0), "hw1_c": (h1, w1)}
        m0 = m1 = None
        if "mask0" in inp:
            data["mask0"], data["mask1"] = torch.from_numpy(inp["mask0"]), torch.from_numpy(inp["mask1"])
            m0, m1 = data["mask0"].flatten(-2), data["mask1"].flatten(-2)
        with torch.no_grad():
            mod(torch.from_numpy(inp["feat_c0"]).to(dt), torch.from_numpy(inp["feat_c1"]).to(dt), data, m0, m1)
        for k in ["b_ids", "i_ids", "j_ids", "mconf", "mkpts0_c", "mkpts1_c"]:
            outs[k + tag] = to_np(data[k])
        if tag == "":
            outs["conf_matrix"] = to_np(data["conf_matrix"])
        else:
            c64 = data["conf_matrix"]
            outs["row_top2_f64"] = to_np(torch.topk(c64, 2, dim=2).values)
            outs["col_top2_f64"] = to_np(torch.topk(c64, 2, dim=1).values.transpose(1, 2))
    return outs


def main():
    ref = ref_import.load_reference()
    torch.set_num_threads(8)
    for case in CASES:
        out = run_case(ref, case)
        path = os.path.join(HERE, case["name"] + ".npz")
        # conf matrices are stored in half the bytes where that loses nothing the tests use
        np.savez_compressed(path, **out)
        print(f"{case['name']}: M={len(out['b_ids'])} (fp64 M={len(out['b_ids_f64'])}) conf.max={float(out['conf_max']):.4f} "
              f"-> {os.path.getsize(path) / 1024:.0f} KiB")


def main_cm():
    ref = ref_import.load_reference()
    for case in CM_CASES:
        out = run_cm_case(ref, case)
        path = os.path.join(HERE, case["name"] + ".npz")
        np.savez_compressed(path, **out)
        nz = (out["conf_matrix"].sum(2) > 0).sum()
        print(f"{case['name']}: M={len(out['b_ids'])} (fp64 {len(out['b_ids_f64'])}) live rows={nz} "
              f"conf.max={out['conf_matrix'].max():.4f} -> {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main_cm()
    main()
