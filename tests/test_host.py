"""CPU-side tests: C-ABI surface, config / state_dict compatibility, error behaviour of the drop-in API."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import loftr_b200
from loftr_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "loftr_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(lb_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/loftr_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), "ctypes binding and header disagree"
    assert _lib.load().lb_version() >= 100


def test_struct_layouts_match_header_field_order():
    header = open(os.path.join(ROOT, "include", "loftr_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    for cls in (_lib.LbEncoderLayerWeights, _lib.LbTransformerState, _lib.LbCoarseMatchArgs,
                _lib.LbFinePreprocessArgs, _lib.LbFineMatchArgs, _lib.LbConvWeights, _lib.LbBackboneWeights):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cls.__name__, cls.__name__), header, re.S).group(1)
        names = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            decl = re.sub(r"\[[^\]]*\]", "", decl)   # array declarators: l1[4] -> l1
            first, *rest = decl.split(",")
            names.append(re.findall(r"[A-Za-z_0-9]+", first)[-1])
            names += [re.findall(r"[A-Za-z_0-9]+", r)[-1] for r in rest]
        assert names == [f[0] for f in cls._fields_], cls.__name__


def test_compute_without_gpu_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    model = loftr_b200.LoFTR(loftr_b200.get_cfg("indoor_ds")).eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        model({"image0": torch.rand(1, 1, 64, 64), "image1": torch.rand(1, 1, 64, 64)})
    # and the library itself refuses as well (no device)
    lib = _lib.load()
    assert lib.lb_split_planes(None, 4, 4, 4, None, None, 4, 0, None) != 0
    assert b"" != lib.lb_last_error()


def test_default_cfg_matches_reference_schema():
    d = loftr_b200.default_cfg
    assert d["coarse"]["temp_bug_fix"] is False and d["match_coarse"]["skh_prefilter"] is True
    assert "sparse_spvs" not in d["match_coarse"]
    c = loftr_b200.get_cfg("indoor_ot")
    assert c["match_coarse"]["match_type"] == "sinkhorn" and c["coarse"]["temp_bug_fix"] is True
    assert loftr_b200.get_cfg("outdoor_ds")["match_coarse"]["thr"] == 0.2


def test_state_dict_names_and_matcher_prefix():
    cfg = loftr_b200.get_cfg("indoor_ot")
    m = loftr_b200.LoFTR(cfg).eval()
    sd = m.state_dict()
    assert len(sd) == 212 and "coarse_matching.bin_score" in sd      # 211 + bin_score (SURVEY.md §9 V9)
    assert "pos_encoding.pe" not in sd                               # non-persistent buffer
    assert sd["loftr_coarse.layers.7.mlp.0.weight"].shape == (512, 512)
    assert sd["fine_preprocess.merge_feat.weight"].shape == (128, 256)
    assert sum(p.numel() for p in loftr_b200.LoFTR(loftr_b200.get_cfg("indoor_ds")).parameters()) == 11561456
    prefixed = {"matcher." + k: v.clone() for k, v in sd.items()}
    m2 = loftr_b200.LoFTR(cfg)
    m2.load_state_dict(prefixed)
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))


def test_training_mode_is_rejected():
    m = loftr_b200.LoFTR(loftr_b200.get_cfg("indoor_ds")).train()
    with pytest.raises(NotImplementedError):
        m({"image0": torch.rand(1, 1, 64, 64), "image1": torch.rand(1, 1, 64, 64)})


def test_backbone_16_4_variant_builds():
    cfg = loftr_b200.get_cfg("indoor_ds")
    cfg["resolution"] = (16, 4)
    cfg["resnetfpn"]["block_dims"] = [128, 196, 256, 512]
    from loftr_b200.backbone import build_backbone
    bb = build_backbone(cfg).eval()
    with torch.no_grad():
        c, f = bb(torch.rand(1, 1, 64, 96))
    assert c.shape == (1, 512, 4, 6) and f.shape == (1, 196, 16, 24)
    assert "layer4_outconv.weight" in bb.state_dict() and "layer2_outconv2.3.weight" in bb.state_dict()


def test_model_with_packed_caches_deepcopies_and_pickles():
    """The packed-weight caches hold ctypes structures with raw pointers; they must not enter copy / pickle state
    (the reference module can be deep-copied, pickled and passed to mp.spawn)."""
    import copy
    import pickle
    model = loftr_b200.LoFTR(loftr_b200.get_cfg("indoor_ds")).eval()
    arr = (_lib.LbEncoderLayerWeights * 2)()
    model.loftr_coarse._packed, model.loftr_coarse._packed_key = (arr, None, []), ("k",)
    model.fine_preprocess._packed, model.fine_preprocess._packed_key = {"x": arr}, ("k",)
    model._tc_backbone._packed, model._tc_backbone._key = (_lib.LbBackboneWeights(), []), ("k",)
    c = copy.deepcopy(model)
    p = pickle.loads(pickle.dumps(model))
    for m in (c, p):
        assert m.loftr_coarse._packed is None and m.fine_preprocess._packed is None and m._tc_backbone._packed is None
        assert m._tc_backbone.m is m.backbone
        assert set(m.state_dict()) == set(model.state_dict())
    assert model.loftr_coarse._packed is not None          # the original keeps its cache
    model.invalidate_packed()
    assert model.loftr_coarse._packed is None and model._tc_backbone._packed is None
    model.loftr_coarse._packed = (arr, None, [])
    model.load_state_dict(c.state_dict())
    assert model.loftr_coarse._packed is None
    model.loftr_coarse._packed = (arr, None, [])
    model.float()
    assert model.loftr_coarse._packed is None


def test_unsupported_shapes_fail_at_construction():
    cfg = loftr_b200.get_cfg("indoor_ds")
    cfg["coarse"]["nhead"] = 4
    with pytest.raises(ValueError, match="coarse transformer"):
        loftr_b200.LoFTR(cfg)
    cfg = loftr_b200.get_cfg("indoor_ds")
    cfg["fine_window_size"] = 7
    with pytest.raises(ValueError, match="fine windows"):
        loftr_b200.LoFTR(cfg)


def test_bench_clock_sampler_filters_by_timestamp():
    """bench.py's nvidia-smi sampler runs for the whole process; only rows stamped inside the timed region count
    (rows within 0.25 s of its end are the fallback when the region was shorter than one sampling period)."""
    import datetime
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    c = bench.ClockSampler.__new__(bench.ClockSampler)   # no nvidia-smi process
    c.proc = None
    now = datetime.datetime.now()
    c.t0, c.t1 = now, now + datetime.timedelta(seconds=0.3)

    def row(dt, clk, cap="Active"):
        ts = (now + datetime.timedelta(seconds=dt)).strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]
        return [ts, str(clk), "1965", "800.1", "Not Active", "Not Active", "Not Active", cap]

    c.rows = [row(-0.2, 1500), row(0.05, 1800), row(0.1, 1820), row(0.4, 1700, "Not Active")]
    s = c.summary()
    assert s["samples"] == 2 and s["sm_mhz"] == 1810.0 and s["sm_max_mhz"] == 1965.0
    assert s["reasons"] == ["sw_power_cap"] and s["sampled"] == "timed region"
    c.rows = [row(-0.6, 1500), row(0.4, 1700)]
    s = c.summary()
    assert s["samples"] == 1 and s["sm_mhz"] == 1700.0 and s["sampled"].startswith("within")
    c.rows = [["garbage"], row(-3.0, 1000)]
    assert c.summary()["samples"] == 0


def test_bench_dump_outputs_dtypes_and_sampling(tmp_path):
    """bench.py --dump-outputs: ids as float64, masks as float32, floats kept; over the byte limit every array keeps
    the same seeded rows, so that the files of two runs stay comparable row for row."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    m = 1000
    out = {"b_ids": torch.arange(m), "gt_mask": torch.zeros(m, dtype=torch.bool), "mconf": torch.rand(m),
           "mkpts0_f": torch.arange(2 * m, dtype=torch.float32).reshape(m, 2), "hw0_i": torch.Size([480, 640]), "bs": 8}
    bench.dump_outputs(out, str(tmp_path / "all"))
    got = {p.stem: np.load(p) for p in (tmp_path / "all").iterdir()}
    assert set(got) == {"b_ids", "gt_mask", "mconf", "mkpts0_f"}
    assert got["b_ids"].dtype == np.float64 and got["gt_mask"].dtype == np.float32
    assert got["mconf"].dtype == np.float32 and np.array_equal(got["mconf"], out["mconf"].numpy())
    limit = 8000
    for d in ("s1", "s2"):
        bench.dump_outputs(out, str(tmp_path / d), max_bytes=limit)
    s1 = {p.stem: np.load(p) for p in (tmp_path / "s1").iterdir()}
    s2 = {p.stem: np.load(p) for p in (tmp_path / "s2").iterdir()}
    assert 0 < sum(a.nbytes for a in s1.values()) <= limit
    assert all(np.array_equal(s1[k], s2[k]) for k in s1)
    rows = s1["b_ids"].astype(np.int64)
    assert (np.diff(rows) > 0).all() and np.array_equal(s1["mkpts0_f"], got["mkpts0_f"][rows])
