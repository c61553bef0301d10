"""CPU suite (-m "not gpu"): pins the oracle against golden vectors recorded from the reference (oracle/gen_golden.py),
checks the host logic and that the C-ABI library loads and exports every declared symbol."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from dd3d_b200.arch import param_specs
from dd3d_b200.config import get_cfg
from dd3d_b200.synthetic import make_inputs, make_state_dict
from oracle.dd3d_oracle import (DD3DOracle, batched_nms_restated, matrix_to_quaternion, predictions_to_boxes3d,
                                quaternion_to_matrix)
from oracle.gen_golden import CASES, case_inputs
from util import det_key, match_by_key, quat_dist

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")


# ------------------------------------------------------------------------------------------------ known answers
def test_kat_predictions_to_boxes3d():
    """Known-answer vector produced by the reference's fcos3d.py:16-52 (values also quoted in SURVEY.md 8c)."""
    k = np.load(os.path.join(GOLDEN_DIR, "kat_boxes3d.npz"))
    cfg = get_cfg("dla34", "kitti_3d")
    inv_K = torch.linalg.inv(torch.tensor(k["K"]))
    out = predictions_to_boxes3d(
        torch.tensor(k["quat_in"]), torch.tensor(k["ctr_in"]), torch.tensor(k["depth_in"]), torch.tensor(k["size_in"]),
        torch.tensor(k["loc"]), inv_K, torch.tensor(k["canon"]), cfg.DD3D.FCOS3D)
    assert quat_dist(out["quat"], k["quat"]).max() < 1e-5
    np.testing.assert_allclose(out["proj_ctr"].numpy(), k["proj_ctr"], rtol=1e-6)
    np.testing.assert_allclose(out["depth"].numpy(), k["depth"].reshape(-1), rtol=1e-6)
    np.testing.assert_allclose(out["size"].numpy(), k["size"], rtol=1e-5)
    np.testing.assert_allclose(out["tvec"].numpy(), k["tvec"], rtol=1e-5, atol=1e-5)
    # the survey's quoted digits
    np.testing.assert_allclose(k["quat"][1], [0.41794351, -0.43590611, 0.57037115, 0.55676377], atol=1e-6)
    np.testing.assert_allclose(k["tvec"][2], [-64.92348480, 17.20170593, 80.0], atol=1e-4)


def test_quaternion_roundtrip():
    g = torch.Generator().manual_seed(0)
    q = torch.randn(256, 4, generator=g)
    q = q / q.norm(dim=1, keepdim=True)
    R = quaternion_to_matrix(q)
    assert (torch.bmm(R, R.transpose(1, 2)) - torch.eye(3)).abs().max() < 1e-5
    q2 = matrix_to_quaternion(R)
    assert quat_dist(q, q2).max() < 1e-5


def test_nms_restated_matches_torchvision():
    from torchvision.ops import batched_nms
    g = torch.Generator().manual_seed(1)
    n = 600
    xy = torch.rand(n, 2, generator=g) * 300
    wh = torch.rand(n, 2, generator=g) * 80 + 4
    boxes = torch.cat([xy, xy + wh], 1)
    scores = torch.rand(n, generator=g)
    cls = torch.randint(0, 5, (n, ), generator=g)
    for thr in (0.3, 0.6, 0.75):
        a = batched_nms_restated(boxes, scores, cls, thr)
        b = batched_nms(boxes, scores, cls, thr)
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ golden vectors
@pytest.mark.parametrize("arch", ["dla34", "v2_99"])
def test_oracle_matches_reference_golden(arch):
    """Oracle (fp32) vs the fixtures produced by the REAL reference forward (oracle/gen_golden.py)."""
    g = np.load(os.path.join(GOLDEN_DIR, f"golden_{arch}.npz"))
    cfg = get_cfg(arch, CASES[arch][0])
    orc = DD3DOracle(cfg, make_state_dict(cfg))
    out = orc.forward(case_inputs(arch))
    for b, o in enumerate(out):
        assert o["box2d"].shape[0] == g[f"boxes{b}"].shape[0]
        # same detections in the same order (NMS order = descending scores_3d)
        assert np.array_equal(o["cls"].numpy(), g[f"classes{b}"])
        assert np.array_equal(o["level"].numpy(), g[f"levels{b}"])
        np.testing.assert_allclose(o["box2d"].numpy(), g[f"boxes{b}"], rtol=1e-4, atol=1e-3)
        np.testing.assert_allclose(o["score"].numpy(), g[f"scores{b}"], rtol=1e-4)
        np.testing.assert_allclose(o["score3d"].numpy(), g[f"scores_3d{b}"], rtol=1e-4)
        assert quat_dist(o["quat"], g[f"quat{b}"]).max() < 1e-4
        np.testing.assert_allclose(o["tvec"].numpy(), g[f"tvec{b}"], rtol=1e-3, atol=1e-3)
        np.testing.assert_allclose(o["size"].numpy(), g[f"size{b}"], rtol=1e-4)


def test_bf16_emulation_stays_close_to_fp32():
    """The bf16-storage emulation (what the engine computes) must keep most detections of the fp32 reference."""
    arch = "dla34"
    cfg = get_cfg(arch, CASES[arch][0])
    sd = make_state_dict(cfg)
    inputs = case_inputs(arch)
    a = DD3DOracle(cfg, sd).forward(inputs)
    b = DD3DOracle(cfg, sd, emulate_bf16=True).forward(inputs)
    for x, y in zip(a, b):
        ka = [det_key(l, p, c) for l, p, c in zip(x["level"], x["loc"], x["cls"])]
        kb = [det_key(l, p, c) for l, p, c in zip(y["level"], y["loc"], y["cls"])]
        ia, ib = match_by_key(ka, kb)
        assert len(ia) >= 0.7 * len(ka)
        assert (x["box2d"][ia] - y["box2d"][ib]).abs().max() < 2.0  # pixels, boxes are tens of pixels wide
        assert (x["score3d"][ia] - y["score3d"][ib]).abs().max() < 0.05


# ------------------------------------------------------------------------------------------------ vs the reference
# reference_checks.npz holds, per case, the reference DD3D's state_dict inventory and its forward on
# make_inputs(1, 128, 256, 721.5, seed_base=7) with the same synthetic weights (oracle/gen_golden.py gen_reference_checks)
def reference_case(name):
    g = np.load(os.path.join(GOLDEN_DIR, "reference_checks.npz"))
    return {k.split("/", 1)[1]: (v if v.dtype.kind == "U" or v.ndim == 0 else torch.from_numpy(v))
            for k, v in g.items() if k.startswith(name + "/")}


def assert_reference_inventory(ref, cfg):
    specs = param_specs(cfg)
    inventory = dict(zip(ref["keys"].tolist(), ref["shapes"].tolist()))
    assert set(inventory) == set(specs), set(inventory) ^ set(specs)
    for k, (shape, _) in specs.items():
        assert inventory[k] == "x".join(map(str, shape)), k


@pytest.mark.parametrize("arch", ["dla34", "v2_99"])
def test_inventory_and_oracle_vs_live_reference(arch):
    cfg = get_cfg(arch, CASES[arch][0])
    ref = reference_case(f"inventory_{arch}")
    assert_reference_inventory(ref, cfg)
    out = DD3DOracle(cfg, make_state_dict(cfg)).forward(make_inputs(1, 128, 256, 721.5, seed_base=7))[0]
    assert ref["boxes"].shape[0] == out["box2d"].shape[0]
    if ref["boxes"].shape[0]:
        assert (ref["boxes"] - out["box2d"]).abs().max() < 1e-3
        assert (ref["scores_3d"] - out["score3d"]).abs().max() < 1e-5
        assert quat_dist(ref["quat"], out["quat"]).max() < 1e-4
        assert (ref["tvec"] - out["tvec"]).abs().max() < 1e-3


FLAG_CASES = [
    dict(FEATURE_LOCATIONS_OFFSET="half"),
    dict(PREDICT_DISTANCE=True),
    dict(PREDICT_ALLOCENTRIC_ROT=False),
    dict(SCALE_DEPTH_BY_FOCAL_LENGTHS=False),
    dict(FEATURE_LOCATIONS_OFFSET="half", PREDICT_DISTANCE=True, PREDICT_ALLOCENTRIC_ROT=False),
]


def apply_flags(cfg, flags):
    for k, v in flags.items():
        if k == "FEATURE_LOCATIONS_OFFSET":
            cfg.DD3D.FEATURE_LOCATIONS_OFFSET = v
        else:
            cfg.DD3D.FCOS3D[k] = v
    return cfg


@pytest.mark.parametrize("flags", FLAG_CASES, ids=lambda f: "+".join(f))
def test_oracle_decode_flags_vs_live_reference(flags):
    """The non-default decode switches the reference reads (core.py:38, fcos3d.py:36-47,306-312): feature-location offset
    "half", PREDICT_DISTANCE, egocentric quaternions, no focal-length depth scaling -- oracle == the reference's forward."""
    cfg = apply_flags(get_cfg("dla34", "kitti_3d"), flags)
    cfg.DD3D.FCOS2D.INFERENCE.PRE_NMS_THRESH = 0.03
    ref = reference_case(f"flags{FLAG_CASES.index(flags)}")
    out = DD3DOracle(cfg, make_state_dict(cfg)).forward(make_inputs(1, 128, 256, 721.5, seed_base=7))[0]
    assert ref["boxes"].shape[0] == out["box2d"].shape[0] > 5
    assert (ref["boxes"] - out["box2d"]).abs().max() < 1e-3
    assert (ref["locations"] - out["loc"]).abs().max() == 0
    assert (ref["scores_3d"] - out["score3d"]).abs().max() < 1e-5
    assert quat_dist(ref["quat"], out["quat"]).max() < 1e-4
    assert (ref["depth"] - out["depth"]).abs().max() < 1e-3
    assert (ref["tvec"] - out["tvec"]).abs().max() < 1e-3


HEAD_CASES = [  # head configurations no shipped experiment uses (VERDICT r1 missing #2)
    dict(THRESH_WITH_CTR=False),
    dict(FCOS3D_USE_SCALE=False),
    dict(FCOS2D_USE_SCALE=False),
    dict(CLASS_AGNOSTIC_BOX3D=True),
    dict(PER_LEVEL_PREDICTORS=True),
    dict(BOX3D_ON=False),
    dict(THRESH_WITH_CTR=False, FCOS3D_USE_SCALE=False, FCOS2D_USE_SCALE=False, CLASS_AGNOSTIC_BOX3D=True,
         PER_LEVEL_PREDICTORS=True),
]


def apply_head_flags(cfg, flags):
    for k, v in flags.items():
        if k == "THRESH_WITH_CTR":
            cfg.DD3D.FCOS2D.INFERENCE.THRESH_WITH_CTR = v
        elif k == "FCOS3D_USE_SCALE":
            cfg.DD3D.FCOS3D.USE_SCALE = v
        elif k == "FCOS2D_USE_SCALE":
            cfg.DD3D.FCOS2D.USE_SCALE = v
        elif k == "BOX3D_ON":
            cfg.MODEL.BOX3D_ON = v
        else:
            cfg.DD3D.FCOS3D[k] = v
    return cfg


@pytest.mark.parametrize("flags", HEAD_CASES, ids=lambda f: "+".join(f))
def test_oracle_head_configs_vs_live_reference(flags):
    """THRESH_WITH_CTR False (fcos2d.py:280-290), USE_SCALE False (fcos2d.py:100-108,145-152; fcos3d.py:116,128-139,175-180),
    CLASS_AGNOSTIC_BOX3D (fcos3d.py:103,333-352), PER_LEVEL_PREDICTORS (fcos3d.py:104,166), BOX3D_ON False (core.py:34-40,
    117-125): the parameter inventory equals the reference's state_dict and the oracle equals the reference's forward."""
    cfg = apply_head_flags(get_cfg("dla34", "kitti_3d"), flags)
    cfg.DD3D.FCOS2D.INFERENCE.PRE_NMS_THRESH = 0.03
    ref = reference_case(f"head{HEAD_CASES.index(flags)}")
    assert_reference_inventory(ref, cfg)
    out = DD3DOracle(cfg, make_state_dict(cfg)).forward(make_inputs(1, 128, 256, 721.5, seed_base=7))[0]
    assert ref["boxes"].shape[0] == out["box2d"].shape[0] > 5
    assert (ref["boxes"] - out["box2d"]).abs().max() < 1e-3
    assert (ref["scores"] - out["score"]).abs().max() < 1e-5
    assert torch.equal(ref["classes"], out["cls"]) and torch.equal(ref["levels"], out["level"])
    assert bool(ref["has_box3d"]) == bool(cfg.MODEL.BOX3D_ON)
    if cfg.MODEL.BOX3D_ON:
        assert (ref["scores_3d"] - out["score3d"]).abs().max() < 1e-5
        assert quat_dist(ref["quat"], out["quat"]).max() < 1e-4
        assert (ref["depth"] - out["depth"]).abs().max() < 1e-3
        assert ((ref["size"] - out["size"]).abs() / out["size"].abs().clamp(min=1e-3)).max() < 1e-4
        assert (ref["tvec"] - out["tvec"]).abs().max() < 1e-3
    else:
        assert "scores_3d" not in ref and "quat" not in ref


# ------------------------------------------------------------------------------------------------ host logic / ABI
def test_identity_intrinsics_raises():
    cfg = get_cfg("dla34", "kitti_3d")
    inputs = make_inputs(1, 128, 128, 700.0)
    inputs[0]["intrinsics"] = torch.eye(3)
    with pytest.raises(ValueError, match="Intrinsics is Identity"):
        DD3DOracle(cfg, make_state_dict(cfg)).preprocess(inputs)
    from dd3d_b200.meta_arch import DD3DB200
    m = DD3DB200(cfg)
    with pytest.raises(ValueError, match="Intrinsics is Identity"):
        m._gather_inputs(inputs, torch.device("cpu"))


def test_unknown_builder_raises_keyerror():
    cfg = get_cfg("dla34", "kitti_3d")
    cfg.FE.BUILDER = "build_something_else"
    from dd3d_b200.meta_arch import DD3DB200
    with pytest.raises(KeyError):
        DD3DB200(cfg)


def test_state_dict_contract():
    from dd3d_b200.meta_arch import DD3DB200
    cfg = get_cfg("v2_99", "nuscenes")
    m = DD3DB200(cfg)
    sd = make_state_dict(cfg)
    assert set(m.state_dict().keys()) == set(sd.keys())
    res = m.load_state_dict(sd)
    assert not res.missing_keys and not res.unexpected_keys
    bad = dict(sd)
    bad["fcos2d_head.cls_logits.weight"] = torch.zeros(3, 256, 3, 3)
    with pytest.raises(RuntimeError, match="size mismatch"):
        m.load_state_dict(bad)
    with pytest.raises(RuntimeError, match="CUDA"):
        m._engine()  # CPU device: must fail loudly, never fall back


def test_gather_inputs_ragged_batch():
    from dd3d_b200.meta_arch import DD3DB200
    cfg = get_cfg("dla34", "kitti_3d")
    m = DD3DB200(cfg)
    inputs = case_inputs("dla34")
    batch, K, sizes, shape, is_u8 = m._gather_inputs(inputs, torch.device("cpu"))
    assert is_u8 and batch.dtype == torch.uint8 and shape == (2, 192, 320)
    assert sizes.tolist() == [[192, 320, 192, 320], [171, 286, 342, 572]]
    assert batch[1, :, 171:, :].sum() == 0 and batch[1, :, :, 286:].sum() == 0
    m.postprocess_in_inference = False
    _, _, sizes, _, _ = m._gather_inputs(inputs, torch.device("cpu"))
    assert sizes.tolist()[1] == [171, 286, 171, 286]


def test_cabi_library_exports_every_declared_symbol():
    """The header is the contract: every dd3d_* function it declares must be exported and bound (no compute calls)."""
    from dd3d_b200 import lib
    header = open(os.path.join(ROOT, "include", "dd3d_b200.h")).read()
    declared = set(re.findall(r"\b(dd3d_[a-z0-9_]+)\s*\(", header))
    assert declared == set(lib.SIGNATURES.keys()), declared ^ set(lib.SIGNATURES.keys())
    L = lib.load()
    for name in declared:
        assert hasattr(L, name)
    import ctypes
    assert ctypes.sizeof(lib.ModelDesc) == 4 * (2 + 3 + 3 + 1 + 1 + 3 + 1 + 2 + 1 + 1 + 1 + 1 + 48 + 1 + 1 + 1 + 6)  # + act_dtype + 6 head switches
    assert ctypes.sizeof(lib.TtaView) == 4 * (1 + 1 + 2 + 2 + 9 + 9)  # dd3d_tta_view
    assert lib.DET_WORDS * 4 == 96  # dd3d_det


def test_tile_decode_fast_division():
    """conv_igemm.cu fast_div (fp32 reciprocal estimate + one correction) restated in numpy: exact for every tile index
    the kernel can see (x < 2^24, launch_conv refuses more) and every divisor a plan can produce."""
    import numpy as np
    rs = np.random.RandomState(0)
    for d in [1, 2, 3, 7, 50, 57, 200, 750, 2850, 11400, 19999] + [int(v) for v in rs.randint(1, 20000, size=40)]:
        inv = np.float32(1.0) / np.float32(d)
        x = np.concatenate([rs.randint(0, 1 << 24, size=50000), [0, d - 1, d, 2 * d - 1, (1 << 24) - 1]]).astype(np.int64)
        q = np.trunc(x.astype(np.float32) * inv).astype(np.int64)
        r = x - q * d
        q = q + (r >= d) - (r < 0)
        assert np.array_equal(q, x // d), d


def test_cabi_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import ctypes as C
    from dd3d_b200 import lib
    L = lib.load()
    desc = lib.desc_from_cfg(get_cfg("dla34", "kitti_3d"))
    h = C.c_void_p()
    st = L.dd3d_create(C.byref(desc), C.byref(h))
    assert st == -3 and not h.value  # DD3D_ERR_CUDA
    assert L.dd3d_last_error(None)
