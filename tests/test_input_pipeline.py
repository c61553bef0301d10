"""GPU input pipeline (SURVEY.md 8f row 3): ResizeShortestEdge + PIL-exact bilinear resampling + intrinsics rescale fused
with the model preprocess.  Integer / byte work: every comparison here is bit-exact."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from oracle import input_oracle as IO

# ((raw h, w), (resized h, w)): nuScenes and KITTI test-time shapes (small crops of them for speed), up- and down-scaling,
# single-axis resizes, strong shrink (long antialiasing kernels)
RESIZE_CASES = [((90, 160), (89, 159)), ((75, 248), (77, 254)), ((74, 244), (96, 317)), ((120, 100), (60, 50)),
                ((64, 80), (160, 200)), ((97, 131), (41, 131)), ((50, 70), (50, 33)), ((150, 200), (38, 45))]
MEAN, STD = [103.530, 116.280, 123.675], [57.375, 57.120, 58.395]


def raw_image(seed, h, w):
    rs = np.random.RandomState(1000 + seed)
    img = rs.randint(0, 256, (h, w, 3)).astype(np.float32)
    yy, xx = np.mgrid[:h, :w]
    img = 0.6 * img + 0.4 * 255.0 * (0.5 + 0.5 * np.sin(0.11 * xx + 0.07 * yy))[..., None]
    return img.round().clip(0, 255).astype(np.uint8)


# ------------------------------------------------------------------------------------------------ CPU
def test_resize_restatement_matches_golden_and_pillow():
    g = np.load(os.path.join(GOLDEN_DIR, "input_pipeline.npz"))
    try:
        from PIL import Image
    except ImportError:  # the fixture was written by Pillow
        Image = None
    for c, ((h, w), (nh, nw)) in enumerate(RESIZE_CASES):
        img = raw_image(c, h, w)
        out = IO.pil_resize_bilinear(img, nh, nw)
        assert np.array_equal(out, g[f"img{c}"]), f"case {c}"
        if Image is not None:
            assert np.array_equal(out, np.asarray(Image.fromarray(img).resize((nw, nh), Image.BILINEAR)))
        K = np.float32([[721.5377, 0, 609.5593], [0, 721.5377, 172.854], [0, 0, 1]])
        assert np.array_equal(IO.scale_intrinsics(K, h, w, nh, nw), g[f"K{c}"])


def test_resize_full_size_matches_pillow():
    Image = pytest.importorskip("PIL.Image")
    for (h, w), size in [((900, 1600), 896), ((375, 1242), 384)]:
        nh, nw = IO.resize_shortest_edge_shape(h, w, size, 100000)
        img = raw_image(50, h, w)
        assert np.array_equal(IO.pil_resize_bilinear(img, nh, nw), np.asarray(Image.fromarray(img).resize((nw, nh), Image.BILINEAR)))


def test_shape_rule_and_cabi_agree():
    """ResizeShortestEdge.get_transform: known shapes of the shipped configs + the C entry point over a sweep."""
    assert IO.resize_shortest_edge_shape(900, 1600, 896, 100000) == (896, 1593)  # dd3d_nusc_v99.yaml:43
    assert IO.resize_shortest_edge_shape(375, 1242, 384, 100000) == (384, 1272)  # dd3d_kitti_dla34.yaml:34
    assert IO.resize_shortest_edge_shape(370, 1224, 384, 100000) == (384, 1270)
    assert IO.resize_shortest_edge_shape(1000, 500, 400, 600) == (600, 300)      # max_size bites
    assert IO.resize_shortest_edge_shape(123, 457, 0, 0) == (123, 457)
    from dd3d_b200 import lib
    L = lib.load()
    rs = np.random.RandomState(0)
    nh, nw = C.c_int32(), C.c_int32()
    for _ in range(2000):
        h, w = int(rs.randint(16, 2000)), int(rs.randint(16, 2000))
        size, mx = int(rs.randint(16, 1200)), int(rs.choice([100000, 1333, 800]))
        assert L.dd3d_resize_shape(h, w, size, mx, C.byref(nh), C.byref(nw)) == 0
        assert (nh.value, nw.value) == IO.resize_shortest_edge_shape(h, w, size, mx), (h, w, size, mx)


def test_intrinsics_rescale_vs_live_reference():
    """The reference's ResizeTransform.apply_intrinsics on the two full-size shapes (reference_checks.npz)."""
    g = np.load(os.path.join(GOLDEN_DIR, "reference_checks.npz"))
    K = np.float32([[1266.4, 0, 816.3], [0, 1266.4, 491.5], [0, 0, 1]])
    for i, ((h, w), (nh, nw)) in enumerate([((900, 1600), (896, 1593)), ((375, 1242), (384, 1272))]):
        assert np.array_equal(g[f"intrinsics{i}/K"], IO.scale_intrinsics(K, h, w, nh, nw))


# ------------------------------------------------------------------------------------------------ GPU
def _expected_input(resized_list, Hp, Wp):
    out = torch.zeros(len(resized_list), Hp, Wp, 4, dtype=torch.bfloat16)
    m, s = torch.tensor(MEAN), torch.tensor(STD)
    for b, r in enumerate(resized_list):
        v = (torch.from_numpy(r).float() - m) / s
        out[b, :r.shape[0], :r.shape[1], :3] = v.to(torch.bfloat16)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("cases,flip", [([0], 0), ([1, 2], 0), ([3, 4, 5], 1), ([6, 7], 0), ([0, 1, 2, 3, 4, 5, 6, 7], 1)])
def test_resize_preprocess_kernel_bit_exact(cases, flip):
    """dd3d_op_resize_preprocess == PIL-exact oracle resize (then np.flip(axis=1) for the test-time-augmentation flip on
    every other image) followed by (x - mean) / std in fp32, rounded to bf16, zero padded; ragged batches share one slot
    size."""
    from dd3d_b200 import lib
    L = lib.load()
    raws = [raw_image(c, *RESIZE_CASES[c][0]) for c in cases]
    news = [RESIZE_CASES[c][1] for c in cases]
    Bn = len(cases)
    raw_h, raw_w = max(r.shape[0] for r in raws), max(r.shape[1] for r in raws)
    Hp = (max(n[0] for n in news) + 63) // 64 * 64
    Wp = (max(n[1] for n in news) + 63) // 64 * 64
    buf = torch.zeros(Bn, raw_h, raw_w, 3, dtype=torch.uint8)
    for b, r in enumerate(raws):
        buf[b, :r.shape[0], :r.shape[1]] = torch.from_numpy(r)
    raw_sizes = torch.tensor([[r.shape[0], r.shape[1]] for r in raws], dtype=torch.int32)
    new_sizes = torch.tensor(news, dtype=torch.int32)
    d_raw = buf.cuda()
    d_out = torch.full((Bn, Hp, Wp, 4), 7.0, dtype=torch.bfloat16, device="cuda")
    mean, std = (C.c_float * 3)(*MEAN), (C.c_float * 3)(*STD)
    flips = torch.tensor([(b % 2 == 0) and flip for b in range(Bn)], dtype=torch.int32)
    st = L.dd3d_op_resize_preprocess(C.c_void_p(d_raw.data_ptr()), raw_h, raw_w, C.c_void_p(raw_sizes.data_ptr()),
                                     C.c_void_p(new_sizes.data_ptr()), C.c_void_p(flips.data_ptr()) if flip else None,
                                     C.c_void_p(d_out.data_ptr()), Bn, Hp, Wp, mean, std,
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert st == 0
    torch.cuda.synchronize()
    resized = [IO.pil_resize_bilinear(r, *n) for r, n in zip(raws, news)]
    resized = [np.ascontiguousarray(np.flip(r, axis=1)) if f else r for r, f in zip(resized, flips.tolist())]
    exp = _expected_input(resized, Hp, Wp)
    assert torch.equal(d_out.cpu().view(torch.int16), exp.view(torch.int16))


@pytest.mark.gpu
def test_forward_raw_equals_mapper_then_forward():
    """forward_raw(raw) == forward([DefaultDatasetMapper-oracle(raw)]): identical detections, bit for bit (the resized
    pixels are bit-identical, so the two runs of the same engine see the same input tensor)."""
    from dd3d_b200.config import get_cfg
    from dd3d_b200.meta_arch import DD3DB200
    from dd3d_b200.synthetic import make_inputs, make_state_dict
    cfg = get_cfg("dla34", "kitti_3d")
    cfg.INPUT.RESIZE.MIN_SIZE_TEST = 192
    cfg.DD3D.FCOS2D.INFERENCE.PRE_NMS_THRESH = 0.02  # the resampled noise images score lower than the calibration set
    model = DD3DB200(cfg).to("cuda")
    model.load_state_dict(make_state_dict(cfg))
    base = make_inputs(2, 188, 620, 721.5)  # KITTI-like aspect; the second image is a little smaller (ragged batch)
    raws = []
    for i, x in enumerate(base):
        img = x["image"].permute(1, 2, 0).contiguous().numpy()
        if i == 1:
            img = np.ascontiguousarray(img[:183, :606])
        raws.append({"image_hwc": img, "intrinsics": x["intrinsics"]})
    out_raw = model.forward_raw(raws)
    mapped = [IO.map_input(r, cfg.INPUT.RESIZE.MIN_SIZE_TEST, cfg.INPUT.RESIZE.MAX_SIZE_TEST) for r in raws]
    assert tuple(mapped[0]["image"].shape) == (3, 192, 633)
    out_map = model(mapped)
    total = 0
    for a, b, r in zip(out_raw, out_map, raws):
        ia, ib = a["instances"], b["instances"]
        assert tuple(ia.image_size) == tuple(ib.image_size) == r["image_hwc"].shape[:2]  # back at the raw resolution
        assert len(ia) == len(ib)
        total += len(ia)
        for f in ("scores", "scores_3d", "pred_classes", "fpn_levels", "locations"):
            assert torch.equal(ia.get(f), ib.get(f)), f
        assert torch.equal(ia.pred_boxes.tensor, ib.pred_boxes.tensor)
        assert torch.equal(ia.pred_boxes3d.vectorize(), ib.pred_boxes3d.vectorize())
    assert total > 5
