"""BEV rotated NMS (SURVEY.md 8f row 1): CPU pins of the oracle + GPU parity of dd3d_op_bev_nms / DO_BEV_NMS forward."""
import math
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from oracle import bev_nms_oracle as B


# ------------------------------------------------------------------------------------------------ independent clipper
def _rect_poly(box):
    return [(x, y) for x, y in B._vertices(tuple(float(v) for v in box))]


def _clip(subject, clip):
    """Sutherland-Hodgman clipping of convex polygons (independent of the Graham-scan formulation under test)."""
    def area2(p):
        return sum(p[i][0] * p[(i + 1) % len(p)][1] - p[(i + 1) % len(p)][0] * p[i][1] for i in range(len(p)))
    if area2(clip) < 0:
        clip = clip[::-1]
    out = subject
    for i in range(len(clip)):
        a, b = clip[i], clip[(i + 1) % len(clip)]
        inp, out = out, []
        if not inp:
            break

        def inside(p):
            return (b[0] - a[0]) * (p[1] - a[1]) - (b[1] - a[1]) * (p[0] - a[0]) >= 0

        def inter(p, q):
            d1 = (b[0] - a[0]) * (p[1] - a[1]) - (b[1] - a[1]) * (p[0] - a[0])
            d2 = (b[0] - a[0]) * (q[1] - a[1]) - (b[1] - a[1]) * (q[0] - a[0])
            t = d1 / (d1 - d2)
            return (p[0] + t * (q[0] - p[0]), p[1] + t * (q[1] - p[1]))
        s = inp[-1]
        for e in inp:
            if inside(e):
                if not inside(s):
                    out.append(inter(s, e))
                out.append(e)
            elif inside(s):
                out.append(inter(s, e))
            s = e
    if len(out) < 3:
        return 0.0
    return abs(sum(out[i][0] * out[(i + 1) % len(out)][1] - out[(i + 1) % len(out)][0] * out[i][1]
                   for i in range(len(out)))) / 2.0


def test_rotated_iou_closed_forms():
    assert abs(B.rotated_iou((0, 0, 4, 2, 0), (0, 0, 4, 2, 0)) - 1.0) < 1e-9
    assert abs(B.rotated_iou((0, 0, 4, 2, 30), (0, 0, 4, 2, 30)) - 1.0) < 1e-9
    # axis aligned, half overlap: inter 2x2=4, union 8+8-4
    assert abs(B.rotated_iou((0, 0, 4, 2, 0), (2, 0, 4, 2, 0)) - 4.0 / 12.0) < 1e-9
    # unit square vs itself rotated by 45 deg: intersection = regular octagon, area 2*(sqrt(2)-1)
    oct_area = 2.0 * (math.sqrt(2.0) - 1.0)
    assert abs(B.rotated_iou((0, 0, 1, 1, 0), (0, 0, 1, 1, 45)) - oct_area / (2.0 - oct_area)) < 1e-9
    assert B.rotated_iou((0, 0, 1, 1, 0), (5, 5, 1, 1, 10)) == 0.0
    # 90-degree rotation swaps w and h
    assert abs(B.rotated_iou((1, 2, 4, 2, 90), (1, 2, 2, 4, 0)) - 1.0) < 1e-9


def test_rotated_iou_vs_independent_clipper():
    rs = np.random.RandomState(0)
    for _ in range(300):
        b1 = (rs.randn() * 2, rs.randn() * 2, rs.rand() * 4 + 0.5, rs.rand() * 4 + 0.5, rs.rand() * 360 - 180)
        b2 = (rs.randn() * 2, rs.randn() * 2, rs.rand() * 4 + 0.5, rs.rand() * 4 + 0.5, rs.rand() * 360 - 180)
        inter = _clip(_rect_poly(b1), _rect_poly(b2))
        ref = inter / (b1[2] * b1[3] + b2[2] * b2[3] - inter)
        assert abs(B.rotated_iou(b1, b2) - ref) < 1e-7
        assert abs(B.rotated_iou(b1, b2) - B.rotated_iou(b2, b1)) < 1e-9


def _random_case(seed, n):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(n, 4, generator=g)
    q = q / q.norm(dim=1, keepdim=True)
    t = torch.randn(n, 3, generator=g) * 4 + torch.tensor([0, 0, 15.0])
    size = torch.rand(n, 3, generator=g) * 3 + 1
    cls = torch.randint(0, 3, (n, ), generator=g)
    score = torch.rand(n, generator=g)
    rs = np.random.RandomState(seed)
    pq = rs.randn(4)
    pq /= np.linalg.norm(pq)
    return dict(quat=q, tvec=t, size=size, cls=cls, score3d=score), pq.astype(np.float32), (rs.randn(3) * 10).astype(np.float32)


def test_bev_oracle_matches_golden():
    """Fixture written by oracle/gen_golden.py from the reference's own nuscenes_sample_aggregate (postprocessing.py)."""
    g = np.load(os.path.join(GOLDEN_DIR, "bev_nms.npz"))
    for c in range(int(g["num_cases"])):
        det, pq, pt = _random_case(100 + c, int(g[f"n{c}"]))
        keep = B.bev_nms_image(det, pq, pt, float(g["thr"]))
        assert np.array_equal(keep.numpy(), g[f"keep{c}"])
        q, t = B.to_global(det["quat"], det["tvec"], pq, pt)
        np.testing.assert_allclose(B.boxes3d_to_rotated_boxes(q, t, det["size"]).numpy(), g[f"rot{c}"], rtol=1e-4, atol=1e-4)


def test_bev_oracle_vs_live_reference():
    """Kept indices recorded from the reference's nuscenes_sample_aggregate (reference_checks.npz, oracle/gen_golden.py)."""
    g = np.load(os.path.join(GOLDEN_DIR, "reference_checks.npz"))
    for c in range(4):
        det, pq, pt = _random_case(7 + c, 40 + 5 * c)
        keep_ref = torch.from_numpy(g[f"bev{c}/keep"])
        assert torch.equal(B.bev_nms_image(det, pq, pt, 0.3), keep_ref)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("seed,n,post", [(0, 90, 1), (1, 128, 0), (2, 7, 1), (3, 0, 1)])
def test_bev_nms_kernel_vs_oracle(seed, n, post):
    import ctypes as C
    from dd3d_b200 import lib
    L = lib.load()
    cap, Bn = 128, 2
    K = torch.tensor([[[700.0, 0.0, 320.0], [0.0, 690.0, 180.0], [0.0, 0.0, 1.0]]]).repeat(Bn, 1, 1)
    inv_K = torch.linalg.inv(K)
    dets = torch.zeros(Bn, cap, 24)
    counts = torch.zeros(Bn, dtype=torch.int32)
    poses = torch.zeros(Bn, 7)
    cases = []
    for b in range(Bn):
        det, pq, pt = _random_case(seed * 10 + b, n)
        order = torch.argsort(det["score3d"], descending=True, stable=True)
        det = {k: v[order] for k, v in det.items()}
        # express tvec through (proj_ctr, depth) like the engine's records
        depth = det["tvec"][:, 2].clamp(min=1.0)
        tv = det["tvec"].clone()
        tv[:, 2] = depth
        uvw = tv @ K[b].T
        pc = uvw[:, :2] / uvw[:, 2:]
        det["tvec"] = (torch.cat([pc, torch.ones(n, 1)], 1) @ inv_K[b].T) * depth[:, None]
        g = torch.Generator().manual_seed(seed + 50 + b)
        xy = torch.rand(n, 2, generator=g) * 300
        det["box2d"] = torch.cat([xy, xy + torch.rand(n, 2, generator=g) * 80], 1)
        dets[b, :n, 0:4] = det["box2d"]
        dets[b, :n, 5] = det["score3d"]
        dets[b, :n, 8:12] = det["quat"]
        dets[b, :n, 12:14] = pc
        dets[b, :n, 14] = depth
        dets[b, :n, 15:18] = det["size"]
        dets.view(torch.int32)[b, :n, 6] = det["cls"].to(torch.int32)
        counts[b] = n
        poses[b, :4] = torch.tensor(pq)
        poses[b, 4:] = torch.tensor(pt)
        cases.append((det, pq, pt))
    sizes = torch.tensor([[360, 640, 360, 640], [360, 640, 180, 320]], dtype=torch.int32)
    d_d, d_c, d_K, d_p, d_s = dets.cuda(), counts.cuda(), K.reshape(Bn, 9).contiguous().cuda(), poses.cuda(), sizes.cuda()
    flags = torch.zeros(1, dtype=torch.int32, device="cuda")
    st = L.dd3d_op_bev_nms(C.c_void_p(d_d.data_ptr()), C.c_void_p(d_c.data_ptr()), C.c_void_p(d_K.data_ptr()),
                           C.c_void_p(d_p.data_ptr()), C.c_void_p(d_s.data_ptr()), C.c_void_p(flags.data_ptr()), Bn, cap,
                           0.3, post, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert st == 0
    torch.cuda.synchronize()
    assert int(flags.item()) == 0
    out, cnt = d_d.cpu(), d_c.cpu()
    for b, (det, pq, pt) in enumerate(cases):
        keep = B.bev_nms_image(det, pq, pt, 0.3)
        ref_box = det["box2d"][keep]
        ref_s = det["score3d"][keep]
        if post:
            sx, sy = sizes[b, 3].item() / sizes[b, 1].item(), sizes[b, 2].item() / sizes[b, 0].item()
            ref_box = ref_box.clone()
            ref_box[:, 0::2] = (ref_box[:, 0::2] * sx).clamp(0, sizes[b, 3].item())
            ref_box[:, 1::2] = (ref_box[:, 1::2] * sy).clamp(0, sizes[b, 2].item())
            ne = ((ref_box[:, 2] - ref_box[:, 0]) > 0) & ((ref_box[:, 3] - ref_box[:, 1]) > 0)
            ref_box, ref_s = ref_box[ne], ref_s[ne]
        m = int(cnt[b])
        assert m == ref_s.shape[0], (b, m, ref_s.shape[0])
        assert torch.equal(out[b, :m, 5], ref_s)  # same survivors in the same order
        np.testing.assert_allclose(out[b, :m, 0:4].numpy(), ref_box.numpy(), rtol=1e-6, atol=1e-4)


@pytest.mark.gpu
def test_forward_with_bev_nms_vs_oracle():
    """DO_BEV_NMS forward == oracle BEV NMS applied to the SAME model's pre-BEV detections (isolates the BEV step from
    the bf16 perturbation of the network), then detector_postprocess."""
    from dd3d_b200.config import get_cfg
    from dd3d_b200.meta_arch import DD3DB200
    from dd3d_b200.synthetic import make_state_dict
    from oracle.dd3d_oracle import DD3DOracle
    from oracle.gen_golden import case_inputs
    cfg = get_cfg("dla34", "kitti_3d")
    cfg.DD3D.INFERENCE.DO_BEV_NMS = True
    cfg.DD3D.INFERENCE.BEV_NMS_IOU_THRESH = 0.05
    sd = make_state_dict(cfg)
    inputs = case_inputs("dla34")
    poses = [([1.0, 0.0, 0.0, 0.0], [0.0, 0.0, 0.0]), ([0.9238795, 0.0, 0.3826834, 0.0], [3.0, -1.0, 2.0])]
    for x, p in zip(inputs, poses):
        x["pose"] = p
    model = DD3DB200(cfg).to("cuda")
    model.load_state_dict(sd)
    out = model(inputs)
    model.do_bev_nms = False
    model.postprocess_in_inference = False
    pre = model(inputs)
    removed = 0
    for b, (o, q) in enumerate(zip(out, pre)):
        pi = q["instances"]
        det = dict(quat=pi.pred_boxes3d.quat.cpu(), tvec=pi.pred_boxes3d.tvec.cpu(), size=pi.pred_boxes3d.size.cpu(),
                   score3d=pi.scores_3d.cpu(), cls=pi.pred_classes.cpu(), box2d=pi.pred_boxes.tensor.cpu())
        keep = B.bev_nms_image(det, poses[b][0], poses[b][1], 0.05)
        removed += len(pi) - len(keep)
        h, w = pi.image_size
        oh, ow = inputs[b].get("height", h), inputs[b].get("width", w)
        ref = DD3DOracle.postprocess({k: v[keep] for k, v in det.items()}, (h, w), (oh, ow))
        inst = o["instances"]
        assert tuple(inst.image_size) == (oh, ow)
        assert len(inst) == ref["box2d"].shape[0]
        assert torch.equal(inst.scores_3d.cpu(), ref["score3d"])
        np.testing.assert_allclose(inst.pred_boxes.tensor.cpu().numpy(), ref["box2d"].numpy(), rtol=1e-6, atol=1e-4)
    assert removed > 0  # the case must actually exercise suppression
