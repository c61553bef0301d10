"""NuscenesDD3D (SURVEY.md 8f row 2; nuscenes_dd3d.py:300-469): attribute / speed predictors on the cls tower and the
cross-camera sample aggregation.  CPU: oracle pinned against fixtures written by the real reference.  GPU: dd3d_op_sample_aggregate and NuscenesDD3DB200.forward."""
import math
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from oracle import bev_nms_oracle as B
from util import det_key, match_by_key, quat_dist, rel_err

AGG_TOKENS = ["a", "a", "a", "b", "b", "b", "a", "a", "a", "b", "b", "b"]  # groups with non-contiguous members


def aggregate_case(seed, num_classes=3):
    """12 images (2 samples x 6 cameras, interleaved) of seeded random 3-D detections sorted by scores_3d, camera poses
    of a nearly parallel rig so that boxes of different cameras overlap in BEV."""
    g = torch.Generator().manual_seed(seed)
    rs = np.random.RandomState(seed)
    dets, poses = [], []
    for i, tok in enumerate(AGG_TOKENS):
        n = int(rs.randint(20, 101)) if i != 5 else 0  # one empty image
        q = torch.randn(n, 4, generator=g)
        q = q / q.norm(dim=1, keepdim=True)
        t = torch.randn(n, 3, generator=g) * torch.tensor([5.0, 0.5, 5.0]) + torch.tensor([0.0, 0.0, 18.0])
        size = torch.rand(n, 3, generator=g) * 3 + 1
        cls = torch.randint(0, num_classes, (n, ), generator=g)
        score = torch.rand(n, generator=g).sort(descending=True).values
        dets.append(dict(quat=q, tvec=t, size=size, cls=cls, score3d=score))
        yaw = math.radians(rs.uniform(-6, 6) + (40.0 if tok == "b" else 0.0))
        # camera (x right, y down, z forward) -> world: forward along (cos yaw, sin yaw, 0)
        R = np.array([[math.sin(yaw), 0.0, math.cos(yaw)], [-math.cos(yaw), 0.0, math.sin(yaw)], [0.0, -1.0, 0.0]])
        from dd3d_b200.structures import matrix_to_quaternion_wxyz
        pq = matrix_to_quaternion_wxyz(torch.tensor(R))
        pt = [float(v) for v in rs.randn(3) * 0.5 + (np.array([50.0, -20.0, 0.0]) if tok == "b" else 0.0)]
        poses.append((pq, pt))
    order = {t: k for k, t in enumerate(dict.fromkeys(AGG_TOKENS))}
    return dets, [order[t] for t in AGG_TOKENS], poses


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("case,max_dets", [(0, 1000), (1, 150)])
def test_sample_aggregate_oracle_matches_golden(case, max_dets):
    """Fixture from the reference's own nuscenes_sample_aggregate (oracle/gen_golden.py)."""
    g = np.load(os.path.join(GOLDEN_DIR, "sample_aggregate.npz"))
    dets, gids, poses = aggregate_case(7 + case)
    out = B.sample_aggregate(dets, gids, poses, 0.3, max_dets)
    total = 0
    for i, (d, o) in enumerate(zip(dets, out)):
        keep = g[f"keep{case}_{i}"]
        total += len(keep)
        assert torch.equal(o["score3d"], d["score3d"][torch.as_tensor(keep, dtype=torch.long)])
        assert quat_dist(o["quat_global"], g[f"quat{case}_{i}"]).max().item() < 1e-5 if len(keep) else True
        np.testing.assert_allclose(o["tvec_global"].numpy(), g[f"tvec{case}_{i}"].reshape(-1, 3), rtol=1e-5, atol=1e-4)
    assert total <= max_dets
    if max_dets == 150:
        assert total == 150  # the cap must bite in this case
    else:
        assert total < sum(d["quat"].shape[0] for d in dets)  # and suppression must happen in the other


def test_sample_aggregate_oracle_vs_live_reference():
    """Kept indices recorded from the reference's nuscenes_sample_aggregate (reference_checks.npz, oracle/gen_golden.py)."""
    g = np.load(os.path.join(GOLDEN_DIR, "reference_checks.npz"))
    dets, gids, poses = aggregate_case(3)
    out = B.sample_aggregate(dets, gids, poses, 0.3, 200)
    assert len(out) == len(dets) == len([k for k in g.files if k.startswith("aggregate/keep")])
    for i, (d, o) in enumerate(zip(dets, out)):
        assert torch.equal(o["score3d"], d["score3d"][torch.from_numpy(g[f"aggregate/keep{i}"])])


def _check_against_golden(out, g, nimg, box_tol, exact_sets):
    matched = total = 0
    for b in range(nimg):
        d = out[b]
        ka = [det_key(l, loc, c) for l, loc, c in zip(d["level"], d["loc"], d["cls"])]
        kb = [det_key(l, loc, c) for l, loc, c in zip(g[f"levels{b}"], g[f"locations{b}"], g[f"classes{b}"])]
        if exact_sets:
            assert sorted(ka) == sorted(kb), f"image {b}: detection sets differ"
        ia, ib = match_by_key(ka, kb)
        matched += len(ia)
        total += len(kb)
        if not len(ia):
            continue
        assert rel_err(d["box2d"][ia], g[f"boxes{b}"][ib], floor=32.0) < box_tol
        assert rel_err(d["score3d"][ia], g[f"scores_3d{b}"][ib], floor=0.05) < box_tol * 4
        assert rel_err(d["speed"][ia], g[f"speed{b}"][ib], floor=1.0) < box_tol * 4
        assert rel_err(d["tvec_global"][ia], g[f"tvec_global{b}"][ib], floor=1.0) < box_tol * 4
        assert quat_dist(d["quat_global"][ia], g[f"quat_global{b}"][ib]).max().item() < box_tol * 8
        agree = (torch.as_tensor(d["attr"])[ia] == torch.as_tensor(g[f"attr{b}"])[ib]).float().mean().item()
        assert agree >= (1.0 if exact_sets else 0.9)
    return matched, total


def test_nuscenes_oracle_matches_reference_golden():
    """fp32 oracle == the reference's NuscenesDD3D.forward on one synthetic 6-camera sample (tests/golden)."""
    from dd3d_b200.config import get_cfg
    from dd3d_b200.synthetic import make_state_dict
    from oracle.dd3d_oracle import DD3DOracle
    from oracle.gen_golden import NUSC_CASE, nusc_case_inputs
    arch = NUSC_CASE[0]
    g = np.load(os.path.join(GOLDEN_DIR, f"golden_nusc_{arch}.npz"))
    cfg = get_cfg(arch, "nuscenes", meta_arch="NuscenesDD3D")
    inputs = nusc_case_inputs()
    out = DD3DOracle(cfg, make_state_dict(cfg)).forward(inputs)
    matched, total = _check_against_golden(out, g, len(inputs), 1e-3, exact_sets=True)
    assert matched == total > 50
    for b in range(len(inputs)):
        assert tuple(int(v) for v in g[f"image_size{b}"]) == (inputs[b]["height"], inputs[b]["width"]) == (256, 384)


def test_nuscenes_group_size_error():
    """get_group_idxs (postprocessing.py:111-119): a sample without exactly 6 images is an error."""
    from dd3d_b200.meta_arch import group_indices
    assert group_indices(["x"] * 6 + ["y"] * 6, 6) == [0] * 6 + [1] * 6
    assert group_indices(AGG_TOKENS, 6) == [0, 0, 0, 1, 1, 1, 0, 0, 0, 1, 1, 1]
    with pytest.raises(ValueError, match="Group sizes"):
        group_indices(["x"] * 5 + ["y"] * 7, 6)


# ------------------------------------------------------------------------------------------------ GPU
def _pack_dets(dets, K, cap):
    """Oracle-style per-image dicts -> engine records ([B][cap][24] words): tvec expressed through (proj_ctr, depth)."""
    Bn = len(dets)
    inv_K = torch.linalg.inv(K)
    buf = torch.zeros(Bn, cap, 24)
    counts = torch.zeros(Bn, dtype=torch.int32)
    packed = []
    for b, det in enumerate(dets):
        det = dict(det)
        n = det["quat"].shape[0]
        depth = det["tvec"][:, 2].clamp(min=1.0)
        tv = det["tvec"].clone()
        tv[:, 2] = depth
        uvw = tv @ K[b].T
        pc = uvw[:, :2] / uvw[:, 2:]
        det["tvec"] = (torch.cat([pc, torch.ones(n, 1)], 1) @ inv_K[b].T) * depth[:, None]
        buf[b, :n, 5] = det["score3d"]
        buf[b, :n, 8:12] = det["quat"]
        buf[b, :n, 12:14] = pc
        buf[b, :n, 14] = depth
        buf[b, :n, 15:18] = det["size"]
        buf.view(torch.int32)[b, :n, 6] = det["cls"].to(torch.int32)
        buf.view(torch.int32)[b, :n, 20] = torch.arange(n, dtype=torch.int32)  # index word: original slot
        counts[b] = n
        packed.append(det)
    return buf, counts, packed


@pytest.mark.gpu
@pytest.mark.parametrize("seed,max_dets", [(7, 500), (8, 150), (11, 1)])
def test_sample_aggregate_kernel_vs_oracle(seed, max_dets):
    import ctypes as C
    from dd3d_b200 import lib
    L = lib.load()
    dets, gids, poses = aggregate_case(seed)
    Bn, cap = len(dets), 128
    K = torch.tensor([[[700.0, 0.0, 320.0], [0.0, 690.0, 180.0], [0.0, 0.0, 1.0]]]).repeat(Bn, 1, 1)
    buf, counts, packed = _pack_dets(dets, K, cap)
    ref = B.sample_aggregate(packed, gids, poses, 0.3, max_dets)
    pose_t = torch.tensor([list(q) + list(t) for q, t in poses], dtype=torch.float32)
    d_d, d_c, d_K, d_p = buf.cuda(), counts.cuda(), K.reshape(Bn, 9).contiguous().cuda(), pose_t.cuda()
    d_g = torch.tensor(gids, dtype=torch.int32).cuda()
    d_glob = torch.zeros(Bn, cap, 10, device="cuda")
    flags = torch.zeros(1, dtype=torch.int32, device="cuda")
    scratch = torch.empty(int(L.dd3d_op_sample_aggregate_scratch_bytes(Bn, cap)), dtype=torch.uint8, device="cuda")
    st = L.dd3d_op_sample_aggregate(C.c_void_p(d_d.data_ptr()), C.c_void_p(d_c.data_ptr()), C.c_void_p(d_K.data_ptr()),
                                    C.c_void_p(d_p.data_ptr()), C.c_void_p(d_g.data_ptr()), max(gids) + 1,
                                    C.c_void_p(d_glob.data_ptr()), C.c_void_p(scratch.data_ptr()),
                                    C.c_void_p(flags.data_ptr()), Bn, cap, 0.3, max_dets,
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert st == 0
    torch.cuda.synchronize()
    assert int(flags.item()) == 0
    out, cnt, glob = d_d.cpu(), d_c.cpu(), d_glob.cpu()
    total = 0
    for b, r in enumerate(ref):
        m = int(cnt[b])
        total += m
        assert m == r["score3d"].shape[0], (b, m, r["score3d"].shape[0])
        assert torch.equal(out[b, :m, 5], r["score3d"])  # same survivors, original order
        if m:
            assert quat_dist(glob[b, :m, 0:4], r["quat_global"]).max().item() < 1e-5
            np.testing.assert_allclose(glob[b, :m, 4:7].numpy(), r["tvec_global"].numpy(), rtol=1e-5, atol=1e-4)
            np.testing.assert_allclose(glob[b, :m, 7:10].numpy(), r["size"].numpy(), rtol=0, atol=0)
    assert total <= max_dets


@pytest.mark.gpu
def test_nuscenes_forward_vs_emulating_oracle_and_golden():
    """NuscenesDD3DB200.forward on one 6-camera sample: (1) against the bf16-emulating oracle of the whole path up to the
    per-image detections, (2) the sample aggregation exactly, by running the oracle's aggregation on the model's own
    pre-aggregation detections, (3) loosely against the fp32 reference golden."""
    from dd3d_b200.config import get_cfg
    from dd3d_b200.meta_arch import NuscenesDD3DB200
    from dd3d_b200.synthetic import make_state_dict
    from oracle.dd3d_oracle import DD3DOracle, pose_of
    from oracle.gen_golden import NUSC_CASE, nusc_case_inputs
    arch = NUSC_CASE[0]
    cfg = get_cfg(arch, "nuscenes", meta_arch="NuscenesDD3D")
    sd = make_state_dict(cfg)
    inputs = nusc_case_inputs()
    model = NuscenesDD3DB200(cfg).to("cuda")
    model.load_state_dict(sd)
    out = model(inputs)
    assert model.overflow_flags() == 0

    def as_dict(inst):
        b3 = inst.pred_boxes3d
        d = dict(level=inst.fpn_levels.cpu(), loc=inst.locations.cpu(), cls=inst.pred_classes.cpu(),
                 box2d=inst.pred_boxes.tensor.cpu(), score3d=inst.scores_3d.cpu(), score=inst.scores.cpu(),
                 quat=b3.quat.cpu(), tvec=b3.tvec.cpu(), size=b3.size.cpu(), attr=inst.pred_attributes.cpu(),
                 speed=inst.pred_speeds.cpu())
        if inst.has("pred_boxes3d_global"):
            d["quat_global"], d["tvec_global"] = inst.pred_boxes3d_global.quat.cpu(), inst.pred_boxes3d_global.tvec.cpu()
        return d

    got = [as_dict(o["instances"]) for o in out]
    # (2) aggregation step in isolation
    model.sample_aggregate_in_inference = False
    pre = [as_dict(o["instances"]) for o in model(inputs)]
    model.sample_aggregate_in_inference = True
    ref = B.sample_aggregate(pre, [0] * 6, [pose_of(x) for x in inputs], cfg.DD3D.INFERENCE.BEV_NMS_IOU_THRESH,
                             cfg.DD3D.NUSC.INFERENCE.MAX_NUM_DETS_PER_SAMPLE)
    assert sum(r["score3d"].shape[0] for r in ref) < sum(p["score3d"].shape[0] for p in pre)  # suppression happened
    for gd, r in zip(got, ref):
        assert torch.equal(gd["score3d"], r["score3d"])
        assert torch.equal(gd["attr"], r["attr"]) and torch.equal(gd["speed"], r["speed"])
        assert quat_dist(gd["quat_global"], r["quat_global"]).max().item() < 1e-5
        np.testing.assert_allclose(gd["tvec_global"].numpy(), r["tvec_global"].numpy(), rtol=1e-5, atol=1e-4)
    # (1) whole path vs the emulating oracle (attributes / speeds of matched detections)
    emu = DD3DOracle(cfg, sd, emulate_bf16=True).forward(inputs)
    matched = total = 0
    for gd, e in zip(got, emu):
        ka = [det_key(l, loc, c) for l, loc, c in zip(gd["level"], gd["loc"], gd["cls"])]
        kb = [det_key(l, loc, c) for l, loc, c in zip(e["level"], e["loc"], e["cls"])]
        ia, ib = match_by_key(ka, kb)
        matched += len(ia)
        total += max(len(ka), len(kb))
        if len(ia):
            assert rel_err(gd["box2d"][ia], e["box2d"][ib], floor=32.0) < 5e-3
            assert rel_err(gd["speed"][ia], e["speed"][ib], floor=1.0) < 2e-2
            assert (gd["attr"][ia] == e["attr"][ib]).float().mean().item() > 0.95
            # global positions: error relative to the camera-frame range (global coordinates carry the ego offset)
            err = (gd["tvec_global"][ia] - e["tvec_global"][ib]).norm(dim=1) / e["tvec"][ib].norm(dim=1).clamp(min=1.0)
            assert err.max().item() < 2e-2
    assert matched >= 0.9 * total
    # (3) fp32 reference golden, loose (bf16 storage)
    g = np.load(os.path.join(GOLDEN_DIR, f"golden_nusc_{arch}.npz"))
    m2, t2 = _check_against_golden(got, g, len(inputs), 5e-2, exact_sets=False)
    assert m2 >= 0.8 * t2
