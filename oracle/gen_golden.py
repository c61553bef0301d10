"""TEST INFRASTRUCTURE -- generates tests/golden/*.npz by running the REAL reference DD3D.forward
(/root/reference/tridet/modeling/dd3d/core.py, imported unmodified under oracle/ref_standin.py) in the build
container.  /root/reference does not exist on the GPU box, so the vectors are committed.

    python -m oracle.gen_golden

Fixtures (all fp32 reference arithmetic, synthetic calibrated weights seed 0, inputs from
dd3d_b200.synthetic.make_inputs):
  golden_<arch>.npz : per image b -> boxes, scores, scores_3d, classes, levels, locations, quat, proj_ctr, depth, size,
                      tvec (post NMS / top-k / postprocess), plus the case description.
  kat_boxes3d.npz   : known-answer vector for predictions_to_boxes3d (fcos3d.py:16-52) from SURVEY.md 8c.
  reference_checks.npz, reference_configs.json : see gen_reference_checks (`--checks` writes only these two).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from dd3d_b200.config import get_cfg  # noqa: E402
from dd3d_b200.synthetic import make_inputs, make_state_dict  # noqa: E402
from oracle import ref_standin  # noqa: E402

CASES = {
    # arch: (dataset, B, H, W, focal, ragged crop of the last image (dh, dw), output size factor of the last image)
    "dla34": ("kitti_3d", 2, 192, 320, 721.5, (21, 34), 2.0),
    "v2_99": ("nuscenes", 2, 128, 192, 1266.4, (0, 0), 1.0),
}
# BASELINE.json shapes (configs[1] / configs[2]), one image each: the full-size parity cases of tests/test_parity_full_gpu.py
FULL_CASES = {
    # name: (arch, dataset, B, H, W, focal)
    "dla34_full": ("dla34", "kitti_3d", 1, 384, 1280, 721.5),
    "v2_99_full": ("v2_99", "nuscenes", 1, 900, 1600, 1266.4),
}
NUSC_CASE = ("v2_99", 1, 128, 192, 1266.4)  # NuscenesDD3D: backbone, samples (x 6 cameras), H, W, focal


TTA_CASE = dict(arch="dla34", dataset="kitti_3d", H=96, W=320, orig=(94, 313), focal=721.5, min_sizes=[64, 96, 128],
                ims_per_batch=4, pre_nms_thresh=0.02)


def tta_case():
    """(cfg, mapped dataset dict) of the TTA fixture: the mapped image is a resized version of a 94x313 original, three
    scales x flip = 6 views run in chunks of 4 (so one chunk mixes two scales and is zero padded)."""
    c = TTA_CASE
    cfg = get_cfg(c["arch"], c["dataset"])
    cfg.DD3D.INFERENCE.DO_POSTPROCESS = False
    cfg.DD3D.FCOS2D.INFERENCE.PRE_NMS_THRESH = c["pre_nms_thresh"]
    cfg.TEST.AUG.MIN_SIZES = list(c["min_sizes"])
    cfg.TEST.IMS_PER_BATCH = c["ims_per_batch"]
    x = make_inputs(1, c["H"], c["W"], c["focal"])[0]
    x["height"], x["width"] = c["orig"]
    return cfg, x


def nusc_case_inputs():
    from dd3d_b200.synthetic import make_nusc_inputs
    _, ns, H, W, focal = NUSC_CASE
    inputs = make_nusc_inputs(ns, H, W, focal)
    for x in inputs:  # the sample aggregation runs AFTER the rescale; detectron2's Instances.cat inside it requires
        x["height"], x["width"] = 2 * H, 2 * W  # one common output size per call (all nuScenes images are 900x1600)
    return inputs


def with_reference_poses(inputs):
    """(quat, tvec) pairs -> the reference's own Pose objects (tridet/structures/pose.py)."""
    ref_standin.install()
    from tridet.structures.pose import Pose
    return [dict(x, pose=Pose(wxyz=np.float32(x["pose"][0]), tvec=np.float32(x["pose"][1]))) for x in inputs]


def reference_sample_aggregate(dets, group_ids, poses, thr, max_dets):
    """Runs the reference's nuscenes_sample_aggregate (postprocessing.py:58-108) on per-image detection dicts;
    returns per image (kept original indices, global quat, global tvec)."""
    ref_standin.install()
    from tridet.modeling.dd3d.postprocessing import nuscenes_sample_aggregate
    from tridet.structures.boxes3d import GenericBoxes3D
    from tridet.structures.pose import Pose
    from collections import OrderedDict

    class _B3(GenericBoxes3D):
        def __getitem__(self, i):
            return _B3(self.quat[i], self.tvec[i], self.size[i])

        def __len__(self):
            return self.quat.shape[0]

        @classmethod
        def cat(cls, l):
            return _B3(torch.cat([b.quat for b in l]), torch.cat([b.tvec for b in l]), torch.cat([b.size for b in l]))

    insts = []
    for d in dets:
        inst = ref_standin.Instances((100, 100))
        inst.pred_boxes3d = _B3(d["quat"], d["tvec"], d["size"])
        inst.pred_classes = d["cls"]
        inst.scores_3d = d["score3d"]
        inst.orig_index = torch.arange(d["quat"].shape[0])
        insts.append(inst)
    groups = OrderedDict()
    for i, g in enumerate(group_ids):
        groups.setdefault(g, []).append(i)
    rposes = [Pose(wxyz=np.float32(q), tvec=np.float32(t)) for q, t in poses]
    num_classes = 1 + max(int(d["cls"].max()) for d in dets if d["cls"].numel())
    out = nuscenes_sample_aggregate(insts, groups, num_classes, rposes, thr, max_num_dets_per_sample=max_dets)
    return [(o.orig_index, o.pred_boxes3d_global.quat, o.pred_boxes3d_global.tvec) for o in out]


def case_cfg(name, **kw):
    """cfg of a golden case: "dla34" / "v2_99" (small, ragged) or "dla34_full" / "v2_99_full" (BASELINE shapes)."""
    if name in FULL_CASES:
        return get_cfg(FULL_CASES[name][0], FULL_CASES[name][1], **kw)
    return get_cfg(name, CASES[name][0], **kw)


def case_inputs(arch):
    if arch in FULL_CASES:
        _, _, B, H, W, focal = FULL_CASES[arch]
        return make_inputs(B, H, W, focal, with_size=True)
    ds, B, H, W, focal, (dh, dw), fac = CASES[arch]
    inputs = make_inputs(B, H, W, focal)
    if dh or dw:
        inputs[-1]["image"] = inputs[-1]["image"][:, :H - dh, :W - dw].contiguous()
    if fac != 1.0:
        inputs[-1]["height"] = int(round((H - dh) * fac))
        inputs[-1]["width"] = int(round((W - dw) * fac))
    return inputs


def reference_bev_keep(det, pose_quat, pose_tvec, thr):
    """Runs the reference's own nuscenes_sample_aggregate (postprocessing.py:58-108, one dummy group per image, as
    core.py:137-151 does) on one image's detections; returns (sorted kept indices, BEV rotated boxes)."""
    ref_standin.install()
    from tridet.layers.bev_nms import boxes3d_to_rotated_boxes
    from tridet.modeling.dd3d.postprocessing import nuscenes_sample_aggregate
    from tridet.structures.boxes3d import GenericBoxes3D
    from tridet.structures.pose import Pose

    class _B3(GenericBoxes3D):  # pred_boxes3d stand-in: only vectorize()/indexing/cat are used
        def __getitem__(self, i):
            return _B3(self.quat[i], self.tvec[i], self.size[i])

        def __len__(self):
            return self.quat.shape[0]

        @classmethod
        def cat(cls, l):
            return _B3(torch.cat([b.quat for b in l]), torch.cat([b.tvec for b in l]), torch.cat([b.size for b in l]))

    n = det["quat"].shape[0]
    inst = ref_standin.Instances((100, 100))
    inst.pred_boxes3d = _B3(det["quat"], det["tvec"], det["size"])
    inst.pred_classes = det["cls"]
    inst.scores_3d = det["score3d"]
    inst.orig_index = torch.arange(n)
    pose = Pose(wxyz=np.float32(pose_quat), tvec=np.float32(pose_tvec))
    out = nuscenes_sample_aggregate([inst], {0: [0]}, 3, [pose], iou_threshold=thr, include_boxes3d_global=True)[0]
    rot = boxes3d_to_rotated_boxes(out.pred_boxes3d_global, pose_cam_global=Pose()).tensor if len(out) else None
    return out.orig_index, rot


def gen_dd3d_goldens(names, out_dir):
    """golden_<name>.npz: the reference's own DD3D.forward (fp32, CPU) on the seeded case."""
    for arch in names:
        cfg = case_cfg(arch)
        model = ref_standin.build_reference_model(cfg).eval()
        model.load_state_dict(make_state_dict(cfg))
        inputs = case_inputs(arch)
        with torch.no_grad():
            outs = model(inputs)
        blob = {}
        for b, o in enumerate(outs):
            inst = o["instances"]
            b3 = inst.pred_boxes3d
            blob.update({
                f"boxes{b}": inst.pred_boxes.tensor.numpy(), f"scores{b}": inst.scores.numpy(),
                f"scores_3d{b}": inst.scores_3d.numpy(), f"classes{b}": inst.pred_classes.numpy(),
                f"levels{b}": inst.fpn_levels.numpy(), f"locations{b}": inst.locations.numpy(),
                f"quat{b}": b3.quat.numpy(), f"proj_ctr{b}": b3.proj_ctr.numpy(), f"depth{b}": b3.depth.numpy(),
                f"size{b}": b3.size.numpy(), f"tvec{b}": b3.tvec.numpy(),
                f"image_size{b}": np.array(inst.image_size),
            })
            print(arch, "image", b, "detections", len(inst))
        np.savez_compressed(os.path.join(out_dir, f"golden_{arch}.npz"), **blob)


def instances_blob(prefix, inst):
    """The fields of one reference Instances as arrays "<prefix>/<field>" (3-D fields only when the model predicts them)."""
    blob = {f"{prefix}/boxes": inst.pred_boxes.tensor.numpy(), f"{prefix}/scores": inst.scores.numpy(),
            f"{prefix}/classes": inst.pred_classes.numpy(), f"{prefix}/levels": inst.fpn_levels.numpy(),
            f"{prefix}/locations": inst.locations.numpy(), f"{prefix}/has_box3d": np.array(inst.has("pred_boxes3d"))}
    if inst.has("pred_boxes3d"):
        b3 = inst.pred_boxes3d
        blob.update({f"{prefix}/scores_3d": inst.scores_3d.numpy(), f"{prefix}/quat": b3.quat.numpy(),
                     f"{prefix}/depth": b3.depth.numpy().reshape(-1), f"{prefix}/size": b3.size.numpy(),
                     f"{prefix}/tvec": b3.tvec.numpy()})
    return blob


def inventory_blob(prefix, model):
    """The reference model's state_dict inventory: sorted keys and their shapes ("64x3x7x7")."""
    sd = model.state_dict()
    keys = sorted(sd)
    return {f"{prefix}/keys": np.array(keys), f"{prefix}/shapes": np.array(["x".join(map(str, sd[k].shape)) for k in keys])}


def gen_reference_checks(out_dir):
    """reference_checks.npz / reference_configs.json: what the oracle and config checks of the CPU suite compare against,
    recorded from the reference itself -- its parameter inventory and forward under the decode / head switches
    (tests/test_cpu_oracle.py), its BEV NMS / sample aggregation / intrinsics rescale on the seeded cases of
    tests/test_bev_nms.py, test_nuscenes.py, test_input_pipeline.py, its model attributes and KITTI3DEvaluator.process()
    rows for the dla34 golden case (tests/boundary_probe.py), and its four DD3D experiments composed by
    tests/hydra_lite.py (tests/test_config_vs_reference.py)."""
    import json
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from hydra_lite import compose_experiment
    from test_bev_nms import _random_case
    from test_config_vs_reference import EXPERIMENTS
    from test_cpu_oracle import FLAG_CASES, HEAD_CASES, apply_flags, apply_head_flags
    from test_nuscenes import aggregate_case

    configs = {e: compose_experiment(os.path.join(ref_standin.REFERENCE_ROOT, "configs"), e) for e, _ in EXPERIMENTS}
    with open(os.path.join(out_dir, "reference_configs.json"), "w") as f:
        json.dump(configs, f, indent=1, sort_keys=True)
        f.write("\n")

    blob = {}
    small = make_inputs(1, 128, 256, 721.5, seed_base=7)
    runs = [(f"inventory_{arch}", get_cfg(arch, CASES[arch][0])) for arch in CASES]
    for i, flags in enumerate(FLAG_CASES):
        runs.append((f"flags{i}", apply_flags(get_cfg("dla34", "kitti_3d"), flags)))
    for i, flags in enumerate(HEAD_CASES):
        runs.append((f"head{i}", apply_head_flags(get_cfg("dla34", "kitti_3d"), flags)))
    for name, cfg in runs:
        if not name.startswith("inventory"):
            cfg.DD3D.FCOS2D.INFERENCE.PRE_NMS_THRESH = 0.03
        model = ref_standin.build_reference_model(cfg).eval()
        blob.update(inventory_blob(name, model))
        model.load_state_dict(make_state_dict(cfg))
        with torch.no_grad():
            inst = model(small)[0]["instances"]
        blob.update(instances_blob(name, inst))
        print(name, "detections", len(inst))

    for c in range(4):
        det, pq, pt = _random_case(7 + c, 40 + 5 * c)
        blob[f"bev{c}/keep"] = reference_bev_keep(det, pq, pt, 0.3)[0].numpy()
    dets, gids, poses = aggregate_case(3)
    for i, (keep, _, _) in enumerate(reference_sample_aggregate(dets, gids, poses, 0.3, 200)):
        blob[f"aggregate/keep{i}"] = keep.numpy()
    from tridet.data.augmentations.resize_transform import ResizeTransform
    K = np.float32([[1266.4, 0, 816.3], [0, 1266.4, 491.5], [0, 0, 1]])
    for i, ((h, w), (nh, nw)) in enumerate([((900, 1600), (896, 1593)), ((375, 1242), (384, 1272))]):
        blob[f"intrinsics{i}/K"] = ResizeTransform(h, w, nh, nw).apply_intrinsics(K)

    # boundary: the reference DD3D's attributes and its evaluator's rows for its own detections on the dla34 golden case
    ref_standin.install_evaluator_stubs()
    from detectron2.data.catalog import DatasetCatalog, MetadataCatalog
    from types import SimpleNamespace
    from tridet.evaluators.kitti_3d_evaluator import KITTI3DEvaluator
    cfg = get_cfg("dla34", "kitti_3d")
    model = ref_standin.build_reference_model(cfg).eval()
    model.load_state_dict(make_state_dict(cfg))
    for attr in ("postprocess_in_inference", "do_nms", "do_bev_nms", "bev_nms_iou_thresh", "only_box2d", "num_classes"):
        blob[f"boundary/{attr}"] = np.array(getattr(model, attr))
    blob["boundary/size_divisibility"] = np.array(model.backbone.size_divisibility)
    inputs = case_inputs("dla34")
    for i, x in enumerate(inputs):
        x["file_name"], x["image_id"] = f"img{i:06d}.png", i
    names = ["Car", "Pedestrian", "Cyclist", "Van", "Truck"]
    DatasetCatalog.register("kitti_probe", lambda: [{"file_name": x["file_name"]} for x in inputs])
    MetadataCatalog.register("kitti_probe", SimpleNamespace(thing_classes=names, contiguous_id_to_name=dict(enumerate(names))))
    with torch.no_grad():
        outs = model(inputs)
    for b, o in enumerate(outs):
        blob[f"boundary/image_size{b}"] = np.array(o["instances"].image_size)
        blob[f"boundary/fields{b}"] = np.array(sorted(o["instances"].get_fields()))
    ev = KITTI3DEvaluator("kitti_probe", iou_thresholds=[0.5, 0.7])
    ev.reset()
    ev.process(inputs, outs)
    rows = ev._predictions_as_json
    blob["boundary/category"] = np.array([r["category"] for r in rows])
    blob["boundary/file_name"] = np.array([r["file_name"] for r in rows])
    blob["boundary/image_id"] = np.array([r["image_id"] for r in rows])
    for k in ("category_id", "bbox3d", "bbox", "score", "score_3d"):
        blob[f"boundary/{k}"] = np.array([r[k] for r in rows])
    print("boundary: evaluator rows", len(rows))
    np.savez_compressed(os.path.join(out_dir, "reference_checks.npz"), **blob)


def main():
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    if "--full" in sys.argv:  # only the BASELINE-shape cases (a V2-99 900x1600 reference forward takes ~10 s here)
        gen_dd3d_goldens(list(FULL_CASES), out_dir)
        return
    if "--checks" in sys.argv:  # only reference_checks.npz / reference_configs.json
        gen_reference_checks(out_dir)
        return
    gen_dd3d_goldens(list(CASES) + list(FULL_CASES), out_dir)

    # NuscenesDD3D (SURVEY.md 8f row 2): the reference's own meta-arch on one 6-camera sample
    arch = NUSC_CASE[0]
    cfg = get_cfg(arch, "nuscenes", meta_arch="NuscenesDD3D")
    model = ref_standin.build_reference_model(cfg).eval()
    model.load_state_dict(make_state_dict(cfg))
    with torch.no_grad():
        outs = model(with_reference_poses(nusc_case_inputs()))
    blob = {}
    for b, o in enumerate(outs):
        inst = o["instances"]
        b3, g3 = inst.pred_boxes3d, inst.pred_boxes3d_global
        blob.update({
            f"boxes{b}": inst.pred_boxes.tensor.numpy(), f"scores{b}": inst.scores.numpy(),
            f"scores_3d{b}": inst.scores_3d.numpy(), f"classes{b}": inst.pred_classes.numpy(),
            f"levels{b}": inst.fpn_levels.numpy(), f"locations{b}": inst.locations.numpy(),
            f"quat{b}": b3.quat.numpy(), f"proj_ctr{b}": b3.proj_ctr.numpy(), f"depth{b}": b3.depth.numpy(),
            f"size{b}": b3.size.numpy(), f"tvec{b}": b3.tvec.numpy(), f"attr{b}": inst.pred_attributes.numpy(),
            f"speed{b}": inst.pred_speeds.numpy(), f"quat_global{b}": g3.quat.numpy(),
            f"tvec_global{b}": g3.tvec.numpy(), f"image_size{b}": np.array(inst.image_size),
        })
        print("nusc", arch, "image", b, "detections", len(inst))
    np.savez_compressed(os.path.join(out_dir, f"golden_nusc_{arch}.npz"), **blob)

    # sample aggregation on seeded random detections: 2 samples x 6 cameras, with and without the 500-cap biting
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_nuscenes import aggregate_case
    blob = {}
    for c, max_dets in enumerate((1000, 150)):
        dets, gids, poses = aggregate_case(7 + c)
        res = reference_sample_aggregate(dets, gids, poses, 0.3, max_dets)
        for i, (keep, q, t) in enumerate(res):
            blob[f"keep{c}_{i}"] = keep.numpy()
            blob[f"quat{c}_{i}"] = q.numpy()
            blob[f"tvec{c}_{i}"] = t.numpy()
        print("aggregate case", c, "kept", sum(len(r[0]) for r in res), "of", sum(d["quat"].shape[0] for d in dets))
    np.savez_compressed(os.path.join(out_dir, "sample_aggregate.npz"), **blob)

    # test-time augmentation (SURVEY.md 8f row 4): the reference's own DD3DWithTTA around its own DD3D
    from tridet.modeling.dd3d.test_time_augmentation import DD3DWithTTA
    cfg, x = tta_case()
    model = ref_standin.build_reference_model(cfg).eval()
    model.load_state_dict(make_state_dict(cfg))
    with torch.no_grad():
        inst = DD3DWithTTA(cfg, model)([x])[0]["instances"]
    b3 = inst.pred_boxes3d
    np.savez_compressed(
        os.path.join(out_dir, "tta_dla34.npz"), boxes=inst.pred_boxes.tensor.numpy(), scores=inst.scores.numpy(),
        scores_3d=inst.scores_3d.numpy(), classes=inst.pred_classes.numpy(), quat=b3.quat.numpy(),
        proj_ctr=b3.proj_ctr.numpy(), depth=b3.depth.numpy(), size=b3.size.numpy(), tvec=b3.tvec.numpy(),
        inv_K=b3.inv_intrinsics.numpy(), image_size=np.array(inst.image_size))
    print("tta merged detections", len(inst))

    # input pipeline (SURVEY.md 8f row 3): real Pillow resize + the reference's own intrinsics rescale
    from PIL import Image
    from test_input_pipeline import RESIZE_CASES, raw_image
    from tridet.data.augmentations.resize_transform import ResizeTransform
    blob = {}
    for c, ((h, w), (nh, nw)) in enumerate(RESIZE_CASES):
        blob[f"img{c}"] = np.asarray(Image.fromarray(raw_image(c, h, w)).resize((nw, nh), Image.BILINEAR))
        K = np.float32([[721.5377, 0, 609.5593], [0, 721.5377, 172.854], [0, 0, 1]])
        blob[f"K{c}"] = ResizeTransform(h, w, nh, nw).apply_intrinsics(K)
    np.savez_compressed(os.path.join(out_dir, "input_pipeline.npz"), **blob)
    print("input pipeline cases", len(RESIZE_CASES))

    # BEV rotated NMS (SURVEY.md 8f row 1): reference nuscenes_sample_aggregate on seeded random boxes / poses
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_bev_nms import _random_case
    from oracle import bev_nms_oracle
    blob = {"num_cases": 4, "thr": 0.3}
    for c in range(4):
        det, pq, pt = _random_case(100 + c, 30 + 10 * c)
        keep, _ = reference_bev_keep(det, pq, pt, 0.3)
        q, t = bev_nms_oracle.to_global(det["quat"], det["tvec"], pq, pt)
        from tridet.structures.boxes3d import GenericBoxes3D
        from tridet.layers.bev_nms import boxes3d_to_rotated_boxes
        from tridet.structures.pose import Pose
        blob[f"n{c}"] = 30 + 10 * c
        blob[f"keep{c}"] = keep.numpy()
        blob[f"rot{c}"] = boxes3d_to_rotated_boxes(GenericBoxes3D(q, t, det["size"]), pose_cam_global=Pose()).tensor.numpy()
        print("bev case", c, "kept", len(keep), "of", 30 + 10 * c)
    np.savez_compressed(os.path.join(out_dir, "bev_nms.npz"), **blob)

    # known-answer test for the 3-D decode, inputs from SURVEY.md 8c (reference function called verbatim)
    ref_standin.install()
    from tridet.modeling.dd3d.fcos3d import predictions_to_boxes3d
    K = torch.tensor([[721.5377, 0, 609.5593], [0, 721.5377, 172.854], [0, 0, 1]])
    quat = torch.tensor([[1, 0, 0, 0], [.5, -.5, .5, .5], [2, .2, -1, .3]])
    ctr = torch.tensor([[0, 0], [12.5, -3.25], [-40, 8]])
    depth = torch.tensor([10, 25.5, 200])
    size = torch.tensor([[0, 0, 0], [.3, -.2, .1], [-1.5, 2, .7]])
    loc = torch.tensor([[609.5593, 172.854], [800, 200], [64, 320]])
    canon = torch.tensor(get_cfg("dla34", "kitti_3d").DD3D.FCOS3D.CANONICAL_BOX3D_SIZES)[:3]
    inv_K = torch.inverse(K)[None].expand(3, 3, 3)
    b3 = predictions_to_boxes3d(quat, ctr, depth, size, loc, inv_K, canon, 0.1, 80.0, 500.0)
    np.savez(os.path.join(out_dir, "kat_boxes3d.npz"), K=K.numpy(), quat_in=quat.numpy(), ctr_in=ctr.numpy(),
             depth_in=depth.numpy(), size_in=size.numpy(), loc=loc.numpy(), canon=canon.numpy(), quat=b3.quat.numpy(),
             proj_ctr=b3.proj_ctr.numpy(), depth=b3.depth.numpy(), size=b3.size.numpy(), tvec=b3.tvec.numpy())
    print("KAT quat", b3.quat.numpy(), "tvec", b3.tvec.numpy())
    gen_reference_checks(out_dir)


if __name__ == "__main__":
    main()
