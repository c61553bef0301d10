"""Run as a subprocess by tests/test_boundary_reference_plumbing.py.

Drives the B200 mirror through the plumbing the reference's scripts use, with the detectron2 stand-in of
oracle/ref_standin.py installed in place of detectron2, and checks it against what the reference produced on the dla34
golden case (tests/golden/reference_checks.npz "boundary/*", recorded by oracle/gen_golden.py):
 1. registry: with the stand-in installed BEFORE dd3d_b200 is imported, `dd3d_b200.meta_arch` registers DD3DB200 /
    NuscenesDD3DB200 in detectron2's META_ARCH_REGISTRY (where the reference's DD3D registers, core.py:18), and the model
    is built the way scripts/train.py:48 -> detectron2 build_model does: META_ARCH_REGISTRY.get(cfg.MODEL.META_ARCHITECTURE)
    (cfg), .to(cfg.MODEL.DEVICE) -- selected purely by the config string; the attributes do_test / DD3DWithTTA poke equal
    the reference DD3D's;
 2. types: the Instances it returns are detectron2's Instances / Boxes, with the reference's fields and image sizes;
 3. evaluator: what the reference's KITTI3DEvaluator.process() (kitti_3d_evaluator.py:66-123) reads from them per
    detection -- class, pred_boxes3d[i].vectorize(), the XYWH 2-D box, scores, scores_3d -- equals the rows it wrote from
    the reference model's own outputs (its KITTI rows are a function of the same values).
The detections fed through DD3DB200._wrap (the product code that turns the C ABI's packed [B][cap][24] buffer into
Instances) are the reference DD3D's own detections on the dla34 golden case (tests/golden/golden_dla34.npz), packed into
the C-ABI layout -- the wrapping needs no GPU.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, os.path.abspath(ROOT))
from oracle import ref_standin  # noqa: E402

ref_standin.install_third_party()
from detectron2.modeling.meta_arch.build import META_ARCH_REGISTRY  # noqa: E402  (stand-in registry)
import dd3d_b200.meta_arch as ma  # noqa: E402  registers DD3DB200 / NuscenesDD3DB200
from dd3d_b200 import lib  # noqa: E402
from dd3d_b200.config import get_cfg  # noqa: E402
from dd3d_b200.synthetic import make_state_dict  # noqa: E402
from oracle.gen_golden import case_inputs  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def build_model(cfg):
    """detectron2.modeling.build_model, restated: registry lookup by config string, then .to(device)."""
    model = META_ARCH_REGISTRY.get(cfg.MODEL.META_ARCHITECTURE)(cfg)
    model.to(torch.device(cfg.MODEL.DEVICE))
    return model


def pack_words(golden, nimg, cap):
    """golden_dla34.npz detections -> the C ABI's [B][cap][24] fp32 words + counts (include/dd3d_b200.h dd3d_det)."""
    out = torch.zeros(nimg, cap, lib.DET_WORDS, dtype=torch.float32)
    oi = out.view(torch.int32)
    counts = torch.zeros(nimg, dtype=torch.int32)
    for b in range(nimg):
        n = golden[f"boxes{b}"].shape[0]
        counts[b] = n
        out[b, :n, 0:4] = torch.from_numpy(golden[f"boxes{b}"])
        out[b, :n, 4] = torch.from_numpy(golden[f"scores{b}"])
        out[b, :n, 5] = torch.from_numpy(golden[f"scores_3d{b}"])
        oi[b, :n, 6] = torch.from_numpy(golden[f"classes{b}"]).to(torch.int32)
        oi[b, :n, 7] = torch.from_numpy(golden[f"levels{b}"]).to(torch.int32)
        out[b, :n, 8:12] = torch.from_numpy(golden[f"quat{b}"])
        out[b, :n, 12:14] = torch.from_numpy(golden[f"proj_ctr{b}"])
        out[b, :n, 14] = torch.from_numpy(golden[f"depth{b}"]).reshape(-1)
        out[b, :n, 15:18] = torch.from_numpy(golden[f"size{b}"])
        out[b, :n, 18:20] = torch.from_numpy(golden[f"locations{b}"])
    return out, counts


def main():
    ref = np.load(os.path.join(GOLDEN, "reference_checks.npz"))
    ref = {k.split("/", 1)[1]: v for k, v in ref.items() if k.startswith("boundary/")}

    # ---- 1. registry / build_model by config string
    assert META_ARCH_REGISTRY.get("DD3DB200") is ma.DD3DB200
    assert META_ARCH_REGISTRY.get("NuscenesDD3DB200") is ma.NuscenesDD3DB200
    cfg = get_cfg("dla34", "kitti_3d")
    assert cfg.MODEL.META_ARCHITECTURE == "DD3D"  # the experiment's own string selects the reference's DD3D
    cfg.MODEL.DEVICE = "cpu"
    cfg.MODEL.META_ARCHITECTURE = "DD3DB200"
    model = build_model(cfg)
    assert type(model) is ma.DD3DB200
    for attr in ("postprocess_in_inference", "do_nms", "do_bev_nms", "bev_nms_iou_thresh", "only_box2d", "num_classes",
                 "device"):  # what do_test / DD3DWithTTA poke (scripts/train.py:206-209, test_time_augmentation.py:107)
        assert hasattr(model, attr), attr
        assert attr == "device" or getattr(model, attr) == ref[attr].item(), attr
    assert model.backbone.size_divisibility == ref["size_divisibility"].item()
    res = model.load_state_dict(make_state_dict(cfg))  # the reference's key set (tests/test_cpu_oracle.py inventory)
    assert not res.missing_keys and not res.unexpected_keys
    try:
        model([{"image": torch.zeros(3, 8, 8, dtype=torch.uint8), "intrinsics": torch.eye(3) * 2}])
        raise SystemExit("forward on cpu must fail loudly")
    except RuntimeError as e:
        assert "no CPU path" in str(e)

    # ---- 2. + 3. the mirror's output containers vs what the reference evaluator read from the reference's own
    inputs = case_inputs("dla34")
    golden = np.load(os.path.join(GOLDEN, "golden_dla34.npz"))
    words, counts = pack_words(golden, len(inputs), model._desc.out_cap)
    assert int(counts.sum()) > 10
    K = torch.stack([x["intrinsics"] for x in inputs]).reshape(len(inputs), 9)
    sizes = torch.tensor([[x["image"].shape[-2], x["image"].shape[-1], x.get("height", x["image"].shape[-2]),
                           x.get("width", x["image"].shape[-1])] for x in inputs], dtype=torch.int32)
    b200_out = model._wrap(words, counts, K, sizes, torch.device("cpu"))  # product code: packed buffer -> Instances
    from detectron2.structures import Boxes, Instances
    from dd3d_b200.structures import Boxes3D
    names = ["Car", "Pedestrian", "Cyclist", "Van", "Truck"]
    rows = []
    for b, o in enumerate(b200_out):
        inst = o["instances"]
        assert type(inst) is Instances and type(inst.pred_boxes) is Boxes and type(inst.pred_boxes3d) is Boxes3D
        assert tuple(inst.image_size) == tuple(ref[f"image_size{b}"].tolist())
        assert sorted(inst.get_fields()) == ref[f"fields{b}"].tolist()
        for i in range(len(inst)):  # the evaluator's per-detection reads (kitti_3d_evaluator.py:84-104)
            x0, y0, x1, y1 = inst.pred_boxes.tensor[i].tolist()
            rows.append(dict(category_id=int(inst.pred_classes[i]), category=names[int(inst.pred_classes[i])],
                             bbox3d=inst.pred_boxes3d[i].vectorize()[0].numpy(), bbox=[x0, y0, x1 - x0, y1 - y0],
                             score=float(inst.scores[i]), score_3d=float(inst.scores_3d[i]),
                             file_name=f"img{b:06d}.png", image_id=b))
    assert len(rows) == len(ref["category_id"]) == int(counts.sum())
    for j, r in enumerate(rows):
        assert r["category_id"] == ref["category_id"][j] and r["category"] == ref["category"][j]
        assert r["file_name"] == ref["file_name"][j] and r["image_id"] == ref["image_id"][j]
        np.testing.assert_allclose(r["bbox3d"], ref["bbox3d"][j], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(r["bbox"], ref["bbox"][j], rtol=1e-6, atol=1e-4)
        assert abs(r["score"] - ref["score"][j]) < 1e-6 and abs(r["score_3d"] - ref["score_3d"][j]) < 1e-6
    print(f"BOUNDARY_OK detections={len(rows)}")


if __name__ == "__main__":
    main()
