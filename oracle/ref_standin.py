"""TEST INFRASTRUCTURE ONLY -- never imported by the product path (dd3d_b200/).

Stand-in for the third-party packages the reference DD3D imports but that are not installable in
this container (detectron2, pytorch3d, fvcore, pyquaternion, mpi4py).  With it installed into
``sys.modules`` the reference's own hot-path files under /root/reference/tridet (core.py, fcos2d.py,
fcos3d.py, dla.py, vovnet.py, boxes3d.py, image_list.py, geometry.py, tensor2d.py, normalization.py)
import and run UNMODIFIED on CPU.  It exists for two purposes only:

  * oracle/gen_golden.py runs the real reference here and writes tests/golden/*.npz;
  * tests/test_oracle_vs_reference.py (skipped when /root/reference is absent) pins oracle/dd3d_oracle.py
    against the real reference.

Every class restates the published semantics of the upstream symbol it replaces (SURVEY.md Appendix A):
detectron2 v0.5-era ``layers.Conv2d / get_norm / FrozenBatchNorm2d / batched_nms``,
``modeling.backbone.FPN / LastLevelP6P7``, ``structures.Instances / Boxes``,
``modeling.postprocessing.detector_postprocess``; pytorch3d >=0.5 ``quaternion_to_matrix /
matrix_to_quaternion`` and the row-vector ``transform3d``.
"""
import importlib.machinery
import sys
import types

import torch
import torch.nn.functional as F
from torch import nn

REFERENCE_ROOT = "/root/reference"


# ----------------------------------------------------------------------------------------------
# detectron2.layers
# ----------------------------------------------------------------------------------------------
class ShapeSpec:
    def __init__(self, channels=None, height=None, width=None, stride=None):
        self.channels, self.height, self.width, self.stride = channels, height, width, stride


class FrozenBatchNorm2d(nn.Module):
    """y = x*s + b with s = weight*rsqrt(running_var+eps), b = bias - running_mean*s; eps=1e-5."""
    _version = 3

    def __init__(self, num_features, eps=1e-5):
        super().__init__()
        self.num_features, self.eps = num_features, eps
        self.register_buffer("weight", torch.ones(num_features))
        self.register_buffer("bias", torch.zeros(num_features))
        self.register_buffer("running_mean", torch.zeros(num_features))
        self.register_buffer("running_var", torch.ones(num_features) - eps)

    def forward(self, x):
        scale = self.weight * (self.running_var + self.eps).rsqrt()
        bias = self.bias - self.running_mean * scale
        return x * scale.reshape(1, -1, 1, 1).to(x.dtype) + bias.reshape(1, -1, 1, 1).to(x.dtype)

    @classmethod
    def convert_frozen_batchnorm(cls, module):
        return module


def get_norm(norm, out_channels):
    if norm is None:
        return None
    if isinstance(norm, str):
        if len(norm) == 0:
            return None
        norm = {
            "BN": nn.BatchNorm2d,
            "SyncBN": nn.BatchNorm2d,
            "FrozenBN": FrozenBatchNorm2d,
            "GN": lambda c: nn.GroupNorm(32, c),
        }[norm]
    return norm(out_channels)


class Conv2d(nn.Conv2d):
    """conv -> norm (if any) -> activation (if any)."""
    def __init__(self, *args, **kwargs):
        norm = kwargs.pop("norm", None)
        activation = kwargs.pop("activation", None)
        super().__init__(*args, **kwargs)
        self.norm = norm
        self.activation = activation

    def forward(self, x):
        x = F.conv2d(x, self.weight, self.bias, self.stride, self.padding, self.dilation, self.groups)
        if self.norm is not None:
            x = self.norm(x)
        if self.activation is not None:
            x = self.activation(x)
        return x


def cat(tensors, dim=0):
    if len(tensors) == 1:
        return tensors[0]
    return torch.cat(tensors, dim)


def _nms_greedy(boxes, scores, thr):
    """torchvision.ops.nms semantics: sort by score desc; keep i unless a kept higher-scored box has
    IoU > thr (strict); IoU = inter / (a + b - inter); returns kept indices in descending-score order."""
    from torchvision.ops import nms
    return nms(boxes, scores, thr)


def batched_nms(boxes, scores, idxs, iou_threshold):
    """detectron2.layers.batched_nms -> torchvision.ops.batched_nms (coordinate-offset trick)."""
    assert boxes.shape[-1] == 4
    if boxes.numel() == 0:
        return torch.empty((0, ), dtype=torch.int64, device=boxes.device)
    boxes = boxes.float()
    max_coordinate = boxes.max()
    offsets = idxs.to(boxes) * (max_coordinate + torch.tensor(1).to(boxes))
    boxes_for_nms = boxes + offsets[:, None]
    return _nms_greedy(boxes_for_nms, scores, iou_threshold)


def batched_nms_rotated(boxes, scores, idxs, iou_threshold):
    """detectron2.layers.nms.batched_nms_rotated: shift the centres by a per-class offset so that boxes of different
    classes never overlap, then greedy rotated NMS (restated in oracle/bev_nms_oracle.py)."""
    assert boxes.shape[-1] == 5
    if boxes.numel() == 0:
        return torch.empty((0, ), dtype=torch.int64, device=boxes.device)
    from oracle.bev_nms_oracle import nms_rotated
    boxes = boxes.float()
    max_coordinate = (torch.max(boxes[:, 0], boxes[:, 1]) + torch.max(boxes[:, 2], boxes[:, 3]) / 2).max()
    min_coordinate = (torch.min(boxes[:, 0], boxes[:, 1]) - torch.max(boxes[:, 2], boxes[:, 3]) / 2).min()
    offsets = idxs.to(boxes) * (max_coordinate - min_coordinate + 1)
    boxes_for_nms = boxes.clone()
    boxes_for_nms[:, :2] += offsets[:, None]
    return nms_rotated(boxes_for_nms, scores, torch.zeros_like(idxs), iou_threshold)


# ----------------------------------------------------------------------------------------------
# detectron2.structures
# ----------------------------------------------------------------------------------------------
class Boxes:
    def __init__(self, tensor):
        if not isinstance(tensor, torch.Tensor):
            tensor = torch.as_tensor(tensor, dtype=torch.float32)
        tensor = tensor.to(torch.float32)
        if tensor.numel() == 0:
            tensor = tensor.reshape((-1, 4))
        assert tensor.dim() == 2 and tensor.size(-1) == 4, tensor.size()
        self.tensor = tensor

    def clone(self):
        return Boxes(self.tensor.clone())

    def to(self, *args, **kwargs):
        return Boxes(self.tensor.to(*args, **kwargs))

    def area(self):
        b = self.tensor
        return (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])

    def clip(self, box_size):
        h, w = box_size
        x1 = self.tensor[:, 0].clamp(min=0, max=w)
        y1 = self.tensor[:, 1].clamp(min=0, max=h)
        x2 = self.tensor[:, 2].clamp(min=0, max=w)
        y2 = self.tensor[:, 3].clamp(min=0, max=h)
        self.tensor = torch.stack((x1, y1, x2, y2), dim=-1)

    def nonempty(self, threshold=0.0):
        b = self.tensor
        return ((b[:, 2] - b[:, 0]) > threshold) & ((b[:, 3] - b[:, 1]) > threshold)

    def scale(self, scale_x, scale_y):
        self.tensor[:, 0::2] *= scale_x
        self.tensor[:, 1::2] *= scale_y

    def __getitem__(self, item):
        if isinstance(item, int):
            return Boxes(self.tensor[item].view(1, -1))
        b = self.tensor[item]
        assert b.dim() == 2
        return Boxes(b)

    def __len__(self):
        return self.tensor.shape[0]

    @classmethod
    def cat(cls, boxes_list):
        if len(boxes_list) == 0:
            return cls(torch.empty(0))
        return cls(torch.cat([b.tensor for b in boxes_list], dim=0))

    @property
    def device(self):
        return self.tensor.device


class RotatedBoxes:
    """detectron2.structures.RotatedBoxes subset: (N, 5) = (cx, cy, w, h, angle_degrees)."""
    def __init__(self, tensor):
        tensor = torch.as_tensor(tensor, dtype=torch.float32)
        if tensor.numel() == 0:
            tensor = tensor.reshape((0, 5))
        assert tensor.dim() == 2 and tensor.size(-1) == 5, tensor.size()
        self.tensor = tensor

    def __len__(self):
        return self.tensor.shape[0]


class Instances:
    def __init__(self, image_size, **kwargs):
        self._image_size = image_size
        self._fields = {}
        for k, v in kwargs.items():
            self.set(k, v)

    @property
    def image_size(self):
        return self._image_size

    def __setattr__(self, name, val):
        if name.startswith("_"):
            super().__setattr__(name, val)
        else:
            self.set(name, val)

    def __getattr__(self, name):
        if name == "_fields" or name not in self._fields:
            raise AttributeError("Cannot find field '{}' in the given Instances!".format(name))
        return self._fields[name]

    def set(self, name, value):
        data_len = len(value)
        if len(self._fields):
            assert len(self) == data_len, "Adding a field of length {} to a Instances of length {}".format(
                data_len, len(self))
        self._fields[name] = value

    def has(self, name):
        return name in self._fields

    def remove(self, name):
        del self._fields[name]

    def get(self, name):
        return self._fields[name]

    def get_fields(self):
        return self._fields

    def to(self, *args, **kwargs):
        ret = Instances(self._image_size)
        for k, v in self._fields.items():
            if hasattr(v, "to"):
                v = v.to(*args, **kwargs)
            ret.set(k, v)
        return ret

    def __getitem__(self, item):
        if type(item) == int:
            if item >= len(self) or item < -len(self):
                raise IndexError("Instances index out of range!")
            item = slice(item, None, len(self))
        ret = Instances(self._image_size)
        for k, v in self._fields.items():
            ret.set(k, v[item])
        return ret

    def __len__(self):
        for v in self._fields.values():
            return v.__len__()
        raise NotImplementedError("Empty Instances does not support __len__!")

    @staticmethod
    def cat(instance_lists):
        assert all(isinstance(i, Instances) for i in instance_lists)
        assert len(instance_lists) > 0
        if len(instance_lists) == 1:
            return instance_lists[0]
        image_size = instance_lists[0].image_size
        for i in instance_lists[1:]:  # detectron2 asserts a common image size
            assert i.image_size == image_size
        ret = Instances(image_size)
        for k in instance_lists[0]._fields.keys():
            values = [i.get(k) for i in instance_lists]
            v0 = values[0]
            if isinstance(v0, torch.Tensor):
                values = torch.cat(values, dim=0)
            elif isinstance(v0, list):
                values = sum(values, [])
            elif hasattr(type(v0), "cat"):
                values = type(v0).cat(values)
            else:
                raise ValueError("Unsupported type {} for concatenation".format(type(v0)))
            ret.set(k, values)
        return ret


def detector_postprocess(results, output_height, output_width, mask_threshold=0.5):
    """sx = W_out / image_size[1], sy = H_out / image_size[0]; scale boxes, clip, drop empty."""
    if isinstance(output_width, torch.Tensor):
        output_width_tmp, output_height_tmp = output_width.float(), output_height.float()
        new_size = torch.stack([output_height, output_width])
    else:
        new_size = (output_height, output_width)
        output_width_tmp, output_height_tmp = output_width, output_height
    scale_x = output_width_tmp / results.image_size[1]
    scale_y = output_height_tmp / results.image_size[0]
    results = Instances(new_size, **results.get_fields())
    output_boxes = results.pred_boxes
    output_boxes.scale(scale_x, scale_y)
    output_boxes.clip(results.image_size)
    results = results[output_boxes.nonempty()]
    return results


# ----------------------------------------------------------------------------------------------
# detectron2.modeling.backbone (FPN and friends), registries, configurable
# ----------------------------------------------------------------------------------------------
class Registry(dict):
    def __init__(self, name):
        super().__init__()
        self._name = name

    def register(self, obj=None):
        if obj is None:
            def deco(func_or_class):
                self[func_or_class.__name__] = func_or_class
                return func_or_class
            return deco
        self[obj.__name__] = obj
        return obj

    def get(self, name):
        if name not in self:
            raise KeyError("No object named '{}' found in '{}' registry!".format(name, self._name))
        return self[name]


BACKBONE_REGISTRY = Registry("BACKBONE")
META_ARCH_REGISTRY = Registry("META_ARCH")


class Backbone(nn.Module):
    @property
    def size_divisibility(self):
        return 0

    def output_shape(self):
        return {
            name: ShapeSpec(channels=self._out_feature_channels[name], stride=self._out_feature_strides[name])
            for name in self._out_features
        }


def configurable(init_func=None, *, from_config=None):
    """detectron2.config.configurable for __init__: if the first positional arg looks like a cfg node,
    call cls.from_config(cfg, *rest) to obtain kwargs."""
    import functools

    def _called_with_cfg(*args, **kwargs):
        if len(args) and hasattr(args[0], "keys") and not isinstance(args[0], (list, tuple, str)):
            return True
        return "cfg" in kwargs

    if init_func is not None:
        @functools.wraps(init_func)
        def wrapped(self, *args, **kwargs):
            if _called_with_cfg(*args, **kwargs):
                explicit = type(self).from_config(*args, **kwargs)
                init_func(self, **explicit)
            else:
                init_func(self, *args, **kwargs)
        return wrapped

    def wrapper(orig_func):
        @functools.wraps(orig_func)
        def wrapped(*args, **kwargs):
            if _called_with_cfg(*args, **kwargs):
                return orig_func(**from_config(*args, **kwargs))
            return orig_func(*args, **kwargs)
        return wrapped
    return wrapper


class LastLevelMaxPool(nn.Module):
    def __init__(self):
        super().__init__()
        self.num_levels = 1
        self.in_feature = "p5"

    def forward(self, x):
        return [F.max_pool2d(x, kernel_size=1, stride=2, padding=0)]


class LastLevelP6P7(nn.Module):
    def __init__(self, in_channels, out_channels, in_feature="res5"):
        super().__init__()
        self.num_levels = 2
        self.in_feature = in_feature
        self.p6 = nn.Conv2d(in_channels, out_channels, 3, 2, 1)
        self.p7 = nn.Conv2d(out_channels, out_channels, 3, 2, 1)

    def forward(self, c5):
        p6 = self.p6(c5)
        p7 = self.p7(F.relu(p6))
        return [p6, p7]


class FPN(Backbone):
    """detectron2.modeling.backbone.FPN (see SURVEY.md Appendix A for the restated semantics)."""
    def __init__(self, bottom_up, in_features, out_channels, norm="", top_block=None, fuse_type="sum"):
        super().__init__()
        import math
        input_shapes = bottom_up.output_shape()
        strides = [input_shapes[f].stride for f in in_features]
        in_channels_per_feature = [input_shapes[f].channels for f in in_features]
        lateral_convs, output_convs = [], []
        use_bias = norm == ""
        for idx, in_channels in enumerate(in_channels_per_feature):
            lateral_norm = get_norm(norm, out_channels)
            output_norm = get_norm(norm, out_channels)
            lateral_conv = Conv2d(in_channels, out_channels, kernel_size=1, bias=use_bias, norm=lateral_norm)
            output_conv = Conv2d(
                out_channels, out_channels, kernel_size=3, stride=1, padding=1, bias=use_bias, norm=output_norm)
            stage = int(math.log2(strides[idx]))
            self.add_module("fpn_lateral{}".format(stage), lateral_conv)
            self.add_module("fpn_output{}".format(stage), output_conv)
            lateral_convs.append(lateral_conv)
            output_convs.append(output_conv)
        self.lateral_convs = lateral_convs[::-1]
        self.output_convs = output_convs[::-1]
        self.top_block = top_block
        self.in_features = tuple(in_features)
        self.bottom_up = bottom_up
        self._out_feature_strides = {"p{}".format(int(math.log2(s))): s for s in strides}
        if self.top_block is not None:
            for s in range(stage, stage + self.top_block.num_levels):
                self._out_feature_strides["p{}".format(s + 1)] = 2**(s + 1)
        self._out_features = list(self._out_feature_strides.keys())
        self._out_feature_channels = {k: out_channels for k in self._out_features}
        self._size_divisibility = strides[-1]
        assert fuse_type in {"avg", "sum"}
        self._fuse_type = fuse_type

    # lateral_convs / output_convs are plain lists: keep them out of the module tree like upstream
    def __setattr__(self, name, value):
        if name in ("lateral_convs", "output_convs"):
            object.__setattr__(self, name, value)
        else:
            super().__setattr__(name, value)

    @property
    def size_divisibility(self):
        return self._size_divisibility

    def forward(self, x):
        bottom_up_features = self.bottom_up(x)
        results = []
        prev_features = self.lateral_convs[0](bottom_up_features[self.in_features[-1]])
        results.append(self.output_convs[0](prev_features))
        for idx, (lateral_conv, output_conv) in enumerate(zip(self.lateral_convs, self.output_convs)):
            if idx > 0:
                features = self.in_features[-idx - 1]
                features = bottom_up_features[features]
                top_down_features = F.interpolate(prev_features, scale_factor=2.0, mode="nearest")
                lateral_features = lateral_conv(features)
                prev_features = lateral_features + top_down_features
                if self._fuse_type == "avg":
                    prev_features /= 2
                results.insert(0, output_conv(prev_features))
        if self.top_block is not None:
            if self.top_block.in_feature in bottom_up_features:
                top_block_in_feature = bottom_up_features[self.top_block.in_feature]
            else:
                top_block_in_feature = results[self._out_features.index(self.top_block.in_feature)]
            results.extend(self.top_block(top_block_in_feature))
        assert len(self._out_features) == len(results)
        return {f: res for f, res in zip(self._out_features, results)}


# ----------------------------------------------------------------------------------------------
# pytorch3d.transforms (>= 0.5 algorithms)
# ----------------------------------------------------------------------------------------------
def quaternion_to_matrix(quaternions):
    r, i, j, k = torch.unbind(quaternions, -1)
    two_s = 2.0 / (quaternions * quaternions).sum(-1)
    o = torch.stack(
        (
            1 - two_s * (j * j + k * k),
            two_s * (i * j - k * r),
            two_s * (i * k + j * r),
            two_s * (i * j + k * r),
            1 - two_s * (i * i + k * k),
            two_s * (j * k - i * r),
            two_s * (i * k - j * r),
            two_s * (j * k + i * r),
            1 - two_s * (i * i + j * j),
        ),
        -1,
    )
    return o.reshape(quaternions.shape[:-1] + (3, 3))


def _sqrt_positive_part(x):
    ret = torch.zeros_like(x)
    positive_mask = x > 0
    ret[positive_mask] = torch.sqrt(x[positive_mask])
    return ret


def matrix_to_quaternion(matrix):
    if matrix.size(-1) != 3 or matrix.size(-2) != 3:
        raise ValueError(f"Invalid rotation matrix shape {matrix.shape}.")
    batch_dim = matrix.shape[:-2]
    m00, m01, m02, m10, m11, m12, m20, m21, m22 = torch.unbind(matrix.reshape(batch_dim + (9, )), dim=-1)
    q_abs = _sqrt_positive_part(
        torch.stack(
            [
                1.0 + m00 + m11 + m22,
                1.0 + m00 - m11 - m22,
                1.0 - m00 + m11 - m22,
                1.0 - m00 - m11 + m22,
            ],
            dim=-1,
        ))
    quat_by_rijk = torch.stack(
        [
            torch.stack([q_abs[..., 0]**2, m21 - m12, m02 - m20, m10 - m01], dim=-1),
            torch.stack([m21 - m12, q_abs[..., 1]**2, m10 + m01, m02 + m20], dim=-1),
            torch.stack([m02 - m20, m10 + m01, q_abs[..., 2]**2, m12 + m21], dim=-1),
            torch.stack([m10 - m01, m20 + m02, m21 + m12, q_abs[..., 3]**2], dim=-1),
        ],
        dim=-2,
    )
    flr = torch.tensor(0.1).to(dtype=q_abs.dtype, device=q_abs.device)
    quat_candidates = quat_by_rijk / (2.0 * q_abs[..., None].max(flr))
    return quat_candidates[F.one_hot(q_abs.argmax(dim=-1), num_classes=4) > 0.5, :].reshape(batch_dim + (4, ))


class Quaternion:
    """Minimal pyquaternion.Quaternion (w, x, y, z) -- the subset tridet/structures/pose.py and
    tridet/evaluators/kitti_3d_evaluator.py (convert_3d_box_to_kitti) use; semantics restated from pyquaternion 0.9.9
    (axis-angle constructor normalises the axis; `axis` = vector part / its norm, zeros when the rotation is the identity;
    `angle` = 2 * atan2(|vector|, scalar) wrapped to (-pi, pi])."""
    def __init__(self, *args, matrix=None, axis=None, radians=None, angle=None):
        import numpy as np
        if axis is not None:
            a = np.asarray(axis, dtype=np.float64)
            m2 = float(np.dot(a, a))
            if m2 == 0.0:
                raise ZeroDivisionError("Provided rotation axis has no length")
            if abs(1.0 - m2) > 1e-12:
                a = a / np.sqrt(m2)
            th = float(radians if radians is not None else angle) / 2.0
            self.q = np.concatenate([[np.cos(th)], a * np.sin(th)])
        elif len(args) == 4:
            self.q = np.asarray(args, dtype=np.float64)
        elif matrix is not None:
            m = np.asarray(matrix, dtype=np.float64)[:3, :3]
            q = matrix_to_quaternion(torch.tensor(m, dtype=torch.float64)[None])[0].numpy()
            if q[0] < 0:
                q = -q
            self.q = q / np.linalg.norm(q)
        elif len(args) == 1 and isinstance(args[0], Quaternion):
            self.q = args[0].q.copy()
        elif len(args) == 1:
            self.q = np.asarray(args[0], dtype=np.float64).copy()
        else:
            self.q = np.array([1.0, 0.0, 0.0, 0.0])

    @property
    def elements(self):
        return self.q

    @property
    def rotation_matrix(self):
        return quaternion_to_matrix(torch.tensor(self.q)[None])[0].numpy()

    def _unit(self):
        import numpy as np
        n = np.linalg.norm(self.q)
        return self.q / n if n > 0 else self.q

    @property
    def axis(self):
        import numpy as np
        v = self._unit()[1:]
        n = np.linalg.norm(v)
        return np.zeros(3) if n < 1e-17 else v / n

    @property
    def angle(self):
        import math
        import numpy as np
        u = self._unit()
        th = 2.0 * math.atan2(float(np.linalg.norm(u[1:])), float(u[0]))
        r = ((th + math.pi) % (2.0 * math.pi)) - math.pi
        return math.pi if r == -math.pi else r

    @property
    def transformation_matrix(self):
        import numpy as np
        m = np.eye(4)
        m[:3, :3] = self.rotation_matrix
        return m

    @property
    def inverse(self):
        import numpy as np
        return Quaternion(self.q * np.array([1.0, -1.0, -1.0, -1.0]) / np.dot(self.q, self.q))

    def rotate(self, v):
        import numpy as np
        return self.rotation_matrix @ np.asarray(v, dtype=np.float64)

    def __mul__(self, o):
        import numpy as np
        a, b = self.q, o.q
        return Quaternion(np.array([
            a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
            a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]]))

    def __eq__(self, o):
        import numpy as np
        return bool(np.allclose(self.q, o.q))

    def __repr__(self):
        return "%.3f %+.3fi %+.3fj %+.3fk" % tuple(self.q)


class _Transform3d:
    """Row-vector convention: p' = [p, 1] @ M. compose(a, b) applies a then b."""
    def __init__(self, matrix):
        self._matrix = matrix

    def compose(self, *others):
        m = self._matrix
        for o in others:
            m = torch.matmul(m, o._matrix)
        return _Transform3d(m)

    def get_matrix(self):
        return self._matrix

    def transform_points(self, points):
        ones = torch.ones(points.shape[:-1] + (1, ), dtype=points.dtype, device=points.device)
        ph = torch.cat([points, ones], dim=-1)
        out = torch.matmul(ph, self._matrix)
        return out[..., :3] / out[..., 3:]


def Transform3d(matrix=None, device="cpu", dtype=torch.float32):
    m = matrix if matrix.dim() == 3 else matrix[None]
    return _Transform3d(m)


def Rotate(R, device="cpu", dtype=torch.float32):
    if R.dim() == 2:
        R = R[None]
    n = R.shape[0]
    m = torch.eye(4, dtype=R.dtype, device=R.device).repeat(n, 1, 1)
    m[:, :3, :3] = R
    return _Transform3d(m)


def Translate(t, device="cpu", dtype=torch.float32):
    n = t.shape[0]
    m = torch.eye(4, dtype=t.dtype, device=t.device).repeat(n, 1, 1)
    m[:, 3, :3] = t
    return _Transform3d(m)


# ----------------------------------------------------------------------------------------------
# installation
# ----------------------------------------------------------------------------------------------
def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__spec__ = importlib.machinery.ModuleSpec(name, None)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


_INSTALLED = False
_THIRD_PARTY_INSTALLED = False


# ----------------------------------------------------------------------------------------------
# fvcore.transforms.transform / detectron2.data.transforms (restated; un-vendored third-party code)
# ----------------------------------------------------------------------------------------------
class Transform:
    """fvcore Transform: apply_box through the four corners, per-class registry of extra data types."""
    def _set_attributes(self, params=None):
        if params:
            for k, v in params.items():
                if k != "self" and not k.startswith("_"):
                    setattr(self, k, v)

    def apply_box(self, box):
        import numpy as np
        idxs = np.array([(0, 1), (2, 1), (0, 3), (2, 3)]).flatten()
        coords = np.asarray(box).reshape(-1, 4)[:, idxs].reshape(-1, 2)
        coords = self.apply_coords(coords).reshape((-1, 4, 2))
        minxy = coords.min(axis=1)
        maxxy = coords.max(axis=1)
        return np.concatenate((minxy, maxxy), axis=1)

    @classmethod
    def register_type(cls, data_type, func):
        def wrapper(transform, x):
            return func(transform, x)
        setattr(cls, "apply_" + data_type, wrapper)

    def inverse(self):
        raise NotImplementedError


class NoOpTransform(Transform):
    def apply_image(self, img):
        return img

    def apply_coords(self, coords):
        return coords

    def inverse(self):
        return self

    def __getattr__(self, name):
        if name.startswith("apply_"):
            return lambda x: x
        raise AttributeError("NoOpTransform object has no attribute {}".format(name))


class HFlipTransform(Transform):
    def __init__(self, width):
        self.width = width

    def apply_image(self, img):
        import numpy as np
        return np.flip(img, axis=1) if img.ndim <= 3 else np.flip(img, axis=-2)

    def apply_coords(self, coords):
        coords[:, 0] = self.width - coords[:, 0]
        return coords

    def inverse(self):
        return self


class VFlipTransform(Transform):
    def __init__(self, height):
        self.height = height

    def apply_image(self, img):
        import numpy as np
        return np.flip(img, axis=0)

    def apply_coords(self, coords):
        coords[:, 1] = self.height - coords[:, 1]
        return coords

    def inverse(self):
        return self


class TransformList(Transform):
    def __init__(self, transforms):
        flat = []
        for t in transforms:
            assert isinstance(t, Transform), t
            flat.extend(t.transforms if isinstance(t, TransformList) else [t])
        self.transforms = flat

    def _apply(self, x, meth):
        for t in self.transforms:
            x = getattr(t, meth)(x)
        return x

    def __getattr__(self, name):
        if name.startswith("apply_"):
            return lambda x: self._apply(x, name)
        raise AttributeError("TransformList object has no attribute {}".format(name))

    def __add__(self, other):
        others = other.transforms if isinstance(other, TransformList) else [other]
        return TransformList(self.transforms + others)

    def __radd__(self, other):
        others = other.transforms if isinstance(other, TransformList) else [other]
        return TransformList(others + self.transforms)

    def __len__(self):
        return len(self.transforms)

    def inverse(self):
        return TransformList([x.inverse() for x in self.transforms[::-1]])


class ResizeTransform(Transform):
    """detectron2 ResizeTransform: uint8 images through PIL (BILINEAR), coordinates scaled by new / old."""
    def __init__(self, h, w, new_h, new_w, interp=None):
        self.h, self.w, self.new_h, self.new_w, self.interp = h, w, new_h, new_w, interp

    def apply_image(self, img, interp=None):
        import numpy as np
        from PIL import Image
        assert img.shape[:2] == (self.h, self.w) and img.dtype == np.uint8
        pil = Image.fromarray(img).resize((self.new_w, self.new_h), Image.BILINEAR)
        return np.asarray(pil)

    def apply_coords(self, coords):
        coords[:, 0] = coords[:, 0] * (self.new_w * 1.0 / self.w)
        coords[:, 1] = coords[:, 1] * (self.new_h * 1.0 / self.h)
        return coords

    def inverse(self):
        return ResizeTransform(self.new_h, self.new_w, self.h, self.w, self.interp)


class ResizeShortestEdge:
    """detectron2 ResizeShortestEdge (sample_style "range" or "choice"; one size at test time)."""
    def __init__(self, short_edge_length, max_size=sys.maxsize, sample_style="range", interp=None):
        if isinstance(short_edge_length, int):
            short_edge_length = (short_edge_length, short_edge_length)
        self.short_edge_length, self.max_size, self.is_range = short_edge_length, max_size, sample_style == "range"

    def get_transform(self, image):
        import numpy as np
        h, w = image.shape[:2]
        if self.is_range:
            size = np.random.randint(self.short_edge_length[0], self.short_edge_length[1] + 1)
        else:
            size = np.random.choice(self.short_edge_length)
        if size == 0:
            return NoOpTransform()
        scale = size * 1.0 / min(h, w)
        if h < w:
            newh, neww = size, scale * w
        else:
            newh, neww = scale * h, size
        if max(newh, neww) > self.max_size:
            scale = self.max_size * 1.0 / max(newh, neww)
            newh = newh * scale
            neww = neww * scale
        return ResizeTransform(h, w, int(newh + 0.5), int(neww + 0.5))


class RandomFlip:
    def __init__(self, prob=0.5, *, horizontal=True, vertical=False):
        self.prob, self.horizontal = prob, horizontal

    def get_transform(self, image):
        import numpy as np
        h, w = image.shape[:2]
        if np.random.uniform() < self.prob:
            return HFlipTransform(w) if self.horizontal else VFlipTransform(h)
        return NoOpTransform()


def apply_augmentations(augmentations, image):
    tfms = []
    for aug in augmentations:
        t = aug.get_transform(image)
        image = t.apply_image(image)
        tfms.append(t)
    return image, TransformList(tfms)


def _noop(*a, **k):
    return None


def install_third_party():
    """Put the stand-in detectron2 / fvcore / pytorch3d / pyquaternion / mpi4py modules on the import path."""
    global _THIRD_PARTY_INSTALLED
    if _THIRD_PARTY_INSTALLED:
        return
    _THIRD_PARTY_INSTALLED = True
    _mod("detectron2")
    _mod("detectron2.config", configurable=configurable)
    _mod("detectron2.layers", Conv2d=Conv2d, get_norm=get_norm, cat=cat, batched_nms=batched_nms,
         FrozenBatchNorm2d=FrozenBatchNorm2d, ShapeSpec=ShapeSpec)
    _mod("detectron2.layers.nms", batched_nms_rotated=batched_nms_rotated, batched_nms=batched_nms)
    _mod("detectron2.structures", Instances=Instances, Boxes=Boxes, RotatedBoxes=RotatedBoxes)
    _mod("detectron2.modeling")
    _mod("detectron2.modeling.backbone", BACKBONE_REGISTRY=BACKBONE_REGISTRY, FPN=FPN, Backbone=Backbone)
    _mod("detectron2.modeling.backbone.build", BACKBONE_REGISTRY=BACKBONE_REGISTRY)
    _mod("detectron2.modeling.backbone.fpn", FPN=FPN, LastLevelMaxPool=LastLevelMaxPool,
         LastLevelP6P7=LastLevelP6P7)
    _mod("detectron2.modeling.meta_arch")
    _mod("detectron2.modeling.meta_arch.build", META_ARCH_REGISTRY=META_ARCH_REGISTRY)
    _mod("detectron2.modeling.postprocessing", detector_postprocess=detector_postprocess)
    _mod("detectron2.utils")
    _mod("detectron2.utils.comm", get_world_size=lambda: 1, get_rank=lambda: 0, is_main_process=lambda: True)
    _mod("detectron2.utils.env", TORCH_VERSION=tuple(int(x) for x in torch.__version__.split(".")[:2]))

    wi = _mod("fvcore.nn.weight_init", c2_msra_fill=_c2_msra_fill, c2_xavier_fill=_c2_xavier_fill)
    _mod("fvcore")
    sl1 = _mod("fvcore.nn.smooth_l1_loss", smooth_l1_loss=_noop)
    _mod("fvcore.nn", sigmoid_focal_loss=_noop, smooth_l1_loss=sl1, weight_init=wi)

    rc = _mod("pytorch3d.transforms.rotation_conversions", quaternion_to_matrix=quaternion_to_matrix,
              matrix_to_quaternion=matrix_to_quaternion)
    t3d = _mod("pytorch3d.transforms.transform3d", Rotate=Rotate, Translate=Translate, Transform3d=Transform3d)
    _mod("pytorch3d")
    _mod("pytorch3d.transforms", rotation_conversions=rc, transform3d=t3d,
         quaternion_to_matrix=quaternion_to_matrix, matrix_to_quaternion=matrix_to_quaternion)

    _mod("pyquaternion", Quaternion=Quaternion)
    _mod("mpi4py", MPI=types.SimpleNamespace(COMM_WORLD=None))


def install(reference_root=REFERENCE_ROOT):
    """Put the stand-in modules and the reference's `tridet` package on the import path."""
    global _INSTALLED
    if _INSTALLED:
        return
    _INSTALLED = True
    install_third_party()

    # The reference's package __init__ files pull in the nuScenes devkit / TTA wrappers; stub the
    # package nodes (not the hot-path modules) so `tridet.modeling.dd3d.core` imports verbatim.
    if reference_root not in sys.path:
        sys.path.insert(0, reference_root)
    import os
    for pkg in ("tridet", "tridet.modeling", "tridet.modeling.dd3d", "tridet.layers", "tridet.structures",
                "tridet.utils"):
        m = types.ModuleType(pkg)
        m.__path__ = [os.path.join(reference_root, *pkg.split("."))]
        m.__spec__ = importlib.machinery.ModuleSpec(pkg, None, is_package=True)
        sys.modules[pkg] = m
    # tridet.layers.__init__ exports (bev_nms needs detectron2 rotated NMS: stubbed above)
    from tridet.layers.iou_loss import IOULoss  # noqa: E402
    from tridet.layers.smooth_l1_loss import smooth_l1_loss  # noqa: E402
    sys.modules["tridet.layers"].IOULoss = IOULoss
    sys.modules["tridet.layers"].smooth_l1_loss = smooth_l1_loss
    from tridet.layers.bev_nms import bev_nms  # noqa: E402  (the reference's own BEV NMS, rotated IoU from the stand-in)
    sys.modules["tridet.layers"].bev_nms = bev_nms
    _mod("tridet.utils.comm", reduce_sum=lambda x: x, get_world_size=lambda: 1)
    # NuscenesDD3D (nuscenes_dd3d.py:13) only needs the constant from the devkit-dependent dataset builder
    for pkg in ("tridet.data", "tridet.data.datasets", "tridet.data.datasets.nuscenes", "tridet.data.augmentations"):
        m = types.ModuleType(pkg)
        m.__path__ = [os.path.join(reference_root, *pkg.split("."))]
        m.__spec__ = importlib.machinery.ModuleSpec(pkg, None, is_package=True)
        sys.modules[pkg] = m

    # fvcore.transforms / detectron2.data.transforms: the transform machinery the dataset mapper and the TTA wrapper use
    _mod("fvcore.transforms", NoOpTransform=NoOpTransform, HFlipTransform=HFlipTransform, VFlipTransform=VFlipTransform,
         Transform=Transform, TransformList=TransformList)
    _mod("fvcore.transforms.transform", NoOpTransform=NoOpTransform, HFlipTransform=HFlipTransform,
         VFlipTransform=VFlipTransform, Transform=Transform, TransformList=TransformList)
    _mod("detectron2.data")
    _mod("detectron2.data.detection_utils", read_image=_noop)
    _mod("detectron2.data.transforms", ResizeTransform=ResizeTransform, ResizeShortestEdge=ResizeShortestEdge,
         RandomFlip=RandomFlip, apply_augmentations=apply_augmentations)
    # the reference's own registrations of intrinsics / box3d handlers on those classes
    import tridet.data.augmentations.resize_transform  # noqa: F401,E402
    import tridet.data.augmentations.flip_transform  # noqa: F401,E402
    _mod("tridet.data.datasets.nuscenes.build", MAX_NUM_ATTRIBUTES=3)  # tridet/data/datasets/nuscenes/build.py:77


def _c2_msra_fill(module):
    nn.init.kaiming_normal_(module.weight, mode="fan_out", nonlinearity="relu")
    if module.bias is not None:
        nn.init.constant_(module.bias, 0)


def _c2_xavier_fill(module):
    nn.init.kaiming_uniform_(module.weight, a=1)
    if module.bias is not None:
        nn.init.constant_(module.bias, 0)


def build_reference_model(cfg):
    """Instantiate the reference's own DD3D (tridet/modeling/dd3d/core.py:19) under the stand-in."""
    install()
    if cfg.MODEL.META_ARCHITECTURE == "NuscenesDD3D":  # tridet/modeling/dd3d/nuscenes_dd3d.py:301
        from tridet.modeling.dd3d.nuscenes_dd3d import NuscenesDD3D
        return NuscenesDD3D(cfg)
    from tridet.modeling.dd3d.core import DD3D
    return DD3D(cfg)


# ------------------------------------------------------------------------------------------------------------------
# Evaluator side (tridet/evaluators/kitti_3d_evaluator.py): the detectron2 / iopath names it imports, and the dataset
# catalog it reads.  Only process() is exercised (the CPU half of the evaluator: per-detection conversion to KITTI
# rows); evaluate() needs numba.cuda (rotate_iou.py selects a CUDA device at import), so that module is stubbed.
# ------------------------------------------------------------------------------------------------------------------
class BoxMode:
    """detectron2.structures.BoxMode subset: the two modes the KITTI evaluator converts between."""
    XYXY_ABS, XYWH_ABS = 0, 1

    @staticmethod
    def convert(box, from_mode, to_mode):
        if from_mode == to_mode:
            return box
        x0, y0, a, b = [float(v) for v in box]
        if from_mode == BoxMode.XYXY_ABS and to_mode == BoxMode.XYWH_ABS:
            return type(box)([x0, y0, a - x0, b - y0]) if isinstance(box, (list, tuple)) else [x0, y0, a - x0, b - y0]
        if from_mode == BoxMode.XYWH_ABS and to_mode == BoxMode.XYXY_ABS:
            return type(box)([x0, y0, x0 + a, y0 + b]) if isinstance(box, (list, tuple)) else [x0, y0, x0 + a, y0 + b]
        raise NotImplementedError((from_mode, to_mode))


class _Catalog(dict):
    def register(self, name, value):
        self[name] = value

    def get(self, name):  # DatasetCatalog: callable -> list[dict]; MetadataCatalog: metadata object
        v = self[name]
        return v() if callable(v) else v


DatasetCatalog = _Catalog()
MetadataCatalog = _Catalog()


class DatasetEvaluator:
    def reset(self):
        pass

    def process(self, inputs, outputs):
        pass

    def evaluate(self):
        pass


def install_evaluator_stubs():
    install()
    _mod("detectron2.data.catalog", DatasetCatalog=DatasetCatalog, MetadataCatalog=MetadataCatalog)
    _mod("detectron2.evaluation")
    _mod("detectron2.evaluation.evaluator", DatasetEvaluator=DatasetEvaluator)
    _mod("detectron2.structures.boxes", BoxMode=BoxMode, Boxes=Boxes)

    class _PathManager:
        def mkdirs(self, path):
            import os
            os.makedirs(path, exist_ok=True)

    _mod("iopath")
    _mod("iopath.common")
    _mod("iopath.common.file_io", PathManager=_PathManager)
    import os
    m = types.ModuleType("tridet.evaluators")
    m.__path__ = [os.path.join(REFERENCE_ROOT, "tridet", "evaluators")]
    m.__spec__ = importlib.machinery.ModuleSpec("tridet.evaluators", None, is_package=True)
    sys.modules["tridet.evaluators"] = m
    _mod("tridet.evaluators.rotate_iou", d3_box_overlap_kernel=None, rotate_iou_gpu_eval=None)
    # detectron2.utils.comm.gather / synchronize are only reached from evaluate()
