"""dd3d_b200/config.py restates the reference's hydra config tree; this pins it: every key get_cfg() carries must equal the
value hydra would resolve for the four shipped DD3D experiments (configs/experiments/dd3d_{kitti,nusc}_{dla34,v99}.yaml on
top of configs/defaults.yaml).  The resolved experiments are recorded in tests/golden/reference_configs.json, composed
from the reference's config tree with PyYAML + tests/hydra_lite.py by oracle/gen_golden.py.  The key list is also checked
so config.py cannot silently drop a key the reference's DD3D.__init__ reads."""
import json
import os

import pytest

from conftest import GOLDEN_DIR
from dd3d_b200.config import get_cfg

EXPERIMENTS = [  # experiment file, get_cfg arguments
    ("dd3d_kitti_dla34", dict(backbone="dla34", dataset="kitti_3d", meta_arch="DD3D")),
    ("dd3d_kitti_v99", dict(backbone="v2_99", dataset="kitti_3d", meta_arch="DD3D")),
    ("dd3d_nusc_dla34", dict(backbone="dla34", dataset="nuscenes", meta_arch="NuscenesDD3D")),
    ("dd3d_nusc_v99", dict(backbone="v2_99", dataset="nuscenes", meta_arch="NuscenesDD3D")),
]
ENGINE_ONLY = {"B200"}  # keys of the engine, absent from the reference
# values that legitimately differ: CKPT is a URL in the experiments (no network here, weights are synthetic)
IGNORED = {("MODEL", "CKPT")}


def _leaves(node, trail=()):
    for k, v in node.items():
        if isinstance(v, dict):
            yield from _leaves(v, trail + (k, ))
        else:
            yield trail + (k, ), v


def _lookup(cfg, path):
    for p in path:
        cfg = cfg[p]
    return cfg


def reference_experiment(name):
    with open(os.path.join(GOLDEN_DIR, "reference_configs.json")) as f:
        return json.load(f)[name]


def _same(a, b):
    if isinstance(a, (list, tuple)) and isinstance(b, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    if isinstance(a, float) or isinstance(b, float):
        return a is not None and b is not None and abs(float(a) - float(b)) <= 1e-9 * max(1.0, abs(float(b)))
    return a == b


@pytest.mark.parametrize("experiment,args", EXPERIMENTS, ids=[e for e, _ in EXPERIMENTS])
def test_config_equals_resolved_reference_experiment(experiment, args):
    ref = reference_experiment(experiment)
    ours = get_cfg(**args)
    bad = []
    for path, val in _leaves(ours):
        if path[0] in ENGINE_ONLY or path in IGNORED:
            continue
        try:
            want = _lookup(ref, path)
        except (KeyError, TypeError):
            bad.append((path, val, "<absent in the reference config>"))
            continue
        if not _same(val, want):
            bad.append((path, val, want))
    assert not bad, "\n".join(f"{'.'.join(p)}: config.py {a!r} != reference {b!r}" for p, a, b in bad)


def test_every_dd3d_key_of_the_reference_is_mirrored():
    """DD3D.__init__ / the heads read cfg.DD3D.*, cfg.FE.*, cfg.MODEL.*: config.py must carry every leaf of those subtrees."""
    ref = reference_experiment("dd3d_nusc_v99")
    ours = get_cfg("v2_99", "nuscenes", meta_arch="NuscenesDD3D")
    missing = []
    for top in ("DD3D", "FE", "MODEL"):
        for path, _ in _leaves(ref[top], (top, )):
            try:
                _lookup(ours, path)
            except (KeyError, TypeError):
                missing.append(".".join(path))
    assert not missing, missing
