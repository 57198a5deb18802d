"""Loader for the UNMODIFIED reference functions of the MVSDet hot path.

TEST INFRASTRUCTURE ONLY.  This module executes the reference's own Python
source from a checkout of the original MVSDet project named by the environment
variable ``MVSDET_REFERENCE_ROOT``; the repository does not contain one.  Nothing
is copied into this repository: the functions are sliced out of the reference
files with ``ast`` at call time and ``exec``-ed in a scratch namespace, exactly
as SURVEY.md section 8(c) describes.

It is used for two things only:
  * ``tests/golden/make_golden.py`` -- generate the committed golden vectors;
  * ``tests/test_oracle_vs_reference.py`` -- pin ``oracle/mvsdet_oracle.py``
    against the live reference when the checkout is given (skipped otherwise).

Reference entry points loaded (all under projects/NeRF-Det/nerfdet/):
  mvs_models/module.py:105-146   homo_warping
  mvsdet.py:43-64                knn
  mvsdet.py:67-104               get_nearest_pose_ids
  mvsdet.py:249-264              MVSDet.collect_proj
  mvsdet.py:266-283              MVSDet.sample_depth_prob
  mvsdet.py:298-317              MVSDet.compute_avg_depth
  mvsdet.py:1124-1156            MVSDet._compute_projection
  mvsdet.py:1316-1327            get_points
  mvsdet.py:1372-1492            backproject_Weigh
  mvsdet.py:1158-1218            MVSDet.compute_depth_scale, compute_depth_scale_MultiIntrin
  mvsdet.py:1272-1313            get_camera_params, lift
  mvsdet.py:319-333              MVSDet.process_rgb_raw
The last two groups call ``.cuda()`` on freshly created tensors (mvsdet.py:1283, :1302, :1313);
``cpu_cuda_shim()`` makes ``Tensor.cuda`` the identity so they run on the CPU
-- the executed source is still the reference's, unmodified.
"""
from __future__ import annotations

import ast
import importlib.util
import math
import os
import types
import warnings

REFERENCE_ROOT = os.environ.get("MVSDET_REFERENCE_ROOT", "")
_NERFDET = os.path.join(REFERENCE_ROOT, "projects", "NeRF-Det", "nerfdet")

_FREE_FUNCS = ("knn", "get_nearest_pose_ids", "get_points", "backproject_Weigh",
               "get_camera_params", "lift")
_METHODS = ("collect_proj", "sample_depth_prob", "compute_avg_depth",
            "_compute_projection", "compute_depth_scale", "compute_depth_scale_MultiIntrin",
            "process_rgb_raw")


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(_NERFDET, "mvsdet.py"))


def _load_module_py():
    path = os.path.join(_NERFDET, "mvs_models", "module.py")
    spec = importlib.util.spec_from_file_location("_mvsdet_ref_module", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load() -> types.SimpleNamespace:
    """Return a namespace holding the reference callables (see module doc)."""
    if not available():
        raise FileNotFoundError(
            f"no MVSDet checkout at MVSDET_REFERENCE_ROOT={REFERENCE_ROOT!r}; set it to the "
            "root of the original project")
    import numpy as np
    import torch
    import torch.nn.functional as F

    warnings.filterwarnings("ignore", message=".*torch.meshgrid.*")
    warnings.filterwarnings("ignore", message=".*align_corners.*")

    ns: dict = {"torch": torch, "np": np, "F": F, "math": math}
    src_path = os.path.join(_NERFDET, "mvsdet.py")
    with open(src_path, "r") as fh:
        tree = ast.parse(fh.read(), filename=src_path)

    picked: list = []
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in _FREE_FUNCS:
            picked.append(node)
        elif isinstance(node, ast.ClassDef) and node.name == "MVSDet":
            for sub in node.body:
                if isinstance(sub, ast.FunctionDef) and sub.name in _METHODS:
                    # strip decorators we cannot resolve except staticmethod
                    picked.append(sub)
    module = ast.Module(body=picked, type_ignores=[])
    exec(compile(module, src_path, "exec"), ns)  # noqa: S102 - reference code

    out = types.SimpleNamespace()
    for name in _FREE_FUNCS + _METHODS:
        setattr(out, name, ns[name])
    out.homo_warping = _load_module_py().homo_warping
    return out


class cpu_cuda_shim:
    """Context manager: ``Tensor.cuda()`` returns the tensor itself (the reference code runs on the CPU)."""

    def __enter__(self):
        import torch
        self._orig = torch.Tensor.cuda
        torch.Tensor.cuda = lambda self_, *a, **k: self_
        return self

    def __exit__(self, *exc):
        import torch
        torch.Tensor.cuda = self._orig
        return False


def make_self(near_far_range, num_depth):
    """Stand-in for the detector instance the sliced methods expect as `self`.

    Mirrors the attributes set in MVSDet.__init__ (mvsdet.py:171,222-225).
    """
    import numpy as np
    self = types.SimpleNamespace()
    self.near_far_range = list(near_far_range)
    self.gs_cfg = types.SimpleNamespace(num_monocular_samples=int(num_depth))
    self.depth_interval = (near_far_range[1] - near_far_range[0]) / num_depth
    self.depth_values = np.arange(near_far_range[0], near_far_range[1],
                                  self.depth_interval, dtype=np.float32)
    assert len(self.depth_values) == num_depth
    return self


def group_correlation_statements():
    """The reference's group-wise correlation arithmetic, executed verbatim: the three assignments
    of ``LSSFPN._generate_cost_volume`` (mvs_models/lss_fpn.py:496-503) that reshape the warped and the
    reference features into channel groups and take ``torch.mean(ref.unsqueeze(3) * warped, axis=2)``.
    ``lss_fpn.py`` cannot be imported (mmdet), so the statements are sliced out with ``ast``.

    -> f(ref_feat [B,C,H,W], warped [B,C,D,H,W], num_groups) -> feat_cost [B,G,D,H,W]"""
    import torch
    path = os.path.join(_NERFDET, "mvs_models", "lss_fpn.py")
    with open(path, "r") as fh:
        tree = ast.parse(fh.read(), filename=path)
    fn = None
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == "_generate_cost_volume":
            fn = node
    if fn is None:
        raise RuntimeError("lss_fpn.py: _generate_cost_volume not found")
    wanted = []
    for node in ast.walk(fn):
        if isinstance(node, ast.Assign) and len(node.targets) == 1 and isinstance(node.targets[0], ast.Name):
            name = node.targets[0].id
            src = ast.unparse(node.value)
            if (name == "warped_stereo_fea" and ".reshape(" in src and "homo_warping" not in src) \
                    or name in ("ref_stereo_feat", "feat_cost"):
                wanted.append(node)
    wanted.sort(key=lambda n: n.lineno)
    if [n.targets[0].id for n in wanted] != ["warped_stereo_fea", "ref_stereo_feat", "feat_cost"]:
        raise RuntimeError("lss_fpn.py: unexpected shape of the group-correlation statements")
    code = compile(ast.Module(body=wanted, type_ignores=[]), path, "exec")

    def run(ref_feat, warped, num_groups):
        b, c, h, w = ref_feat.shape
        ns = {"torch": torch, "self": types.SimpleNamespace(num_groups=num_groups, num_samples=warped.shape[2]),
              "batch_size": b, "num_channels": c, "height": h, "width": w,
              "stereo_feats_all_sweeps": [ref_feat], "sweep_index": 0, "warped_stereo_fea": warped}
        exec(code, ns)  # noqa: S102 - reference code
        return ns["feat_cost"]
    return run
