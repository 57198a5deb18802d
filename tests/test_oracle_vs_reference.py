"""Pin the oracle and the product's geometry against the reference.

``oracle/ref_loader.py`` slices the reference's own functions out of a checkout
of the original MVSDet project (``MVSDET_REFERENCE_ROOT``) and executes them
verbatim; with it, fresh seeded scenes -- not the ones frozen in tests/golden --
go through both the reference chain (tests/golden/make_golden.py: mvsdet.py:404-515
followed statement by statement) and ``oracle.hot_path``.  The repository does
not contain that checkout, so the tests that need it skip without it; the
geometry comparison falls back to the reference outputs stored in tests/golden.
"""
import importlib.util
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN_CASES, assert_close, load_golden, oracle_chain
from mvsdet_b200.scene import make_scene, tiny_config
from oracle import ref_loader

needs_reference = pytest.mark.skipif(
    not ref_loader.available(),
    reason="needs a checkout of the original MVSDet project in MVSDET_REFERENCE_ROOT")

CASES = [
    (tiny_config(n_views=6, channels=8, num_depth=8), 101),
    (tiny_config(n_views=3, channels=8, num_depth=4, topk=2, per_view_intrinsics=True,
                 near_far_range=(0.5, 5.5)), 102),
    (tiny_config(n_views=7, channels=4, num_depth=16, topk=3, n_voxels=(10, 8, 4)), 103),
]


def _make_golden_module():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_golden.py")
    spec = importlib.util.spec_from_file_location("_make_golden", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def ref():
    return ref_loader.load()


@needs_reference
@pytest.mark.parametrize("cfg,seed", CASES)
def test_oracle_equals_live_reference(ref, cfg, seed):
    mg = _make_golden_module()
    scene = make_scene(cfg, seed)
    want = mg.reference_chain(ref, scene)
    got = oracle_chain(scene)
    for key in ("neighbor_ids", "est_idx", "valid", "count"):
        assert np.array_equal(got[key].numpy(), want[key].numpy()), key
    for key in ("variance", "prob_volume", "off_pred", "est_depth", "est_densities",
                "depth_coding", "volume_mean", "projection", "points",
                "g_feature_from_variance", "g_feature_from_voxels", "g_cost_out"):
        assert_close(got[key], want[key], rtol=1e-6, atol=1e-6, what=key)


def test_geometry_mirrors_equal_live_reference():
    """The product's host-side geometry (mvsdet_b200/geometry.py) against the
    reference's knn / get_nearest_pose_ids / collect_proj / get_points /
    _compute_projection: bit for bit against their outputs stored in tests/golden
    for the golden scenes and, with the reference checkout, live on one more camera set."""
    from mvsdet_b200 import geometry as G
    for case in GOLDEN_CASES:
        scene, gold = load_golden(case)
        cfg, meta = scene["cfg"], scene["img_meta"]
        w2c = torch.tensor(np.array(meta["lidar2img"]["extrinsic"]))
        c2w = w2c.inverse()
        nbr = G.get_nearest_pose_ids(c2w, c2w, min(2, cfg.n_views - 1), maskself=True)   # mvsdet.py:432-434
        assert np.array_equal(nbr.numpy(), gold["neighbor_ids"]), case
        kf = G.feature_intrinsics(torch.tensor(np.array(meta["lidar2img"]["intrinsic"])), cfg.ratio)
        ref_proj, nei_projs = G.collect_proj(w2c, kf, nbr)
        assert np.array_equal(ref_proj.numpy(), gold["ref_proj"]), case
        assert np.array_equal(torch.stack(nei_projs).numpy(), gold["nei_projs"]), case
        assert np.array_equal(G.compute_projection(meta, cfg.stride).numpy(), gold["projection"]), case
        points = G.get_points(cfg.n_voxels, cfg.voxel_size, meta["lidar2img"]["origin"])
        assert np.array_equal(points.numpy(), gold["points"]), case
    if not ref_loader.available():
        return
    ref = ref_loader.load()
    cfg = tiny_config(n_views=9, channels=4)
    scene = make_scene(cfg, 7)
    meta = scene["img_meta"]
    w2c = torch.tensor(np.array(meta["lidar2img"]["extrinsic"]))
    c2w = w2c.inverse()
    a = ref.get_nearest_pose_ids(c2w, c2w, 2, maskself=True)
    b = G.get_nearest_pose_ids(c2w, c2w, 2, maskself=True)
    assert torch.equal(a, b)
    self = ref_loader.make_self(cfg.near_far_range, cfg.num_depth)
    intr = torch.tensor(np.array(meta["lidar2img"]["intrinsic"]))
    kf = G.feature_intrinsics(intr, cfg.ratio)
    pa, na = ref.collect_proj(self, w2c, kf, a)
    pb, nb = G.collect_proj(w2c, kf, b)
    assert torch.equal(pa, pb) and all(torch.equal(x, y) for x, y in zip(na, nb))
    assert torch.equal(ref._compute_projection(meta, cfg.stride, None),
                       G.compute_projection(meta, cfg.stride))
    pts = ref.get_points(n_voxels=torch.tensor(cfg.n_voxels), voxel_size=torch.tensor(cfg.voxel_size),
                         origin=torch.tensor(meta["lidar2img"]["origin"]))
    assert torch.equal(pts, G.get_points(cfg.n_voxels, cfg.voxel_size, meta["lidar2img"]["origin"]))


@needs_reference
def test_costreg_restatement_equals_reference_class():
    """oracle/costreg_oracle.CostRegNet3DGS (what the GPU tests attach to the drop-in) against the
    reference's CostRegNet_3DGS (mvs_models/mvsnet.py:73-113), loaded under a synthetic package
    because mvsnet.py uses ``from .module import *``: same state_dict keys and shapes, same
    output with the same weights."""
    import sys
    import types
    from oracle import costreg_oracle
    root = os.path.join(ref_loader.REFERENCE_ROOT, "projects", "NeRF-Det", "nerfdet", "mvs_models")
    pkg = types.ModuleType("_ref_mvs_models")
    pkg.__path__ = [root]
    sys.modules["_ref_mvs_models"] = pkg
    for name in ("module", "mvsnet"):
        spec = importlib.util.spec_from_file_location(f"_ref_mvs_models.{name}", os.path.join(root, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = mod
        spec.loader.exec_module(mod)
    torch.manual_seed(0)
    theirs = sys.modules["_ref_mvs_models.mvsnet"].CostRegNet_3DGS()
    mine = costreg_oracle.CostRegNet3DGS()
    sd = theirs.state_dict()
    assert list(sd.keys()) == list(mine.state_dict().keys())
    assert all(sd[k].shape == v.shape for k, v in mine.state_dict().items())
    assert sum(p.numel() for p in mine.parameters()) == 4871554          # SURVEY.md 8c
    mine.load_state_dict(sd)
    x = torch.randn(1, 256, 4, 8, 8)
    for train in (False, True):
        theirs.train(train)
        mine.train(train)
        assert torch.equal(theirs(x.clone()), mine(x.clone()))


@needs_reference
def test_group_correlation_equals_reference_statements(ref):
    """SURVEY 8f rank 4: the oracle's group-wise correlation against the reference's own statements
    (mvs_models/lss_fpn.py:496-503, sliced and executed verbatim) fed with the reference's own
    homo_warping of the same neighbours."""
    from oracle import mvsdet_oracle as O
    cfg = tiny_config(n_views=5, channels=32, num_depth=6)
    scene = make_scene(cfg, 211)
    feature = scene["feature"]
    groups = 8
    got = O.scene_group_correlation(feature, scene["img_meta"], near_far_range=cfg.near_far_range,
                                    num_depth=cfg.num_depth, num_groups=groups, stride=cfg.stride)
    stmts = ref_loader.group_correlation_statements()
    v = feature.shape[0]
    ratio = scene["img_meta"]["ori_shape"][0] / (scene["img_meta"]["img_shape"][0] / cfg.stride)
    w2c = torch.as_tensor(np.array(scene["img_meta"]["lidar2img"]["extrinsic"]))
    k_feat = O.feature_intrinsics(torch.as_tensor(np.array(scene["img_meta"]["lidar2img"]["intrinsic"])), ratio)
    nbr = ref.get_nearest_pose_ids(w2c.inverse(), w2c.inverse(), 2, maskself=True)       # mvsdet.py:434
    proj = torch.matmul(k_feat.unsqueeze(0).repeat(v, 1, 1), w2c)
    dvals = torch.as_tensor(O.depth_values_for(cfg.near_far_range, cfg.num_depth)).unsqueeze(0).repeat(v, 1)
    assert tuple(got.shape) == (v, 2, groups, cfg.num_depth, *cfg.feat_hw)
    for j in range(2):
        warped = ref.homo_warping(feature[nbr[:, j]], proj[nbr[:, j]], proj, dvals)
        want = stmts(feature, warped, groups)
        assert_close(got[:, j], want, rtol=1e-6, atol=1e-6, what=f"group correlation, neighbour {j}")
