"""The own-view forward of a view-sharded scene, the parts that run without a GPU: ``mvsd_halo_gather_p2p`` is
declared, exported and typed, and rejects every malformed request in its own name before any launch;
``sharded.halo_gather_table`` points every halo row of a rank at its owner's row of that view, so gathering
from the owners' own-view buffers rebuilds the block + halo buffer the replicated-input forms pack; and
``sharded.owned_views`` names the views ``ShardedScenePipeline.load`` has always given a rank."""
import ctypes
import os
import re

import pytest
import torch

import test_abi as A
from mvsdet_b200 import _lib as L_
from mvsdet_b200 import geometry as G
from mvsdet_b200 import sharded
from mvsdet_b200.hotpath import MVSDetHotPath
from mvsdet_b200.scene import SceneConfig, make_scene

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRY = "mvsd_halo_gather_p2p"


# ---- the symbol: header, export, ctypes table ----------------------------------------------------------------
def test_gather_is_declared_exported_and_typed():
    with open(os.path.join(REPO, "include", "mvsdet_b200.h")) as fh:
        header = fh.read()
    decl = re.search(r"int mvsd_halo_gather_p2p\(([^)]*)\);", header)
    assert decl, "mvsd_halo_gather_p2p is not declared in the header"
    params = [p.strip() for p in decl.group(1).split(",")]
    assert params == ["void* const* feat_ptrs", "const int32_t* gather_sources", "int world", "int rank",
                      "int n_own", "int n_halo", "int64_t view_bytes", "void* stream"]
    assert L_.SIGNATURES[ENTRY] == ([ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 4
                                    + [ctypes.c_int64, ctypes.c_void_p], ctypes.c_int)
    lib = A._build_if_needed().load()
    fn = getattr(lib, ENTRY)
    assert fn.argtypes == L_.SIGNATURES[ENTRY][0] and fn.restype is ctypes.c_int
    assert lib.mvsd_abi_version() == L_.ABI_VERSION == 3


# ---- argument checks: the rules of mvsd_halo_reduce_p2p in the same order, plus n_halo and 8-byte rows ----------
_ARGS = ("feat_ptrs", "src", "world", "rank", "n_own", "n_halo", "view_bytes", "stream")
_VALID = dict(feat_ptrs=True, src=True, world=2, rank=1, n_own=3, n_halo=2, view_bytes=64, stream=None)
_SIZE = "halo_gather_p2p: bad view count / size"
_RULES = [
    *[(f"null-{p}", {p: False}, "halo_gather_p2p: null pointer") for p in ("feat_ptrs", "src")],
    ("world=0", {"world": 0, "rank": 0}, "halo_gather_p2p: bad world/rank (0/0)"),
    ("world>16", {"world": 17}, "halo_gather_p2p: bad world/rank (1/17)"),
    ("rank<0", {"rank": -1}, "halo_gather_p2p: bad world/rank (-1/2)"),
    ("rank=world", {"rank": 2}, "halo_gather_p2p: bad world/rank (2/2)"),
    ("n_own=0", {"n_own": 0}, _SIZE),
    ("n_own>65535", {"n_own": 65536}, _SIZE),
    ("n_halo=0", {"n_halo": 0}, _SIZE),
    ("n_halo<0", {"n_halo": -1}, _SIZE),
    ("n_halo>65535", {"n_halo": 65536}, _SIZE),
    ("view_bytes=0", {"view_bytes": 0}, _SIZE),
    ("view_bytes<0", {"view_bytes": -8}, _SIZE),
    *[(f"view_bytes%8={r}", {"view_bytes": 64 + r}, _SIZE) for r in (1, 2, 4, 6)],
    ("null-before-world", {"feat_ptrs": False, "world": 0}, "halo_gather_p2p: null pointer"),
    ("world-before-size", {"world": 0, "view_bytes": 3}, "halo_gather_p2p: bad world/rank (1/0)"),
]


@pytest.mark.parametrize("overrides,message", [pytest.param(o, m, id=r) for r, o, m in _RULES])
def test_gather_rejects_before_any_launch(overrides, message):
    lib = A._build_if_needed().load()
    args = {**_VALID, **overrides}
    dummy = ctypes.c_void_p(16)
    before = lib.mvsd_launch_count()
    st = getattr(lib, ENTRY)(*[(dummy if args[p] else None) if p in ("feat_ptrs", "src") else args[p]
                               for p in _ARGS])
    assert lib.mvsd_launch_count() == before
    assert (st, lib.mvsd_last_error().decode()) == (L_.ERR_INVALID_ARG, message)


def test_gather_launcher_raises_with_its_name(monkeypatch):
    """the Python launcher passes n_halo as the table's rows and reports the C-side rejection as ValueError"""
    A._build_if_needed()
    monkeypatch.setattr(L_, "_stream", lambda: 0)
    with pytest.raises(ValueError, match=r"^mvsd_halo_gather_p2p: halo_gather_p2p: bad view count / size$"):
        L_.halo_gather_p2p(16, torch.zeros((65536, 2), dtype=torch.int32), world=2, rank=0, n_own=2, view_bytes=64)
    with pytest.raises(ValueError, match=r"^mvsd_halo_gather_p2p: halo_gather_p2p: bad view count / size$"):
        L_.halo_gather_p2p(16, torch.zeros((1, 2), dtype=torch.int32), world=2, rank=0, n_own=2, view_bytes=36)


# ---- halo_gather_table ---------------------------------------------------------------------------------------
CASES = [(8, 2), (20, 3), (20, 4), (80, 8), (5, 8)]


def _hot(cfg):
    return MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                         stride=cfg.stride)


def _scene_ids(v, world, pose_clustered):
    """whole-scene neighbour ids of a synthetic scan in the numbering the ranks shard"""
    cfg = SceneConfig(n_views=v)
    scene = make_scene(cfg, seed=7, with_grads=False)
    order, meta, nbr = sharded._view_plan(_hot(cfg), scene["img_meta"], world, pose_clustered)
    return order, nbr


@pytest.mark.parametrize("pose_clustered", [False, True], ids=["index", "pose"])
@pytest.mark.parametrize("v,world", CASES)
def test_gather_table_points_at_each_halo_views_owner_row(v, world, pose_clustered):
    order, nbr = _scene_ids(v, world, pose_clustered)
    assert sorted(order) == list(range(v)) and (pose_clustered or order == list(range(v)))
    blocks = [sharded.partition_views(v, world, q) for q in range(world)]
    g = torch.Generator().manual_seed(v * 10 + world)
    feature = torch.randn((v, 3, 2, 2), generator=g)                 # in the sharded numbering
    own_bufs = [feature[b:e].clone() for b, e in blocks]             # what each owner packs: its own views only
    n_halo_total = 0
    for r, (b, e) in enumerate(blocks):
        src = sharded.halo_gather_table(nbr, world, r)
        assert src.dtype == torch.int32 and src.dim() == 2 and src.shape[1] == 2
        if e <= b:
            assert src.shape[0] == 0
            continue
        views, _ = sharded.halo_views(nbr[b:e], b, e)
        assert src.shape[0] == len(views) - (e - b)
        for j, (q, row) in enumerate(src.tolist()):
            qb, qe = blocks[q]
            assert q != r, "a halo row never points at the rank itself"
            assert 0 <= row < qe - qb and qb + row == views[e - b + j]
        local = torch.cat([own_bufs[r]] + [own_bufs[q][row:row + 1] for q, row in src.tolist()])
        assert torch.equal(local, feature[views]), f"rank {r}: gathered rows differ from feature[views]"
        n_halo_total += src.shape[0]
    assert n_halo_total == sum(sharded.halo_counts(nbr, world))
    rows = max(e - b + h for (b, e), h in zip(blocks, sharded.halo_counts(nbr, world)))
    assert sharded._max_local_views(nbr, world) == rows


def test_gather_table_of_a_single_rank_is_empty():
    order, nbr = _scene_ids(9, 1, True)
    assert order == list(range(9))
    assert tuple(sharded.halo_gather_table(nbr, 1, 0).shape) == (0, 2)


# ---- owned_views: the views load() has always given a rank --------------------------------------------------
def _load_plan_before(hot, img_meta, world, rank, pose_clustered):
    """the planning steps ShardedScenePipeline.load ran inline before they became owned_views"""
    geo_full = hot.geometry(img_meta, "cpu", prologue="host")
    v_all = geo_full.neighbor_ids_host.shape[0]
    begin, end = sharded.partition_views(v_all, world, rank)
    order = list(range(v_all))
    if pose_clustered:
        order = sharded.pose_order(img_meta["lidar2img"]["extrinsic"], geo_full.neighbor_ids_host, world)
        if order != list(range(v_all)):
            img_meta = sharded.permute_img_meta(img_meta, order)
            geo_full = hot.geometry(img_meta, "cpu", prologue="host")
    return order, torch.tensor(order[begin:end], dtype=torch.int64), geo_full.neighbor_ids_host, img_meta


@pytest.mark.parametrize("pose_clustered", [False, True], ids=["index", "pose"])
@pytest.mark.parametrize("v,world,per_view", [(80, 8, False), (40, 8, True), (20, 3, False), (9, 2, True)])
def test_owned_views_is_what_load_computed(v, world, per_view, pose_clustered):
    cfg = SceneConfig(n_views=v, per_view_intrinsics=per_view)
    scene = make_scene(cfg, seed=7, with_grads=False)
    hot = _hot(cfg)
    for rank in range(world):
        want_order, want_ids, want_nbr, want_meta = _load_plan_before(hot, scene["img_meta"], world, rank,
                                                                      pose_clustered)
        order, view_ids = sharded.owned_views(hot, scene["img_meta"], world, rank, pose_clustered=pose_clustered)
        assert order == want_order and view_ids.dtype == torch.int64 and torch.equal(view_ids, want_ids)
        order2, meta, nbr = sharded._view_plan(hot, scene["img_meta"], world, pose_clustered)
        assert order2 == want_order and torch.equal(nbr, want_nbr)
        assert meta["lidar2img"]["extrinsic"] == want_meta["lidar2img"]["extrinsic"]
    if pose_clustered and v == 80:
        assert order != list(range(v)), "the helix scan should be re-ordered into pose clusters"
    # every view is owned by exactly one rank
    owned = torch.cat([sharded.owned_views(hot, scene["img_meta"], world, r, pose_clustered)[1]
                       for r in range(world)])
    assert sorted(owned.tolist()) == list(range(v))


def test_owned_views_geometry_matches_the_sharded_ids():
    """the rows a rank's geometry slice gets in the sharded numbering are its owned views' rows of the scene"""
    cfg = SceneConfig(n_views=20)
    scene = make_scene(cfg, seed=3, with_grads=False)
    hot = _hot(cfg)
    kw = dict(stride=cfg.stride, near_far_range=cfg.near_far_range, num_depth=cfg.num_depth,
              n_voxels=cfg.n_voxels, voxel_size=cfg.voxel_size, device="cpu", prologue="host")
    geo = G.scene_geometry(scene["img_meta"], **kw)
    order, meta, _ = sharded._view_plan(hot, scene["img_meta"], 4, True)
    for rank in range(4):
        _, view_ids = sharded.owned_views(hot, scene["img_meta"], 4, rank)
        b, e = sharded.partition_views(20, 4, rank)
        geo_r = G.scene_geometry(meta, view_slice=slice(b, e), **kw)
        assert torch.equal(geo_r.projection, geo.projection[view_ids])
