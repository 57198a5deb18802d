"""The deterministic training-step forms, the parts that run without a GPU: mvsd_halo_reduce_p2p_fixed is
exported, typed like its fp32 twin and rejects every rule of it, in its own name, before any launch;
``ScenePipeline(deterministic=True)`` and a ``ShardedScenePipeline`` over a deterministic hot path enqueue
only the fixed-point (``*_det``) scatter entry points, the fixed-point halo pull and
``mvsd_fixed_to_float`` (the launchers are recorded, nothing is launched), and run silently under
``torch.use_deterministic_algorithms(True)``, while their default forms keep alerting."""
import contextlib
import ctypes
import types

import pytest
import torch

import test_abi as A
from mvsdet_b200 import _lib as L_
from mvsdet_b200.pipeline import ScenePipeline
from mvsdet_b200.scene import tiny_config
from mvsdet_b200.sharded import ShardedScenePipeline
from test_det_routes_cpu import det_flag  # noqa: F401  (fixture)

HALO = ("mvsd_halo_reduce_p2p", "mvsd_halo_reduce_p2p_fixed")


def test_fixed_halo_pull_is_exported_and_typed_like_its_twin():
    lib = A._build_if_needed().load()
    assert L_.SIGNATURES["mvsd_halo_reduce_p2p_fixed"] == L_.SIGNATURES["mvsd_halo_reduce_p2p"]
    fn = lib.mvsd_halo_reduce_p2p_fixed
    assert fn.argtypes == L_.SIGNATURES["mvsd_halo_reduce_p2p_fixed"][0] and fn.restype is ctypes.c_int


# ---- argument checks: the rules of mvsd_halo_reduce_p2p, in the same order, each entry point in its name ----
_HALO_ARGS = ("g_ptrs", "offs", "src", "world", "rank", "n_own", "view_elems", "stream")
_HALO_VALID = dict(g_ptrs=True, offs=True, src=True, world=2, rank=1, n_own=3, view_elems=64, stream=None)
_HALO_RULES = [
    *[(f"null-{p}", {p: False}, "{who}: null pointer") for p in ("g_ptrs", "offs", "src")],
    ("world=0", {"world": 0, "rank": 0}, "{who}: bad world/rank (0/0)"),
    ("world>16", {"world": 17}, "{who}: bad world/rank (1/17)"),
    ("rank<0", {"rank": -1}, "{who}: bad world/rank (-1/2)"),
    ("rank=world", {"rank": 2}, "{who}: bad world/rank (2/2)"),
    ("n_own=0", {"n_own": 0}, "{who}: bad view count / size"),
    ("n_own>65535", {"n_own": 65536}, "{who}: bad view count / size"),
    ("view_elems=0", {"view_elems": 0}, "{who}: bad view count / size"),
    ("view_elems<0", {"view_elems": -4}, "{who}: bad view count / size"),
    *[(f"view_elems%4={r}", {"view_elems": 64 + r}, "{who}: bad view count / size") for r in (1, 2, 3)],
    ("null-before-world", {"g_ptrs": False, "world": 0}, "{who}: null pointer"),
    ("world-before-size", {"world": 0, "view_elems": 3}, "{who}: bad world/rank (1/0)"),
]


@pytest.mark.parametrize("entry", HALO)
@pytest.mark.parametrize("overrides,message", [pytest.param(o, m, id=r) for r, o, m in _HALO_RULES])
def test_halo_pull_rejects_before_any_launch(entry, overrides, message):
    lib = A._build_if_needed().load()
    args = {**_HALO_VALID, **overrides}
    dummy = ctypes.c_void_p(16)
    before = lib.mvsd_launch_count()
    st = getattr(lib, entry)(*[(dummy if args[p] else None) if p in ("g_ptrs", "offs", "src") else args[p]
                               for p in _HALO_ARGS])
    assert lib.mvsd_launch_count() == before
    assert (st, lib.mvsd_last_error().decode()) == (L_.ERR_INVALID_ARG, message.format(who=entry[len("mvsd_"):]))


def test_halo_pull_launcher_raises_with_its_name(monkeypatch):
    """the Python launcher reports the C-side rejection as ValueError naming the entry point"""
    A._build_if_needed()
    monkeypatch.setattr(L_, "_stream", lambda: 0)
    offs = torch.zeros(1, dtype=torch.int32)                       # n_own = 0
    with pytest.raises(ValueError, match=r"^mvsd_halo_reduce_p2p_fixed: halo_reduce_p2p_fixed: bad view count"):
        L_.halo_reduce_p2p_fixed(16, offs, torch.zeros((1, 2), dtype=torch.int32), world=2, rank=0, view_elems=64)


# ---- routing: which entry points the training-step forms enqueue -------------------------------------------
class _Stream:
    """stands in for torch.cuda.Stream: the schedule's stream edges are host calls with no effect here"""

    def __init__(self, *args, **kwargs):
        pass

    def wait_stream(self, other):
        pass


@pytest.fixture
def calls(monkeypatch):
    """records the entry points the launchers call (nothing is launched); the CUDA streams are stand-ins"""
    rec = []
    monkeypatch.setattr(L_, "call", lambda name, *args: rec.append(name))
    monkeypatch.setattr(L_, "_stream", lambda: 0)
    monkeypatch.setattr(torch.cuda, "Stream", _Stream)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: _Stream())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    return rec


CFG = tiny_config(n_views=4, channels=16, num_depth=4, topk=2, n_voxels=(4, 4, 4))


def _geometry(v, k=2):
    hf, wf = CFG.feat_hw
    h, w = CFG.crop_hw
    n = CFG.n_voxels[0] * CFG.n_voxels[1] * CFG.n_voxels[2]
    return types.SimpleNamespace(neighbor_ids=torch.zeros((v, k), dtype=torch.int32), hom=torch.zeros((v, k, 12)),
                                 depth_values=torch.zeros((v, CFG.num_depth)), points=torch.zeros((3, n)),
                                 projection=torch.zeros((v, 3, 4)), height=h, width=w)


# the fp32-RED scatter entry points and their fixed-point forms
FP32 = {"mvsd_backproject_bwd", "mvsd_plane_sweep_bwd", "mvsd_halo_reduce_p2p"}
FIXED = {"mvsd_backproject_bwd_det", "mvsd_plane_sweep_bwd_det", "mvsd_halo_reduce_p2p_fixed"}


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("overlap", [True, False], ids=["overlapped", "back-to-back"])
def test_scene_pipeline_deterministic_step_enqueues_fixed_point_only(feature_dtype, overlap, calls, det_flag):  # noqa: F811
    det_flag(True)                                   # the deterministic form runs silently under the flag
    pipe = ScenePipeline(CFG, "cpu", feature_dtype=feature_dtype, deterministic=True)
    assert pipe.g_feat_q.dtype == torch.int64 and pipe.g_pn_q.dtype == torch.int64
    assert pipe.g_feat_q.shape == pipe.g_feat_cl.shape and pipe.g_pn_q.shape == pipe.g_pn.shape
    pipe.overlap_small = overlap
    pipe.set_geometry(_geometry(CFG.n_views))
    pipe.step()
    assert not FP32 & set(calls)
    scatter = [c for c in calls if c in FIXED]
    assert scatter == ["mvsd_backproject_bwd_det", "mvsd_plane_sweep_bwd_det"] or \
        scatter == ["mvsd_plane_sweep_bwd_det", "mvsd_backproject_bwd_det"]
    # g_pn is converted before the prob-norm backward reads it, g_feat after both scatters, before the unpack
    i_bp, i_pn = calls.index("mvsd_backproject_bwd_det"), calls.index("mvsd_prob_norm_bwd")
    assert calls[i_bp + 1] == "mvsd_fixed_to_float" and i_pn == i_bp + 2
    assert calls[-2:] == ["mvsd_fixed_to_float", "mvsd_unpack_nhwc_to_nchw"]
    assert calls.index("mvsd_plane_sweep_bwd_det") < len(calls) - 2
    assert calls.count("mvsd_fixed_to_float") == 2
    bytes_ = pipe.algorithmic_bytes()
    assert {"backproject_bwd_det", "plane_sweep_bwd_det", "fixed_to_float_pn", "fixed_to_float_feat"} <= set(bytes_)
    assert not {"backproject_bwd", "plane_sweep_bwd"} & set(bytes_)


def test_scene_pipeline_default_step_is_unchanged_and_still_alerts(calls, det_flag):  # noqa: F811
    assert ScenePipeline.deterministic is False and ShardedScenePipeline.deterministic is False
    pipe = ScenePipeline(CFG, "cpu")
    assert not pipe.deterministic and not hasattr(pipe, "g_feat_q")
    pipe.set_geometry(_geometry(CFG.n_views))
    det_flag(False)
    pipe.step()
    assert {"mvsd_backproject_bwd", "mvsd_plane_sweep_bwd"} <= set(calls)
    assert not FIXED & set(calls) and "mvsd_fixed_to_float" not in calls
    calls.clear()
    det_flag(True)
    with pytest.raises(RuntimeError, match="^ScenePipeline.step does not have a deterministic"):
        pipe.step()
    assert calls == []
    assert set(pipe.algorithmic_bytes()) == {"pack", "plane_sweep_fwd", "depth_topk_fwd", "backproject_fwd",
                                             "backproject_bwd", "prob_norm_bwd", "depth_topk_bwd",
                                             "plane_sweep_bwd", "unpack"}


def _sharded(deterministic, world=2, rank=0, vb=2, vl=3, n_pull=1):
    """a ShardedScenePipeline after load() and its first backward's allocation, with CPU tensors and
    stand-ins for the process group's peer-mapped buffer (built without __init__: no process group)"""
    hf, wf = CFG.feat_hw
    c, d, t = CFG.channels, CFG.num_depth, CFG.topk
    n = CFG.n_voxels[0] * CFG.n_voxels[1] * CFG.n_voxels[2]
    ve = hf * wf * c
    p = ShardedScenePipeline.__new__(ShardedScenePipeline)
    p.hot = types.SimpleNamespace(deterministic=deterministic)
    p.deterministic = deterministic
    p.cfg, p.device, p.c, p.n, p.world, p.rank = CFG, torch.device("cpu"), c, n, world, rank
    p.vl, p.vb = vl, vb
    p.lg = types.SimpleNamespace(geo=_geometry(vb), neighbor_ids_local=torch.zeros((vb, 2), dtype=torch.int32))
    p.feat_cl = torch.zeros((vl, hf, wf, c)).permute(0, 3, 1, 2)
    p.cost_out = torch.zeros((vb, 2, d, hf, wf))
    p.est_depth = p.est_dens = torch.zeros((vb, t, hf, wf))
    p.est_idx = torch.zeros((vb, t, hf, wf), dtype=torch.int64)
    p._red = [types.SimpleNamespace(count_local=torch.zeros(n, dtype=torch.int32))] * 2
    p._last_slot, p.s_aux = 0, _Stream()
    p._g_feat = torch.zeros(vl * ve, dtype=torch.int64 if deterministic else torch.float32)
    p._h_g = types.SimpleNamespace(barrier=lambda channel: None, buffer_ptrs_dev=16)
    p._pull_offs = torch.tensor([0, n_pull] + [n_pull] * (vb - 1), dtype=torch.int32)
    p._pull_src, p._n_pull = torch.zeros((n_pull, 2), dtype=torch.int32), n_pull
    p.g_pn = torch.zeros((vb, t, hf, wf))
    p.g_est_dens = torch.zeros((vb, t, hf, wf))
    p.g_cost_out = torch.zeros((vb, 2, d, hf, wf))
    p.g_feature = torch.zeros((vb, c, hf, wf))
    if deterministic:
        p.g_pn_q = torch.zeros((vb, t, hf, wf), dtype=torch.int64)
        p.g_feat_own = torch.zeros(vb * ve)
    g_vol = torch.zeros((c,) + tuple(CFG.n_voxels))
    g_var = torch.zeros((vb, d, hf, wf, c)).permute(0, 4, 1, 2, 3)
    return p, g_vol, g_var


def test_sharded_backward_follows_a_deterministic_hot_path(calls, det_flag):  # noqa: F811
    det_flag(True)
    pipe, g_vol, g_var = _sharded(True)
    pipe.backward(g_vol, g_var, use_graph=False)
    assert not FP32 & set(calls)
    assert FIXED <= set(calls)
    # the pull runs after both scatters; the owned rows are converted after it, then unpacked
    i_pull = calls.index("mvsd_halo_reduce_p2p_fixed")
    assert max(calls.index("mvsd_backproject_bwd_det"), calls.index("mvsd_plane_sweep_bwd_det")) < i_pull
    assert calls[i_pull + 1:] == ["mvsd_fixed_to_float", "mvsd_unpack_nhwc_to_nchw"]
    assert calls.count("mvsd_fixed_to_float") == 2                   # g_pn_q, then the owned rows


def test_sharded_backward_default_is_unchanged_and_still_alerts(calls, det_flag):  # noqa: F811
    pipe, g_vol, g_var = _sharded(False)
    det_flag(False)
    pipe.backward(g_vol, g_var, use_graph=False)
    assert {"mvsd_backproject_bwd", "mvsd_plane_sweep_bwd", "mvsd_halo_reduce_p2p"} <= set(calls)
    assert not FIXED & set(calls) and "mvsd_fixed_to_float" not in calls
    calls.clear()
    det_flag(True)
    with pytest.raises(RuntimeError, match="^ShardedScenePipeline.backward does not have a deterministic"):
        pipe.backward(g_vol, g_var, use_graph=False)
    assert calls == []

