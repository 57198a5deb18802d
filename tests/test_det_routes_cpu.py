"""torch.use_deterministic_algorithms and the deterministic backwards, the parts that run without a GPU:
the two new entry points (mvsd_homo_warp_bwd_det, mvsd_backproject_bwd_det_mode) are exported and typed
and reject every rule of their fp32 twins with their own names before any launch; the one policy
(ops._deterministic) sends every scatter backward to its fixed-point entry point under the flag, with or
without a gradient sink; the captured training-step forms alert as ATen does."""
import ctypes
import re
import warnings

import pytest
import torch

import test_abi as A
from mvsdet_b200 import _lib as L_
from mvsdet_b200 import ops
from mvsdet_b200._lib import BP_MEAN, BP_PER_VIEW, BP_SUM


@pytest.fixture
def det_flag():
    """turns torch.use_deterministic_algorithms on inside the test; restores the flag and warn_only"""
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()

    def set_flag(on, warn_only=False):
        torch.use_deterministic_algorithms(on, warn_only=warn_only)
    yield set_flag
    torch.use_deterministic_algorithms(was, warn_only=warn)


def test_entry_points_are_exported_and_typed():
    lib = A._build_if_needed().load()
    for name, twin in (("mvsd_homo_warp_bwd_det", "mvsd_homo_warp_bwd"),
                       ("mvsd_backproject_bwd_det_mode", "mvsd_backproject_bwd")):
        assert L_.SIGNATURES[name] == L_.SIGNATURES[twin]
        fn = getattr(lib, name)
        assert fn.argtypes == L_.SIGNATURES[name][0] and fn.restype is ctypes.c_int


def _call(lib, entry, params, args):
    dummy = ctypes.c_void_p(16)
    before = lib.mvsd_launch_count()
    st = getattr(lib, entry)(*[(dummy if args[p] else None) if p in _PTRS else args[p] for p in params])
    assert lib.mvsd_launch_count() == before
    return st, lib.mvsd_last_error().decode()


# ---- mvsd_homo_warp_bwd_det: the rules of mvsd_homo_warp_bwd (test_abi's table), in its own name ---------
def _warp_cases():
    for rule, overrides, expect in A._SWEEP_RULES:
        if "warp_bwd" in expect:
            status, message = expect["warp_bwd"]
            # the fp32 form names its grid after the kernel family and its dtype error after itself
            message = re.sub(r"^(\{who\}|homo_warp_bwd|plane_sweep_bwd):", "homo_warp_bwd_det:", message)
            yield pytest.param(overrides, status, message, id=rule)


_PTRS = A._POINTERS + ("count", "points", "projection", "prob")


@pytest.mark.parametrize("overrides,status,message", list(_warp_cases()))
def test_homo_warp_bwd_det_rejects_before_any_launch(overrides, status, message):
    lib = A._build_if_needed().load()
    assert _call(lib, "mvsd_homo_warp_bwd_det", A._WARP_BWD, {**A._VALID, **overrides}) == (status, message)


# ---- mvsd_backproject_bwd_det_mode: the rules of mvsd_backproject_bwd, in its own name -------------------
_BP_BWD = ("g_out", "layout", "mode", "count", "feat", "feat_dtype", "feat_h", "feat_w", "points", "projection",
           "depth", "prob", "sv", "sy", "sx", "st", "vs_z", "g_feat", "g_pn", "V", "C", "h", "w", "T", "N",
           "stream")
_BP_VALID = dict(layout=0, mode=BP_SUM, feat_dtype=0, feat_h=4, feat_w=4, sv=48, sy=12, sx=3, st=1, vs_z=0.1,
                 V=2, C=8, h=4, w=4, T=3, N=10, stream=None,
                 **{p: True for p in ("g_out", "count", "feat", "points", "projection", "depth", "prob",
                                      "g_feat", "g_pn")})
_BP_NULLABLE = ("count", "g_pn")
# (rule, overrides, message of both entry points, or {entry: message}); {who} is the entry point's name
_BP_RULES = [
    *[(f"{d}=0", {d: 0}, (A._ARG, "{who}: non-positive dimension")) for d in ("V", "C", "h", "w", "T", "N")],
    ("crop", {"h": 5}, (A._ARG, "{who}: crop [5,4] exceeds the map [4,4]")),
    ("C%4", {"C": 6}, (A._UNS, "{who}: C=6 must be a multiple of 4 and <= 512")),
    ("C>512", {"C": 516}, (A._UNS, "{who}: C=516 must be a multiple of 4 and <= 512")),
    ("T>8", {"T": 9}, (A._UNS, "{who}: T=9 > 8")),
    ("mode", {"mode": 3}, (A._ARG, "{who}: bad mode 3")),
    ("layout", {"layout": 2}, (A._ARG, "{who}: bad layout 2")),
    ("per-view-channels-first", {"mode": BP_PER_VIEW, "layout": 1},
     (A._UNS, "{who}: per-view volumes are channels-last only")),
    *[(f"null-{p}", {p: None}, (A._ARG, "{who}: null pointer"))
      for p in ("g_out", "feat", "points", "projection", "depth", "prob", "g_feat")],
    ("dims-before-null", {"V": 0, "g_out": None}, (A._ARG, "{who}: non-positive dimension")),
    ("null-before-dtype", {"feat": None, "feat_dtype": 2}, (A._ARG, "{who}: null pointer")),
    ("dtype", {"feat_dtype": 2}, {"mvsd_backproject_bwd": (A._ARG, "backproject: bad dtype"),
                                  "mvsd_backproject_bwd_det_mode": (A._ARG, "{who}: bad dtype")}),
    ("mean", {"mode": BP_MEAN}, {"mvsd_backproject_bwd_det_mode": (
        A._UNS, "{who}: the MEAN mode's deterministic backward is mvsd_backproject_bwd_det")}),
    ("mean-no-count", {"mode": BP_MEAN, "count": None}, {
        "mvsd_backproject_bwd": (A._ARG, "{who}: count is required in MEAN mode"),
        "mvsd_backproject_bwd_det_mode": (A._UNS, "{who}: the MEAN mode's deterministic backward is "
                                                  "mvsd_backproject_bwd_det")}),
]


def _bp_cases():
    for entry in ("mvsd_backproject_bwd", "mvsd_backproject_bwd_det_mode"):
        who = entry[len("mvsd_"):]
        for rule, overrides, expect in _BP_RULES:
            if isinstance(expect, dict):
                if entry not in expect:
                    continue
                expect = expect[entry]
            yield pytest.param(entry, overrides, expect[0], expect[1].format(who=who), id=f"{who}-{rule}")


@pytest.mark.parametrize("entry,overrides,status,message", list(_bp_cases()))
def test_backproject_bwd_det_mode_rejects_like_its_twin(entry, overrides, status, message):
    """the same rules in the same order as mvsd_backproject_bwd (run on both), before any launch"""
    lib = A._build_if_needed().load()
    assert _call(lib, entry, _BP_BWD, {**_BP_VALID, **overrides}) == (status, message)


# ---- routing: which entry point each backward calls, flag off and on --------------------------------------
@pytest.fixture
def calls(monkeypatch):
    """records the entry points the launchers call (nothing is launched); fixed_to_float is recorded too"""
    rec = []
    monkeypatch.setattr(L_, "call", lambda name, *args: rec.append(name))
    monkeypatch.setattr(L_, "_stream", lambda: 0)
    monkeypatch.setattr(ops, "fixed_to_float",
                        lambda q: (rec.append("mvsd_fixed_to_float"), torch.zeros(q.shape))[1])
    return rec


V, C, H, W, D, K, G, T, N = 3, 16, 5, 7, 4, 2, 4, 2, 11


def _feat(dtype=torch.float32):
    return torch.zeros((V, H, W, C), dtype=dtype).permute(0, 3, 1, 2)


def _sweep_inputs():
    nbr = torch.zeros((V, K), dtype=torch.int32)
    return _feat(), nbr, torch.zeros((V, K, 12)), torch.zeros((V, D))


def _bp_inputs(strided=False):
    big = torch.zeros((V, T, H + 2, W)) if strided else torch.zeros((V, T, H, W))
    hyp = big[:, :, 1:1 + H] if strided else big
    return _feat(), torch.zeros((3, N)), torch.zeros((V, 3, 4)), hyp, hyp


ROUTES = {
    "variance": ("mvsd_plane_sweep_bwd", "mvsd_plane_sweep_bwd_det"),
    "correlation": ("mvsd_plane_sweep_groupcorr_bwd", "mvsd_plane_sweep_groupcorr_bwd_det"),
    "bp-mean": ("mvsd_backproject_bwd", "mvsd_backproject_bwd_det"),
    "bp-sum": ("mvsd_backproject_bwd", "mvsd_backproject_bwd_det_mode"),
    "bp-sum-strided": ("mvsd_backproject_bwd", "mvsd_backproject_bwd_det_mode"),
    "bp-per-view": ("mvsd_backproject_bwd", "mvsd_backproject_bwd_det_mode"),
    "homo-warp": ("mvsd_homo_warp_bwd", "mvsd_homo_warp_bwd_det"),
}


def _run_route(route, acc=None):
    """one backward of ``route`` on CPU tensors (the launchers are recorded) -> the feature gradient"""
    if route == "variance":
        feat, nbr, hom, dv = _sweep_inputs()
        g = torch.zeros((V, D, H, W, C)).permute(0, 4, 1, 2, 3)
        return ops._sweep_bwd_raw(g, feat, nbr, hom, dv, 0, acc)
    if route == "correlation":
        feat, nbr, hom, dv = _sweep_inputs()
        g = torch.zeros((V, K, D, H, W, G)).permute(0, 1, 5, 2, 3, 4)
        return ops._corr_bwd_raw(g, feat, nbr, hom, dv, 0, acc)
    if route.startswith("bp-") and route != "bp-per-view":
        feat, pts, proj, depth, dens = _bp_inputs(strided=route.endswith("strided"))
        mode = BP_MEAN if route == "bp-mean" else BP_SUM
        g_feat, g_prob = ops._bp_bwd_raw(torch.zeros((C, N)), feat, pts, proj, depth, dens,
                                         torch.zeros(N, dtype=torch.int32), 0.1, H, W, mode, True, acc)
        assert g_prob.stride() == dens.stride()
        return g_feat
    if route == "bp-per-view":
        feat = _feat().requires_grad_(True)
        hyp = torch.zeros((V, H * W, 1, T))
        vol, _ = ops._BackprojectPerView.apply(feat, torch.zeros((3, N)), torch.zeros((V, 3, 4)), hyp, hyp,
                                               0.1, H, W)
        g, = torch.autograd.grad(vol, feat, torch.zeros(vol.shape))
        return g
    src = _feat().requires_grad_(True)                                    # homo-warp
    out = ops._HomoWarp.apply(src, torch.zeros((V, 12)), torch.zeros((V, D)), torch.float32)
    g, = torch.autograd.grad(out, src, torch.zeros(out.shape))
    return g


@pytest.mark.parametrize("flag", [False, True], ids=["flag-off", "flag-on"])
@pytest.mark.parametrize("route", list(ROUTES))
def test_policy_routes_every_backward(route, flag, calls, det_flag):
    """without a sink: the fp32-RED entry point, or under the flag the fixed-point one, converted once"""
    det_flag(flag)
    g = _run_route(route)
    assert ROUTES[route][flag] in calls and ROUTES[route][not flag] not in calls
    assert ("mvsd_fixed_to_float" in calls) == flag
    assert g.dtype == torch.float32 and tuple(g.shape) == (V, C, H, W)


@pytest.mark.parametrize("flag", [False, True], ids=["flag-off", "flag-on"])
@pytest.mark.parametrize("route", ["variance", "correlation", "bp-mean", "bp-sum"])
def test_sink_dtype_follows_the_policy_at_first_use(route, flag, calls, det_flag):
    """a sink made with deterministic=False becomes int64 under the flag; its consumers follow its dtype"""
    sink = ops.FeatureGradSink((V, C, H, W), "cpu", deterministic=False)
    det_flag(flag)
    acc = sink.get()
    assert acc.dtype == (torch.int64 if flag else torch.float32)
    det_flag(not flag)                         # the dtype is fixed at the first get()
    assert sink.get() is acc
    assert _run_route(route, acc) is None
    assert ROUTES[route][flag] in calls and ROUTES[route][not flag] not in calls
    calls.clear()
    assert sink.take().dtype == torch.float32
    assert calls == (["mvsd_fixed_to_float"] if flag else [])


def test_explicit_deterministic_sink_is_fixed_point_without_the_flag(det_flag):
    det_flag(False)
    assert ops._deterministic(True) and not ops._deterministic()
    assert ops.FeatureGradSink((V, C, H, W), "cpu", deterministic=True).get().dtype == torch.int64
    det_flag(True)
    assert ops._deterministic() and ops._deterministic(False)


# ---- the alert of the captured training-step forms ---------------------------------------------------------
def test_alert_raises_warns_or_stays_silent(det_flag):
    det_flag(False)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        ops._alert_not_deterministic("X.step")
    det_flag(True)
    with pytest.raises(RuntimeError, match=r"^X\.step does not have a deterministic implementation, but you set "
                                           r"'torch\.use_deterministic_algorithms\(True\)'"):
        ops._alert_not_deterministic("X.step")
    det_flag(True, warn_only=True)
    with pytest.warns(UserWarning, match=r"^X\.step does not have a deterministic implementation"):
        ops._alert_not_deterministic("X.step")


def test_training_step_forms_alert_before_enqueueing(calls, det_flag):
    from mvsdet_b200.pipeline import ScenePipeline
    from mvsdet_b200.sharded import ShardedScenePipeline
    pipe = ScenePipeline.__new__(ScenePipeline)
    pipe.geo = object()                                  # set_geometry() done; nothing else is touched
    sharded = ShardedScenePipeline.__new__(ShardedScenePipeline)
    det_flag(True)
    with pytest.raises(RuntimeError, match="^ScenePipeline.step does not have a deterministic"):
        pipe.step()
    with pytest.raises(RuntimeError, match="^ShardedScenePipeline.backward does not have a deterministic"):
        sharded.backward(None, None)
    assert calls == []


def test_hot_path_dispatcher_rejection_names_the_flag():
    from mvsdet_b200.hotpath import MVSDetHotPath
    with pytest.raises(ValueError, match=r"dispatcher_ops=True.*torch\.use_deterministic_algorithms\(True\)"):
        MVSDetHotPath([4, 4, 4], [0.1] * 3, [0.2, 5.0], deterministic=True, dispatcher_ops=True)
