"""The deterministic group-correlation backward, the parts that run without a GPU: both entry points
are exported and typed, give every rejection rule of mvsd_plane_sweep_groupcorr_bwd with their own
names before any launch, and the launchers pick the entry point from the depth rank."""
import ctypes

import pytest
import torch

import test_abi as A
from mvsdet_b200 import _lib as L_
from mvsdet_b200 import ops

DET = ("mvsd_plane_sweep_groupcorr_bwd_det", "mvsd_plane_sweep_groupcorr_bwd_det_px")
V, C, H, W, D, K, G = 3, 16, 5, 7, 4, 2, 4


def test_entry_points_are_exported_and_typed():
    lib = A._build_if_needed().load()
    for name in DET:
        assert L_.SIGNATURES[name] == L_.SIGNATURES["mvsd_plane_sweep_groupcorr_bwd"]
        fn = getattr(lib, name)
        assert fn.argtypes == L_.SIGNATURES[name][0] and fn.restype is ctypes.c_int


# The deterministic form always takes the pixel kernel, so its grid errors name that kernel in both
# the fp32 and the bf16 case (the fp32-RED form reports the family, or for bf16 and k = 2 the run kernel).
_GRID_MESSAGE = "plane_sweep_groupcorr_bwd_det: grid too large"


def _det_cases():
    for entry in DET:
        who = entry[len("mvsd_"):]
        for rule, overrides, expect in A._SWEEP_RULES:
            if "corr_bwd" not in expect:
                continue
            status, message = expect["corr_bwd"]
            if rule.startswith("grid"):
                message = _GRID_MESSAGE
            yield pytest.param(entry, overrides, status, message.format(who=who), id=f"{who}-{rule}")


@pytest.mark.parametrize("entry,overrides,status,message", list(_det_cases()))
def test_det_entry_points_reject_before_any_launch(entry, overrides, status, message):
    lib = A._build_if_needed().load()
    args = {**A._VALID, **overrides}
    dummy = ctypes.c_void_p(16)
    before = lib.mvsd_launch_count()
    st = getattr(lib, entry)(*[(dummy if args[p] else None) if p in A._POINTERS else args[p] for p in A._CORR_BWD])
    assert lib.mvsd_launch_count() == before
    assert (st, lib.mvsd_last_error().decode()) == (status, message)


def _capture(monkeypatch):
    calls = []
    monkeypatch.setattr(L_, "call", lambda name, *args: calls.append((name, args)))
    monkeypatch.setattr(L_, "_stream", lambda: 0)
    return calls


def _inputs(per_pixel):
    feat = torch.empty((V, H, W, C)).permute(0, 3, 1, 2)
    nbr = torch.zeros((V, K), dtype=torch.int32)
    hom = torch.zeros((V, K, 12))
    dv = torch.zeros((V, D, H, W) if per_pixel else (V, D))
    g = torch.zeros((V, K, D, H, W, G)).permute(0, 1, 5, 2, 3, 4)
    return g, feat, nbr, hom, dv


@pytest.mark.parametrize("per_pixel", [False, True], ids=["per_view", "per_pixel"])
def test_launcher_picks_the_entry_point_from_the_depth_rank(per_pixel, monkeypatch):
    calls = _capture(monkeypatch)
    g, feat, nbr, hom, dv = _inputs(per_pixel)
    L_.plane_sweep_groupcorr_bwd_det(g, feat, nbr, hom, dv, torch.zeros(feat.shape, dtype=torch.int64),
                                     ref_begin=0)
    name, args = calls[0]
    assert name == DET[per_pixel]
    assert len(args) == len(L_.SIGNATURES[name][0])
    assert any(tuple(args[i:i + 7]) == (V, C, D, H, W, K, G) for i in range(len(args)))


@pytest.mark.parametrize("per_pixel", [False, True], ids=["per_view", "per_pixel"])
def test_corr_bwd_raw_routes_an_int64_accumulator_to_the_det_entry_point(per_pixel, monkeypatch):
    """an int64 sink goes to the deterministic entry point and nothing is returned; an fp32 sink and no
    sink keep the fp32-RED entry point"""
    calls = _capture(monkeypatch)
    g, feat, nbr, hom, dv = _inputs(per_pixel)
    sfx = "_px" if per_pixel else ""
    assert ops._corr_bwd_raw(g, feat, nbr, hom, dv, 0, torch.zeros(feat.shape, dtype=torch.int64)) is None
    assert ops._corr_bwd_raw(g, feat, nbr, hom, dv, 0, torch.zeros(feat.shape)) is None
    assert [n for n, _ in calls] == [f"mvsd_plane_sweep_groupcorr_bwd_det{sfx}", f"mvsd_plane_sweep_groupcorr_bwd{sfx}"]


def test_hot_path_accepts_deterministic_group_correlation():
    from mvsdet_b200.hotpath import MVSDetHotPath
    mod = MVSDetHotPath([4, 4, 4], [0.1] * 3, [0.2, 5.0], cost_volume="group_correlation", deterministic=True)
    assert mod.deterministic and mod.cost_volume == "group_correlation"
    with pytest.raises(ValueError, match="dispatcher_ops=True"):
        MVSDetHotPath([4, 4, 4], [0.1] * 3, [0.2, 5.0], cost_volume="group_correlation", deterministic=True,
                      dispatcher_ops=True)
