"""Per-pixel depth hypotheses in the fused plane sweeps, the parts that run without a GPU: the
*_px entry points of the C ABI validate their arguments on the host and name themselves, and the
dispatcher ops' fake implementations take a [V,D,H,W] depth_values."""
import ctypes

import pytest
import torch

from mvsdet_b200 import _lib as L_
from mvsdet_b200 import library as L

V, C, H, W, D, K = 3, 16, 5, 7, 4, 2


def _lib():
    from mvsdet_b200 import build
    import os
    if not os.path.isfile(L_.LIB_PATH):
        build.build()
    return L_.load()


def test_px_entry_points_validate_before_any_launch():
    lib = _lib()
    before = lib.mvsd_launch_count()
    one = ctypes.c_void_p(16)                            # non-null dummy: rejected before any dereference
    st = lib.mvsd_plane_sweep_fwd_px(None, 0, None, None, None, None, 0, 0, 2, 8, 4, 4, 4, 0, 0, 2, None)
    assert st == L_.ERR_INVALID_ARG and lib.mvsd_last_error() == b"plane_sweep_fwd_px: null pointer"
    st = lib.mvsd_plane_sweep_fwd_px(one, 0, one, one, one, one, 0, 0, 2, 8, 4, 4, 4, 2, 1, 2, None)
    assert st == L_.ERR_INVALID_ARG and b"plane_sweep_fwd_px: reference views" in lib.mvsd_last_error()
    st = lib.mvsd_plane_sweep_bwd_px(None, 0, 0, None, 0, None, None, None, None, 2, 8, 4, 4, 4, 1, 0, 2, None)
    assert st == L_.ERR_INVALID_ARG and lib.mvsd_last_error() == b"plane_sweep_bwd_px: null pointer"
    st = lib.mvsd_plane_sweep_bwd_det_px(one, 0, 0, one, 0, one, one, one, one, 2, 6, 4, 4, 4, 1, 0, 2, None)
    assert st == L_.ERR_UNSUPPORTED and lib.mvsd_last_error().startswith(b"plane_sweep_bwd_det_px:")
    st = lib.mvsd_plane_sweep_groupcorr_fwd_px(one, 0, one, one, one, one, 2, 24, 4, 4, 4, 1, 2, 0, 2, None)
    assert st == L_.ERR_UNSUPPORTED and b"plane_sweep_groupcorr_fwd_px:" in lib.mvsd_last_error()
    st = lib.mvsd_plane_sweep_groupcorr_bwd_px(one, one, 0, one, one, one, one, 2, 24, 4, 4, 4, 1, 5, 0, 2, None)
    assert st == L_.ERR_INVALID_ARG and b"plane_sweep_groupcorr_bwd_px:" in lib.mvsd_last_error()
    assert lib.mvsd_launch_count() == before


@pytest.mark.parametrize("per_pixel", [False, True], ids=["per_view", "per_pixel"])
def test_launchers_pick_the_entry_point_from_the_depth_rank(per_pixel, monkeypatch):
    calls = []
    monkeypatch.setattr(L_, "call", lambda name, *args: calls.append((name, args)))
    monkeypatch.setattr(L_, "_stream", lambda: 0)
    feat = torch.empty((V, H, W, C)).permute(0, 3, 1, 2)
    nbr = torch.zeros((V, K), dtype=torch.int32)
    hom = torch.zeros((V, K, 12))
    dv = torch.zeros((V, D, H, W) if per_pixel else (V, D))
    vol = torch.empty((V, D, H, W, C)).permute(0, 4, 1, 2, 3)
    L_.plane_sweep_fwd(feat, nbr, hom, dv, vol)
    L_.plane_sweep_bwd(vol, feat, nbr, hom, dv, feat)
    L_.plane_sweep_bwd_det(vol, feat, nbr, hom, dv, feat)
    corr = torch.empty((V, K, D, H, W, 4)).permute(0, 1, 5, 2, 3, 4)
    L_.plane_sweep_groupcorr_fwd(feat, nbr, hom, dv, corr)
    L_.plane_sweep_groupcorr_bwd(corr, feat, nbr, hom, dv, feat)
    sfx = "_px" if per_pixel else ""
    assert [n for n, _ in calls] == [f"mvsd_plane_sweep_fwd{sfx}", f"mvsd_plane_sweep_bwd{sfx}",
                                     f"mvsd_plane_sweep_bwd_det{sfx}", f"mvsd_plane_sweep_groupcorr_fwd{sfx}",
                                     f"mvsd_plane_sweep_groupcorr_bwd{sfx}"]
    for name, args in calls:                             # D is depth_values.shape[1] in both forms
        assert len(args) == len(L_.SIGNATURES[name][0])
        assert any(tuple(args[i:i + 6]) == (V, C, D, H, W, K) for i in range(len(args))), name


def _meta(depth_shape):
    feat = torch.empty((V, H, W, C), device="meta").permute(0, 3, 1, 2).requires_grad_(True)
    nbr = torch.empty((V, K), dtype=torch.int32, device="meta")
    hom = torch.empty((V, K, 12), device="meta")
    return feat, nbr, hom, torch.empty(depth_shape, device="meta")


def test_fake_implementations_take_per_pixel_depth():
    feat, nbr, hom, dv = _meta((V, D, H, W))
    var = L.plane_sweep_variance(feat, nbr, hom, dv)
    assert tuple(var.shape) == (V, C, D, H, W) and var.permute(0, 2, 3, 4, 1).is_contiguous()
    g, = torch.autograd.grad(var, feat, torch.empty_like(var))
    assert tuple(g.shape) == (V, C, H, W)
    cost = L.plane_sweep_group_correlation(feat, nbr, hom, dv, 4)
    assert tuple(cost.shape) == (V, K, 4, D, H, W) and cost.permute(0, 1, 3, 4, 5, 2).is_contiguous()
