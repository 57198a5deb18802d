"""The depth top-k over per-pixel depth hypotheses, the parts that run without a GPU: the *_px entry
points of the C ABI validate their arguments on the host and name themselves, the launchers pick
the entry point from ``depth_values``, and the dispatcher ops' fake implementations give the
shapes of the outputs and of the gradients."""
import ctypes
import os

import pytest
import torch

from mvsdet_b200 import _lib as L_
from mvsdet_b200 import library as L

V, D, H, W, T = 2, 12, 5, 7, 3


def _lib():
    from mvsdet_b200 import build
    if not os.path.isfile(L_.LIB_PATH):
        build.build()
    return L_.load()


ONE = ctypes.c_void_p(16)              # non-null dummy: rejected before any dereference


def _fwd_args(**kw):
    a = dict(cost_out=ONE, s_v=0, s_c=0, s_d=0, s_p=0, depth_values=ONE, interval_map=None, interval=0.5,
             prob_volume=None, off_pred=None, est_depth=ONE, est_dens=ONE, est_idx=ONE, depth_coding=None,
             ray_intrinsics=None, ray_per_view=0, opacity=None, depth_scale=None, est_ray_depth=None,
             ray_depth_coding=None, raw=0, V=V, D=D, H=H, W=W, T=T, stream=None)
    a.update(kw)
    return list(a.values())


def _bwd_args(**kw):
    a = dict(cost_out=ONE, s_v=0, s_c=0, s_d=0, s_p=0, est_idx=ONE, depth_values=ONE, interval_map=None,
             interval=0.5, g_prob_volume=None, g_off_pred=None, g_est_depth=None, g_est_dens=None,
             g_depth_coding=None, ray_intrinsics=None, ray_per_view=0, g_est_ray_depth=None,
             g_ray_depth_coding=None, g_cost_out=ONE, g_depth_values=None, g_interval_map=None, raw=0,
             V=V, D=D, H=H, W=W, T=T, stream=None)
    a.update(kw)
    return list(a.values())


NULL = b"null pointer"
CASES = [
    ("fwd", dict(cost_out=None), L_.ERR_INVALID_ARG, NULL),
    ("fwd", dict(depth_values=None), L_.ERR_INVALID_ARG, NULL),
    ("fwd", dict(est_depth=None), L_.ERR_INVALID_ARG, NULL),
    ("fwd", dict(est_dens=None), L_.ERR_INVALID_ARG, NULL),
    ("fwd", dict(D=65), L_.ERR_UNSUPPORTED, b"D=65 > 64"),
    ("fwd", dict(D=2, T=3), L_.ERR_UNSUPPORTED, b"T=3 must be <= min(D, 8)"),
    ("fwd", dict(T=0), L_.ERR_INVALID_ARG, b"non-positive dimension"),
    ("fwd", dict(depth_scale=ONE), L_.ERR_INVALID_ARG, b"ray outputs need ray_intrinsics"),
    ("bwd", dict(cost_out=None), L_.ERR_INVALID_ARG, NULL),
    ("bwd", dict(est_idx=None), L_.ERR_INVALID_ARG, NULL),
    ("bwd", dict(depth_values=None), L_.ERR_INVALID_ARG, NULL),
    ("bwd", dict(g_cost_out=None), L_.ERR_INVALID_ARG, NULL),
    ("bwd", dict(D=65), L_.ERR_UNSUPPORTED, b"D=65 > 64"),
    ("bwd", dict(D=2, T=3), L_.ERR_UNSUPPORTED, b"T=3 must be <= min(D, 8)"),
    ("bwd", dict(g_interval_map=ONE), L_.ERR_INVALID_ARG, b"g_interval_map needs interval_map"),
    ("bwd", dict(g_est_ray_depth=ONE), L_.ERR_INVALID_ARG, b"ray gradients need ray_intrinsics"),
]


@pytest.mark.parametrize("which,override,status,message", CASES,
                         ids=[f"{w}-{'-'.join(o)}-{m.decode().split()[0]}" for w, o, _, m in CASES])
def test_px_entry_points_validate_before_any_launch(which, override, status, message):
    lib = _lib()
    before = lib.mvsd_launch_count()
    if which == "fwd":
        st = lib.mvsd_depth_topk_fwd_px(*_fwd_args(**override))
    else:
        st = lib.mvsd_depth_topk_bwd_px(*_bwd_args(**override))
    assert st == status
    assert lib.mvsd_last_error() == f"depth_topk_{which}_px: ".encode() + message
    assert lib.mvsd_launch_count() == before


@pytest.mark.parametrize("per_pixel,interval_map", [(False, False), (True, False), (True, True)],
                         ids=["per_view", "per_pixel", "per_pixel_map"])
def test_launchers_pick_the_entry_point(per_pixel, interval_map, monkeypatch):
    calls = []
    monkeypatch.setattr(L_, "call", lambda name, *args: calls.append((name, args)))
    monkeypatch.setattr(L_, "_stream", lambda: 0)
    cost = torch.zeros(V, 2, D, H, W)
    prob = torch.zeros(V, D, H, W)
    hyp = torch.zeros(V, T, H, W)
    idx = torch.zeros(V, T, H, W, dtype=torch.int64)
    coding = torch.zeros(V, H, W)
    dv = torch.zeros(V, D, H, W) if per_pixel else None
    imap = torch.zeros(V, H, W) if interval_map else None
    interval = imap if interval_map else 0.25
    L_.depth_topk_fwd(cost, prob, prob, hyp, hyp, idx, coding, near=0.5, interval=interval, depth_values=dv)
    g_dv = torch.zeros(V, D, H, W) if per_pixel else None
    L_.depth_topk_bwd(cost, idx, prob, prob, hyp, hyp, coding, cost, near=0.5, interval=interval,
                      depth_values=dv, g_depth_values=g_dv, g_interval_map=imap)
    sfx = "_px" if per_pixel else ""
    assert [n for n, _ in calls] == [f"mvsd_depth_topk_fwd{sfx}", f"mvsd_depth_topk_bwd{sfx}"]
    for name, args in calls:
        assert len(args) == len(L_.SIGNATURES[name][0]), name
        assert tuple(args[-7:-1]) == (0, V, D, H, W, T), name
    if per_pixel:
        fwd, bwd = calls[0][1], calls[1][1]
        assert fwd[5] == dv.data_ptr() and bwd[6] == dv.data_ptr()
        assert fwd[6] == bwd[7] == (imap.data_ptr() if interval_map else None)
        assert fwd[7] == bwd[8] == (0.0 if interval_map else 0.25)
        assert bwd[-9] == g_dv.data_ptr() and bwd[-8] == (imap.data_ptr() if interval_map else None)
    else:
        assert calls[0][1][-9:-7] == (0.5, 0.25) and calls[1][1][-9:-7] == (0.5, 0.25)


@pytest.mark.parametrize("with_map", [False, True], ids=["scalar", "map"])
def test_fake_implementations_and_gradients(with_map):
    f32 = dict(device="meta", dtype=torch.float32)
    cost = torch.empty(V, 2, D, H, W, **f32).requires_grad_(True)
    dv = torch.empty(V, D, H, W, **f32).requires_grad_(True)
    imap = torch.empty(V, H, W, **f32).requires_grad_(True) if with_map else None
    outs = L.depth_topk_px(cost, dv, imap, 0.3, T)
    shapes = [(V, D, H, W), (V, D, H, W), (V, T, H, W), (V, T, H, W), (V, T, H, W), (V, H, W)]
    assert [tuple(o.shape) for o in outs] == shapes
    assert [o.dtype for o in outs] == [torch.float32] * 4 + [torch.int64, torch.float32]
    diff = [outs[i] for i in (0, 1, 2, 3, 5)]
    inputs = (cost, dv) + ((imap,) if with_map else ())
    grads = torch.autograd.grad(diff, inputs, [torch.empty_like(o) for o in diff])
    assert [tuple(g.shape) for g in grads] == [tuple(x.shape) for x in inputs]
    assert all(g.dtype == torch.float32 for g in grads)
    g = L.depth_topk_px_bwd(cost.detach(), outs[4], dv.detach(), None if imap is None else imap.detach(),
                            None, None, None, None, None, 0.3, False)
    assert tuple(g[2].shape) == ((V, H, W) if with_map else (0,))
