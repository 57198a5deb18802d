"""``torch.library`` registration of the path's fused operators (SURVEY.md §8b, "what
calls it"): dispatcher-visible ops ``torch.ops.mvsdet_b200.*`` with

* a CUDA implementation only (``device_types="cuda"``) that enqueues the sm_100a
  kernels through the C ABI -- a CPU tensor has no kernel to dispatch to and raises;
* a fake (meta) implementation giving sizes, strides and dtypes without touching the
  library, so the ops trace under ``FakeTensorMode`` / ``torch.export`` / a compiler that
  wraps the surrounding detector (the ops themselves stay opaque: they are never lowered);
* autograd through ``register_autograd`` whose backward formulas call the ``*_bwd`` ops,
  themselves registered, so double tracing (AOT autograd) sees only these ops.

The ``torch.autograd.Function`` layer in ``ops.py`` is the same arithmetic (both allocate
through the ``_*_raw`` helpers there, check arguments with the same functions and launch
through ``_lib``); it additionally offers caller-owned output buffers for the peer-memory
multi-GPU combine, which a functional dispatcher op cannot (no aliasing of inputs).
``MVSDetHotPath(dispatcher_ops=True)`` routes the drop-in through this module.

Operators (reference lines as in ``ops.py``):

  plane_sweep_variance(feat, nbr_ids, hom, depth_values, out_bf16=False, ref_begin=0) -> variance
      mvsdet.py:439-467 + mvs_models/module.py:105-146; depth_values [V,D] or per-pixel
      [V,D,H,W] (module.py:130-133), in this op and in plane_sweep_group_correlation
  plane_sweep_group_correlation(feat, nbr_ids, hom, depth_values, num_groups=8, ref_begin=0) -> [V,k,G,D,H,W]
      mvs_models/lss_fpn.py:485-506 over mvs_models/module.py:105-146 (optional operator)
  depth_topk(cost_out, near, interval, topk, raw=False)
      -> (prob_volume, off_pred, est_depth, est_densities, est_idx, depth_coding)
      mvsdet.py:470-482, :266-283, :298-317
  depth_topk_px(cost_out, depth_values, interval_map, interval, topk, raw=False) -> the same six
      over per-pixel hypotheses [V,D,H,W] with an [V,H,W] interval map (or None: the scalar);
      its backward also gives dL/ddepth_values and dL/dinterval_map
  backproject_aggregate(feat, points, projection, est_depth, est_dens, vs_z, height, width,
                        sum_only=False, channels_first=True) -> (volume, count)
      mvsdet.py:1372-1492, :511-515, :681-682 (sum_only: the multi-GPU partials)
  voxel_normalize(volume_sum, count) -> volume_mean                      mvsdet.py:514-515
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import ops as _ops
from ._lib import BP_MEAN, BP_SUM

__all__ = ["plane_sweep_variance", "plane_sweep_group_correlation", "depth_topk", "depth_topk_px",
           "backproject_aggregate", "voxel_normalize"]

_NS = "mvsdet_b200"


# --------------------------------------------------------------------------
# plane sweep
# --------------------------------------------------------------------------
@torch.library.custom_op(f"{_NS}::plane_sweep_variance", mutates_args=(), device_types="cuda")
def plane_sweep_variance(feat: Tensor, nbr_ids: Tensor, hom: Tensor, depth_values: Tensor,
                         out_bf16: bool = False, ref_begin: int = 0) -> Tensor:
    _ops._check_sweep(feat, nbr_ids, hom, depth_values, ref_begin)
    return _ops._sweep_fwd_raw(feat, nbr_ids, hom.contiguous(), depth_values.contiguous(),
                               torch.bfloat16 if out_bf16 else torch.float32, int(ref_begin))


@plane_sweep_variance.register_fake
def _(feat, nbr_ids, hom, depth_values, out_bf16=False, ref_begin=0):
    _, c, h, w = feat.shape
    return _ops._empty_ndhwc(nbr_ids.shape[0], c, depth_values.shape[1], h, w,
                             torch.bfloat16 if out_bf16 else torch.float32, feat.device)


@torch.library.custom_op(f"{_NS}::plane_sweep_variance_bwd", mutates_args=(), device_types="cuda")
def plane_sweep_variance_bwd(g: Tensor, feat: Tensor, nbr_ids: Tensor, hom: Tensor,
                             depth_values: Tensor, ref_begin: int) -> Tensor:
    return _ops._sweep_bwd_raw(g, feat, nbr_ids, hom, depth_values, int(ref_begin))


@plane_sweep_variance_bwd.register_fake
def _(g, feat, nbr_ids, hom, depth_values, ref_begin):
    v, c, h, w = feat.shape
    return _ops._empty_nhwc(v, c, h, w, feat.dtype, feat.device)


def _sweep_setup(ctx, inputs, output):
    feat, nbr_ids, hom, depth_values, _out_bf16, ref_begin = inputs
    ctx.save_for_backward(feat, nbr_ids, hom, depth_values)
    ctx.ref_begin = ref_begin


def _sweep_backward(ctx, g):
    feat, nbr_ids, hom, depth_values = ctx.saved_tensors
    g_feat = plane_sweep_variance_bwd(g, feat, nbr_ids, hom.contiguous(), depth_values.contiguous(),
                                      ctx.ref_begin)
    return g_feat, None, None, None, None, None


plane_sweep_variance.register_autograd(_sweep_backward, setup_context=_sweep_setup)


# --------------------------------------------------------------------------
# group-wise correlation volume (optional operator, SURVEY.md 8f rank 4)
# --------------------------------------------------------------------------
@torch.library.custom_op(f"{_NS}::plane_sweep_group_correlation", mutates_args=(), device_types="cuda")
def plane_sweep_group_correlation(feat: Tensor, nbr_ids: Tensor, hom: Tensor, depth_values: Tensor,
                                  num_groups: int = 8, ref_begin: int = 0) -> Tensor:
    _ops._check_corr(feat, nbr_ids, hom, depth_values, num_groups, ref_begin)
    return _ops._corr_fwd_raw(feat, nbr_ids, hom.contiguous(), depth_values.contiguous(), int(num_groups),
                              int(ref_begin))


@plane_sweep_group_correlation.register_fake
def _(feat, nbr_ids, hom, depth_values, num_groups=8, ref_begin=0):
    _, _, h, w = feat.shape
    v, k = nbr_ids.shape
    return torch.empty((v, k, depth_values.shape[1], h, w, num_groups), dtype=torch.float32,
                       device=feat.device).permute(0, 1, 5, 2, 3, 4)


@torch.library.custom_op(f"{_NS}::plane_sweep_group_correlation_bwd", mutates_args=(), device_types="cuda")
def plane_sweep_group_correlation_bwd(g: Tensor, feat: Tensor, nbr_ids: Tensor, hom: Tensor,
                                      depth_values: Tensor, num_groups: int, ref_begin: int) -> Tensor:
    return _ops._corr_bwd_raw(g, feat, nbr_ids, hom, depth_values, int(ref_begin))


@plane_sweep_group_correlation_bwd.register_fake
def _(g, feat, nbr_ids, hom, depth_values, num_groups, ref_begin):
    v, c, h, w = feat.shape
    return _ops._empty_nhwc(v, c, h, w, feat.dtype, feat.device)


def _corr_setup(ctx, inputs, output):
    feat, nbr_ids, hom, depth_values, num_groups, ref_begin = inputs
    ctx.save_for_backward(feat, nbr_ids, hom, depth_values)
    ctx.meta = (num_groups, ref_begin)


def _corr_backward(ctx, g):
    feat, nbr_ids, hom, depth_values = ctx.saved_tensors
    num_groups, ref_begin = ctx.meta
    g_feat = plane_sweep_group_correlation_bwd(g, feat, nbr_ids, hom.contiguous(), depth_values.contiguous(),
                                               num_groups, ref_begin)
    return g_feat, None, None, None, None, None


plane_sweep_group_correlation.register_autograd(_corr_backward, setup_context=_corr_setup)


# --------------------------------------------------------------------------
# softmax / sigmoid / top-k / expectation
# --------------------------------------------------------------------------
def _topk_outputs(cost_out, topk):
    v, _, d, h, w = cost_out.shape
    f32 = dict(dtype=torch.float32, device=cost_out.device)
    return (torch.empty((v, d, h, w), **f32), torch.empty((v, d, h, w), **f32),
            torch.empty((v, topk, h, w), **f32), torch.empty((v, topk, h, w), **f32),
            torch.empty((v, topk, h, w), dtype=torch.int64, device=cost_out.device),
            torch.empty((v, h, w), **f32))


@torch.library.custom_op(f"{_NS}::depth_topk", mutates_args=(), device_types="cuda")
def depth_topk(cost_out: Tensor, near: float, interval: float, topk: int,
               raw: bool = False) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    _ops._check_cost("cost_out", cost_out)
    _, outs = _ops._topk_fwd_raw(cost_out, near, interval, int(topk), int(raw))
    return outs


@depth_topk.register_fake
def _(cost_out, near, interval, topk, raw=False):
    return _topk_outputs(cost_out, topk)


@torch.library.custom_op(f"{_NS}::depth_topk_bwd", mutates_args=(), device_types="cuda")
def depth_topk_bwd(cost_out: Tensor, est_idx: Tensor, g_prob: Optional[Tensor], g_off: Optional[Tensor],
                   g_depth: Optional[Tensor], g_dens: Optional[Tensor], g_coding: Optional[Tensor],
                   near: float, interval: float, topk: int, raw: bool) -> Tensor:
    return _ops._topk_bwd_raw(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding,
                              near, interval, int(raw))


@depth_topk_bwd.register_fake
def _(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding, near, interval, topk, raw):
    v, _, d, h, w = cost_out.shape
    return torch.empty((v, 2, d, h, w), dtype=torch.float32, device=cost_out.device)


def _topk_setup(ctx, inputs, output):
    cost_out, near, interval, topk, raw = inputs
    ctx.save_for_backward(cost_out, output[4])
    ctx.consts = (float(near), float(interval), int(topk), bool(raw))


def _topk_backward(ctx, g_prob, g_off, g_depth, g_dens, _g_idx, g_coding):
    cost_out, est_idx = ctx.saved_tensors
    near, interval, topk, raw = ctx.consts
    g_cost = depth_topk_bwd(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding,
                            near, interval, topk, raw)
    if g_cost.dtype != cost_out.dtype:
        g_cost = g_cost.to(cost_out.dtype)
    return g_cost, None, None, None, None


depth_topk.register_autograd(_topk_backward, setup_context=_topk_setup)


@torch.library.custom_op(f"{_NS}::depth_topk_px", mutates_args=(), device_types="cuda")
def depth_topk_px(cost_out: Tensor, depth_values: Tensor, interval_map: Optional[Tensor], interval: float,
                  topk: int, raw: bool = False) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    iv = interval if interval_map is None else interval_map
    _ops._check_topk_px("cost_out", cost_out, depth_values, iv)
    _, outs = _ops._topk_fwd_raw(cost_out, None, iv if interval_map is None else interval_map.contiguous(),
                                 int(topk), int(raw), depth_values=depth_values.contiguous())
    return outs


@depth_topk_px.register_fake
def _(cost_out, depth_values, interval_map, interval, topk, raw=False):
    return _topk_outputs(cost_out, topk)


@torch.library.custom_op(f"{_NS}::depth_topk_px_bwd", mutates_args=(), device_types="cuda")
def depth_topk_px_bwd(cost_out: Tensor, est_idx: Tensor, depth_values: Tensor, interval_map: Optional[Tensor],
                      g_prob: Optional[Tensor], g_off: Optional[Tensor], g_depth: Optional[Tensor],
                      g_dens: Optional[Tensor], g_coding: Optional[Tensor], interval: float,
                      raw: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (dL/dcost_out, dL/ddepth_values, dL/dinterval_map: [V,H,W], or [0] without a map)"""
    depth_values = depth_values.contiguous()
    g_dv = torch.empty_like(depth_values)
    if interval_map is None:
        g_im = torch.empty((0,), dtype=torch.float32, device=cost_out.device)
        iv = interval
    else:
        iv = interval_map.contiguous()
        g_im = torch.empty_like(iv)
    g_cost = _ops._topk_bwd_raw(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding, None, iv, int(raw),
                                depth_values=depth_values, g_depth_values=g_dv,
                                g_interval_map=None if interval_map is None else g_im)
    return g_cost, g_dv, g_im


@depth_topk_px_bwd.register_fake
def _(cost_out, est_idx, depth_values, interval_map, g_prob, g_off, g_depth, g_dens, g_coding, interval, raw):
    v, _, d, h, w = cost_out.shape
    f32 = dict(dtype=torch.float32, device=cost_out.device)
    return (torch.empty((v, 2, d, h, w), **f32), torch.empty((v, d, h, w), **f32),
            torch.empty((0,) if interval_map is None else (v, h, w), **f32))


def _topk_px_setup(ctx, inputs, output):
    cost_out, depth_values, interval_map, interval, topk, raw = inputs
    ctx.save_for_backward(cost_out, output[4], depth_values, interval_map)
    ctx.consts = (float(interval), bool(raw))


def _topk_px_backward(ctx, g_prob, g_off, g_depth, g_dens, _g_idx, g_coding):
    cost_out, est_idx, depth_values, interval_map = ctx.saved_tensors
    interval, raw = ctx.consts
    g_cost, g_dv, g_im = depth_topk_px_bwd(cost_out, est_idx, depth_values, interval_map, g_prob, g_off, g_depth,
                                           g_dens, g_coding, interval, raw)
    if g_cost.dtype != cost_out.dtype:
        g_cost = g_cost.to(cost_out.dtype)
    return g_cost, g_dv, (None if interval_map is None else g_im), None, None, None


depth_topk_px.register_autograd(_topk_px_backward, setup_context=_topk_px_setup)


# --------------------------------------------------------------------------
# back-projection + aggregation
# --------------------------------------------------------------------------
@torch.library.custom_op(f"{_NS}::backproject_aggregate", mutates_args=(), device_types="cuda")
def backproject_aggregate(feat: Tensor, points: Tensor, projection: Tensor, est_depth: Tensor,
                          est_dens: Tensor, vs_z: float, height: int, width: int,
                          sum_only: bool = False, channels_first: bool = True) -> Tuple[Tensor, Tensor]:
    _ops._check_bp(feat, points, projection, est_depth, est_dens, height, width)
    if est_depth.stride() != est_dens.stride():
        est_depth, est_dens = est_depth.contiguous(), est_dens.contiguous()
    return _ops._bp_fwd_raw(feat, points.contiguous().float(), projection.contiguous().float(),
                            est_depth, est_dens, float(vs_z), int(height), int(width),
                            BP_SUM if sum_only else BP_MEAN, bool(channels_first))


@backproject_aggregate.register_fake
def _(feat, points, projection, est_depth, est_dens, vs_z, height, width, sum_only=False,
      channels_first=True):
    c = feat.shape[1]
    n = points.numel() // 3
    vol = torch.empty((c, n) if channels_first else (n, c), dtype=torch.float32, device=feat.device)
    return (vol if channels_first else vol.t()), torch.empty((n,), dtype=torch.int32, device=feat.device)


@torch.library.custom_op(f"{_NS}::backproject_aggregate_bwd", mutates_args=(), device_types="cuda")
def backproject_aggregate_bwd(g_out: Tensor, feat: Tensor, points: Tensor, projection: Tensor,
                              est_depth: Tensor, est_dens: Tensor, count: Tensor, vs_z: float,
                              height: int, width: int, sum_only: bool,
                              channels_first: bool) -> Tuple[Tensor, Tensor]:
    if est_depth.stride() != est_dens.stride():
        est_depth, est_dens = est_depth.contiguous(), est_dens.contiguous()
    return _ops._bp_bwd_raw(g_out, feat, points.contiguous().float(), projection.contiguous().float(),
                            est_depth, est_dens, count, float(vs_z), int(height), int(width),
                            BP_SUM if sum_only else BP_MEAN, bool(channels_first))


@backproject_aggregate_bwd.register_fake
def _(g_out, feat, points, projection, est_depth, est_dens, count, vs_z, height, width, sum_only,
      channels_first):
    v, c, fh, fw = feat.shape
    if est_depth.stride() != est_dens.stride():
        est_dens = est_dens.contiguous()
    return (_ops._empty_nhwc(v, c, fh, fw, feat.dtype, feat.device),
            torch.empty_strided(est_dens.size(), est_dens.stride(), dtype=est_dens.dtype,
                                device=est_dens.device))


def _bp_setup(ctx, inputs, output):
    feat, points, projection, est_depth, est_dens, vs_z, height, width, sum_only, channels_first = inputs
    ctx.save_for_backward(feat, points, projection, est_depth, est_dens, output[1])
    ctx.consts = (float(vs_z), int(height), int(width), bool(sum_only), bool(channels_first))


def _bp_backward(ctx, g_out, _g_count):
    feat, points, projection, est_depth, est_dens, count = ctx.saved_tensors
    vs_z, height, width, sum_only, channels_first = ctx.consts
    g_feat, g_prob = backproject_aggregate_bwd(g_out, feat, points, projection, est_depth, est_dens,
                                               count, vs_z, height, width, sum_only, channels_first)
    return g_feat, None, None, None, g_prob, None, None, None, None, None


backproject_aggregate.register_autograd(_bp_backward, setup_context=_bp_setup)


# --------------------------------------------------------------------------
# normalisation of all-reduced partials
# --------------------------------------------------------------------------
@torch.library.custom_op(f"{_NS}::voxel_normalize", mutates_args=(), device_types="cuda")
def voxel_normalize(volume_sum: Tensor, count: Tensor) -> Tensor:
    return _ops.voxel_normalize(volume_sum, count)


@voxel_normalize.register_fake
def _(volume_sum, count):
    return torch.empty_strided(volume_sum.size(), volume_sum.stride(), dtype=volume_sum.dtype,
                               device=volume_sum.device)
