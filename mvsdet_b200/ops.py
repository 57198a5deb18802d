"""PyTorch custom-op layer over the C ABI (include/mvsdet_b200.h).

Each op is a ``torch.autograd.Function`` whose forward and backward enqueue the
hand-written sm_100a kernels on ``torch.cuda.current_stream()`` through ctypes;
PyTorch only owns the memory.  There is deliberately no CPU / eager fallback:
a CPU tensor is a ``ValueError`` and a missing library an exception at first
use.

Tensor conventions: feature maps have logical shape [V,C,H,W] in
``torch.channels_last`` memory format; volumes have logical shape [V,C,D,H,W]
in ``torch.channels_last_3d`` -- the reference's logical shapes
(mvs_models/module.py:105-111, mvsdet.py:439-467), with the memory format the
kernels (and cuDNN's Conv3d after them) want.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import BP_MEAN, BP_PER_VIEW, BP_SUM

__all__ = ["pack_features", "plane_sweep_variance", "homo_warp", "depth_topk", "depth_topk_nvs",
           "topk_hypotheses", "ray_depth_scale", "rgb_downsample4", "backproject_aggregate",
           "backproject_per_view", "voxel_normalize", "scene_setup", "volume_to_ncdhw", "FeatureGradSink"]


# --------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------
def _need_cuda(name: str, t: torch.Tensor) -> None:
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{name} must be a tensor")
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor: mvsdet_b200 has no CPU path")


def _is_nhwc(t: torch.Tensor) -> bool:
    return t.dim() == 4 and t.permute(0, 2, 3, 1).is_contiguous()


def _is_ndhwc(t: torch.Tensor) -> bool:
    return t.dim() == 5 and t.permute(0, 2, 3, 4, 1).is_contiguous()


def _empty_nhwc(v, c, h, w, dtype, device) -> torch.Tensor:
    return torch.empty((v, h, w, c), dtype=dtype, device=device).permute(0, 3, 1, 2)


def _zeros_nhwc(v, c, h, w, dtype, device) -> torch.Tensor:
    return torch.zeros((v, h, w, c), dtype=dtype, device=device).permute(0, 3, 1, 2)


def _empty_ndhwc(v, c, d, h, w, dtype, device) -> torch.Tensor:
    return torch.empty((v, d, h, w, c), dtype=dtype, device=device).permute(0, 4, 1, 2, 3)


# Re-layouts of a volume-sized gradient are a hidden 1.2 GB transpose per scene: they are counted so a
# caller (and tests/test_gpu_costreg.py, with the real CostRegNet_3DGS attached) can assert that the
# upstream gradient arrives in channels_last_3d and that no copy fires.
relayout_count = {"g_variance": 0, "g_variance_cast": 0}


def _as_ndhwc(t: torch.Tensor, dtype=None) -> torch.Tensor:
    if dtype is not None and t.dtype != dtype:
        relayout_count["g_variance_cast"] += 1
        t = t.to(dtype)
    if _is_ndhwc(t):
        return t
    relayout_count["g_variance"] += 1
    return t.contiguous(memory_format=torch.channels_last_3d)


# --------------------------------------------------------------------------
# layout: [V,C,H,W] fp32 contiguous <-> channels-last
# --------------------------------------------------------------------------
class FeatureGradSink:
    """One fp32 channels-last gradient accumulator shared by every consumer of a packed feature
    tensor (the training-step form ``ScenePipeline`` uses, expressed in autograd).

    Without it each backward node allocates and zero-fills its own 98 MB accumulator, the engine
    casts every partial gradient to the packed tensor's dtype (bf16: 2^-9 relative rounding),
    adds the partials, and the pack node converts back to fp32 before the transpose.  With a sink
    the plane-sweep and back-projection backward kernels RED into ONE accumulator in fp32, return
    no gradient for the packed tensor, and ``pack_features``' backward transposes the accumulator
    to the FPN's fp32 NCHW layout once: fp32 accumulation end to end, ~0.5 GB less traffic per
    scene.  Created by ``pack_features(x, dtype, sink=True)``; an implementation detail of
    ``MVSDetHotPath.forward``."""

    def __init__(self, shape, device, deterministic: bool = False):
        self.shape = tuple(shape)          # logical [V,C,H,W]
        self.device = device
        self.deterministic = bool(deterministic)
        self.buf: Optional[torch.Tensor] = None

    def get(self) -> torch.Tensor:
        """the accumulator (logical [V,C,H,W], channels-last memory), zero-filled on first use.
        (Pre-filling it at forward time on a side stream was measured: the cross-stream
        ``record_stream`` defeats the caching allocator's block reuse, 820 -> 692 scenes/s.)
        ``deterministic``: int64 fixed point (32 fractional bits) for the ``*_det`` kernels, whose
        integer REDs make the sum independent of the order the warps arrive in."""
        if self.buf is None:
            v, c, h, w = self.shape
            self.buf = _zeros_nhwc(v, c, h, w, torch.int64 if self.deterministic else torch.float32, self.device)
        return self.buf

    def take(self) -> Optional[torch.Tensor]:
        """-> the fp32 accumulator (converted once from fixed point in the deterministic form)"""
        buf, self.buf = self.buf, None
        if buf is not None and self.deterministic:
            buf = fixed_to_float(buf)
        return buf


def fixed_to_float(q: torch.Tensor) -> torch.Tensor:
    """mvsd_fixed_to_float: an int64 fixed-point accumulator of the ``*_det`` kernels -> fp32, same
    shape and memory layout."""
    _need_cuda("accumulator", q)
    if q.dtype != torch.int64:
        raise ValueError("fixed_to_float takes an int64 accumulator")
    out = torch.empty_like(q, dtype=torch.float32)
    if q.numel():
        _lib.fixed_to_float(q, out)
    return out


def _pack(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    out = _empty_nhwc(*x.shape, dtype, x.device)
    _lib.pack(x, out)
    return out


def _unpack(acc: torch.Tensor) -> torch.Tensor:
    out = torch.empty(acc.shape, dtype=torch.float32, device=acc.device)
    _lib.unpack(acc, out)
    return out


class _PackFeaturesSink(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: torch.Tensor, dtype: torch.dtype, sink: FeatureGradSink):
        out = _pack(x, dtype)
        ctx.sink = sink
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, g):
        acc = ctx.sink.take()
        if g is not None:                   # a consumer that does not know the sink
            g = g.float()
            acc = g if acc is None else acc.add_(g)
        if acc is None:
            return None, None, None
        if not _is_nhwc(acc):
            acc = acc.contiguous(memory_format=torch.channels_last)
        return _unpack(acc), None, None


class _PackFeatures(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: torch.Tensor, dtype: torch.dtype):
        return _pack(x, dtype)

    @staticmethod
    def backward(ctx, g: torch.Tensor):
        if g.dtype != torch.float32 or not _is_nhwc(g):
            g = g.float().contiguous(memory_format=torch.channels_last)
        return _unpack(g), None


def pack_features(x: torch.Tensor, dtype: torch.dtype = torch.float32, sink: bool = False,
                  deterministic: bool = False):
    """[V,C,H,W] features -> the same logical tensor in channels_last memory
    format and ``dtype`` (fp32 or bf16).  A tensor that already has that layout
    and dtype is returned as is; an fp32 NCHW-contiguous tensor (the reference's
    FPN output, mvsdet.py:373-376) goes through the transpose kernel.

    ``sink=True`` returns ``(packed, FeatureGradSink | None)``: when ``x`` needs a gradient and goes
    through the transpose kernel, the sink collects the fp32 gradients of the consumers that are
    given it (``plane_sweep_variance(..., grad_sink=)``, ``backproject_aggregate(..., grad_sink=)``)."""
    _need_cuda("features", x)
    if x.dim() != 4:
        raise ValueError("features must be [V,C,H,W]")
    if _is_nhwc(x) and x.shape[1] > 1:
        out = x if x.dtype == dtype else x.to(dtype)
        return (out, None) if sink else out
    if x.dtype != torch.float32 or not x.is_contiguous():
        x = x.float().contiguous()
    if sink and x.requires_grad and torch.is_grad_enabled():
        gs = FeatureGradSink(x.shape, x.device, deterministic)
        return _PackFeaturesSink.apply(x, dtype, gs), gs
    out = _PackFeatures.apply(x, dtype)
    return (out, None) if sink else out


class _VolumeToNCDHW(torch.autograd.Function):
    """[V,C,D,H,W] logical volume in channels_last_3d memory -> the reference's strict NCDHW
    contiguous memory (and back for the gradient), with the same transpose kernels as the feature
    maps: a volume is a feature map with H' = D*H."""

    @staticmethod
    def forward(ctx, vol):
        return _unpack(vol)

    @staticmethod
    def backward(ctx, g):
        g = g.float().contiguous()
        out = _empty_ndhwc(*g.shape, torch.float32, g.device)
        _lib.pack(g, out)
        return out


def volume_to_ncdhw(vol: torch.Tensor) -> torch.Tensor:
    """The variance volume as the reference materialises it: [V,C,D,H,W] fp32 CONTIGUOUS
    (mvsdet.py:439-467).  The kernels produce channels_last_3d, which cuDNN's Conv3d (the only
    consumer, mvsnet.py:76) takes as is; a consumer that needs strict NCDHW memory pays one extra
    transpose pass here (2.4 GB of traffic at the benchmark size, ~0.4 ms)."""
    _need_cuda("volume", vol)
    if vol.dim() != 5:
        raise ValueError("volume must be [V,C,D,H,W]")
    if vol.is_contiguous():
        return vol
    if vol.dtype != torch.float32 or not _is_ndhwc(vol):
        raise ValueError("volume_to_ncdhw takes an fp32 channels_last_3d volume")
    return _VolumeToNCDHW.apply(vol)


# --------------------------------------------------------------------------
# plane sweep
# --------------------------------------------------------------------------
def _sweep_fwd_raw(feat, nbr_ids, hom, depth_values, out_dtype, ref_begin):
    """-> variance, logical [V,C,D,H,W] in channels_last_3d"""
    _, c, h, w = feat.shape
    out = _empty_ndhwc(nbr_ids.shape[0], c, depth_values.shape[1], h, w, out_dtype, feat.device)
    _lib.plane_sweep_fwd(feat, nbr_ids, hom, depth_values, out, ref_begin=ref_begin)
    return out


def _sweep_bwd_raw(g, feat, nbr_ids, hom, depth_values, ref_begin, acc=None):
    """-> dL/dfeat in feat's dtype, channels_last.  ``acc``: an fp32 channels-last accumulator to
    RED into instead (FeatureGradSink); returns None then."""
    gdt = torch.bfloat16 if (g.dtype == torch.bfloat16 and feat.dtype == torch.bfloat16) else torch.float32
    g = _as_ndhwc(g, gdt)
    if acc is not None and acc.dtype == torch.int64:        # deterministic sink: fixed-point integer REDs
        _lib.plane_sweep_bwd_det(g, feat, nbr_ids, hom, depth_values, acc, ref_begin=ref_begin)
        return None
    g_feat = acc if acc is not None else _zeros_nhwc(*feat.shape, torch.float32, feat.device)
    _lib.plane_sweep_bwd(g, feat, nbr_ids, hom, depth_values, g_feat, ref_begin=ref_begin)
    return None if acc is not None else g_feat.to(feat.dtype)


class _PlaneSweepVariance(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, nbr_ids, hom, depth_values, out_dtype, ref_begin, sink=None):
        out = _sweep_fwd_raw(feat, nbr_ids, hom, depth_values, out_dtype, ref_begin)
        ctx.save_for_backward(feat, nbr_ids, hom, depth_values)
        ctx.ref_begin = ref_begin
        ctx.sink = sink
        return out

    @staticmethod
    def backward(ctx, g):
        feat, nbr_ids, hom, depth_values = ctx.saved_tensors
        acc = ctx.sink.get() if ctx.sink is not None else None
        g_feat = _sweep_bwd_raw(g, feat, nbr_ids, hom, depth_values, ctx.ref_begin, acc)
        return g_feat, None, None, None, None, None, None


# The argument checks of an operator (_check_*) are shared by its function here and its
# dispatcher op in library.py.
def _check_sweep(feat, nbr_ids, hom, depth_values, ref_begin, grad_sink=None) -> None:
    for n, t in (("feat", feat), ("nbr_ids", nbr_ids), ("hom", hom), ("depth_values", depth_values)):
        _need_cuda(n, t)
    if not _is_nhwc(feat):
        raise ValueError("feat must be channels_last; use ops.pack_features")
    if nbr_ids.dtype != torch.int32 or not nbr_ids.is_contiguous():
        raise ValueError("nbr_ids must be contiguous int32 [V,k]")
    v, k = nbr_ids.shape
    if tuple(hom.shape) != (v, k, 12) or depth_values.shape[0] != v:
        raise ValueError("nbr_ids [V,k], hom [V,k,12] and depth_values [V,D] must agree")
    if ref_begin < 0 or ref_begin + v > feat.shape[0]:
        raise ValueError("reference views [ref_begin, ref_begin+V) exceed feat")
    if hom.dtype != torch.float32 or depth_values.dtype != torch.float32:
        raise ValueError("hom and depth_values must be float32")
    if grad_sink is not None and grad_sink.shape != tuple(feat.shape):
        raise ValueError("grad_sink belongs to a different feature tensor")


def plane_sweep_variance(feat: torch.Tensor, nbr_ids: torch.Tensor, hom: torch.Tensor,
                         depth_values: torch.Tensor,
                         out_dtype: torch.dtype = torch.float32,
                         ref_begin: int = 0, grad_sink: Optional[FeatureGradSink] = None) -> torch.Tensor:
    """Fused mvsdet.py:439-467: channels-last features [Vf,C,H,W] (fp32/bf16),
    neighbour ids [V,k] int32 (indices into feat), homographies [V,k,12], depth
    planes [V,D] -> variance volume, logical [V,C,D,H,W] in channels_last_3d.
    Reference view v is feat[ref_begin + v]; V < Vf sweeps a slice of the views
    (view-sharded multi-GPU)."""
    _check_sweep(feat, nbr_ids, hom, depth_values, ref_begin, grad_sink)
    return _PlaneSweepVariance.apply(feat, nbr_ids, hom.contiguous(), depth_values.contiguous(),
                                     out_dtype, int(ref_begin), grad_sink)


def _corr_fwd_raw(feat, nbr_ids, hom, depth_values, num_groups, ref_begin):
    """-> logical [V,k,G,D,H,W] fp32, groups innermost in memory"""
    _, _, h, w = feat.shape
    v, k = nbr_ids.shape
    out = torch.empty((v, k, depth_values.shape[1], h, w, num_groups), dtype=torch.float32,
                      device=feat.device).permute(0, 1, 5, 2, 3, 4)
    _lib.plane_sweep_groupcorr_fwd(feat, nbr_ids, hom, depth_values, out, ref_begin=ref_begin)
    return out


def _corr_bwd_raw(g, feat, nbr_ids, hom, depth_values, ref_begin, acc=None):
    """-> dL/dfeat in feat's dtype (channels_last), or None when it was accumulated into the fp32
    accumulator ``acc`` (FeatureGradSink)"""
    # no copy when it arrives in the forward's layout
    g = g.float().permute(0, 1, 3, 4, 5, 2).contiguous().permute(0, 1, 5, 2, 3, 4)
    if acc is not None and acc.dtype != torch.float32:
        raise ValueError("the group-correlation backward has no deterministic form")
    g_feat = acc if acc is not None else _zeros_nhwc(*feat.shape, torch.float32, feat.device)
    _lib.plane_sweep_groupcorr_bwd(g, feat, nbr_ids, hom, depth_values, g_feat, ref_begin=ref_begin)
    return None if acc is not None else g_feat.to(feat.dtype)


class _GroupCorrelation(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, nbr_ids, hom, depth_values, num_groups, ref_begin, sink=None):
        out = _corr_fwd_raw(feat, nbr_ids, hom, depth_values, num_groups, ref_begin)
        ctx.save_for_backward(feat, nbr_ids, hom, depth_values)
        ctx.ref_begin = ref_begin
        ctx.sink = sink
        return out

    @staticmethod
    def backward(ctx, g):
        feat, nbr_ids, hom, depth_values = ctx.saved_tensors
        acc = ctx.sink.get() if ctx.sink is not None else None
        g_feat = _corr_bwd_raw(g, feat, nbr_ids, hom, depth_values, ctx.ref_begin, acc)
        return g_feat, None, None, None, None, None, None


def _check_corr(feat, nbr_ids, hom, depth_values, num_groups, ref_begin, grad_sink=None) -> None:
    _check_sweep(feat, nbr_ids, hom, depth_values, ref_begin, grad_sink)
    if nbr_ids.shape[1] < 1:
        raise ValueError("group correlation needs at least one neighbour")
    if depth_values.dim() != 2:
        raise ValueError("nbr_ids [V,k], hom [V,k,12] and depth_values [V,D] must agree")
    if num_groups < 1 or feat.shape[1] % num_groups != 0:
        raise ValueError("the channel count must be divisible by num_groups")


def plane_sweep_group_correlation(feat: torch.Tensor, nbr_ids: torch.Tensor, hom: torch.Tensor,
                                  depth_values: torch.Tensor, num_groups: int = 8, ref_begin: int = 0,
                                  grad_sink: Optional[FeatureGradSink] = None) -> torch.Tensor:
    """Group-wise correlation cost volumes over the plane sweep (SURVEY.md 8f rank 4; the reference's
    arithmetic is mvs_models/lss_fpn.py:485-506, the warp mvs_models/module.py:105-146): same arguments
    as ``plane_sweep_variance``; -> logical [V,k,num_groups,D,H,W] fp32, one volume per neighbour,
    ``mean over the group's channels of ref * warped_j``.  C / num_groups must be 4 ... 128 and divide
    128.  The memory order is [V,k,D,H,W,num_groups]."""
    _check_corr(feat, nbr_ids, hom, depth_values, num_groups, ref_begin, grad_sink)
    return _GroupCorrelation.apply(feat, nbr_ids, hom.contiguous(), depth_values.contiguous(),
                                   int(num_groups), int(ref_begin), grad_sink)


class _HomoWarp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, hom, depth_values, out_dtype):
        b, c, h, w = src.shape
        out = _empty_ndhwc(b, c, depth_values.shape[1], h, w, out_dtype, src.device)
        _lib.homo_warp_fwd(src, hom, depth_values, out)
        ctx.save_for_backward(hom, depth_values)
        ctx.src_meta = (src.shape, src.dtype)
        return out

    @staticmethod
    def backward(ctx, g):
        hom, depth_values = ctx.saved_tensors
        shape, sdtype = ctx.src_meta
        g = _as_ndhwc(g, torch.float32 if g.dtype != torch.bfloat16 else torch.bfloat16)
        g_src = _zeros_nhwc(*shape, torch.float32, g.device)
        _lib.homo_warp_bwd(g, hom, depth_values, g_src)
        return g_src.to(sdtype), None, None, None


def homo_warp(src: torch.Tensor, hom: torch.Tensor, depth_values: torch.Tensor,
              out_dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """mvs_models/module.py:105-146 with the homography already reduced to
    [B,12] (rot rows, trans): channels-last [B,C,H,W] -> [B,C,D,H,W].
    ``depth_values`` is [B,D] or the per-pixel form [B,D,H,W] (module.py:130-133)."""
    for n, t in (("src", src), ("hom", hom), ("depth_values", depth_values)):
        _need_cuda(n, t)
    if not _is_nhwc(src):
        raise ValueError("src must be channels_last; use ops.pack_features")
    if depth_values.dim() not in (2, 4) or depth_values.shape[0] != src.shape[0] or \
            (depth_values.dim() == 4 and tuple(depth_values.shape[2:]) != tuple(src.shape[2:])):
        raise ValueError("depth_values must be [B,D] or [B,D,H,W]")
    return _HomoWarp.apply(src, hom.contiguous().float(), depth_values.contiguous().float(), out_dtype)


# --------------------------------------------------------------------------
# softmax / sigmoid / top-k / expectation
# --------------------------------------------------------------------------
def _as_cost(cost_out: torch.Tensor) -> torch.Tensor:
    """fp32, NCDHW-contiguous or channels_last_3d (any strides with s_h = W * s_w)"""
    if cost_out.dtype != torch.float32:
        cost_out = cost_out.float()
    sv, sc, sd, sh, sw = cost_out.stride()
    if sh != cost_out.shape[4] * sw or (cost_out.numel() and min(sv, sc, sd, sw) < 1):
        cost_out = cost_out.contiguous()
    return cost_out


def _ray_intr(ray_intr, v):
    """[4,4] or [V,4,4] fp32 feature-level intrinsics"""
    if ray_intr is None:
        return None
    _need_cuda("ray_intrinsics", ray_intr)
    k = ray_intr.float().contiguous()
    if tuple(k.shape) in ((4, 4), (v, 4, 4)):
        return k
    raise ValueError(f"ray intrinsics must be [4,4] or [{v},4,4], got {tuple(ray_intr.shape)}")


def _topk_fwd_raw(cost_out, near, interval, topk, raw, ray_intr=None):
    """-> (cost_out as the kernel read it, the six outputs, and with ``ray_intr`` the four NVS
    outputs opacity, depth_scale, est_ray_depth, ray_depth_coding)"""
    cost_out = _as_cost(cost_out)
    v, _, d, h, w = cost_out.shape
    dev = cost_out.device
    f32 = dict(dtype=torch.float32, device=dev)
    prob = torch.empty((v, d, h, w), **f32)
    off = torch.empty((v, d, h, w), **f32)
    est_depth = torch.empty((v, topk, h, w), **f32)
    est_dens = torch.empty((v, topk, h, w), **f32)
    est_idx = torch.empty((v, topk, h, w), dtype=torch.int64, device=dev)
    coding = torch.empty((v, h, w), **f32)
    kmat = _ray_intr(ray_intr, v)
    nvs = ()
    if kmat is not None:
        nvs = (torch.empty((v, h, w), **f32), torch.empty((v, h, w), **f32),
               torch.empty((v, topk, h, w), **f32), torch.empty((v, h, w), **f32))
    _lib.depth_topk_fwd(cost_out, prob, off, est_depth, est_dens, est_idx, coding, near=near,
                        interval=interval, raw=raw, ray_intr=kmat, nvs=nvs or (None,) * 4)
    return cost_out, (prob, off, est_depth, est_dens, est_idx, coding) + nvs


def _topk_bwd_raw(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding, near, interval,
                  raw, ray_intr=None, g_ray_depth=None, g_ray_coding=None):
    """-> dL/dcost_out (any of the upstream gradients may be None)"""
    cost_out = _as_cost(cost_out)

    def prep(g):
        return None if g is None else g.contiguous().float()
    g_prob, g_off, g_depth, g_dens, g_coding, g_ray_depth, g_ray_coding = map(
        prep, (g_prob, g_off, g_depth, g_dens, g_coding, g_ray_depth, g_ray_coding))
    kmat = _ray_intr(ray_intr, cost_out.shape[0])
    g_cost = torch.empty(cost_out.shape, dtype=torch.float32, device=cost_out.device)
    _lib.depth_topk_bwd(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding, g_cost, near=near,
                        interval=interval, raw=raw, ray_intr=kmat, g_ray_depth=g_ray_depth,
                        g_ray_coding=g_ray_coding)
    return g_cost


def _check_cost(name, cost_out) -> None:
    _need_cuda(name, cost_out)
    if cost_out.dim() != 5 or cost_out.shape[1] != 2:
        raise ValueError(f"{name} must be [V,2,D,H,W]")


class _DepthTopk(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cost_out, near, interval, topk, raw):
        cost_out, outs = _topk_fwd_raw(cost_out, near, interval, topk, raw)
        ctx.save_for_backward(cost_out, outs[4])
        ctx.consts = (float(near), float(interval), int(raw))
        ctx.mark_non_differentiable(outs[4])
        return outs

    @staticmethod
    def backward(ctx, g_prob, g_off, g_depth, g_dens, _g_idx, g_coding):
        cost_out, est_idx = ctx.saved_tensors
        near, interval, raw = ctx.consts
        g_cost = _topk_bwd_raw(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding,
                               near, interval, raw)
        return g_cost, None, None, None, None


class _DepthTopkNVS(torch.autograd.Function):
    """depth_topk plus the NVS-branch epilogue; opacity is the top-1 density and shares its
    gradient path, depth_scale is a constant of the intrinsics."""

    @staticmethod
    def forward(ctx, cost_out, near, interval, topk, ray_intr):
        cost_out, outs = _topk_fwd_raw(cost_out, near, interval, topk, 0, ray_intr)
        ctx.save_for_backward(cost_out, outs[4], ray_intr)
        ctx.consts = (float(near), float(interval))
        ctx.mark_non_differentiable(outs[4], outs[7])
        return outs

    @staticmethod
    def backward(ctx, g_prob, g_off, g_depth, g_dens, _g_idx, g_coding, g_opacity, _g_scale,
                 g_ray_depth, g_ray_coding):
        cost_out, est_idx, ray_intr = ctx.saved_tensors
        near, interval = ctx.consts
        if g_opacity is not None:                      # opacity == est_dens[:, 0]
            g_dens = torch.zeros_like(est_idx, dtype=torch.float32) if g_dens is None else g_dens.clone()
            g_dens[:, 0] += g_opacity
        g_cost = _topk_bwd_raw(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding,
                               near, interval, 0, ray_intr, g_ray_depth, g_ray_coding)
        return g_cost, None, None, None, None


def depth_topk(cost_out: torch.Tensor, near: float, interval: float, topk: int):
    """Fused mvsdet.py:470-482 + sample_depth_prob (:266-283) + compute_avg_depth
    (:298-317).  cost_out [V,2,D,H,W] -> (prob_volume [V,D,H,W], off_pred
    [V,D,H,W], est_depth [V,T,H,W], est_densities [V,T,H,W], est_idx int64
    [V,T,H,W], depth_coding [V,H,W])."""
    _check_cost("cost_out", cost_out)
    return _DepthTopk.apply(cost_out, near, interval, int(topk), 0)


def depth_topk_nvs(cost_out: torch.Tensor, near: float, interval: float, topk: int,
                   k_feat: torch.Tensor):
    """``depth_topk`` with the NVS-branch consumers computed in the same kernel (SURVEY.md 8f
    rank 3).  ``k_feat``: feature-level intrinsics [4,4] or [V,4,4].  Returns the six outputs of
    ``depth_topk`` followed by
      opacity [V,H,W]           max_d prob_volume                          mvsdet.py:579
      depth_scale [V,H,W]       compute_depth_scale[_MultiIntrin]          mvsdet.py:1158-1218
      est_ray_depth [V,T,H,W]   est_depth / (depth_scale + 1e-8)           mvsdet.py:494
      ray_depth_coding [V,H,W]  depth_coding / (depth_scale + 1e-8)        mvsdet.py:583
    (full, un-cropped maps; the caller crops / reshapes as it does est_depth)."""
    _check_cost("cost_out", cost_out)
    kmat = _ray_intr(k_feat, cost_out.shape[0])
    return _DepthTopkNVS.apply(cost_out, near, interval, int(topk), kmat)


def ray_depth_scale(k_feat: torch.Tensor, n_views: int, height: int, width: int) -> torch.Tensor:
    """compute_depth_scale / compute_depth_scale_MultiIntrin (mvsdet.py:1158-1218) alone:
    [4,4] or [V,4,4] feature-level intrinsics -> depth_scale [V,height,width]."""
    kmat = _ray_intr(k_feat, n_views)
    out = torch.empty((n_views, height, width), dtype=torch.float32, device=kmat.device)
    _lib.ray_depth_scale(kmat, out)
    return out


def rgb_downsample4(rgb: torch.Tensor, src_ids, height: int, width: int) -> torch.Tensor:
    """process_rgb_raw (mvsdet.py:319-333) for ratio 4: rgb [V,3,H,W] fp32 -> [1, n, height*width, 3]."""
    _need_cuda("rgb", rgb)
    if rgb.dim() != 4 or rgb.shape[1] != 3:
        raise ValueError("rgb must be [V,3,H,W]")
    rgb = rgb.float().contiguous()
    v = rgb.shape[0]
    ids = None
    n = v
    if src_ids is not None:
        ids = torch.as_tensor(src_ids, dtype=torch.int64).reshape(-1)
        if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= v):
            raise ValueError("src_id outside the image batch")
        ids = ids.to(rgb.device)
        n = ids.numel()
    out = torch.empty((1, n, height * width, 3), dtype=torch.float32, device=rgb.device)
    _lib.rgb_downsample4(rgb, ids, out, height=int(height), width=int(width))
    return out


def topk_hypotheses(prob_off: torch.Tensor, near: float, interval: float, topk: int):
    """Stand-alone form of ``depth_topk`` for inputs that are already
    probabilities / offsets: prob_off [V,2,D,H,W] = stack(prob_volume, off_pred).
    Same six outputs (the first two are pass-through copies)."""
    _check_cost("prob_off", prob_off)
    return _DepthTopk.apply(prob_off, near, interval, int(topk), 1)


# --------------------------------------------------------------------------
# back-projection
# --------------------------------------------------------------------------
def _zeros_strided_like(t: torch.Tensor) -> torch.Tensor:
    """zeros with exactly t's sizes AND strides (zeros_like falls back to
    contiguous strides for views with gaps, e.g. a row-cropped map)."""
    return torch.empty_strided(t.size(), t.stride(), dtype=t.dtype, device=t.device).zero_()


def _bp_fwd_raw(feat, points, projection, est_depth, est_dens, vs_z, h, w, mode, channels_first,
                out=None, count=None):
    """aggregating modes; -> (volume logical [C,N], count)"""
    c = feat.shape[1]
    n = points.numel() // 3
    dev = feat.device
    shape = (c, n) if channels_first else (n, c)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    elif tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous fp32 {shape} tensor (memory order of the volume)")
    if count is None:
        count = torch.empty((n,), dtype=torch.int32, device=dev)
    elif count.numel() != n or count.dtype != torch.int32 or not count.is_contiguous():
        raise ValueError("count must be a contiguous int32 [N] tensor")
    vol = out if channels_first else out.t()
    _lib.backproject_fwd(feat, points, projection, est_depth, est_dens, vol, vs_z=vs_z, mode=mode, height=h,
                         width=w, channels_first=channels_first, count=count)
    return vol, count


def _bp_bwd_raw(g_out, feat, points, projection, est_depth, est_dens, count, vs_z, h, w, mode,
                channels_first, acc=None):
    """back-projection + prob-norm backward; -> (dL/dfeat, dL/dest_dens); with ``acc``
    (FeatureGradSink accumulator) the feature gradient is RED-added there and None is returned"""
    g_out = g_out.float()
    g_mem = g_out.contiguous() if channels_first else g_out.t().contiguous().t()
    if acc is not None and acc.dtype == torch.int64:        # deterministic sink (MEAN mode only)
        if mode != BP_MEAN:
            raise ValueError("the deterministic backward is built for the mean aggregation only")
        g_pn_q = torch.zeros(est_dens.shape, dtype=torch.int64, device=feat.device)
        g_prob = _zeros_strided_like(est_dens)
        if g_pn_q.stride() != est_depth.stride():           # g_pn_q: contiguous [V,T,fh,fw]
            raise ValueError("the deterministic backward needs contiguous [V,T,H,W] hypotheses")
        _lib.backproject_bwd_det(g_mem, count, feat, points, projection, est_depth, est_dens, acc, g_pn_q,
                                 vs_z=vs_z, height=h, width=w, channels_first=channels_first)
        _lib.prob_norm_bwd(est_dens, fixed_to_float(g_pn_q), g_prob, height=h, width=w)
        return None, g_prob
    g_feat = acc if acc is not None else _zeros_nhwc(*feat.shape, torch.float32, feat.device)
    g_pn = _zeros_strided_like(est_dens)
    g_prob = _zeros_strided_like(est_dens)
    _lib.backproject_bwd(g_mem, feat, points, projection, est_depth, est_dens, g_feat, g_pn, vs_z=vs_z,
                         mode=mode, height=h, width=w, channels_first=channels_first,
                         count=count if mode == BP_MEAN else None)
    _lib.prob_norm_bwd(est_dens, g_pn, g_prob, height=h, width=w)
    return (None if acc is not None else g_feat.to(feat.dtype)), g_prob


class _BackprojectAggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, points, projection, est_depth, est_dens, vs_z, h, w, mode, channels_first,
                out=None, count=None, sink=None):
        external = out is not None or count is not None
        res, count = _bp_fwd_raw(feat, points, projection, est_depth, est_dens, vs_z, h, w, mode,
                                 channels_first, out, count)
        # Only MEAN mode needs the count in its backward (s_u = 1/(count+1e-8)); SUM mode saves
        # nothing that aliases caller-owned (reused, peer-mapped) buffers, so a later call that
        # overwrites them cannot corrupt this graph.
        # With a caller-owned count buffer (a slice of a batch tensor, a peer-mapped buffer) the
        # backward keeps its own copy (N int32 = 100 KB): a later writer cannot change s_u.
        keep = None
        if mode == BP_MEAN:
            keep = count.clone() if external else count
        ctx.save_for_backward(feat, points, projection, est_depth, est_dens, keep)
        ctx.consts = (float(vs_z), h, w, mode, channels_first)
        ctx.sink = sink
        ctx.mark_non_differentiable(count)
        return res, count

    @staticmethod
    def backward(ctx, g_out, _g_count):
        feat, points, projection, est_depth, est_dens, count = ctx.saved_tensors
        vs_z, h, w, mode, channels_first = ctx.consts
        acc = ctx.sink.get() if ctx.sink is not None else None
        g_feat, g_prob = _bp_bwd_raw(g_out, feat, points, projection, est_depth, est_dens, count,
                                     vs_z, h, w, mode, channels_first, acc)
        return g_feat, None, None, None, g_prob, None, None, None, None, None, None, None, None


def _check_hyp(name, t, v, fh, fw):
    _need_cuda(name, t)
    if t.dim() != 4 or t.shape[0] != v or t.shape[2] != fh or t.shape[3] != fw:
        raise ValueError(f"{name} must be [V,T,{fh},{fw}] (the full, un-cropped map)")
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32")


def _check_bp(feat, points, projection, est_depth, est_dens, height, width, grad_sink=None) -> None:
    _need_cuda("feat", feat)
    if not _is_nhwc(feat):
        raise ValueError("feat must be channels_last; use ops.pack_features")
    v, _, fh, fw = feat.shape
    _check_hyp("est_depth", est_depth, v, fh, fw)
    _check_hyp("est_dens", est_dens, v, fh, fw)
    _need_cuda("points", points)
    _need_cuda("projection", projection)
    if tuple(projection.shape) != (v, 3, 4):
        raise ValueError("projection must be [V,3,4]")
    if height > fh or width > fw:
        raise ValueError("crop exceeds the feature map")
    if grad_sink is not None and grad_sink.shape != tuple(feat.shape):
        raise ValueError("grad_sink belongs to a different feature tensor")


def backproject_aggregate(feat, points, projection, est_depth, est_dens, vs_z: float,
                          height: int, width: int, *, mode: str = "mean",
                          channels_first: bool = True, out: Optional[torch.Tensor] = None,
                          count_out: Optional[torch.Tensor] = None,
                          grad_sink: Optional[FeatureGradSink] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Fused backproject_Weigh (mvsdet.py:1372-1492) + aggregation (:511-515,
    :681-682).

    feat        channels-last [V,C,Hf,Wf] (only [:height,:width] is addressed)
    points      [3,nx,ny,nz] fp32;  projection [V,3,4] fp32
    est_depth, est_dens   [V,T,Hf,Wf] fp32 as ``depth_topk`` returns them
    mode        "mean" -> (volume_mean [C,N], count [N] int32)
                "sum"  -> (volume_sum  [C,N], count) partials for multi-GPU
    The result is logical [C,N]; with channels_first=False its memory is [N,C]
    (channels_last_3d once viewed as [C,nx,ny,nz]).  ``out`` / ``count_out``: write into
    caller-owned buffers (memory order of the volume: [C,N] or [N,C] contiguous) -- the
    view-sharded path lets the kernel write its partials straight into peer-mapped memory, the
    batched drop-in lets it write each scene's volume into its slot of the stacked batch tensor
    (mvsdet.py:695).  The buffers are overwritten in place without bumping autograd's version
    counters; the backward keeps a private copy of the count, so reusing the buffers later cannot
    corrupt this graph -- but the VALUES handed back are the buffers themselves."""
    _check_bp(feat, points, projection, est_depth, est_dens, height, width, grad_sink)
    if est_depth.stride() != est_dens.stride():
        est_depth, est_dens = est_depth.contiguous(), est_dens.contiguous()
    m = {"mean": BP_MEAN, "sum": BP_SUM}[mode]
    return _BackprojectAggregate.apply(feat, points.contiguous().float(),
                                       projection.contiguous().float(), est_depth, est_dens,
                                       float(vs_z), int(height), int(width), m, bool(channels_first),
                                       out, count_out, grad_sink)


def _per_view_hyp(t, h, w):
    """[V, h*w, 1, T] -> the [V,T,h,w] view the kernels take"""
    return t.view(t.shape[0], h, w, t.shape[3]).permute(0, 3, 1, 2)


class _BackprojectPerView(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, points, projection, depth, prob, vs_z, h, w):
        v, c = feat.shape[:2]
        n = points.numel() // 3
        dev = feat.device
        out = torch.zeros((v, n, c), dtype=torch.float32, device=dev)
        valid = torch.empty((v, n), dtype=torch.uint8, device=dev)
        _lib.backproject_fwd(feat, points, projection, _per_view_hyp(depth, h, w), _per_view_hyp(prob, h, w),
                             out.permute(0, 2, 1), vs_z=vs_z, mode=BP_PER_VIEW, height=h, width=w, valid=valid)
        ctx.save_for_backward(feat, points, projection, depth, prob)
        ctx.consts = (float(vs_z), h, w)
        valid = valid.bool()
        ctx.mark_non_differentiable(valid)
        return out.permute(0, 2, 1), valid

    @staticmethod
    def backward(ctx, g_out, _g_valid):
        feat, points, projection, depth, prob = ctx.saved_tensors
        vs_z, h, w = ctx.consts
        g_mem = g_out.float().permute(0, 2, 1).contiguous().permute(0, 2, 1)
        g_feat = _zeros_nhwc(*feat.shape, torch.float32, feat.device)
        g_pn = _zeros_strided_like(prob)
        g_prob = _zeros_strided_like(prob)
        prob_t = _per_view_hyp(prob, h, w)
        _lib.backproject_bwd(g_mem, feat, points, projection, _per_view_hyp(depth, h, w), prob_t, g_feat, g_pn,
                             vs_z=vs_z, mode=BP_PER_VIEW, height=h, width=w)
        _lib.prob_norm_bwd(prob_t, g_pn, g_prob, height=h, width=w)
        return g_feat.to(feat.dtype), None, None, None, g_prob, None, None, None


def backproject_per_view(feat, points, projection, depth, prob, vs_z: float, height: int,
                         width: int):
    """Un-aggregated back-projection with the reference's argument layout:
    ``depth`` / ``prob`` are [V, height*width, num_surface, T] (any strides with
    a common layout, mvsdet.py:484,495).  Returns (volume logical [V,C,N] with
    memory [V,N,C], valid bool [V,N])."""
    _need_cuda("feat", feat)
    if not _is_nhwc(feat):
        raise ValueError("feat must be channels_last; use ops.pack_features")
    v = feat.shape[0]
    if depth.shape != prob.shape or depth.dim() != 4 or depth.shape[0] != v \
            or depth.shape[1] != height * width:
        raise ValueError("depth and prob must be [V, h*w, num_surface, T]")
    t = depth.shape[2] * depth.shape[3]
    depth = depth.float()
    prob = prob.float()
    if depth.shape[2] != 1 or depth.stride() != prob.stride():
        depth = depth.reshape(v, height * width, 1, t).contiguous()
        prob = prob.reshape(v, height * width, 1, t).contiguous()
    return _BackprojectPerView.apply(feat, points.contiguous().float(),
                                     projection.contiguous().float(), depth, prob, float(vs_z),
                                     int(height), int(width))


def voxel_normalize(volume_sum: torch.Tensor, count: torch.Tensor) -> torch.Tensor:
    """sum / (count + 1e-8), zero where count == 0 (mvsdet.py:514-515) for a
    [C,N] (either memory order) partial sum after the multi-GPU all-reduce."""
    _need_cuda("volume_sum", volume_sum)
    channels_first = volume_sum.is_contiguous()
    if not channels_first and not volume_sum.t().is_contiguous():
        raise ValueError("volume_sum must be [C,N] contiguous or the transpose of [N,C]")
    out = torch.empty_like(volume_sum)          # same memory order
    _lib.voxel_normalize(volume_sum, count, out, channels_first=channels_first)
    return out


# --------------------------------------------------------------------------
# per-scene camera geometry (device prologue)
# --------------------------------------------------------------------------
def scene_setup(w2c: torch.Tensor, k_feat: torch.Tensor, ref_proj: torch.Tensor, inv_ref: torch.Tensor,
                k: int, ref_begin: int = 0, n_ref: Optional[int] = None):
    """mvsd_scene_setup: neighbour ids, homographies and projections of one scene in one launch
    (mvsdet.py:43-104, :249-264, :432-434, :1124-1156; module.py:116-118).  All inputs are DEVICE
    fp32 tensors: w2c [V,4,4], k_feat [4,4] or [V,4,4] (feature level), ref_proj = K_feat @ w2c and
    its inverse [V,4,4] (both from the host's ATen calls, see geometry.scene_geometry).
    -> (nbr_ids [n_ref,k] int32, hom [n_ref,k,12], projection [n_ref,3,4])."""
    for n, t in (("w2c", w2c), ("k_feat", k_feat), ("ref_proj", ref_proj), ("inv_ref", inv_ref)):
        _need_cuda(n, t)
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"{n} must be contiguous float32")
    v = w2c.shape[0]
    n_ref = v - ref_begin if n_ref is None else int(n_ref)
    dev = w2c.device
    out = torch.empty(n_ref * k * 13 + n_ref * 12, dtype=torch.float32, device=dev)
    nbr = out[:n_ref * k].view(torch.int32).view(n_ref, k)
    hom = out[n_ref * k:n_ref * k * 13].view(n_ref, k, 12)
    proj = out[n_ref * k * 13:].view(n_ref, 3, 4)
    _lib.scene_setup(w2c, k_feat, ref_proj, inv_ref, nbr, hom, proj, ref_begin=int(ref_begin))
    return nbr, hom, proj
