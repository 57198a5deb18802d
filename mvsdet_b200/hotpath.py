"""Drop-in replacement for the per-scene block of ``MVSDet.extract_feat``
(projects/NeRF-Det/nerfdet/mvsdet.py:404-515 and :681-682).

``MVSDetHotPath`` takes what that block takes -- one scene's FPN features
[V,C,Hf,Wf], its ``img_meta`` and the cost-regularisation net -- and returns
what it produces (volume_mean, per-voxel valid count, the depth hypotheses and
probabilities the NVS branch consumes), but runs three fused kernels instead
of ~150 ATen launches with host syncs:

    features --pack--> channels-last (fp32 | bf16)
        plane_sweep_variance            mvsdet.py:439-467
        cost_regularization (cuDNN)     mvsdet.py:470   (not part of the path)
        depth_topk                      mvsdet.py:472-482, :266-283, :298-317
        backproject_aggregate           mvsdet.py:499-515, :681-682

Constructor arguments are the detector's own (mvsdet.py:125-155):
``near_far_range``, ``num_monocular_samples`` (gs_cfg), ``topk``, ``n_voxels``,
``voxel_size``.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional, Sequence

import torch
import torch.nn as nn

from . import library, ops
from .geometry import SceneGeometry, scene_geometry

__all__ = ["MVSDetHotPath"]


class MVSDetHotPath(nn.Module):
    def __init__(self, n_voxels: Sequence[int], voxel_size: Sequence[float],
                 near_far_range: Sequence[float], num_monocular_samples: int = 12, topk: int = 3,
                 cost_regularization: Optional[nn.Module] = None, stride: int = 4,
                 feature_dtype: torch.dtype = torch.float32,
                 variance_dtype: torch.dtype = torch.float32,
                 channels_first_volume: bool = True, num_neighbors: int = 2,
                 dispatcher_ops: bool = False, strict_ncdhw_variance: bool = False,
                 deterministic: bool = False, cost_volume: str = "variance", num_groups: int = 8):
        super().__init__()
        self.n_voxels = [int(n) for n in n_voxels]
        self.voxel_size = [float(s) for s in voxel_size]
        self.near_far_range = [float(x) for x in near_far_range]
        self.num_depth = int(num_monocular_samples)
        # mvsdet.py:222 -- python float, becomes fp32 inside the ops
        self.depth_interval = (self.near_far_range[1] - self.near_far_range[0]) / self.num_depth
        self.topk = int(topk)
        self.stride = int(stride)
        self.cost_regularization = cost_regularization
        self.feature_dtype = feature_dtype
        self.variance_dtype = variance_dtype
        self.channels_first_volume = channels_first_volume
        self.num_neighbors = num_neighbors      # k = min(2, V-1), mvsdet.py:432
        # True: go through the torch.library ops (torch.ops.mvsdet_b200.*, library.py) instead of
        # the autograd.Function layer -- same launchers, same kernels, traceable with fake tensors
        self.dispatcher_ops = bool(dispatcher_ops)
        # True: hand the cost-regularisation net the variance in the reference's strict NCDHW
        # contiguous memory (one extra transpose pass) instead of channels_last_3d
        self.strict_ncdhw_variance = bool(strict_ncdhw_variance)
        # True: bit-reproducible feature / cost gradients -- the backward kernels (variance or group-
        # correlation sweep, back-projection) accumulate in 64-bit fixed point with integer REDs
        # (order-independent) instead of fp32 REDs.  A scene's forward + backward with the variance
        # takes 7.3 ms instead of 1.2 ms (un-merged scatter, scalar 64-bit REDs): a reproducibility
        # mode, not the fast path; the forward is deterministic either way.
        self.deterministic = bool(deterministic)
        # "variance" (the reference, mvsdet.py:439-467) or "group_correlation": hand the cost-regularisation
        # net the k group-wise correlation volumes [V,k,num_groups,D,H,W] instead (SURVEY 8f rank 4; the
        # arithmetic of mvs_models/lss_fpn.py:485-506) -- for a lighter net than CostRegNet_3DGS
        if cost_volume not in ("variance", "group_correlation"):
            raise ValueError("cost_volume must be 'variance' or 'group_correlation'")
        self.cost_volume = cost_volume
        self.num_groups = int(num_groups)
        if self.deterministic and self.dispatcher_ops:
            raise ValueError("deterministic=True uses the shared gradient accumulator of the autograd.Function "
                             "layer; it is not available with dispatcher_ops=True")

    def geometry(self, img_meta: dict, device, view_slice=None, prologue=None) -> SceneGeometry:
        """Per-scene parameter block (mvsdet.py:407-450).  ``prologue``: "device" (default: two
        host ATen calls + one setup kernel) or "host" (the reference's own ops on the host)."""
        return scene_geometry(img_meta, stride=self.stride, near_far_range=self.near_far_range,
                              num_depth=self.num_depth, n_voxels=self.n_voxels,
                              voxel_size=self.voxel_size, num_neighbors=self.num_neighbors,
                              device=device, view_slice=view_slice, prologue=prologue)

    # -- stages ------------------------------------------------------------
    def variance(self, feat_cl: torch.Tensor, geo: SceneGeometry, ref_begin: int = 0,
                 grad_sink=None, depth_values: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The variance volume over the scene's neighbour ids and homographies.  ``depth_values``
        (default: the scene's planes ``geo.depth_values`` [V,D]) may be the caller's own planes, e.g.
        per-pixel hypotheses [V,D,Hf,Wf] for a second, narrow sweep around ``est_depth``; with the
        ``grad_sink`` of the first sweep both sweeps' feature gradients go to one accumulator."""
        depth = geo.depth_values if depth_values is None else depth_values
        if self.dispatcher_ops:
            if self.variance_dtype not in (torch.float32, torch.bfloat16):
                raise ValueError("variance_dtype must be float32 or bfloat16")
            return library.plane_sweep_variance(feat_cl, geo.neighbor_ids, geo.hom, depth,
                                                self.variance_dtype == torch.bfloat16, ref_begin)
        return ops.plane_sweep_variance(feat_cl, geo.neighbor_ids, geo.hom, depth,
                                        out_dtype=self.variance_dtype, ref_begin=ref_begin,
                                        grad_sink=grad_sink)

    def hypotheses(self, cost_out: torch.Tensor, k_feat: Optional[torch.Tensor] = None,
                   depth_values: Optional[torch.Tensor] = None, interval=None):
        """(prob_volume, off_pred, est_depth, est_densities, est_idx, depth_coding); with the
        feature-level intrinsics ``k_feat`` also the NVS-branch outputs (opacity, depth_scale,
        est_ray_depth, ray_depth_coding) from the same kernel (mvsdet.py:494, :579, :583).
        ``depth_values`` [V,D,Hf,Wf]: the per-pixel planes the cost volume was swept over (a second
        sweep, ``variance(..., depth_values=)``), with ``interval`` their offset scale -- a float or
        an [V,Hf,Wf] map; the scene's interval is no default for them.  Both may carry gradients."""
        if depth_values is not None:
            if interval is None:
                raise ValueError("per-pixel depth_values need their own interval (a float or an [V,H,W] map)")
            if k_feat is not None:
                return ops.depth_topk_nvs(cost_out, 0.0, interval, self.topk, k_feat, depth_values=depth_values)
            if self.dispatcher_ops:
                if isinstance(interval, torch.Tensor):
                    return library.depth_topk_px(cost_out, depth_values, interval, 0.0, self.topk)
                return library.depth_topk_px(cost_out, depth_values, None, float(interval), self.topk)
            return ops.depth_topk(cost_out, 0.0, interval, self.topk, depth_values=depth_values)
        if k_feat is not None:
            return ops.depth_topk_nvs(cost_out, self.near_far_range[0], self.depth_interval, self.topk, k_feat)
        if self.dispatcher_ops:
            return library.depth_topk(cost_out, self.near_far_range[0], self.depth_interval, self.topk)
        return ops.depth_topk(cost_out, self.near_far_range[0], self.depth_interval, self.topk)

    def voxels(self, feat_cl, geo: SceneGeometry, est_depth, est_dens, mode: str = "mean", grad_sink=None,
               out=None, count_out=None):
        if self.dispatcher_ops and out is None:
            return library.backproject_aggregate(feat_cl, geo.points, geo.projection, est_depth, est_dens,
                                                 self.voxel_size[2], geo.height, geo.width,
                                                 {"mean": False, "sum": True}[mode],
                                                 self.channels_first_volume)
        return ops.backproject_aggregate(feat_cl, geo.points, geo.projection, est_depth, est_dens,
                                         self.voxel_size[2], geo.height, geo.width, mode=mode,
                                         channels_first=self.channels_first_volume, grad_sink=grad_sink,
                                         out=out, count_out=count_out)

    # -- the whole block ---------------------------------------------------
    def forward(self, feature: torch.Tensor, img_meta: dict,
                cost_regularization: Optional[Callable] = None,
                geometry: Optional[SceneGeometry] = None, nvs: bool = False,
                volume_out: Optional[torch.Tensor] = None,
                count_out: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """feature [V,C,Hf,Wf] (fp32 NCHW as the reference's FPN gives it, or
        already channels_last / bf16).  Returns a dict with
          volume_mean [C,nx,ny,nz], valid [1,nx,ny,nz] (float count, as
          extract_feat returns it, mvsdet.py:698), count int32 [N],
          variance (the cost volume handed to the net: the variance, or with
          ``cost_volume="group_correlation"`` the [V,k,G,D,Hf,Wf] correlation volumes),
          prob_volume, off_pred, est_depth, est_densities, est_idx, opacity,
          depth_coding [V,1,h,w] -- the reference's intermediates; ``nvs=True`` adds
          depth_scale [V,h*w,1], est_ray_depth [V,h*w,1,T] and ray_depth_coding [V,h*w,1]
          in the reference's layouts (mvsdet.py:488-494, :583), from the top-k kernel."""
        cost_net = cost_regularization or self.cost_regularization
        if cost_net is None:
            raise ValueError("a cost_regularization callable is required (mvsdet.py:470)")
        geo = geometry or self.geometry(img_meta, feature.device)
        # one fp32 gradient accumulator shared by the two consumers of the packed features
        # (ops.FeatureGradSink); the torch.library route keeps plain functional autograd
        feat_cl, sink = ops.pack_features(feature, self.feature_dtype, sink=True, deterministic=self.deterministic)
        if self.dispatcher_ops:
            sink = None
        if self.cost_volume == "group_correlation":
            if self.dispatcher_ops:
                from . import library
                variance = library.plane_sweep_group_correlation(feat_cl, geo.neighbor_ids, geo.hom,
                                                                 geo.depth_values, self.num_groups, 0)
            else:
                variance = ops.plane_sweep_group_correlation(feat_cl, geo.neighbor_ids, geo.hom, geo.depth_values,
                                                             self.num_groups, grad_sink=sink)
        else:
            variance = self.variance(feat_cl, geo, grad_sink=sink)
            if self.strict_ncdhw_variance:
                variance = ops.volume_to_ncdhw(variance)
        cost_out = cost_net(variance)
        hyp = self.hypotheses(cost_out, geo.k_feat if nvs else None)
        prob, off, est_depth, est_dens, est_idx, coding = hyp[:6]
        vol, count = self.voxels(feat_cl, geo, est_depth, est_dens, grad_sink=sink, out=volume_out,
                                 count_out=count_out)
        nx, ny, nz = self.n_voxels
        c = feat_cl.shape[1]
        volume_mean = vol.view(c, nx, ny, nz) if vol.is_contiguous() else vol.unflatten(1, (nx, ny, nz))
        out = dict(volume_mean=volume_mean, valid=count.view(1, nx, ny, nz).float(), count=count,
                   variance=variance, cost_out=cost_out, prob_volume=prob, off_pred=off, est_depth=est_depth,
                   est_densities=est_dens, est_idx=est_idx,
                   # NVS branch: opacity = max_d prob_volume (mvsdet.py:579) is the top-1
                   # hypothesis probability, bit for bit
                   opacity=est_dens[:, 0],
                   depth_coding=coding[:, :geo.height, :geo.width].unsqueeze(1),
                   # int32 on the device (device prologue); .long() gives the reference's dtype
                   neighbor_ids=geo.neighbor_ids)
        if nvs:
            v, h, w = est_depth.shape[0], geo.height, geo.width
            opacity, scale, ray_depth, ray_coding = hyp[6:]
            out["opacity"] = opacity
            out["depth_scale"] = scale[:, :h, :w].reshape(v, h * w, 1)
            out["est_ray_depth"] = ray_depth[:, :, :h, :w].reshape(v, self.topk, h * w).transpose(2, 1).unsqueeze(2)
            out["ray_depth_coding"] = ray_coding[:, :h, :w].reshape(v, h * w, 1)
        return out

    def forward_batch(self, features, img_metas, cost_regularization: Optional[Callable] = None,
                      nvs: bool = False):
        """The scene loop of ``extract_feat`` (mvsdet.py:404-698) up to the neck: every scene's
        volume is written by the back-projection kernel straight into its slot of the stacked
        batch tensor (the reference appends to a list and ``torch.stack``s, :684-696 -- two extra
        passes over 26 MB per scene).  -> (x [B,C,nx,ny,nz] -- the input of ``neck_3d`` --,
        valids [B,1,nx,ny,nz] float counts as ``extract_feat`` returns them (:698), per-scene dicts)."""
        if len(features) != len(img_metas) or not len(features):
            raise ValueError("one img_meta per scene")
        if not self.channels_first_volume:
            raise ValueError("forward_batch stacks [C,nx,ny,nz] volumes: channels_first_volume=True")
        b = len(features)
        c = features[0].shape[1]
        nx, ny, nz = self.n_voxels
        dev = features[0].device
        x = torch.empty((b, c, nx * ny * nz), dtype=torch.float32, device=dev)
        counts = torch.empty((b, nx * ny * nz), dtype=torch.int32, device=dev)
        outs, vols = [], []
        for i, (feature, meta) in enumerate(zip(features, img_metas)):
            out = self.forward(feature, meta, cost_regularization, nvs=nvs, volume_out=x[i], count_out=counts[i])
            outs.append(out)
            vols.append(out["volume_mean"])
        xb = x.view(b, c, nx, ny, nz)
        if any(v.requires_grad for v in vols):
            # the kernels already wrote every scene into x: wire the scenes' autograd nodes behind
            # the batch tensor without copying (the backward hands each scene its slice of the gradient)
            xb = _StackFilled.apply(xb, *vols)
        return xb, counts.view(b, 1, nx, ny, nz).float(), outs


class _StackFilled(torch.autograd.Function):
    """``torch.stack(vols)`` when ``filled`` already holds the stacked values (each vols[i] IS
    filled[i]): forward returns the filled tensor, backward returns the per-scene gradient slices."""

    @staticmethod
    def forward(ctx, filled, *vols):
        ctx.shapes = [tuple(v.shape) for v in vols]
        return filled.detach()

    @staticmethod
    def backward(ctx, g):
        return (None,) + tuple(g[i].reshape(shape) for i, shape in enumerate(ctx.shapes))
