#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ by EXECUTING THE REFERENCE.

Needs a checkout of the original MVSDet project:

    MVSDET_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py

For every case below it builds a seeded synthetic scene
(mvsdet_b200.scene.make_scene), runs the reference's own functions -- sliced
verbatim out of that checkout by oracle/ref_loader.py -- through the glue
of MVSDet.extract_feat (projects/NeRF-Det/nerfdet/mvsdet.py:404-515, :681-682,
followed statement by statement, out-of-place training branch :458-459), and
stores inputs, every intermediate the parity tests compare, and the autograd
gradients in ``tests/golden/<case>.npz``.

CostRegNet_3DGS (mvs_models/mvsnet.py:73-113) sits between the stages and is
not part of the path (SURVEY.md 8a): its output is replaced by the scene's
seeded ``cost_out`` tensor, and the gradient that would reach the variance
volume by the scene's ``g_variance``.
"""
from __future__ import annotations

import dataclasses
import json
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from mvsdet_b200.scene import SceneConfig, make_scene, tiny_config  # noqa: E402
from oracle import ref_loader  # noqa: E402

CASES = {
    # name: (config, seed)
    "scannet_tiny": (tiny_config(n_views=5, channels=16), 1),
    "arkit_tiny": (tiny_config(n_views=4, channels=16, near_far_range=(0.5, 5.5),
                               per_view_intrinsics=True, num_depth=12), 2),
    "two_views": (tiny_config(n_views=2, channels=8, num_depth=4, topk=2), 3),
    "wide_c": (tiny_config(n_views=3, channels=132, num_depth=4, topk=1,
                           n_voxels=(8, 8, 4), img_shape=(31, 48), pad_shape=(32, 48),
                           ori_shape=(124, 192)), 4),
}


def reference_chain(ref, scene, training=True):
    cfg = scene["cfg"]
    meta = scene["img_meta"]
    feature = scene["feature"].clone().requires_grad_(True)
    cost_out = scene["cost_out"].clone().requires_grad_(True)
    self = ref_loader.make_self(cfg.near_far_range, cfg.num_depth)
    stride = cfg.stride

    # mvsdet.py:407-413
    projection = ref._compute_projection(meta, stride, None)
    points = ref.get_points(n_voxels=torch.tensor(cfg.n_voxels),
                            voxel_size=torch.tensor(cfg.voxel_size),
                            origin=torch.tensor(meta["lidar2img"]["origin"]))
    # :416-428
    height = meta["img_shape"][0] // stride
    width = meta["img_shape"][1] // stride
    src_w2c = torch.tensor(np.array(meta["lidar2img"]["extrinsic"]))
    src_intrinsic = torch.tensor(np.array(meta["lidar2img"]["intrinsic"]))
    intrin_list_flag = isinstance(meta["lidar2img"]["intrinsic"], list)
    ratio = meta["ori_shape"][0] / (meta["img_shape"][0] / stride)
    src_feat_intrinsic = src_intrinsic.clone()
    if not intrin_list_flag:
        src_feat_intrinsic[:2] /= ratio
    else:
        src_feat_intrinsic[:, :2] /= ratio
    # :432-434
    num_src = feature.shape[0]
    k = min(2, num_src - 1)
    src_c2w = src_w2c.inverse()
    neighbor_ids = ref.get_nearest_pose_ids(src_c2w, src_c2w, k, maskself=True)
    # :437-467
    num_depth = cfg.num_depth
    ref_volume = feature.unsqueeze(2).repeat(1, 1, num_depth, 1, 1)
    volume_sum = ref_volume
    volume_sq_sum = ref_volume ** 2
    nei_features = feature[neighbor_ids.view(-1)].view(num_src, k, *feature.shape[1:])
    nei_features = torch.unbind(nei_features, dim=1)
    ref_proj, nei_projs = ref.collect_proj(self, src_w2c, src_feat_intrinsic, neighbor_ids)
    depth_values = torch.tensor(self.depth_values).unsqueeze(0).repeat(num_src, 1)
    warped_all = []
    for nei_fea, nei_proj in zip(nei_features, nei_projs):
        warped_volume = ref.homo_warping(nei_fea, nei_proj, ref_proj, depth_values)
        warped_all.append(warped_volume.detach())
        volume_sum = volume_sum + warped_volume
        volume_sq_sum = volume_sq_sum + warped_volume ** 2
    volume_variance = volume_sq_sum.div_(k + 1).sub_(volume_sum.div_(k + 1).pow_(2))
    # :470-475 with the stand-in for the cost-regularisation net
    cost_reg, off_pred = torch.unbind(cost_out, dim=1)
    prob_volume = F.softmax(cost_reg, dim=1)
    off_pred = torch.sigmoid(off_pred)
    # :478-484,495
    est_depth_full, est_dens_full = ref.sample_depth_prob(self, prob_volume, off_pred, topk=cfg.topk)
    est_idx = prob_volume.topk(k=cfg.topk, dim=1)[1]
    est_depth = est_depth_full[:, :, :height, :width]
    est_densities = est_dens_full[:, :, :height, :width]
    depth_coding = ref.compute_avg_depth(self, prob_volume, off_pred)[:, :height, :width].unsqueeze(1)
    est_depth = est_depth.view(*est_depth.shape[:2], -1).transpose(2, 1).unsqueeze(2)
    est_densities = est_densities.reshape(*est_densities.shape[:2], -1).transpose(2, 1).unsqueeze(2)
    # :499-507
    volume, valid, gap, rmse = ref.backproject_Weigh(
        feature[:, :, :height, :width], points, projection, est_depth,
        list(cfg.voxel_size), est_densities, gt_depth=None, save_dir=None,
        img_meta=meta, depth_mean=depth_coding.squeeze(1))
    per_view_valid = valid
    # :511-515, :681-682
    volume_sum_v = volume.sum(dim=0)
    valid_cnt = valid.sum(dim=0)
    volume_mean = volume_sum_v / (valid_cnt + 1e-8)
    volume_mean[:, valid_cnt[0] == 0] = .0

    g_feat_var, = torch.autograd.grad(volume_variance, feature, scene["g_variance"],
                                      retain_graph=True)
    g_feat_vox, g_cost = torch.autograd.grad(volume_mean, (feature, cost_out),
                                             scene["g_volume_mean"], allow_unused=True)
    return dict(
        neighbor_ids=neighbor_ids, warped0=warped_all[0][:, :4],
        variance=volume_variance.detach(), prob_volume=prob_volume.detach(),
        off_pred=off_pred.detach(), est_depth=est_depth_full.detach(),
        est_densities=est_dens_full.detach(), est_idx=est_idx,
        depth_coding=depth_coding.detach(), projection=projection, points=points,
        valid=per_view_valid, volume_mean=volume_mean.detach(), count=valid_cnt,
        g_feature_from_variance=g_feat_var, g_feature_from_voxels=g_feat_vox,
        g_cost_out=g_cost, ref_proj=ref_proj, nei_projs=torch.stack(nei_projs, 0),
        gap=gap, rmse=rmse)


def reference_nvs(ref, scene, chain):
    """The NVS-branch consumers of the path (SURVEY.md 8f rank 3), by the reference's own code:
    compute_depth_scale[_MultiIntrin] (mvsdet.py:1158-1218 -> get_camera_params / lift), the
    ray-depth conversions of extract_feat (:488-494, :583), opacity (:579) and process_rgb_raw
    (:319-333).  get_camera_params / lift call ``.cuda()``: run under ref_loader.cpu_cuda_shim."""
    cfg = scene["cfg"]
    meta = scene["img_meta"]
    self = ref_loader.make_self(cfg.near_far_range, cfg.num_depth)
    stride = cfg.stride
    height, width = meta["img_shape"][0] // stride, meta["img_shape"][1] // stride
    v = cfg.n_views
    with ref_loader.cpu_cuda_shim():
        if isinstance(meta["lidar2img"]["intrinsic"], list):                       # :490-492
            scale = ref.compute_depth_scale_MultiIntrin(self, height, width, "cpu", meta, stride, v)
        else:                                                                      # :487-489
            scale = ref.compute_depth_scale(self, height, width, "cpu", meta, stride, v)
    cur_depth_scale = scale.squeeze(0)                                             # (V, h*w, 1)
    est_depth = chain["est_depth"][:, :, :height, :width]
    est_depth = est_depth.view(*est_depth.shape[:2], -1).transpose(2, 1).unsqueeze(2)   # :484
    est_ray_depth = est_depth / (cur_depth_scale.unsqueeze(-1).repeat(1, 1, 1, est_depth.shape[-1]) + 1e-8)
    depth_coding = chain["depth_coding"]                                           # (V,1,h,w)
    dc = depth_coding.view(*depth_coding.shape[:2], -1).unsqueeze(0).transpose(3, 2)     # :562
    ray_depth_coding = dc / (cur_depth_scale.unsqueeze(0) + 1e-8)                  # :583
    opacity = torch.max(chain["prob_volume"], dim=1)[0]                            # :579
    rgb = torch.rand(v, 3, cfg.pad_shape[0], cfg.pad_shape[1],
                     generator=torch.Generator().manual_seed(77))
    src_id = list(range(0, v, 2))
    rgb_raw = ref.process_rgb_raw(self, rgb, stride, height, width, src_id)
    return dict(depth_scale=scale, est_ray_depth=est_ray_depth, ray_depth_coding=ray_depth_coding,
                opacity=opacity, rgb=rgb, src_id=np.asarray(src_id, dtype=np.int64), rgb_raw=rgb_raw)


def main():
    ref = ref_loader.load()
    out_dir = os.path.dirname(os.path.abspath(__file__))
    only_nvs = "--only-nvs" in sys.argv
    for name in ("scannet_tiny", "arkit_tiny"):
        cfg, seed = CASES[name]
        scene = make_scene(cfg, seed)
        chain = reference_chain(ref, scene)
        nvs = reference_nvs(ref, scene, chain)
        path = os.path.join(out_dir, "nvs_" + name + ".npz")
        np.savez_compressed(path, **{k: (v.numpy() if torch.is_tensor(v) else v) for k, v in nvs.items()})
        print(f"nvs_{name}: wrote {path} ({os.path.getsize(path) / 1e6:.2f} MB)")
    if only_nvs:
        return
    for name, (cfg, seed) in CASES.items():
        scene = make_scene(cfg, seed)
        res = reference_chain(ref, scene)
        meta = scene["img_meta"]
        blob = {
            "in_feature": scene["feature"].numpy(),
            "in_cost_out": scene["cost_out"].numpy(),
            "in_g_volume_mean": scene["g_volume_mean"].numpy(),
            "in_g_variance": scene["g_variance"].numpy(),
            "in_w2c": np.stack(meta["lidar2img"]["extrinsic"]),
            "in_intrinsic": np.array(meta["lidar2img"]["intrinsic"]),
            "seed": np.int64(seed),
            "cfg_json": np.array(json.dumps(dataclasses.asdict(cfg))),
        }
        for key, val in res.items():
            blob["out_" + key] = val.numpy() if torch.is_tensor(val) else np.asarray(val)
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **blob)
        nvalid = int(res["valid"].sum())
        print(f"{name}: wrote {path} ({os.path.getsize(path) / 1e6:.2f} MB), "
              f"valid pairs {nvalid}, occupied voxels {int((res['count'] > 0).sum())}")


if __name__ == "__main__":
    main()
