#!/usr/bin/env python
"""Cost of the deterministic training step: CUDA-event times per scene, at V = 20, C = 256, D = 12, 60 x 80
feature maps, bf16 features, fp32 variance (the shape bench.py times), of

  step_default   ScenePipeline.step replayed from a CUDA graph (fp32-RED backward)
  step_det       ScenePipeline(deterministic=True).step replayed from a CUDA graph (fixed-point backward)
  eager_det      MVSDetHotPath(deterministic=True) forward + autograd backward, un-captured

on the same scene and upstream gradients.  The three alternate within every round (the order reverses every
other round); each window runs ``--iters`` scenes back to back.  Medians and min / max over the rounds are
printed with the GPU's name and power limit.

    python tools/bench_det_pipeline.py [--rounds 9] [--iters 20] [--out result.json]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

from bench_det_routes import _gpu_info  # noqa: E402
from mvsdet_b200.hotpath import MVSDetHotPath  # noqa: E402
from mvsdet_b200.pipeline import ScenePipeline  # noqa: E402
from mvsdet_b200.scene import SceneConfig, make_scene  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--iters", type=int, default=20, help="scenes per timed window")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool only measures on the GPU")
    dev = torch.device("cuda")
    cfg = SceneConfig(n_views=20)
    scene = make_scene(cfg, seed=0)
    hot = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        stride=cfg.stride, feature_dtype=torch.bfloat16, deterministic=True)
    geo = hot.geometry(scene["img_meta"], dev)
    graphs = {}
    for name, det in (("step_default", False), ("step_det", True)):
        pipe = ScenePipeline(cfg, dev, feature_dtype=torch.bfloat16, deterministic=det)
        pipe.set_geometry(geo)
        pipe.load_scene(scene)
        graphs[name] = (pipe, pipe.capture())
    feature0, cost0 = scene["feature"].to(dev), scene["cost_out"].to(dev)
    g_var, g_vol = scene["g_variance"].to(dev), scene["g_volume_mean"].to(dev)

    def eager():
        feat = feature0.detach().requires_grad_(True)
        cost = cost0.detach().requires_grad_(True)
        out = hot(feat, scene["img_meta"], cost_regularization=lambda var: cost, geometry=geo)
        torch.autograd.backward([out["variance"], out["volume_mean"]], [g_var, g_vol])

    def one(name):
        if name == "eager_det":
            eager()
        else:
            graphs[name][1].replay()

    def window(name):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.iters):
            one(name)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / a.iters

    names = ("step_default", "step_det", "eager_det")
    for name in names:                              # warm-up: module load, allocator, every form
        window(name)
    times = {n: [] for n in names}
    for r in range(a.rounds):
        for name in (names if r % 2 == 0 else names[::-1]):
            times[name].append(window(name))
    torch.cuda.synchronize()
    same = bool(torch.equal(graphs["step_det"][0].volume_mean, graphs["step_default"][0].volume_mean))
    res = {"gpu": _gpu_info(),
           "shape": dict(V=cfg.n_views, C=cfg.channels, D=cfg.num_depth, H=cfg.feat_hw[0], W=cfg.feat_hw[1],
                         T=cfg.topk, voxels=list(cfg.n_voxels), feature_dtype="bf16", variance_dtype="fp32"),
           "rounds": a.rounds, "scenes_per_window": a.iters, "ms_per_scene": {},
           "det_volume_mean_is_default_bits": same}
    for name, t in times.items():
        res["ms_per_scene"][name] = dict(median=round(statistics.median(t), 4), min=round(min(t), 4),
                                         max=round(max(t), 4))
    base = statistics.median(times["step_default"])
    for name in ("step_det", "eager_det"):
        res["ms_per_scene"][name]["vs_step_default"] = round(statistics.median(times[name]) / base, 3)
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
