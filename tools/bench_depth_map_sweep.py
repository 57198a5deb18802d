#!/usr/bin/env python
"""Cost of per-pixel depth hypotheses in the fused variance sweep: CUDA-event times of the forward
and the fp32-RED backward, per-view planes [V,D] against per-pixel maps [V,D,H,W], at the benchmark
shape (V = 20, C = 256, D = 12, 60 x 80 feature maps, bf16 features, k = 2, fp32 variance).

Two per-pixel inputs:
  px_const   the per-view planes broadcast to [V,D,H,W] -- the same samples, so the difference to
             per_view is the cost of the variant itself;
  px_narrow  a narrow second sweep (+-10 % around a smooth per-pixel depth), the intended use.
Three scene buffer sets rotate (bf16 features 3 x 49 MB, variance / gradient volumes 1.18 GB each),
so the timed working set is far larger than the 126 MB L2.  The variants alternate within every
round; medians and min / max over the rounds are printed with the GPU's name and power limit.

    python tools/bench_depth_map_sweep.py [--rounds 9] [--iters 12] [--out result.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from mvsdet_b200 import _lib, ops  # noqa: E402
from mvsdet_b200.hotpath import MVSDetHotPath  # noqa: E402
from mvsdet_b200.scene import SceneConfig, make_scene  # noqa: E402

NBUF = 3


def _gpu_info():
    info = {"name": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info["power_limit, max_sm_clock"] = q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit, max_sm_clock"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--iters", type=int, default=12, help="launches per timed window (rotating buffer sets)")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool only measures on the GPU")
    dev = torch.device("cuda")
    cfg = SceneConfig(n_views=20)
    hf, wf = cfg.feat_hw
    mod = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        stride=cfg.stride, feature_dtype=torch.bfloat16)
    gen = torch.Generator().manual_seed(0)
    sets = []
    for b in range(NBUF):
        scene = make_scene(cfg, seed=b, with_grads=False)
        geo = mod.geometry(scene["img_meta"], dev)
        feat = ops.pack_features(scene["feature"].to(dev), torch.bfloat16)
        planes = geo.depth_values
        const = planes[:, :, None, None].expand(-1, -1, hf, wf).contiguous()
        center = cfg.near_far_range[0] + (cfg.near_far_range[1] - cfg.near_far_range[0]) * \
            (0.3 + 0.4 * torch.rand(cfg.n_views, 1, hf, wf, generator=gen))
        center = torch.nn.functional.avg_pool2d(center, 9, stride=1, padding=4, count_include_pad=False)
        steps = torch.linspace(-0.1, 0.1, cfg.num_depth).view(1, -1, 1, 1)
        narrow = (center * (1 + steps)).contiguous().to(dev)
        out = torch.empty((cfg.n_views, cfg.num_depth, hf, wf, cfg.channels), device=dev).permute(0, 4, 1, 2, 3)
        g = torch.randn(out.shape, generator=gen).to(dev).contiguous(memory_format=torch.channels_last_3d)
        g_feat = torch.zeros(feat.shape, device=dev).contiguous(memory_format=torch.channels_last)
        sets.append(dict(feat=feat, nbr=geo.neighbor_ids, hom=geo.hom, out=out, g=g, g_feat=g_feat,
                         depth=dict(per_view=planes, px_const=const, px_narrow=narrow)))
    variants = ("per_view", "px_const", "px_narrow")

    def launch(kind, variant, s):
        if kind == "fwd":
            _lib.plane_sweep_fwd(s["feat"], s["nbr"], s["hom"], s["depth"][variant], s["out"])
        else:
            _lib.plane_sweep_bwd(s["g"], s["feat"], s["nbr"], s["hom"], s["depth"][variant], s["g_feat"])

    def window(kind, variant):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.iters):
            launch(kind, variant, sets[i % NBUF])
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / a.iters

    for kind in ("fwd", "bwd"):                     # warm-up: module load, every shape and variant
        for variant in variants:
            window(kind, variant)
    times = {(k, v): [] for k in ("fwd", "bwd") for v in variants}
    for r in range(a.rounds):
        order = variants if r % 2 == 0 else variants[::-1]
        for kind in ("fwd", "bwd"):
            for variant in order:
                times[(kind, variant)].append(window(kind, variant))
    torch.cuda.synchronize()
    res = {"gpu": _gpu_info(),
           "shape": dict(V=cfg.n_views, C=cfg.channels, D=cfg.num_depth, H=hf, W=wf, k=2,
                         feature_dtype="bf16", variance_dtype="fp32"),
           "rounds": a.rounds, "launches_per_window": a.iters, "ms_per_call": {}}
    for (kind, variant), t in times.items():
        res["ms_per_call"][f"{kind}_{variant}"] = dict(median=round(statistics.median(t), 4),
                                                       min=round(min(t), 4), max=round(max(t), 4))
    for kind in ("fwd", "bwd"):
        base = statistics.median(times[(kind, "per_view")])
        for variant in variants[1:]:
            res["ms_per_call"][f"{kind}_{variant}"]["vs_per_view"] = round(
                statistics.median(times[(kind, variant)]) / base, 3)
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
