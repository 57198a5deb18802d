#!/usr/bin/env python
"""Cost of the deterministic group-correlation backward: CUDA-event times of
mvsd_plane_sweep_groupcorr_bwd (fp32 REDs; for bf16 features and k = 2 the run-merging kernel) against
mvsd_plane_sweep_groupcorr_bwd_det (64-bit fixed-point integer REDs, pixel-per-warp kernel), at
V = 20, C = 256, G = 8, D = 12, 60 x 80 feature maps, bf16 features, k = 2.

Two depth forms:
  per_view   the scene's planes [V,D];
  px_narrow  a narrow second sweep (+-10 % around a smooth per-pixel depth) [V,D,H,W].
Three scene buffer sets rotate (bf16 features 3 x 49 MB, cost-volume gradients 3 x 74 MB, fp32 and
int64 accumulators 3 x 98 MB and 3 x 197 MB), so the timed working set is far larger than the
126 MB L2.  The accumulators are not cleared between launches (the sums only grow; the time does
not depend on the values), and the fixed_to_float conversion is not part of the timed window.  The
two forms alternate within every round; medians and min / max over the rounds are printed with the
GPU's name and power limit.

    python tools/bench_groupcorr_det.py [--rounds 9] [--iters 12] [--out result.json]
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
GROUPS = 8


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
        k = geo.neighbor_ids.shape[1]
        center = cfg.near_far_range[0] + (cfg.near_far_range[1] - cfg.near_far_range[0]) * \
            (0.3 + 0.4 * torch.rand(cfg.n_views, 1, hf, wf, generator=gen))
        center = torch.nn.functional.avg_pool2d(center, 9, stride=1, padding=4, count_include_pad=False)
        steps = torch.linspace(-0.1, 0.1, cfg.num_depth).view(1, -1, 1, 1)
        narrow = (center * (1 + steps)).contiguous().to(dev)
        g = torch.randn((cfg.n_views, k, cfg.num_depth, hf, wf, GROUPS), generator=gen).to(dev)
        acc = dict(red=torch.zeros(feat.shape, device=dev).contiguous(memory_format=torch.channels_last),
                   det=torch.zeros(feat.shape, dtype=torch.int64, device=dev)
                   .contiguous(memory_format=torch.channels_last))
        sets.append(dict(feat=feat, nbr=geo.neighbor_ids, hom=geo.hom, g=g.permute(0, 1, 5, 2, 3, 4), acc=acc,
                         depth=dict(per_view=geo.depth_values, px_narrow=narrow)))
    forms = ("red", "det")
    depths = ("per_view", "px_narrow")
    bwd = dict(red=_lib.plane_sweep_groupcorr_bwd, det=_lib.plane_sweep_groupcorr_bwd_det)

    def window(form, depth):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.iters):
            s = sets[i % NBUF]
            bwd[form](s["g"], s["feat"], s["nbr"], s["hom"], s["depth"][depth], s["acc"][form])
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / a.iters

    for depth in depths:                            # warm-up: module load, every form and depth form
        for form in forms:
            window(form, depth)
    times = {(f, d): [] for d in depths for f in forms}
    for r in range(a.rounds):
        order = forms if r % 2 == 0 else forms[::-1]
        for depth in depths:
            for form in order:
                times[(form, depth)].append(window(form, depth))
    torch.cuda.synchronize()
    res = {"gpu": _gpu_info(),
           "shape": dict(V=cfg.n_views, C=cfg.channels, G=GROUPS, D=cfg.num_depth, H=hf, W=wf,
                         k=int(sets[0]["nbr"].shape[1]), feature_dtype="bf16"),
           "rounds": a.rounds, "launches_per_window": a.iters, "ms_per_call": {}}
    for (form, depth), t in times.items():
        res["ms_per_call"][f"bwd_{form}_{depth}"] = dict(median=round(statistics.median(t), 4),
                                                         min=round(min(t), 4), max=round(max(t), 4))
    for depth in depths:
        res["ms_per_call"][f"bwd_det_{depth}"]["vs_red"] = round(
            statistics.median(times[("det", depth)]) / statistics.median(times[("red", depth)]), 3)
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
