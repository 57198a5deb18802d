#!/usr/bin/env python
"""Cost of the deterministic backwards that torch.use_deterministic_algorithms(True) selects on the routes
outside MVSDetHotPath: CUDA-event times of each fp32-RED entry point against its fixed-point form
(64-bit integer REDs), at V = 20, C = 256, D = 12, 60 x 80 feature maps, bf16 features:

  homo_warp        mvsd_homo_warp_bwd            vs mvsd_homo_warp_bwd_det       (bf16 upstream gradient)
  bp_sum           mvsd_backproject_bwd (SUM)    vs mvsd_backproject_bwd_det_mode, channels-first volume
  bp_per_view      mvsd_backproject_bwd (PER_VIEW) vs mvsd_backproject_bwd_det_mode

The back-projection runs over the scene's voxel grid with the hypotheses of ``depth_topk`` on the scene's
cost volume.  Two buffer sets rotate so consecutive launches do not reuse the same inputs; accumulators
are not cleared between launches (the time does not depend on the values), and the fixed_to_float
conversion is not part of the timed window.  The two forms alternate within every round; medians and
min / max over the rounds are printed with the GPU's name and power limit.

    python tools/bench_det_routes.py [--rounds 9] [--iters 10] [--out result.json]
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
from mvsdet_b200._lib import BP_PER_VIEW, BP_SUM  # noqa: E402
from mvsdet_b200.hotpath import MVSDetHotPath  # noqa: E402
from mvsdet_b200.scene import SceneConfig, make_scene  # noqa: E402

NBUF = 2


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
    ap.add_argument("--iters", type=int, default=10, help="launches per timed window (rotating buffer sets)")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool only measures on the GPU")
    dev = torch.device("cuda")
    cfg = SceneConfig(n_views=20)
    hf, wf = cfg.feat_hw
    v, c, d = cfg.n_views, cfg.channels, cfg.num_depth
    mod = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        stride=cfg.stride, feature_dtype=torch.bfloat16)
    gen = torch.Generator().manual_seed(0)
    sets = []
    for b in range(NBUF):
        scene = make_scene(cfg, seed=b, with_grads=False)
        geo = mod.geometry(scene["img_meta"], dev)
        feat = ops.pack_features(scene["feature"].to(dev), torch.bfloat16)
        with torch.no_grad():
            _, _, est_depth, est_dens, _, _ = ops.depth_topk(scene["cost_out"].to(dev), cfg.near_far_range[0],
                                                             cfg.depth_interval, cfg.topk)
        n = geo.points.numel() // 3
        g_warp = torch.randn((v, d, hf, wf, c), generator=gen).to(dev, torch.bfloat16).permute(0, 4, 1, 2, 3)
        g_sum = torch.randn((c, n), generator=gen).to(dev)
        g_view = torch.randn((v, n, c), generator=gen).to(dev).permute(0, 2, 1)

        def acc(dtype):
            return torch.zeros(feat.shape, dtype=dtype, device=dev).contiguous(memory_format=torch.channels_last)
        sets.append(dict(feat=feat, hom=geo.hom[:, 0].contiguous(), depth=geo.depth_values, pts=geo.points,
                         proj=geo.projection, est_depth=est_depth, est_dens=est_dens, h=geo.height, w=geo.width,
                         g_warp=g_warp, g_sum=g_sum, g_view=g_view,
                         red=acc(torch.float32), det=acc(torch.int64),
                         pn_red=torch.zeros_like(est_dens), pn_det=torch.zeros_like(est_dens, dtype=torch.int64)))

    def launch(form, what, s):
        if what == "homo_warp":
            fn = _lib.homo_warp_bwd if form == "red" else _lib.homo_warp_bwd_det
            fn(s["g_warp"], s["hom"], s["depth"], s[form])
            return
        mode = BP_SUM if what == "bp_sum" else BP_PER_VIEW
        g = s["g_sum"] if mode == BP_SUM else s["g_view"]
        args = (g, s["feat"], s["pts"], s["proj"], s["est_depth"], s["est_dens"], s[form], s["pn_" + form])
        kw = dict(vs_z=cfg.voxel_size[2], mode=mode, height=s["h"], width=s["w"], channels_first=mode == BP_SUM)
        if form == "red":
            _lib.backproject_bwd(*args, **kw)
        else:
            _lib.backproject_bwd_det_mode(*args, **kw)

    def window(form, what):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.iters):
            launch(form, what, sets[i % NBUF])
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / a.iters

    forms = ("red", "det")
    whats = ("homo_warp", "bp_sum", "bp_per_view")
    for what in whats:                              # warm-up: module load, every form
        for form in forms:
            window(form, what)
    times = {(f, w): [] for w in whats for f in forms}
    for r in range(a.rounds):
        order = forms if r % 2 == 0 else forms[::-1]
        for what in whats:
            for form in order:
                times[(form, what)].append(window(form, what))
    torch.cuda.synchronize()
    res = {"gpu": _gpu_info(),
           "shape": dict(V=v, C=c, D=d, H=hf, W=wf, T=cfg.topk, N=int(sets[0]["pts"].numel() // 3),
                         feature_dtype="bf16"),
           "rounds": a.rounds, "launches_per_window": a.iters, "ms_per_call": {}}
    for (form, what), t in times.items():
        res["ms_per_call"][f"{what}_{form}"] = dict(median=round(statistics.median(t), 4), min=round(min(t), 4),
                                                    max=round(max(t), 4))
    for what in whats:
        res["ms_per_call"][f"{what}_det"]["vs_red"] = round(
            statistics.median(times[("det", what)]) / statistics.median(times[("red", what)]), 3)
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
