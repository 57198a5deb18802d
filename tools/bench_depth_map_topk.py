#!/usr/bin/env python
"""Cost of per-pixel depth hypotheses in the depth top-k epilogue: CUDA-event times of the forward
and the backward, per-view planes (near, interval) against per-pixel planes [V,D,H,W] with a
per-pixel spacing map [V,H,W], at V = 20, 60 x 80 maps, T = 3, for D = 12 (the coarse sweep) and
D = 8 (a narrow second sweep).  The per-pixel backward also writes dL/ddepth_values and
dL/dinterval_map.

Eight buffer sets rotate (cost volumes, outputs, gradients: ~15 MB per set at D = 12), so the timed
working set (~120 MB at D = 12) is not served from the 126 MB L2 the way one set would be.  The
variants alternate within every round; medians and min / max over the rounds are printed with the
GPU's name and power limit.

    python tools/bench_depth_map_topk.py [--rounds 9] [--iters 40] [--out result.json]
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

from bench_depth_map_sweep import _gpu_info  # noqa: E402
from mvsdet_b200 import _lib  # noqa: E402

NBUF = 8
V, H, W, T = 20, 60, 80, 3
NEAR, INTERVAL = 0.5, 0.3125


def _buffers(d, gen, dev):
    f32 = dict(dtype=torch.float32)
    cost = (torch.randn(V, 2, d, H, W, generator=gen) * 3).to(dev)
    planes = (0.5 + 4 * torch.rand(V, 1, H, W, generator=gen)) * (1 + torch.linspace(-0.05, 0.05, d).view(1, d, 1, 1))
    s = dict(cost=cost, depth=planes.contiguous().to(dev), spacing=(planes[:, 0] * 0.1 / (d - 1)).to(dev),
             prob=torch.empty(V, d, H, W, device=dev, **f32), off=torch.empty(V, d, H, W, device=dev, **f32),
             est_depth=torch.empty(V, T, H, W, device=dev, **f32), est_dens=torch.empty(V, T, H, W, device=dev, **f32),
             est_idx=torch.empty(V, T, H, W, device=dev, dtype=torch.int64),
             coding=torch.empty(V, H, W, device=dev, **f32), g_cost=torch.empty_like(cost),
             g_depth=torch.empty(V, d, H, W, device=dev, **f32), g_int=torch.empty(V, H, W, device=dev, **f32))
    s["grads"] = [torch.randn(x.shape, generator=gen).to(dev)
                  for x in (s["prob"], s["off"], s["est_depth"], s["est_dens"], s["coding"])]
    return s


def _launch(kind, variant, s):
    px = variant == "per_pixel"
    interval = s["spacing"] if px else INTERVAL
    dv = s["depth"] if px else None
    if kind == "fwd":
        _lib.depth_topk_fwd(s["cost"], s["prob"], s["off"], s["est_depth"], s["est_dens"], s["est_idx"], s["coding"],
                            near=NEAR, interval=interval, depth_values=dv)
    else:
        _lib.depth_topk_bwd(s["cost"], s["est_idx"], *s["grads"], s["g_cost"], near=NEAR, interval=interval,
                            depth_values=dv, g_depth_values=s["g_depth"] if px else None,
                            g_interval_map=s["g_int"] if px else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=9)
    ap.add_argument("--iters", type=int, default=40, help="launches per timed window (rotating buffer sets)")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool only measures on the GPU")
    dev = torch.device("cuda")
    gen = torch.Generator().manual_seed(0)
    variants = ("per_view", "per_pixel")
    res = {"gpu": _gpu_info(), "shape": dict(V=V, H=H, W=W, T=T), "rounds": a.rounds,
           "launches_per_window": a.iters, "ms_per_call": {}}
    for d in (12, 8):
        sets = [_buffers(d, gen, dev) for _ in range(NBUF)]
        for s in sets:                              # est_idx for the backward
            _launch("fwd", "per_pixel", s)

        def window(kind, variant):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(a.iters):
                _launch(kind, variant, sets[i % NBUF])
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1) / a.iters

        for kind in ("fwd", "bwd"):                 # warm-up: module load, every variant
            for variant in variants:
                window(kind, variant)
        times = {(k, v): [] for k in ("fwd", "bwd") for v in variants}
        for r in range(a.rounds):
            order = variants if r % 2 == 0 else variants[::-1]
            for kind in ("fwd", "bwd"):
                for variant in order:
                    times[(kind, variant)].append(window(kind, variant))
        for (kind, variant), t in times.items():
            res["ms_per_call"][f"D{d}_{kind}_{variant}"] = dict(
                median=round(statistics.median(t), 5), min=round(min(t), 5), max=round(max(t), 5))
        for kind in ("fwd", "bwd"):
            res["ms_per_call"][f"D{d}_{kind}_per_pixel"]["vs_per_view"] = round(
                statistics.median(times[(kind, "per_pixel")]) / statistics.median(times[(kind, "per_view")]), 3)
        del sets
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
