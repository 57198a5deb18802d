#!/usr/bin/env python
"""Plane-sweep backward: a variant selected by the test hook mvsd_set_tuning(5, x) against the
generic pixel kernel (5 = 1) on the same inputs, on several shapes (ragged tiles, ragged channels,
the benchmarked size), with CUDA-event timings at the benchmarked size.

    python tools/check_bwd_variant.py --variants 0 20 [--g-dtype f32]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from mvsdet_b200 import _lib, ops  # noqa: E402
from mvsdet_b200.hotpath import MVSDetHotPath  # noqa: E402
from mvsdet_b200.scene import SceneConfig, make_scene, tiny_config  # noqa: E402


def inputs(cfg, seed, g_dtype):
    dev = torch.device("cuda")
    scene = make_scene(cfg, seed=seed)
    mod = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk)
    geo = mod.geometry(scene["img_meta"], dev)
    feat = ops.pack_features(scene["feature"].to(dev), torch.bfloat16)
    v, c, h, w = feat.shape
    gen = torch.Generator(device="cuda").manual_seed(seed)
    g = torch.randn(v, cfg.num_depth, h, w, c, device=dev, generator=gen).to(g_dtype).permute(0, 4, 1, 2, 3)
    return feat, geo, g


def run(variant, feat, geo, g):
    old = _lib.set_tuning(5, variant)
    try:
        acc = torch.zeros(feat.shape, dtype=torch.float32, device=feat.device).contiguous(memory_format=torch.channels_last)
        _lib.plane_sweep_bwd(g, feat, geo.neighbor_ids, geo.hom, geo.depth_values, acc)
        torch.cuda.synchronize()
    finally:
        _lib.set_tuning(5, old)
    return acc


def timed(variant, feat, geo, g, reps=12):
    old = _lib.set_tuning(5, variant)
    acc = torch.zeros(feat.shape, dtype=torch.float32, device=feat.device).contiguous(memory_format=torch.channels_last)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=feat.device)
    ms = []
    try:
        for _ in range(reps):
            flush.zero_()
            acc.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.plane_sweep_bwd(g, feat, geo.neighbor_ids, geo.hom, geo.depth_values, acc)
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
    finally:
        _lib.set_tuning(5, old)
    return round(statistics.median(ms[2:]), 4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--variants", type=int, nargs="+", default=[0, 20])
    ap.add_argument("--g-dtype", default="f32")
    ap.add_argument("--no-small", action="store_true")
    a = ap.parse_args()
    gdt = torch.float32 if a.g_dtype == "f32" else torch.bfloat16
    out = {"lib": os.path.basename(os.environ.get("MVSDET_B200_LIB", "default")), "cases": []}
    cases = []
    if not a.no_small:
        for (h, w, c, v, d) in [(13, 21, 40, 4, 6), (9, 7, 256, 4, 5), (17, 40, 256, 5, 12), (16, 33, 132, 4, 7),
                                (12, 16, 128, 6, 9)]:
            cases.append((f"{h}x{w}x{c} V{v} D{d}", tiny_config(n_views=v, channels=c, num_depth=d,
                          img_shape=(4 * h - 1, 4 * w), pad_shape=(4 * h, 4 * w), ori_shape=(16 * h - 4, 16 * w))))
    cases.append(("benchmarked 60x80x256 V20 D12", SceneConfig(n_views=20)))
    for name, cfg in cases:
        feat, geo, g = inputs(cfg, 3, gdt)
        ref = run(1, feat, geo, g).double()
        rms = float(ref.pow(2).mean().sqrt())
        rec = {"case": name, "rms": rms}
        for var in a.variants:
            got = run(var, feat, geo, g).double()
            rec[f"v{var}_max_err_over_rms"] = float((got - ref).abs().max() / rms)
        out["cases"].append(rec)
        print(json.dumps(rec), flush=True)
    feat, geo, g = inputs(SceneConfig(n_views=20), 3, gdt)
    out["ms"] = {f"v{var}": timed(var, feat, geo, g) for var in a.variants}
    print(json.dumps(out["ms"]), flush=True)


if __name__ == "__main__":
    main()
