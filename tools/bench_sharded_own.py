"""The view-sharded pipeline fed with every view's maps (``load``) against the same pipeline fed with each
rank's own views only (``load_own``: the halo maps are pulled from their owners over NVLink every forward,
after one more cross-rank barrier).  The two run on the same scene in the same process, alternating round by
round, and are checked to give the same bits:

* V=80 test-time scene (BASELINE.json configs[2]), forward with the p2p combine: one scene alone, and a
  stream of 8 scenes (``forward_stream``);
* the ARKitScenes-shaped V=40 scene (configs[3]), forward + backward.

    torchrun --nproc-per-node N tools/bench_sharded_own.py [--rounds 7] [--iters 20] [--out FILE]

Per rank: halo maps and bytes pulled per forward, pack bytes saved (the halo maps ``load`` packs from its fp32
copy), CUDA-event medians over the rounds (each round's time is the max over ranks); the card's name and power
limit.  One JSON line on rank 0 (also written to ``--out``)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mvsdet_b200 import sharded  # noqa: E402
from mvsdet_b200.hotpath import MVSDetHotPath  # noqa: E402
from mvsdet_b200.scene import ARKIT, SceneConfig, make_scene  # noqa: E402


def card(dev) -> dict:
    idx = dev.index or 0
    try:
        limit = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return {"name": torch.cuda.get_device_name(dev), "power_limit": limit}


def timed(fn, iters, dev) -> float:
    """ms per call, CUDA events on this rank, max over ranks"""
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def pair(hot, cfg, scene, dev, world, rank):
    """the same scene in a load-fed and a load_own-fed pipeline"""
    a = sharded.ShardedScenePipeline(hot, cfg, dev)
    a.load(scene["feature"], scene["cost_out"], scene["img_meta"])
    ids = a.view_ids
    b = sharded.ShardedScenePipeline(hot, cfg, dev)
    b.load_own(scene["feature"][ids], scene["cost_out"][ids], scene["img_meta"])
    hf, wf = cfg.feat_hw
    elems = cfg.channels * hf * wf
    n_halo = a.vl - a.vb
    packed = elems * torch.empty((), dtype=hot.feature_dtype).element_size()
    stats = {"rank": rank, "own_views": a.vb, "halo_views": n_halo, "halo_bytes_pulled": n_halo * packed,
             "pack_bytes_saved": n_halo * (4 * elems + packed)}
    return a, b, stats


def compare(name, fn_a, fn_b, rounds, iters, dev, warmup=3):
    for _ in range(warmup):
        fn_a()
        fn_b()
    ts = {"load": [], "load_own": []}
    for r in range(rounds):                              # alternate which goes first
        order = (("load", fn_a), ("load_own", fn_b)) if r % 2 == 0 else (("load_own", fn_b), ("load", fn_a))
        for key, fn in order:
            ts[key].append(timed(fn, iters, dev))
    med = {k: round(statistics.median(v), 4) for k, v in ts.items()}
    return {"leg": name, "ms_median_load": med["load"], "ms_median_load_own": med["load_own"],
            "ms_added_by_own_view_input": round(med["load_own"] - med["load"], 4),
            "ms_rounds": {k: [round(x, 4) for x in v] for k, v in ts.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--views", type=int, default=80)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    try:
        legs, per_rank = [], {}
        # configs[2]: V=80 forward, p2p combine
        cfg = SceneConfig(n_views=args.views)
        scene = make_scene(cfg, seed=7, with_grads=False)
        hot = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                            feature_dtype=torch.bfloat16)
        a, b, per_rank["v80"] = pair(hot, cfg, scene, dev, world, rank)
        ra, rb = a.forward("p2p"), b.forward("p2p")
        same = torch.equal(ra["volume_mean"], rb["volume_mean"]) and torch.equal(ra["count"], rb["count"])
        leg = compare(f"V={cfg.n_views} forward, one scene alone", lambda: a.forward("p2p"),
                      lambda: b.forward("p2p"), args.rounds, args.iters, dev)
        leg["bits_equal"] = bool(same)
        legs.append(leg)
        leg = compare(f"V={cfg.n_views} forward, stream of 8 scenes (ms per scene x 8)",
                      lambda: a.forward_stream("p2p", 8), lambda: b.forward_stream("p2p", 8),
                      args.rounds, max(1, args.iters // 4), dev)
        legs.append(leg)
        a.close()
        b.close()
        del a, b, scene
        torch.cuda.empty_cache()
        # configs[3]: ARKit-shaped V=40, forward + backward
        cfg = ARKIT
        scene = make_scene(cfg, seed=11)
        hot = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                            feature_dtype=torch.bfloat16)
        a, b, per_rank["arkit"] = pair(hot, cfg, scene, dev, world, rank)
        g_vol = scene["g_volume_mean"].to(dev)
        g_var = scene["g_variance"][a.view_ids].to(dev).contiguous(memory_format=torch.channels_last_3d)

        def step(p):
            p.forward("p2p")
            return p.backward(g_vol, g_var)
        ga = step(a)[0].clone()
        gb = step(b)[0]
        scale = float(ga.abs().max())
        leg = compare(f"ARKit-shaped V={cfg.n_views} forward + backward", lambda: step(a), lambda: step(b),
                      args.rounds, args.iters, dev)
        leg["g_feature_max_rel_diff"] = float((ga - gb).abs().max()) / max(scale, 1e-30)
        legs.append(leg)
        a.close()
        b.close()
        ranks = [None] * world
        dist.all_gather_object(ranks, {"rank": rank, "card": card(dev), **per_rank})
        if rank == 0:
            line = {"tool": "bench_sharded_own", "world": world, "legs": legs, "per_rank": ranks,
                    "what": "load = every view's fp32 maps resident, block + halo packed locally; load_own = own "
                            "views resident, halo maps pulled over NVLink after a cross-rank barrier; ms are "
                            "CUDA-event medians over alternating rounds, max over ranks per round"}
            text = json.dumps(line)
            print(text, flush=True)
            if args.out:
                os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
                with open(args.out, "w") as fh:
                    fh.write(text + "\n")
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
