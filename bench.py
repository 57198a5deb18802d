#!/usr/bin/env python
"""bench.py -- scenes/s of the MVSDet plane-sweep + depth-top-k + voxel
back-projection path (forward + backward) on B200, with the HBM roofline of the
dominant kernel and the CPU baseline beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): one synthetic ScanNet-shaped scene per step
-- V=20 views, 320x240 images -> 60x80 FPN features x 256 channels, D=12 depth
planes, k=2 neighbours, T=3 hypotheses, 40x40x16 voxels -- forward+backward,
bf16 features / fp32 accumulation, fp32 variance volume.  The cost-regularisation
3-D U-Net that sits between the stages is not part of the path (SURVEY.md 8a):
its output and the gradient it returns to the variance volume are synthetic
inputs of the step.  A "step" = ScenePipeline.step(): pack, sweep fwd, top-k
fwd, voxels fwd, voxels bwd, pn bwd, top-k bwd, sweep bwd, unpack.

N > 1 (torchrun): scenes are independent, so every rank runs its own scenes
(weak scaling, no data-path collective); the timed region is bracketed by a
barrier + synchronize and the slowest rank's device time is used.

`--impl reference` times the CPU oracle (the restatement of the reference's
PyTorch path, oracle/mvsdet_oracle.py) on the host cores for the same metric.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "scenes/sec for plane-sweep+voxel backproj fwd+bwd; % of HBM roofline"
UNIT = "scenes/s"
NBUF = 3   # rotating scene buffer sets: a set is re-read after >= 2 other steps (> 4 GB of traffic)


def _dist_env():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bind_to_gpu_numa_node(gpu_index: int):
    """Pin this rank's threads (and therefore the pages of its pinned host buffers, which are
    first-touched by the allocating thread) to the NUMA node the GPU hangs off: with 8 ranks the
    host <-> device copies of the e2e leg otherwise cross the socket interconnect.  Best effort:
    returns the node id, or None when sysfs / nvidia-smi do not say."""
    try:
        bdf = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if not bdf:
            return None
        if len(bdf.split(":")[0]) == 8:                    # 00000000:1B:00.0 -> 0000:1b:00.0
            bdf = bdf[4:]
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as fh:
            node = int(fh.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:                                      # noqa: BLE001
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, period_ms: int = 100):
        self.gpu = gpu_index
        self.samples = []          # (t, sm, max, [reasons])
        self.proc = None
        self.period_ms = period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu), "-lms", str(self.period_ms)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        threading.Thread(target=self._reader, daemon=True).start()

    def _reader(self):
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm, mx = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            reasons = [n for n, p in zip(names, parts[4:8]) if p.lower().startswith("active")]
            self.samples.append((time.time(), sm, mx, reasons))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0: float, t1: float):
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = sorted({r for s in inside for r in s[3]})
        return {"sm_mhz": statistics.median(s[1] for s in inside),
                "sm_max_mhz": max(s[2] for s in inside), "reasons": reasons,
                "samples": len(inside)}


# ---------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle on the host cores
# ---------------------------------------------------------------------------
def cpu_reference_step(scene, n_sample_views: int):
    """fwd+bwd of the oracle restricted to the first ``n_sample_views``
    reference views (plane sweep, top-k and back-projection all scale linearly
    in the number of reference views; neighbours are still drawn from all V)."""
    from oracle import mvsdet_oracle as O
    cfg = scene["cfg"]
    feature = scene["feature"].clone().requires_grad_(True)
    vs = n_sample_views
    cost_out = scene["cost_out"][:vs].clone().requires_grad_(True)
    res = O.hot_path(feature, scene["img_meta"], lambda var: cost_out,
                     near_far_range=cfg.near_far_range, num_depth=cfg.num_depth, topk=cfg.topk,
                     n_voxels=cfg.n_voxels, voxel_size=cfg.voxel_size, stride=cfg.stride,
                     training=True, view_subset=vs)
    torch.autograd.backward([res["variance"], res["volume_mean"]],
                            [scene["g_variance"][:vs], scene["g_volume_mean"]])
    return feature.grad, cost_out.grad


CPU_SAMPLE_VIEWS = 4          # reference views swept per CPU step: FIXED (round-1 picked 1, 2 or 4 by a
                              # wall-clock budget, which moved the number by 1.9x between runs)


def time_cpu_reference(cfg, steps: int, warmup: int, budget_s=None):
    """The oracle on the host cores: always ``CPU_SAMPLE_VIEWS`` of the scene's reference views per
    step (every stage of the path is linear in the number of reference views; the neighbours are
    still drawn from all V), ``warmup`` untimed + ``steps`` timed steps, MEDIAN step time, scaled to
    a scene.  With ``budget_s`` the number of timed steps is bounded by it (never below 3)."""
    from mvsdet_b200.scene import make_scene
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    scene = make_scene(cfg, seed=0)
    v = cfg.n_views
    vs = min(CPU_SAMPLE_VIEWS, v)
    t0 = time.perf_counter()
    cpu_reference_step(scene, vs)                      # first warm-up step, also the calibration
    t_first = time.perf_counter() - t0
    for _ in range(max(0, warmup - 1)):
        cpu_reference_step(scene, vs)
    n_timed = steps if budget_s is None else max(3, min(max(1, steps), int(budget_s / max(t_first, 1e-3))))
    times = []
    for _ in range(n_timed):
        t0 = time.perf_counter()
        cpu_reference_step(scene, vs)
        times.append(time.perf_counter() - t0)
    t_step = statistics.median(times)
    scenes_per_s = 1.0 / (t_step * v / vs)
    sample = (f"{vs} of {v} reference views per step, fixed (plane sweep + top-k + back-projection "
              f"fwd+bwd of the oracle, fp32, torch {torch.__version__} CPU, {threads} threads), scaled "
              f"x{v / vs:g} to a scene; {len(times)} timed steps, median {t_step:.3f} s/step "
              f"(min {min(times):.3f}, max {max(times):.3f})")
    return scenes_per_s, t_step, threads, sample, len(times)


def run_reference_arm(args, cfg, cfg_json):
    rank, local, world = _dist_env()
    if rank != 0:
        return
    val, t_step, threads, sample, nsteps = time_cpu_reference(cfg, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": nsteps, "warmup": args.warmup, "ms_per_step": t_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg_json,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# own arm
# ---------------------------------------------------------------------------
SURVEY_PATH_MB = 3034.0     # SURVEY.md 8(d): algorithmic bytes of the path per scene, fwd+bwd, fp32 sizes


def _build_pipes(cfg, dev, feat_dtype, mod, rank, capture=True, variance_dtype=torch.float32):
    from mvsdet_b200.pipeline import ScenePipeline
    from mvsdet_b200.scene import make_scene
    pipes, graphs, first_scene = [], [], None
    for b in range(NBUF):
        scene = make_scene(cfg, seed=1000 * rank + b)
        pipe = ScenePipeline(cfg, dev, feature_dtype=feat_dtype, variance_dtype=variance_dtype)
        pipe.set_geometry(mod.geometry(scene["img_meta"], dev))
        pipe.load_scene(scene)
        pipes.append(pipe)
        if b == 0:
            first_scene = scene
    torch.cuda.synchronize()
    if capture:
        graphs = [p.capture() for p in pipes]
    return pipes, graphs, first_scene


def _time_steps(step_fn, steps, warmup, barrier):
    """W untimed + K timed steps on the current stream, CUDA events, barrier + synchronize on both
    sides; returns (ms_total, wall0, wall1)."""
    for i in range(warmup):
        step_fn(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.time()
    e0.record()
    for i in range(steps):
        step_fn(i)
    e1.record()
    barrier()
    return e0.elapsed_time(e1), wall0, time.time()


DUMP_BUDGET = 64 << 20       # bytes: all dumped files together


def snapshot_outputs(pipe):
    """What ``pipe``'s last step handed its caller, in the caller's logical layouts, as float32 host
    arrays: the variance volume [V,C,D,Hf,Wf] (input of the cost-regularisation net), the top-k
    products, volume_mean [C,nx,ny,nz], count [nx,ny,nz], g_feature [V,C,Hf,Wf] and g_cost_out.
    Each output gets an equal share of DUMP_BUDGET; a larger one is reduced to the elements at
    fixed, seeded positions of its logical (row-major) index, so two builds sample the same ones."""
    import numpy as np
    cfg = pipe.cfg
    outs = {
        "variance": pipe.variance.permute(0, 4, 1, 2, 3),
        "prob_volume": pipe.prob_volume, "off_pred": pipe.off_pred,
        "est_depth": pipe.est_depth, "est_densities": pipe.est_dens, "est_idx": pipe.est_idx,
        "depth_coding": pipe.depth_coding,
        "volume_mean": pipe.volume_mean.view(cfg.channels, *cfg.n_voxels),
        "count": pipe.count.view(*cfg.n_voxels),
        "g_feature": pipe.g_feature, "g_cost_out": pipe.g_cost_out,
    }
    cap = DUMP_BUDGET // (4 * len(outs))             # float32 elements per output
    arrays, info = {}, {}
    for seed, (name, t) in enumerate(outs.items()):
        if t.numel() <= cap:
            arrays[name] = t.float().cpu().numpy()
            info[name] = {"shape": list(t.shape)}
            continue
        flat = np.sort(np.random.default_rng(seed).choice(t.numel(), cap, replace=False))
        idx = torch.from_numpy(np.stack(np.unravel_index(flat, tuple(t.shape)))).to(t.device)
        arrays[name] = t[tuple(idx)].float().cpu().numpy()
        info[name] = {"shape": list(t.shape), "sampled": cap,
                      "sample": f"np.sort(np.random.default_rng({seed}).choice({t.numel()}, {cap}, "
                                "replace=False)) of the row-major index"}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BUDGET:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_BUDGET}-byte budget")
    return arrays, info


def write_outputs(directory, arrays):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def _kernel_table(pipes, ksteps):
    timers = {}
    for i in range(ksteps):
        pipes[i % NBUF].step(timers)
    torch.cuda.synchronize()
    abytes = pipes[0].algorithmic_bytes()
    kernels = {}
    for name, evs in timers.items():
        ms = statistics.mean(a.elapsed_time(b) for a, b in evs)
        kernels[name] = {"ms": round(ms, 5), "algorithmic_mb": round(abytes[name] / 1e6, 2),
                         "gbs": round(abytes[name] / (ms * 1e-3) / 1e9, 1)}
    return kernels, abytes


def time_eager_gpu(cfg, scene, dev, reps=3):
    """SURVEY.md 8d 'eager-GPU comparison': the reference's PyTorch path (the oracle's ATen ops on
    CUDA tensors, fp32, ~150 eager launches with host syncs) on the SAME GPU and scene, fwd+bwd."""
    from oracle import mvsdet_oracle as O
    feature0 = scene["feature"].to(dev)
    cost0 = scene["cost_out"].to(dev)
    g_var = scene["g_variance"].to(dev)
    g_vol = scene["g_volume_mean"].to(dev)

    def step():
        feature = feature0.clone().requires_grad_(True)
        cost_out = cost0.clone().requires_grad_(True)
        res = O.hot_path(feature, scene["img_meta"], lambda var: cost_out,
                         near_far_range=cfg.near_far_range, num_depth=cfg.num_depth, topk=cfg.topk,
                         n_voxels=cfg.n_voxels, voxel_size=cfg.voxel_size, stride=cfg.stride, training=True)
        torch.autograd.backward([res["variance"], res["volume_mean"]], [g_var, g_vol])

    step()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    out = {"value": 1e3 / ms, "unit": UNIT, "ms_per_scene": round(ms, 3), "steps": reps,
           "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 1e9, 2),
           "what": "reference PyTorch path (oracle ops) on CUDA tensors, fp32, eager ATen kernels, same GPU"}
    del feature0, cost0, g_var, g_vol
    torch.cuda.empty_cache()
    return out


def time_group_correlation(pipe, cfg, peak, groups=8, reps=20):
    """mvsd_plane_sweep_groupcorr_fwd / _bwd on the benchmark scene's packed features (G = 8 groups of
    32 channels): CUDA-event means, an L2 flush between repetitions."""
    from mvsdet_b200 import _lib
    dev = pipe.feat_cl.device
    geo = pipe.geo
    v, d, k = cfg.n_views, cfg.num_depth, geo.k
    hf, wf = cfg.feat_hw
    c = cfg.channels
    out = torch.empty((v, k, d, hf, wf, groups), dtype=torch.float32, device=dev)
    g_out = torch.randn_like(out)
    acc = torch.zeros((v, hf, wf, c), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    fdt = _lib.BF16 if pipe.feat_cl.dtype == torch.bfloat16 else _lib.F32

    def fwd():
        _lib.call("mvsd_plane_sweep_groupcorr_fwd", pipe.feat_cl.data_ptr(), fdt, geo.neighbor_ids.data_ptr(),
                  geo.hom.data_ptr(), geo.depth_values.data_ptr(), out.data_ptr(), v, c, d, hf, wf, k, groups,
                  0, v, st)

    def bwd():
        _lib.call("mvsd_plane_sweep_groupcorr_bwd", g_out.data_ptr(), pipe.feat_cl.data_ptr(), fdt,
                  geo.neighbor_ids.data_ptr(), geo.hom.data_ptr(), geo.depth_values.data_ptr(), acc.data_ptr(),
                  v, c, d, hf, wf, k, groups, 0, v, st)

    res = {}
    for name, fn in (("fwd", fwd), ("bwd", bwd)):
        ms = []
        for _ in range(reps + 3):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        res[name] = statistics.mean(ms[3:])
    feat_b = pipe.feat_cl.numel() * pipe.feat_cl.element_size()
    fwd_b = feat_b + out.numel() * 4
    bwd_b = feat_b + out.numel() * 4 + acc.numel() * 4
    return {"what": f"optional operator (SURVEY 8f rank 4): group-wise correlation volumes [V,k,{groups},D,H,W] over the "
                    "same homography sweep (lss_fpn.py:485-506 arithmetic, warp-shuffle group sums); not part of the step",
            "groups": groups, "fwd_ms": round(res["fwd"], 5), "bwd_ms": round(res["bwd"], 5),
            "fwd_algorithmic_mb": round(fwd_b / 1e6, 1), "bwd_algorithmic_mb": round(bwd_b / 1e6, 1),
            "fwd_frac_of_hbm_peak": round(fwd_b / (res["fwd"] * 1e-3) / 1e9 / peak, 4),
            "bwd_frac_of_hbm_peak": round(bwd_b / (res["bwd"] * 1e-3) / 1e9 / peak, 4),
            "note": "the output is 16x smaller than the variance volume, so the kernels are bound by the gather "
                    "(L1 / L2 tap traffic and, in the backward, the un-merged fp32 RED payload), not by HBM"}


def run_sharded_leg(args, dev, rank, world, dist):
    """BASELINE.json configs[2]: ONE test-time scene (V = --sharded-views, forward only) with its
    reference views sharded over the ranks and the voxel partials combined over NVLink, against
    the same forward on one GPU.  Reported as the ``sharded`` key of the N > 1 bench line."""
    from mvsdet_b200 import sharded
    from mvsdet_b200.hotpath import MVSDetHotPath
    from mvsdet_b200.scene import SceneConfig, make_scene
    cfg = SceneConfig(n_views=args.sharded_views)
    scene = make_scene(cfg, seed=7, with_grads=False)          # the same scene on every rank
    hot = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        feature_dtype=torch.bfloat16)
    feat = scene["feature"].to(dev)
    cost = scene["cost_out"].to(dev)
    iters = 30

    def timed(fn, n=iters):
        for _ in range(3):
            fn()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # one GPU, whole scene (every rank runs it on its own GPU; no communication)
    geo_full = hot.geometry(scene["img_meta"], dev)
    with torch.no_grad():
        whole = hot(feat, scene["img_meta"], cost_regularization=lambda var: cost, geometry=geo_full)
        ms_eager = timed(lambda: hot(feat, scene["img_meta"], cost_regularization=lambda var: cost,
                                     geometry=geo_full))
        # the same forward replayed as a CUDA graph: the 1-GPU baseline gets the treatment the sharded
        # chain gets (the speed-up is quoted against the FASTER of the two)
        ms_graph = None
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                hot(feat, scene["img_meta"], cost_regularization=lambda var: cost, geometry=geo_full)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g1 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1):
                out_g = hot(feat, scene["img_meta"], cost_regularization=lambda var: cost, geometry=geo_full)
            ms_graph = timed(g1.replay)
            if not torch.equal(out_g["count"], whole["count"]):
                ms_graph = None
            del g1, out_g
        except Exception:                                  # noqa: BLE001
            ms_graph = None
    ms_whole = min(ms_eager, ms_graph) if ms_graph else ms_eager
    out = {"workload": f"BASELINE.json configs[2]: V={cfg.n_views} test-time scene, forward, reference views "
                       f"sharded over {world} GPUs, voxel sums + counts combined once per scene",
           "views": cfg.n_views, "ms_whole_scene_1gpu": round(ms_whole, 4),
           "ms_whole_scene_1gpu_eager": round(ms_eager, 4),
           "ms_whole_scene_1gpu_graph": None if ms_graph is None else round(ms_graph, 4),
           "bytes": int(whole["volume_mean"].numel() * 4 + whole["count"].numel() * 4)}
    pipe = sharded.ShardedScenePipeline(hot, cfg, dev)
    pipe.load(scene["feature"], scene["cost_out"], scene["img_meta"])      # pose-clustered blocks
    out["partition"] = ("pose-clustered blocks (sharded.pose_order)" if pipe.view_order != list(range(cfg.n_views))
                        else "contiguous blocks")
    out["halo_views_per_rank"] = pipe.halo_counts
    out["halo_views_per_rank_contiguous"] = sharded.halo_counts(geo_full.neighbor_ids_ref(), world)
    results = {}
    for mode in ("p2p", "nccl"):
        try:
            res = pipe.forward(mode)
            torch.cuda.synchronize()
            ok_count = bool(torch.equal(res["count"], whole["count"]))
            err = float((res["volume_mean"].reshape(-1) - whole["volume_mean"].reshape(-1)).abs().max())
            chk = res["volume_mean"].double().sum().reshape(1)
            gathered = [torch.zeros_like(chk) for _ in range(world)]
            dist.all_gather(gathered, chk)
            flags = torch.tensor([int(ok_count), int(err <= 1e-5 * max(1.0, float(whole["volume_mean"].abs().max())))],
                                 device=dev)
            dist.all_reduce(flags, op=dist.ReduceOp.MIN)
            ms_lat = timed(lambda: pipe.forward(mode))
            ms_thr = timed(lambda: pipe.forward_stream(mode, 8), n=6) / 8
            results[mode] = {"ms_per_scene_latency": round(ms_lat, 4), "ms_per_scene_pipelined": round(ms_thr, 4),
                             "counts_bit_exact": bool(flags[0].item()), "volume_close": bool(flags[1].item()),
                             "max_abs_err_vs_1gpu": err,
                             "replicas_identical": all(float(g) == float(gathered[0]) for g in gathered)}
        except Exception as exc:                          # noqa: BLE001 -- keep the other mode's number
            results[mode] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    out["modes"] = results
    best = min((m for m in results if "ms_per_scene_pipelined" in results[m]),
               key=lambda m: results[m]["ms_per_scene_pipelined"], default=None)
    if best is not None:
        out.update(collective=best, ms=results[best]["ms_per_scene_pipelined"],
                   ms_latency=results[best]["ms_per_scene_latency"],
                   speedup_vs_1gpu=round(ms_whole / results[best]["ms_per_scene_pipelined"], 3),
                   speedup_vs_1gpu_latency=round(ms_whole / results[best]["ms_per_scene_latency"], 3),
                   what_ms_is="per-scene time of a stream of scenes, the combine of scene i overlapped with "
                              "the sweep of scene i+1 (two CUDA streams, double-buffered peer partials); "
                              "ms_latency = one scene alone")
    pipe.close()
    return out


def run_sharded_train_leg(args, dev, rank, world, dist):
    """BASELINE.json configs[3]: ONE ARKitScenes-shaped training scene (40 views, per-view intrinsics,
    near/far 0.5-5.5 m, the shipped 40x40x16 grid; SURVEY.md section 5), forward + backward, reference
    views sharded over the ranks: forward partials combined over NVLink peer memory, backward with the
    halo pull of the feature gradient.  Against the same scene's graph-replayed step on one GPU.
    Reported as the ``sharded_train`` key of the N > 1 bench line."""
    from mvsdet_b200 import sharded
    from mvsdet_b200.hotpath import MVSDetHotPath
    from mvsdet_b200.pipeline import ScenePipeline
    from mvsdet_b200.scene import ARKIT, make_scene
    cfg = ARKIT
    scene = make_scene(cfg, seed=11)                           # the same scene on every rank
    hot = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        feature_dtype=torch.bfloat16)
    iters = 20

    def timed(fn, n=iters):
        for _ in range(3):
            fn()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # one GPU, whole scene: the captured step (every rank runs it on its own GPU, no communication)
    p1 = ScenePipeline(cfg, dev, feature_dtype=torch.bfloat16)
    p1.set_geometry(hot.geometry(scene["img_meta"], dev))
    p1.load_scene(scene)
    p1.step()
    torch.cuda.synchronize()
    g1 = p1.capture()
    ms_whole = timed(g1.replay)
    pipe = sharded.ShardedScenePipeline(hot, cfg, dev)
    pipe.load(scene["feature"], scene["cost_out"], scene["img_meta"])      # pose-clustered blocks
    own = pipe.view_ids.to(dev)                                             # the views this rank owns
    ref_vol, ref_count = p1.volume_mean.clone(), p1.count.clone()
    ref_g_feat, ref_g_cost = p1.g_feature[own].clone(), p1.g_cost_out[own].clone()
    g_scale = float(p1.g_feature.abs().max())
    del g1, p1
    torch.cuda.empty_cache()
    g_vol = scene["g_volume_mean"].to(dev)
    g_var = scene["g_variance"][pipe.view_ids].to(dev).contiguous(memory_format=torch.channels_last_3d)
    out = {"workload": f"BASELINE.json configs[3]: ARKitScenes-shaped scene (V={cfg.n_views}, per-view intrinsics, "
                       f"near/far {cfg.near_far_range}), forward + backward, reference views sharded over {world} GPUs",
           "views": cfg.n_views, "ms_whole_scene_1gpu_graph": round(ms_whole, 4),
           "partition": "pose-clustered blocks (sharded.pose_order)" if pipe.view_order != list(range(cfg.n_views))
                        else "contiguous blocks",
           "halo_views_per_rank": pipe.halo_counts,
           "halo_views_per_rank_contiguous": sharded.halo_counts(
               hot.geometry(scene["img_meta"], "cpu", prologue="host").neighbor_ids_host, world)}
    results = {}
    for mode in ("p2p", "nccl"):
        try:
            def step(mode=mode):
                res = pipe.forward(mode)
                gf, gc = pipe.backward(g_vol, g_var)
                return res, gf, gc
            res, gf, gc = step()
            torch.cuda.synchronize()
            flags = torch.tensor([
                int(torch.equal(res["count"].reshape(-1), ref_count.reshape(-1))),
                int(float((res["volume_mean"].reshape(-1) - ref_vol.reshape(-1)).abs().max())
                    <= 1e-5 * max(1.0, float(ref_vol.abs().max()))),
                int(float((gf - ref_g_feat).abs().max()) <= 1e-4 * g_scale),
                int(float((gc - ref_g_cost).abs().max()) <= 1e-4 * max(1.0, float(ref_g_cost.abs().max())))],
                device=dev)
            dist.all_reduce(flags, op=dist.ReduceOp.MIN)
            ms = timed(step)
            results[mode] = {"ms_per_scene": round(ms, 4), "counts_bit_exact": bool(flags[0].item()),
                             "volume_close": bool(flags[1].item()), "g_feature_close_1e-4": bool(flags[2].item()),
                             "g_cost_out_close_1e-4": bool(flags[3].item())}
        except Exception as exc:                          # noqa: BLE001 -- keep the other mode's number
            results[mode] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    out["modes"] = results
    best = min((m for m in results if "ms_per_scene" in results[m]), key=lambda m: results[m]["ms_per_scene"],
               default=None)
    if best is not None:
        out.update(collective=best, ms=results[best]["ms_per_scene"],
                   speedup_vs_1gpu=round(ms_whole / results[best]["ms_per_scene"], 3),
                   what_ms_is="one scene, forward (captured chain + combine) then backward (captured local "
                              "chain, halo pull over NVLink between two barriers, unpack); max over ranks")
    pipe.close()
    return out


def run_own_arm(args, cfg, cfg_json):
    import torch.distributed as dist
    from mvsdet_b200 import _lib
    from mvsdet_b200.hotpath import MVSDetHotPath

    rank, local, world = _dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: mvsdet_b200 has no CPU path "
                           "(use --impl reference for the CPU baseline)")
    numa_node = bind_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    feat_dtype = torch.bfloat16 if args.feature_dtype == "bf16" else torch.float32
    mod = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        stride=cfg.stride)
    use_graph = not args.no_graph
    pipes, graphs, host_scene = _build_pipes(cfg, dev, feat_dtype, mod, rank, capture=use_graph)
    launches_before = _lib.launch_count()
    pipes[0].step()
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - launches_before

    def one_step(i):
        if use_graph:
            graphs[i % NBUF].replay()
        else:
            pipes[i % NBUF].step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(x):
        if world > 1:
            t = torch.tensor([x], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    # ---- value: device-resident inputs --------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    ms_total, wall0, wall1 = _time_steps(one_step, args.steps, args.warmup, barrier)
    ms_total = rank_max(ms_total)
    ms_per_step = ms_total / args.steps
    value = world * args.steps / (ms_total * 1e-3)
    # the outputs of the last timed step, before any later leg reuses the buffers
    dump = None
    if args.dump_outputs and rank == 0:
        arrays, dump = snapshot_outputs(pipes[(args.steps - 1) % NBUF])
        write_outputs(args.dump_outputs, arrays)
        del arrays
    # the same measurement over a long run (sustained clocks / power), on request
    sustained = None
    if args.steps < args.sustained_steps:
        ms_s, ws0, ws1 = _time_steps(one_step, args.sustained_steps, 3, barrier)
        ms_s = rank_max(ms_s)
        sustained = {"value": world * args.sustained_steps / (ms_s * 1e-3), "unit": UNIT,
                     "steps": args.sustained_steps, "ms_per_step": ms_s / args.sustained_steps,
                     "clocks": sampler.summary(ws0, ws1)}

    # ---- e2e: host buffers through the public pipeline call -------------
    p0 = pipes[0]
    host = p0.host_buffers()
    host["feature"].copy_(host_scene["feature"])
    host["cost_out"].copy_(host_scene["cost_out"])
    host["g_volume_mean"].copy_(host_scene["g_volume_mean"].reshape(host["g_volume_mean"].shape))
    host["g_variance"].copy_(host_scene["g_variance"].permute(0, 2, 3, 4, 1))
    e2e_steps = max(3, min(args.steps, args.e2e_steps))
    from mvsdet_b200.pipeline import HostPipelinedRunner
    runner = HostPipelinedRunner(pipes, graphs if use_graph else None)
    host_in = {n: host[n] for n in p0.INPUTS}
    runner.run(host_in, 2 * NBUF)                       # warm-up: every buffer set, twice
    barrier()
    e2, e3 = runner.run(host_in, e2e_steps)             # H2D / compute / D2H overlapped across steps
    barrier()
    ms_e2e = rank_max(e2.elapsed_time(e3))
    # the same call without overlap (one stream), for reference
    for _ in range(2):
        p0.run_host(graphs[0] if use_graph else None)
    barrier()
    e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e4.record()
    for _ in range(min(e2e_steps, 10)):
        p0.run_host(graphs[0] if use_graph else None)
    e5.record()
    barrier()
    ms_e2e_serial = e4.elapsed_time(e5) / min(e2e_steps, 10)
    e2e_value = world * e2e_steps / (ms_e2e * 1e-3)
    sampler.stop()
    clocks = sampler.summary(wall0, wall1)
    # sanity of the e2e result: compare the host copy of the outputs with the device ones
    e2e_ok = bool(torch.equal(host["count"], p0.count.cpu()))
    h2d_parts = {n: getattr(p0, n).numel() * getattr(p0, n).element_size() for n in p0.INPUTS}

    # ---- per-kernel device times (CUDA events around each launch, same stream)
    ksteps = max(3, min(args.steps, 30))
    kernels, abytes = _kernel_table(pipes, ksteps)
    peak, peak_src = _peaks()
    path_names = [n for n in kernels if n not in ("pack", "unpack")]
    top = max(kernels, key=lambda n: kernels[n]["ms"])
    total_ms = sum(k["ms"] for k in kernels.values())
    achieved = kernels[top]["gbs"]
    own_path_mb = sum(abytes[n] for n in path_names) / 1e6
    roofline = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": abytes[top],
                "kernel_ms": kernels[top]["ms"],
                "share_of_step": round(kernels[top]["ms"] / total_ms, 3),
                # whole path: SURVEY.md 8(d)'s 3 034 MB per scene (fp32 sizes, pack / unpack NOT counted)
                "path_algorithmic_mb": SURVEY_PATH_MB,
                "path_achieved_gbs": round(SURVEY_PATH_MB * 1e6 / (ms_per_step * 1e-3) / 1e9, 1),
                "path_frac": round(SURVEY_PATH_MB * 1e6 / (ms_per_step * 1e-3) / 1e9 / peak, 4),
                # the same with the bytes this configuration actually has to move (bf16 features are smaller)
                "path_algorithmic_mb_own_dtypes": round(own_path_mb, 1),
                "path_frac_own_dtypes": round(own_path_mb * 1e6 / (ms_per_step * 1e-3) / 1e9 / peak, 4),
                "layout_overhead": {"what": "pack (FPN fp32 NCHW -> channels-last) + unpack of the gradient: "
                                            "self-inflicted layout cost, not algorithmic bytes",
                                    "mb": round((abytes["pack"] + abytes["unpack"]) / 1e6, 1),
                                    "ms": round(kernels["pack"]["ms"] + kernels["unpack"]["ms"], 5)}}
    # SURVEY.md 8(d): both denominators (measured copy bandwidth and the nominal 8 TB/s), and the
    # back-projection's data-dependent traffic (passing (view, voxel) pairs x C x bytes per feature)
    roofline["frac_of_nominal_8tbs"] = round(achieved / 8000.0, 4)
    roofline["path_frac_of_nominal_8tbs"] = round(SURVEY_PATH_MB * 1e6 / (ms_per_step * 1e-3) / 1e9 / 8000.0, 4)
    pairs = int(p0.count.sum().item())
    roofline["backproject_passing_pairs"] = pairs
    roofline["backproject_pairs_feature_mb"] = round(pairs * cfg.channels * p0.feat_cl.element_size() / 1e6, 1)
    ncu_traffic = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(ncu_traffic):
        try:
            with open(ncu_traffic) as fh:
                tj = json.load(fh)
            roofline["traffic"] = tj.get(top)
            red = tj.get(top + "_red_payload")
            if red:
                # the scatter kernel's second stream: fp32 REDs into L2.  Ceiling measured by
                # tools/microbench_red.cu on this pool's B200 (profiles/r01_b_microbench_red.txt).
                red_gbs = red / (kernels[top]["ms"] * 1e-3) / 1e9
                roofline["limiter"] = {"what": "fp32 red.global.add.v4 payload into L2 (ncu l1tex2xbar write bytes)",
                                       "red_payload_bytes": red, "achieved_gbs": round(red_gbs, 1),
                                       "ceiling_gbs": 5700.0, "frac": round(red_gbs / 5700.0, 3),
                                       "binding": red_gbs / 5700.0 > 0.8}
        except Exception:
            pass

    # ---- the autograd drop-in (MVSDetHotPath + torch.autograd, scene geometry every call):
    # what a maintainer gets from INTEGRATION.md level 1, wall clock incl. host work
    module_api = None
    if world == 1:
        hot = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                            stride=cfg.stride, feature_dtype=feat_dtype)
        m_feat = p0.feature.detach().clone().requires_grad_(True)
        m_cost = p0.cost_out.detach().clone().requires_grad_(True)
        m_gvar = p0.g_variance.permute(0, 4, 1, 2, 3)       # channels_last_3d view, as cuDNN returns it
        m_gvol = p0.g_volume_mean.view(cfg.channels, *cfg.n_voxels)

        def module_step():
            res = hot(m_feat, host_scene["img_meta"], cost_regularization=lambda var: m_cost)
            torch.autograd.backward([res["variance"], res["volume_mean"]], [m_gvar, m_gvol])
            m_feat.grad = None
            m_cost.grad = None

        for _ in range(5):
            module_step()
        torch.cuda.synchronize()
        n_mod = 60
        t0 = time.perf_counter()
        for _ in range(n_mod):
            module_step()
        t_host = (time.perf_counter() - t0) / n_mod * 1e3          # host time to ENQUEUE a scene
        torch.cuda.synchronize()
        ms_mod = (time.perf_counter() - t0) / n_mod * 1e3
        module_api = {"value": 1e3 / ms_mod, "unit": UNIT, "ms_per_scene": round(ms_mod, 4), "steps": n_mod,
                      "host_enqueue_ms_per_scene": round(t_host, 4),
                      "fraction_of_graph_value": round((1e3 / ms_mod) / value, 4),
                      "what": "MVSDetHotPath forward + torch.autograd backward, scene geometry rebuilt every "
                              "call (two host ATen calls + one setup kernel), shared fp32 gradient accumulator, "
                              "caching allocator, no CUDA graph"}
        if not args.no_extras:
            # the opt-in bit-reproducible backward (64-bit fixed-point integer REDs, un-merged scatter)
            hot_det = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                                    stride=cfg.stride, feature_dtype=feat_dtype, deterministic=True)

            def det_step():
                res = hot_det(m_feat, host_scene["img_meta"], cost_regularization=lambda var: m_cost)
                torch.autograd.backward([res["variance"], res["volume_mean"]], [m_gvar, m_gvol])
                g = m_feat.grad
                m_feat.grad = None
                m_cost.grad = None
                return g
            g_a = det_step().clone()
            g_b = det_step().clone()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(20):
                det_step()
            torch.cuda.synchronize()
            ms_det = (time.perf_counter() - t0) / 20 * 1e3
            module_api["deterministic"] = {"value": 1e3 / ms_det, "unit": UNIT, "ms_per_scene": round(ms_det, 4),
                                           "bit_identical_runs": bool(torch.equal(g_a, g_b)),
                                           "what": "MVSDetHotPath(deterministic=True): backward accumulates in 64-bit "
                                                   "fixed point with integer REDs (mvsd_*_bwd_det); opt-in"}
            del hot_det, g_a, g_b
        del hot, m_feat, m_cost

    # ---- fp32-feature line (1e-4 parity is proven on fp32 features; their backward is the lean kernel)
    f32_line = None
    if world == 1 and feat_dtype == torch.bfloat16 and not args.no_extras:
        pipes32, graphs32, _ = _build_pipes(cfg, dev, torch.float32, mod, rank, capture=use_graph)

        def step32(i):
            if use_graph:
                graphs32[i % NBUF].replay()
            else:
                pipes32[i % NBUF].step()
        n32 = max(20, min(args.steps, 100))
        ms32, _, _ = _time_steps(step32, n32, 3, barrier)
        k32, _ = _kernel_table(pipes32, 10)
        f32_line = {"value": n32 / (ms32 * 1e-3), "unit": UNIT, "steps": n32, "ms_per_step": ms32 / n32,
                    "dtype": "f32 features, f32 accumulate",
                    "kernels_ms": {n: k32[n]["ms"] for n in k32}}
        del pipes32, graphs32
        torch.cuda.empty_cache()

    # ---- bf16 hand-off line: variance / g_variance exchanged with the cost-regularisation net as bf16
    # channels_last_3d (what that net computes in under autocast), fp32 accumulation inside the kernels.
    # NOT the headline: BASELINE configs[1] names fp32 accumulation and the headline keeps fp32 volumes.
    bf16_line = None
    if world == 1 and feat_dtype == torch.bfloat16 and not args.no_extras:
        pipes16, graphs16, _ = _build_pipes(cfg, dev, torch.bfloat16, mod, rank, capture=use_graph,
                                            variance_dtype=torch.bfloat16)

        def step16(i):
            if use_graph:
                graphs16[i % NBUF].replay()
            else:
                pipes16[i % NBUF].step()
        n16 = max(20, min(args.steps, 100))
        ms16, _, _ = _time_steps(step16, n16, 3, barrier)
        k16, ab16 = _kernel_table(pipes16, 10)
        path16 = sum(ab16[n] for n in ab16 if n not in ("pack", "unpack"))
        bf16_line = {"value": n16 / (ms16 * 1e-3), "unit": UNIT, "steps": n16, "ms_per_step": ms16 / n16,
                     "dtype": "bf16 features, bf16 variance / g_variance hand-off, f32 accumulate",
                     "path_algorithmic_mb_own_dtypes": round(path16 / 1e6, 1),
                     "path_frac_own_dtypes": round(path16 / (ms16 / n16 * 1e-3) / 1e9 / peak, 4),
                     "kernels_ms": {n: k16[n]["ms"] for n in k16},
                     "note": "half the bytes of the two 1.18 GB volumes; an option of the hand-off "
                             "(tests/test_gpu_costreg.py, test_gpu_benchmarked.py), not the headline configuration"}
        del pipes16, graphs16
        torch.cuda.empty_cache()

    # ---- optional operator: group-wise correlation volume over the same sweep (SURVEY 8f rank 4)
    corr_line = None
    if world == 1 and feat_dtype == torch.bfloat16 and not args.no_extras:
        try:
            corr_line = time_group_correlation(p0, cfg, peak)
        except Exception as exc:                       # noqa: BLE001
            corr_line = {"error": f"{type(exc).__name__}: {exc}"[:200]}

    eager = None
    if world == 1 and not args.no_extras:
        try:
            eager = time_eager_gpu(cfg, host_scene, dev)
        except Exception as exc:                       # noqa: BLE001
            eager = {"error": f"{type(exc).__name__}: {exc}"[:200]}

    sharded_line = None
    if world > 1 and not args.no_sharded:
        try:
            sharded_line = run_sharded_leg(args, dev, rank, world, dist)
        except Exception as exc:                       # noqa: BLE001
            sharded_line = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    sharded_train_line = None
    if world > 1 and not args.no_sharded:
        try:
            sharded_train_line = run_sharded_train_leg(args, dev, rank, world, dist)
        except Exception as exc:                       # noqa: BLE001
            sharded_train_line = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    if rank == 0:
        cpu_line = None
        if world == 1 and not args.no_cpu_baseline:
            val, t_step, threads, sample, _ = time_cpu_reference(cfg, 3, 1, 30.0)
            cpu_line = {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16 features, f32 accumulate" if feat_dtype == torch.bfloat16 else "f32",
            "data": "synthetic", "config": cfg_json,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": p0.h2d_bytes(),
                    "d2h_bytes_per_step": p0.d2h_bytes(), "steps": e2e_steps,
                    "ms_per_step": ms_e2e / e2e_steps, "outputs_match_device": e2e_ok,
                    "overlap": "H2D / compute / D2H on three streams over %d buffer sets" % NBUF,
                    "ms_per_step_serial": ms_e2e_serial,
                    "h2d_bytes_by_input": h2d_parts, "host_numa_node": numa_node,
                    "h2d_fraction_g_variance": round(h2d_parts["g_variance"] / p0.h2d_bytes(), 3),
                    "note": "g_variance (the gradient the cost-regularisation net returns) is 90 % of the "
                            "upload: on a real detector it is produced on the device; here it is a synthetic "
                            "input and is copied in every step, so e2e is PCIe-bound"},
            "gpu_launches": launches_per_step * args.steps,
            "gpu_launches_per_step": launches_per_step,
            "cuda_graph": use_graph,
            "roofline": roofline, "kernels": kernels,
        }
        if sustained is not None:
            line["sustained"] = sustained
        if dump is not None:
            line["dumped_outputs"] = {"dir": args.dump_outputs, "dtype": "float32", "step": args.steps - 1,
                                      "outputs": dump}
        if module_api is not None:
            line["module_api"] = module_api
        if f32_line is not None:
            line["f32_features"] = f32_line
        if bf16_line is not None:
            line["bf16_handoff"] = bf16_line
        if corr_line is not None:
            line["group_correlation"] = corr_line
        if eager is not None:
            line["eager_gpu"] = eager
        if sharded_line is not None:
            line["sharded"] = sharded_line
        if sharded_train_line is not None:
            line["sharded_train"] = sharded_train_line
        if cpu_line is not None:
            line["cpu_baseline"] = cpu_line
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_sweep(args):
    """BASELINE.json configs[4]: D in {12..64} x V in {10..100} x feature maps up to 480x640, achieved
    algorithmic GB/s of the two sweep kernels against the measured HBM peak (1 GPU; view-chunked)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("sweep_chart", os.path.join(ROOT, "tools", "sweep_chart.py"))
    sc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sc)
    rows = sc.sweep(quick=args.sweep == "quick", verbose=False)
    print(json.dumps({"metric": "plane-sweep kernels, achieved algorithmic GB/s vs HBM roofline",
                      "config": {"workload": "BASELINE.json configs[4]: depth-plane / view-count / resolution sweep",
                                 "channels": 256, "dtype": "bf16 features, f32 variance"},
                      "hbm_peak_gbs": sc.peak(), "n_gpus": 1, "data": "synthetic", "rows": rows}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--views", type=int, default=20)
    ap.add_argument("--feature-dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=30)
    ap.add_argument("--sustained-steps", type=int, default=0,
                    help="a second timed run of this many steps when --steps is shorter (sustained clocks); "
                         "reported apart from the headline, off by default")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32, 64 MB in all; "
                         "a large output as a fixed, seeded sample), for comparing two builds")
    ap.add_argument("--no-extras", action="store_true", help="skip the fp32-feature and eager-GPU legs")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the view-sharded V=80 leg")
    ap.add_argument("--sharded-views", type=int, default=80)
    ap.add_argument("--sweep", choices=["quick", "full"], default=None,
                    help="BASELINE.json configs[4] instead of the step benchmark: depth-plane / view-count / "
                         "resolution sweep of the plane-sweep kernels (tools/sweep_chart.py), one JSON line")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "own":
        ap.error("--dump-outputs needs --impl own")
    if args.sweep:
        run_sweep(args)
        return
    args.warmup = max(args.warmup, 3 if args.impl == "own" else 1)

    from mvsdet_b200.scene import SceneConfig
    cfg = SceneConfig(n_views=args.views)
    hf, wf = cfg.feat_hw
    cfg_json = {
        "workload": "BASELINE.json configs[1]: mvsdet_res50_2x_low_res, 1 scene/step, fwd+bwd of "
                    "plane-sweep variance + depth top-k + voxel back-projection",
        "views": cfg.n_views, "channels": cfg.channels, "depth_planes": cfg.num_depth,
        "feature_map": [hf, wf], "image": [cfg.pad_shape[0], cfg.pad_shape[1]],
        "neighbors": cfg.num_neighbors, "topk": cfg.topk, "voxels": list(cfg.n_voxels),
        "feature_in": "fp32 NCHW (FPN layout), packed in-step to channels-last "
                      + ("bf16" if args.feature_dtype == "bf16" else "fp32"),
        "variance": "fp32 channels_last_3d", "scenes_per_step_per_gpu": 1,
        "parallelism": f"scene-parallel x{args.gpus} (no collective)",
        "l2": f"working set 2.6 GB/step >> 126 MB L2; {NBUF} rotating scene buffer sets",
        "cost_reg_net": "excluded (synthetic cost_out / g_variance inputs)",
    }
    if args.impl == "reference":
        run_reference_arm(args, cfg, cfg_json)
    else:
        run_own_arm(args, cfg, cfg_json)


if __name__ == "__main__":
    main()
