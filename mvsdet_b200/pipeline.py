"""Pre-allocated, CUDA-graph-capturable forward+backward of the hot path for
one scene -- the training-step form of ``MVSDetHotPath``.

``MVSDetHotPath`` (hotpath.py) is the autograd drop-in for
mvsdet.py:404-515.  In a training step the cost-regularisation net sits between
the stages, so its output and the gradient it sends back to the variance volume
are *inputs* of the path (SURVEY.md 8d).  ``ScenePipeline`` owns every buffer of
that step, enqueues the eight kernels through the C ABI without touching the
allocator, and can therefore be captured once into a CUDA graph and replayed:

    pack          feature fp32 NCHW      -> channels-last fp32|bf16
    sweep fwd     packed feature         -> variance            (-> cost-reg net)
    top-k fwd     cost_out               -> prob, hypotheses, depth_coding
    voxels fwd    packed feature, hyp.   -> volume_mean, count
    voxels bwd    g_volume_mean          -> g_feat += , g_pn
    pn bwd        g_pn                   -> g_est_densities
    top-k bwd     g_est_densities        -> g_cost_out         (-> cost-reg net bwd)
    sweep bwd     g_variance             -> g_feat +=
    unpack        g_feat channels-last   -> g_feature fp32 NCHW

It also provides the host-buffer form of the same call (``run_host``): pinned
host inputs are copied in, the step runs, results are copied out -- the
end-to-end path bench.py reports as ``e2e``.

``deterministic=True`` gives the bit-reproducible form of the same step: the two
scatter backwards (voxels bwd, sweep bwd) add into int64 fixed-point accumulators
(``*_det`` kernels, integer REDs) that ``mvsd_fixed_to_float`` converts once, so
``g_feature`` and ``g_cost_out`` are the bits of ``MVSDetHotPath(deterministic=True)``
on every run.  It is the form that runs under ``torch.use_deterministic_algorithms(True)``.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _lib, ops
from ._lib import BP_MEAN
from .geometry import SceneGeometry
from .scene import SceneConfig

__all__ = ["ScenePipeline"]


class ScenePipeline:
    INPUTS = ("feature", "cost_out", "g_volume_mean", "g_variance")
    OUTPUTS = ("volume_mean", "count", "g_feature", "g_cost_out")
    deterministic = False          # fp32-RED backward (the default, fastest form)

    def __init__(self, cfg: SceneConfig, device="cuda", feature_dtype=torch.bfloat16,
                 variance_dtype=torch.float32, pack_input: bool = True, deterministic: bool = False):
        self.cfg = cfg
        self.deterministic = bool(deterministic)
        self.device = torch.device(device)
        self.feature_dtype = feature_dtype
        self.variance_dtype = variance_dtype
        self.pack_input = pack_input
        v, c, d, t = cfg.n_views, cfg.channels, cfg.num_depth, cfg.topk
        hf, wf = cfg.feat_hw
        nx, ny, nz = cfg.n_voxels
        n = nx * ny * nz
        dev = self.device
        f32 = dict(dtype=torch.float32, device=dev)
        # inputs
        self.feature = torch.empty((v, c, hf, wf), **f32)                         # FPN output, NCHW
        self.cost_out = torch.empty((v, 2, d, hf, wf), **f32)
        self.g_volume_mean = torch.empty((c, n), **f32)
        self.g_variance = torch.empty((v, d, hf, wf, c), dtype=variance_dtype, device=dev)
        # intermediates
        self.feat_cl = torch.empty((v, hf, wf, c), dtype=feature_dtype, device=dev)
        self.variance = torch.empty((v, d, hf, wf, c), dtype=variance_dtype, device=dev)
        self.prob_volume = torch.empty((v, d, hf, wf), **f32)
        self.off_pred = torch.empty((v, d, hf, wf), **f32)
        self.est_depth = torch.empty((v, t, hf, wf), **f32)
        self.est_dens = torch.empty((v, t, hf, wf), **f32)
        self.est_idx = torch.empty((v, t, hf, wf), dtype=torch.int64, device=dev)
        self.depth_coding = torch.empty((v, hf, wf), **f32)
        self.g_pn = torch.empty((v, t, hf, wf), **f32)
        self.g_est_dens = torch.zeros((v, t, hf, wf), **f32)
        self.g_feat_cl = torch.empty((v, hf, wf, c), **f32)
        if self.deterministic:
            # the fixed-point accumulators of the *_det kernels; g_feat_cl and g_pn take their conversions
            self.g_feat_q = torch.empty((v, hf, wf, c), dtype=torch.int64, device=dev)
            self.g_pn_q = torch.empty((v, t, hf, wf), dtype=torch.int64, device=dev)
            self._g_feat_q = self.g_feat_q.permute(0, 3, 1, 2)
        # outputs
        self.volume_mean = torch.empty((c, n), **f32)
        self.count = torch.empty((n,), dtype=torch.int32, device=dev)
        self.g_feature = torch.empty((v, c, hf, wf), **f32)
        self.g_cost_out = torch.empty((v, 2, d, hf, wf), **f32)
        # the logical [V,C,H,W] / [V,C,D,H,W] views of the channels-last buffers the kernels take
        self._feat = self.feat_cl.permute(0, 3, 1, 2)
        self._g_feat = self.g_feat_cl.permute(0, 3, 1, 2)
        self._variance = self.variance.permute(0, 4, 1, 2, 3)
        self._g_variance = self.g_variance.permute(0, 4, 1, 2, 3)
        self.geo: Optional[SceneGeometry] = None
        self._host = None
        self._side = torch.cuda.Stream(device=dev)     # zero-fills of the gradient accumulators
        self._aux = torch.cuda.Stream(device=dev, priority=-1)   # the small kernels, see step()
        self.overlap_small = True

    # ------------------------------------------------------------------
    def set_geometry(self, geo: SceneGeometry) -> None:
        self.geo = geo

    def load_scene(self, scene: Dict) -> None:
        """Copy a host scene (scene.make_scene) into the input buffers."""
        self.feature.copy_(scene["feature"])
        self.cost_out.copy_(scene["cost_out"])
        self.g_volume_mean.copy_(scene["g_volume_mean"].reshape(self.g_volume_mean.shape))
        self.g_variance.copy_(scene["g_variance"].permute(0, 2, 3, 4, 1))
        if not self.pack_input:
            self.feat_cl.copy_(scene["feature"].permute(0, 2, 3, 1))

    def algorithmic_bytes(self) -> Dict[str, int]:
        """Compulsory traffic of each kernel: every input read once, every
        output written once (SURVEY.md 8d)."""
        cfg = self.cfg
        v, c, d, t = cfg.n_views, cfg.channels, cfg.num_depth, cfg.topk
        hf, wf = cfg.feat_hw
        h, w = cfg.crop_hw
        n = cfg.n_voxels[0] * cfg.n_voxels[1] * cfg.n_voxels[2]
        bf = self.feat_cl.element_size()
        bv = self.variance.element_size()
        feat = v * c * hf * wf
        vol = v * c * d * hf * wf
        out = {
            "pack": feat * 4 + feat * bf,
            "plane_sweep_fwd": feat * bf + vol * bv,
            "depth_topk_fwd": 2 * v * d * hf * wf * 4 + 2 * v * d * hf * wf * 4
                              + 2 * v * t * hf * wf * 4 + v * t * hf * wf * 8 + v * hf * wf * 4,
            "backproject_fwd": v * c * h * w * bf + 2 * v * h * w * t * 4 + c * n * 4 + n * 4,
            "backproject_bwd": c * n * 4 + v * c * h * w * bf + v * c * h * w * 4 + v * h * w * t * 4,
            "prob_norm_bwd": 3 * v * h * w * t * 4,
            "depth_topk_bwd": 2 * v * d * hf * wf * 4 + v * t * hf * wf * 12 + 2 * v * d * hf * wf * 4,
            "plane_sweep_bwd": vol * bv + feat * bf + feat * 4,
            "unpack": feat * 4 * 2,
        }
        if self.deterministic:
            # the scatter backwards write 8-byte fixed-point accumulators, each converted once (read 8, write 4)
            out["backproject_bwd_det"] = out.pop("backproject_bwd") + v * c * h * w * 4 + v * h * w * t * 4
            out["plane_sweep_bwd_det"] = out.pop("plane_sweep_bwd") + feat * 4
            out["fixed_to_float_pn"] = v * t * hf * wf * (8 + 4)
            out["fixed_to_float_feat"] = feat * (8 + 4)
        return out

    # ------------------------------------------------------------------
    def step(self, timers: Optional[Dict] = None) -> None:
        """Enqueue forward+backward on the current stream.  No allocation, no
        synchronisation: capturable in a CUDA graph.  ``timers`` (name ->
        list of (start, end) event pairs) makes it time every kernel."""
        geo = self.geo
        if geo is None:
            raise RuntimeError("set_geometry() first")
        det = self.deterministic
        if not det:
            # its backward kernels RED in fp32, in an order that varies from run to run
            ops._alert_not_deterministic("ScenePipeline.step")
        cfg = self.cfg
        h, w = geo.height, geo.width
        near, interval = cfg.near_far_range[0], cfg.depth_interval
        sweep = (self._feat, geo.neighbor_ids, geo.hom, geo.depth_values)
        hyp = (self._feat, geo.points, geo.projection, self.est_depth, self.est_dens)
        bp = dict(vs_z=cfg.voxel_size[2], mode=BP_MEAN, height=h, width=w, channels_first=True, count=self.count)

        def run(name, launch, *args, **kwargs):
            if timers is None:
                launch(*args, **kwargs)
                return
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            launch(*args, **kwargs)
            e1.record()
            timers.setdefault(name, []).append((e0, e1))

        def small_kernels():
            with torch.cuda.stream(aux):
                run("depth_topk_fwd", _lib.depth_topk_fwd, self.cost_out, self.prob_volume, self.off_pred,
                    self.est_depth, self.est_dens, self.est_idx, self.depth_coding, near=near, interval=interval)
                run("backproject_fwd", _lib.backproject_fwd, *hyp, self.volume_mean, **bp)
                # ---- backward
                aux.wait_stream(self._side)
                if det:
                    run("backproject_bwd_det", _lib.backproject_bwd_det, self.g_volume_mean, self.count, *hyp,
                        self._g_feat_q, self.g_pn_q, vs_z=cfg.voxel_size[2], height=h, width=w, channels_first=True)
                    run("fixed_to_float_pn", _lib.fixed_to_float, self.g_pn_q, self.g_pn)
                else:
                    run("backproject_bwd", _lib.backproject_bwd, self.g_volume_mean, *hyp, self._g_feat, self.g_pn,
                        **bp)
                run("prob_norm_bwd", _lib.prob_norm_bwd, self.est_dens, self.g_pn, self.g_est_dens, height=h,
                    width=w)
                run("depth_topk_bwd", _lib.depth_topk_bwd, self.cost_out, self.est_idx, None, None, None,
                    self.g_est_dens, None, self.g_cost_out, near=near, interval=interval)

        # Three streams (fork/join edges once the step is captured into a graph):
        #   cur    pack -> sweep fwd -> sweep bwd -> unpack      (the two 1.2 GB streaming kernels)
        #   _aux   top-k fwd -> voxels fwd -> voxels bwd -> pn bwd -> top-k bwd
        #          small latency-bound kernels (2-3 waves, L2-resident operands) that depend only
        #          on pack; they run under the sweep kernels at higher stream priority.  The two
        #          backward kernels accumulate into g_feat_cl with commutative REDs -- with
        #          ``deterministic`` into g_feat_q with integer REDs, which also commute (and
        #          associate), so the overlap leaves the fixed-point sums' bits unchanged.
        #   _side  zero-fills of the gradient accumulators (98 MB + 1 MB; int64: twice that), no producer
        # With ``timers`` the kernels run back to back on ``cur`` so each can be timed alone.
        cur = torch.cuda.current_stream()
        overlap = timers is None and self.overlap_small
        aux = self._aux if overlap else cur
        if self.pack_input:
            run("pack", _lib.pack, self.feature, self._feat)
        # the fills start after the pack (which is HBM-bound on its own: 0.029 ms alone, 0.045 ms
        # next to a 98 MB memset) and run under the forward sweep instead
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            if det:
                self.g_feat_q.zero_()
                self.g_pn_q.zero_()
            else:
                self.g_feat_cl.zero_()
                self.g_pn.zero_()
        if overlap:
            aux.wait_stream(cur)
            small_kernels()
        run("plane_sweep_fwd", _lib.plane_sweep_fwd, *sweep, self._variance)
        if overlap:
            cur.wait_stream(self._side)
        else:
            small_kernels()
        if det:
            run("plane_sweep_bwd_det", _lib.plane_sweep_bwd_det, self._g_variance, *sweep, self._g_feat_q)
        else:
            run("plane_sweep_bwd", _lib.plane_sweep_bwd, self._g_variance, *sweep, self._g_feat)
        if overlap:
            cur.wait_stream(aux)
        if det:
            run("fixed_to_float_feat", _lib.fixed_to_float, self.g_feat_q, self.g_feat_cl)
        run("unpack", _lib.unpack, self._g_feat, self.g_feature)

    # ------------------------------------------------------------------
    def capture(self) -> "torch.cuda.CUDAGraph":
        """Warm up once, then capture ``step`` into a CUDA graph."""
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.step()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.step()
        return graph

    # ------------------------------------------------------------------
    def host_buffers(self) -> Dict[str, torch.Tensor]:
        """Pinned host mirrors of the inputs and outputs (allocated once)."""
        if self._host is None:
            self._host = {n: torch.empty(getattr(self, n).shape, dtype=getattr(self, n).dtype,
                                         pin_memory=True) for n in self.INPUTS + self.OUTPUTS}
        return self._host

    def h2d_bytes(self) -> int:
        return sum(getattr(self, n).numel() * getattr(self, n).element_size() for n in self.INPUTS)

    def d2h_bytes(self) -> int:
        return sum(getattr(self, n).numel() * getattr(self, n).element_size() for n in self.OUTPUTS)

    def run_host(self, graph: Optional["torch.cuda.CUDAGraph"] = None) -> None:
        """Host-buffer form: pinned inputs -> device, step, outputs -> pinned
        host; all on the current stream (the caller synchronises)."""
        host = self.host_buffers()
        for n in self.INPUTS:
            getattr(self, n).copy_(host[n], non_blocking=True)
        if graph is not None:
            graph.replay()
        else:
            self.step()
        for n in self.OUTPUTS:
            host[n].copy_(getattr(self, n), non_blocking=True)


class HostPipelinedRunner:
    """Host-buffer steps over several ``ScenePipeline`` buffer sets with the
    copies overlapped with compute: three streams (H2D, compute, D2H), step i
    uses buffer set i % n.  Every step still copies its own inputs in from
    pinned host memory and its own results out; only the *overlap* differs from
    ``ScenePipeline.run_host``.  PCIe is full duplex, so the steady state is
    bound by the slowest of {H2D, compute, D2H}.

        runner = HostPipelinedRunner(pipes, graphs)
        runner.run(host_inputs, n_steps)      # enqueue; returns (start, end) events
    """

    def __init__(self, pipes, graphs=None):
        if not pipes:
            raise ValueError("need at least one ScenePipeline")
        self.pipes = list(pipes)
        self.graphs = list(graphs) if graphs else [None] * len(self.pipes)
        dev = self.pipes[0].device
        self.s_in = torch.cuda.Stream(device=dev)
        self.s_run = torch.cuda.Stream(device=dev)
        self.s_out = torch.cuda.Stream(device=dev)
        self._ev_run = [None] * len(self.pipes)     # last compute on the set (inputs consumed)
        self._ev_out = [None] * len(self.pipes)     # last D2H of the set (outputs drained)

    def run(self, host_inputs: Dict[str, torch.Tensor], n_steps: int):
        """Enqueue ``n_steps`` host-buffer steps.  ``host_inputs`` are pinned
        tensors named as ScenePipeline.INPUTS; results land in each set's
        ``host_buffers()``.  Returns (start_event, end_event) recorded around the
        whole region; the caller synchronises."""
        cur = torch.cuda.current_stream()
        for s in (self.s_in, self.s_run, self.s_out):
            s.wait_stream(cur)
        start = torch.cuda.Event(enable_timing=True)
        end = torch.cuda.Event(enable_timing=True)
        start.record(self.s_in)
        n = len(self.pipes)
        for i in range(n_steps):
            b = i % n
            p = self.pipes[b]
            host_out = p.host_buffers()
            with torch.cuda.stream(self.s_in):
                if self._ev_run[b] is not None:
                    self.s_in.wait_event(self._ev_run[b])
                for name in p.INPUTS:
                    getattr(p, name).copy_(host_inputs[name], non_blocking=True)
                ev_in = torch.cuda.Event()
                ev_in.record(self.s_in)
            with torch.cuda.stream(self.s_run):
                self.s_run.wait_event(ev_in)
                if self._ev_out[b] is not None:
                    self.s_run.wait_event(self._ev_out[b])
                if self.graphs[b] is not None:
                    self.graphs[b].replay()
                else:
                    p.step()
                ev_run = torch.cuda.Event()
                ev_run.record(self.s_run)
                self._ev_run[b] = ev_run
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(ev_run)
                for name in p.OUTPUTS:
                    host_out[name].copy_(getattr(p, name), non_blocking=True)
                ev_out = torch.cuda.Event()
                ev_out.record(self.s_out)
                self._ev_out[b] = ev_out
        self.s_out.wait_stream(self.s_in)
        self.s_out.wait_stream(self.s_run)
        end.record(self.s_out)
        cur.wait_stream(self.s_out)
        return start, end
