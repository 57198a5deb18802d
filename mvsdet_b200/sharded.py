"""View-sharded forward of ONE scene over the ranks of a process group
(BASELINE.json configs[2]: test-time scenes with 50-100 source views).

Reference views are independent in the plane sweep and in the back-projection
(per-view loops, projects/NeRF-Det/nerfdet/mvsdet.py:453, :1401, :1458); only
the sum over views and the per-voxel valid count couple them (mvsdet.py:511-515).
So every rank sweeps a contiguous block of reference views, back-projects them
into *partial* voxel sums and counts (``MVSD_BP_SUM``), and the partials
(``C*N + N`` words, 26.3 MB for the shipped 40x40x16 grid) are combined once per
scene, giving replicas that are bit-identical across ranks.  Two combines exist:

* ``P2PVoxelReducer`` (default): the back-projection writes its partials into a
  peer-mapped buffer and ``mvsd_voxel_reduce_p2p`` does reduce-scatter +
  ``sum / (count + 1e-8)`` (mvsdet.py:514-515, :681-682) + all-gather in one kernel
  over NVLink peer pointers (V=80 on 8 B200: 0.38 ms per scene against 0.59 ms);
* ``p2p=False``: ONE NCCL all-reduce of the packed partials, then
  ``mvsd_voxel_normalize`` on every rank.  The counts travel as fp32 in the same
  buffer: they are integers <= V <= 2^24, so the sum is exact.

The FPN feature maps of all V views are resident on every rank (the k=2 pose
neighbours of a local view may belong to another rank, SURVEY.md 8e caveat 1);
only the reference-view work is partitioned: a rank packs (fp32 NCHW -> channels-last
bf16/fp32) just its own block plus the few neighbour views outside it ("halo"), and
the neighbour ids are re-based onto that compact buffer.

The partition / packing / all-reduce helpers are device-agnostic host logic and
are exercised with a world-size-2 gloo group on CPU (tests/test_sharded_cpu.py);
``ShardedSceneForward`` itself launches the CUDA kernels and needs a GPU.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib, ops
from ._lib import BP_MEAN, BP_SUM

__all__ = ["partition_views", "halo_views", "halo_pull_table", "halo_counts", "pose_order", "permute_img_meta",
           "pack_partials", "unpack_partials", "allreduce_partials", "LocalGeometry", "ShardedSceneForward",
           "ShardedScenePipeline"]


def halo_views(neighbor_ids: torch.Tensor, begin: int, end: int) -> Tuple[List[int], torch.Tensor]:
    """Views a rank must hold to sweep reference views [begin, end): the block
    itself followed by the neighbour views outside it, ascending.  Returns
    (global view ids in local order, neighbour ids re-based to local indices
    [V_local,k] int32).  Pure host logic (tested on CPU)."""
    nbr = neighbor_ids.to(torch.int64).cpu()
    own = list(range(begin, end))
    extra = sorted(set(int(x) for x in nbr.reshape(-1).tolist()) - set(own))
    order = own + extra
    lut = {g: i for i, g in enumerate(order)}
    local = torch.tensor([[lut[int(x)] for x in row] for row in nbr.tolist()],
                         dtype=torch.int32).reshape(nbr.shape[0], nbr.shape[1] if nbr.dim() > 1 else 0)
    return order, local


def halo_pull_table(neighbor_ids: torch.Tensor, world: int, rank: int):
    """Backward of a view-sharded scene: which peers hold gradient contributions for the views this
    rank owns.  ``neighbor_ids`` [V,k] are the FULL scene's ids (every rank computes the same
    table from them).  Rank q's sweep backward scatters into its halo views -- the neighbours of
    its block that it does not own; the owner pulls them.  Returns (offsets int32 [n_own+1],
    sources int32 [n_pull,2] = (peer rank, view index in the peer's local buffer)), CSR over this
    rank's owned views, peers in rank order.  Pure host logic (tested on CPU)."""
    nbr = neighbor_ids.to(torch.int64).cpu()
    v = nbr.shape[0]
    begin, end = partition_views(v, world, rank)
    per_view: List[List[Tuple[int, int]]] = [[] for _ in range(end - begin)]
    for q in range(world):
        if q == rank:
            continue
        qb, qe = partition_views(v, world, q)
        if qe <= qb:
            continue
        order, _ = halo_views(nbr[qb:qe], qb, qe)
        for local_idx, g in enumerate(order):
            if local_idx >= qe - qb and begin <= g < end:           # a halo view of q that this rank owns
                per_view[g - begin].append((q, local_idx))
    offs = [0]
    src: List[Tuple[int, int]] = []
    for lst in per_view:
        src.extend(lst)
        offs.append(len(src))
    return (torch.tensor(offs, dtype=torch.int32),
            torch.tensor(src, dtype=torch.int32).reshape(-1, 2))


def halo_counts(neighbor_ids: torch.Tensor, world: int, order: Optional[List[int]] = None) -> List[int]:
    """Halo views per rank (neighbours of a rank's block that it does not own) when rank r owns the views
    ``order[begin_r:end_r]`` (``order`` = identity when None).  Pure host logic."""
    nbr = neighbor_ids.to(torch.int64).cpu()
    v = nbr.shape[0]
    order = list(range(v)) if order is None else [int(x) for x in order]
    out = []
    for r in range(world):
        b, e = partition_views(v, world, r)
        own = set(order[b:e])
        need = set(int(x) for i in order[b:e] for x in nbr[i].tolist())
        out.append(len(need - own))
    return out


def pose_order(w2c, neighbor_ids: torch.Tensor, world: int) -> List[int]:
    """A permutation of the views such that the contiguous blocks of ``partition_views`` are pose
    clusters (SURVEY.md 8e: "contiguous or pose-clustered blocks"): the pose neighbours of a view are
    often NOT its index neighbours -- on a multi-turn scan the nearest cameras sit one turn away -- and
    every neighbour outside a rank's block is a halo map the rank has to hold, pack and, in the backward,
    have pulled from it.  Candidates: the given order, and the azimuth of the camera centres around their
    centroid in the plane of their two largest principal axes (a ring / helix scan unrolled by angle, not
    by time).  The candidate with the smaller worst-rank halo count wins (then the smaller total; ties keep
    the given order).  V=80 on 8 ranks, synthetic helix: 11-20 halo maps per rank -> 1-3.
    Every rank computes the same order from the same inputs (numpy, deterministic).  Pure host logic."""
    import numpy as np
    w = np.asarray(w2c, dtype=np.float64).reshape(-1, 4, 4)
    v = w.shape[0]
    ident = list(range(v))
    if world <= 1 or v <= 2:
        return ident
    centres = -np.einsum("vji,vj->vi", w[:, :3, :3], w[:, :3, 3])       # c2w translation = -R^T t
    x = centres - centres.mean(axis=0, keepdims=True)
    _, _, vt = np.linalg.svd(x, full_matrices=False)
    az = np.arctan2(x @ vt[1], x @ vt[0])
    by_angle = [int(i) for i in np.argsort(az, kind="stable")]
    best, best_key = ident, (max(halo_counts(neighbor_ids, world)), sum(halo_counts(neighbor_ids, world)))
    hc = halo_counts(neighbor_ids, world, by_angle)
    if (max(hc), sum(hc)) < best_key:
        best = by_angle
    return best


def permute_img_meta(img_meta: dict, order: List[int]) -> dict:
    """The scene's meta dict with its views re-ordered (extrinsics, per-view intrinsics)."""
    import numpy as np
    l2i = dict(img_meta["lidar2img"])
    l2i["extrinsic"] = [img_meta["lidar2img"]["extrinsic"][i] for i in order]
    intr = img_meta["lidar2img"]["intrinsic"]
    if not (hasattr(intr, "shape") and np.asarray(intr).ndim == 2):      # a list / array of V matrices (ARKit)
        l2i["intrinsic"] = [intr[i] for i in order]
    out = dict(img_meta)
    out["lidar2img"] = l2i
    return out


@dataclass
class LocalGeometry:
    """A rank's slice of the scene parameter block plus its halo bookkeeping."""
    geo: object                    # SceneGeometry of reference views [begin, end)
    views: List[int]               # global view ids held locally (block first, then halo)
    neighbor_ids_local: torch.Tensor   # [V_local,k] int32 on the device, indices into ``views``
    begin: int
    end: int


def partition_views(n_views: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous, balanced block [begin, end) of reference views for ``rank``
    (the first ``n_views % world_size`` ranks get one extra view; a rank may get
    an empty block when world_size > n_views)."""
    if n_views < 0 or world_size <= 0 or not 0 <= rank < world_size:
        raise ValueError(f"bad partition request: V={n_views}, world={world_size}, rank={rank}")
    base, extra = divmod(n_views, world_size)
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def pack_partials(volume_sum: torch.Tensor, count: torch.Tensor,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[C,N] fp32 sums (any memory order) + [N] integer counts -> one flat fp32
    buffer ``[C*N + N]`` in the memory order of ``volume_sum``."""
    c, n = volume_sum.shape
    if count.numel() != n:
        raise ValueError("count must have one entry per voxel")
    mem = volume_sum if volume_sum.is_contiguous() else volume_sum.t()
    if not mem.is_contiguous():
        raise ValueError("volume_sum must be [C,N] contiguous or the transpose of a contiguous [N,C]")
    if out is None:
        out = torch.empty(c * n + n, dtype=torch.float32, device=volume_sum.device)
    out[:c * n].copy_(mem.reshape(-1))
    out[c * n:].copy_(count.reshape(-1))       # int -> fp32, exact for counts <= 2^24
    return out


def unpack_partials(buf: torch.Tensor, c: int, n: int, channels_first: bool = True):
    """Inverse of pack_partials -> (volume_sum logical [C,N] view, count int32 [N])."""
    vol = buf[:c * n].view(c, n) if channels_first else buf[:c * n].view(n, c).t()
    count = buf[c * n:].round().to(torch.int32)
    return vol, count


def allreduce_partials(buf: torch.Tensor, group=None) -> torch.Tensor:
    """Sum the packed partials over the group, in place.  One collective per
    scene; a no-op without an initialised process group (single-rank run)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return buf


class P2PVoxelReducer:
    """Sum-over-ranks + normalise of the voxel partials over NVLink peer memory
    (``mvsd_voxel_reduce_p2p``): one reduce-scatter / normalise / all-gather kernel
    bracketed by two cross-rank barriers, instead of an NCCL all-reduce followed by a
    normalise kernel.  Buffers are torch symmetric memory (P2P-mapped on every rank of
    the group); torch provides the allocation, the pointer exchange and the barrier
    kernel, the data path is ours.

        red = P2PVoxelReducer(C, N, channels_first, device, group)
        volume_mean, count = red(volume_sum, count)        # identical bits on every rank

    LIFETIME: the returned tensors are views of the reducer's peer-mapped result buffer, which the
    next call (this rank's and the peers' P2P stores) overwrites.  Clone them to keep them
    (``ShardedSceneForward`` does).
    """

    def __init__(self, channels: int, n_voxels: int, channels_first: bool, device, group=None):
        import torch.distributed._symmetric_memory as symm
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("P2PVoxelReducer needs an initialised process group")
        self.group = group if group is not None else dist.group.WORLD
        self.c, self.n, self.cfirst = int(channels), int(n_voxels), bool(channels_first)
        self.total = self.c * self.n
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        self.part = symm.empty(self.total + self.n, dtype=torch.float32, device=device)
        self.out = symm.empty(self.total + self.n, dtype=torch.float32, device=device)
        self.h_part = symm.rendezvous(self.part, self.group)
        self.h_out = symm.rendezvous(self.out, self.group)
        self.count_local = torch.empty(self.n, dtype=torch.int32, device=device)

    def partial_buffers(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """(sum, count) views of this rank's peer-mapped partial buffer, in the volume's
        memory order: pass them as ``out=`` / ``count_out=`` of the back-projection so the
        kernel writes its partials where the peers will read them."""
        shape = (self.c, self.n) if self.cfirst else (self.n, self.c)
        return self.part[:self.total].view(shape), self.part[self.total:].view(torch.int32)

    def __call__(self, volume_sum: torch.Tensor, count: torch.Tensor):
        mem = volume_sum if volume_sum.is_contiguous() else volume_sum.t()
        if not mem.is_contiguous() or mem.numel() != self.total:
            raise ValueError("volume_sum must be [C,N] contiguous or the transpose of a contiguous [N,C]")
        if mem.data_ptr() != self.part.data_ptr():           # not already written in place
            self.part[:self.total].copy_(mem.reshape(-1))
            self.part[self.total:].view(torch.int32).copy_(count.reshape(-1))
        self.h_part.barrier(channel=0)          # every rank's partials are complete and visible
        _lib.voxel_reduce_p2p(self.h_part.buffer_ptrs_dev, self.h_out.buffer_ptrs_dev, self.count_local,
                              world=self.world, rank=self.rank, channels=self.c, channels_first=self.cfirst)
        self.h_out.barrier(channel=0)           # every rank's slice has landed in every out buffer
        vol = self.out[:self.total]
        vol = vol.view(self.c, self.n) if self.cfirst else vol.view(self.n, self.c).t()
        return vol, self.out[self.total:].view(torch.int32)


class ShardedSceneForward:
    """Forward of one scene with the reference views split over the group.

        sharded = ShardedSceneForward(hot_path)            # an MVSDetHotPath
        out = sharded(feature, img_meta, cost_regularization)
        out["volume_mean"], out["count"]                   # identical on every rank

    ``feature`` holds ALL views on every rank.  The all-reduce runs on the
    current stream right after the local back-projection (there is nothing left
    to overlap it with inside one scene; a multi-scene caller overlaps it with
    the next scene's sweep by calling from a side stream)."""

    def __init__(self, hot_path, group=None, p2p: bool = True):
        self.hot = hot_path
        self.group = group
        self.p2p = p2p                 # combine over NVLink peer memory (default); False = NCCL all-reduce
        self._reducer = None

    def _world(self) -> Tuple[int, int]:
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(self.group), dist.get_world_size(self.group)
        return 0, 1

    def local_geometry(self, img_meta: dict, n_views: int, device) -> Optional[LocalGeometry]:
        """This rank's slice of the per-scene parameter block and its halo (host
        work, ~2 ms; a caller that revisits a scene passes it back in as
        ``geometry``)."""
        rank, world = self._world()
        begin, end = partition_views(n_views, world, rank)
        if end <= begin:
            return None
        geo = self.hot.geometry(img_meta, device, view_slice=slice(begin, end), prologue="host")
        views, nbr_local = halo_views(geo.neighbor_ids_host, begin, end)
        return LocalGeometry(geo=geo, views=views, neighbor_ids_local=nbr_local.to(device),
                             begin=begin, end=end)

    def _pack_local(self, feature: torch.Tensor, lg: LocalGeometry) -> torch.Tensor:
        """fp32 NCHW [V,C,H,W] -> channels-last buffer of the views in ``lg.views``
        (contiguous runs of views go through one transpose launch each)."""
        v, c, h, w = feature.shape
        dt = self.hot.feature_dtype
        if feature.dtype != torch.float32 or not feature.is_contiguous():
            return ops.pack_features(feature[lg.views], dt)       # already channels-last / bf16 inputs
        out = ops._empty_nhwc(len(lg.views), c, h, w, dt, feature.device)
        i = 0
        while i < len(lg.views):
            j = i
            while j + 1 < len(lg.views) and lg.views[j + 1] == lg.views[j] + 1:
                j += 1
            _lib.pack(feature[lg.views[i]:lg.views[j] + 1], out[i:j + 1])
            i = j + 1
        return out

    def local_partials(self, feature: torch.Tensor, img_meta: dict, cost_net: Callable,
                       geometry: Optional[LocalGeometry] = None, rank_world: Optional[Tuple[int, int]] = None,
                       partial_out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
        """This rank's contribution before the collective: (volume_sum logical
        [C,N], count int32 [N], (begin, end)).  ``rank_world`` overrides the
        process group (used by the single-GPU tests to play every rank)."""
        hot = self.hot
        rank, world = rank_world or self._world()
        v_all = feature.shape[0]
        begin, end = partition_views(v_all, world, rank)
        c = feature.shape[1]
        nx, ny, nz = hot.n_voxels
        n = nx * ny * nz
        dev = feature.device
        if end > begin:
            lg = geometry
            if lg is None:
                geo = hot.geometry(img_meta, dev, view_slice=slice(begin, end), prologue="host")
                views, nbr_local = halo_views(geo.neighbor_ids_host, begin, end)
                lg = LocalGeometry(geo, views, nbr_local.to(dev), begin, end)
            geo = lg.geo
            feat_cl = self._pack_local(feature, lg)            # block + halo only
            variance = ops.plane_sweep_variance(feat_cl, lg.neighbor_ids_local, geo.hom,
                                                geo.depth_values, out_dtype=hot.variance_dtype,
                                                ref_begin=0)
            cost_out = cost_net(variance)
            _, _, est_depth, est_dens, est_idx, _ = hot.hypotheses(cost_out)
            vol_sum, count = ops.backproject_aggregate(
                feat_cl[:end - begin], geo.points, geo.projection, est_depth, est_dens,
                hot.voxel_size[2], geo.height, geo.width, mode="sum",
                channels_first=hot.channels_first_volume,
                out=None if partial_out is None else partial_out[0],
                count_out=None if partial_out is None else partial_out[1])
        else:                                   # more ranks than views: contribute zeros
            shape = (c, n) if hot.channels_first_volume else (n, c)
            vol_sum = torch.zeros(shape, dtype=torch.float32, device=dev)
            vol_sum = vol_sum if hot.channels_first_volume else vol_sum.t()
            count = torch.zeros(n, dtype=torch.int32, device=dev)
        return vol_sum, count, (begin, end)

    def __call__(self, feature: torch.Tensor, img_meta: dict,
                 cost_regularization: Optional[Callable] = None, geometry=None) -> Dict[str, torch.Tensor]:
        hot = self.hot
        cost_net = cost_regularization or hot.cost_regularization
        if cost_net is None:
            raise ValueError("a cost_regularization callable is required (mvsdet.py:470)")
        c = feature.shape[1]
        nx, ny, nz = hot.n_voxels
        n = nx * ny * nz
        use_p2p = self.p2p and self._world()[1] > 1
        if use_p2p and self._reducer is None:
            self._reducer = P2PVoxelReducer(c, n, hot.channels_first_volume, feature.device, self.group)
        vol_sum, count, (begin, end) = self.local_partials(
            feature, img_meta, cost_net, geometry,
            partial_out=self._reducer.partial_buffers() if use_p2p else None)
        if use_p2p:
            # the reducer's result buffers are peer-mapped and reused by the next scene (peers store
            # into them): hand the caller its own copy, as the NCCL branch does (the reference
            # keeps every scene's volume in a list and stacks them later, mvsdet.py:681-696)
            volume_mean, count = self._reducer(vol_sum.detach(), count)
            volume_mean, count = volume_mean.clone(), count.clone()
        else:
            buf = pack_partials(vol_sum.detach(), count)
            allreduce_partials(buf, self.group)
            vol_sum, count = unpack_partials(buf, c, n, hot.channels_first_volume)
            volume_mean = ops.voxel_normalize(vol_sum, count)
        vm = (volume_mean.view(c, nx, ny, nz) if volume_mean.is_contiguous()
              else volume_mean.unflatten(1, (nx, ny, nz)))
        return dict(volume_mean=vm, valid=count.view(1, nx, ny, nz).float(), count=count,
                    view_range=(begin, end))


class ShardedScenePipeline:
    """Pre-allocated view-sharded forward (+ backward) of ONE large scene per rank -- the
    multi-GPU counterpart of ``pipeline.ScenePipeline`` (BASELINE.json configs[2] / [3]).

    Per rank: the fp32 FPN maps of its block of reference views plus the halo views (the pose
    neighbours it does not own) are resident ("pre-placed halos", SURVEY.md 8e caveat 1); the
    chain  pack -> plane sweep -> top-k -> back-projection(SUM)  writes the partial voxel sums and
    counts straight into a peer-mapped buffer and is replayed as ONE CUDA graph; the combine
    (sum over ranks + ``sum / (count + 1e-8)``, mvsdet.py:511-515, :681-682) is either
    ``mvsd_voxel_reduce_p2p`` over NVLink peer pointers between two symmetric-memory barriers
    ("p2p") or NCCL all-reduces + ``mvsd_voxel_normalize`` ("nccl").  Partial and result buffers are
    double-buffered, so in a stream of scenes the combine of scene i runs on a second CUDA
    stream under the sweep of scene i+1 (``forward_stream``).

    Backward (``backward``): every rank holds ``g_volume_mean`` (replicated, like the forward's
    result) and the gradient its cost-regularisation net returned for ITS views' variance;
    back-projection / prob-norm / top-k / sweep backward run locally into one fp32 accumulator
    over block + halo views, then each owner pulls its peers' halo contributions over NVLink
    (``mvsd_halo_reduce_p2p``): the result is dL/dfeature for the rank's own block -- a
    reduce-scatter of the scene's feature gradient with 2-4 views of traffic per rank.

    A hot path with ``deterministic=True`` makes the backward deterministic, as it makes the hot path's
    own: the scatter backwards add into an int64 fixed-point accumulator (``*_det`` kernels) and the
    owners pull with ``mvsd_halo_reduce_p2p_fixed``.  Every contribution to a view is then summed as an
    integer, in no particular order, so a rank's ``g_feature`` rows are the bits of the single-GPU
    deterministic gradient of those views, for any number of ranks and any split of the views."""
    deterministic = False          # fp32-RED backward

    def __init__(self, hot_path, cfg, device, group=None):
        import torch.distributed._symmetric_memory as symm
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("ShardedScenePipeline needs an initialised process group")
        self.hot, self.cfg, self.device = hot_path, cfg, torch.device(device)
        self.deterministic = bool(hot_path.deterministic)
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        self._symm = symm
        self.c = cfg.channels
        self.n = cfg.n_voxels[0] * cfg.n_voxels[1] * cfg.n_voxels[2]
        dev = self.device
        # per slot: the peer-mapped partial and result buffers and the p2p combine over them
        self._red = [P2PVoxelReducer(self.c, self.n, True, dev, self.group) for _ in range(2)]
        self.nccl_out = [torch.empty(self.c * self.n, dtype=torch.float32, device=dev) for _ in range(2)]
        # higher priority: the combine's barrier / reduce CTAs are dispatched as soon as SM slots free up,
        # ahead of the next scene's queued sweep CTAs (at equal priority they wait for the sweep's last wave)
        self.s_comm = torch.cuda.Stream(device=dev, priority=-1)
        self.s_aux = torch.cuda.Stream(device=dev, priority=-1)      # small backward kernels under the sweep
        self._ev_part = [None, None]      # partials of slot written (compute stream)
        self._ev_free = [None, None]      # slot's partial buffer consumed by the combine (comm stream)
        self._graphs = [None, None]
        self.lg: Optional[LocalGeometry] = None
        self._g_feat = None
        self._bwd_graphs: Dict = {}
        self._slot = 0

    # ------------------------------------------------------------------ setup
    def load(self, feature: torch.Tensor, cost_out: torch.Tensor, img_meta: dict,
             pose_clustered: bool = True) -> None:
        """Place this rank's share of a scene: ``feature`` [V,C,Hf,Wf] fp32 and ``cost_out``
        [V,2,D,Hf,Wf] (host or device, ALL views; only block + halo maps are kept).
        ``pose_clustered``: the ranks' blocks are pose clusters (``pose_order``) instead of index ranges;
        ``self.view_ids`` (also ``view_ids`` in ``forward``'s result) lists the views this rank owns, in the
        order of the rows ``backward`` takes and returns."""
        hot, cfg, dev = self.hot, self.cfg, self.device
        v_all = feature.shape[0]
        begin, end = partition_views(v_all, self.world, self.rank)
        if end <= begin:
            raise ValueError("more ranks than reference views")
        geo_full = hot.geometry(img_meta, "cpu", prologue="host")           # ids of the whole scene
        order = list(range(v_all))
        if pose_clustered:
            order = pose_order(img_meta["lidar2img"]["extrinsic"], geo_full.neighbor_ids_host, self.world)
            if order != list(range(v_all)):
                img_meta = permute_img_meta(img_meta, order)
                geo_full = hot.geometry(img_meta, "cpu", prologue="host")   # ids in the permuted numbering
        self.view_order = order
        self.view_ids = torch.tensor(order[begin:end], dtype=torch.int64)
        self.nbr_full = geo_full.neighbor_ids_host
        self.halo_counts = halo_counts(self.nbr_full, self.world)
        geo = hot.geometry(img_meta, dev, view_slice=slice(begin, end), prologue="host")
        views, nbr_local = halo_views(geo.neighbor_ids_host, begin, end)
        self.lg = LocalGeometry(geo, views, nbr_local.to(dev), begin, end)
        vl, vb = len(views), end - begin
        d, t = cfg.num_depth, cfg.topk
        hf, wf = cfg.feat_hw
        f32 = dict(dtype=torch.float32, device=dev)
        self.feature = feature[[order[i] for i in views]].to(dev, dtype=torch.float32).contiguous()
        self.cost_out = cost_out[order[begin:end]].to(dev, dtype=torch.float32).contiguous()
        self.feat_cl = ops._empty_nhwc(vl, self.c, hf, wf, hot.feature_dtype, dev)
        self.variance = ops._empty_ndhwc(vb, self.c, d, hf, wf, hot.variance_dtype, dev)
        self.est_depth = torch.empty((vb, t, hf, wf), **f32)
        self.est_dens = torch.empty((vb, t, hf, wf), **f32)
        self.est_idx = torch.empty((vb, t, hf, wf), dtype=torch.int64, device=dev)
        self.vl, self.vb = vl, vb
        self._graphs = [None, None]
        self._g_feat = None
        self._bwd_graphs = {}
        torch.cuda.synchronize(dev)

    def _enqueue_compute(self, slot: int) -> None:
        """pack -> sweep -> top-k -> back-projection(SUM) into the slot's partials; current stream; capturable."""
        cfg, lg, geo = self.cfg, self.lg, self.lg.geo
        _lib.pack(self.feature, self.feat_cl)
        _lib.plane_sweep_fwd(self.feat_cl, lg.neighbor_ids_local, geo.hom, geo.depth_values, self.variance)
        _lib.depth_topk_fwd(self.cost_out, None, None, self.est_depth, self.est_dens, self.est_idx, None,
                            near=cfg.near_far_range[0], interval=cfg.depth_interval)
        vol_sum, count = self._red[slot].partial_buffers()
        _lib.backproject_fwd(self.feat_cl, geo.points, geo.projection, self.est_depth, self.est_dens, vol_sum,
                             vs_z=cfg.voxel_size[2], mode=BP_SUM, height=geo.height, width=geo.width,
                             channels_first=True, count=count)

    def _compute(self, slot: int, use_graph: bool = True) -> None:
        if not use_graph:
            self._enqueue_compute(slot)
            return
        if self._graphs[slot] is None:
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._enqueue_compute(slot)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._enqueue_compute(slot)
            self._graphs[slot] = g
        self._graphs[slot].replay()

    def _combine(self, slot: int, mode: str) -> Dict[str, torch.Tensor]:
        """sum over ranks + normalise, on the current stream -> views of this slot's result buffers"""
        c, n = self.c, self.n
        nx, ny, nz = self.cfg.n_voxels
        red = self._red[slot]
        if mode == "p2p":
            vol, count = red(*red.partial_buffers())
            vol = vol.view(c, nx, ny, nz)
        elif mode == "nccl":
            vol_sum, cnt = red.partial_buffers()
            dist.all_reduce(vol_sum, op=dist.ReduceOp.SUM, group=self.group)
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=self.group)
            red.count_local.copy_(cnt)
            _lib.voxel_normalize(vol_sum, cnt, self.nccl_out[slot].view(c, n), channels_first=True)
            vol = self.nccl_out[slot].view(c, nx, ny, nz)
            count = red.count_local
        else:
            raise ValueError("mode must be 'p2p' or 'nccl'")
        return dict(volume_mean=vol, count=count, valid=count.view(1, nx, ny, nz),
                    view_range=(self.lg.begin, self.lg.end), view_ids=self.view_ids)

    # ------------------------------------------------------------------ forward
    def forward(self, mode: str = "p2p", use_graph: bool = True) -> Dict[str, torch.Tensor]:
        """One scene, everything on the current stream.  The returned tensors are views of
        reused (p2p: peer-mapped) buffers: valid until the next-but-one forward; clone to keep."""
        slot = self._slot
        self._slot ^= 1
        self._compute(slot, use_graph)
        res = self._combine(slot, mode)
        self._last_slot = slot
        return res

    def forward_stream(self, mode: str = "p2p", n_scenes: int = 8, use_graph: bool = True):
        """A stream of ``n_scenes`` scenes (the resident scene replayed): the chain of scene i+1 runs
        on the current stream while the combine of scene i runs on the communication stream."""
        cur = torch.cuda.current_stream()
        res = None
        for _ in range(n_scenes):
            slot = self._slot
            self._slot ^= 1
            if self._ev_free[slot] is not None:
                cur.wait_event(self._ev_free[slot])          # the slot's partials were consumed
            self._compute(slot, use_graph)
            ev = torch.cuda.Event()
            ev.record(cur)
            with torch.cuda.stream(self.s_comm):
                self.s_comm.wait_event(ev)
                res = self._combine(slot, mode)
                done = torch.cuda.Event()
                done.record(self.s_comm)
            self._ev_free[slot] = done
            self._last_slot = slot
        cur.wait_stream(self.s_comm)
        return res

    # ------------------------------------------------------------------ backward
    def backward(self, g_volume_mean: torch.Tensor, g_variance: torch.Tensor, use_graph: bool = True):
        """After ``forward`` (same slot): ``g_volume_mean`` [C,nx,ny,nz] (replicated on every rank),
        ``g_variance`` logical [Vb,C,D,Hf,Wf] in channels_last_3d for this rank's reference views (rows in
        the order of ``self.view_ids``).
        -> (g_feature [Vb,C,Hf,Wf] fp32 for the rank's own views ``self.view_ids``, g_cost_out [Vb,2,D,Hf,Wf])."""
        det = self.deterministic
        if not det:
            # its backward kernels RED in fp32, in an order that varies from run to run
            ops._alert_not_deterministic("ShardedScenePipeline.backward")
        cfg, lg, geo = self.cfg, self.lg, self.lg.geo
        dev = self.device
        vl, vb, c, n = self.vl, self.vb, self.c, self.n
        d, t = cfg.num_depth, cfg.topk
        hf, wf = cfg.feat_hw
        view_elems = hf * wf * c
        if self._g_feat is None:
            # every rank allocates for the same (maximum) number of local views: symmetric allocation
            vl_max = torch.tensor([vl], device=dev)
            dist.all_reduce(vl_max, op=dist.ReduceOp.MAX, group=self.group)
            # deterministic: the accumulator is int64 fixed point, g_pn_q too; the owned rows of the
            # accumulator are converted into g_feat_own after the pull (the halo rows are scratch)
            acc_dtype = torch.int64 if det else torch.float32
            self._g_feat = self._symm.empty(int(vl_max.item()) * view_elems, dtype=acc_dtype, device=dev)
            self._h_g = self._symm.rendezvous(self._g_feat, self.group)
            offs, src = halo_pull_table(self.nbr_full, self.world, self.rank)
            self._pull_offs, self._pull_src = offs.to(dev), src.to(dev)
            self._n_pull = int(src.shape[0])
            self.g_pn = torch.empty((vb, t, hf, wf), dtype=torch.float32, device=dev)
            self.g_est_dens = torch.zeros((vb, t, hf, wf), dtype=torch.float32, device=dev)
            self.g_cost_out = torch.empty((vb, 2, d, hf, wf), dtype=torch.float32, device=dev)
            self.g_feature = torch.empty((vb, c, hf, wf), dtype=torch.float32, device=dev)
            if det:
                self.g_pn_q = torch.empty((vb, t, hf, wf), dtype=torch.int64, device=dev)
                self.g_feat_own = torch.empty(vb * view_elems, dtype=torch.float32, device=dev)
        slot = self._last_slot
        g_vol = g_volume_mean.reshape(c, n).float().contiguous()
        gv = g_variance if g_variance.permute(0, 2, 3, 4, 1).is_contiguous() else \
            g_variance.contiguous(memory_format=torch.channels_last_3d)

        def enqueue_local():
            """zero-fills + back-projection / prob-norm / top-k / sweep backward into the accumulator;
            current stream; capturable (no allocation, no host sync)"""
            cur = torch.cuda.current_stream()
            hyp = (self.feat_cl, geo.points, geo.projection, self.est_depth, self.est_dens)
            self._g_feat.zero_()
            (self.g_pn_q if det else self.g_pn).zero_()
            # the three small kernels run on a higher-priority side stream under the sweep backward
            # (all of them RED into the same accumulator: the order does not matter)
            self.s_aux.wait_stream(cur)
            with torch.cuda.stream(self.s_aux):
                count = self._red[slot].count_local
                if det:
                    _lib.backproject_bwd_det(g_vol, count, *hyp, self._g_feat, self.g_pn_q, vs_z=cfg.voxel_size[2],
                                             height=geo.height, width=geo.width, channels_first=True)
                    _lib.fixed_to_float(self.g_pn_q, self.g_pn)
                else:
                    _lib.backproject_bwd(g_vol, *hyp, self._g_feat, self.g_pn, vs_z=cfg.voxel_size[2], mode=BP_MEAN,
                                         height=geo.height, width=geo.width, channels_first=True, count=count)
                _lib.prob_norm_bwd(self.est_dens, self.g_pn, self.g_est_dens, height=geo.height, width=geo.width)
                _lib.depth_topk_bwd(self.cost_out, self.est_idx, None, None, None, self.g_est_dens, None,
                                    self.g_cost_out, near=cfg.near_far_range[0], interval=cfg.depth_interval)
            sweep_bwd = _lib.plane_sweep_bwd_det if det else _lib.plane_sweep_bwd
            sweep_bwd(gv, self.feat_cl, lg.neighbor_ids_local, geo.hom, geo.depth_values, self._g_feat)
            cur.wait_stream(self.s_aux)

        # the local chain is replayed as one CUDA graph while the caller keeps handing in the same
        # gradient buffers (a training loop's pre-allocated ones); new pointers -> captured again
        key = (slot, g_vol.data_ptr(), gv.data_ptr(), gv.dtype)
        if use_graph and g_vol.data_ptr() == g_volume_mean.data_ptr():
            ent = self._bwd_graphs.get(key)
            if ent is None:
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    enqueue_local()
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize(dev)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    enqueue_local()
                if len(self._bwd_graphs) >= 4:
                    self._bwd_graphs.clear()
                ent = self._bwd_graphs[key] = (g, g_vol, gv)          # keeps the captured buffers alive
            ent[0].replay()
        else:
            enqueue_local()
        # owners pull the halo contributions of their peers
        self._h_g.barrier(channel=0)
        if self._n_pull:
            pull = _lib.halo_reduce_p2p_fixed if det else _lib.halo_reduce_p2p
            pull(self._h_g.buffer_ptrs_dev, self._pull_offs, self._pull_src, world=self.world, rank=self.rank,
                 view_elems=view_elems)
        self._h_g.barrier(channel=0)
        if det:
            _lib.fixed_to_float(self._g_feat[:vb * view_elems], self.g_feat_own)
            _lib.unpack(self.g_feat_own, self.g_feature)
        else:
            _lib.unpack(self._g_feat, self.g_feature)
        return self.g_feature, self.g_cost_out

    def close(self) -> None:
        """Drop the captured graphs and peer-mapped buffers before the process group goes away."""
        torch.cuda.synchronize(self.device)
        self._graphs = [None, None]
        self._bwd_graphs = {}
        self._g_feat = None
