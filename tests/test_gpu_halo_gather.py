"""The own-view forward of a view-sharded scene on the GPU.

``mvsd_halo_gather_p2p`` is checked with several "ranks" that are buffers of one device: bf16 and fp32 rows,
rows of 16-byte and of 8-byte multiples; the halo rows get the source bits and nothing else is written.  Playing
1-4 ranks on one device, each rank's own-row pack plus gather is the bits of the block + halo pack of the
replicated-input forward, and its partial voxel sums are those of that forward's chain.  Through the process
group (one rank here, two when two GPUs are visible): ``ShardedScenePipeline.load_own`` gives the bits of
``load`` (forward, stream of forwards, deterministic backward; the default backward within the bound of
tests/test_gpu_p2p.py), ``ShardedSceneForward.forward_own`` the bits of ``__call__``, and a stream of
scenes whose own-view input is rewritten between scenes gives every scene the bits of its single forward."""
import os
import socket

import pytest
import torch

from mvsdet_b200 import _lib, sharded
from mvsdet_b200.hotpath import MVSDetHotPath
from mvsdet_b200.scene import make_scene, tiny_config

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
BF16, F32 = torch.bfloat16, torch.float32


def _bits(x):
    return x.view(torch.int16) if x.dtype == BF16 else x.view(torch.int32)


# ---- the kernel, ranks played by buffers of one device ---------------------------------------------------------
@pytest.mark.parametrize("dtype,chw", [(BF16, (64, 6, 8)), (F32, (64, 6, 8)), (BF16, (132, 59, 81)),
                                       (F32, (132, 59, 81)), (BF16, (4, 1, 1))],
                         ids=["bf16-16B", "f32-16B", "bf16-8B-59x81x132", "f32-59x81x132", "bf16-8B-one-pixel"])
@pytest.mark.parametrize("rank", [0, 2])
def test_gather_copies_the_halo_rows_and_nothing_else(dtype, chw, rank):
    c, h, w = chw
    elems = c * h * w
    view_bytes = elems * torch.empty((), dtype=dtype).element_size()
    assert (view_bytes % 16 != 0) == (dtype == BF16 and (h * w) % 2 == 1 and c % 8 == 4)
    g = torch.Generator().manual_seed(elems + rank)
    bufs = [torch.randn((8 + q, elems), generator=g).to(DEV, dtype) for q in range(3)]
    before = [b.clone() for b in bufs]
    n_own = 2
    sources = [(q, row) for q, row in ((1, 2), (2, 0), (1, 0), (0, 4), (2, 6)) if q != rank]
    src = torch.tensor(sources, dtype=torch.int32, device=DEV)
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=DEV)
    _lib.halo_gather_p2p(ptrs.data_ptr(), src, world=3, rank=rank, n_own=n_own, view_bytes=view_bytes)
    torch.cuda.synchronize()
    mine = bufs[rank]
    for j, (q, row) in enumerate(sources):
        assert torch.equal(_bits(mine[n_own + j]), _bits(before[q][row])), f"halo row {j}"
    assert torch.equal(_bits(mine[:n_own]), _bits(before[rank][:n_own])), "own rows were written"
    end = n_own + len(sources)
    assert torch.equal(_bits(mine[end:]), _bits(before[rank][end:])), "rows past the halo rows were written"
    for q in range(3):
        if q != rank:
            assert torch.equal(_bits(bufs[q]), _bits(before[q])), f"peer {q} was written"


# ---- own-row pack + gather against the replicated-input pack and chain, ranks played on one device ------------
def _hot(cfg, feature_dtype=BF16, deterministic=False):
    return MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                         stride=cfg.stride, feature_dtype=feature_dtype, deterministic=deterministic)


@pytest.mark.parametrize("pose_clustered", [False, True], ids=["index", "pose"])
@pytest.mark.parametrize("feature_dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_own_pack_plus_gather_is_the_block_and_halo_pack(world, feature_dtype, pose_clustered):
    cfg = tiny_config(n_views=9, channels=64)
    scene = make_scene(cfg, seed=5, with_grads=False)
    hot = _hot(cfg, feature_dtype)
    runner = sharded.ShardedSceneForward(hot)
    order, meta, nbr = sharded._view_plan(hot, scene["img_meta"], world, pose_clustered)
    feature = scene["feature"].to(DEV)[order].contiguous()             # the sharded numbering
    cost = scene["cost_out"].to(DEV)[order].contiguous()
    c, hf, wf = feature.shape[1:]
    rows = sharded._max_local_views(nbr, world)
    view_elems = c * hf * wf
    flat = [torch.full((rows * view_elems,), 7.0, device=DEV).to(feature_dtype) for _ in range(world)]
    packed, lgs = [], []
    for r in range(world):
        b, e = sharded.partition_views(cfg.n_views, world, r)
        geo = hot.geometry(meta, DEV, view_slice=slice(b, e), prologue="host")
        views, nbr_local = sharded.halo_views(geo.neighbor_ids_host, b, e)
        lgs.append(sharded.LocalGeometry(geo, views, nbr_local.to(DEV), b, e))
        packed.append(flat[r][:len(views) * view_elems].view(len(views), hf, wf, c).permute(0, 3, 1, 2))
        _lib.pack(feature[b:e], packed[r][:e - b])                    # each owner packs its own views only
    ptrs = torch.tensor([f.data_ptr() for f in flat], dtype=torch.int64, device=DEV)
    for r, lg in enumerate(lgs):
        src = sharded.halo_gather_table(nbr, world, r).to(DEV)
        if src.shape[0]:
            _lib.halo_gather_p2p(ptrs.data_ptr(), src, world=world, rank=r, n_own=lg.end - lg.begin,
                                 view_bytes=view_elems * feature.new_empty((), dtype=feature_dtype).element_size())
    for r, lg in enumerate(lgs):
        want = runner._pack_local(feature, lg)
        assert torch.equal(_bits(packed[r].contiguous(memory_format=torch.channels_last)),
                           _bits(want.contiguous(memory_format=torch.channels_last))), f"rank {r}: packed rows"
        net = (lambda b, e: (lambda var: cost[b:e]))(lg.begin, lg.end)
        vol_a, cnt_a, _ = runner.local_partials(feature, meta, net, geometry=lg, rank_world=(r, world))
        vol_b, cnt_b = runner._chain(packed[r], lg, net, None)
        torch.cuda.synchronize()
        assert torch.equal(cnt_a, cnt_b), f"rank {r}: counts"
        assert torch.equal(vol_a.view(torch.int32), vol_b.view(torch.int32)), f"rank {r}: partial sums"


# ---- through the process group: load_own against load, forward_own against __call__ ---------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _same(a, b):
    return bool(torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32)))


def _stream_of(pipe, inputs, mode):
    """a stream of scenes scheduled as ``forward_stream`` schedules them, with the resident own-view input
    rewritten in place on the compute stream before each scene -> cloned (volume_mean, count) per scene"""
    cur = torch.cuda.current_stream()
    outs = []
    for x in inputs:
        slot = pipe._slot
        pipe._slot ^= 1
        if pipe._ev_free[slot] is not None:
            cur.wait_event(pipe._ev_free[slot])
        pipe.feature.copy_(x)
        pipe._compute(slot)
        ev = torch.cuda.Event()
        ev.record(cur)
        with torch.cuda.stream(pipe.s_comm):
            pipe.s_comm.wait_event(ev)
            res = pipe._combine(slot, mode)
            outs.append((res["volume_mean"].clone(), res["count"].clone()))
            done = torch.cuda.Event()
            done.record(pipe.s_comm)
        pipe._ev_free[slot] = done
    cur.wait_stream(pipe.s_comm)
    torch.cuda.synchronize()
    return outs


def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cfg = tiny_config(n_views=9, channels=64)
        scene = make_scene(cfg, seed=5)
        feature, cost, meta = scene["feature"], scene["cost_out"], scene["img_meta"]
        g_vol, g_var = scene["g_volume_mean"].to(dev), scene["g_variance"].to(dev)
        ok = {}
        for det in (True, False):
            hot = _hot(cfg, deterministic=det)
            for pose in (True, False):
                key = f"{'det' if det else 'default'}-{'pose' if pose else 'index'}"
                a = sharded.ShardedScenePipeline(hot, cfg, dev)
                a.load(feature, cost, meta, pose_clustered=pose)
                ids = a.view_ids
                b = sharded.ShardedScenePipeline(hot, cfg, dev)
                with pytest.raises(ValueError, match="one row per owned view"):
                    b.load_own(feature[ids][1:], cost[ids][1:], meta, pose_clustered=pose)
                b.load_own(feature[ids], cost[ids], meta, pose_clustered=pose)
                _, want_ids = sharded.owned_views(hot, meta, world, rank, pose_clustered=pose)
                ok[key + "-view_ids"] = bool(torch.equal(b.view_ids, ids) and torch.equal(want_ids, ids))
                ok[key + "-resident"] = tuple(b.feature.shape) == (len(ids), cfg.channels, *cfg.feat_hw)
                for mode in ("p2p", "nccl"):
                    for n in (1, 2, 3):                      # both slots, then the first again
                        ra, rb = a.forward(mode), b.forward(mode)
                        ok[f"{key}-{mode}-fwd{n}"] = _same(ra["volume_mean"], rb["volume_mean"]) and \
                            bool(torch.equal(ra["count"], rb["count"]))
                    ra = a.forward_stream(mode, 4)
                    rb = b.forward_stream(mode, 4)
                    torch.cuda.synchronize()
                    ok[f"{key}-{mode}-stream"] = _same(ra["volume_mean"], rb["volume_mean"]) and \
                        bool(torch.equal(ra["count"], rb["count"]))
                own = ids.to(dev)
                gv = g_var[own].contiguous(memory_format=torch.channels_last_3d)
                a.forward("p2p")
                b.forward("p2p")
                for _ in range(2):                           # twice: the accumulators are reused
                    ga, gca = a.backward(g_vol, gv)
                    ga, gca = ga.clone(), gca.clone()
                    gb, gcb = b.backward(g_vol, gv)
                torch.cuda.synchronize()
                if det:
                    ok[key + "-bwd"] = _same(ga, gb) and _same(gca, gcb)
                else:
                    scale = float(ga.abs().max())
                    ok[key + "-bwd"] = (float((ga - gb).abs().max()) <= 1e-4 * scale
                                        and float((gca - gcb).abs().max()) <= 1e-4)
                if det and pose:
                    # reuse: own-view input A, B, A, B in a stream of scenes, rewritten in place between scenes
                    g = torch.Generator().manual_seed(11)
                    sets = [feature[ids].to(dev), torch.randn(feature[ids].shape, generator=g).to(dev)]
                    for mode in ("p2p", "nccl"):
                        single = []
                        for x in sets:
                            b.feature.copy_(x)
                            r = b.forward(mode)
                            single.append((r["volume_mean"].clone(), r["count"].clone()))
                        outs = _stream_of(b, [sets[0], sets[1], sets[0], sets[1]], mode)
                        ok[f"reuse-{mode}"] = all(_same(v, single[i % 2][0]) and torch.equal(c, single[i % 2][1])
                                                  for i, (v, c) in enumerate(outs))
                        ok[f"reuse-{mode}-differs"] = not _same(single[0][0], single[1][0])
                a.close()
                b.close()
        # the one-call form: forward_own over index blocks is __call__ on the whole scene's maps
        hot = _hot(cfg)
        fdev, cdev = feature.to(dev), cost.to(dev)
        for p2p in (True, False):
            run = sharded.ShardedSceneForward(hot, p2p=p2p)
            begin, end = sharded.partition_views(cfg.n_views, world, rank)
            for n in range(2):                               # the buffers are reused scene after scene
                want = run(fdev, meta, cost_regularization=lambda var: cdev[begin:end])
                got = run.forward_own(fdev[begin:end], meta, cost_regularization=lambda var: cdev[begin:end],
                                      pose_clustered=False)
                ok[f"forward_own-p2p{int(p2p)}-{n}"] = (
                    _same(want["volume_mean"], got["volume_mean"]) and bool(torch.equal(want["count"], got["count"]))
                    and got["view_range"] == want["view_range"]
                    and got["view_ids"].tolist() == list(range(begin, end)))
            _, ids = sharded.owned_views(hot, meta, world, rank)
            got = run.forward_own(fdev[ids.to(dev)], meta, cost_regularization=lambda var: cdev[ids.to(dev)])
            ok[f"forward_own-pose-p2p{int(p2p)}-count"] = bool(torch.equal(got["count"], want["count"])) and \
                torch.equal(got["view_ids"], ids)
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


def _spawn(world):
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    for rank in range(world):
        bad = [k for k, v in ret[rank].items() if not v]
        assert not bad, f"rank {rank} of {world}: {bad}"
        assert len(ret[rank]) >= 50


def test_own_view_forms_one_rank_are_the_replicated_input_bits():
    _spawn(1)


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_own_view_forms_two_gpus_are_the_replicated_input_bits():
    _spawn(2)
