"""The deterministic training-step forms on the GPU.

``ScenePipeline(deterministic=True)``, eager and replayed from a CUDA graph, gives the bits of
``MVSDetHotPath(deterministic=True)``'s autograd backward on the same inputs (both add the same fixed-point
contributions with integer REDs and convert once), the forward bits of the default pipeline, and
gradients within 1e-5 of the rms of the default pipeline's fp32-RED ones; it steps and captures under
``torch.use_deterministic_algorithms(True)``.

``mvsd_halo_reduce_p2p_fixed`` is checked with several "ranks" that are buffers of one device: exact
integer sums near the int64 range, untouched rows, the same bits for a permuted pull table.  The property it
gives the view-sharded backward -- a rank's feature-gradient rows are the bits of the whole-scene
deterministic gradient, whatever the number of ranks -- is checked by playing 1-4 ranks' local chains on
one device, and with two GPUs through ``ShardedScenePipeline`` itself (skipped below two)."""
import os
import socket

import pytest
import torch

from mvsdet_b200 import _lib, sharded
from mvsdet_b200.hotpath import MVSDetHotPath
from mvsdet_b200.pipeline import ScenePipeline
from mvsdet_b200.scene import SceneConfig, make_scene, tiny_config
from test_det_routes_cpu import det_flag  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
BF16, F32 = torch.bfloat16, torch.float32
DTYPES = [(BF16, F32), (F32, F32), (BF16, BF16)]
DTYPE_IDS = ["bf16", "f32", "bf16-bf16var"]


def _hot(cfg, feature_dtype=BF16, variance_dtype=F32, deterministic=True):
    return MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                         stride=cfg.stride, feature_dtype=feature_dtype, variance_dtype=variance_dtype,
                         deterministic=deterministic)


def _autograd(scene, geo, feature_dtype, variance_dtype):
    """whole-scene forward + backward of MVSDetHotPath(deterministic=True) -> (feat.grad, cost.grad, out)"""
    hot = _hot(scene["cfg"], feature_dtype, variance_dtype)
    feat = scene["feature"].to(DEV).requires_grad_(True)
    cost = scene["cost_out"].to(DEV).requires_grad_(True)
    out = hot(feat, scene["img_meta"], cost_regularization=lambda var: cost, geometry=geo)
    torch.autograd.backward([out["variance"], out["volume_mean"]],
                            [scene["g_variance"].to(DEV), scene["g_volume_mean"].to(DEV)])
    return feat.grad, cost.grad, out


def _pipeline(scene, geo, feature_dtype, variance_dtype, deterministic):
    pipe = ScenePipeline(scene["cfg"], DEV, feature_dtype=feature_dtype, variance_dtype=variance_dtype,
                         deterministic=deterministic)
    pipe.set_geometry(geo)
    pipe.load_scene(scene)
    return pipe


def _outputs(pipe):
    return {n: getattr(pipe, n).clone() for n in ("volume_mean", "count", "g_feature", "g_cost_out")}


def _near(det, red, what):
    d, r = det.double(), red.double()
    rms = float(r.pow(2).mean().sqrt())
    err = (d - r).abs()
    assert rms > 0 and float(err.max()) <= 1e-5 * rms, f"{what}: max err {float(err.max()):.3e}, rms {rms:.3e}"


def _check_pipeline(scene, feature_dtype, variance_dtype):
    geo = _hot(scene["cfg"]).geometry(scene["img_meta"], DEV)
    pipe = _pipeline(scene, geo, feature_dtype, variance_dtype, True)
    pipe.step()                                           # eager, overlapped streams
    torch.cuda.synchronize()
    runs = [_outputs(pipe)]
    graph = pipe.capture()
    for _ in range(3):
        pipe.g_feature.zero_()
        pipe.g_cost_out.zero_()
        graph.replay()
        torch.cuda.synchronize()
        runs.append(_outputs(pipe))
    for i, r in enumerate(runs[1:], 1):
        for n in r:
            assert torch.equal(r[n], runs[0][n]), f"replay {i}: {n} bits differ from the eager step"
    g_feat, g_cost, out = _autograd(scene, geo, feature_dtype, variance_dtype)
    torch.cuda.synchronize()
    assert torch.equal(runs[0]["g_feature"], g_feat), "g_feature differs from the deterministic autograd route"
    assert torch.equal(runs[0]["g_cost_out"], g_cost), "g_cost_out differs from the deterministic autograd route"
    del graph, pipe
    ref = _pipeline(scene, geo, feature_dtype, variance_dtype, False)
    ref.step()
    torch.cuda.synchronize()
    assert torch.equal(runs[0]["volume_mean"], ref.volume_mean) and torch.equal(runs[0]["count"], ref.count)
    assert torch.equal(runs[0]["volume_mean"], out["volume_mean"].reshape(ref.volume_mean.shape))
    _near(runs[0]["g_feature"], ref.g_feature, "g_feature against the fp32-RED step")
    _near(runs[0]["g_cost_out"], ref.g_cost_out, "g_cost_out against the fp32-RED step")


@pytest.mark.parametrize("feature_dtype,variance_dtype", DTYPES, ids=DTYPE_IDS)
def test_deterministic_step_is_the_autograd_bits_small(feature_dtype, variance_dtype):
    _check_pipeline(make_scene(tiny_config(n_views=6, channels=64), seed=31), feature_dtype, variance_dtype)


def test_deterministic_step_is_the_autograd_bits_benchmarked_shape():
    """V=20, 60x80x256, D=12, bf16 features: the shape bench.py times"""
    _check_pipeline(make_scene(SceneConfig(n_views=20), seed=3), BF16, F32)


def test_deterministic_step_runs_and_captures_under_the_flag(det_flag):  # noqa: F811
    scene = make_scene(tiny_config(n_views=5, channels=32), seed=33)
    geo = _hot(scene["cfg"]).geometry(scene["img_meta"], DEV)
    pipe = _pipeline(scene, geo, BF16, F32, True)
    pipe.step()
    torch.cuda.synchronize()
    want = _outputs(pipe)
    det_flag(True)
    pipe.step()
    graph = pipe.capture()
    graph.replay()
    torch.cuda.synchronize()
    det_flag(False)
    got = _outputs(pipe)
    for n in want:
        assert torch.equal(got[n], want[n]), n


# ---- the fixed-point halo pull, with the "ranks" as buffers of one device ----------------------------------
VIEW_ELEMS = 40_000                     # 20 000 16-byte vectors: more than 64 CTAs of 256 cover, grid-stride
# owner rank 0 of a world of 3; rank q holds 4 + q local views; (peer rank, peer view) per owned view
PULLS = [[(1, 2), (2, 0)], [], [(1, 0)], [(2, 1), (1, 1), (2, 5)]]


def _table(pulls):
    offs = [0]
    src = []
    for lst in pulls:
        src.extend(lst)
        offs.append(len(src))
    return (torch.tensor(offs, dtype=torch.int32, device=DEV),
            torch.tensor(src, dtype=torch.int32, device=DEV).reshape(-1, 2))


def _ranks(dtype, world=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    if dtype == torch.int64:
        bound = 2 ** 62 // world                          # |sum| stays below 2^63 for up to `world` + 1 terms
        return [torch.randint(-bound, bound, (4 + q, VIEW_ELEMS), generator=g, dtype=torch.int64).to(DEV)
                for q in range(world)]
    return [torch.randn((4 + q, VIEW_ELEMS), generator=g).to(DEV) for q in range(world)]


def _pull(bufs, pulls, fixed, rank=0):
    ptrs = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=DEV)
    offs, src = _table(pulls)
    launch = _lib.halo_reduce_p2p_fixed if fixed else _lib.halo_reduce_p2p
    launch(ptrs.data_ptr(), offs, src, world=len(bufs), rank=rank, view_elems=VIEW_ELEMS)
    torch.cuda.synchronize()


def test_fixed_halo_pull_is_the_exact_integer_sum():
    bufs = _ranks(torch.int64)
    before = [b.cpu() for b in bufs]
    _pull(bufs, PULLS, fixed=True)
    for d, lst in enumerate(PULLS):
        want = before[0][d].clone()
        for q, j in lst:
            want += before[q][j]
        assert torch.equal(bufs[0][d].cpu(), want), f"owned view {d}"
    assert torch.equal(bufs[0][len(PULLS):].cpu(), before[0][len(PULLS):]), "rows past the owned views"
    for q in (1, 2):
        assert torch.equal(bufs[q].cpu(), before[q]), f"peer {q} was written"
    # values near the range: a negative and a positive sum of four terms each close to +-2^62 / 3
    assert float(before[0].abs().max()) > 0.99 * 2 ** 62 / 3


def test_fixed_halo_pull_does_not_depend_on_the_table_order():
    a, b = _ranks(torch.int64, seed=1), _ranks(torch.int64, seed=1)
    _pull(a, PULLS, fixed=True)
    _pull(b, [lst[::-1] for lst in PULLS], fixed=True)
    assert torch.equal(a[0], b[0])


def test_fp32_halo_pull_adds_in_table_order():
    """the fp32 pull (shares the kernel body): own + sources in table order, one rounding each"""
    bufs = _ranks(torch.float32, seed=2)
    before = [b.cpu() for b in bufs]
    _pull(bufs, PULLS, fixed=False)
    for d, lst in enumerate(PULLS):
        want = before[0][d].clone()
        for q, j in lst:
            want = want + before[q][j]
        assert torch.equal(bufs[0][d].cpu(), want), f"owned view {d}"
    assert torch.equal(bufs[0][len(PULLS):].cpu(), before[0][len(PULLS):])


# ---- the view-sharded feature gradient is the single-GPU one, bit for bit, for any number of ranks --------
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_sharded_feature_gradient_is_the_whole_scene_bits_on_one_device(world):
    """each rank's local chain of ShardedScenePipeline.backward (sweep + back-projection backward into an int64
    accumulator over block + halo views), then every owner's fixed-point pull and conversion, played on one
    device with the whole scene's geometry rows; the owned rows equal the whole-scene autograd gradient"""
    from mvsdet_b200 import ops
    cfg = tiny_config(n_views=9, channels=64)
    scene = make_scene(cfg, seed=5)
    geo = _hot(cfg).geometry(scene["img_meta"], DEV)
    g_feat, _, out = _autograd(scene, geo, BF16, F32)
    nbr = geo.neighbor_ids.cpu().to(torch.int64)
    hf, wf = cfg.feat_hw
    c, t = cfg.channels, cfg.topk
    ve = hf * wf * c
    feat_cl = ops.pack_features(scene["feature"].to(DEV), BF16)
    g_var = scene["g_variance"].to(DEV).contiguous(memory_format=torch.channels_last_3d)
    g_vol = scene["g_volume_mean"].to(DEV).reshape(c, -1).contiguous()
    est_depth, est_dens, count = out["est_depth"].detach(), out["est_densities"].detach(), out["count"]
    accs, blocks = [], []
    for r in range(world):
        b, e = sharded.partition_views(cfg.n_views, world, r)
        views, nbr_local = sharded.halo_views(nbr[b:e], b, e)
        local = torch.stack([feat_cl[v] for v in views]).contiguous(memory_format=torch.channels_last)
        acc = torch.zeros((len(views), hf, wf, c), dtype=torch.int64, device=DEV)
        g_pn_q = torch.zeros((e - b, t, hf, wf), dtype=torch.int64, device=DEV)
        _lib.plane_sweep_bwd_det(g_var[b:e], local, nbr_local.to(DEV), geo.hom[b:e], geo.depth_values[b:e],
                                 acc.permute(0, 3, 1, 2))
        _lib.backproject_bwd_det(g_vol, count, local, geo.points, geo.projection[b:e], est_depth[b:e],
                                 est_dens[b:e], acc.permute(0, 3, 1, 2), g_pn_q, vs_z=cfg.voxel_size[2],
                                 height=geo.height, width=geo.width, channels_first=True)
        accs.append(acc)
        blocks.append((b, e))
    ptrs = torch.tensor([a.data_ptr() for a in accs], dtype=torch.int64, device=DEV)
    for r, (b, e) in enumerate(blocks):
        offs, src = sharded.halo_pull_table(nbr, world, r)
        if src.shape[0]:
            _lib.halo_reduce_p2p_fixed(ptrs.data_ptr(), offs.to(DEV), src.to(DEV), world=world, rank=r,
                                       view_elems=ve)
    for r, (b, e) in enumerate(blocks):
        g_own = torch.empty((e - b, hf, wf, c), dtype=torch.float32, device=DEV)
        _lib.fixed_to_float(accs[r][:e - b], g_own)
        g = torch.empty((e - b, c, hf, wf), dtype=torch.float32, device=DEV)
        _lib.unpack(g_own, g)
        torch.cuda.synchronize()
        assert torch.equal(g, g_feat[b:e]), f"rank {r} of {world}: g_feature rows differ from the whole scene"


# ---- ShardedScenePipeline over a deterministic hot path ------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cfg = tiny_config(n_views=9, channels=64)
        scene = make_scene(cfg, seed=5)
        hot = _hot(cfg)
        feat = scene["feature"].to(dev).requires_grad_(True)
        cost = scene["cost_out"].to(dev).requires_grad_(True)
        g_vol, g_var = scene["g_volume_mean"].to(dev), scene["g_variance"].to(dev)
        # the whole scene on one GPU, with the host prologue the sharded pipeline builds its geometry with
        whole = hot(feat, scene["img_meta"], cost_regularization=lambda var: cost,
                    geometry=hot.geometry(scene["img_meta"], dev, prologue="host"))
        torch.autograd.backward([whole["variance"], whole["volume_mean"]], [g_var, g_vol])
        ok = {}
        for pose_clustered in (True, False):
            pipe = sharded.ShardedScenePipeline(hot, cfg, dev)
            pipe.load(scene["feature"], scene["cost_out"], scene["img_meta"], pose_clustered=pose_clustered)
            own = pipe.view_ids.to(dev)
            pipe.forward("p2p")
            for _ in range(2):                              # twice: the accumulators are reused
                g_feature, g_cost = pipe.backward(g_vol, g_var[own].contiguous(memory_format=torch.channels_last_3d))
            torch.cuda.synchronize()
            ok["pose" if pose_clustered else "index"] = (
                pipe.deterministic, bool(torch.equal(g_feature, feat.grad[own])),
                bool(torch.equal(g_cost, cost.grad[own])))
            pipe.close()
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


def _spawn(world):
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    for rank in range(world):
        for key, (det, g_ok, c_ok) in ret[rank].items():
            assert det, "the pipeline did not take deterministic from the hot path"
            assert g_ok, f"rank {rank} ({key} blocks): g_feature differs from the whole-scene deterministic rows"
            assert c_ok, f"rank {rank} ({key} blocks): g_cost_out differs from the whole-scene deterministic rows"


def test_sharded_pipeline_one_rank_is_the_whole_scene_bits():
    _spawn(1)


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_pipeline_two_gpus_is_the_whole_scene_bits():
    _spawn(2)
