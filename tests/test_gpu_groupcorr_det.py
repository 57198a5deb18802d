"""The deterministic group-correlation backward (mvsd_plane_sweep_groupcorr_bwd_det[_px]): against the
oracle's autograd at the bar of test_gpu_groupcorr.py, against the fp32-RED form, bit for bit from run
to run, independent of how the reference views are split into calls, per-view planes equal to constant
per-pixel maps, and MVSDetHotPath(cost_volume="group_correlation", deterministic=True) end to end."""
import pytest
import torch

import test_gpu_depth_map_sweep as S
from mvsdet_b200.scene import make_scene, tiny_config
from oracle import mvsdet_oracle as O

pytestmark = pytest.mark.gpu

DEV = S.DEV
_close = S._close


def _ragged(**kw):
    h, w = 13, 21
    return tiny_config(img_shape=(4 * h - 1, 4 * w), pad_shape=(4 * h, 4 * w), ori_shape=(16 * h - 4, 16 * w), **kw)


def _depth(geo, cfg, per_pixel):
    return S._depth_maps(geo.depth_values, *cfg.feat_hw) if per_pixel else geo.depth_values.cpu()


def _det_vs_oracle(cfg, seed, k, groups, feature_dtype, per_pixel):
    from mvsdet_b200 import ops
    feature, _, geo, all_proj = S._setup(cfg, seed, k, feature_dtype)
    depth = _depth(geo, cfg, per_pixel)
    f_ref = feature.clone().requires_grad_(True)
    want = S._oracle_corr(f_ref, all_proj, geo.neighbor_ids_ref(), depth, groups)
    g = torch.randn(want.shape, generator=torch.Generator().manual_seed(seed + 1))
    want_g, = torch.autograd.grad(want, f_ref, g)
    f_dev = feature.to(DEV).requires_grad_(True)
    feat_cl, sink = ops.pack_features(f_dev, feature_dtype, sink=True, deterministic=True)
    assert sink.deterministic
    got = ops.plane_sweep_group_correlation(feat_cl, geo.neighbor_ids, geo.hom, depth.to(DEV), groups,
                                            grad_sink=sink)
    got_g, = torch.autograd.grad(got, f_dev, g.to(DEV))
    torch.cuda.synchronize()
    return got_g, want_g


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("channels,groups", [(32, 8), (64, 8), (256, 8), (128, 1), (132, 33)],
                         ids=["width4", "width8", "width32", "width128", "C132_G33"])
def test_det_backward_matches_oracle(channels, groups, feature_dtype):
    cfg = tiny_config(n_views=5, channels=channels, num_depth=6)
    got_g, want_g = _det_vs_oracle(cfg, 31 + channels, 2, groups, feature_dtype, False)
    _close(got_g, want_g, f"C={channels} G={groups}: dL/dfeature")


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("per_pixel", [False, True], ids=["planes", "maps"])
@pytest.mark.parametrize("k", [1, 2, 3])
def test_det_backward_ragged_map_matches_oracle(k, per_pixel, feature_dtype):
    """13 x 21 map (H not a multiple of the 2-row CTA patch, W not of the 4-pixel one), k = 1, 2, 3"""
    cfg = _ragged(n_views=5, channels=64, num_depth=5)
    got_g, want_g = _det_vs_oracle(cfg, 50 + k, k, 8, feature_dtype, per_pixel)
    _close(got_g, want_g, f"k={k} per_pixel={per_pixel}: dL/dfeature")


# ---- the raw entry points -------------------------------------------------------------------------
def _raw_inputs(feature_dtype, per_pixel, k=2, channels=256, groups=8, seed=3):
    """-> (packed features, geometry, depth_values on the device, upstream gradient in the forward's layout)"""
    from mvsdet_b200 import ops
    cfg = _ragged(n_views=6, channels=channels, num_depth=8)
    feature, _, geo, _ = S._setup(cfg, seed, k, feature_dtype)
    feat = ops.pack_features(feature.to(DEV), feature_dtype)
    depth = _depth(geo, cfg, per_pixel).to(DEV)
    h, w = cfg.feat_hw
    g = torch.randn((cfg.n_views, k, cfg.num_depth, h, w, groups), generator=torch.Generator().manual_seed(seed))
    return feat, geo, depth, g.to(DEV).permute(0, 1, 5, 2, 3, 4)


def _det(g, feat, nbr, hom, depth, q=None, ref_begin=0):
    from mvsdet_b200 import _lib
    if q is None:
        q = torch.zeros(feat.shape, dtype=torch.int64, device=DEV).contiguous(memory_format=torch.channels_last)
    _lib.plane_sweep_groupcorr_bwd_det(g, feat, nbr, hom, depth, q, ref_begin=ref_begin)
    return q


def _red(g, feat, nbr, hom, depth):
    from mvsdet_b200 import _lib
    r = torch.zeros(feat.shape, device=DEV).contiguous(memory_format=torch.channels_last)
    _lib.plane_sweep_groupcorr_bwd(g, feat, nbr, hom, depth, r)
    return r


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("per_pixel", [False, True], ids=["planes", "maps"])
@pytest.mark.parametrize("variant", [0, 1], ids=["default_kernel", "pixel_kernel"])
def test_det_backward_is_close_to_fp32_red(variant, per_pixel, feature_dtype):
    """within 1e-5 of the rms of the fp32-RED result, both for the kernel the fp32-RED form picks by
    default (bf16, k = 2: the run kernel) and for its pixel kernel (test hook mvsd_set_tuning(5, 1))"""
    from mvsdet_b200 import _lib, ops
    feat, geo, depth, g = _raw_inputs(feature_dtype, per_pixel)
    old = _lib.set_tuning(5, variant)
    try:
        red = _red(g, feat, geo.neighbor_ids, geo.hom, depth)
    finally:
        _lib.set_tuning(5, old)
    det = ops.fixed_to_float(_det(g, feat, geo.neighbor_ids, geo.hom, depth))
    torch.cuda.synchronize()
    rms = float(red.double().pow(2).mean().sqrt())
    err = float((det.double() - red.double()).abs().max())
    assert rms > 0 and err <= 1e-5 * rms, (err, rms)


@pytest.mark.parametrize("per_pixel", [False, True], ids=["planes", "maps"])
def test_det_backward_is_bit_reproducible(per_pixel):
    from mvsdet_b200 import ops
    feat, geo, depth, g = _raw_inputs(torch.bfloat16, per_pixel)
    runs = []
    for _ in range(3):
        q = _det(g, feat, geo.neighbor_ids, geo.hom, depth)
        runs.append((q, ops.fixed_to_float(q)))
    torch.cuda.synchronize()
    assert bool(runs[0][0].ne(0).any())
    for q, f in runs[1:]:
        assert torch.equal(q, runs[0][0]), "int64 accumulator differs between runs"
        assert torch.equal(f, runs[0][1]), "fp32 gradient differs between runs"


@pytest.mark.parametrize("per_pixel", [False, True], ids=["planes", "maps"])
def test_det_backward_is_independent_of_the_reference_split(per_pixel):
    """reference views [0, a) and [a, V) swept in two calls, in either order, into one accumulator give
    the whole-scene call's bits"""
    feat, geo, depth, g = _raw_inputs(torch.float32, per_pixel, k=3)
    nbr, hom = geo.neighbor_ids, geo.hom
    whole = _det(g, feat, nbr, hom, depth)
    a = 2
    parts = {"lo": slice(0, a), "hi": slice(a, nbr.shape[0])}
    for order in (("lo", "hi"), ("hi", "lo")):
        q = None
        for name in order:
            s = parts[name]
            q = _det(g[s], feat, nbr[s], hom[s], depth[s], q, ref_begin=s.start)
        torch.cuda.synchronize()
        assert torch.equal(q, whole), f"split {order}"


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("k", [1, 2, 3])
def test_constant_map_gives_the_per_view_accumulator(k, feature_dtype):
    feat, geo, planes, g = _raw_inputs(feature_dtype, False, k=k, seed=60 + k)
    h, w = feat.shape[2:]
    maps = planes[:, :, None, None].expand(-1, -1, h, w).contiguous()
    a = _det(g, feat, geo.neighbor_ids, geo.hom, planes)
    b = _det(g, feat, geo.neighbor_ids, geo.hom, maps)
    torch.cuda.synchronize()
    assert bool(a.ne(0).any()) and torch.equal(a, b)


# ---- the hot path -----------------------------------------------------------------------------------
def test_hot_path_deterministic_group_correlation():
    """MVSDetHotPath(cost_volume="group_correlation", deterministic=True) with the small cost net of
    test_gpu_groupcorr.py: bit-identical feature and cost gradients over three runs, at that test's
    tolerance of the oracle"""
    from mvsdet_b200.hotpath import MVSDetHotPath
    cfg = tiny_config(n_views=5, channels=32, num_depth=8)
    scene = make_scene(cfg, 13)
    groups = 8
    torch.manual_seed(0)
    net = torch.nn.Conv3d(2 * groups, 2, 3, padding=1)
    hf, wf = cfg.feat_hw

    def cost_net_for(mod):
        def run(vol):
            ramp = torch.arange(cfg.num_depth, dtype=torch.float32, device=vol.device).view(1, 1, -1, 1, 1)
            return mod(vol.reshape(vol.shape[0], 2 * groups, cfg.num_depth, hf, wf)) * 3.0 + 0.01 * ramp
        return run

    f_ref = scene["feature"].clone().requires_grad_(True)
    corr = O.scene_group_correlation(f_ref, scene["img_meta"], near_far_range=cfg.near_far_range,
                                     num_depth=cfg.num_depth, num_groups=groups, stride=cfg.stride)
    want_cost = cost_net_for(net)(corr)
    want_cost.retain_grad()
    want = O.hot_path(f_ref, scene["img_meta"], lambda var: want_cost, near_far_range=cfg.near_far_range,
                      num_depth=cfg.num_depth, topk=cfg.topk, n_voxels=cfg.n_voxels, voxel_size=cfg.voxel_size,
                      stride=cfg.stride)
    g_vol = scene["g_volume_mean"]
    want["volume_mean"].backward(g_vol)
    net_d = torch.nn.Conv3d(2 * groups, 2, 3, padding=1).to(DEV)
    net_d.load_state_dict(net.state_dict())
    mod = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        stride=cfg.stride, cost_volume="group_correlation", num_groups=groups, deterministic=True)
    want_cost_d = want_cost.detach().to(DEV)

    def cost_net_cuda(vol):
        # the oracle's values, the CUDA net's gradient (see test_gpu_groupcorr.py)
        cost = cost_net_for(net_d)(vol)
        return cost + (want_cost_d - cost).detach()

    runs = []
    with torch.backends.cudnn.flags(allow_tf32=False, deterministic=True):
        for _ in range(3):
            f_dev = scene["feature"].to(DEV).requires_grad_(True)
            res = mod(f_dev, scene["img_meta"], cost_regularization=cost_net_cuda)
            res["cost_out"].retain_grad()
            res["volume_mean"].backward(g_vol.to(DEV))
            torch.cuda.synchronize()
            runs.append((f_dev.grad.clone(), res["cost_out"].grad.clone()))
    for gf, gc in runs[1:]:
        assert torch.equal(gf, runs[0][0]), "feature gradient differs between runs"
        assert torch.equal(gc, runs[0][1]), "cost gradient differs between runs"
    _close(runs[0][0], f_ref.grad, "deterministic dL/dfeature", rtol=1e-3, atol_scale=1e-3)
    _close(runs[0][1], want_cost.grad, "deterministic dL/dcost_out", rtol=1e-3, atol_scale=1e-3)


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_deterministic_second_correlation_sweep_is_bit_reproducible(feature_dtype):
    """a per-view and a per-pixel correlation sweep into the same fixed-point accumulator: bit-identical
    feature gradients run to run, and the fp32-RED accumulation to 1e-5"""
    from mvsdet_b200 import ops
    cfg = tiny_config(n_views=5, channels=64, num_depth=6)
    feature, _, geo, _ = S._setup(cfg, 5, 2, feature_dtype)
    depth = S._depth_maps(geo.depth_values, *cfg.feat_hw).to(DEV)
    gen = torch.Generator().manual_seed(9)
    g1 = torch.randn((cfg.n_views, 2, 8, cfg.num_depth, *cfg.feat_hw), generator=gen).to(DEV)
    g2 = torch.randn(g1.shape, generator=gen).to(DEV)

    def grads(deterministic):
        f = feature.to(DEV).requires_grad_(True)
        feat_cl, sink = ops.pack_features(f, feature_dtype, sink=True, deterministic=deterministic)
        c1 = ops.plane_sweep_group_correlation(feat_cl, geo.neighbor_ids, geo.hom, geo.depth_values, 8,
                                               grad_sink=sink)
        c2 = ops.plane_sweep_group_correlation(feat_cl, geo.neighbor_ids, geo.hom, depth, 8, grad_sink=sink)
        gf, = torch.autograd.grad((c1 * g1).sum() + (c2 * g2).sum(), f)
        torch.cuda.synchronize()
        return gf

    a, b, c = grads(True), grads(True), grads(True)
    assert torch.equal(a, b) and torch.equal(a, c)
    _close(a, grads(False), "deterministic vs fp32-RED", rtol=1e-5, atol_scale=1e-5)
