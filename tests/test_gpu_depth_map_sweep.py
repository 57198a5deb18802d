"""Per-pixel depth hypotheses [V,D,H,W] in the fused plane sweeps (homo_warping's branch,
mvs_models/module.py:130-133): variance and group-correlation volumes, forward and backward,
against the oracle's warp with autograd, at the bar of test_gpu_parity.py
(1e-4 * rms + 1e-4 * |ref|, bf16 features at the fp32 bar on the same rounded features).

The depth maps vary in x and in y, and alternate rows differ by 30 %: the row hand-off of the
bf16 backward kernel decides from the adjacent rows' samples, so a hand-off decided with the wrong
row's depth sends a weighted vector to a row that does not have the tap and fails here."""
import numpy as np
import pytest
import torch

from mvsdet_b200.scene import make_scene, tiny_config
from oracle import mvsdet_oracle as O

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda")


def _close(a, b, what, rtol=1e-4, atol_scale=1e-4):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    rms = float(b.pow(2).mean().sqrt())
    err = (a - b).abs()
    bad = err > atol_scale * rms + rtol * b.abs()
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())}/{bad.numel()} out of tolerance, "
                                 f"max abs err {float(err.max()):.3e} (rms {rms:.3e})")


def _setup(cfg, seed, k, feature_dtype):
    """-> (feature [V,C,Hf,Wf] fp32 (bf16-rounded for bf16), module, device geometry, oracle projections)"""
    from mvsdet_b200.hotpath import MVSDetHotPath
    scene = make_scene(cfg, seed, with_grads=False)
    feature = scene["feature"]
    if feature_dtype == torch.bfloat16:
        feature = feature.to(torch.bfloat16).float()            # both sides see the same rounded features
    mod = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        stride=cfg.stride, feature_dtype=feature_dtype, num_neighbors=k)
    geo = mod.geometry(scene["img_meta"], DEV)
    meta = scene["img_meta"]
    ratio = meta["ori_shape"][0] / (meta["img_shape"][0] / cfg.stride)
    w2c = torch.as_tensor(np.array(meta["lidar2img"]["extrinsic"]))
    k_feat = O.feature_intrinsics(torch.as_tensor(np.array(meta["lidar2img"]["intrinsic"])), ratio)
    all_proj = torch.matmul(k_feat if k_feat.dim() == 3 else k_feat.unsqueeze(0).repeat(w2c.shape[0], 1, 1), w2c)
    return feature, mod, geo, all_proj


def _depth_maps(planes, hf, wf):
    """[V,D] planes -> per-pixel hypotheses [V,D,hf,wf] that vary smoothly in x and y and jump by 30 %
    between adjacent rows"""
    ys = torch.arange(hf, dtype=torch.float32).view(hf, 1)
    xs = torch.arange(wf, dtype=torch.float32).view(1, wf)
    f = (1.0 + 0.3 * (ys % 2)) * (1.0 + 0.08 * torch.sin(0.7 * xs + 0.4 * ys))
    return (planes.cpu()[:, :, None, None] * f).contiguous()


def _warped(feature, all_proj, nbr, j, depth):
    v = feature.shape[0]
    return O.homo_warping(feature[nbr[:, j]], all_proj[nbr[:, j]], all_proj[:v], depth)


def _oracle_variance(feature, all_proj, nbr, depth):
    """the oracle's plane_sweep_variance (mvsdet.py:439-467) with the per-pixel warp"""
    k, d = nbr.shape[1], depth.shape[1]
    ref = feature.unsqueeze(2).repeat(1, 1, d, 1, 1)
    s1, s2 = ref, ref ** 2
    for j in range(k):
        w = _warped(feature, all_proj, nbr, j, depth)
        s1 = s1 + w
        s2 = s2 + w ** 2
    return s2 / (k + 1) - (s1 / (k + 1)) ** 2


def _oracle_corr(feature, all_proj, nbr, depth, groups):
    """the oracle's group_correlation (mvs_models/lss_fpn.py:496-503) with the per-pixel warp"""
    v, c, h, w = feature.shape
    d = depth.shape[1]
    ref = feature.reshape(v, groups, c // groups, h, w)
    costs = []
    for j in range(nbr.shape[1]):
        warped = _warped(feature, all_proj, nbr, j, depth).reshape(v, groups, c // groups, d, h, w)
        costs.append(torch.mean(ref.unsqueeze(3) * warped, axis=2))
    return torch.stack(costs, dim=1)


def _variance_vs_oracle(cfg, seed, k, feature_dtype):
    from mvsdet_b200 import ops
    feature, mod, geo, all_proj = _setup(cfg, seed, k, feature_dtype)
    depth = _depth_maps(geo.depth_values, *cfg.feat_hw)
    f_ref = feature.clone().requires_grad_(True)
    want = _oracle_variance(f_ref, all_proj, geo.neighbor_ids_ref(), depth)
    g = torch.randn(want.shape, generator=torch.Generator().manual_seed(seed + 1))
    want_g, = torch.autograd.grad(want, f_ref, g)
    f_dev = feature.to(DEV).requires_grad_(True)
    feat_cl, sink = ops.pack_features(f_dev, feature_dtype, sink=True)
    got = mod.variance(feat_cl, geo, grad_sink=sink, depth_values=depth.to(DEV))
    got_g, = torch.autograd.grad(got, f_dev, g.to(DEV))
    torch.cuda.synchronize()
    return got, want.detach(), got_g, want_g


# (k, test hook key 5): k = 1, 2 through the run kernels (bf16: hand-off, fp32: lean), k = 3 and the
# k = 2 test hook through the generic pixel kernel
KERNELS = [(1, 0), (2, 0), (3, 0), (2, 1)]


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("k,variant", KERNELS, ids=["k1", "k2", "k3", "k2_generic"])
def test_variance_ragged_map_matches_oracle(k, variant, feature_dtype):
    """13 x 21 map: H not a multiple of the 4-row CTA, W not a multiple of the 8-pixel run"""
    from mvsdet_b200 import _lib
    h, w = 13, 21
    cfg = tiny_config(n_views=5, channels=40, num_depth=6, img_shape=(4 * h - 1, 4 * w),
                      pad_shape=(4 * h, 4 * w), ori_shape=(16 * h - 4, 16 * w))
    old = _lib.set_tuning(5, variant)
    try:
        got, want, got_g, want_g = _variance_vs_oracle(cfg, 41 + k, k, feature_dtype)
    finally:
        _lib.set_tuning(5, old)
    _close(got, want, f"k={k} variant {variant}: variance")
    _close(got_g, want_g, f"k={k} variant {variant}: dL/dfeature")


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("channels", [256, 132])
def test_variance_channel_counts_match_oracle(channels, feature_dtype):
    cfg = tiny_config(n_views=4, channels=channels, num_depth=5)
    got, want, got_g, want_g = _variance_vs_oracle(cfg, 7 + channels, 2, feature_dtype)
    _close(got, want, f"C={channels}: variance")
    _close(got_g, want_g, f"C={channels}: dL/dfeature")


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("k", [1, 2, 3])
def test_constant_map_gives_the_per_view_sweep(k, feature_dtype):
    """[V,D] planes broadcast to [V,D,H,W]: the forward and the deterministic backward are bit-identical
    to the per-view call, the fp32-RED backward agrees to summation order"""
    from mvsdet_b200 import _lib, ops
    h, w = 13, 21
    cfg = tiny_config(n_views=5, channels=256, num_depth=6, img_shape=(4 * h - 1, 4 * w),
                      pad_shape=(4 * h, 4 * w), ori_shape=(16 * h - 4, 16 * w))
    feature, mod, geo, _ = _setup(cfg, 60 + k, k, feature_dtype)
    planes = geo.depth_values
    maps = planes[:, :, None, None].expand(-1, -1, h, w).contiguous()
    feat = ops.pack_features(feature.to(DEV), feature_dtype)
    nbr, hom = geo.neighbor_ids, geo.hom
    var_v = ops.plane_sweep_variance(feat, nbr, hom, planes)
    var_p = ops.plane_sweep_variance(feat, nbr, hom, maps)
    assert torch.equal(var_v, var_p)
    g = torch.randn(var_v.shape, generator=torch.Generator().manual_seed(k)).to(DEV)
    g = g.contiguous(memory_format=torch.channels_last_3d)
    acc = {}
    for name, dv in (("view", planes), ("pixel", maps)):
        q = torch.zeros(feat.shape, dtype=torch.int64, device=DEV).contiguous(memory_format=torch.channels_last)
        _lib.plane_sweep_bwd_det(g, feat, nbr, hom, dv, q)
        r = torch.zeros(feat.shape, device=DEV).contiguous(memory_format=torch.channels_last)
        _lib.plane_sweep_bwd(g, feat, nbr, hom, dv, r)
        acc[name] = (q, r)
    torch.cuda.synchronize()
    assert torch.equal(acc["view"][0], acc["pixel"][0]), "deterministic backward"
    _close(acc["pixel"][1], acc["view"][1], "fp32-RED backward", rtol=1e-5, atol_scale=1e-6)


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
def test_deterministic_second_sweep_is_bit_reproducible(feature_dtype):
    """MVSDetHotPath(deterministic=True): a per-view sweep and a per-pixel second sweep into the same
    fixed-point accumulator give bit-identical feature gradients run to run, and match the
    fp32-RED accumulation"""
    from mvsdet_b200 import ops
    cfg = tiny_config(n_views=5, channels=64, num_depth=6)
    feature, mod, geo, _ = _setup(cfg, 5, 2, feature_dtype)
    depth = _depth_maps(geo.depth_values, *cfg.feat_hw).to(DEV)
    gen = torch.Generator().manual_seed(9)
    g1 = torch.randn((cfg.n_views, cfg.channels, cfg.num_depth, *cfg.feat_hw), generator=gen).to(DEV)
    g2 = torch.randn(g1.shape, generator=gen).to(DEV)

    def grads(deterministic):
        mod.deterministic = deterministic
        f = feature.to(DEV).requires_grad_(True)
        feat_cl, sink = ops.pack_features(f, feature_dtype, sink=True, deterministic=mod.deterministic)
        v1 = mod.variance(feat_cl, geo, grad_sink=sink)
        v2 = mod.variance(feat_cl, geo, grad_sink=sink, depth_values=depth)
        gf, = torch.autograd.grad((v1 * g1).sum() + (v2 * g2).sum(), f)
        torch.cuda.synchronize()
        return gf

    a, b = grads(True), grads(True)
    assert torch.equal(a, b)
    _close(a, grads(False), "deterministic vs fp32-RED", rtol=1e-5, atol_scale=1e-5)


@pytest.mark.parametrize("feature_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("k", [1, 2])
def test_group_correlation_matches_oracle(k, feature_dtype):
    from mvsdet_b200 import ops
    h, w, groups = 13, 21, 8
    cfg = tiny_config(n_views=5, channels=256, num_depth=6, img_shape=(4 * h - 1, 4 * w),
                      pad_shape=(4 * h, 4 * w), ori_shape=(16 * h - 4, 16 * w))
    feature, mod, geo, all_proj = _setup(cfg, 80 + k, k, feature_dtype)
    depth = _depth_maps(geo.depth_values, h, w)
    f_ref = feature.clone().requires_grad_(True)
    want = _oracle_corr(f_ref, all_proj, geo.neighbor_ids_ref(), depth, groups)
    g = torch.randn(want.shape, generator=torch.Generator().manual_seed(k))
    want_g, = torch.autograd.grad(want, f_ref, g)
    f_dev = feature.to(DEV).requires_grad_(True)
    feat_cl, sink = ops.pack_features(f_dev, feature_dtype, sink=True)
    got = ops.plane_sweep_group_correlation(feat_cl, geo.neighbor_ids, geo.hom, depth.to(DEV), groups,
                                            grad_sink=sink)
    got_g, = torch.autograd.grad(got, f_dev, g.to(DEV))
    torch.cuda.synchronize()
    _close(got, want.detach(), f"k={k}: correlation volumes")
    _close(got_g, want_g, f"k={k}: dL/dfeature")


def _small_sweep():
    from mvsdet_b200 import ops
    cfg = tiny_config(n_views=4, channels=32, num_depth=4)
    feature, mod, geo, _ = _setup(cfg, 3, 2, torch.float32)
    feat = ops.pack_features(feature.to(DEV), torch.float32).detach().requires_grad_(True)
    depth = _depth_maps(geo.depth_values, *cfg.feat_hw).to(DEV)
    return cfg, feat, geo, depth


def test_opcheck_with_per_pixel_depth():
    from mvsdet_b200 import library as L
    _, feat, geo, depth = _small_sweep()
    checks = ("test_schema", "test_faketensor", "test_autograd_registration")
    torch.library.opcheck(L.plane_sweep_variance, (feat, geo.neighbor_ids, geo.hom, depth), test_utils=checks)
    torch.library.opcheck(L.plane_sweep_group_correlation, (feat, geo.neighbor_ids, geo.hom, depth, 4),
                          test_utils=checks)


def test_dispatcher_op_matches_autograd_function():
    from mvsdet_b200 import library as L, ops
    _, feat, geo, depth = _small_sweep()
    a = ops.plane_sweep_variance(feat, geo.neighbor_ids, geo.hom, depth)
    b = L.plane_sweep_variance(feat, geo.neighbor_ids, geo.hom, depth)
    assert torch.equal(a, b)
    a = ops.plane_sweep_group_correlation(feat, geo.neighbor_ids, geo.hom, depth, 4)
    b = L.plane_sweep_group_correlation(feat, geo.neighbor_ids, geo.hom, depth, 4)
    assert torch.equal(a, b)


def test_bad_depth_shapes_raise():
    """anything but [V,D] or [V,D,H,W] with the feature map's H,W is a ValueError (a [V,D,H',W'] tensor
    used to pass the check and be read as [V,D] planes)"""
    from mvsdet_b200 import library as L, ops
    cfg, feat, geo, depth = _small_sweep()
    v, d = geo.depth_values.shape
    h, w = cfg.feat_hw
    bad = [torch.ones(v, d, h + 1, w, device=DEV), torch.ones(v, d, h, device=DEV),
           torch.ones(v, d, h, w, 1, device=DEV)]
    nbr, hom = geo.neighbor_ids, geo.hom
    for dv in bad:
        for fn in (lambda: ops.plane_sweep_variance(feat, nbr, hom, dv),
                   lambda: L.plane_sweep_variance(feat, nbr, hom, dv),
                   lambda: ops.plane_sweep_group_correlation(feat, nbr, hom, dv, 4),
                   lambda: L.plane_sweep_group_correlation(feat, nbr, hom, dv, 4)):
            with pytest.raises(ValueError):
                fn()
