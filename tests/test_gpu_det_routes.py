"""torch.use_deterministic_algorithms(True) on every route of the package that scatters in its backward:
pre-packed fp32 / bf16 features without a gradient sink, the stand-alone operators, back-projection in
SUM and PER_VIEW mode and with strided hypotheses, ``functional.homo_warping`` and
``functional.backproject_Weigh``, the dispatcher ops and ``MVSDetHotPath(dispatcher_ops=True)``.

Under the flag each route's feature gradient is bit-identical over three runs and within 1e-5 of the rms
of its fp32-RED form (flag off); its forward outputs are the bits of the flag-off run.  The new
back-projection modes stay within the fixed-point bounds of tests/ref64.py, and a sink made with
``deterministic=False`` gives, under the flag, the bits of the explicit ``deterministic=True`` call.
References are computed outside the flag (the flag makes cuBLAS need a workspace setting and fills
``torch.empty`` with NaN); only the product path runs under it."""
import pytest
import torch

import bp_cases as BC
import ref64
import test_gpu_backproject_edges as E
import test_gpu_depth_map_sweep as S
from mvsdet_b200 import functional as F_
from mvsdet_b200 import library as L
from mvsdet_b200 import ops
from mvsdet_b200.scene import tiny_config
from test_det_routes_cpu import det_flag  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


def _sweep_scene(channels=64, seed=7):
    cfg = tiny_config(n_views=5, channels=channels, num_depth=6)
    feature, _, geo, all_proj = S._setup(cfg, seed, 2, torch.float32)
    return cfg, feature, geo, all_proj


def _bp_scene(seed=5):
    return BC.random_scene(6, 132, 3, 170, seed=seed)


def _grad_like(t, seed):
    return torch.randn(t.shape, generator=torch.Generator().manual_seed(seed)).to(DEV)


def _leaf(t, dtype=torch.float32):
    """a channels-last leaf (features that arrive already packed)"""
    return ops.pack_features(t.to(DEV), dtype).detach().requires_grad_(True)


# Each route: () -> (forward outputs, gradients), on inputs built outside the flag.
def _routes():
    cfg, feature, geo, all_proj = _sweep_scene()
    depth_px = S._depth_maps(geo.depth_values, *cfg.feat_hw).to(DEV)
    nbr, hom = geo.neighbor_ids, geo.hom
    sc = _bp_scene()
    pts, proj = sc["points"].to(DEV), sc["projection"].to(DEV)
    depth_b, dens_b = sc["depth"].to(DEV), sc["prob"].to(DEV)
    strided = E._hyp(sc["prob"], True)
    strided_depth = E._hyp(sc["depth"], True)

    def sweep(dtype, depth, corr=False):
        def f():
            x = _leaf(feature, dtype)
            out = ops.plane_sweep_group_correlation(x, nbr, hom, depth, 4) if corr else \
                ops.plane_sweep_variance(x, nbr, hom, depth)
            return (out,), torch.autograd.grad(out, x, _grad_like(out, 1))
        return f

    def bp(mode, cfirst, hyp=(depth_b, dens_b)):
        def f():
            x = _leaf(sc["feat"])
            dens = hyp[1].detach().clone().requires_grad_(True) if hyp[1].is_contiguous() else \
                hyp[1].detach().requires_grad_(True)
            vol, cnt = ops.backproject_aggregate(x, pts, proj, hyp[0], dens, sc["vs_z"], sc["h"], sc["w"],
                                                 mode=mode, channels_first=cfirst)
            return (vol, cnt), torch.autograd.grad(vol, (x, dens), _grad_like(vol, 2))
        return f

    def homo_warping():
        j = nbr[:, 0].long().cpu()
        src = feature[j].to(DEV).requires_grad_(True)
        out = F_.homo_warping(src, all_proj[j], all_proj[:nbr.shape[0]], geo.depth_values.cpu())
        return (out,), torch.autograd.grad(out, src, _grad_like(out, 3))

    def backproject_weigh():
        v, t, h, w = sc["prob"].shape[0], sc["prob"].shape[1], sc["h"], sc["w"]
        feat = sc["feat"][:, :, :h, :w].to(DEV).requires_grad_(True)
        dr = E._crop(depth_b, sc).permute(0, 2, 3, 1).reshape(v, h * w, 1, t)
        pr = E._crop(dens_b, sc).permute(0, 2, 3, 1).reshape(v, h * w, 1, t).detach().requires_grad_(True)
        vol, valid, _, _ = F_.backproject_Weigh(feat, pts.view(3, -1, 1, 1), proj, dr, [0.1, 0.1, sc["vs_z"]], pr)
        return (vol, valid), torch.autograd.grad(vol, (feat, pr), _grad_like(vol, 4))

    def dispatcher(dtype):
        def f():
            x = _leaf(feature, dtype)
            var = L.plane_sweep_variance(x, nbr, hom, depth_px)
            cor = L.plane_sweep_group_correlation(x, nbr, hom, geo.depth_values, 4)
            xb = _leaf(sc["feat"], dtype)
            vol, cnt = L.backproject_aggregate(xb, pts, proj, depth_b, dens_b, sc["vs_z"], sc["h"], sc["w"], True)
            g = torch.autograd.grad((var, cor, vol), (x, xb), (_grad_like(var, 5), _grad_like(cor, 6),
                                                              _grad_like(vol, 7)))
            return (var, cor, vol, cnt), g
        return f

    return {
        "variance-prepacked-f32": sweep(torch.float32, geo.depth_values),
        "variance-prepacked-bf16": sweep(torch.bfloat16, geo.depth_values),
        "variance-px-prepacked": sweep(torch.float32, depth_px),
        "correlation-prepacked": sweep(torch.float32, geo.depth_values, corr=True),
        "correlation-px-prepacked-bf16": sweep(torch.bfloat16, depth_px, corr=True),
        "bp-mean-no-sink": bp("mean", True),
        "bp-sum-cfirst": bp("sum", True),
        "bp-sum-clast": bp("sum", False),
        "bp-sum-strided": bp("sum", True, (strided_depth, strided)),
        "homo-warping": homo_warping,
        "backproject-weigh": backproject_weigh,
        "dispatcher-f32": dispatcher(torch.float32),
        "dispatcher-bf16": dispatcher(torch.bfloat16),
    }


ROUTES = [
    "variance-prepacked-f32", "variance-prepacked-bf16", "variance-px-prepacked", "correlation-prepacked",
    "correlation-px-prepacked-bf16", "bp-mean-no-sink", "bp-sum-cfirst", "bp-sum-clast", "bp-sum-strided",
    "homo-warping", "backproject-weigh", "dispatcher-f32", "dispatcher-bf16"]


def _near(det, red, what):
    """within 1e-5 of the rms of the fp32-RED gradient.  A bf16 gradient is within one bf16 ulp of its
    partial sums instead: the two forms' fp32 sums may round to neighbouring bf16 values, and autograd adds
    the bf16 partials of several consumers (bounded here by |red| + rms)."""
    d, r = det.double(), red.double()
    rms = float(r.pow(2).mean().sqrt())
    tol = 1e-5 * rms + (2.0 ** -7 * (r.abs() + rms) if det.dtype == torch.bfloat16 else 0.0)
    err = (d - r).abs()
    assert rms > 0 and not bool((err > tol).any()), f"{what}: max err {float(err.max()):.3e}, rms {rms:.3e}"


@pytest.mark.parametrize("route", ROUTES)
def test_route_is_deterministic_under_the_flag(route, det_flag):  # noqa: F811
    fn = _routes()[route]
    det_flag(False)
    outs_red, grads_red = fn()
    det_flag(True)
    runs = [fn() for _ in range(3)]
    torch.cuda.synchronize()
    det_flag(False)
    outs, grads = runs[0]
    for i, (o, g) in enumerate(runs[1:], 1):
        for a, b in zip(g, grads):
            assert torch.equal(a, b), f"{route}: run {i} gradient bits differ"
    for a, b in zip(outs, outs_red):
        assert torch.equal(a, b), f"{route}: forward outputs differ with the flag on"
    for n, (a, b) in enumerate(zip(grads, grads_red)):
        assert a.dtype == b.dtype and a.shape == b.shape
        _near(a, b, f"{route}: gradient {n} against the fp32-RED form")


# ---- the new back-projection modes against fp64, through the sink and without one -----------------------
@pytest.mark.parametrize("case,fdt", [(c, f) for c in ("sum-cfirst", "sum-clast", "sum-strided") for f in ("f32", "bf16")]
                         + [("per-view", "f32")])
def test_new_backproject_modes_within_fixed_point_bounds(case, fdt, det_flag):  # noqa: F811
    """run under the flag: SUM goes through a sink made with deterministic=False (int64 under the flag),
    PER_VIEW through backproject_per_view, which has no sink and so returns the gradient in the features'
    dtype (fp32 here: a bf16 gradient is outside an fp32 bound, in either form)"""
    sc = BC.random_scene(17, 256, 3, 190, seed=40 + len(case), bf16=fdt == "bf16")
    mode = ref64.PER_VIEW if case == "per-view" else ref64.SUM
    det_flag(True)
    got = E.run(sc, mode, case != "sum-clast", E.FDT[fdt], strided=case == "sum-strided", g_seed=3)
    again = E.run(sc, mode, case != "sum-clast", E.FDT[fdt], strided=case == "sum-strided", g_seed=3)
    det_flag(False)
    assert torch.equal(got["g_feat"], again["g_feat"]) and torch.equal(got["g_prob"], again["g_prob"])
    E.check(sc, got, E.reference(sc, mode, got["g_out"]), f"{case} {fdt} under the flag", det=True)


@pytest.mark.parametrize("mode", [ref64.MEAN, ref64.SUM])
def test_sink_under_the_flag_gives_the_explicit_bits(mode, det_flag):  # noqa: F811
    sc = _bp_scene(seed=11)
    explicit = E.run(sc, mode, True, det=True, g_seed=8)
    det_flag(True)
    flagged = E.run(sc, mode, True, det=False, g_seed=8)
    det_flag(False)
    assert torch.equal(flagged["g_feat"], explicit["g_feat"]) and torch.equal(flagged["g_prob"], explicit["g_prob"])


def test_variance_sink_under_the_flag_gives_the_explicit_bits(det_flag):  # noqa: F811
    cfg, feature, geo, _ = _sweep_scene(seed=9)

    def grad(det):
        x = feature.to(DEV).requires_grad_(True)
        feat_cl, sink = ops.pack_features(x, torch.bfloat16, sink=True, deterministic=det)
        var = ops.plane_sweep_variance(feat_cl, geo.neighbor_ids, geo.hom, geo.depth_values, grad_sink=sink)
        return torch.autograd.grad(var, x, _grad_like(var, 9))[0]
    explicit = grad(True)
    det_flag(True)
    flagged = grad(False)
    det_flag(False)
    assert torch.equal(flagged, explicit)


def test_explicit_deterministic_with_prepacked_features():
    """deterministic=True gives pre-packed features a fixed-point sink too (no flag): bit-reproducible"""
    cfg, feature, geo, _ = _sweep_scene(seed=13)
    sc = _bp_scene(seed=13)

    def grad():
        x = _leaf(feature, torch.bfloat16)
        feat_cl, sink = ops.pack_features(x, torch.bfloat16, sink=True, deterministic=True)
        assert sink is not None and feat_cl.dtype == torch.bfloat16
        var = ops.plane_sweep_variance(feat_cl, geo.neighbor_ids, geo.hom, geo.depth_values, grad_sink=sink)
        g = torch.autograd.grad(var, x, _grad_like(var, 10))[0]
        assert sink.buf is None and g.dtype == torch.bfloat16
        return g
    a, b = grad(), grad()
    assert torch.equal(a, b)
    xb = _leaf(sc["feat"])
    feat_cl, sink = ops.pack_features(xb, torch.float32, sink=True, deterministic=True)
    vol, _ = ops.backproject_aggregate(feat_cl, sc["points"].to(DEV), sc["projection"].to(DEV),
                                       sc["depth"].to(DEV), sc["prob"].to(DEV), sc["vs_z"], sc["h"], sc["w"],
                                       grad_sink=sink)
    g = torch.autograd.grad(vol, xb, _grad_like(vol, 11))[0]
    assert g.dtype == torch.float32 and bool(g.abs().sum() > 0)


def test_opcheck_dispatcher_ops_under_the_flag(det_flag):  # noqa: F811
    _, feat, geo, depth = S._small_sweep()
    sc = _bp_scene(seed=17)
    xb = _leaf(sc["feat"])
    checks = ("test_schema", "test_faketensor", "test_autograd_registration")
    det_flag(True)
    torch.library.opcheck(L.plane_sweep_variance, (feat, geo.neighbor_ids, geo.hom, depth), test_utils=checks)
    torch.library.opcheck(L.plane_sweep_group_correlation, (feat, geo.neighbor_ids, geo.hom, depth, 4),
                          test_utils=checks)
    for sum_only in (False, True):
        torch.library.opcheck(L.backproject_aggregate,
                              (xb, sc["points"].to(DEV), sc["projection"].to(DEV), sc["depth"].to(DEV),
                               sc["prob"].to(DEV).requires_grad_(True), sc["vs_z"], sc["h"], sc["w"], sum_only),
                              test_utils=checks)


def test_hot_path_dispatcher_ops_end_to_end_under_the_flag(det_flag):  # noqa: F811
    """MVSDetHotPath(dispatcher_ops=True) with pre-packed bf16 features and a small conv net: the feature
    and weight gradients are bit-identical over three runs"""
    from mvsdet_b200.hotpath import MVSDetHotPath
    cfg = tiny_config(n_views=5, channels=32, num_depth=4)
    feature, _, _, _ = S._setup(cfg, 21, 2, torch.bfloat16)
    from mvsdet_b200.scene import make_scene
    meta = make_scene(cfg, 21, with_grads=False)["img_meta"]
    mod = MVSDetHotPath(cfg.n_voxels, cfg.voxel_size, cfg.near_far_range, cfg.num_depth, cfg.topk,
                        stride=cfg.stride, feature_dtype=torch.bfloat16, dispatcher_ops=True)
    geo = mod.geometry(meta, DEV)
    torch.manual_seed(0)
    net = torch.nn.Conv3d(cfg.channels, 2, 3, padding=1).to(DEV)
    g_vol = None
    det_flag(True)
    runs = []
    for _ in range(3):
        x = _leaf(feature, torch.bfloat16)
        out = mod(x, meta, cost_regularization=net, geometry=geo)
        vol = out["volume_mean"]
        if g_vol is None:
            g_vol = torch.randn(vol.shape, generator=torch.Generator().manual_seed(1)).to(DEV)
        loss = (vol * g_vol).sum() + out["est_depth"].sum()
        runs.append(torch.autograd.grad(loss, (x, net.weight)))
    torch.cuda.synchronize()
    det_flag(False)
    assert runs[0][0].dtype == torch.bfloat16 and bool(runs[0][0].float().abs().sum() > 0)
    for r in runs[1:]:
        assert torch.equal(r[0], runs[0][0]) and torch.equal(r[1], runs[0][1])
