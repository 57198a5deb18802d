"""The depth top-k over per-pixel depth hypotheses [V,D,H,W] (``depth_values=``, the planes of a
second sweep around an earlier ``est_depth``), forward and backward.

1. Planes z_d = fl(fl(d*interval) + near) with the scalar interval or a constant map give the
   per-view call's bits: all ten outputs and dL/dcost_out, at every DMAX template.
2. Non-uniform planes (sorted, unsorted, per-pixel spacing) against fp64 with per-element bounds
   (tests/ref64_px.py), est_idx against the kernel's own probabilities and fp64 where decided.
3. The backward, including dL/ddepth_values and dL/dinterval_map, against fp64 autograd.
4. NaN plane depths propagate as in the restatement.
5. The dispatcher ops give the autograd.Function route's bits and pass opcheck.
6. A coarse-to-fine chain through MVSDetHotPath's stages against the oracle.
"""
import pytest
import torch

import ref64
import ref64_px as R
from mvsdet_b200 import _lib, library as L, ops

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
NEAR, INTERVAL = 0.41, 0.37            # neither exact in fp32: the reduction rule sees real roundings
H, W = 5, 27                           # 135 pixels: one full CTA of 128 and a 7-pixel tail
DIFF = (0, 1, 2, 3, 5)                 # the differentiable outputs of depth_topk


def _cost(v, d, seed, raw=False):
    gen = torch.Generator().manual_seed(seed)
    c = torch.randn(v, 2, d, H, W, generator=gen) * 3.0
    if raw:
        p = torch.rand(v, d, H, W, generator=gen)
        c = torch.stack((p / p.sum(1, keepdim=True), torch.rand(v, d, H, W, generator=gen)), 1)
    return c


def _uniform_planes(v, d):
    """z_d = fl(fl(d * interval) + near) in fp32, as the per-view kernel forms it"""
    z = torch.arange(d, dtype=torch.float32) * torch.tensor(INTERVAL, dtype=torch.float32)
    z = z + torch.tensor(NEAR, dtype=torch.float32)
    return z.view(1, d, 1, 1).expand(v, d, H, W).contiguous()


def _grads(v, d, t, seed):
    gen = torch.Generator().manual_seed(seed)
    return (torch.randn(v, d, H, W, generator=gen), torch.randn(v, d, H, W, generator=gen),
            torch.randn(v, t, H, W, generator=gen), torch.randn(v, t, H, W, generator=gen),
            torch.randn(v, H, W, generator=gen))


def _k_feat(v):
    k = torch.zeros(v, 4, 4)
    for i in range(v):
        k[i] = torch.tensor([[20.0 + i, 0.3 * i, 13.0, 0], [0, 21.0 - i, 2.5 + i, 0], [0, 0, 1, 0], [0, 0, 0, 1]])
    return k.to(DEV)


DT = sorted({(d, t) for d in (1, 12, 13, 16, 17, 32, 33, 64) for t in (1, min(d, 3), min(d, 8))})


# --------------------------------------------------------------------------
# 1. reduction rule
# --------------------------------------------------------------------------
@pytest.mark.parametrize("d,t", DT)
def test_uniform_planes_give_the_per_view_bits(d, t):
    v = 2
    planes = _uniform_planes(v, d).to(DEV)
    imap = torch.full((v, H, W), INTERVAL, device=DEV)
    grads = [g.to(DEV) for g in _grads(v, d, t, 10 * d + t)]
    for raw in (False, True):
        cost = _cost(v, d, 100 * d + t, raw=raw).to(DEV)
        fn = ops.topk_hypotheses if raw else ops.depth_topk
        c0 = cost.clone().requires_grad_(True)
        want = fn(c0, NEAR, INTERVAL, t)
        g_want, = torch.autograd.grad([want[i] for i in DIFF], c0, [grads[i] for i in range(5)])
        for name, iv in (("scalar", INTERVAL), ("map", imap)):
            c1 = cost.clone().requires_grad_(True)
            got = fn(c1, 123.0, iv, t, depth_values=planes)     # near is ignored with depth_values
            for i, (a, b) in enumerate(zip(got, want)):
                assert torch.equal(a, b), f"D={d} T={t} raw={raw} {name}: output {i}"
            g_got, = torch.autograd.grad([got[i] for i in DIFF], c1, [grads[i] for i in range(5)])
            assert torch.equal(g_got, g_want), f"D={d} T={t} raw={raw} {name}: dL/dcost_out"
    # the NVS epilogue, with every upstream gradient including the ray terms
    cost = _cost(v, d, 7 * d + t).to(DEV)
    k = _k_feat(v)
    gen = torch.Generator().manual_seed(d + t)
    g_ray = [torch.randn(v, H, W, generator=gen).to(DEV), torch.randn(v, t, H, W, generator=gen).to(DEV),
             torch.randn(v, H, W, generator=gen).to(DEV)]      # opacity, est_ray_depth, ray_depth_coding
    nvs_grads = list(grads) + g_ray
    res = []
    for kw in (dict(near=NEAR, interval=INTERVAL), dict(near=0.0, interval=INTERVAL, depth_values=planes),
               dict(near=0.0, interval=imap, depth_values=planes)):
        c = cost.clone().requires_grad_(True)
        outs = ops.depth_topk_nvs(c, kw.pop("near"), kw.pop("interval"), t, k, **kw)
        g, = torch.autograd.grad([outs[i] for i in (0, 1, 2, 3, 5, 6, 8, 9)], c, nvs_grads)
        res.append(list(outs) + [g])
    for name, r in zip(("scalar", "map"), res[1:]):
        for i, (a, b) in enumerate(zip(r, res[0])):
            assert torch.equal(a, b), f"NVS D={d} T={t} {name}: output {i}"


# --------------------------------------------------------------------------
# 2. non-uniform planes against fp64
# --------------------------------------------------------------------------
def _planes(kind, v, d, seed):
    gen = torch.Generator().manual_seed(seed)
    base = 0.5 + 4 * torch.rand(v, 1, H, W, generator=gen)
    steps = 0.01 + 0.2 * torch.rand(v, d, H, W, generator=gen)
    z = base + torch.cumsum(steps, dim=1) - steps[:, :1]
    if kind == "unsorted":
        z = z[:, torch.randperm(d, generator=gen)]
    spacing = 0.05 + 0.3 * torch.rand(v, H, W, generator=gen) if kind == "spacing" else 0.23
    return z.contiguous(), spacing


def _on(x):
    return x.to(DEV) if torch.is_tensor(x) else x


@pytest.mark.parametrize("kind", ["sorted", "unsorted", "spacing"])
@pytest.mark.parametrize("d,t", [(1, 1), (8, 3), (12, 3), (13, 8), (33, 8), (64, 8)])
def test_non_uniform_planes_against_fp64(d, t, kind):
    v = 2
    cost = _cost(v, d, 31 * d + t)
    if d >= 2:   # planted exact ties above every other plane: resolved to the lower plane index
        gen = torch.Generator().manual_seed(d)
        a = torch.randint(0, d, (v, H, W), generator=gen)
        b = torch.randint(0, d, (v, H, W), generator=gen)
        top = cost[:, 0].max(dim=1).values + 1.0
        vi, yi, xi = torch.meshgrid(torch.arange(v), torch.arange(H), torch.arange(W), indexing="ij")
        cost[vi, 0, a, yi, xi] = top
        cost[vi, 0, b, yi, xi] = top
    z, iv = _planes(kind, v, d, 5 * d + t)
    outs = ops.depth_topk(cost.to(DEV), 0.0, _on(iv), t, depth_values=z.to(DEV))
    prob, off, dep, dens, idx, coding = (o.cpu() for o in outs)
    rp, ro, rdep, rcod = R.px_forward_reference(cost, z, iv)
    ref64.check_bound(prob, rp.v, rp.e, "prob")
    ref64.check_bound(off, ro.v, ro.e, "off")
    ref64.check_bound(coding, rcod.v, rcod.e, "depth_coding")
    ref64.check_bound(dep, torch.gather(rdep.v, 1, idx), torch.gather(rdep.e, 1, idx), "est_depth")
    assert torch.equal(dens, torch.gather(prob, 1, idx))
    assert torch.equal(idx, torch.sort(prob, dim=1, descending=True, stable=True).indices[:, :t]), \
        "est_idx is not the top-T of the kernel's own probabilities"
    sure, order = R.decided_ranks(rp.v, rp.e, t)
    assert torch.equal(idx[sure], order[sure]), "est_idx differs from the fp64 top-T where it is decided"
    print(f"D={d} T={t} {kind}: {int((~sure).sum())} of {sure.numel()} ranks within rounding")
    if d >= 2:
        lo, hi = torch.minimum(a, b), torch.maximum(a, b)
        one = a == b
        assert torch.equal(idx[:, 0], lo)
        if t >= 2:
            assert torch.equal(idx[:, 1][~one], hi[~one])


# --------------------------------------------------------------------------
# 3. backward against fp64 autograd
# --------------------------------------------------------------------------
def _check_backward(cost, z, iv, idx, grads, got, what, raw=False, g_depth_b=None, g_coding_b=None):
    """got = (g_cost, g_z, g_I or None) from the kernel; grads = (g_prob, g_off, g_depth, g_dens,
    g_coding) fp32 CPU (g_depth / g_coding as the kernel combined them with the ray terms: B's)"""
    (c, zz, imap), outs = R.px_restatement(cost, z, iv, idx, raw=raw)
    gd = g_depth_b.v if g_depth_b is not None else grads[2].double()
    gcod = g_coding_b.v if g_coding_b is not None else grads[4].double()
    leaves = [c, zz] + ([imap] if imap is not None else [])
    ref = torch.autograd.grad(outs, leaves, [grads[0].double(), grads[1].double(), gd, grads[3].double(), gcod])
    b0, b1, bz, bi = R.px_backward_bound(cost, z, iv, idx, grads[0], grads[1],
                                         g_depth_b if g_depth_b is not None else ref64.B(grads[2].double()),
                                         grads[3],
                                         g_coding_b if g_coding_b is not None else ref64.B(grads[4].double()),
                                         raw=raw)
    r = [ref64.check_bound(got[0][:, 0].cpu(), ref[0][:, 0], b0, f"{what}: dL/dlogits"),
         ref64.check_bound(got[0][:, 1].cpu(), ref[0][:, 1], b1, f"{what}: dL/doffsets"),
         ref64.check_bound(got[1].cpu(), ref[1], bz, f"{what}: dL/ddepth_values")]
    if imap is not None:
        r.append(ref64.check_bound(got[2].cpu(), ref[2], bi, f"{what}: dL/dinterval_map"))
    print(f"{what}: backward uses {max(x[0] for x in r):.3f} of its bound")


@pytest.mark.parametrize("kind", ["unsorted", "spacing"])
@pytest.mark.parametrize("d,t", [(8, 3), (12, 3), (17, 8), (64, 8)])
@pytest.mark.parametrize("raw", [False, True], ids=["logits", "raw"])
def test_backward_against_fp64(d, t, kind, raw):
    v = 2
    cost = _cost(v, d, 3 * d + t, raw=raw)
    z, iv = _planes(kind, v, d, d + 17 * t)
    grads = _grads(v, d, t, d * 7 + t)
    c = cost.to(DEV).requires_grad_(True)
    zd = z.to(DEV).requires_grad_(True)
    ivd = _on(iv).requires_grad_(True) if torch.is_tensor(iv) else iv
    fn = ops.topk_hypotheses if raw else ops.depth_topk
    outs = fn(c, 0.0, ivd, t, depth_values=zd)
    leaves = [c, zd] + ([ivd] if torch.is_tensor(iv) else [])
    got = torch.autograd.grad([outs[i] for i in DIFF], leaves, [g.to(DEV) for g in grads])
    _check_backward(cost, z, iv, outs[4].cpu(), grads, list(got) + [None], f"D={d} T={t} {kind} raw={raw}",
                    raw=raw)


@pytest.mark.parametrize("used", [(), (0,), (1,), (2,), (3,), (4,), (2, 4)],
                         ids=["none", "prob", "off", "depth", "dens", "coding", "depth+coding"])
def test_backward_with_missing_upstream_gradients(used):
    """gradients of only some outputs (the others arrive as None / zeros)"""
    v, d, t = 2, 12, 3
    cost = _cost(v, d, 5)
    z, iv = _planes("spacing", v, d, 9)
    full = _grads(v, d, t, 3)
    grads = tuple(g if i in used else torch.zeros_like(g) for i, g in enumerate(full))
    c = cost.to(DEV).requires_grad_(True)
    zd = z.to(DEV).requires_grad_(True)
    ivd = iv.to(DEV).requires_grad_(True)
    outs = ops.depth_topk(c, 0.0, ivd, t, depth_values=zd)
    if not used:     # no upstream gradient at all: every gradient is zero
        g_cost = torch.empty_like(c)
        g_z = torch.full_like(zd, float("nan"))
        g_i = torch.full_like(ivd, float("nan"))
        _lib.depth_topk_bwd(c.detach(), outs[4], None, None, None, None, None, g_cost, near=0.0, interval=ivd.detach(),
                            depth_values=zd.detach(), g_depth_values=g_z, g_interval_map=g_i)
        torch.cuda.synchronize()
        assert not bool(g_cost.any()) and not bool(g_z.any()) and not bool(g_i.any())
        return
    sel = [DIFF[i] for i in used]
    got = torch.autograd.grad([outs[i] for i in sel], [c, zd, ivd], [full[i].to(DEV) for i in used])
    _check_backward(cost, z, iv, outs[4].cpu(), grads, got, f"upstream {used}")


def test_backward_with_ray_gradients():
    """depth_topk_nvs over per-pixel hypotheses: opacity, est_ray_depth and ray_depth_coding feed
    dL/ddepth_values and dL/dinterval_map through the kernel's fold of the ray terms"""
    v, d, t = 3, 13, 3
    cost = _cost(v, d, 21)
    z, iv = _planes("spacing", v, d, 22)
    grads = _grads(v, d, t, 23)
    gen = torch.Generator().manual_seed(24)
    g_opa, g_rd, g_rc = (torch.randn(v, H, W, generator=gen), torch.randn(v, t, H, W, generator=gen),
                         torch.randn(v, H, W, generator=gen))
    c = cost.to(DEV).requires_grad_(True)
    zd = z.to(DEV).requires_grad_(True)
    ivd = iv.to(DEV).requires_grad_(True)
    outs = ops.depth_topk_nvs(c, 0.0, ivd, t, _k_feat(v), depth_values=zd)
    got = torch.autograd.grad([outs[i] for i in (0, 1, 2, 3, 5, 6, 8, 9)], [c, zd, ivd],
                              [x.to(DEV) for x in list(grads) + [g_opa, g_rd, g_rc]])
    # the kernel folds the ray terms: gz = fmaf(g_ray_depth, 1/fl(scale + 1e-8), g_depth), likewise gcod
    scale = outs[7].cpu().double()
    inv = ref64.B(torch.ones_like(scale)).div(ref64.B(scale) + 1e-8)
    inv_t = ref64.B(inv.v.unsqueeze(1), inv.e.unsqueeze(1))
    gz = ref64.B(g_rd.double()).fma(inv_t, ref64.B(grads[2].double()))
    gcod = ref64.B(g_rc.double()).fma(inv, ref64.B(grads[4].double()))
    g_dens = grads[3].clone()
    g_dens[:, 0] += g_opa                      # opacity is est_dens[:, 0], added in fp32 as ops does
    _check_backward(cost, z, iv, outs[4].cpu(), (grads[0], grads[1], grads[2], g_dens, grads[4]), got,
                    "ray gradients", g_depth_b=gz, g_coding_b=gcod)


def test_map_gradients_are_written_only_when_requested():
    """the launcher with one of g_depth_values / g_interval_map: the other stays untouched, the given
    one is overwritten (NaN-filled beforehand), and dL/dcost_out does not depend on the request"""
    v, d, t = 2, 16, 3
    cost = _cost(v, d, 40).to(DEV)
    z, iv = _planes("spacing", v, d, 41)
    z, iv = z.to(DEV), iv.to(DEV)
    outs = ops.depth_topk(cost, 0.0, iv, t, depth_values=z)
    idx = outs[4]
    grads = [g.to(DEV) for g in _grads(v, d, t, 42)]
    res = {}
    for want_z, want_i in ((True, True), (True, False), (False, True), (False, False)):
        g_cost = torch.empty_like(cost)
        g_z = torch.full_like(z, float("nan"))
        g_i = torch.full_like(iv, float("nan"))
        _lib.depth_topk_bwd(cost, idx, *grads, g_cost, near=0.0, interval=iv, depth_values=z,
                            g_depth_values=g_z if want_z else None, g_interval_map=g_i if want_i else None)
        torch.cuda.synchronize()
        res[want_z, want_i] = (g_cost, g_z, g_i)
        assert bool(g_z.isnan().all()) != want_z and bool(g_i.isnan().all()) != want_i
    full = res[True, True]
    assert not bool(full[1].isnan().any()) and not bool(full[2].isnan().any())
    for (want_z, want_i), r in res.items():
        assert torch.equal(r[0], full[0])
        if want_z:
            assert torch.equal(r[1], full[1])
        if want_i:
            assert torch.equal(r[2], full[2])
    # through autograd: a depth_values that needs no gradient gets none, an interval map likewise
    c = cost.clone().requires_grad_(True)
    zd = z.clone().requires_grad_(True)
    o = ops.depth_topk(c, 0.0, iv, t, depth_values=zd)
    gc, gz = torch.autograd.grad([o[i] for i in DIFF], [c, zd], [grads[i] for i in range(5)])
    assert torch.equal(gc, full[0]) and torch.equal(gz, full[1])


# --------------------------------------------------------------------------
# 4. NaN planes
# --------------------------------------------------------------------------
def test_nan_planes_propagate_as_the_restatement():
    v, d, t = 2, 12, 3
    cost = _cost(v, d, 50)
    z, iv = _planes("spacing", v, d, 51)
    gen = torch.Generator().manual_seed(52)
    z[torch.rand(z.shape, generator=gen) < 0.05] = float("nan")
    grads = _grads(v, d, t, 53)
    c = cost.to(DEV).requires_grad_(True)
    zd = z.to(DEV).requires_grad_(True)
    ivd = iv.to(DEV).requires_grad_(True)
    outs = ops.depth_topk(c, 0.0, ivd, t, depth_values=zd)
    got = torch.autograd.grad([outs[i] for i in DIFF], [c, zd, ivd], [g.to(DEV) for g in grads])
    idx = outs[4].cpu()
    leaves, ref_outs = R.px_restatement(cost, z, iv, idx)
    ref_g = torch.autograd.grad(ref_outs, list(leaves), [g.double() for g in grads])
    for i, (a, b) in enumerate(zip([outs[j] for j in DIFF], ref_outs)):
        assert torch.equal(a.detach().cpu().isnan(), b.detach().isnan()), f"output {DIFF[i]}"
    assert bool(outs[2].isnan().any()) and bool(outs[5].isnan().any())
    for i, (a, b) in enumerate(zip(got, ref_g)):
        assert torch.equal(a.cpu().isnan(), b.isnan()), f"gradient {i}"


# --------------------------------------------------------------------------
# 5. dispatcher ops
# --------------------------------------------------------------------------
@pytest.mark.parametrize("with_map", [False, True], ids=["scalar", "map"])
def test_dispatcher_route_matches_autograd_function(with_map):
    v, d, t = 2, 12, 3
    cost = _cost(v, d, 60).to(DEV)
    z, iv = _planes("spacing" if with_map else "unsorted", v, d, 61)
    z, iv = z.to(DEV), _on(iv)
    grads = [g.to(DEV) for g in _grads(v, d, t, 62)]
    res = []
    for route in ("ops", "library"):
        c = cost.clone().requires_grad_(True)
        zd = z.clone().requires_grad_(True)
        ivd = iv.clone().requires_grad_(True) if with_map else iv
        if route == "ops":
            outs = ops.depth_topk(c, 0.0, ivd, t, depth_values=zd)
        else:
            outs = L.depth_topk_px(c, zd, ivd if with_map else None, 0.0 if with_map else iv, t)
        leaves = [c, zd] + ([ivd] if with_map else [])
        g = torch.autograd.grad([outs[i] for i in DIFF], leaves, [grads[i] for i in range(5)])
        res.append([o.detach() for o in outs] + list(g))
    for i, (a, b) in enumerate(zip(*res)):
        assert torch.equal(a, b), f"item {i}"
    c = cost.clone().requires_grad_(True)
    zd = z.clone().requires_grad_(True)
    checks = ("test_schema", "test_faketensor", "test_autograd_registration")
    if with_map:
        ivd = iv.clone().requires_grad_(True)
        torch.library.opcheck(L.depth_topk_px, (c, zd, ivd, 0.0, t), test_utils=checks)
        o = L.depth_topk_px(cost, z, iv, 0.0, t)
        args = (cost, o[4], z, iv, *grads, 0.0, False)
    else:
        torch.library.opcheck(L.depth_topk_px, (c, zd, None, iv, t), test_utils=checks)
        o = L.depth_topk_px(cost, z, None, iv, t)
        args = (cost, o[4], z, None, *grads, iv, False)
    torch.library.opcheck(L.depth_topk_px_bwd, args, test_utils=("test_schema", "test_faketensor"))


def test_bad_arguments_raise():
    v, d, t = 2, 12, 3
    cost = _cost(v, d, 70).to(DEV)
    z = _uniform_planes(v, d).to(DEV)
    imap = torch.full((v, H, W), INTERVAL, device=DEV)
    bad = [dict(depth_values=z[:, :-1]), dict(depth_values=z.cpu()), dict(depth_values=z.double()),
           dict(depth_values=z[..., :-1]), dict(depth_values=z, interval=imap[:, :-1]),
           dict(depth_values=z, interval=imap.cpu()), dict(depth_values=z, interval=imap.double()),
           dict(depth_values=z, interval="0.3")]
    for kw in bad:
        kw = dict(kw)
        iv = kw.pop("interval", INTERVAL)
        with pytest.raises(ValueError):
            ops.depth_topk(cost, NEAR, iv, t, **kw)
        with pytest.raises(ValueError):
            ops.topk_hypotheses(cost, NEAR, iv, t, **kw)
        with pytest.raises(ValueError):
            ops.depth_topk_nvs(cost, NEAR, iv, t, _k_feat(v), **kw)
        if not kw["depth_values"].is_cuda or (isinstance(iv, torch.Tensor) and not iv.is_cuda):
            continue             # the dispatcher op has no CPU kernel to dispatch a mixed call to
        if isinstance(iv, torch.Tensor):
            with pytest.raises(ValueError):
                L.depth_topk_px(cost, kw["depth_values"], iv, 0.0, t)
        elif isinstance(iv, float):
            with pytest.raises(ValueError):
                L.depth_topk_px(cost, kw["depth_values"], None, iv, t)


# --------------------------------------------------------------------------
# 6. coarse-to-fine through MVSDetHotPath's stages against the oracle
# --------------------------------------------------------------------------
def _close(a, b, what, rtol=1e-4, atol_scale=1e-4):
    """the bar of test_gpu_parity.py: |a - b| <= 1e-4 rms(b) + 1e-4 |b|"""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    assert a.shape == b.shape, f"{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    rms = float(b.pow(2).mean().sqrt())
    err = (a - b).abs()
    bad = err > atol_scale * rms + rtol * b.abs()
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())}/{bad.numel()} out of tolerance, "
                                 f"max abs err {float(err.max()):.3e} (rms {rms:.3e})")


def _rank_agreement(prob_ref, idx, what, rel=1e-4):
    """the oracle's top-T (its own probabilities) equals the kernel's est_idx wherever the oracle's
    gaps to the neighbouring ranks exceed rel * max prob; returns the number not decided"""
    t = idx.shape[1]
    srt, order = torch.sort(prob_ref.detach(), dim=1, descending=True, stable=True)
    thr = rel * srt[:, :1]
    apart = (srt[:, :-1] - srt[:, 1:]) > thr
    sure = torch.ones(idx.shape, dtype=torch.bool)
    for i in range(t):
        if i > 0:
            sure[:, i] &= apart[:, i - 1]
        if i + 1 < srt.shape[1]:
            sure[:, i] &= apart[:, i]
    assert torch.equal(order[:, :t][sure], idx[sure]), f"{what}: the oracle's top-T differs where it is decided"
    return int((~sure).sum())


def test_coarse_to_fine_through_the_stages_matches_the_oracle():
    from oracle import mvsdet_oracle as O
    from mvsdet_b200.scene import tiny_config
    from test_gpu_depth_map_sweep import _oracle_variance, _setup

    d1, d2 = 12, 8
    cfg = tiny_config(n_views=5, channels=32, num_depth=d1, topk=3)
    feature, mod, geo, all_proj = _setup(cfg, 11, 2, torch.float32)
    c, t = cfg.channels, cfg.topk
    hf, wf = cfg.feat_hw
    h, w = geo.height, geo.width
    nets = []
    for seed in (1, 2):
        torch.manual_seed(seed)
        nets.append(torch.nn.Conv3d(c, 2, 3, padding=1))
    gen = torch.Generator().manual_seed(12)
    g_vol = torch.randn(c, *cfg.n_voxels, generator=gen)
    g_ed = torch.randn(cfg.n_views, t, hf, wf, generator=gen)
    g_cod = torch.randn(cfg.n_views, hf, wf, generator=gen)
    factors = 1 + torch.linspace(-0.05, 0.05, d2)

    # the kernels, through the stage API
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        dnets = [torch.nn.Conv3d(c, 2, 3, padding=1).to(DEV) for _ in nets]
        for a, b in zip(dnets, nets):
            a.load_state_dict(b.state_dict())
        f = feature.to(DEV).requires_grad_(True)
        feat_cl, sink = ops.pack_features(f, torch.float32, sink=True)
        coarse = mod.hypotheses(dnets[0](mod.variance(feat_cl, geo, grad_sink=sink)))
        ed1 = coarse[2][:, :1]
        planes = ed1 * factors.to(DEV).view(1, d2, 1, 1)                # not detached
        spacing = ed1[:, 0] * (0.1 / 7)
        fine = mod.hypotheses(dnets[1](mod.variance(feat_cl, geo, grad_sink=sink, depth_values=planes)),
                              depth_values=planes, interval=spacing)
        vol, count = mod.voxels(feat_cl, geo, fine[2], fine[3], grad_sink=sink)
        nx, ny, nz = cfg.n_voxels
        vol = vol.view(c, nx, ny, nz)
        params = [p for n in dnets for p in n.parameters()]
        g = torch.autograd.grad([vol, fine[2], fine[5]], [f] + params,
                                [g_vol.to(DEV), g_ed.to(DEV), g_cod.to(DEV)])
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32 = tf32

    # the oracle, with the kernel's ranks where they are within rounding
    fr = feature.clone().requires_grad_(True)
    nbr = geo.neighbor_ids_ref()
    dplanes = geo.depth_values.cpu()[:, :, None, None].expand(-1, -1, hf, wf).contiguous()
    prob1, off1 = O.depth_probability(nets[0](_oracle_variance(fr, all_proj, nbr, dplanes)))
    idx1 = coarse[4].cpu()
    n_undecided = _rank_agreement(prob1, idx1, "coarse")
    dep1 = torch.arange(d1).view(1, d1, 1, 1) * mod.depth_interval + torch.tensor(cfg.near_far_range[0]) \
        + off1 * torch.tensor(mod.depth_interval)
    ed1_ref = torch.gather(dep1, 1, idx1[:, :1])
    planes_ref = ed1_ref * factors.view(1, d2, 1, 1)
    spacing_ref = ed1_ref[:, 0] * (0.1 / 7)
    # the sweep gives depth_values no gradient (the reference builds its grid under no_grad)
    prob2, off2 = O.depth_probability(nets[1](_oracle_variance(fr, all_proj, nbr, planes_ref.detach())))
    idx2 = fine[4].cpu()
    n_undecided += _rank_agreement(prob2, idx2, "fine")
    dep2 = planes_ref + off2 * spacing_ref.unsqueeze(1)
    ed2_ref = torch.gather(dep2, 1, idx2)
    dens2_ref = torch.gather(prob2, 1, idx2)
    cod2_ref = (prob2 * dep2).sum(dim=1)
    _close(fine[2], ed2_ref, "fine est_depth")
    _close(fine[3], dens2_ref, "fine est_densities")
    _close(fine[5], cod2_ref, "fine depth_coding")

    # back-projection: the window tests on the kernel's est_depth (the same fp32 values the kernel
    # tested), the oracle's own depths must agree wherever they are not within rounding of an edge
    import bp_cases
    pts = geo.points.cpu().reshape(3, -1)
    proj = geo.projection.cpu()
    vs_z = cfg.voxel_size[2]
    ed2_k = fine[2].detach().cpu()[:, :, :h, :w]
    r_k, inb = bp_cases.window_margin(pts, proj, ed2_k, vs_z, h, w)
    r_o, _ = bp_cases.window_margin(pts, proj, ed2_ref.detach()[:, :, :h, :w], vs_z, h, w)
    sure = inb.unsqueeze(-1) & ((r_o - 1).abs() > 1e-4)
    assert torch.equal((r_k < 1)[sure], (r_o < 1)[sure]), "a depth-test window differs where it is decided"
    n_window = int((inb.unsqueeze(-1) & ~sure.bool()).sum())
    print(f"ranks within rounding: {n_undecided}; depth-test windows within rounding: {n_window}")
    depth_r = ed2_k.reshape(cfg.n_views, t, -1).transpose(2, 1).unsqueeze(2)
    dens_r = dens2_ref[:, :, :h, :w].reshape(cfg.n_views, t, -1).transpose(2, 1).unsqueeze(2)
    volume, valid = O.backproject_weigh(fr[:, :, :h, :w], geo.points.cpu(), proj, depth_r, cfg.voxel_size, dens_r)
    vol_ref, count_ref = O.aggregate_views(volume, valid)
    _close(vol, vol_ref, "volume_mean")
    assert torch.equal(count.cpu().long(), count_ref.reshape(-1).long()), "count"
    ref_params = [p for n in nets for p in n.parameters()]
    g_ref = torch.autograd.grad([vol_ref, ed2_ref, cod2_ref], [fr] + ref_params, [g_vol, g_ed, g_cod])
    _close(g[0], g_ref[0], "dL/dfeature")
    names = [f"{s} {n}" for s in ("coarse", "fine") for n, _ in nets[0].named_parameters()]
    for name, a, b in zip(names, g[1:], g_ref[1:]):
        _close(a, b, f"dL/d{name}")
