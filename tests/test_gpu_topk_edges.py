"""The depth top-k epilogue (softmax, sigmoid, top-T hypotheses, expectation; forward and
backward) at every plane count around its DMAX templates {12, 16, 32, 64} and T up to 8, against
fp64 with per-element bounds (tests/ref64.py).

Forward bounds follow the kernel op by op: ``expf`` is within 2 ulp, every other operation is
correctly rounded.  The backward recomputes the probabilities with ``__expf`` (within
2 + floor(|1.173 a|) ulp for argument a) and ``__fdividef`` (2 ulp), so its bound grows with the
spread of the logits; ``ref64.topk_backward_bound`` derives it.  The tests print the largest
observed error as a fraction of its bound.
"""
import pytest
import torch

import ref64
from mvsdet_b200 import ops

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
NEAR, INTERVAL = 0.5, 0.3125
H, W = 5, 27            # 135 pixels: one full CTA of 128 and a 7-pixel tail


def _cost(v, d, seed, spread=3.0, ties=True, neg_inf=False):
    gen = torch.Generator().manual_seed(seed)
    c = torch.randn(v, 2, d, H, W, generator=gen) * spread
    if spread > 10:
        c = (torch.rand(v, 2, d, H, W, generator=gen) * 2 - 1) * spread
    if ties and d >= 2:
        # planted exact ties: two planes share the pixel's largest logit (equal logits -> equal
        # probabilities, bit for bit) -- resolved to the lower plane index
        a = torch.randint(0, d, (v, H, W), generator=gen)
        b = torch.randint(0, d, (v, H, W), generator=gen)
        top = c[:, 0].max(dim=1).values + 1.0
        rows = torch.rand(v, H, W, generator=gen) < 0.5
        vi, yi, xi = rows.nonzero(as_tuple=True)
        c[vi, 0, a[rows], yi, xi] = top[rows]
        c[vi, 0, b[rows], yi, xi] = top[rows]
    if neg_inf and d >= 3:
        m = torch.rand(v, d, H, W, generator=gen) < 0.3
        m[:, 0] = False                      # keep one finite plane per pixel
        c[:, 0][m] = float("-inf")
    return c


def _topk_of_own_probs(prob, t):
    """the top-T of the kernel's own fp32 probabilities, ties to the lower plane index"""
    return torch.sort(prob, dim=1, descending=True, stable=True).indices[:, :t]


def _grads(v, d, t, seed):
    gen = torch.Generator().manual_seed(seed + 7)
    return (torch.randn(v, d, H, W, generator=gen), torch.randn(v, d, H, W, generator=gen),
            torch.randn(v, t, H, W, generator=gen), torch.randn(v, t, H, W, generator=gen),
            torch.randn(v, H, W, generator=gen))


def _fwd_check(cost, outs, t, what, raw=False):
    prob, off, dep, dens, idx, coding = (o.detach().cpu() for o in outs[:6])
    rp, ro, rdep, rcod = ref64.topk_forward_reference(cost, NEAR, INTERVAL, raw=raw)
    r = [ref64.check_bound(prob, rp.v, rp.e, f"{what}: prob")]
    r.append(ref64.check_bound(off, ro.v, ro.e, f"{what}: off"))
    r.append(ref64.check_bound(coding, rcod.v, rcod.e, f"{what}: depth_coding"))
    r.append(ref64.check_bound(dep, torch.gather(rdep.v.expand(*prob.shape), 1, idx),
                               torch.gather(rdep.e.expand(*prob.shape), 1, idx), f"{what}: est_depth"))
    assert torch.equal(dens, torch.gather(prob, 1, idx)), f"{what}: est_dens != prob.gather(est_idx)"
    assert torch.equal(idx, _topk_of_own_probs(prob, t)), f"{what}: est_idx is not the top-T of prob"
    # against fp64 wherever the rank is decided: the fp64 gap to the neighbours above and below
    # exceeds 8 ulp and the two elements' bounds
    srt, order = torch.sort(rp.v, dim=1, descending=True, stable=True)
    eb = torch.gather(rp.e, 1, order)
    gap = srt[:, :-1] - srt[:, 1:]
    thr = torch.maximum(8 * ref64.ULP * srt[:, :-1].abs(), eb[:, :-1] + eb[:, 1:])
    apart = gap > thr                                   # rank i and i + 1 are decided
    sure = torch.ones_like(idx, dtype=torch.bool)
    d = srt.shape[1]
    for i in range(t):
        if i > 0:
            sure[:, i] &= apart[:, i - 1]
        if i + 1 < d:
            sure[:, i] &= apart[:, i]
    assert torch.equal(idx[sure], order[:, :t][sure]), f"{what}: est_idx differs from the fp64 top-T"
    return max(x[0] for x in r)


DT = sorted({(d, t) for d in (1, 2, 11, 12, 13, 16, 17, 31, 32, 33, 63, 64)
             for t in (1, min(d, 3), min(d, 8))})


@pytest.mark.parametrize("d,t", DT)
def test_planes_and_hypotheses(d, t):
    cost = _cost(2, d, seed=100 * d + t)
    cd = cost.to(DEV).requires_grad_(True)
    outs = ops.depth_topk(cd, NEAR, INTERVAL, t)
    ratio = _fwd_check(cost, outs, t, f"D={d} T={t}")
    idx = outs[4].cpu()
    if d >= 2:    # planted ties: the lower plane wins
        srt = torch.sort(cost[:, 0], dim=1, descending=True, stable=True)
        tie = srt.values[:, 0] == srt.values[:, 1]
        assert bool(tie.any())
        assert torch.equal(idx[:, 0][tie], srt.indices[:, 0][tie]), "an exact tie was not resolved to the lower plane"
        if t >= 2:
            assert torch.equal(idx[:, 1][tie], srt.indices[:, 1][tie])
    grads = _grads(2, d, t, d * 10 + t)
    g, = torch.autograd.grad([outs[i] for i in (0, 1, 2, 3, 5)], cd, [x.to(DEV) for x in grads])
    ref = ref64.topk_autograd_reference(cost, idx, grads, NEAR, INTERVAL)
    b0, b1 = ref64.topk_backward_bound(cost, idx, grads, NEAR, INTERVAL)
    r0 = ref64.check_bound(g[:, 0].cpu(), ref[:, 0], b0, f"D={d} T={t}: dL/dlogits")
    r1 = ref64.check_bound(g[:, 1].cpu(), ref[:, 1], b1, f"D={d} T={t}: dL/doffsets")
    print(f"D={d} T={t}: forward uses {ratio:.3f} of its bound, backward {max(r0[0], r1[0]):.3f} "
          f"(max abs err {max(r0[1], r1[1]):.2e})")


@pytest.mark.parametrize("d,t", [(12, 3), (33, 8), (64, 8)])
def test_backward_wide_logits(d, t):
    """logits spread over +-80 (where __expf's error grows with |a|) and planes at -inf"""
    cost = _cost(2, d, seed=7 * d, spread=80.0, ties=False, neg_inf=True)
    cd = cost.to(DEV).requires_grad_(True)
    outs = ops.depth_topk(cd, NEAR, INTERVAL, t)
    _fwd_check(cost, outs, t, f"wide D={d}")
    idx = outs[4].cpu()
    grads = _grads(2, d, t, d)
    g, = torch.autograd.grad([outs[i] for i in (0, 1, 2, 3, 5)], cd, [x.to(DEV) for x in grads])
    ref = ref64.topk_autograd_reference(cost, idx, grads, NEAR, INTERVAL)
    b0, b1 = ref64.topk_backward_bound(cost, idx, grads, NEAR, INTERVAL)
    r0 = ref64.check_bound(g[:, 0].cpu(), ref[:, 0], b0, f"wide D={d}: dL/dlogits")
    r1 = ref64.check_bound(g[:, 1].cpu(), ref[:, 1], b1, f"wide D={d}: dL/doffsets")
    print(f"wide D={d} T={t}: backward uses {max(r0[0], r1[0]):.3f} of its bound "
          f"(max abs err {max(r0[1], r1[1]):.2e})")


def test_raw_mode():
    """ops.topk_hypotheses: channel 0 / 1 are already probabilities / offsets"""
    d, t = 64, 8
    gen = torch.Generator().manual_seed(3)
    p = torch.rand(2, d, H, W, generator=gen)
    p[:, 5] = p[:, 9] = 1.5                        # an exact tie above everything
    po = torch.stack((p / p.sum(1, keepdim=True), torch.rand(2, d, H, W, generator=gen)), 1)
    cd = po.to(DEV).requires_grad_(True)
    outs = ops.topk_hypotheses(cd, NEAR, INTERVAL, t)
    assert torch.equal(outs[0].detach().cpu(), po[:, 0]) and torch.equal(outs[1].detach().cpu(), po[:, 1])
    _fwd_check(po, outs, t, "raw", raw=True)
    idx = outs[4].cpu()
    assert bool((idx[:, 0] == 5).all()) and bool((idx[:, 1] == 9).all())
    grads = _grads(2, d, t, 5)
    g, = torch.autograd.grad([outs[i] for i in (0, 1, 2, 3, 5)], cd, [x.to(DEV) for x in grads])
    ref = ref64.topk_autograd_reference(po, idx, grads, NEAR, INTERVAL, raw=True)
    b0, b1 = ref64.topk_backward_bound(po, idx, grads, NEAR, INTERVAL, raw=True)
    ref64.check_bound(g[:, 0].cpu(), ref[:, 0], b0, "raw: dL/dprob")
    ref64.check_bound(g[:, 1].cpu(), ref[:, 1], b1, "raw: dL/doff")


@pytest.mark.parametrize("d,t", [(13, 3), (64, 8)])
def test_channels_last_cost(d, t):
    """a channels_last_3d cost_out is read through its strides: same bits, forward and backward"""
    cost = _cost(2, d, seed=d).to(DEV)
    grads = [x.to(DEV) for x in _grads(2, d, t, 1)]
    res = []
    for c in (cost.contiguous(), cost.contiguous(memory_format=torch.channels_last_3d)):
        c = c.detach().requires_grad_(True)
        outs = ops.depth_topk(c, NEAR, INTERVAL, t)
        g, = torch.autograd.grad([outs[i] for i in (0, 1, 2, 3, 5)], c, grads)
        res.append([o.detach() for o in outs] + [g.contiguous()])
    for a, b in zip(*res):
        assert torch.equal(a, b)


def test_nvs_epilogue():
    """depth_topk_nvs at D = 64, T = 8 with per-view intrinsics: the ray depths are the kernel's own
    est_depth / depth_coding divided by (depth_scale + 1e-8), bit for bit; opacity is the top-1
    density"""
    d, t, v = 64, 8, 3
    cost = _cost(v, d, seed=11).to(DEV)
    k = torch.zeros(v, 4, 4)
    for i in range(v):
        k[i] = torch.tensor([[20.0 + i, 0.3 * i, 13.0, 0], [0, 21.0 - i, 2.5 + i, 0], [0, 0, 1, 0], [0, 0, 0, 1]])
    outs = ops.depth_topk_nvs(cost, NEAR, INTERVAL, t, k.to(DEV))
    prob, off, dep, dens, idx, coding, opacity, scale, ray_dep, ray_cod = outs
    plain = ops.depth_topk(cost, NEAR, INTERVAL, t)
    for a, b in zip(outs[:6], plain):
        assert torch.equal(a, b)
    den = scale + 1e-8
    assert torch.equal(ray_dep, dep / den.unsqueeze(1))
    assert torch.equal(ray_cod, coding / den)
    assert torch.equal(opacity, dens[:, 0])
    assert torch.equal(scale, ops.ray_depth_scale(k.to(DEV), v, H, W))
    _fwd_check(cost.cpu(), outs, t, "nvs")
