"""Hand-built inputs for the back-projection edge tests (test infrastructure, CPU tensors).

``random_scene`` builds cameras around a small voxel block and depth maps whose every
(view, voxel, hypothesis) decision is far from any rounding question; ``exact_scene`` builds
projections whose every product and quotient is exact in fp32, so that the rounding, window and
routing edges are hit exactly.  ``tests/test_bp_topk_cases_cpu.py`` checks on CPU that both are
what they claim to be.
"""
from __future__ import annotations

import math

import torch

BACKGROUND = 15.0     # depth of an unused hypothesis: > 2 vs_z from every voxel's z (z is 1.5 .. 4.5)


def _look_at(gen, radius):
    """world -> camera rotation and centre of a camera on a sphere looking at the origin"""
    az = float(torch.rand((), generator=gen)) * 2 * math.pi
    el = (float(torch.rand((), generator=gen)) - 0.5) * 1.2
    c = torch.tensor([math.cos(el) * math.cos(az), math.cos(el) * math.sin(az), math.sin(el)]) * radius
    fwd = -c / c.norm()
    up = torch.tensor([0.0, 0.0, 1.0])
    right = torch.linalg.cross(fwd, up)
    right = right / right.norm()
    down = torch.linalg.cross(fwd, right)
    return torch.stack((right, down, fwd)), c


def project(points, projection):
    """the oracle's fp32 projection (bmm, then round half-to-even): -> x, y [V,N] int64, z [V,N]"""
    v = projection.shape[0]
    pts = torch.cat((points, torch.ones_like(points[:1])), 0).unsqueeze(0).expand(v, 4, -1)
    p = torch.bmm(projection, pts)
    return (p[:, 0] / p[:, 2]).round().long(), (p[:, 1] / p[:, 2]).round().long(), p[:, 2]


def window_margin(points, projection, depth, vs_z, h, w):
    """|z - d| / vs_z of every in-bounds (view, voxel, hypothesis) -> ([V,N,T] ratio, [V,N] in-bounds)"""
    x, y, z = project(points, projection)
    inb = (x >= 0) & (y >= 0) & (x < w) & (y < h) & (z > 0)
    v, t = depth.shape[:2]
    xs, ys = x.clamp(0, w - 1), y.clamp(0, h - 1)
    d = depth[torch.arange(v).view(v, 1, 1), torch.arange(t).view(1, 1, t), ys.unsqueeze(-1), xs.unsqueeze(-1)]
    return (z.unsqueeze(-1) - d).abs() / vs_z, inb


def random_scene(v, c, t, n, seed, *, h=21, w=28, fh=24, fw=31, vs_z=0.03125, bf16=False):
    """V random cameras 2.5-3.5 units from a voxel block in [-0.6, 0.6]^3, an [fh,fw] feature map
    of which [h,w] is the crop, T hypotheses per pixel.  About 40 % of the in-bounds (view, voxel)
    pairs get their projected z (+- 0.4 vs_z) written into a random hypothesis of their pixel,
    15 % get z +- 2.2..3 vs_z, the rest see only BACKGROUND.  A hypothesis that two voxels share
    and that ends up within [0.5, 2] vs_z of either is reset to BACKGROUND, so every decision has
    a margin of at least half the window: it cannot depend on rounding or FMA contraction.
    Features are rounded to bf16 values when ``bf16`` (the kernels then read them exactly)."""
    gen = torch.Generator().manual_seed(seed)
    points = (torch.rand(3, n, generator=gen) * 1.2 - 0.6).float()
    proj = []
    for _ in range(v):
        rot, cen = _look_at(gen, 2.5 + float(torch.rand((), generator=gen)))
        f = w * (1.1 + 0.3 * float(torch.rand((), generator=gen)))
        k = torch.tensor([[f, 0.0, w / 2 + float(torch.randn((), generator=gen))],
                          [0.0, f, h / 2 + float(torch.randn((), generator=gen))],
                          [0.0, 0.0, 1.0]])
        proj.append(k @ torch.cat((rot, -(rot @ cen).unsqueeze(1)), 1))
    proj = torch.stack(proj).float()
    x, y, z = project(points, proj)
    inb = (x >= 0) & (y >= 0) & (x < w) & (y < h) & (z > 0)
    depth = BACKGROUND + torch.rand(v, t, fh, fw, generator=gen) * 5
    prob = 0.05 + torch.rand(v, t, fh, fw, generator=gen) * 0.95
    roll = torch.rand(v, n, generator=gen)
    hyp = torch.randint(0, t, (v, n), generator=gen)
    off = (torch.rand(v, n, generator=gen) * 0.8 - 0.4) * vs_z
    far = (2.2 + 0.8 * torch.rand(v, n, generator=gen)) * vs_z * torch.where(
        torch.rand(v, n, generator=gen) < 0.5, -1.0, 1.0)
    val = torch.where(roll < 0.4, z + off, z + far)
    sel = inb & (roll < 0.55)
    vi = torch.arange(v).view(v, 1).expand(v, n)
    depth[vi[sel], hyp[sel], y[sel], x[sel]] = val[sel].float()
    ratio, _ = window_margin(points, proj, depth, vs_z, h, w)
    amb = inb.unsqueeze(-1) & (ratio >= 0.5) & (ratio <= 2.0)
    if bool(amb.any()):
        vv, nn, tt = amb.nonzero(as_tuple=True)
        depth[vv, tt, y[vv, nn], x[vv, nn]] = BACKGROUND
    feat = torch.randn(v, c, fh, fw, generator=gen)
    if bf16:
        feat = feat.bfloat16().float()
    return dict(points=points, projection=proj, depth=depth, prob=prob.float(), feat=feat, vs_z=vs_z,
                h=h, w=w, fh=fh, fw=fw)


def add_blind_views(sc, extra, seed):
    """append ``extra`` views that never pass: the projection of view 0 negated, so z < 0 for
    every voxel (same x, y).  Their features and hypotheses are random."""
    gen = torch.Generator().manual_seed(seed)
    v0, c, fh, fw = sc["feat"].shape
    t = sc["depth"].shape[1]
    out = dict(sc)
    out["projection"] = torch.cat((sc["projection"], -sc["projection"][:1].expand(extra, 3, 4)), 0)
    out["feat"] = torch.cat((sc["feat"], torch.randn(extra, c, fh, fw, generator=gen)), 0)
    if bool((sc["feat"] == sc["feat"].bfloat16().float()).all()):
        out["feat"] = out["feat"].bfloat16().float()
    out["depth"] = torch.cat((sc["depth"], -torch.rand(extra, t, fh, fw, generator=gen) * 4), 0)
    out["prob"] = torch.cat((sc["prob"], 0.05 + torch.rand(extra, t, fh, fw, generator=gen)), 0)
    return out


# --------------------------------------------------------------------------
# constructed exact geometry
# --------------------------------------------------------------------------
EXACT_VS_Z = 0.25
EXACT_H, EXACT_W, EXACT_FH, EXACT_FW, EXACT_T = 6, 6, 8, 9, 3
FAR = 50.0
ULP1 = 2.0 ** -23                     # one ulp above 1.0 (and of 1.25 - 0.25 from below: 1 - 2^-23 is exact)
ROUND_COORDS = (-0.5, 0.5, 1.5, 2.5, EXACT_W - 1.5, EXACT_W - 0.5, float(torch.tensor(-0.50001)))
ROUND_EXPECT = (0, 0, 2, 2, 4, 6, -1)  # half-to-even; 6 == w is outside, -1 is outside
# window row y = 5, x = 0..5: hypothesis 0's depth and whether z = 1 passes it
WINDOW_DEPTHS = (1.25, 0.75, 1.25 - ULP1, 0.75 + ULP1, float("nan"), FAR)
WINDOW_PASS = (False, False, True, True, False, False)


def exact_scene(c=8, seed=0):
    """Three views over a 6x6 crop of an 8x9 map, T = 3, vs_z = 0.25, voxels at Z = 0.

    view 0: rows [1,0,0,0], [0,1,0,0], [0,0,0,1]: z = 1, x = X, y = Y exactly.
      - x rounding: X in ROUND_COORDS at Y = 2 (x = -0.5 -> 0 inside, w - 0.5 -> w outside);
        the same in y at X = 3.  Hypothesis 0 of pixels x (or y) in {0, 2, 4} is 1.0 (passes),
        every other pixel is FAR, so a voxel rounded to the wrong pixel fails.
      - window: row y = 5, x = 0..5, hypothesis 0 = WINDOW_DEPTHS: z == d - vs_z, z == d + vs_z
        (both fail), one ulp inside each edge (both pass), NaN, and at x = 5 a non-passing
        j = 0 next to a passing j = 1 of probability 0 (valid, but no hypothesis is routed).
      - ties: pixel (y=1, x=1) has j = 1 and j = 2 passing with equal probability (route to 1),
        pixel (y=1, x=4) has j = 0 and j = 1 passing with equal probability (route to 0).
    view 1: third row 0: p2 = 0, x = X / 0 is +-inf or NaN: never in bounds.
    view 2: every row negated: x = X, y = Y in bounds but p2 = -1: never passes (its depth map is
      -1 everywhere, which z = -1 would pass).
    Returns the scene and ``expect``: per voxel of view 0 the pixel (x, y), in-bounds, valid and
    the routed hypothesis (-1: none)."""
    vox, expect = [], []
    for xv, ex in zip(ROUND_COORDS, ROUND_EXPECT):
        vox.append((xv, 2.0))
        inb = 0 <= ex < EXACT_W
        expect.append(dict(x=ex, y=2, inb=inb, valid=inb, jstar=0 if inb else -1))
    for yv, ey in zip(ROUND_COORDS, ROUND_EXPECT):
        vox.append((3.0, yv))
        inb = 0 <= ey < EXACT_H
        expect.append(dict(x=3, y=ey, inb=inb, valid=inb, jstar=0 if inb else -1))
    for xi, ok in enumerate(WINDOW_PASS):
        vox.append((float(xi), 5.0))
        valid = ok or xi == 5
        expect.append(dict(x=xi, y=5, inb=True, valid=valid, jstar=0 if ok else -1))
    vox.append((1.0, 1.0))
    expect.append(dict(x=1, y=1, inb=True, valid=True, jstar=1))
    vox.append((4.0, 1.0))
    expect.append(dict(x=4, y=1, inb=True, valid=True, jstar=0))
    points = torch.tensor([[a for a, _ in vox], [b for _, b in vox], [0.0] * len(vox)], dtype=torch.float32)

    p0 = torch.tensor([[1.0, 0, 0, 0], [0, 1.0, 0, 0], [0, 0, 0, 1.0]])
    p1 = torch.tensor([[1.0, 0, 0, 0], [0, 1.0, 0, 0], [0, 0, 0, 0.0]])
    proj = torch.stack((p0, p1, -p0)).float()

    t, fh, fw = EXACT_T, EXACT_FH, EXACT_FW
    depth = torch.full((3, t, fh, fw), FAR)
    prob = torch.full((3, t, fh, fw), 0.5)
    depth[1] = 0.0
    depth[2] = -1.0
    passp = torch.tensor([0.6, 0.25, 0.15])
    for i in (0, 2, 4):
        depth[0, 0, 2, i] = 1.0
        depth[0, 0, i, 3] = 1.0
        prob[0, :, 2, i] = passp
        prob[0, :, i, 3] = passp
    for xi, d in enumerate(WINDOW_DEPTHS):
        depth[0, 0, 5, xi] = d
        prob[0, :, 5, xi] = passp
    depth[0, 1, 5, 5] = 1.0
    prob[0, :, 5, 5] = torch.tensor([0.5, 0.0, 0.5])
    depth[0, :, 1, 1] = torch.tensor([FAR, 1.0, 1.0])
    prob[0, :, 1, 1] = torch.tensor([0.4, 0.3, 0.3])
    depth[0, :, 1, 4] = torch.tensor([1.0, 1.0, FAR])
    prob[0, :, 1, 4] = torch.tensor([0.4, 0.4, 0.2])
    gen = torch.Generator().manual_seed(seed)
    feat = torch.randn(3, c, fh, fw, generator=gen)
    sc = dict(points=points, projection=proj, depth=depth.float(), prob=prob.float(), feat=feat,
              vs_z=EXACT_VS_Z, h=EXACT_H, w=EXACT_W, fh=fh, fw=fw)
    return sc, expect
