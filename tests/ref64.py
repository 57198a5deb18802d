"""fp64 references with per-element error bounds for the voxel half of the path (back-projection,
view aggregation, prob-norm backward) and for the depth top-k epilogue (test infrastructure).

The integer decisions of the back-projection -- pixel x, y, in-bounds, ``passed[v, n, j]``, the
routed hypothesis j* and ``valid`` -- come from the fp32 oracle (``oracle.mvsdet_oracle.
backproject_weigh``), because the kernels must reproduce the reference's fp32 arithmetic there bit
for bit.  Every float is then recomputed in fp64 from those decisions, next to a bound on how far a
correct fp32 kernel can be from it.  Comparisons are element by element against that bound, never
against the rms of the result, so one mis-weighted view among 100 or a gradient routed to the
wrong hypothesis cannot hide under the bulk of the values.

Bounds use u = 2^-24 (the unit roundoff of a correctly rounded fp32 operation) and the standard
model: a chain of k roundings whose exact terms have absolute values summing to A is off by at most
gamma_k * A, gamma_k = k u / (1 - k u) <= (k + 1) u for the k used here.  The k of each value is
derived in the docstring of the function that builds it.
"""
from __future__ import annotations

import math

import torch

from oracle import mvsdet_oracle as O

U = 2.0 ** -24            # fp32 unit roundoff (round to nearest)
ULP = 2.0 ** -23          # one fp32 ulp of a value in [1, 2), relative: the unit of documented ulp errors
FIXED_HALF = 2.0 ** -33   # rounding of one fp32 contribution to the 2^-32 fixed-point grid of the *_det kernels
MEAN, SUM, PER_VIEW = "mean", "sum", "per_view"


# --------------------------------------------------------------------------
# back-projection
# --------------------------------------------------------------------------
def bp_decisions(points, projection, depth, prob, vs_z, h, w):
    """Integer decisions of the back-projection, from the fp32 oracle on CPU.

    points [3,N], projection [V,3,4], depth / prob [V,T,h,w] (the crop) -> dict of
      x, y [V,N] int64, z [V,N] fp32, inb [V,N], passed [V,N,T], valid [V,N] bool,
      pix [V,N] (y*w + x, 0 where out of bounds), jstar [V,N] (first maximum of the candidate
      weights, as torch.max routes its gradient), jpass [V,N] (j* is itself a passing hypothesis:
      only then does the weight, and its gradient, belong to a probability)."""
    points, projection = points.float().cpu(), projection.float().cpu()
    depth, prob = depth.float().cpu(), prob.float().cpu()
    v, t = depth.shape[:2]
    n = points.shape[1]
    d_r = depth.permute(0, 2, 3, 1).reshape(v, h * w, 1, t)
    p_r = prob.permute(0, 2, 3, 1).reshape(v, h * w, 1, t)
    feats = torch.zeros(v, 1, h, w)             # the decisions do not depend on the features
    _, valid, dbg = O.backproject_weigh(feats, points.reshape(3, n, 1, 1), projection, d_r,
                                        (vs_z, vs_z, vs_z), p_r, return_debug=True)
    inb, passed = dbg["inb"], dbg["passed"]
    pix = torch.where(inb, dbg["y"] * w + dbg["x"], torch.zeros_like(dbg["x"]))
    pf = p_r.reshape(v, h * w, t)
    pn = pf / pf.sum(dim=-1, keepdim=True)
    pn_at = torch.gather(pn, 1, pix.unsqueeze(-1).expand(v, n, t))
    cand = torch.where(passed, pn_at, torch.zeros_like(pn_at))
    best = cand.max(dim=-1, keepdim=True).values
    jstar = (cand == best).int().argmax(dim=-1)          # first maximal index
    jpass = torch.gather(passed, 2, jstar.unsqueeze(-1)).squeeze(-1)
    return dict(x=dbg["x"], y=dbg["y"], z=dbg["z"], inb=inb, passed=passed,
                valid=valid.reshape(v, n), pix=pix, jstar=jstar, jpass=jpass)


def bp_reference(feat, dec, prob, mode, g_out=None):
    """fp64 back-projection forward (and, with ``g_out``, backward) from the oracle's decisions.

    feat [V,C,h,w] (the crop, fp32 values; bf16 features are given here already rounded, so the
    bound stays the fp32 one), prob [V,T,h,w], mode "mean" | "sum" | "per_view".
    g_out: [C,N] (aggregating modes) or [V,C,N] (per view).

    Returns a dict of (value, bound) pairs and exact integers:
      count [N], valid [V,N]
      out   [C,N] or [V,C,N]
      g_feat [V,C,h,w], g_pn [V,T,h,w], g_prob [V,T,h,w]   (with g_out)
      g_feat_det, g_pn_det  bounds of the deterministic (fixed-point) backward

    Derivation of the bounds (T hypotheses, m = number of terms of a sum):
      weight   pn = p_j* / sum_T p: the fp32 sum has T - 1 roundings, the division one: T.
      out      term = feat * weight: T + 1; summed over m views in view order: m - 1 more,
               so k = m + T (+1 for gamma).  MEAN divides by fl(count + 1e-8) = count (1e-8 is
               below half an ulp of any count >= 1) where the reference divides by count + 1e-8:
               one rounding plus 1e-8 relative, k += 2.  PER_VIEW: one term, k = T + 2.
      g_feat   term = fl(g / den) * weight: T + 1 (+2 MEAN); m terms RED-added in any order:
               k = m + T + 1 (+2).
      g_pn     dot over C: each lane runs 4 G fmas (G = ceil(C/128) channel slices), then a
               5-level butterfly: 4 G + 5 roundings (+2 MEAN for g / den); m voxels atomically
               added: k = 4 G + 5 + m (+2).
      g_prob   g_m / S - (sum_j g_j p_j) / S^2 in fp32 (S: T - 1 roundings, 1/S: 1, the dot:
               T fmas, the fma and the product: 2) gives 3 T + 4 on |g_m| / S + sum_j |g_j| p_j / S^2;
               the error of the kernel's own g_pn (bound b) adds (b_m + sum_j b_j p_j / S) / S.
      *_det    every fp32 contribution has the term error of the default form (no summation
               error: integer adds are exact), is rounded to the 2^-32 grid (<= 2^-33 each) and the
               exact sum is rounded to fp32 once: T + 2 (+2) per term, m * 2^-33, u * |result|.
    """
    feat = feat.double().cpu()
    p64 = prob.double().cpu()
    v, c, h, w = feat.shape
    t = p64.shape[1]
    n = dec["valid"].shape[1]
    valid, pix, jstar = dec["valid"], dec["pix"], dec["jstar"]
    routed = valid & dec["jpass"]                                  # weight = pn[j*]
    pn = (p64 / p64.sum(dim=1, keepdim=True)).reshape(v, t, h * w)
    pn_flat = pn.permute(0, 2, 1)                                   # [V,hw,T]
    w64 = pn_flat[torch.arange(v).unsqueeze(1), pix, jstar]         # [V,N]
    w64 = torch.where(routed, w64, torch.zeros_like(w64))
    fflat = feat.reshape(v, c, h * w)
    f_at = torch.gather(fflat, 2, pix.unsqueeze(1).expand(v, c, n))  # [V,C,N]
    f_at = torch.where(valid.unsqueeze(1), f_at, torch.zeros_like(f_at))
    terms = f_at * w64.unsqueeze(1)                                  # [V,C,N]
    count = valid.sum(dim=0)                                         # [N]
    res = dict(count=count.to(torch.int32), valid=valid)
    mean = mode == MEAN
    if mode == PER_VIEW:
        res["out"] = (terms, (t + 2) * U * terms.abs())
    else:
        s = terms.sum(dim=0)
        a = terms.abs().sum(dim=0)
        k = count.double() + t + 1
        if mean:
            den = count.double() + 1e-8
            nz = count > 0
            res["out"] = (torch.where(nz, s / den, torch.zeros_like(s)),
                          torch.where(nz, (k + 2) * U * a / den, torch.zeros_like(a)))
        else:
            res["out"] = (s, k * U * a)
    if g_out is None:
        return res

    g = g_out.double().cpu()
    if mean:
        den = count.double() + 1e-8
        g = torch.where(count > 0, g / den, torch.zeros_like(g))
    gv = g.unsqueeze(0).expand(v, c, n) if mode != PER_VIEW else g      # [V,C,N]
    gv = torch.where(valid.unsqueeze(1), gv, torch.zeros_like(gv))
    extra = 2 if mean else 0
    flat = (torch.arange(v).unsqueeze(1) * (h * w) + pix)                # [V,N] into [V*hw]
    sel = valid.reshape(-1)
    idx = flat.reshape(-1)[sel]

    # g_feat[v, :, pix] += g_vol[:, n] * weight[v, n]
    gterm = (gv * w64.unsqueeze(1)).permute(0, 2, 1).reshape(v * n, c)[sel]
    gf = torch.zeros(v * h * w, c, dtype=torch.float64).index_add_(0, idx, gterm)
    ga = torch.zeros(v * h * w, c, dtype=torch.float64).index_add_(0, idx, gterm.abs())
    m = torch.zeros(v * h * w, dtype=torch.float64).index_add_(0, idx, torch.ones(idx.numel(), dtype=torch.float64))
    m = m.unsqueeze(1)

    def nchw(x):
        return x.reshape(v, h, w, c).permute(0, 3, 1, 2)
    res["g_feat"] = (nchw(gf), nchw((m + t + 2 + extra) * U * ga))
    res["g_feat_det"] = (nchw(gf), nchw((t + 3 + extra) * U * ga + m * FIXED_HALF + U * gf.abs()))

    # g_pn[v, j*, pix] += sum_c g_vol[c, n] feat[v, c, pix]   (only where j* passes)
    dot = (gv * f_at).sum(dim=1)                                         # [V,N]
    dota = (gv * f_at).abs().sum(dim=1)
    rsel = routed.reshape(-1)
    pidx = (torch.arange(v).unsqueeze(1) * (t * h * w) + jstar * (h * w) + pix).reshape(-1)[rsel]
    gp = torch.zeros(v * t * h * w, dtype=torch.float64).index_add_(0, pidx, dot.reshape(-1)[rsel])
    gpa = torch.zeros(v * t * h * w, dtype=torch.float64).index_add_(0, pidx, dota.reshape(-1)[rsel])
    mp = torch.zeros(v * t * h * w, dtype=torch.float64).index_add_(
        0, pidx, torch.ones(pidx.numel(), dtype=torch.float64))
    g_slices = (c + 127) // 128
    gp, gpa, mp = (x.reshape(v, t, h, w) for x in (gp, gpa, mp))
    b_pn = (4 * g_slices + 6 + extra + mp) * U * gpa
    b_pn_det = (4 * g_slices + 6 + extra) * U * gpa + mp * FIXED_HALF + U * gp.abs()
    res["g_pn"] = (gp, b_pn)
    res["g_pn_det"] = (gp, b_pn_det)
    res["g_prob"] = prob_norm_reference(p64, gp, b_pn)
    res["g_prob_det"] = prob_norm_reference(p64, gp, b_pn_det)
    return res


def prob_norm_reference(prob, g_pn, b_pn):
    """pn = p / sum_T p backward in fp64: g_p_m = g_m / S - (sum_j g_j p_j) / S^2, with the bound
    derived in ``bp_reference`` (prob, g_pn, b_pn: [V,T,h,w])."""
    p = prob.double()
    t = p.shape[1]
    s = p.sum(dim=1, keepdim=True)
    dot = (g_pn * p).sum(dim=1, keepdim=True)
    val = g_pn / s - dot / (s * s)
    mag = ((g_pn.abs() + b_pn) + ((g_pn.abs() + b_pn) * p).sum(dim=1, keepdim=True) / s) / s
    prop = (b_pn + (b_pn * p).sum(dim=1, keepdim=True) / s) / s
    return val, prop + (3 * t + 5) * U * mag


# --------------------------------------------------------------------------
# depth top-k
# --------------------------------------------------------------------------
class B:
    """A value computed in fp64 with a bound on how far the kernel's fp32 evaluation of the same
    expression, operation by operation, can be from it (first-order error propagation plus the
    rounding of each fp32 operation).  ``v`` is the exact value of the expression for the fp32
    inputs (to fp64 accuracy), ``e`` the bound."""

    __slots__ = ("v", "e")

    def __init__(self, v, e=None):
        self.v = v
        self.e = torch.zeros_like(v) if e is None else e

    @staticmethod
    def _r(v, e, k=1.0):
        return B(v, e + k * U * (v.abs() + e))

    def __add__(self, o):
        o = _b(o)
        return B._r(self.v + o.v, self.e + o.e)

    def __sub__(self, o):
        o = _b(o)
        return B._r(self.v - o.v, self.e + o.e)

    def __mul__(self, o):
        o = _b(o)
        return B._r(self.v * o.v, self.v.abs() * o.e + o.v.abs() * self.e + self.e * o.e)

    def __truediv__(self, o):
        return self.div(o)

    def div(self, o, ulps=None):
        """IEEE division (one rounding) or, with ``ulps``, an approximate one of that max error"""
        o = _b(o)
        v = self.v / o.v
        e = (self.e + v.abs() * o.e) / (o.v.abs() - o.e)
        if ulps is None:
            return B._r(v, e)
        return B(v, e + ulps * ULP * (v.abs() + e))

    def fma(self, b, c):
        """fl(self * b + c): one rounding"""
        b, c = _b(b), _b(c)
        v = self.v * b.v + c.v
        return B._r(v, self.v.abs() * b.e + b.v.abs() * self.e + self.e * b.e + c.e)

    def exp(self, ulps):
        """exp with a documented max error of ``ulps`` (a tensor or number) ulps; a -inf argument
        gives an exact 0"""
        v = torch.exp(self.v)
        prop = v * torch.expm1(self.e)
        prop = torch.where(torch.isinf(self.v), torch.zeros_like(v), prop)
        ulps = torch.as_tensor(ulps, dtype=torch.float64)
        ulps = torch.where(torch.isinf(self.v), torch.zeros_like(v), ulps.expand_as(v))
        # results below the normal range lose relative precision: an absolute 2^-126 covers them
        return B(v, prop + ulps * ULP * (v + prop) + 2.0 ** -126)


def _b(x):
    if isinstance(x, B):
        return x
    if not torch.is_tensor(x):
        x = torch.tensor(float(x), dtype=torch.float64)
    return B(x.double())


def topk_forward_reference(cost, near, interval, raw=False):
    """fp64 forward of the top-k epilogue for cost [V,2,D,H,W] (fp32 values) with bounds for the
    kernel's fp32 evaluation (``depth_topk_fwd_kernel``, op by op):

      a_d = fl(c_d - max) (one rounding, relative |a_d| u on exp), e_d = expf(a_d) (2 ulp),
      S = sum in plane order (D - 1 roundings), prob_d = e_d / S (one rounding);
      off_d = 1 / (1 + expf(-o_d)) (2 ulp, one add, one division);
      depth_d = fl(fl(fl(d I) + near) + fl(off_d I));
      coding = fmaf chain over d (D roundings).
    ``raw``: channel 0 / 1 already hold probabilities / offsets (pass-through).
    Returns B's prob, off [V,D,H,W], depth [V,D,H,W] and coding [V,H,W]."""
    c = cost.double().cpu()
    x, o = c[:, 0], c[:, 1]
    d = x.shape[1]
    if raw:
        prob, off = B(x), B(o)
    else:
        mx = x.max(dim=1, keepdim=True).values
        a = B._r(x - mx, torch.zeros_like(x))
        e = a.exp(2.0)
        s = B(e.v[:, 0], e.e[:, 0])
        for i in range(1, d):
            s = s + B(e.v[:, i], e.e[:, i])
        prob = e.div(B(s.v.unsqueeze(1), s.e.unsqueeze(1)))
        eo = B(-o).exp(2.0)
        off = B(torch.ones_like(o)).div(eo + 1.0)
    planes = torch.arange(d, dtype=torch.float64).view(1, d, 1, 1)
    dep = (B(planes * interval, U * (planes * interval).abs()) + near) + off * interval
    coding = None
    for i in range(d):
        pi, di = B(prob.v[:, i], prob.e[:, i]), B(dep.v[:, i], dep.e[:, i])
        coding = (pi * di) if coding is None else pi.fma(di, coding)
    return prob, off, dep, coding


def topk_backward_bound(cost, est_idx, grads, near, interval, raw=False):
    """Bound on dL/dcost_out of ``depth_topk_bwd_kernel`` (the FAST form) against fp64 autograd.

    The backward recomputes the probabilities with ``__expf`` -- max error 2 + floor(|1.173 a|) ulp
    for argument a (CUDA C Programming Guide, intrinsic functions) -- and ``__fdividef`` -- max
    error 2 ulp for divisors in [2^-126, 2^126] -- then, op by op:
      gp_d = fmaf(gcod, depth_d, g_prob_d);  gs_d = fmaf(fl(gcod p_d), I, g_off_d)
      gp_idx += g_dens;  gs_idx = fmaf(g_depth, I, gs_idx)        (t = 0 .. T-1)
      dot = fmaf chain of p_d gp_d;  g_c_d = fl(p_d fl(gp_d - dot));  g_o_d = fl(fl(gs_d s_d)(1 - s_d)).
    The fp32 compiler may contract ``gp_d - dot`` products no further (each step above is written
    with its rounding).  grads = (g_prob, g_off, g_depth, g_dens, g_coding), fp32 values."""
    c = cost.double().cpu()
    x, o = c[:, 0], c[:, 1]
    v, d, h, w = x.shape
    g_prob, g_off, g_depth, g_dens, g_coding = (B(g.double().cpu()) for g in grads)
    idx = est_idx.cpu()
    if raw:
        prob, off = B(x), B(o)
    else:
        mx = x.max(dim=1, keepdim=True).values
        a = B._r(x - mx, torch.zeros_like(x))
        e = a.exp(2.0 + torch.floor(1.173 * (a.v.abs() + a.e)))
        s = B(e.v[:, 0], e.e[:, 0])
        for i in range(1, d):
            s = s + B(e.v[:, i], e.e[:, i])
        inv = B(torch.ones_like(s.v)).div(s, ulps=2.0)
        prob = e * B(inv.v.unsqueeze(1), inv.e.unsqueeze(1))
        eo = B(-o).exp(2.0 + torch.floor(1.173 * o.abs()))
        off = B(torch.ones_like(o)).div(eo + 1.0, ulps=2.0)
    planes = torch.arange(d, dtype=torch.float64).view(1, d, 1, 1)
    dep = (B(planes * interval, U * (planes * interval).abs()) + near) + off * interval
    gc = B(g_coding.v.unsqueeze(1), g_coding.e.unsqueeze(1))
    gp = gc.fma(dep, g_prob)
    gs = (gc * prob).fma(B(torch.full_like(x, interval)), g_off)
    gpv, gpe, gsv, gse = gp.v.clone(), gp.e.clone(), gs.v.clone(), gs.e.clone()
    for t in range(idx.shape[1]):
        it = idx[:, t:t + 1]
        cur_p = B(torch.gather(gpv, 1, it), torch.gather(gpe, 1, it)) + B(g_dens.v[:, t:t + 1])
        cur_s = B(g_depth.v[:, t:t + 1]).fma(B(torch.full_like(cur_p.v, interval)),
                                             B(torch.gather(gsv, 1, it), torch.gather(gse, 1, it)))
        gpv.scatter_(1, it, cur_p.v), gpe.scatter_(1, it, cur_p.e)
        gsv.scatter_(1, it, cur_s.v), gse.scatter_(1, it, cur_s.e)
    gp, gs = B(gpv, gpe), B(gsv, gse)
    dot = None
    for i in range(d):
        pi, gi = B(prob.v[:, i], prob.e[:, i]), B(gp.v[:, i], gp.e[:, i])
        dot = (pi * gi) if dot is None else pi.fma(gi, dot)
    if raw:
        return gp.e, gs.e
    g0 = prob * (gp - B(dot.v.unsqueeze(1), dot.e.unsqueeze(1)))
    g1 = (gs * off) * (B(torch.ones_like(o)) - off)
    return g0.e, g1.e


def topk_autograd_reference(cost, est_idx, grads, near, interval, raw=False):
    """fp64 autograd of softmax / sigmoid / plane depths / gather / expectation
    (mvsdet.py:470-482, :266-283, :298-317) -> dL/dcost_out [V,2,D,H,W]"""
    c = cost.double().cpu().clone().requires_grad_(True)
    x, o = c[:, 0], c[:, 1]
    d = x.shape[1]
    prob, off = (x, o) if raw else (torch.softmax(x, dim=1), torch.sigmoid(o))
    planes = torch.arange(d, dtype=torch.float64).view(1, d, 1, 1)
    dep = planes * interval + near + off * interval
    idx = est_idx.cpu()
    est_depth = torch.gather(dep, 1, idx)
    est_dens = torch.gather(prob, 1, idx)
    coding = (prob * dep).sum(dim=1)
    outs = (prob, off, est_depth, est_dens, coding)
    g, = torch.autograd.grad(outs, (c,), [gi.double().cpu() for gi in grads])
    return g


def check_bound(got, ref, bound, what, exact_zero_ok=True):
    """element-wise |got - ref| <= bound; the message reports the worst element and the largest
    ratio err / bound (how much of the bound a correct kernel uses)."""
    got = got.detach().double().cpu()
    ref, bound = ref.double(), bound.double()
    assert got.shape == ref.shape, f"{what}: shape {tuple(got.shape)} vs {tuple(ref.shape)}"
    err = (got - ref).abs()
    err = torch.where(torch.isnan(got) | torch.isnan(ref), torch.full_like(err, math.inf), err)
    bad = err > bound
    ratio = torch.where(bound > 0, err / bound, torch.where(err > 0, torch.full_like(err, math.inf), 0 * err))
    worst = int(ratio.reshape(-1).argmax()) if ratio.numel() else 0
    msg = (f"{what}: {int(bad.sum())}/{bad.numel()} elements outside the fp64 bound; worst at flat index "
           f"{worst}: got {float(got.reshape(-1)[worst]):.9g} ref {float(ref.reshape(-1)[worst]):.9g} "
           f"err {float(err.reshape(-1)[worst]):.3e} bound {float(bound.reshape(-1)[worst]):.3e}")
    assert not bool(bad.any()), msg
    return float(ratio.max()) if ratio.numel() else 0.0, float(err.max()) if err.numel() else 0.0
