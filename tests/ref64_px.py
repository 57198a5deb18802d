"""fp64 references with per-element bounds for the depth top-k over per-pixel depth hypotheses
(``depth_topk_{fwd,bwd}_kernel<DMAX, PX = true>``), built from ``ref64.B`` the way
``ref64.topk_forward_reference`` / ``ref64.topk_backward_bound`` are for the per-view planes
(test infrastructure).

Per pixel, z_d = depth_values[v,d,y,x] and I = interval_map[v,y,x] (or the scalar interval) take the
place of fl(fl(d*interval) + near) and interval:  depth_d = fl(z_d + fl(off_d I)).
"""
from __future__ import annotations

import torch

import ref64
from ref64 import B


def _col(x, i):
    return B(x.v[:, i], x.e[:, i])


def fp32(x):
    """a scalar interval as the kernels receive it: rounded to fp32 by the C ABI's float argument"""
    return float(torch.tensor(float(x), dtype=torch.float32))


def _interval(interval, like):
    """-> exact B of I broadcast against [V,1,H,W]"""
    if torch.is_tensor(interval):
        return B(interval.double().cpu().unsqueeze(1))
    return B(torch.full_like(like[:, :1], fp32(interval)))


def px_forward_reference(cost, depth_values, interval, raw=False):
    """fp64 forward with bounds: B's prob, off, depth [V,D,H,W] and coding [V,H,W].  prob and off
    are those of ``ref64.topk_forward_reference`` (the same softmax / sigmoid code)."""
    prob, off, _, _ = ref64.topk_forward_reference(cost, 0.0, 1.0, raw=raw)
    z = B(depth_values.double().cpu())
    dep = z + off * _interval(interval, z.v)
    coding = None
    for i in range(dep.v.shape[1]):
        pi, di = _col(prob, i), _col(dep, i)
        coding = (pi * di) if coding is None else pi.fma(di, coding)
    return prob, off, dep, coding


def _fast_prob_off(cost, raw):
    """the backward's recomputed probabilities and offsets (``__expf``, ``__fdividef``), as
    ``ref64.topk_backward_bound`` bounds them"""
    c = cost.double().cpu()
    x, o = c[:, 0], c[:, 1]
    if raw:
        return B(x), B(o)
    mx = x.max(dim=1, keepdim=True).values
    a = B._r(x - mx, torch.zeros_like(x))
    e = a.exp(2.0 + torch.floor(1.173 * (a.v.abs() + a.e)))
    s = _col(e, 0)
    for i in range(1, x.shape[1]):
        s = s + _col(e, i)
    inv = B(torch.ones_like(s.v)).div(s, ulps=2.0)
    prob = e * B(inv.v.unsqueeze(1), inv.e.unsqueeze(1))
    eo = B(-o).exp(2.0 + torch.floor(1.173 * o.abs()))
    off = B(torch.ones_like(o)).div(eo + 1.0, ulps=2.0)
    return prob, off


def _scatter_add(x, idx, val, fma_with=None):
    """x[idx] = x[idx] + val (or fmaf(val, fma_with, x[idx])) along dim 1, in B arithmetic"""
    cur = B(torch.gather(x.v, 1, idx), torch.gather(x.e, 1, idx))
    new = cur + val if fma_with is None else val.fma(fma_with, cur)
    v, e = x.v.clone(), x.e.clone()
    v.scatter_(1, idx, new.v)
    e.scatter_(1, idx, new.e)
    return B(v, e)


def px_backward_bound(cost, depth_values, interval, est_idx, g_prob, g_off, g_depth, g_dens, g_coding,
                      raw=False):
    """Bounds of the PX backward against fp64 autograd, op by op:
      gp_d = fmaf(gcod, depth_d, g_prob_d);  gcp_d = fl(gcod p_d);  gs_d = fmaf(gcp_d, I, g_off_d)
      gp_idx = fl(gp_idx + g_dens_t);  gs_idx = fmaf(gz_t, I, gs_idx)          (t = 0 .. T-1)
      g_cost as ``ref64.topk_backward_bound``
      g_z_d = gcp_d, then g_z_idx = fl(g_z_idx + gz_t);
      g_I = fmaf(gcod, sum_ps, g_int), sum_ps = fmaf chain of p_d s_d, g_int = fmaf chain of gz_t s_idx_t.
    g_depth (gz) and g_coding (gcod) are B's [V,T,H,W] and [V,H,W] (they carry the ray terms'
    rounding), the other gradients fp32 tensors.  -> bounds (g_logits, g_offsets, g_z, g_I)."""
    prob, off = _fast_prob_off(cost, raw)
    z = B(depth_values.double().cpu())
    iv = _interval(interval, z.v)
    dep = z + off * iv
    gc = B(g_coding.v.unsqueeze(1), g_coding.e.unsqueeze(1))
    gp = gc.fma(dep, B(g_prob.double().cpu()))
    gcp = gc * prob
    gs = gcp.fma(iv, B(g_off.double().cpu()))
    gz_map = gcp
    idx = est_idx.cpu()
    dens = B(g_dens.double().cpu())
    ivt = B(iv.v.expand(-1, 1, -1, -1).clone())
    for t in range(idx.shape[1]):
        it = idx[:, t:t + 1]
        gp = _scatter_add(gp, it, B(dens.v[:, t:t + 1]))
        gs = _scatter_add(gs, it, B(g_depth.v[:, t:t + 1], g_depth.e[:, t:t + 1]), fma_with=ivt)
    for t in range(idx.shape[1]):
        gz_map = _scatter_add(gz_map, idx[:, t:t + 1], B(g_depth.v[:, t:t + 1], g_depth.e[:, t:t + 1]))
    dot = None
    sum_ps = None
    for i in range(prob.v.shape[1]):
        pi, gi, si = _col(prob, i), _col(gp, i), _col(off, i)
        dot = (pi * gi) if dot is None else pi.fma(gi, dot)
        sum_ps = (pi * si) if sum_ps is None else pi.fma(si, sum_ps)
    g_int = B(torch.zeros_like(g_coding.v))
    for t in range(idx.shape[1]):
        st = torch.gather(off.v, 1, idx[:, t:t + 1])[:, 0]
        se = torch.gather(off.e, 1, idx[:, t:t + 1])[:, 0]
        g_int = B(g_depth.v[:, t], g_depth.e[:, t]).fma(B(st, se), g_int)
    g_i = g_coding.fma(sum_ps, g_int)
    if raw:
        return gp.e, gs.e, gz_map.e, g_i.e
    g0 = prob * (gp - B(dot.v.unsqueeze(1), dot.e.unsqueeze(1)))
    g1 = (gs * off) * (B(torch.ones_like(off.v)) - off)
    return g0.e, g1.e, gz_map.e, g_i.e


def px_restatement(cost, depth_values, interval, est_idx, raw=False, dtype=torch.float64):
    """autograd restatement (softmax, sigmoid, z + off*I, gather with the kernel's est_idx,
    expectation) -> (leaves (cost, depth_values, interval map or None), outputs
    (prob, off, est_depth, est_dens, coding))"""
    c = cost.detach().to(dtype).cpu().requires_grad_(True)
    z = depth_values.detach().to(dtype).cpu().requires_grad_(True)
    imap = interval.detach().to(dtype).cpu().requires_grad_(True) if torch.is_tensor(interval) else None
    iv = imap.unsqueeze(1) if imap is not None else fp32(interval)
    x, o = c[:, 0], c[:, 1]
    prob, off = (x, o) if raw else (torch.softmax(x, dim=1), torch.sigmoid(o))
    dep = z + off * iv
    idx = est_idx.cpu()
    outs = (prob, off, torch.gather(dep, 1, idx), torch.gather(prob, 1, idx), (prob * dep).sum(dim=1))
    return (c, z, imap), outs


def decided_ranks(prob_ref, bound, t):
    """[V,T,H,W] mask of the hypotheses whose rank fp64 decides (gap to the neighbours above and
    below larger than 8 ulp and the two bounds), and fp64's own top-T order"""
    srt, order = torch.sort(prob_ref, dim=1, descending=True, stable=True)
    eb = torch.gather(bound, 1, order)
    apart = (srt[:, :-1] - srt[:, 1:]) > torch.maximum(8 * ref64.ULP * srt[:, :-1].abs(), eb[:, :-1] + eb[:, 1:])
    sure = torch.ones(order[:, :t].shape, dtype=torch.bool)
    d = srt.shape[1]
    for i in range(t):
        if i > 0:
            sure[:, i] &= apart[:, i - 1]
        if i + 1 < d:
            sure[:, i] &= apart[:, i]
    return sure, order[:, :t]
