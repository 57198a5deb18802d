"""CPU checks of the hand-built back-projection cases (tests/bp_cases.py): the rounding ties are
exact .5, the window edges are exact, the fp32 oracle takes the decisions the cases claim, and the
random scenes keep every decision far from the window edges.  A change to a case builder fails
here, not as a confusing mismatch on the GPU."""
import pytest
import torch

import bp_cases as BC
import ref64


def test_rounding_ties_are_exact_halves():
    x = torch.tensor(BC.ROUND_COORDS, dtype=torch.float32)
    frac = x - torch.floor(x)
    assert (frac[:6] == 0.5).all(), "the first six coordinates must be exact .5 ties"
    assert float(x[6]) < -0.5, "-0.50001 must round below -0.5"
    # half to even, as torch.round (and the kernels' rintf) does
    assert torch.round(x).long().tolist() == list(BC.ROUND_EXPECT)
    # roundf (half away from zero) would differ on four of them: the case can tell the two apart
    away = (torch.sign(x) * torch.floor(x.abs() + 0.5)).long().tolist()
    assert sum(a != b for a, b in zip(away, BC.ROUND_EXPECT)) == 4


def test_window_edges_are_exact():
    vs = torch.tensor(BC.EXACT_VS_Z, dtype=torch.float32)
    d = torch.tensor(BC.WINDOW_DEPTHS, dtype=torch.float32)
    one = torch.tensor(1.0, dtype=torch.float32)
    lo, hi = d - vs, d + vs                           # fp32, as the kernels compute them
    assert float(lo[0]) == 1.0, "z == d - vs_z exactly"
    assert float(hi[1]) == 1.0, "z == d + vs_z exactly"
    assert float(lo[2]) == 1.0 - BC.ULP1 and float(hi[2]) > 1.0, "one ulp inside the lower edge"
    assert float(hi[3]) == 1.0 + BC.ULP1 and float(lo[3]) < 1.0, "one ulp inside the upper edge"
    assert torch.isnan(d[4])
    passed = (one > lo) & (one < hi)
    assert passed.tolist() == list(BC.WINDOW_PASS)
    assert ((one >= lo) & (one <= hi)).tolist() != list(BC.WINDOW_PASS), "closed window must differ"


def test_exact_scene_decisions():
    sc, expect = BC.exact_scene()
    x, y, z = BC.project(sc["points"], sc["projection"])
    assert (z[0] == 1.0).all() and (z[1] == 0.0).all() and (z[2] == -1.0).all()
    crop = lambda t: t[:, :, :sc["h"], :sc["w"]]              # noqa: E731
    dec = ref64.bp_decisions(sc["points"], sc["projection"], crop(sc["depth"]), crop(sc["prob"]),
                             sc["vs_z"], sc["h"], sc["w"])
    for n, e in enumerate(expect):
        got = dict(x=int(dec["x"][0, n]), y=int(dec["y"][0, n]), inb=bool(dec["inb"][0, n]),
                   valid=bool(dec["valid"][0, n]),
                   jstar=int(dec["jstar"][0, n]) if bool(dec["jpass"][0, n]) else -1)
        assert got == e, f"voxel {n} at {tuple(sc['points'][:2, n].tolist())}: {got} != {e}"
    assert not bool(dec["inb"][1:].any()), "views 1 (p2 = 0) and 2 (p2 < 0) are never in bounds"
    # view 2 is in the crop in x and y: only p2 > 0 keeps it out
    assert bool(((x[2] >= 0) & (x[2] < sc["w"]) & (y[2] >= 0) & (y[2] < sc["h"])).any())
    # the two ties are exact in the normalised probabilities
    p = sc["prob"][0]
    pn = p / p.sum(0, keepdim=True)
    assert float(pn[1, 1, 1]) == float(pn[2, 1, 1]) and float(pn[0, 1, 4]) == float(pn[1, 1, 4])


@pytest.mark.parametrize("v,t,seed", [(17, 3, 1), (65, 8, 2), (5, 1, 3)])
def test_random_scene_margins(v, t, seed):
    sc = BC.random_scene(v, 4, t, 300, seed)
    h, w = sc["h"], sc["w"]
    ratio, inb = BC.window_margin(sc["points"], sc["projection"], sc["depth"], sc["vs_z"], h, w)
    r = ratio[inb.unsqueeze(-1).expand_as(ratio)]
    assert bool(((r < 0.5) | (r > 2.0)).all()), "a decision lies within [0.5, 2] vs_z of the window"
    passes = (ratio < 1.0) & inb.unsqueeze(-1)
    frac = float(passes.any(-1).float().mean())
    assert 0.15 < frac < 0.5, f"{frac:.2f} of the (view, voxel) pairs pass; about a third is intended"
    assert bool(passes.any(-1).any(-1).all()), "every view must have passing pairs"
    blind = BC.add_blind_views(sc, 3, seed)
    _, _, z = BC.project(blind["points"], blind["projection"])
    assert bool((z[v:] < 0).all())
