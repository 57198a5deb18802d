"""Back-projection, view aggregation, prob-norm backward and voxel normalisation at their view,
channel, hypothesis, voxel-tail and rounding edges, against the fp64 reference of tests/ref64.py.

Inputs are built directly (tests/bp_cases.py), not through make_scene, so V = 100 stays cheap.
Counts and per-view masks are compared bit for bit; every float element by element against its
fp64 error bound.  Gradients are taken through the production autograd path with the shared fp32
accumulator (``pack_features(..., sink=True)``), so bf16 features get an fp32 gradient.
"""
import pytest
import torch

import bp_cases as BC
import ref64
from mvsdet_b200 import _lib, ops

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


def _crop(t, sc):
    return t[:, :, :sc["h"], :sc["w"]]


def _hyp(t, strided):
    """[V,T,fh,fw] on the GPU; ``strided``: a row-cropped view of a taller map (gaps between the
    T planes), the ``_zeros_strided_like`` path of the backward"""
    t = t.to(DEV)
    if not strided:
        return t
    big = torch.full((t.shape[0], t.shape[1], t.shape[2] + 3, t.shape[3]), 7.0, device=DEV)
    big[:, :, 1:1 + t.shape[2]] = t
    return big[:, :, 1:1 + t.shape[2]]


def run(sc, mode, channels_first=True, fdtype=torch.float32, det=False, strided=False, g_seed=0):
    """one forward + backward through ops -> dict of CPU results and the upstream gradient"""
    v, c = sc["feat"].shape[:2]
    n = sc["points"].shape[1]
    x = sc["feat"].to(DEV).requires_grad_(True)
    dens_leaf = sc["prob"].clone().requires_grad_(True)
    dens = _hyp(dens_leaf, strided)
    depth = _hyp(sc["depth"], strided)
    pts, proj = sc["points"].to(DEV), sc["projection"].to(DEV)
    gen = torch.Generator().manual_seed(1000 + g_seed)
    out = {}
    if mode == ref64.PER_VIEW:
        packed = ops.pack_features(x, fdtype)
        h, w = sc["h"], sc["w"]
        dr = _crop(depth, sc).permute(0, 2, 3, 1).reshape(v, h * w, 1, -1)
        pr = _crop(dens, sc).permute(0, 2, 3, 1).reshape(v, h * w, 1, -1)
        vol, valid = ops.backproject_per_view(packed, pts, proj, dr, pr, sc["vs_z"], h, w)
        out["valid"] = valid.cpu()
        g_out = torch.randn(v, c, n, generator=gen)
    else:
        packed, sink = ops.pack_features(x, fdtype, sink=True, deterministic=det)
        vol, cnt = ops.backproject_aggregate(packed, pts, proj, depth, dens, sc["vs_z"], sc["h"], sc["w"],
                                             mode=mode, channels_first=channels_first, grad_sink=sink)
        out["count"] = cnt.cpu()
        g_out = torch.randn(c, n, generator=gen)
    out["out"] = vol.detach().cpu()
    g_x, g_dens = torch.autograd.grad(vol, (x, dens_leaf), g_out.to(DEV))
    out["g_feat"], out["g_prob"] = g_x.cpu(), g_dens.cpu()
    out["g_out"] = g_out
    return out


def reference(sc, mode, g_out):
    dec = ref64.bp_decisions(sc["points"], sc["projection"], _crop(sc["depth"], sc), _crop(sc["prob"], sc),
                             sc["vs_z"], sc["h"], sc["w"])
    return ref64.bp_reference(_crop(sc["feat"], sc), dec, _crop(sc["prob"], sc), mode, g_out)


def check(sc, got, ref, what, det=False):
    if "count" in got:
        assert torch.equal(got["count"], ref["count"]), f"{what}: count differs from the oracle's decisions"
    if "valid" in got:
        assert torch.equal(got["valid"], ref["valid"]), f"{what}: per-view valid differs from the oracle"
    ref64.check_bound(got["out"], *ref["out"], f"{what}: volume")
    gf, bf = ref["g_feat_det" if det else "g_feat"]
    h, w = sc["h"], sc["w"]
    ref64.check_bound(_crop(got["g_feat"], sc), gf, bf, f"{what}: dL/dfeat")
    ref64.check_bound(_crop(got["g_prob"], sc), *ref["g_prob_det" if det else "g_prob"], f"{what}: dL/dprob")
    outside = torch.ones(got["g_feat"].shape[2:], dtype=torch.bool)
    outside[:h, :w] = False
    assert not bool(got["g_feat"][:, :, outside].any()), f"{what}: gradient outside the crop"
    assert not bool(got["g_prob"][:, :, outside].any()), f"{what}: dL/dprob outside the crop"


FDT = {"f32": torch.float32, "bf16": torch.bfloat16}


@pytest.mark.parametrize("fdt", ["f32", "bf16"])
@pytest.mark.parametrize("cfirst", [True, False])
@pytest.mark.parametrize("v", [1, 15, 16, 17, 31, 32, 33, 64, 65, 100])
def test_views(v, cfirst, fdt):
    """32 views per ballot, the pair kernel up to 16 views and the loop kernel from 17: every view
    count around those edges, MEAN mode, C = 256"""
    sc = BC.random_scene(v, 256, 3, 210, seed=v, bf16=fdt == "bf16")
    got = run(sc, ref64.MEAN, cfirst, FDT[fdt], g_seed=v)
    check(sc, got, reference(sc, ref64.MEAN, got["g_out"]), f"V={v} cfirst={cfirst} {fdt}")


@pytest.mark.parametrize("fdt", ["f32", "bf16"])
@pytest.mark.parametrize("v", [5, 17])
@pytest.mark.parametrize("c", [4, 124, 128, 132, 256, 260, 384, 388, 508, 512])
def test_channels(c, v, fdt):
    """1, 2 and 4 slices of 128 channels with the 128 g + 4 lane >= C guard, in both kernel forms"""
    sc = BC.random_scene(v, c, 2, 100, seed=c + v, bf16=fdt == "bf16")
    mode = ref64.SUM if c % 8 else ref64.MEAN          # the ragged widths also run the SUM mode
    got = run(sc, mode, c % 3 == 0, FDT[fdt], g_seed=c)
    check(sc, got, reference(sc, mode, got["g_out"]), f"C={c} V={v} {fdt}")


@pytest.mark.parametrize("t", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("mode", [ref64.MEAN, ref64.SUM, ref64.PER_VIEW])
def test_modes_and_hypotheses(mode, t):
    sc = BC.random_scene(20, 64, t, 150, seed=40 + t)
    got = run(sc, mode, True, g_seed=t)
    check(sc, got, reference(sc, mode, got["g_out"]), f"{mode} T={t}")


@pytest.mark.parametrize("cfirst", [True, False])
@pytest.mark.parametrize("n", [1, 31, 33, 32 * 5 + 7])
def test_voxel_tails(n, cfirst):
    """a last CTA with 1..31 voxels: with channels_first its transposed tile is only partly stored"""
    sc = BC.random_scene(9, 132, 3, n, seed=n)
    got = run(sc, ref64.MEAN, cfirst, g_seed=n)
    check(sc, got, reference(sc, ref64.MEAN, got["g_out"]), f"N={n} cfirst={cfirst}")


def test_strided_hypotheses():
    """hypotheses as a row-cropped view: the kernels read the strides, the backward allocates its
    gradients with the same strides"""
    sc = BC.random_scene(17, 128, 3, 120, seed=77)
    got = run(sc, ref64.MEAN, True, strided=True, g_seed=77)
    check(sc, got, reference(sc, ref64.MEAN, got["g_out"]), "strided hypotheses")


@pytest.mark.parametrize("mode", [ref64.MEAN, ref64.SUM, ref64.PER_VIEW])
@pytest.mark.parametrize("extra", [0, 14])
def test_exact_geometry(mode, extra):
    """the constructed exact cases (tests/bp_cases.exact_scene): half-to-even rounding at -0.5 /
    w - 0.5, the strict window at z == d +- vs_z and one ulp inside, p2 = 0 and p2 < 0, NaN depth,
    equal-probability ties routed to the lower j, a passing j of probability 0; ``extra`` appends
    never-passing views so the loop kernel (V = 17) runs them too"""
    sc, expect = BC.exact_scene(c=8)
    if extra:
        sc = BC.add_blind_views(sc, extra, seed=5)
    got = run(sc, mode, True)
    ref = reference(sc, mode, got["g_out"])
    check(sc, got, ref, f"exact geometry {mode} V={sc['feat'].shape[0]}")
    want_valid = torch.tensor([e["valid"] for e in expect])
    assert torch.equal(ref["valid"][0], want_valid)
    if mode == ref64.PER_VIEW:
        assert torch.equal(got["valid"][0], want_valid)
        assert not bool(got["valid"][1:].any())
    else:
        assert torch.equal(got["count"], want_valid.int())
    # routing: the reference's dL/dpn lands only on the expected hypothesis (the kernel's is checked
    # through dL/dprob above, whose bound is 0 wherever no gradient is routed)
    gp, _ = ref["g_pn"]
    for n, e in enumerate(expect):
        if e["valid"]:
            row = gp[0, :, e["y"], e["x"]]
            want = [e["jstar"]] if e["jstar"] >= 0 else []
            assert row.nonzero().flatten().tolist() == want, f"voxel {n}: routed to {row.tolist()}"
    assert bool(got["g_prob"][0, :, 5, 5].eq(0).all()), "a probability-0 passing hypothesis got a gradient"


def _blind_pair(v0=16, extras=(1, 17, 49), seed=3):
    base = BC.random_scene(v0, 256, 3, 150, seed=seed)
    return base, [BC.add_blind_views(base, e, seed=seed + e) for e in extras]


@pytest.mark.parametrize("cfirst", [True, False])
def test_same_bits_in_both_kernel_forms(cfirst):
    """V = 16 (pair kernel) and the same scene padded with never-passing views to V = 17, 33, 65
    (loop kernel): both gather in ascending view order, so the volume and the count are the same
    bits; the deterministic backward's integer sums are too, and its extra views stay zero"""
    base, padded = _blind_pair()
    ref = run(base, ref64.MEAN, cfirst, g_seed=9)
    ref_det = run(base, ref64.MEAN, cfirst, det=True, g_seed=9)
    r64 = reference(base, ref64.MEAN, ref["g_out"])
    check(base, ref, r64, "V=16")
    check(base, ref_det, r64, "V=16 deterministic", det=True)
    for sc in padded:
        v = sc["feat"].shape[0]
        got = run(sc, ref64.MEAN, cfirst, g_seed=9)
        assert torch.equal(got["count"], ref["count"]), f"V={v}: count"
        assert torch.equal(got["out"], ref["out"]), f"V={v}: volume bits differ from V=16"
        r = reference(sc, ref64.MEAN, got["g_out"])
        check(sc, got, r, f"V={v} padded")
        det = run(sc, ref64.MEAN, cfirst, det=True, g_seed=9)
        assert torch.equal(det["g_feat"][:16], ref_det["g_feat"]), f"V={v}: deterministic dL/dfeat bits"
        assert torch.equal(det["g_prob"][:16], ref_det["g_prob"]), f"V={v}: deterministic dL/dprob bits"
        assert not bool(det["g_feat"][16:].any()) and not bool(det["g_prob"][16:].any())


@pytest.mark.parametrize("fdt", ["f32", "bf16"])
@pytest.mark.parametrize("v", [5, 33])
def test_deterministic_backward_against_fp64(v, fdt):
    """the fixed-point backward: every fp32 contribution rounded to 2^-32, summed exactly, so
    |det - ref64| <= n_terms 2^-33 + the per-term fp32 bound; and within the sum of both bounds of
    the default (RED) backward"""
    sc = BC.random_scene(v, 256, 3, 200, seed=90 + v, bf16=fdt == "bf16")
    for cfirst in (True, False):
        det = run(sc, ref64.MEAN, cfirst, FDT[fdt], det=True, g_seed=v)
        red = run(sc, ref64.MEAN, cfirst, FDT[fdt], g_seed=v)
        ref = reference(sc, ref64.MEAN, det["g_out"])
        check(sc, det, ref, f"det V={v} {fdt}", det=True)
        check(sc, red, ref, f"red V={v} {fdt}")
        for key, kd, kr in (("g_feat", "g_feat_det", "g_feat"), ("g_prob", "g_prob_det", "g_prob")):
            ref64.check_bound(_crop(det[key], sc), _crop(red[key], sc).double(), ref[kd][1] + ref[kr][1],
                              f"det vs red {key}")


@pytest.mark.parametrize("v", [5, 17])
@pytest.mark.parametrize("cfirst", [True, False])
def test_normalise_is_mean(v, cfirst):
    """MEAN == voxel_normalize(SUM, count) bit for bit: both divide by __fadd_rn(count, 1e-8f);
    voxels with count 0 give 0"""
    sc = BC.random_scene(v, 132, 3, 180, seed=200 + v)
    sc["points"][:, :4] = 40.0                      # far outside every view: count 0
    pts, proj = sc["points"].to(DEV), sc["projection"].to(DEV)
    feat = ops.pack_features(sc["feat"].to(DEV))
    depth, dens = sc["depth"].to(DEV), sc["prob"].to(DEV)
    args = (feat, pts, proj, depth, dens, sc["vs_z"], sc["h"], sc["w"])
    mean, cnt = ops.backproject_aggregate(*args, mode="mean", channels_first=cfirst)
    s, cnt2 = ops.backproject_aggregate(*args, mode="sum", channels_first=cfirst)
    assert torch.equal(cnt, cnt2)
    assert bool((cnt == 0).any()) and bool((cnt > 1).any())
    norm = ops.voxel_normalize(s, cnt)
    assert norm.is_contiguous() == cfirst
    assert torch.equal(norm, mean)
    assert not bool(mean[:, cnt == 0].any())


def test_prob_norm_backward_alone():
    """mvsd_prob_norm_bwd against fp64 for T = 1..8 with given fp32 g_pn (no upstream error)"""
    for t in (1, 2, 3, 5, 8):
        gen = torch.Generator().manual_seed(t)
        prob = 0.01 + torch.rand(4, t, 9, 13, generator=gen)
        g_pn = torch.randn(4, t, 9, 13, generator=gen)
        out = torch.zeros_like(prob, device=DEV)
        _lib.prob_norm_bwd(prob.to(DEV), g_pn.to(DEV), out, height=9, width=13)
        val, bound = ref64.prob_norm_reference(prob.double(), g_pn.double(), torch.zeros(4, t, 9, 13).double())
        ref64.check_bound(out.cpu(), val, bound, f"prob_norm_bwd T={t}")
