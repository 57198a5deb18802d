"""CPU-side checks of the drop-in boundary (no compute calls, no GPU needed):
the C-ABI library loads, exports every symbol include/mvsdet_b200.h declares
and nothing is declared in the ctypes layer that the header does not have;
the host-side mirrors validate their arguments and refuse CPU tensors."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mvsdet_b200.h")


def _header_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)            # strip comments
    # every prototype of the form  <type> mvsd_xxx(
    return sorted(set(re.findall(r"\b(mvsd_[a-z0-9_]+)\s*\(", text)))


def _build_if_needed():
    from mvsdet_b200 import _lib, build
    if not os.path.isfile(_lib.LIB_PATH):
        build.build()
    return _lib


def test_header_declares_entry_points():
    names = _header_functions()
    for must in ("mvsd_plane_sweep_fwd", "mvsd_plane_sweep_bwd", "mvsd_depth_topk_fwd",
                 "mvsd_depth_topk_bwd", "mvsd_backproject_fwd", "mvsd_backproject_bwd",
                 "mvsd_homo_warp_fwd", "mvsd_homo_warp_bwd", "mvsd_voxel_normalize"):
        assert must in names


def test_library_exports_every_declared_symbol():
    _lib = _build_if_needed()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in _header_functions():
        assert hasattr(lib, name), f"{name} is declared in the header but not exported"


def test_ctypes_table_matches_header():
    _lib = _build_if_needed()
    assert sorted(_lib.SIGNATURES) == _header_functions()


def test_prototype_arity_matches_ctypes_table():
    """Count the parameters of every prototype in the header and compare with
    the ctypes argtypes: a drifted signature would corrupt the stack silently."""
    _lib = _build_if_needed()
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name, (argtypes, _) in _lib.SIGNATURES.items():
        m = re.search(r"\b%s\s*\(([^)]*)\)" % name, text)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ("", "void") else len(params.split(","))
        assert n == len(argtypes), f"{name}: header has {n} parameters, ctypes {len(argtypes)}"


def test_load_info_and_status_strings():
    _lib = _build_if_needed()
    lib = _lib.load()
    assert lib.mvsd_abi_version() == _lib.ABI_VERSION == 3
    assert b"sm_100a" in lib.mvsd_build_info()
    assert lib.mvsd_status_string(0) == b"ok"
    assert lib.mvsd_status_string(1) == b"invalid argument"
    assert lib.mvsd_launch_count() >= 0


def test_invalid_arguments_fail_before_any_launch():
    """Argument validation happens on the host side of the ABI: a null pointer
    or a non-positive dimension is rejected with MVSD_ERR_INVALID_ARG and a
    message, without touching the (absent) device."""
    _lib = _build_if_needed()
    lib = _lib.load()
    before = lib.mvsd_launch_count()
    one = ctypes.c_void_p(16)                            # non-null dummy: rejected before any dereference
    st = lib.mvsd_depth_topk_fwd(None, 0, 0, 0, 0, None, None, None, None, None, None,
                                 None, 0, None, None, None, None, 0.2, 0.4, 0, 1, 100, 4, 4, 3, None)
    assert st == _lib.ERR_UNSUPPORTED                    # D > 64
    st = lib.mvsd_scene_setup(one, one, 0, one, one, one, one, one, 4, 4, 0, 4, None)
    assert st == _lib.ERR_UNSUPPORTED                    # k must be <= V-1
    st = lib.mvsd_scene_setup(one, one, 0, one, one, one, one, one, 4, 2, 3, 2, None)
    assert st == _lib.ERR_INVALID_ARG                    # reference views [3,5) of 4
    st = lib.mvsd_backproject_fwd(None, 0, 4, 4, None, None, None, None, 0, 0, 0, 0, 0.2, 7, None,
                                  0, None, None, None, 1, 8, 4, 4, 3, 10, None)
    assert st == _lib.ERR_INVALID_ARG                    # bad mode
    with pytest.raises(ValueError):
        _lib.call("mvsd_voxel_normalize", None, None, None, 0, 4, 4, None)
    assert lib.mvsd_launch_count() == before


# ---- the plane-sweep entry points: every rejection rule, with its exact status and message ----------
# Argument names in header order.  Pointer arguments get a non-null dummy address unless a rule nulls
# them; every case must be rejected on the host, so no kernel is ever launched at the dummy.
_FWD = ("feat", "feat_dtype", "nbr", "hom", "depth", "out", "out_dtype", "layout",
        "V", "C", "D", "H", "W", "k", "ref_begin", "n_feat", "stream")
_BWD = ("g_out", "g_dtype", "layout", "feat", "feat_dtype", "nbr", "hom", "depth", "g_feat",
        "V", "C", "D", "H", "W", "k", "ref_begin", "n_feat", "stream")
_WARP_FWD = ("feat", "feat_dtype", "hom", "depth", "out", "out_dtype", "layout", "V", "C", "D", "H", "W",
             "per_pixel", "stream")
_WARP_BWD = ("g_out", "g_dtype", "layout", "hom", "depth", "g_feat", "V", "C", "D", "H", "W", "per_pixel",
             "stream")
_CORR_FWD = ("feat", "feat_dtype", "nbr", "hom", "depth", "out", "V", "C", "D", "H", "W", "k", "groups",
             "ref_begin", "n_feat", "stream")
_CORR_BWD = ("g_out", "feat", "feat_dtype", "nbr", "hom", "depth", "g_feat", "V", "C", "D", "H", "W", "k",
             "groups", "ref_begin", "n_feat", "stream")
_POINTERS = ("feat", "nbr", "hom", "depth", "out", "g_out", "g_feat")

# entry point -> (argument names, family); a family shares its rules and messages
_SWEEP_ENTRIES = {
    "mvsd_plane_sweep_fwd": (_FWD, "fwd"), "mvsd_plane_sweep_fwd_px": (_FWD, "fwd"),
    "mvsd_homo_warp_fwd": (_WARP_FWD, "warp_fwd"),
    "mvsd_plane_sweep_bwd": (_BWD, "bwd"), "mvsd_plane_sweep_bwd_px": (_BWD, "bwd"),
    "mvsd_plane_sweep_bwd_det": (_BWD, "det"), "mvsd_plane_sweep_bwd_det_px": (_BWD, "det"),
    "mvsd_homo_warp_bwd": (_WARP_BWD, "warp_bwd"),
    "mvsd_plane_sweep_groupcorr_fwd": (_CORR_FWD, "corr"), "mvsd_plane_sweep_groupcorr_fwd_px": (_CORR_FWD, "corr"),
    "mvsd_plane_sweep_groupcorr_bwd": (_CORR_BWD, "corr_bwd"),
    "mvsd_plane_sweep_groupcorr_bwd_px": (_CORR_BWD, "corr_bwd"),
}
# a call every entry point accepts (k = 2: the variance backward takes its run kernel)
_VALID = dict(feat_dtype=0, out_dtype=0, g_dtype=0, layout=0, V=2, C=8, D=4, H=4, W=4, k=2, groups=2,
              ref_begin=0, n_feat=2, per_pixel=0, stream=None, **{p: True for p in _POINTERS})

_ARG, _UNS = 1, 2                                        # MVSD_ERR_INVALID_ARG, MVSD_ERR_UNSUPPORTED
_ALL = ("fwd", "warp_fwd", "bwd", "det", "warp_bwd", "corr", "corr_bwd")
_FUSED = ("fwd", "bwd", "det", "corr", "corr_bwd")      # the entry points with k and reference views
_CORR = ("corr", "corr_bwd")
_NULL_ALL = {p: None for p in _POINTERS}
_GRID = dict(V=2 ** 30, n_feat=2 ** 30, H=8, W=8)        # 2^31 CTAs or more for every sweep kernel
_BAD_GROUPS = "{who}: %d channels per group (must be 4, 8, 16, 32, 64 or 128)"


def _each(families, status, message):
    return {f: (status, message) for f in families}


# (rule, argument overrides, family -> (status, message)): a rule applies to the families it lists and
# overrides only the arguments an entry point has; {who} is the entry point without "mvsd_"
_SWEEP_RULES = [
    *[(f"{d}=0", {d: 0}, _each(_ALL, _ARG, "{who}: non-positive dimension")) for d in "VCDHW"],
    ("k<0", {"k": -1}, _each(_FUSED, _ARG, "{who}: non-positive dimension")),
    ("C%4", {"C": 6}, _each(_ALL, _UNS, "{who}: C=6 must be a multiple of 4 and <= 512")),
    ("C>512", {"C": 516}, _each(_ALL, _UNS, "{who}: C=516 must be a multiple of 4 and <= 512")),
    ("k>4", {"k": 5}, _each(_FUSED, _UNS, "{who}: k=5 > 4")),
    ("HWC>=2^31", {"H": 2048, "W": 2048, "C": 512},
     _each(_ALL, _UNS, "{who}: one feature map must stay below 2^31 elements")),
    ("layout", {"layout": 1}, _each(("fwd", "warp_fwd", "bwd", "det", "warp_bwd"), _UNS,
                                    "{who}: only MVSD_CHANNELS_LAST volumes are implemented")),
    *[(f"null-{p}", {p: None}, _each({f for params, f in _SWEEP_ENTRIES.values() if p in params}, _ARG,
                                     "{who}: null pointer")) for p in _POINTERS],
    ("ref<0", {"ref_begin": -1}, _each(_FUSED, _ARG, "{who}: reference views [-1, 1) exceed the 2 feature views")),
    ("ref>n_feat", {"ref_begin": 1}, _each(_FUSED, _ARG, "{who}: reference views [1, 3) exceed the 2 feature views")),
    # the order of the checks
    ("dims-before-null", {"V": 0, **_NULL_ALL}, _each(_ALL, _ARG, "{who}: non-positive dimension")),
    ("null-before-ref", {"ref_begin": 1, "depth": None}, _each(_FUSED, _ARG, "{who}: null pointer")),
    ("ref-before-groups", {"ref_begin": 1, "groups": 5},
     _each(_CORR, _ARG, "{who}: reference views [1, 3) exceed the 2 feature views")),
    # dtypes
    ("dtype-feat", {"feat_dtype": 2}, {
        "fwd": (_ARG, "plane_sweep_fwd: bad dtype"), "warp_fwd": (_ARG, "plane_sweep_fwd: bad dtype"),
        "bwd": (_UNS, "plane_sweep_bwd: dtype combination not built"),
        "det": (_UNS, "{who}: dtype combination not built"), **_each(_CORR, _ARG, "{who}: bad dtype")}),
    ("dtype-out", {"out_dtype": 2}, _each(("fwd", "warp_fwd"), _ARG, "plane_sweep_fwd: bad dtype")),
    ("dtype-grad", {"g_dtype": 2}, {
        "bwd": (_UNS, "plane_sweep_bwd: dtype combination not built"),
        "det": (_UNS, "{who}: dtype combination not built"), "warp_bwd": (_ARG, "homo_warp_bwd: bad dtype")}),
    ("dtype-fp32-feat-bf16-grad", {"g_dtype": 1}, {
        "bwd": (_UNS, "plane_sweep_bwd: dtype combination not built"),
        "det": (_UNS, "{who}: dtype combination not built")}),
    ("dtype-fp32-feat-bf16-grad-pixel-kernel", {"g_dtype": 1, "k": 3},
     _each(("bwd",), _UNS, "{who}: dtype combination not built")),
    # group correlation
    ("k=0", {"k": 0}, _each(_CORR, _ARG, "{who}: needs at least one neighbour")),
    ("k=0-null-nbr", {"k": 0, "nbr": None}, _each(_CORR, _ARG, "{who}: null pointer")),
    ("C%groups", {"C": 24, "groups": 5}, _each(_CORR, _ARG, "{who}: C=24 is not divisible by num_groups=5")),
    ("groups=0", {"groups": 0}, _each(_CORR, _ARG, "{who}: C=8 is not divisible by num_groups=0")),
    ("group-width-12", {"C": 24, "groups": 2}, _each(_CORR, _UNS, _BAD_GROUPS % 12)),
    ("group-width-2", {"C": 8, "groups": 4}, _each(_CORR, _UNS, _BAD_GROUPS % 2)),
    ("group-width-256", {"C": 512, "groups": 2}, _each(_CORR, _UNS, _BAD_GROUPS % 256)),
    # launch grids of 2^31 CTAs or more, per kernel
    ("grid", _GRID, {
        "fwd": (_UNS, "plane_sweep_fwd: grid too large"), "warp_fwd": (_UNS, "plane_sweep_fwd: grid too large"),
        "bwd": (_UNS, "plane_sweep_bwd: grid too large"), "det": (_UNS, "plane_sweep_bwd_det: grid too large"),
        "warp_bwd": (_UNS, "plane_sweep_bwd: grid too large"),
        **_each(_CORR, _UNS, "plane_sweep_groupcorr: grid too large")}),
    ("grid-bf16", {**_GRID, "feat_dtype": 1}, {
        "bwd": (_UNS, "plane_sweep_bwd: grid too large"),
        "corr_bwd": (_UNS, "plane_sweep_groupcorr_bwd: grid too large")}),
    ("grid-pixel-kernel", {**_GRID, "k": 3}, _each(("bwd",), _UNS, "plane_sweep_bwd: grid too large")),
]


def _sweep_cases():
    for entry, (params, family) in _SWEEP_ENTRIES.items():
        for rule, overrides, expect in _SWEEP_RULES:
            if family in expect:
                status, message = expect[family]
                yield pytest.param(entry, overrides, status, message.format(who=entry[len("mvsd_"):]),
                                   id=f"{entry[len('mvsd_'):]}-{rule}")


@pytest.mark.parametrize("entry,overrides,status,message", list(_sweep_cases()))
def test_sweep_entry_points_reject_before_any_launch(entry, overrides, status, message):
    """Each argument rule of the plane-sweep entry points fails on the host with its exact status and
    message, before any kernel is launched (the launch counter stays put)."""
    lib = _build_if_needed().load()
    params, _ = _SWEEP_ENTRIES[entry]
    args = {**_VALID, **overrides}
    dummy = ctypes.c_void_p(16)
    before = lib.mvsd_launch_count()
    st = getattr(lib, entry)(*[(dummy if args[p] else None) if p in _POINTERS else args[p] for p in params])
    assert lib.mvsd_launch_count() == before
    assert (st, lib.mvsd_last_error().decode()) == (status, message)


def test_ops_refuse_cpu_tensors():
    from mvsdet_b200 import functional as F_, ops
    x = torch.randn(2, 8, 4, 4)
    with pytest.raises(ValueError, match="no CPU path"):
        ops.pack_features(x)
    with pytest.raises(ValueError):
        ops.depth_topk(torch.randn(2, 2, 4, 4, 4), 0.2, 0.4, 3)
    with pytest.raises(ValueError):
        F_.backproject_Weigh(x, torch.zeros(3, 2, 2, 2), torch.zeros(2, 3, 4),
                             torch.zeros(2, 16, 1, 3), [0.1, 0.1, 0.1], torch.zeros(2, 16, 1, 3),
                             gt_depth=torch.zeros(1))


def test_product_package_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under mvsdet_b200/ may import it."""
    pkg = os.path.join(ROOT, "mvsdet_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
