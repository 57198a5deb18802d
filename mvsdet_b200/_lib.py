"""ctypes binding of libmvsdet_b200.so -- the C ABI declared in
include/mvsdet_b200.h.  There is no fallback: if the library is missing or a
call fails this raises, loudly."""
from __future__ import annotations

import ctypes as C
import math
import os
import threading

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MVSDET_B200_LIB") or os.path.join(HERE, "lib", "libmvsdet_b200.so")

ABI_VERSION = 3
OK, ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_CUDA = 0, 1, 2, 3
F32, BF16 = 0, 1
CHANNELS_LAST, CHANNELS_FIRST = 0, 1
BP_MEAN, BP_SUM, BP_PER_VIEW = 0, 1, 2

_p, _i, _f, _l = C.c_void_p, C.c_int, C.c_float, C.c_int64

# name -> argtypes; every symbol include/mvsdet_b200.h declares
SIGNATURES = {
    "mvsd_abi_version": ([], _i),
    "mvsd_build_info": ([], C.c_char_p),
    "mvsd_status_string": ([_i], C.c_char_p),
    "mvsd_last_error": ([], C.c_char_p),
    "mvsd_set_tuning": ([_i, _i], _i),
    "mvsd_launch_count": ([], _l),
    "mvsd_pack_nchw_to_nhwc": ([_p, _p, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_unpack_nhwc_to_nchw": ([_p, _p, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_scene_setup": ([_p, _p, _i, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p], _i),
    "mvsd_plane_sweep_fwd": ([_p, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_plane_sweep_bwd": ([_p, _i, _i, _p, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_plane_sweep_bwd_det": ([_p, _i, _i, _p, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_fixed_to_float": ([_p, _p, _l, _p], _i),
    "mvsd_backproject_bwd_det": ([_p, _i, _p, _p, _i, _i, _i, _p, _p, _p, _p, _l, _l, _l, _l,
                                  _f, _p, _p, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_plane_sweep_groupcorr_fwd": ([_p, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_plane_sweep_groupcorr_bwd": ([_p, _p, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_homo_warp_fwd": ([_p, _i, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_homo_warp_bwd": ([_p, _i, _i, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_depth_topk_fwd": ([_p, _l, _l, _l, _l, _p, _p, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p,
                             _f, _f, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_depth_topk_bwd": ([_p, _l, _l, _l, _l, _p, _p, _p, _p, _p, _p, _p, _i, _p, _p, _p,
                             _f, _f, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_ray_depth_scale": ([_p, _i, _p, _i, _i, _i, _p], _i),
    "mvsd_rgb_downsample4": ([_p, _p, _i, _p, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_backproject_fwd": ([_p, _i, _i, _i, _p, _p, _p, _p, _l, _l, _l, _l, _f, _i, _p, _i,
                              _p, _p, _p, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_backproject_bwd": ([_p, _i, _i, _p, _p, _i, _i, _i, _p, _p, _p, _p, _l, _l, _l, _l,
                              _f, _p, _p, _i, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_prob_norm_bwd": ([_p, _p, _p, _l, _l, _l, _l, _i, _i, _i, _i, _p], _i),
    "mvsd_voxel_normalize": ([_p, _p, _p, _i, _i, _i, _p], _i),
    "mvsd_voxel_reduce_p2p": ([_p, _p, _p, _i, _i, _i, _i, _i, _p], _i),
    "mvsd_halo_reduce_p2p": ([_p, _p, _p, _i, _i, _i, _l, _p], _i),
}


# --------------------------------------------------------------------------
# Launchers: one per status-returning entry point, the only code that knows its argument order.
# They take tensors with logical shapes in the memory format the kernel reads (ops.py's
# convention), derive dims, strides and dtype codes from them, pass None as NULL and enqueue on
# torch's current stream.  They never allocate, copy or validate: the captured pipelines stay
# allocation-free, and the autograd drop-in pays no host time for checks its callers already did.
# --------------------------------------------------------------------------
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> int:
    """cudaStream_t of torch's current stream on the current device.  torch.cuda.current_stream()
    builds a Stream object through three layers of device-index helpers (16 us per call, ten calls
    per scene: 15 % of the drop-in's host time); the raw getter inductor uses is one C call."""
    if _raw_stream is not None:
        return _raw_stream(torch._C._cuda_getDevice())
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else t.data_ptr()


def _code(dtype) -> int:
    if dtype == torch.float32:
        return F32
    if dtype == torch.bfloat16:
        return BF16
    raise ValueError(f"mvsdet_b200 kernels take float32 or bfloat16, got {dtype}")


def _layout(channels_first: bool) -> int:
    return CHANNELS_FIRST if channels_first else CHANNELS_LAST


def _per_view(intrinsics) -> int:
    return int(intrinsics is not None and intrinsics.dim() == 3)


def pack(src, dst):
    """fp32 NCHW src -> channels-last dst, both [V,C,H,W] (or [V,C,D,H,W]: H' = D*H)"""
    v, c, *hs, w = src.shape
    call("mvsd_pack_nchw_to_nhwc", src.data_ptr(), dst.data_ptr(), _code(dst.dtype), v, c, math.prod(hs), w,
         _stream())


def unpack(src, dst, *, accumulate=False):
    """fp32 channels-last src -> fp32 NCHW dst, shapes as ``pack``"""
    v, c, *hs, w = dst.shape
    call("mvsd_unpack_nhwc_to_nchw", src.data_ptr(), dst.data_ptr(), int(accumulate), v, c, math.prod(hs), w,
         _stream())


def scene_setup(w2c, k_feat, ref_proj, inv_ref, nbr_ids, hom, projection, *, ref_begin):
    k = hom.shape[1]
    call("mvsd_scene_setup", w2c.data_ptr(), k_feat.data_ptr(), _per_view(k_feat), ref_proj.data_ptr(),
         inv_ref.data_ptr(), _ptr(nbr_ids) if k else None, _ptr(hom) if k else None, projection.data_ptr(),
         w2c.shape[0], k, ref_begin, projection.shape[0], _stream())


def plane_sweep_fwd(feat, nbr_ids, hom, depth_values, out, *, ref_begin=0):
    """feat [Vf,C,H,W], nbr_ids [V,k], depth_values [V,D] -> out [V,C,D,H,W]"""
    vf, c, h, w = feat.shape
    v, k = nbr_ids.shape
    call("mvsd_plane_sweep_fwd", feat.data_ptr(), _code(feat.dtype), nbr_ids.data_ptr(), hom.data_ptr(),
         depth_values.data_ptr(), out.data_ptr(), _code(out.dtype), CHANNELS_LAST, v, c, depth_values.shape[1],
         h, w, k, ref_begin, vf, _stream())


def _sweep_bwd(name, g, feat, nbr_ids, hom, depth_values, g_feat, ref_begin):
    vf, c, h, w = feat.shape
    v, k = nbr_ids.shape
    call(name, g.data_ptr(), _code(g.dtype), CHANNELS_LAST, feat.data_ptr(), _code(feat.dtype), nbr_ids.data_ptr(),
         hom.data_ptr(), depth_values.data_ptr(), g_feat.data_ptr(), v, c, depth_values.shape[1], h, w, k,
         ref_begin, vf, _stream())


def plane_sweep_bwd(g, feat, nbr_ids, hom, depth_values, g_feat, *, ref_begin=0):
    """g [V,C,D,H,W] -> RED into the fp32 channels-last g_feat (feat's shape)"""
    _sweep_bwd("mvsd_plane_sweep_bwd", g, feat, nbr_ids, hom, depth_values, g_feat, ref_begin)


def plane_sweep_bwd_det(g, feat, nbr_ids, hom, depth_values, g_feat_q, *, ref_begin=0):
    """``plane_sweep_bwd`` into an int64 fixed-point accumulator"""
    _sweep_bwd("mvsd_plane_sweep_bwd_det", g, feat, nbr_ids, hom, depth_values, g_feat_q, ref_begin)


def plane_sweep_groupcorr_fwd(feat, nbr_ids, hom, depth_values, out, *, ref_begin=0):
    """-> fp32 out [V,k,G,D,H,W], groups innermost in memory"""
    vf, c, h, w = feat.shape
    v, k = nbr_ids.shape
    call("mvsd_plane_sweep_groupcorr_fwd", feat.data_ptr(), _code(feat.dtype), nbr_ids.data_ptr(), hom.data_ptr(),
         depth_values.data_ptr(), out.data_ptr(), v, c, depth_values.shape[1], h, w, k, out.shape[2], ref_begin,
         vf, _stream())


def plane_sweep_groupcorr_bwd(g, feat, nbr_ids, hom, depth_values, g_feat, *, ref_begin=0):
    """fp32 g laid out as the forward's out -> RED into the fp32 g_feat"""
    vf, c, h, w = feat.shape
    v, k = nbr_ids.shape
    call("mvsd_plane_sweep_groupcorr_bwd", g.data_ptr(), feat.data_ptr(), _code(feat.dtype), nbr_ids.data_ptr(),
         hom.data_ptr(), depth_values.data_ptr(), g_feat.data_ptr(), v, c, depth_values.shape[1], h, w, k,
         g.shape[2], ref_begin, vf, _stream())


def homo_warp_fwd(src, hom, depth_values, out):
    """src [B,C,H,W], depth_values [B,D] or [B,D,H,W] -> out [B,C,D,H,W]"""
    b, c, h, w = src.shape
    call("mvsd_homo_warp_fwd", src.data_ptr(), _code(src.dtype), hom.data_ptr(), depth_values.data_ptr(),
         out.data_ptr(), _code(out.dtype), CHANNELS_LAST, b, c, depth_values.shape[1], h, w,
         int(depth_values.dim() == 4), _stream())


def homo_warp_bwd(g, hom, depth_values, g_src):
    b, c, h, w = g_src.shape
    call("mvsd_homo_warp_bwd", g.data_ptr(), _code(g.dtype), CHANNELS_LAST, hom.data_ptr(), depth_values.data_ptr(),
         g_src.data_ptr(), b, c, depth_values.shape[1], h, w, int(depth_values.dim() == 4), _stream())


def depth_topk_fwd(cost_out, prob, off, est_depth, est_dens, est_idx, coding, *, near, interval, raw=False,
                   ray_intr=None, nvs=(None,) * 4):
    """cost_out [V,2,D,H,W] -> [V,D,H,W], [V,T,H,W] and [V,H,W] outputs (prob, off, coding may be
    None); with ``ray_intr`` also ``nvs`` = (opacity, depth_scale, est_ray_depth, ray_depth_coding)"""
    v, _, d, h, w = cost_out.shape
    sv, sc, sd, _, sp = cost_out.stride()
    call("mvsd_depth_topk_fwd", cost_out.data_ptr(), sv, sc, sd, sp, _ptr(prob), _ptr(off), est_depth.data_ptr(),
         est_dens.data_ptr(), est_idx.data_ptr(), _ptr(coding), _ptr(ray_intr), _per_view(ray_intr),
         *map(_ptr, nvs), float(near), float(interval), int(raw), v, d, h, w, est_depth.shape[1], _stream())


def depth_topk_bwd(cost_out, est_idx, g_prob, g_off, g_depth, g_dens, g_coding, g_cost, *, near, interval,
                   raw=False, ray_intr=None, g_ray_depth=None, g_ray_coding=None):
    v, _, d, h, w = cost_out.shape
    sv, sc, sd, _, sp = cost_out.stride()
    call("mvsd_depth_topk_bwd", cost_out.data_ptr(), sv, sc, sd, sp, est_idx.data_ptr(), _ptr(g_prob), _ptr(g_off),
         _ptr(g_depth), _ptr(g_dens), _ptr(g_coding), _ptr(ray_intr), _per_view(ray_intr), _ptr(g_ray_depth),
         _ptr(g_ray_coding), g_cost.data_ptr(), float(near), float(interval), int(raw), v, d, h, w,
         est_idx.shape[1], _stream())


def ray_depth_scale(intrinsics, out):
    v, h, w = out.shape
    call("mvsd_ray_depth_scale", intrinsics.data_ptr(), _per_view(intrinsics), out.data_ptr(), v, h, w, _stream())


def rgb_downsample4(rgb, src_ids, out, *, height, width):
    """rgb [V,3,H,W], src_ids [n] or None -> out [1,n,height*width,3]"""
    v, _, hh, ww = rgb.shape
    call("mvsd_rgb_downsample4", rgb.data_ptr(), _ptr(src_ids), out.shape[1], out.data_ptr(), v, hh, ww, height,
         width, _stream())


def backproject_fwd(feat, points, projection, depth, prob, out, *, vs_z, mode, height, width,
                    channels_first=False, count=None, valid=None):
    """feat [Vf,C,Hf,Wf]; depth, prob [V,T,.,.] views of feat's first V views' hypotheses -> out [C,N]
    ([V,C,N] per view)"""
    _, c, fh, fw = feat.shape
    v, t = depth.shape[:2]
    sv, st, sy, sx = depth.stride()
    call("mvsd_backproject_fwd", feat.data_ptr(), _code(feat.dtype), fh, fw, points.data_ptr(), projection.data_ptr(),
         depth.data_ptr(), prob.data_ptr(), sv, sy, sx, st, float(vs_z), mode, out.data_ptr(),
         _layout(channels_first), _ptr(count), _ptr(valid), None, v, c, height, width, t, out.shape[-1], _stream())


def backproject_bwd(g_out, feat, points, projection, depth, prob, g_feat, g_pn, *, vs_z, mode, height, width,
                    channels_first=False, count=None):
    """g_out shaped as ``backproject_fwd``'s out -> RED into g_feat and g_pn (prob's strides)"""
    _, c, fh, fw = feat.shape
    v, t = depth.shape[:2]
    sv, st, sy, sx = depth.stride()
    call("mvsd_backproject_bwd", g_out.data_ptr(), _layout(channels_first), mode, _ptr(count), feat.data_ptr(),
         _code(feat.dtype), fh, fw, points.data_ptr(), projection.data_ptr(), depth.data_ptr(), prob.data_ptr(),
         sv, sy, sx, st, float(vs_z), g_feat.data_ptr(), g_pn.data_ptr(), v, c, height, width, t,
         g_out.shape[-1], _stream())


def backproject_bwd_det(g_out, count, feat, points, projection, depth, prob, g_feat_q, g_pn_q, *, vs_z, height,
                        width, channels_first=False):
    _, c, fh, fw = feat.shape
    v, t = depth.shape[:2]
    sv, st, sy, sx = depth.stride()
    call("mvsd_backproject_bwd_det", g_out.data_ptr(), _layout(channels_first), count.data_ptr(), feat.data_ptr(),
         _code(feat.dtype), fh, fw, points.data_ptr(), projection.data_ptr(), depth.data_ptr(), prob.data_ptr(),
         sv, sy, sx, st, float(vs_z), g_feat_q.data_ptr(), g_pn_q.data_ptr(), v, c, height, width, t,
         g_out.shape[-1], _stream())


def prob_norm_bwd(prob, g_pn, g_prob, *, height, width):
    v, t = prob.shape[:2]
    sv, st, sy, sx = prob.stride()
    call("mvsd_prob_norm_bwd", prob.data_ptr(), g_pn.data_ptr(), g_prob.data_ptr(), sv, sy, sx, st, v, height,
         width, t, _stream())


def voxel_normalize(volume_sum, count, out, *, channels_first):
    c, n = volume_sum.shape
    call("mvsd_voxel_normalize", volume_sum.data_ptr(), count.data_ptr(), out.data_ptr(), _layout(channels_first),
         c, n, _stream())


def voxel_reduce_p2p(part_ptrs, out_ptrs, count_local, *, world, rank, channels, channels_first):
    call("mvsd_voxel_reduce_p2p", part_ptrs, out_ptrs, count_local.data_ptr(), world, rank, _layout(channels_first),
         channels, count_local.numel(), _stream())


def halo_reduce_p2p(g_ptrs, pull_offsets, pull_sources, *, world, rank, view_elems):
    call("mvsd_halo_reduce_p2p", g_ptrs, pull_offsets.data_ptr(), pull_sources.data_ptr(), world, rank,
         pull_offsets.numel() - 1, view_elems, _stream())


def fixed_to_float(src, dst):
    call("mvsd_fixed_to_float", src.data_ptr(), dst.data_ptr(), src.numel(), _stream())


_lock = threading.Lock()
_lib = None


class MvsdError(RuntimeError):
    pass


def load() -> C.CDLL:
    """dlopen the library and type every entry point (no compute happens)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.isfile(LIB_PATH):
                raise MvsdError(
                    f"{LIB_PATH} is missing. Build it with `python -m mvsdet_b200.build` "
                    "(nvcc, sm_100a). mvsdet_b200 has no CPU or PyTorch fallback.")
            lib = C.CDLL(LIB_PATH)
            for name, (argtypes, restype) in SIGNATURES.items():
                fn = getattr(lib, name)          # AttributeError if a symbol is missing
                fn.argtypes = argtypes
                fn.restype = restype
            if lib.mvsd_abi_version() != ABI_VERSION:
                raise MvsdError("libmvsdet_b200.so ABI version mismatch; rebuild")
            _lib = lib
    return _lib


def call(name: str, *args) -> None:
    """Invoke a status-returning entry point; non-zero status -> exception
    (ValueError for caller mistakes, RuntimeError otherwise)."""
    lib = load()
    status = getattr(lib, name)(*args)
    if status != OK:
        msg = lib.mvsd_last_error().decode() or lib.mvsd_status_string(status).decode()
        if status in (ERR_INVALID_ARG, ERR_UNSUPPORTED):
            raise ValueError(f"{name}: {msg}")
        raise MvsdError(f"{name}: {msg}")


def launch_count() -> int:
    return int(load().mvsd_launch_count())


def set_tuning(key: int, value: int) -> int:
    return int(load().mvsd_set_tuning(key, value))
