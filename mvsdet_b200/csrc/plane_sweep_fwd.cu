// Plane-sweep variance volume, forward (and the stand-alone homography warp).
// See plane_sweep.cuh for the design; mvsdet.py:439-467, module.py:105-146.
#include "plane_sweep.cuh"

namespace mvsd {

template <typename TIn, typename TOut, int KMAX, int G, bool FULL, bool WARP_ONLY>
__global__ void __launch_bounds__(kSweepThreads) sweep_fwd_kernel(const SweepParams p) {
  __shared__ WarpSample s_tab[kSweepWarps][kSlots];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const SweepCoord c = sweep_coord<G>(p, warp, lane);
  if (!c.ok) return;                            // warps are independent: no CTA barrier below
  const int C = p.C, k = p.k, HW = p.H * p.W;
  const TIn* feat = static_cast<const TIn*>(p.feat);
  const unsigned pix = (unsigned)(c.y * p.W + c.x);
  TOut* out_pix = static_cast<TOut*>(p.out) + ((size_t)c.v * p.D * HW + pix) * C + c.c0;
  const size_t plane_stride = (size_t)HW * C;

  float4 ref[G], ref2[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    ref[g] = f4zero();
    if (!WARP_ONLY && group_on<FULL>(c.c0, g, C))
      ref[g] = Io<TIn>::ld(feat + ((size_t)(c.v + p.ref_begin) * HW + pix) * C + c.c0 + 128 * g);
    ref2[g] = f4mul(ref[g], ref[g]);
  }
  const TIn* nsrc[KMAX];
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    int n = c.v + p.ref_begin;
    if (!WARP_ONLY && j < k) n = __ldg(p.nbr + (size_t)c.v * k + j);
    nsrc[j] = feat + (size_t)n * HW * C + c.c0;
  }
  const float inv_n = 1.0f / (float)(k + 1);
  const int dc = k > 0 ? kSlots / k : p.D;      // planes per geometry pass

  for (int d0 = 0; d0 < p.D; d0 += dc) {
    if (k > 0) {
      __syncwarp();
      fill_samples<WARP_ONLY ? kDepthEither : kDepthPlanes>(s_tab[warp], p, c, d0, dc, lane);
      __syncwarp();
    }
    const int dend = min(p.D, d0 + dc);
    for (int d = d0; d < dend; ++d) {
      float4 s1[G], s2[G];
#pragma unroll
      for (int g = 0; g < G; ++g) {
        s1[g] = ref[g];
        s2[g] = ref2[g];
      }
#pragma unroll
      for (int j = 0; j < KMAX; ++j) {
        if (j >= k) break;
        const WarpSample s = s_tab[warp][(d - d0) * k + j];
        if (s.p00 == kNoSample) continue;       // all four taps outside: adds 0
        float4 wv[G];
        gather_taps<TIn, G, FULL>(nsrc[j], s, c.c0, C, wv);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          s1[g] = f4add(s1[g], wv[g]);
          s2[g] = f4fma(wv[g], wv[g], s2[g]);
        }
      }
      TOut* o = out_pix + (size_t)d * plane_stride;
#pragma unroll
      for (int g = 0; g < G; ++g) {
        if (!group_on<FULL>(c.c0, g, C)) continue;
        float4 r;
        if (WARP_ONLY) {
          r = s1[g];
        } else {
          // var = S2/n - (S1/n)^2 (mvsdet.py:467); "/n" as "*(1/n)", which is what
          // ATen's CUDA division by a scalar does.  S2/n and (S1/n)^2 are rounded
          // separately as in the reference (no FMA contraction), which keeps the
          // variance of a single view (k = 0) exactly 0.
          const float4 m = f4scale(s1[g], inv_n);
          r.x = __fsub_rn(s2[g].x * inv_n, __fmul_rn(m.x, m.x));
          r.y = __fsub_rn(s2[g].y * inv_n, __fmul_rn(m.y, m.y));
          r.z = __fsub_rn(s2[g].z * inv_n, __fmul_rn(m.z, m.z));
          r.w = __fsub_rn(s2[g].w * inv_n, __fmul_rn(m.w, m.w));
        }
        Io<TOut>::st_stream(o + 128 * g, r);
      }
    }
  }
}

// Packed-arithmetic forward (default): identical decomposition, the per-lane 4-channel
// vectors are f32x2 pairs so the bilinear blend and the S1 / S2 accumulation
// issue as FMUL2 / FFMA2 / FADD2 -- the scalar kernel above is issue-bound
// (profiles/r01_a_ncu_sweep_summary.txt: 81% issue-active, 314 instructions per
// pixel-plane of which 160 are fp32 math).
// CTA of the packed forward: a 2 x 2 pixel patch, 4 warps.  Measured on B200 (profiles/r02_bwd_experiments.md):
// 4 x 2 (8 warps, the shape of the other pixel-per-warp kernels) 0.2606 ms, 2 x 2 and 4 x 1 0.2534, 2 x 1
// 0.2626, 1 x 1 0.2759, 4 x 4 / 8 x 2 0.367 -- with 64 registers an SM holds 32 warps either way, smaller CTAs
// drain and refill in finer steps, and below 4 warps the shared taps of neighbouring pixels stop meeting in L1.
constexpr int kFwdPatchW = 2, kFwdPatchH = 2;
constexpr int kFwdWarps = kFwdPatchW * kFwdPatchH, kFwdThreads = kFwdWarps * 32;

// PX: per-pixel depth hypotheses [V,D,H,W] (mvsd_plane_sweep_fwd_px); PX = false is the per-view kernel.
template <typename TIn, typename TOut, int KMAX, int G, bool FULL, bool PX>
// 8 CTAs x 4 warps per SM = 64 registers (9 CTAs at 56 registers measured the same, 10 at 48 spill: 0.313 ms)
__global__ void __launch_bounds__(kFwdThreads, 8) sweep_fwd_p_kernel(const SweepParams p) {
  __shared__ WarpSample s_tab[kFwdWarps][kSlots];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  SweepCoord c;
  {
    int t = blockIdx.x;
    const int tx = t % p.tiles_x; t /= p.tiles_x;
    const int ty = t % p.tiles_y; t /= p.tiles_y;
    const int slice = t % p.slices;
    c.v = t / p.slices;
    c.x = tx * kFwdPatchW + (warp % kFwdPatchW);
    c.y = ty * kFwdPatchH + (warp / kFwdPatchW);
    c.ok = c.x < p.W && c.y < p.H;
    c.c0 = slice * 128 * G + 4 * lane;
  }
  if (!c.ok) return;
  const int C = p.C, k = p.k, HW = p.H * p.W;
  const TIn* feat = static_cast<const TIn*>(p.feat);
  const unsigned pix = (unsigned)(c.y * p.W + c.x);
  TOut* out_pix = static_cast<TOut*>(p.out) + ((size_t)c.v * p.D * HW + pix) * C + c.c0;
  const size_t plane_stride = (size_t)HW * C;

  P4 ref[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    ref[g] = p4zero();
    if (group_on<FULL>(c.c0, g, C))
      ref[g] = p4from(Raw<TIn>::ld(feat + ((size_t)(c.v + p.ref_begin) * HW + pix) * C + c.c0 + 128 * g));
  }
  TOut* o = out_pix;
  const TIn* nsrc[KMAX];
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    int n = c.v + p.ref_begin;
    if (j < k) n = __ldg(p.nbr + (size_t)c.v * k + j);
    nsrc[j] = feat + (size_t)n * HW * C + c.c0;
    asm volatile("" : "+l"(nsrc[j]));           // keep the base in registers (ptxas re-derives it per plane otherwise)
  }
  const float inv_n = 1.0f / (float)(k + 1);
  const u64 inv_n2 = pk2(inv_n, inv_n);
  const int dc = k > 0 ? kSlots / k : p.D;

  for (int d0 = 0; d0 < p.D; d0 += dc) {
    if (k > 0) {
      __syncwarp();
      fill_samples<PX ? kDepthPixels : kDepthPlanes>(s_tab[warp], p, c, d0, dc, lane);
      __syncwarp();
    }
    const int dend = min(p.D, d0 + dc);
    for (int d = d0; d < dend; ++d) {
      const WarpSample* tab = s_tab[warp] + (d - d0) * k;
      // The variance + store tail is instantiated once per control path (which
      // neighbours have a sample), so no path pays register moves at a merge.
      auto emit = [&](const P4 (&s1)[G], const P4 (&s2)[G]) {
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (!group_on<FULL>(c.c0, g, C)) continue;
          // var = S2/n - (S1/n)^2, every step rounded on its own (see the scalar kernel): mul.rn.f32x2 /
          // sub.rn.f32x2 round each element exactly like the scalar _rn intrinsics, no contraction
          const P4 m = p4scale(s1[g], inv_n2);
          const P4 q = p4scale(s2[g], inv_n2);
          Io<TOut>::st_stream(o + 128 * g, p4to(p4sub(q, p4mul(m, m))));
        }
      };
      if (KMAX <= 2) {
        const bool v0 = k > 0 && tab[0].p00 != kNoSample;
        const bool v1 = KMAX == 2 && k > 1 && tab[1].p00 != kNoSample;
        if (v0 && v1) {
          // both neighbours' 8*G loads in flight before the first blend
          RawTaps<TIn, G> r0, r1;
          load_taps<TIn, G, FULL>(nsrc[0], tab[0], c.c0, C, r0);
          load_taps<TIn, G, FULL>(nsrc[KMAX - 1], tab[KMAX - 1], c.c0, C, r1);
          P4 s1[G], s2[G], wa[G], wb[G];
          blend_taps<TIn, G>(r0, tab[0], wa);
          blend_taps<TIn, G>(r1, tab[KMAX - 1], wb);
#pragma unroll
          for (int g = 0; g < G; ++g) {
            s1[g] = p4add(p4add(ref[g], wa[g]), wb[g]);
            s2[g] = p4fma(wb[g], wb[g], p4fma(wa[g], wa[g], p4mul(ref[g], ref[g])));
          }
          emit(s1, s2);
        } else if (v0) {
          P4 s1[G], s2[G], wv[G];
          gather_taps_p<TIn, G, FULL>(nsrc[0], tab[0], c.c0, C, wv);
#pragma unroll
          for (int g = 0; g < G; ++g) {
            s1[g] = p4add(ref[g], wv[g]);
            s2[g] = p4fma(wv[g], wv[g], p4mul(ref[g], ref[g]));
          }
          emit(s1, s2);
        } else if (v1) {
          P4 s1[G], s2[G], wv[G];
          gather_taps_p<TIn, G, FULL>(nsrc[KMAX - 1], tab[KMAX - 1], c.c0, C, wv);
#pragma unroll
          for (int g = 0; g < G; ++g) {
            s1[g] = p4add(ref[g], wv[g]);
            s2[g] = p4fma(wv[g], wv[g], p4mul(ref[g], ref[g]));
          }
          emit(s1, s2);
        } else {
          P4 s2[G];
#pragma unroll
          for (int g = 0; g < G; ++g) s2[g] = p4mul(ref[g], ref[g]);
          emit(ref, s2);
        }
      } else {
        P4 s1[G], s2[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
          s1[g] = ref[g];
          s2[g] = p4mul(ref[g], ref[g]);
        }
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
          if (j >= k) break;
          if (tab[j].p00 == kNoSample) continue;   // all four taps outside: adds 0
          P4 wv[G];
          gather_taps_p<TIn, G, FULL>(nsrc[j], tab[j], c.c0, C, wv);
#pragma unroll
          for (int g = 0; g < G; ++g) {
            s1[g] = p4add(s1[g], wv[g]);
            s2[g] = p4fma(wv[g], wv[g], s2[g]);
          }
        }
        emit(s1, s2);
      }
      o += plane_stride;
      asm volatile("" : "+l"(o));
    }
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
int sweep_check(const char* who, int V, int C, int D, int H, int W, int k, int layout) {
  if (V <= 0 || C <= 0 || D <= 0 || H <= 0 || W <= 0 || k < 0)
    return fail(MVSD_ERR_INVALID_ARG, "%s: non-positive dimension", who);
  if (C % 4 != 0 || C > MVSD_MAX_C)
    return fail(MVSD_ERR_UNSUPPORTED, "%s: C=%d must be a multiple of 4 and <= %d", who, C, MVSD_MAX_C);
  if (k > MVSD_MAX_K) return fail(MVSD_ERR_UNSUPPORTED, "%s: k=%d > %d", who, k, MVSD_MAX_K);
  if ((long long)H * W * C >= (1LL << 31))
    return fail(MVSD_ERR_UNSUPPORTED, "%s: one feature map must stay below 2^31 elements", who);
  if (layout != MVSD_CHANNELS_LAST)
    return fail(MVSD_ERR_UNSUPPORTED, "%s: only MVSD_CHANNELS_LAST volumes are implemented", who);
  return MVSD_OK;
}

// Channel groups (of 128) per warp: 2 keeps all 256 FPN channels of a tap in one
// warp (fewest instructions per byte).
int sweep_groups(int C) { return C > 128 ? 2 : 1; }

bool sweep_grid(SweepParams& p, int G, dim3& grid) {
  p.tiles_x = (p.W + kPatchW - 1) / kPatchW;
  p.tiles_y = (p.H + kPatchH - 1) / kPatchH;
  p.slices = (p.C + 128 * G - 1) / (128 * G);
  const long long blocks = (long long)p.V * p.slices * p.tiles_y * p.tiles_x;
  if (blocks > 2147483647LL) return false;
  grid = dim3((unsigned)blocks);
  return true;
}

template <typename TIn, typename TOut, bool WARP_ONLY>
static int launch_fwd_k(SweepParams& p, cudaStream_t st) {
  dim3 grid;
  const int G = sweep_groups(p.C);
  if (!sweep_grid(p, G, grid)) return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_fwd: grid too large");
  if constexpr (!WARP_ONLY) {                 // the packed kernel has its own CTA patch
    p.tiles_x = (p.W + kFwdPatchW - 1) / kFwdPatchW;
    p.tiles_y = (p.H + kFwdPatchH - 1) / kFwdPatchH;
    const long long blocks = (long long)p.V * p.slices * p.tiles_y * p.tiles_x;
    if (blocks > 2147483647LL) return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_fwd: grid too large");
    grid = dim3((unsigned)blocks);
  }
  const bool full = p.C % (128 * G) == 0;
  const int kmax = WARP_ONLY ? 1 : (p.k <= 1 ? 1 : (p.k == 2 ? 2 : 4));
#define MVSD_FWD(KM, GG, FU)                                                           \
  do {                                                                                 \
    if constexpr (WARP_ONLY)                                                           \
      sweep_fwd_kernel<TIn, TOut, KM, GG, FU, true><<<grid, kSweepThreads, 0, st>>>(p); \
    else if (p.depth_per_pixel)                                                        \
      sweep_fwd_p_kernel<TIn, TOut, KM, GG, FU, true><<<grid, kFwdThreads, 0, st>>>(p); \
    else                                                                               \
      sweep_fwd_p_kernel<TIn, TOut, KM, GG, FU, false><<<grid, kFwdThreads, 0, st>>>(p); \
  } while (0)
#define MVSD_FWD_G(KM)                                                            \
  do {                                                                            \
    if (G == 2) { if (full) MVSD_FWD(KM, 2, true); else MVSD_FWD(KM, 2, false); } \
    else { if (full) MVSD_FWD(KM, 1, true); else MVSD_FWD(KM, 1, false); }        \
  } while (0)
  if constexpr (WARP_ONLY) {
    MVSD_FWD_G(1);                        // stand-alone warp: the scalar kernel, one source
  } else {
    // k = 2 is the reference's configuration (mvsdet.py:432) and gets the un-predicated
    // instantiation; k = 0, 1 (one- and two-view scenes) and k = 3, 4 share the predicated ones
    if (kmax == 2) MVSD_FWD_G(2);
    else if (kmax == 1) { if (G == 2) MVSD_FWD(1, 2, false); else MVSD_FWD(1, 1, false); }
    else { if (G == 2) MVSD_FWD(4, 2, false); else MVSD_FWD(4, 1, false); }
  }
#undef MVSD_FWD_G
#undef MVSD_FWD
  count_launch();
  return check_launch("plane_sweep_fwd");
}

template <bool WARP_ONLY>
static int launch_fwd(SweepParams& p, int in_dtype, int out_dtype, cudaStream_t st) {
  if (in_dtype == MVSD_F32 && out_dtype == MVSD_F32) return launch_fwd_k<float, float, WARP_ONLY>(p, st);
  if (in_dtype == MVSD_BF16 && out_dtype == MVSD_F32)
    return launch_fwd_k<__nv_bfloat16, float, WARP_ONLY>(p, st);
  if (in_dtype == MVSD_BF16 && out_dtype == MVSD_BF16)
    return launch_fwd_k<__nv_bfloat16, __nv_bfloat16, WARP_ONLY>(p, st);
  if (in_dtype == MVSD_F32 && out_dtype == MVSD_BF16)
    return launch_fwd_k<float, __nv_bfloat16, WARP_ONLY>(p, st);
  return fail(MVSD_ERR_INVALID_ARG, "plane_sweep_fwd: bad dtype");
}

}  // namespace mvsd

using namespace mvsd;

// per_pixel: depth_values is [V,D,H,W] (homo_warping's per-pixel branch, module.py:130-133)
static int plane_sweep_fwd(const char* who, const void* feat, int feat_dtype, const int32_t* nbr_ids,
                           const float* hom, const float* depth_values, void* out, int out_dtype,
                           int out_layout, int V, int C, int D, int H, int W, int k, int ref_begin,
                           int n_feat_views, bool per_pixel, void* stream) {
  if (int e = sweep_check(who, V, C, D, H, W, k, out_layout)) return e;
  if (!feat || !out || !depth_values || (k > 0 && (!nbr_ids || !hom)))
    return fail(MVSD_ERR_INVALID_ARG, "%s: null pointer", who);
  if (ref_begin < 0 || (long long)ref_begin + V > n_feat_views)
    return fail(MVSD_ERR_INVALID_ARG, "%s: reference views [%d, %d) exceed the %d feature views",
                who, ref_begin, ref_begin + V, n_feat_views);
  SweepParams p{};
  p.feat = feat; p.nbr = nbr_ids; p.hom = hom; p.depth = depth_values; p.out = out;
  p.V = V; p.C = C; p.D = D; p.H = H; p.W = W; p.k = k; p.ref_begin = ref_begin; p.n_feat = n_feat_views;
  p.depth_per_pixel = per_pixel ? 1 : 0;
  return launch_fwd<false>(p, feat_dtype, out_dtype, static_cast<cudaStream_t>(stream));
}

extern "C" int mvsd_plane_sweep_fwd(const void* feat, int feat_dtype, const int32_t* nbr_ids,
                                    const float* hom, const float* depth_values, void* out,
                                    int out_dtype, int out_layout, int V, int C, int D, int H,
                                    int W, int k, int ref_begin, int n_feat_views, void* stream) {
  return plane_sweep_fwd("plane_sweep_fwd", feat, feat_dtype, nbr_ids, hom, depth_values, out, out_dtype,
                         out_layout, V, C, D, H, W, k, ref_begin, n_feat_views, false, stream);
}

extern "C" int mvsd_plane_sweep_fwd_px(const void* feat, int feat_dtype, const int32_t* nbr_ids,
                                       const float* hom, const float* depth_values, void* out,
                                       int out_dtype, int out_layout, int V, int C, int D, int H,
                                       int W, int k, int ref_begin, int n_feat_views, void* stream) {
  return plane_sweep_fwd("plane_sweep_fwd_px", feat, feat_dtype, nbr_ids, hom, depth_values, out, out_dtype,
                         out_layout, V, C, D, H, W, k, ref_begin, n_feat_views, true, stream);
}

extern "C" int mvsd_homo_warp_fwd(const void* src, int src_dtype, const float* hom,
                                  const float* depth_values, void* out, int out_dtype,
                                  int out_layout, int B, int C, int D, int H, int W,
                                  int depth_per_pixel, void* stream) {
  if (int e = sweep_check("homo_warp_fwd", B, C, D, H, W, 1, out_layout)) return e;
  if (!src || !hom || !depth_values || !out)
    return fail(MVSD_ERR_INVALID_ARG, "homo_warp_fwd: null pointer");
  SweepParams p{};
  p.feat = src; p.nbr = nullptr; p.hom = hom; p.depth = depth_values; p.out = out;
  p.V = B; p.C = C; p.D = D; p.H = H; p.W = W; p.k = 1; p.ref_begin = 0; p.n_feat = B;
  p.depth_per_pixel = depth_per_pixel ? 1 : 0;
  return launch_fwd<true>(p, src_dtype, out_dtype, static_cast<cudaStream_t>(stream));
}
