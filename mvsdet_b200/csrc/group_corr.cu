// Group-wise correlation cost volume over the same homography sweep (SURVEY.md 8f rank 4; the
// variant BASELINE.json's north_star alludes to with "group-wise correlation / variance reduction
// ... warp-shuffle reductions").  In the reference it exists only in code no shipped config
// reaches, projects/NeRF-Det/nerfdet/mvs_models/lss_fpn.py:485-506: per neighbour ("sweep") j
//     cost_j[v, g, d, y, x] = mean_{c in group g} ref[v, c, y, x] * warped_j[v, c, d, y, x]
// with the channels split into num_groups contiguous groups; the warp is MVSDet's homo_warping
// (mvs_models/module.py:105-146), i.e. the sample geometry of plane_sweep.cuh.  It is offered
// as an optional operator next to the variance volume for a lighter cost-regularisation net:
// the output is C / num_groups times smaller than the variance volume (74 MB instead of 1.18 GB
// at the headline configuration), so the kernel is gather-bound, not write-bound.
//
// Decomposition: pixel-per-warp like the forward sweep (lane l <-> channels 128 g' + 4 l .. + 3);
// the per-lane products are summed over the lanes of a channel group with shfl.xor (a group is
// cg / 4 consecutive lanes), the first lane of every group writes one float.  Output memory is
// [V, k, D, H, W, num_groups] (groups innermost: the eight values of a pixel-plane are one 32-byte
// sector); the Python layer hands it out as the logical [V, k, num_groups, D, H, W].
// Backward: d ref += sum_j sum_d g_j / cg * warped_j ; d warped_j = g_j / cg * ref -> bilinear
// scatter with fp32 vector REDs: for bf16 features and k = 2 through the run-merging hand-off kernel of
// the variance backward (plane_sweep_bwd_run.cu, MODE 1: same gather, column merging and row hand-off,
// the correlation algebra in the pixel body), otherwise the un-merged pixel-per-warp kernel below.  The
// deterministic form (*_bwd_det) is always that pixel kernel, with 64-bit fixed-point integer REDs.
#include "plane_sweep.cuh"

namespace mvsd {

struct CorrParams {
  SweepParams s;       // s.out: cost volume (fwd); s.g_out: its gradient (bwd); s.g_feat: dL/dfeat
  int groups;          // num_groups
  int cg;              // channels per group
  int lpg;             // lanes per group = cg / 4
  float inv_cg;
};

__device__ __forceinline__ float lane_sum4(P4 v) {
  float a, b, c, d;
  upk2(v.lo, a, b);
  upk2(v.hi, c, d);
  return (a + b) + (c + d);
}

// KMAX = 2: exactly two neighbours (the reference's k, mvsdet.py:432), both neighbours' taps in flight
// before the first blend (one L2 round trip per pixel-plane, like the forward sweep); KMAX = 4: any
// k <= 4, one neighbour at a time.
// CTA = 2 x 2 pixels, 4 warps, like the packed forward sweep (plane_sweep_fwd.cu: smaller CTAs measured faster)
constexpr int kCorrPatchW = 2, kCorrPatchH = 2;
constexpr int kCorrWarps = kCorrPatchW * kCorrPatchH, kCorrThreads = kCorrWarps * 32;

// PX (both kernels): per-pixel depth hypotheses [V,D,H,W] (the *_px entry points)
template <typename TIn, int KMAX, int G, bool FULL, bool PX = false>
__global__ void __launch_bounds__(kCorrThreads, 8) corr_fwd_kernel(const CorrParams q) {
  const SweepParams& p = q.s;
  __shared__ WarpSample s_tab[kCorrWarps][kSlots];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  SweepCoord c;
  {
    int t = blockIdx.x;
    const int tx = t % p.tiles_x; t /= p.tiles_x;
    const int ty = t % p.tiles_y; t /= p.tiles_y;
    const int slice = t % p.slices;
    c.v = t / p.slices;
    c.x = tx * kCorrPatchW + (warp % kCorrPatchW);
    c.y = ty * kCorrPatchH + (warp / kCorrPatchW);
    c.ok = c.x < p.W && c.y < p.H;
    c.c0 = slice * 128 * G + 4 * lane;
  }
  if (!c.ok) return;
  const int C = p.C, k = p.k, HW = p.H * p.W;
  const TIn* feat = static_cast<const TIn*>(p.feat);
  const unsigned pix = (unsigned)(c.y * p.W + c.x);
  P4 ref[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    ref[g] = p4zero();
    if (group_on<FULL>(c.c0, g, C))
      ref[g] = p4from(Raw<TIn>::ld(feat + ((size_t)(c.v + p.ref_begin) * HW + pix) * C + c.c0 + 128 * g));
  }
  const TIn* nsrc[KMAX];
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    const int n = j < k ? __ldg(p.nbr + (size_t)c.v * k + j) : 0;
    nsrc[j] = feat + (size_t)n * HW * C + c.c0;      // only dereferenced behind a valid sample (id checked in the fill)
    asm volatile("" : "+l"(nsrc[j]));
  }
  // this lane's output slot: first lane of every channel group writes the group's mean
  const bool writer = (lane % q.lpg) == 0;
  int grp[G];
#pragma unroll
  for (int g = 0; g < G; ++g) grp[g] = group_on<FULL>(c.c0, g, C) ? (c.c0 + 128 * g) / q.cg : -1;
  const size_t nbr_stride = (size_t)p.D * HW * q.groups, plane_stride = (size_t)HW * q.groups;
  float* o = static_cast<float*>(p.out) + ((size_t)c.v * k * p.D * HW + pix) * q.groups;
  const int dc = kSlots / k;
  for (int d0 = 0; d0 < p.D; d0 += dc) {
    __syncwarp();
    fill_samples<PX ? kDepthPixels : kDepthPlanes>(s_tab[warp], p, c, d0, dc, lane);
    __syncwarp();
    const int dend = min(p.D, d0 + dc);
    for (int d = d0; d < dend; ++d) {
      const WarpSample* tab = s_tab[warp] + (d - d0) * k;
      float part[KMAX][G];
#pragma unroll
      for (int j = 0; j < KMAX; ++j)
#pragma unroll
        for (int g = 0; g < G; ++g) part[j][g] = 0.f;
      if (KMAX == 2) {
        const bool v0 = tab[0].p00 != kNoSample, v1 = tab[1].p00 != kNoSample;
        RawTaps<TIn, G> r0, r1;
        if (v0) load_taps<TIn, G, FULL>(nsrc[0], tab[0], c.c0, C, r0);
        if (v1) load_taps<TIn, G, FULL>(nsrc[KMAX - 1], tab[KMAX - 1], c.c0, C, r1);
        P4 wv[G];
        if (v0) {
          blend_taps<TIn, G>(r0, tab[0], wv);
#pragma unroll
          for (int g = 0; g < G; ++g) part[0][g] = lane_sum4(p4mul(ref[g], wv[g]));
        }
        if (v1) {
          blend_taps<TIn, G>(r1, tab[KMAX - 1], wv);
#pragma unroll
          for (int g = 0; g < G; ++g) part[KMAX - 1][g] = lane_sum4(p4mul(ref[g], wv[g]));
        }
      } else {
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
          if (j >= k || tab[j].p00 == kNoSample) continue;     // all four taps outside: warped = 0, cost = 0
          P4 wv[G];
          gather_taps_p<TIn, G, FULL>(nsrc[j], tab[j], c.c0, C, wv);
#pragma unroll
          for (int g = 0; g < G; ++g) part[j][g] = lane_sum4(p4mul(ref[g], wv[g]));
        }
      }
      if (KMAX == 2 && G == 2 && q.lpg == 8) {
        // The shipped shape (256 channels, 8 groups: 8 lanes per group, 2 neighbours x 2 channel blocks =
        // 4 values per lane).  A butterfly per value is 12 SHFL per pixel-plane, and shuffles travel through
        // the same L1TEX data stage as the tap loads that bound this kernel.  Halving instead: at every step
        // a lane keeps half of its values and hands the other half to its partner -- 2 + 1 + 1 = 4 SHFL --
        // and lane (bit2, bit1) of a group ends up owning value (neighbour bit2, block bit1).
        const bool b2 = lane & 4, b1 = lane & 2;
        const float s0 = b2 ? part[0][0] : part[1][0], s1 = b2 ? part[0][1] : part[1][1];
        float k0 = (b2 ? part[1][0] : part[0][0]) + __shfl_xor_sync(0xffffffffu, s0, 4);
        float k1 = (b2 ? part[1][1] : part[0][1]) + __shfl_xor_sync(0xffffffffu, s1, 4);
        float m = (b1 ? k1 : k0) + __shfl_xor_sync(0xffffffffu, b1 ? k0 : k1, 2);
        m += __shfl_xor_sync(0xffffffffu, m, 1);
        const int gsel = b1 ? grp[G - 1] : grp[0];
        if (!(lane & 1) && gsel >= 0) __stcs(o + (b2 ? nbr_stride : (size_t)0) + gsel, m * q.inv_cg);
        o += plane_stride;
        continue;
      }
      for (int sh = q.lpg >> 1; sh > 0; sh >>= 1) {
#pragma unroll
        for (int j = 0; j < KMAX; ++j)
#pragma unroll
          for (int g = 0; g < G; ++g) part[j][g] += __shfl_xor_sync(0xffffffffu, part[j][g], sh);
      }
      if (writer) {
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
          if (j >= k) continue;
#pragma unroll
          for (int g = 0; g < G; ++g)
            if (grp[g] >= 0) __stcs(o + j * nbr_stride + grp[g], part[j][g] * q.inv_cg);
        }
      }
      o += plane_stride;
    }
  }
}

// The gradient accumulator of the TAcc form, read where it is used: a pointer hoisted to the top of
// corr_bwd_kernel changed the register allocation of the fp32-RED kernels.
template <typename TAcc>
__device__ __forceinline__ TAcc* acc_ptr(const SweepParams& p) {
  if constexpr (sizeof(TAcc) == 8) return p.g_feat_q;
  else return p.g_feat;
}

// TAcc = float: fp32 vector REDs into p.g_feat; TAcc = long long: the deterministic form, fixed-point
// integer REDs into p.g_feat_q (common.cuh)
template <typename TIn, int G, bool FULL, typename TAcc = float, bool PX = false>
__global__ void __launch_bounds__(kSweepThreads) corr_bwd_kernel(const CorrParams q) {
  const SweepParams& p = q.s;
  __shared__ WarpSample s_tab[kSweepWarps][kSlots];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const SweepCoord c = sweep_coord<G>(p, warp, lane);
  if (!c.ok) return;
  const int C = p.C, k = p.k, HW = p.H * p.W;
  const TIn* feat = static_cast<const TIn*>(p.feat);
  const unsigned pix = (unsigned)(c.y * p.W + c.x);
  const size_t ref_off = ((size_t)(c.v + p.ref_begin) * HW + pix) * C + c.c0;
  float4 ref[G], gref[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    ref[g] = gref[g] = f4zero();
    if (group_on<FULL>(c.c0, g, C)) ref[g] = Io<TIn>::ld(feat + ref_off + 128 * g);
  }
  const float* g_out = static_cast<const float*>(p.g_out);
  const int dc = kSlots / k;
  for (int d0 = 0; d0 < p.D; d0 += dc) {
    __syncwarp();
    fill_samples<PX ? kDepthPixels : kDepthPlanes>(s_tab[warp], p, c, d0, dc, lane);
    __syncwarp();
    const int dend = min(p.D, d0 + dc);
    for (int d = d0; d < dend; ++d) {
      for (int j = 0; j < k; ++j) {
        const WarpSample s = s_tab[warp][(d - d0) * k + j];
        if (s.p00 == kNoSample) continue;       // warped = 0: no gradient to the reference view either
        const int n = __ldg(p.nbr + (size_t)c.v * k + j);
        const float* g_pp = g_out + ((((size_t)c.v * k + j) * p.D + d) * HW + pix) * q.groups;
        float4 wv[G], gw[G];
        gather_taps<TIn, G, FULL>(feat + (size_t)n * HW * C + c.c0, s, c.c0, C, wv);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          float gq = 0.f;
          if (group_on<FULL>(c.c0, g, C)) gq = __ldg(g_pp + (c.c0 + 128 * g) / q.cg) * q.inv_cg;
          gref[g] = f4fma(wv[g], gq, gref[g]);
          gw[g] = f4scale(ref[g], gq);
        }
        TAcc* dst = acc_ptr<TAcc>(p) + (size_t)n * HW * C + c.c0;
        red_tap<G, FULL, TAcc>(dst, s.p00, gw, s.w00, c.c0, C);
        red_tap<G, FULL, TAcc>(dst, s.p01, gw, s.w01, c.c0, C);
        red_tap<G, FULL, TAcc>(dst, s.p10, gw, s.w10, c.c0, C);
        red_tap<G, FULL, TAcc>(dst, s.p11, gw, s.w11, c.c0, C);
      }
    }
  }
  TAcc* dst = acc_ptr<TAcc>(p) + ref_off;
#pragma unroll
  for (int g = 0; g < G; ++g)
    if (group_on<FULL>(c.c0, g, C)) red_vec(dst + 128 * g, gref[g]);
}

static int corr_setup(const char* who, CorrParams& q, int num_groups) {
  SweepParams& p = q.s;
  if (p.k <= 0) return fail(MVSD_ERR_INVALID_ARG, "%s: needs at least one neighbour", who);
  if (num_groups <= 0 || p.C % num_groups != 0)
    return fail(MVSD_ERR_INVALID_ARG, "%s: C=%d is not divisible by num_groups=%d", who, p.C, num_groups);
  const int cg = p.C / num_groups;
  if (cg % 4 != 0 || cg > 128 || 128 % cg != 0)
    return fail(MVSD_ERR_UNSUPPORTED, "%s: %d channels per group (must be 4, 8, 16, 32, 64 or 128)", who, cg);
  q.groups = num_groups;
  q.cg = cg;
  q.lpg = cg / 4;
  q.inv_cg = 1.0f / (float)cg;                   // a power of two: exact
  p.corr_groups = num_groups;
  p.corr_inv_cg = q.inv_cg;
  p.corr_cg_shift = 0;
  while ((1 << p.corr_cg_shift) < cg) ++p.corr_cg_shift;
  return MVSD_OK;
}

// TAcc = long long: the deterministic backward, built with FULL = false only (ragged C by predication), as
// the variance's deterministic kernel is
template <bool BWD, typename TIn, typename TAcc>
static int corr_launch_t(CorrParams& q, cudaStream_t st) {
  constexpr bool det = std::is_same_v<TAcc, long long>;
  const char* name = det ? "plane_sweep_groupcorr_bwd_det"
                         : BWD ? "plane_sweep_groupcorr_bwd" : "plane_sweep_groupcorr_fwd";
  // the forward has its own CTA patch; grid errors name the family, or the deterministic kernel
  return sweep_launch(q.s, det ? name : "plane_sweep_groupcorr", BWD ? kPatchW : kCorrPatchW,
                      BWD ? kPatchH : kCorrPatchH, name, [&](dim3 grid, auto G2, auto FULL, auto PX) {
    constexpr int GG = G2 ? 2 : 1;
    if constexpr (det) corr_bwd_kernel<TIn, GG, false, TAcc, PX><<<grid, kSweepThreads, 0, st>>>(q);
    else if constexpr (BWD) corr_bwd_kernel<TIn, GG, FULL, TAcc, PX><<<grid, kSweepThreads, 0, st>>>(q);
    else if (q.s.k == 2) corr_fwd_kernel<TIn, 2, GG, FULL, PX><<<grid, kCorrThreads, 0, st>>>(q);
    else corr_fwd_kernel<TIn, 4, GG, FULL, PX><<<grid, kCorrThreads, 0, st>>>(q);
  });
}

template <bool BWD, typename TAcc = float>
static int corr_launch(CorrParams& q, const char* who, int feat_dtype, cudaStream_t st) {
  if (feat_dtype == MVSD_F32) return corr_launch_t<BWD, float, TAcc>(q, st);
  if (feat_dtype == MVSD_BF16) return corr_launch_t<BWD, __nv_bfloat16, TAcc>(q, st);
  return fail(MVSD_ERR_INVALID_ARG, "%s: bad dtype", who);
}

// per_pixel: depth_values is [V,D,H,W] (homo_warping's per-pixel branch, module.py:130-133)
static int groupcorr_fwd(const char* who, const void* feat, int feat_dtype, const int32_t* nbr_ids,
                         const float* hom, const float* depth_values, float* out, int V, int C, int D, int H,
                         int W, int k, int num_groups, int ref_begin, int n_feat_views, bool per_pixel,
                         void* stream) {
  CorrParams q{};
  if (int e = sweep_setup(q.s, who, {feat, out}, true, feat, nbr_ids, hom, depth_values, V, C, D, H, W, k,
                          MVSD_CHANNELS_LAST, ref_begin, n_feat_views, per_pixel))
    return e;
  q.s.out = out;
  if (int e = corr_setup(who, q, num_groups)) return e;
  return corr_launch<false>(q, who, feat_dtype, static_cast<cudaStream_t>(stream));
}

// g_acc: dL/dfeat, fp32 (TAcc = float) or the deterministic form's 64-bit fixed point (TAcc = long long)
template <typename TAcc>
static int groupcorr_bwd(const char* who, const float* g_out, const void* feat, int feat_dtype,
                         const int32_t* nbr_ids, const float* hom, const float* depth_values, TAcc* g_acc,
                         int V, int C, int D, int H, int W, int k, int num_groups, int ref_begin,
                         int n_feat_views, bool per_pixel, void* stream) {
  constexpr bool det = std::is_same_v<TAcc, long long>;
  CorrParams q{};
  if (int e = sweep_setup(q.s, who, {g_out, feat, g_acc}, true, feat, nbr_ids, hom, depth_values, V, C, D, H, W,
                          k, MVSD_CHANNELS_LAST, ref_begin, n_feat_views, per_pixel))
    return e;
  q.s.g_out = g_out;
  if constexpr (det) q.s.g_feat_q = g_acc;
  else q.s.g_feat = g_acc;
  if (int e = corr_setup(who, q, num_groups)) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // bf16 features, k = 2: the run-merging hand-off kernel of the variance backward with the correlation
  // algebra in its pixel body (same gather, same merged scatter); anything else, the deterministic form
  // and the test hook mvsd_set_tuning(5, 1): the pixel-per-warp kernel above
  if (!det && feat_dtype == MVSD_BF16 && k == 2 && tuning(5) != 1) return launch_bwd_run_corr(q.s, st);
  return corr_launch<true, TAcc>(q, who, feat_dtype, st);
}

}  // namespace mvsd

using namespace mvsd;

extern "C" int mvsd_plane_sweep_groupcorr_fwd(const void* feat, int feat_dtype, const int32_t* nbr_ids,
                                              const float* hom, const float* depth_values, float* out,
                                              int V, int C, int D, int H, int W, int k, int num_groups,
                                              int ref_begin, int n_feat_views, void* stream) {
  return groupcorr_fwd("plane_sweep_groupcorr_fwd", feat, feat_dtype, nbr_ids, hom, depth_values, out, V, C, D, H,
                       W, k, num_groups, ref_begin, n_feat_views, false, stream);
}

extern "C" int mvsd_plane_sweep_groupcorr_fwd_px(const void* feat, int feat_dtype, const int32_t* nbr_ids,
                                                 const float* hom, const float* depth_values, float* out,
                                                 int V, int C, int D, int H, int W, int k, int num_groups,
                                                 int ref_begin, int n_feat_views, void* stream) {
  return groupcorr_fwd("plane_sweep_groupcorr_fwd_px", feat, feat_dtype, nbr_ids, hom, depth_values, out, V, C, D,
                       H, W, k, num_groups, ref_begin, n_feat_views, true, stream);
}

extern "C" int mvsd_plane_sweep_groupcorr_bwd(const float* g_out, const void* feat, int feat_dtype,
                                              const int32_t* nbr_ids, const float* hom,
                                              const float* depth_values, float* g_feat, int V, int C,
                                              int D, int H, int W, int k, int num_groups, int ref_begin,
                                              int n_feat_views, void* stream) {
  return groupcorr_bwd("plane_sweep_groupcorr_bwd", g_out, feat, feat_dtype, nbr_ids, hom, depth_values, g_feat, V,
                       C, D, H, W, k, num_groups, ref_begin, n_feat_views, false, stream);
}

extern "C" int mvsd_plane_sweep_groupcorr_bwd_px(const float* g_out, const void* feat, int feat_dtype,
                                                 const int32_t* nbr_ids, const float* hom,
                                                 const float* depth_values, float* g_feat, int V, int C,
                                                 int D, int H, int W, int k, int num_groups, int ref_begin,
                                                 int n_feat_views, void* stream) {
  return groupcorr_bwd("plane_sweep_groupcorr_bwd_px", g_out, feat, feat_dtype, nbr_ids, hom, depth_values,
                       g_feat, V, C, D, H, W, k, num_groups, ref_begin, n_feat_views, true, stream);
}

extern "C" int mvsd_plane_sweep_groupcorr_bwd_det(const float* g_out, const void* feat, int feat_dtype,
                                                  const int32_t* nbr_ids, const float* hom,
                                                  const float* depth_values, int64_t* g_feat_q, int V, int C,
                                                  int D, int H, int W, int k, int num_groups, int ref_begin,
                                                  int n_feat_views, void* stream) {
  return groupcorr_bwd("plane_sweep_groupcorr_bwd_det", g_out, feat, feat_dtype, nbr_ids, hom, depth_values,
                       reinterpret_cast<long long*>(g_feat_q), V, C, D, H, W, k, num_groups, ref_begin,
                       n_feat_views, false, stream);
}

extern "C" int mvsd_plane_sweep_groupcorr_bwd_det_px(const float* g_out, const void* feat, int feat_dtype,
                                                     const int32_t* nbr_ids, const float* hom,
                                                     const float* depth_values, int64_t* g_feat_q, int V,
                                                     int C, int D, int H, int W, int k, int num_groups,
                                                     int ref_begin, int n_feat_views, void* stream) {
  return groupcorr_bwd("plane_sweep_groupcorr_bwd_det_px", g_out, feat, feat_dtype, nbr_ids, hom, depth_values,
                       reinterpret_cast<long long*>(g_feat_q), V, C, D, H, W, k, num_groups, ref_begin,
                       n_feat_views, true, stream);
}
