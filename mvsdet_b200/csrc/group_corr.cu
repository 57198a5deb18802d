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
// the correlation algebra in the pixel body), otherwise the un-merged pixel-per-warp kernel below.
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

template <int G, bool FULL>
__device__ __forceinline__ void corr_red_tap(float* dst, unsigned off, const float4 (&gw)[G], float w,
                                             int c0, int C) {
  if (w == 0.f) return;                         // clamped (outside) tap: contributes nothing
  float* a = at(dst, off);
#pragma unroll
  for (int g = 0; g < G; ++g)
    if (group_on<FULL>(c0, g, C)) red_add_f32x4(a + 128 * g, f4scale(gw[g], w));
}

template <typename TIn, int G, bool FULL, bool PX = false>
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
        float* dst = p.g_feat + (size_t)n * HW * C + c.c0;
        corr_red_tap<G, FULL>(dst, s.p00, gw, s.w00, c.c0, C);
        corr_red_tap<G, FULL>(dst, s.p01, gw, s.w01, c.c0, C);
        corr_red_tap<G, FULL>(dst, s.p10, gw, s.w10, c.c0, C);
        corr_red_tap<G, FULL>(dst, s.p11, gw, s.w11, c.c0, C);
      }
    }
  }
  float* dst = p.g_feat + ref_off;
#pragma unroll
  for (int g = 0; g < G; ++g)
    if (group_on<FULL>(c.c0, g, C)) red_add_f32x4(dst + 128 * g, gref[g]);
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

template <bool BWD, typename TIn, bool PX>
static int corr_launch(CorrParams& q, cudaStream_t st) {
  dim3 grid;
  const int G = sweep_groups(q.s.C);
  if (!sweep_grid(q.s, G, grid)) return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_groupcorr: grid too large");
  if constexpr (!BWD) {                          // the forward has its own CTA patch
    q.s.tiles_x = (q.s.W + kCorrPatchW - 1) / kCorrPatchW;
    q.s.tiles_y = (q.s.H + kCorrPatchH - 1) / kCorrPatchH;
    const long long blocks = (long long)q.s.V * q.s.slices * q.s.tiles_y * q.s.tiles_x;
    if (blocks > 2147483647LL) return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_groupcorr: grid too large");
    grid = dim3((unsigned)blocks);
  }
  const bool full = q.s.C % (128 * G) == 0;
#define MVSD_CORR(GG, FU)                                                        \
  do {                                                                           \
    if constexpr (BWD) corr_bwd_kernel<TIn, GG, FU, PX><<<grid, kSweepThreads, 0, st>>>(q); \
    else if (q.s.k == 2) corr_fwd_kernel<TIn, 2, GG, FU, PX><<<grid, kCorrThreads, 0, st>>>(q); \
    else corr_fwd_kernel<TIn, 4, GG, FU, PX><<<grid, kCorrThreads, 0, st>>>(q);  \
  } while (0)
  if (G == 2) { if (full) MVSD_CORR(2, true); else MVSD_CORR(2, false); }
  else { if (full) MVSD_CORR(1, true); else MVSD_CORR(1, false); }
#undef MVSD_CORR
  count_launch();
  return check_launch(BWD ? "plane_sweep_groupcorr_bwd" : "plane_sweep_groupcorr_fwd");
}

int launch_bwd_run_corr(SweepParams& p, int feat_dtype, cudaStream_t st);     // plane_sweep_bwd_run.cu

template <bool BWD, typename TIn>
static int corr_launch_px(CorrParams& q, cudaStream_t st) {
  return q.s.depth_per_pixel ? corr_launch<BWD, TIn, true>(q, st) : corr_launch<BWD, TIn, false>(q, st);
}

// per_pixel: depth_values is [V,D,H,W] (homo_warping's per-pixel branch, module.py:130-133)
static int groupcorr_fwd(const char* who, const void* feat, int feat_dtype, const int32_t* nbr_ids,
                         const float* hom, const float* depth_values, float* out, int V, int C, int D, int H,
                         int W, int k, int num_groups, int ref_begin, int n_feat_views, bool per_pixel,
                         void* stream) {
  if (int e = sweep_check(who, V, C, D, H, W, k, MVSD_CHANNELS_LAST)) return e;
  if (!feat || !out || !depth_values || !nbr_ids || !hom)
    return fail(MVSD_ERR_INVALID_ARG, "%s: null pointer", who);
  if (ref_begin < 0 || (long long)ref_begin + V > n_feat_views)
    return fail(MVSD_ERR_INVALID_ARG, "%s: reference views [%d, %d) exceed the %d feature views",
                who, ref_begin, ref_begin + V, n_feat_views);
  CorrParams q{};
  SweepParams& p = q.s;
  p.feat = feat; p.nbr = nbr_ids; p.hom = hom; p.depth = depth_values; p.out = out;
  p.V = V; p.C = C; p.D = D; p.H = H; p.W = W; p.k = k; p.ref_begin = ref_begin; p.n_feat = n_feat_views;
  p.depth_per_pixel = per_pixel ? 1 : 0;
  if (int e = corr_setup(who, q, num_groups)) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (feat_dtype == MVSD_F32) return corr_launch_px<false, float>(q, st);
  if (feat_dtype == MVSD_BF16) return corr_launch_px<false, __nv_bfloat16>(q, st);
  return fail(MVSD_ERR_INVALID_ARG, "%s: bad dtype", who);
}

static int groupcorr_bwd(const char* who, const float* g_out, const void* feat, int feat_dtype,
                         const int32_t* nbr_ids, const float* hom, const float* depth_values, float* g_feat,
                         int V, int C, int D, int H, int W, int k, int num_groups, int ref_begin,
                         int n_feat_views, bool per_pixel, void* stream) {
  if (int e = sweep_check(who, V, C, D, H, W, k, MVSD_CHANNELS_LAST)) return e;
  if (!g_out || !feat || !g_feat || !depth_values || !nbr_ids || !hom)
    return fail(MVSD_ERR_INVALID_ARG, "%s: null pointer", who);
  if (ref_begin < 0 || (long long)ref_begin + V > n_feat_views)
    return fail(MVSD_ERR_INVALID_ARG, "%s: reference views [%d, %d) exceed the %d feature views",
                who, ref_begin, ref_begin + V, n_feat_views);
  CorrParams q{};
  SweepParams& p = q.s;
  p.feat = feat; p.nbr = nbr_ids; p.hom = hom; p.depth = depth_values; p.g_out = g_out; p.g_feat = g_feat;
  p.V = V; p.C = C; p.D = D; p.H = H; p.W = W; p.k = k; p.ref_begin = ref_begin; p.n_feat = n_feat_views;
  p.depth_per_pixel = per_pixel ? 1 : 0;
  if (int e = corr_setup(who, q, num_groups)) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // bf16 features, k = 2: the run-merging hand-off kernel of the variance backward with the correlation
  // algebra in its pixel body (same gather, same merged scatter); anything else (and the test hook
  // mvsd_set_tuning(5, 1)): the pixel-per-warp kernel above
  if (tuning(5) != 1) {
    const int rc = launch_bwd_run_corr(p, feat_dtype, st);
    if (rc >= 0) return rc;
  }
  if (feat_dtype == MVSD_F32) return corr_launch_px<true, float>(q, st);
  if (feat_dtype == MVSD_BF16) return corr_launch_px<true, __nv_bfloat16>(q, st);
  return fail(MVSD_ERR_INVALID_ARG, "%s: bad dtype", who);
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
