// Plane-sweep variance volume, backward (and the homography warp's backward).
// See plane_sweep.cuh for the design.  What autograd computes through
// mvsdet.py:439-467 (SURVEY.md Appendix A.4), with n = k+1, mu = S1/n:
//   dL/dref       += sum_d G (2/n) (ref - mu_d)        (registers, one RED at the end)
//   dL/dwarped_j   = G (2/n) (warped_j - mu)            -> bilinear scatter into neighbour j
// The scatter uses fp32 16-byte vector REDs (red.global.add.v4.f32); ncu shows
// the L2 atomic unit (32 B / clk / slice) as the binding resource of this kernel.
#include "plane_sweep.cuh"

namespace mvsd {

// TAcc = float: fp32 vector REDs; TAcc = long long: the deterministic fixed-point form (common.cuh)
__device__ __forceinline__ void red_vec(float* a, float4 v) { red_add_f32x4(a, v); }
__device__ __forceinline__ void red_vec(long long* a, float4 v) { red_add_fixed4(a, v); }

template <int G, bool FULL, typename TAcc>
__device__ __forceinline__ void red_tap(TAcc* dst, unsigned off, const float4 (&gw)[G], float w,
                                        int c0, int C) {
  if (w == 0.f) return;                         // clamped (outside) tap: contributes nothing
  TAcc* a = at(dst, off);
#pragma unroll
  for (int g = 0; g < G; ++g)
    if (group_on<FULL>(c0, g, C)) red_vec(a + 128 * g, f4scale(gw[g], w));
}

// PX: per-pixel depth hypotheses [V,D,H,W] (the *_px entry points)
template <typename TIn, typename TG, int KMAX, int G, bool FULL, bool WARP_ONLY, typename TAcc = float,
          bool PX = false>
__global__ void __launch_bounds__(kSweepThreads) sweep_bwd_kernel(const SweepParams p) {
  TAcc* const g_acc = sizeof(TAcc) == 8 ? reinterpret_cast<TAcc*>(p.g_feat_q) : reinterpret_cast<TAcc*>(p.g_feat);
  __shared__ WarpSample s_tab[kSweepWarps][kSlots];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const SweepCoord c = sweep_coord<G>(p, warp, lane);
  if (!c.ok) return;
  const int C = p.C, k = p.k, HW = p.H * p.W;
  const TIn* feat = static_cast<const TIn*>(p.feat);
  const unsigned pix = (unsigned)(c.y * p.W + c.x);
  const size_t ref_off = ((size_t)(c.v + p.ref_begin) * HW + pix) * C + c.c0;
  const TG* g_pix = static_cast<const TG*>(p.g_out) + ((size_t)c.v * p.D * HW + pix) * C + c.c0;
  const size_t plane_stride = (size_t)HW * C;

  float4 ref[G], gref[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    ref[g] = f4zero();
    gref[g] = f4zero();
    if (!WARP_ONLY && group_on<FULL>(c.c0, g, C)) ref[g] = Io<TIn>::ld(feat + ref_off + 128 * g);
  }
  const TIn* nsrc[KMAX];
  TAcc* ndst[KMAX];
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    int n = c.v + p.ref_begin;
    if (!WARP_ONLY && j < k) n = __ldg(p.nbr + (size_t)c.v * k + j);
    nsrc[j] = feat + (size_t)n * HW * C + c.c0;
    ndst[j] = g_acc + (size_t)n * HW * C + c.c0;
  }
  const float inv_n = 1.0f / (float)(k + 1);
  const float two_inv_n = 2.0f * inv_n;
  const int dc = k > 0 ? kSlots / k : p.D;

  for (int d0 = 0; d0 < p.D; d0 += dc) {
    if (k > 0) {
      __syncwarp();
      fill_samples<WARP_ONLY ? kDepthEither : (PX ? kDepthPixels : kDepthPlanes)>(s_tab[warp], p, c, d0, dc, lane);
      __syncwarp();
    }
    const int dend = min(p.D, d0 + dc);
    for (int d = d0; d < dend; ++d) {
      const TG* gp = g_pix + (size_t)d * plane_stride;
      float4 gv[G], mu[G];
      float4 wv[KMAX][G];
      WarpSample smp[KMAX];
#pragma unroll
      for (int g = 0; g < G; ++g) {
        gv[g] = group_on<FULL>(c.c0, g, C) ? Io<TG>::ld_stream(gp + 128 * g) : f4zero();
        mu[g] = ref[g];
      }
#pragma unroll
      for (int j = 0; j < KMAX; ++j) {
#pragma unroll
        for (int g = 0; g < G; ++g) wv[j][g] = f4zero();
        if (j >= k) continue;
        smp[j] = s_tab[warp][(d - d0) * k + j];
        if (WARP_ONLY || smp[j].p00 == kNoSample) continue;
        gather_taps<TIn, G, FULL>(nsrc[j], smp[j], c.c0, C, wv[j]);
#pragma unroll
        for (int g = 0; g < G; ++g) mu[g] = f4add(mu[g], wv[j][g]);
      }
      if (!WARP_ONLY) {
#pragma unroll
        for (int g = 0; g < G; ++g) {
          mu[g] = f4scale(mu[g], inv_n);
          gv[g] = f4scale(gv[g], two_inv_n);
          gref[g] = f4fma(gv[g], f4sub(ref[g], mu[g]), gref[g]);
        }
      }
#pragma unroll
      for (int j = 0; j < KMAX; ++j) {
        if (j >= k) continue;
        const WarpSample s = smp[j];
        if (s.p00 == kNoSample) continue;
        float4 gw[G];
#pragma unroll
        for (int g = 0; g < G; ++g)
          gw[g] = WARP_ONLY ? gv[g] : f4mul(gv[g], f4sub(wv[j][g], mu[g]));
        red_tap<G, FULL, TAcc>(ndst[j], s.p00, gw, s.w00, c.c0, C);
        red_tap<G, FULL, TAcc>(ndst[j], s.p01, gw, s.w01, c.c0, C);
        red_tap<G, FULL, TAcc>(ndst[j], s.p10, gw, s.w10, c.c0, C);
        red_tap<G, FULL, TAcc>(ndst[j], s.p11, gw, s.w11, c.c0, C);
      }
    }
  }
  if (!WARP_ONLY) {
    TAcc* dst = g_acc + ref_off;
#pragma unroll
    for (int g = 0; g < G; ++g)
      if (group_on<FULL>(c.c0, g, C)) red_vec(dst + 128 * g, gref[g]);
  }
}

template <typename TIn, typename TG, bool WARP_ONLY>
static int launch_bwd_k(SweepParams& p, cudaStream_t st) {
  dim3 grid;
  const int G = sweep_groups(p.C);
  if (!sweep_grid(p, G, grid)) return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_bwd: grid too large");
  // generic fallback (k = 3, 4, the stand-alone warp, and the test hook): one instantiation per
  // dtype and channel-group count, every k <= 4 and ragged C handled by predication
#define MVSD_BWD(KM, GG, PX) sweep_bwd_kernel<TIn, TG, KM, GG, false, WARP_ONLY, float, PX><<<grid, kSweepThreads, 0, st>>>(p)
  if constexpr (WARP_ONLY) {
    if (G == 2) MVSD_BWD(1, 2, false); else MVSD_BWD(1, 1, false);
  } else if (p.depth_per_pixel) {
    if (G == 2) MVSD_BWD(4, 2, true); else MVSD_BWD(4, 1, true);
  } else {
    if (G == 2) MVSD_BWD(4, 2, false); else MVSD_BWD(4, 1, false);
  }
#undef MVSD_BWD
  count_launch();
  return check_launch("plane_sweep_bwd");
}

// deterministic form: the pixel-per-warp kernel with 64-bit fixed-point integer REDs
template <typename TIn, typename TG>
static int launch_bwd_det(SweepParams& p, cudaStream_t st) {
  dim3 grid;
  const int G = sweep_groups(p.C);
  if (!sweep_grid(p, G, grid)) return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_bwd_det: grid too large");
#define MVSD_BWD_DET(GG, PX) sweep_bwd_kernel<TIn, TG, 4, GG, false, false, long long, PX><<<grid, kSweepThreads, 0, st>>>(p)
  if (p.depth_per_pixel) {
    if (G == 2) MVSD_BWD_DET(2, true); else MVSD_BWD_DET(1, true);
  } else {
    if (G == 2) MVSD_BWD_DET(2, false); else MVSD_BWD_DET(1, false);
  }
#undef MVSD_BWD_DET
  count_launch();
  return check_launch("plane_sweep_bwd_det");
}

int launch_bwd_run(SweepParams& p, int feat_dtype, int g_dtype, cudaStream_t st);

__global__ void fixed_to_float_kernel(const long long* __restrict__ src, float* __restrict__ dst, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (float)((double)src[i] * (1.0 / 4294967296.0));      // one rounding, to nearest
}

}  // namespace mvsd

using namespace mvsd;

// per_pixel: depth_values is [V,D,H,W] (homo_warping's per-pixel branch, module.py:130-133)
static int plane_sweep_bwd(const char* who, const void* g_out, int g_dtype, int g_layout, const void* feat,
                           int feat_dtype, const int32_t* nbr_ids, const float* hom,
                           const float* depth_values, float* g_feat, int V, int C, int D, int H, int W,
                           int k, int ref_begin, int n_feat_views, bool per_pixel, void* stream) {
  if (int e = sweep_check(who, V, C, D, H, W, k, g_layout)) return e;
  if (!g_out || !feat || !g_feat || !depth_values || (k > 0 && (!nbr_ids || !hom)))
    return fail(MVSD_ERR_INVALID_ARG, "%s: null pointer", who);
  if (ref_begin < 0 || (long long)ref_begin + V > n_feat_views)
    return fail(MVSD_ERR_INVALID_ARG, "%s: reference views [%d, %d) exceed the %d feature views",
                who, ref_begin, ref_begin + V, n_feat_views);
  SweepParams p{};
  p.feat = feat; p.nbr = nbr_ids; p.hom = hom; p.depth = depth_values; p.g_out = g_out;
  p.g_feat = g_feat;
  p.V = V; p.C = C; p.D = D; p.H = H; p.W = W; p.k = k; p.ref_begin = ref_begin; p.n_feat = n_feat_views;
  p.depth_per_pixel = per_pixel ? 1 : 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Kernel selection.  k in {1, 2} (the reference uses k = min(2, V-1), mvsdet.py:432): the
  // run-merging kernels of plane_sweep_bwd_run.cu -- row hand-off + pipelined loads for bf16
  // features, the lean kernel for fp32 features.  Any other k (and the stand-alone warp): the
  // pixel-per-warp kernel above.  mvsd_set_tuning(5, 1) is a TEST hook, never used on the product
  // path: it sends k in {1, 2} to the pixel kernel too.
  if ((k == 1 || k == 2) && tuning(5) != 1) return launch_bwd_run(p, feat_dtype, g_dtype, st);
  if (feat_dtype == MVSD_F32 && g_dtype == MVSD_F32) return launch_bwd_k<float, float, false>(p, st);
  if (feat_dtype == MVSD_BF16 && g_dtype == MVSD_F32)
    return launch_bwd_k<__nv_bfloat16, float, false>(p, st);
  if (feat_dtype == MVSD_BF16 && g_dtype == MVSD_BF16)
    return launch_bwd_k<__nv_bfloat16, __nv_bfloat16, false>(p, st);
  return fail(MVSD_ERR_UNSUPPORTED, "%s: dtype combination not built", who);
}

static int plane_sweep_bwd_det(const char* who, const void* g_out, int g_dtype, int g_layout, const void* feat,
                               int feat_dtype, const int32_t* nbr_ids, const float* hom,
                               const float* depth_values, int64_t* g_feat_q, int V, int C, int D, int H,
                               int W, int k, int ref_begin, int n_feat_views, bool per_pixel, void* stream) {
  if (int e = sweep_check(who, V, C, D, H, W, k, g_layout)) return e;
  if (!g_out || !feat || !g_feat_q || !depth_values || (k > 0 && (!nbr_ids || !hom)))
    return fail(MVSD_ERR_INVALID_ARG, "%s: null pointer", who);
  if (ref_begin < 0 || (long long)ref_begin + V > n_feat_views)
    return fail(MVSD_ERR_INVALID_ARG, "%s: reference views [%d, %d) exceed the %d feature views",
                who, ref_begin, ref_begin + V, n_feat_views);
  SweepParams p{};
  p.feat = feat; p.nbr = nbr_ids; p.hom = hom; p.depth = depth_values; p.g_out = g_out;
  p.g_feat_q = reinterpret_cast<long long*>(g_feat_q);
  p.V = V; p.C = C; p.D = D; p.H = H; p.W = W; p.k = k; p.ref_begin = ref_begin; p.n_feat = n_feat_views;
  p.depth_per_pixel = per_pixel ? 1 : 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (feat_dtype == MVSD_F32 && g_dtype == MVSD_F32) return launch_bwd_det<float, float>(p, st);
  if (feat_dtype == MVSD_BF16 && g_dtype == MVSD_F32) return launch_bwd_det<__nv_bfloat16, float>(p, st);
  if (feat_dtype == MVSD_BF16 && g_dtype == MVSD_BF16) return launch_bwd_det<__nv_bfloat16, __nv_bfloat16>(p, st);
  return fail(MVSD_ERR_UNSUPPORTED, "%s: dtype combination not built", who);
}

extern "C" int mvsd_plane_sweep_bwd(const void* g_out, int g_dtype, int g_layout, const void* feat,
                                    int feat_dtype, const int32_t* nbr_ids, const float* hom,
                                    const float* depth_values, float* g_feat, int V, int C, int D,
                                    int H, int W, int k, int ref_begin, int n_feat_views,
                                    void* stream) {
  return plane_sweep_bwd("plane_sweep_bwd", g_out, g_dtype, g_layout, feat, feat_dtype, nbr_ids, hom, depth_values,
                         g_feat, V, C, D, H, W, k, ref_begin, n_feat_views, false, stream);
}

extern "C" int mvsd_plane_sweep_bwd_px(const void* g_out, int g_dtype, int g_layout, const void* feat,
                                       int feat_dtype, const int32_t* nbr_ids, const float* hom,
                                       const float* depth_values, float* g_feat, int V, int C, int D,
                                       int H, int W, int k, int ref_begin, int n_feat_views,
                                       void* stream) {
  return plane_sweep_bwd("plane_sweep_bwd_px", g_out, g_dtype, g_layout, feat, feat_dtype, nbr_ids, hom,
                         depth_values, g_feat, V, C, D, H, W, k, ref_begin, n_feat_views, true, stream);
}

extern "C" int mvsd_plane_sweep_bwd_det(const void* g_out, int g_dtype, int g_layout, const void* feat,
                                        int feat_dtype, const int32_t* nbr_ids, const float* hom,
                                        const float* depth_values, int64_t* g_feat_q, int V, int C, int D,
                                        int H, int W, int k, int ref_begin, int n_feat_views,
                                        void* stream) {
  return plane_sweep_bwd_det("plane_sweep_bwd_det", g_out, g_dtype, g_layout, feat, feat_dtype, nbr_ids, hom,
                             depth_values, g_feat_q, V, C, D, H, W, k, ref_begin, n_feat_views, false, stream);
}

extern "C" int mvsd_plane_sweep_bwd_det_px(const void* g_out, int g_dtype, int g_layout, const void* feat,
                                           int feat_dtype, const int32_t* nbr_ids, const float* hom,
                                           const float* depth_values, int64_t* g_feat_q, int V, int C, int D,
                                           int H, int W, int k, int ref_begin, int n_feat_views,
                                           void* stream) {
  return plane_sweep_bwd_det("plane_sweep_bwd_det_px", g_out, g_dtype, g_layout, feat, feat_dtype, nbr_ids, hom,
                             depth_values, g_feat_q, V, C, D, H, W, k, ref_begin, n_feat_views, true, stream);
}

extern "C" int mvsd_fixed_to_float(const int64_t* src, float* dst, int64_t n, void* stream) {
  if (n <= 0) return fail(MVSD_ERR_INVALID_ARG, "fixed_to_float: non-positive size");
  if (!src || !dst) return fail(MVSD_ERR_INVALID_ARG, "fixed_to_float: null pointer");
  const long long blocks = (n + 255) / 256;
  if (blocks > 2147483647LL) return fail(MVSD_ERR_UNSUPPORTED, "fixed_to_float: too many elements");
  fixed_to_float_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const long long*>(src), dst, (long long)n);
  count_launch();
  return check_launch("fixed_to_float");
}

extern "C" int mvsd_homo_warp_bwd(const void* g_out, int g_dtype, int g_layout, const float* hom,
                                  const float* depth_values, float* g_src, int B, int C, int D,
                                  int H, int W, int depth_per_pixel, void* stream) {
  if (int e = sweep_check("homo_warp_bwd", B, C, D, H, W, 1, g_layout)) return e;
  if (!g_out || !hom || !depth_values || !g_src)
    return fail(MVSD_ERR_INVALID_ARG, "homo_warp_bwd: null pointer");
  SweepParams p{};
  p.feat = nullptr; p.nbr = nullptr; p.hom = hom; p.depth = depth_values; p.g_out = g_out;
  p.g_feat = g_src;
  p.V = B; p.C = C; p.D = D; p.H = H; p.W = W; p.k = 1; p.ref_begin = 0; p.n_feat = B;
  p.depth_per_pixel = depth_per_pixel ? 1 : 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (g_dtype == MVSD_F32) return launch_bwd_k<float, float, true>(p, st);
  if (g_dtype == MVSD_BF16) return launch_bwd_k<float, __nv_bfloat16, true>(p, st);
  return fail(MVSD_ERR_INVALID_ARG, "homo_warp_bwd: bad dtype");
}
