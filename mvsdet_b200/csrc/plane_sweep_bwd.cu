// Plane-sweep variance volume, backward (and the homography warp's backward).
// See plane_sweep.cuh for the design.  What autograd computes through
// mvsdet.py:439-467 (SURVEY.md Appendix A.4), with n = k+1, mu = S1/n:
//   dL/dref       += sum_d G (2/n) (ref - mu_d)        (registers, one RED at the end)
//   dL/dwarped_j   = G (2/n) (warped_j - mu)            -> bilinear scatter into neighbour j
// The scatter uses fp32 16-byte vector REDs (red.global.add.v4.f32); ncu shows
// the L2 atomic unit (32 B / clk / slice) as the binding resource of this kernel.
#include "plane_sweep.cuh"

namespace mvsd {

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

// The pixel-per-warp kernel: the variance backward for k = 0, 3, 4 (and every k through the test hook),
// its deterministic form (TAcc = long long) and the stand-alone warp.  One instantiation per dtype and
// channel-group count: every k <= 4 and ragged C handled by predication.
template <typename TIn, typename TG, bool WARP_ONLY, typename TAcc>
static int launch_bwd_k(SweepParams& p, cudaStream_t st) {
  const char* name = sizeof(TAcc) == 8 ? "plane_sweep_bwd_det" : "plane_sweep_bwd";
  return sweep_launch(p, name, kPatchW, kPatchH, name, [&](dim3 grid, auto G2, auto /*FULL*/, auto PX) {
    constexpr int GG = G2 ? 2 : 1;
    if constexpr (WARP_ONLY)              // reads either depth form (fill_samples<kDepthEither>)
      sweep_bwd_kernel<TIn, TG, 1, GG, false, true><<<grid, kSweepThreads, 0, st>>>(p);
    else
      sweep_bwd_kernel<TIn, TG, 4, GG, false, false, TAcc, PX><<<grid, kSweepThreads, 0, st>>>(p);
  });
}

__global__ void fixed_to_float_kernel(const long long* __restrict__ src, float* __restrict__ dst, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (float)((double)src[i] * (1.0 / 4294967296.0));      // one rounding, to nearest
}

}  // namespace mvsd

using namespace mvsd;

// per_pixel: depth_values is [V,D,H,W] (homo_warping's per-pixel branch, module.py:130-133).
// g_acc: dL/dfeat, fp32 (TAcc = float) or the deterministic form's 64-bit fixed point (TAcc = long long).
template <typename TAcc>
static int plane_sweep_bwd(const char* who, const void* g_out, int g_dtype, int g_layout, const void* feat,
                           int feat_dtype, const int32_t* nbr_ids, const float* hom,
                           const float* depth_values, TAcc* g_acc, int V, int C, int D, int H, int W,
                           int k, int ref_begin, int n_feat_views, bool per_pixel, void* stream) {
  constexpr bool det = std::is_same_v<TAcc, long long>;
  SweepParams p;
  if (int e = sweep_setup(p, who, {g_out, feat, g_acc}, k > 0, feat, nbr_ids, hom, depth_values, V, C, D, H, W,
                          k, g_layout, ref_begin, n_feat_views, per_pixel))
    return e;
  p.g_out = g_out;
  if constexpr (det) p.g_feat_q = g_acc;
  else p.g_feat = g_acc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // Kernel selection.  k in {1, 2} (the reference uses k = min(2, V-1), mvsdet.py:432): the
  // run-merging kernels of plane_sweep_bwd_run.cu -- row hand-off + pipelined loads for bf16
  // features, the lean kernel for fp32 features.  Any other k, and the deterministic form: the
  // pixel-per-warp kernel above.  mvsd_set_tuning(5, 1) is a TEST hook, never used on the product
  // path: it sends k in {1, 2} to the pixel kernel too.
  if (!det && (k == 1 || k == 2) && tuning(5) != 1) return launch_bwd_run(p, feat_dtype, g_dtype, st);
  if (feat_dtype == MVSD_F32 && g_dtype == MVSD_F32) return launch_bwd_k<float, float, false, TAcc>(p, st);
  if (feat_dtype == MVSD_BF16 && g_dtype == MVSD_F32)
    return launch_bwd_k<__nv_bfloat16, float, false, TAcc>(p, st);
  if (feat_dtype == MVSD_BF16 && g_dtype == MVSD_BF16)
    return launch_bwd_k<__nv_bfloat16, __nv_bfloat16, false, TAcc>(p, st);
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
  return plane_sweep_bwd("plane_sweep_bwd_det", g_out, g_dtype, g_layout, feat, feat_dtype, nbr_ids, hom,
                         depth_values, reinterpret_cast<long long*>(g_feat_q), V, C, D, H, W, k, ref_begin,
                         n_feat_views, false, stream);
}

extern "C" int mvsd_plane_sweep_bwd_det_px(const void* g_out, int g_dtype, int g_layout, const void* feat,
                                           int feat_dtype, const int32_t* nbr_ids, const float* hom,
                                           const float* depth_values, int64_t* g_feat_q, int V, int C, int D,
                                           int H, int W, int k, int ref_begin, int n_feat_views,
                                           void* stream) {
  return plane_sweep_bwd("plane_sweep_bwd_det_px", g_out, g_dtype, g_layout, feat, feat_dtype, nbr_ids, hom,
                         depth_values, reinterpret_cast<long long*>(g_feat_q), V, C, D, H, W, k, ref_begin,
                         n_feat_views, true, stream);
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
  SweepParams p;
  if (int e = sweep_setup(p, "homo_warp_bwd", {g_out, hom, g_src}, false, nullptr, nullptr, hom, depth_values, B, C,
                          D, H, W, 1, g_layout, 0, B, depth_per_pixel != 0))
    return e;
  p.g_out = g_out;
  p.g_feat = g_src;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (g_dtype == MVSD_F32) return launch_bwd_k<float, float, true, float>(p, st);
  if (g_dtype == MVSD_BF16) return launch_bwd_k<float, __nv_bfloat16, true, float>(p, st);
  return fail(MVSD_ERR_INVALID_ARG, "homo_warp_bwd: bad dtype");
}
