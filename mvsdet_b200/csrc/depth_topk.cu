// Depth probability epilogue of the cost-regularisation net, for sm_100a:
// softmax over the D planes, sigmoid sub-plane offsets, top-T hypotheses with
// their depths, and the depth expectation -- one pass, one thread per pixel.
//
// Replaces projects/NeRF-Det/nerfdet/mvsdet.py:470-482 together with
// MVSDet.sample_depth_prob (:266-283) and MVSDet.compute_avg_depth (:298-317):
// in the reference that is softmax + sigmoid + topk(T) + gather + topk(D)
// (a full sort) + gather, ~10 launches over [V,D,H,W] tensors.
//
// Each thread reads the 2*D values of its pixel (coalesced across the warp:
// consecutive threads are consecutive pixels), keeps them in registers
// (DMAX-sized arrays, D <= DMAX predicated), and writes every output once.
// ~18 MB of traffic per 20-view scene: latency-bound, not bandwidth-bound.
//
// Optional NVS-branch epilogue (SURVEY.md 8f rank 3), same registers, no extra pass:
//   opacity          = max_d prob_volume                         mvsdet.py:579
//   depth_scale      = z component of the unit ray through pixel (x, y) of a camera with the
//                      feature-level intrinsics and identity pose
//                      (compute_depth_scale[_MultiIntrin] mvsdet.py:1158-1218 through
//                      get_camera_params / lift, :1272-1313)
//   est_ray_depth    = est_depth    / (depth_scale + 1e-8)        mvsdet.py:494
//   ray_depth_coding = depth_coding / (depth_scale + 1e-8)        mvsdet.py:583
//
// Numerical notes.  depth_coding is accumulated in plane order; the reference sums the same
// terms in probability-sorted order (compute_avg_depth sorts with a full-length topk first), so
// the two agree to fp32 summation rounding (~1 ulp of the result, tested at 1e-6), not bit for
// bit.  A pixel whose logits contain NaN / +inf has an all-NaN softmax: no plane compares
// greater, and the hypotheses are then the lowest planes not yet taken (distinct indices, NaN
// densities) -- torch.topk also returns distinct indices there, in unspecified order.
#include "common.cuh"

namespace mvsd {

struct TopkParams {
  const float* cost;
  int64_t s_v, s_c, s_d, s_p;
  float* prob; float* off; float* est_depth; float* est_dens; int64_t* est_idx; float* coding;
  const int64_t* idx_in;
  const float* g_prob; const float* g_off; const float* g_depth; const float* g_dens;
  const float* g_coding; float* g_cost;
  float near, interval;
  int V, D, HW, T;
  int raw;   // 1: channel 0 already holds probabilities, channel 1 offsets
  // NVS epilogue (all optional)
  int W;                      // map width (pixel -> x, y)
  const float* ray_intr;      // [1 or V][16] feature-level intrinsics, or NULL
  int ray_per_view;
  float* opacity;             // [V,H,W]
  float* depth_scale;         // [V,H,W]
  float* est_ray_depth;       // [V,T,H,W]
  float* ray_coding;          // [V,H,W]
  const float* g_ray_depth;   // backward: dL/dest_ray_depth, dL/dray_depth_coding
  const float* g_ray_coding;
  // per-pixel depth hypotheses (the *_px entry points)
  const float* depth_values;  // [V,D,H,W] plane depths z_d
  const float* interval_map;  // [V,H,W] offset scale per pixel, or NULL: the scalar interval
  float* g_depth_values;      // backward: dL/ddepth_values, dL/dinterval_map (NULL = not requested)
  float* g_interval_map;
};

// 1 / (depth_scale + 1e-8) for pixel (x, y): lift() with z = 1 (mvsdet.py:1300-1313), identity
// pose, F.normalize; every step rounded separately as the reference's ATen ops do.
__device__ __forceinline__ float ray_depth_scale(const float* __restrict__ K, float x, float y) {
  const float fx = __ldg(K + 0), sk = __ldg(K + 1), cx = __ldg(K + 2), fy = __ldg(K + 5), cy = __ldg(K + 6);
  float xl = __fsub_rn(x, cx);
  xl = __fadd_rn(xl, __fdiv_rn(__fmul_rn(cy, sk), fy));
  xl = __fsub_rn(xl, __fdiv_rn(__fmul_rn(sk, y), fy));
  xl = __fdiv_rn(xl, fx);
  const float yl = __fdiv_rn(__fsub_rn(y, cy), fy);
  const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(xl, xl), __fmul_rn(yl, yl)), 1.0f));
  return __fdiv_rn(1.0f, fmaxf(nrm, 1e-12f));
}

// FAST (backward only): ex2.approx-based exp and approximate division -- the
// backward needs the probabilities to ~1e-6 relative for the gradient, not the
// bit pattern that decided the top-k (the indices come from the forward).
template <int DMAX, bool FAST>
__device__ __forceinline__ void load_pixel(const TopkParams& p, int v, int pix, float (&prob)[DMAX],
                                           float (&off)[DMAX]) {
  const float* c0 = p.cost + v * p.s_v + pix * p.s_p;
  const float* c1 = c0 + p.s_c;
  float mx = -INFINITY;
#pragma unroll
  for (int d = 0; d < DMAX; ++d) {
    if (d < p.D) {
      prob[d] = __ldg(c0 + d * p.s_d);
      off[d] = __ldg(c1 + d * p.s_d);
      mx = fmaxf(mx, prob[d]);
    }
  }
  if (p.raw) return;
  float sum = 0.f;
#pragma unroll
  for (int d = 0; d < DMAX; ++d) {
    if (d < p.D) {
      prob[d] = FAST ? __expf(prob[d] - mx) : expf(prob[d] - mx);
      sum += prob[d];
      off[d] = FAST ? __fdividef(1.0f, 1.0f + __expf(-off[d])) : 1.0f / (1.0f + expf(-off[d]));
    }
  }
  const float inv = FAST ? __fdividef(1.0f, sum) : 0.f;
#pragma unroll
  for (int d = 0; d < DMAX; ++d)
    if (d < p.D) prob[d] = FAST ? prob[d] * inv : prob[d] / sum;
}

// depth of plane d with its offset: (d*interval + near) + off*interval, each
// step rounded separately as in sample_depth_prob (mvsdet.py:278-281).
__device__ __forceinline__ float plane_depth(int d, float off, float near, float interval) {
  return __fadd_rn(__fadd_rn(__fmul_rn((float)d, interval), near), __fmul_rn(off, interval));
}

// The offset scale I of a pixel: the scalar interval, or with PX the pixel's entry of interval_map.
template <bool PX>
__device__ __forceinline__ float pixel_interval(const TopkParams& p, int v, int pix) {
  return PX && p.interval_map ? __ldg(p.interval_map + (size_t)v * p.HW + pix) : p.interval;
}

// Depth of hypothesis d of a pixel with its offset; o = (v*D + d)*HW + pix.  PX: z_d + off*I with
// z_d = depth_values[o], loaded here -- plane_depth's rounding sequence with fl(fl(d*interval) + near)
// replaced by z_d, so planes z_d = fl(fl(d*interval) + near) with I = interval give its bits.
template <bool PX>
__device__ __forceinline__ float hyp_depth(const TopkParams& p, size_t o, int d, float off, float I) {
  if constexpr (PX) return __fadd_rn(__ldg(p.depth_values + o), __fmul_rn(off, I));
  else return plane_depth(d, off, p.near, p.interval);
}

// PX: per-pixel hypotheses (depth_values, interval_map) instead of the planes d*interval + near.
template <int DMAX, bool PX>
__global__ void __launch_bounds__(128) depth_topk_fwd_kernel(const TopkParams p) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  const int v = blockIdx.y;
  if (pix >= p.HW) return;
  float prob[DMAX], off[DMAX];
  load_pixel<DMAX, false>(p, v, pix, prob, off);
  const float I = pixel_interval<PX>(p, v, pix);

  float coding = 0.f;
#pragma unroll
  for (int d = 0; d < DMAX; ++d) {
    if (d < p.D) {
      const size_t o = ((size_t)v * p.D + d) * p.HW + pix;
      if (p.prob) p.prob[o] = prob[d];
      if (p.off) p.off[o] = off[d];
      coding = fmaf(prob[d], hyp_depth<PX>(p, o, d, off[d], I), coding);
    }
  }
  if (p.coding) p.coding[(size_t)v * p.HW + pix] = coding;
  float ray_den = 1.0f;
  if (p.ray_intr) {
    const int y = pix / p.W, x = pix - y * p.W;
    const float sc = ray_depth_scale(p.ray_intr + (p.ray_per_view ? (size_t)v * 16 : 0), (float)x, (float)y);
    ray_den = __fadd_rn(sc, 1e-8f);
    if (p.depth_scale) p.depth_scale[(size_t)v * p.HW + pix] = sc;
    if (p.ray_coding) p.ray_coding[(size_t)v * p.HW + pix] = __fdiv_rn(coding, ray_den);
  }

  // top-T by repeated arg-max; strict '>' while scanning upwards keeps the
  // lowest plane index among equal probabilities.
  unsigned long long taken = 0ull;
  for (int t = 0; t < p.T; ++t) {
    float best = -INFINITY;
    int bi = -1;
    float boff = 0.f;
#pragma unroll
    for (int d = 0; d < DMAX; ++d) {
      if (d < p.D && !((taken >> d) & 1ull) && (prob[d] > best)) {
        best = prob[d];
        bi = d;
        boff = off[d];
      }
    }
    if (bi < 0) {              // NaN (or all -inf) probabilities: lowest plane not yet taken, indices stay distinct
      bi = __ffsll((long long)~taken) - 1;
#pragma unroll
      for (int d = 0; d < DMAX; ++d)
        if (d == bi) { best = prob[d]; boff = off[d]; }
    }
    taken |= 1ull << bi;
    const size_t o = ((size_t)v * p.T + t) * p.HW + pix;
    p.est_dens[o] = best;
    const float dep = hyp_depth<PX>(p, ((size_t)v * p.D + bi) * p.HW + pix, bi, boff, I);
    p.est_depth[o] = dep;
    if (p.est_idx) p.est_idx[o] = bi;
    if (t == 0 && p.opacity) p.opacity[(size_t)v * p.HW + pix] = best;
    if (p.est_ray_depth) p.est_ray_depth[o] = __fdiv_rn(dep, ray_den);
  }
}

// Backward.  With p = softmax(c), s = sigmoid(o), depth_d = d*I + near + s_d*I (PX: z_d + s_d*I):
//   dL/dp_d  = g_prob_d + g_coding*depth_d + [d == idx_t] g_dens_t
//   dL/ds_d  = g_off_d + g_coding*p_d*I + [d == idx_t] g_depth_t*I
//   dL/dc_d  = p_d (dL/dp_d - sum_e p_e dL/dp_e);   dL/do_d = dL/ds_d s_d (1 - s_d)
// and with PX
//   dL/dz_d  = g_coding*p_d + [d == idx_t] g_depth_t
//   dL/dI    = g_coding * sum_d p_d s_d + sum_t g_depth_t s_idx_t
// dL/dz_d is written in the plane loop and the hypotheses' terms are added to it in global memory
// (the thread's own stores) in a second pass over t, so it needs no third DMAX array.
template <int DMAX, bool PX>
__global__ void __launch_bounds__(128) depth_topk_bwd_kernel(const TopkParams p) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  const int v = blockIdx.y;
  if (pix >= p.HW) return;
  float prob[DMAX], off[DMAX], gp[DMAX], gs[DMAX];
  load_pixel<DMAX, true>(p, v, pix, prob, off);
  const float I = pixel_interval<PX>(p, v, pix);
  float gcod = p.g_coding ? __ldg(p.g_coding + (size_t)v * p.HW + pix) : 0.f;
  float ray_inv = 0.f;
  if (p.ray_intr && (p.g_ray_depth || p.g_ray_coding)) {
    const int y = pix / p.W, x = pix - y * p.W;
    const float sc = ray_depth_scale(p.ray_intr + (p.ray_per_view ? (size_t)v * 16 : 0), (float)x, (float)y);
    ray_inv = 1.0f / __fadd_rn(sc, 1e-8f);
    if (p.g_ray_coding) gcod = fmaf(__ldg(p.g_ray_coding + (size_t)v * p.HW + pix), ray_inv, gcod);
  }
#pragma unroll
  for (int d = 0; d < DMAX; ++d) {
    if (d < p.D) {
      const size_t o = ((size_t)v * p.D + d) * p.HW + pix;
      gp[d] = p.g_prob ? __ldg(p.g_prob + o) : 0.f;
      gs[d] = p.g_off ? __ldg(p.g_off + o) : 0.f;
      gp[d] = fmaf(gcod, hyp_depth<PX>(p, o, d, off[d], I), gp[d]);
      const float gcp = gcod * prob[d];
      // the per-view form reads p.interval at its use, as it always did: its code stays unchanged
      gs[d] = fmaf(gcp, PX ? I : p.interval, gs[d]);
      if constexpr (PX)
        if (p.g_depth_values) p.g_depth_values[o] = gcp;
    }
  }
  for (int t = 0; t < p.T; ++t) {
    const size_t o = ((size_t)v * p.T + t) * p.HW + pix;
    const int bi = (int)p.idx_in[o];
    const float gd = p.g_dens ? __ldg(p.g_dens + o) : 0.f;
    float gz = p.g_depth ? __ldg(p.g_depth + o) : 0.f;
    if (p.g_ray_depth && p.ray_intr) gz = fmaf(__ldg(p.g_ray_depth + o), ray_inv, gz);
#pragma unroll
    for (int d = 0; d < DMAX; ++d) {
      if (d == bi) {
        gp[d] += gd;
        gs[d] = fmaf(gz, PX ? I : p.interval, gs[d]);
      }
    }
  }
  float dot = 0.f;
#pragma unroll
  for (int d = 0; d < DMAX; ++d)
    if (d < p.D) dot = fmaf(prob[d], gp[d], dot);
  float sum_ps = 0.f;           // PX: sum_d p_d s_d, for dL/dI
#pragma unroll
  for (int d = 0; d < DMAX; ++d) {
    if (d < p.D) {
      const size_t o0 = (((size_t)v * 2 + 0) * p.D + d) * p.HW + pix;
      const size_t o1 = (((size_t)v * 2 + 1) * p.D + d) * p.HW + pix;
      p.g_cost[o0] = p.raw ? gp[d] : prob[d] * (gp[d] - dot);
      p.g_cost[o1] = p.raw ? gs[d] : gs[d] * off[d] * (1.0f - off[d]);
      if constexpr (PX) sum_ps = fmaf(prob[d], off[d], sum_ps);
    }
  }
  if constexpr (PX) {
    // the hypotheses' terms of dL/dz and dL/dI in a second pass over t, once gp and gs are dead
    float g_int = 0.f;
    for (int t = 0; t < p.T; ++t) {
      const size_t o = ((size_t)v * p.T + t) * p.HW + pix;
      const int bi = (int)p.idx_in[o];
      if ((unsigned)bi >= (unsigned)p.D) continue;
      float gz = p.g_depth ? __ldg(p.g_depth + o) : 0.f;
      if (p.g_ray_depth && p.ray_intr) gz = fmaf(__ldg(p.g_ray_depth + o), ray_inv, gz);
      float boff = 0.f;
#pragma unroll
      for (int d = 0; d < DMAX; ++d)
        if (d == bi) boff = off[d];
      if (p.g_depth_values) p.g_depth_values[((size_t)v * p.D + bi) * p.HW + pix] += gz;
      g_int = fmaf(gz, boff, g_int);
    }
    if (p.g_interval_map) p.g_interval_map[(size_t)v * p.HW + pix] = fmaf(gcod, sum_ps, g_int);
  }
}

// compute_depth_scale / compute_depth_scale_MultiIntrin alone (mvsdet.py:1158-1218)
__global__ void __launch_bounds__(128) ray_depth_scale_kernel(const float* __restrict__ intr, int per_view,
                                                              float* __restrict__ out, int HW, int W) {
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  const int v = blockIdx.y;
  if (pix >= HW) return;
  const int y = pix / W, x = pix - y * W;
  out[(size_t)v * HW + pix] = ray_depth_scale(intr + (per_view ? (size_t)v * 16 : 0), (float)x, (float)y);
}

static int check_topk(const char* who, int V, int D, int H, int W, int T) {
  if (V <= 0 || D <= 0 || H <= 0 || W <= 0 || T <= 0)
    return fail(MVSD_ERR_INVALID_ARG, "%s: non-positive dimension", who);
  if (D > MVSD_MAX_D) return fail(MVSD_ERR_UNSUPPORTED, "%s: D=%d > %d", who, D, MVSD_MAX_D);
  if (T > D || T > MVSD_MAX_T)
    return fail(MVSD_ERR_UNSUPPORTED, "%s: T=%d must be <= min(D, %d)", who, T, MVSD_MAX_T);
  if (V > 65535) return fail(MVSD_ERR_UNSUPPORTED, "%s: V=%d > 65535", who, V);
  return MVSD_OK;
}

template <bool BWD, bool PX>
static int launch_topk(const char* who, const TopkParams& p, cudaStream_t st) {
  dim3 grid((p.HW + 127) / 128, p.V);
  if (p.D <= 12) {                      // the shipped configs: D = num_monocular_samples = 12
    if (BWD) depth_topk_bwd_kernel<12, PX><<<grid, 128, 0, st>>>(p);
    else depth_topk_fwd_kernel<12, PX><<<grid, 128, 0, st>>>(p);
  } else if (p.D <= 16) {
    if (BWD) depth_topk_bwd_kernel<16, PX><<<grid, 128, 0, st>>>(p);
    else depth_topk_fwd_kernel<16, PX><<<grid, 128, 0, st>>>(p);
  } else if (p.D <= 32) {
    if (BWD) depth_topk_bwd_kernel<32, PX><<<grid, 128, 0, st>>>(p);
    else depth_topk_fwd_kernel<32, PX><<<grid, 128, 0, st>>>(p);
  } else {
    if (BWD) depth_topk_bwd_kernel<64, PX><<<grid, 128, 0, st>>>(p);
    else depth_topk_fwd_kernel<64, PX><<<grid, 128, 0, st>>>(p);
  }
  count_launch();
  return check_launch(who);
}

// The forward and backward behind both entry point pairs; depth_values != NULL selects the PX kernels.
static int topk_fwd(const char* who, const float* cost_out, int64_t s_v, int64_t s_c, int64_t s_d, int64_t s_p,
                    const float* depth_values, const float* interval_map, float near, float interval,
                    float* prob_volume, float* off_pred, float* est_depth, float* est_dens, int64_t* est_idx,
                    float* depth_coding, const float* ray_intrinsics, int ray_per_view, float* opacity,
                    float* depth_scale, float* est_ray_depth, float* ray_depth_coding, int raw, int V, int D,
                    int H, int W, int T, void* stream) {
  TopkParams p{};
  p.cost = cost_out; p.s_v = s_v; p.s_c = s_c; p.s_d = s_d; p.s_p = s_p;
  p.prob = prob_volume; p.off = off_pred; p.est_depth = est_depth; p.est_dens = est_dens;
  p.est_idx = est_idx; p.coding = depth_coding;
  p.W = W; p.ray_intr = ray_intrinsics; p.ray_per_view = ray_per_view ? 1 : 0; p.opacity = opacity;
  p.depth_scale = depth_scale; p.est_ray_depth = est_ray_depth; p.ray_coding = ray_depth_coding;
  p.near = near; p.interval = interval; p.V = V; p.D = D; p.HW = H * W; p.T = T;
  p.raw = raw ? 1 : 0;
  p.depth_values = depth_values; p.interval_map = interval_map;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  return depth_values ? launch_topk<false, true>(who, p, st) : launch_topk<false, false>(who, p, st);
}

static int topk_bwd(const char* who, const float* cost_out, int64_t s_v, int64_t s_c, int64_t s_d, int64_t s_p,
                    const int64_t* est_idx, const float* depth_values, const float* interval_map, float near,
                    float interval, const float* g_prob_volume, const float* g_off_pred, const float* g_est_depth,
                    const float* g_est_dens, const float* g_depth_coding, const float* ray_intrinsics,
                    int ray_per_view, const float* g_est_ray_depth, const float* g_ray_depth_coding,
                    float* g_cost_out, float* g_depth_values, float* g_interval_map, int raw, int V, int D,
                    int H, int W, int T, void* stream) {
  TopkParams p{};
  p.cost = cost_out; p.s_v = s_v; p.s_c = s_c; p.s_d = s_d; p.s_p = s_p;
  p.idx_in = est_idx; p.g_prob = g_prob_volume; p.g_off = g_off_pred; p.g_depth = g_est_depth;
  p.g_dens = g_est_dens; p.g_coding = g_depth_coding; p.g_cost = g_cost_out;
  p.W = W; p.ray_intr = ray_intrinsics; p.ray_per_view = ray_per_view ? 1 : 0;
  p.g_ray_depth = g_est_ray_depth; p.g_ray_coding = g_ray_depth_coding;
  p.near = near; p.interval = interval; p.V = V; p.D = D; p.HW = H * W; p.T = T;
  p.raw = raw ? 1 : 0;
  p.depth_values = depth_values; p.interval_map = interval_map;
  p.g_depth_values = g_depth_values; p.g_interval_map = g_interval_map;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  return depth_values ? launch_topk<true, true>(who, p, st) : launch_topk<true, false>(who, p, st);
}

}  // namespace mvsd

using namespace mvsd;

extern "C" int mvsd_depth_topk_fwd(const float* cost_out, int64_t s_v, int64_t s_c, int64_t s_d,
                                   int64_t s_p, float* prob_volume, float* off_pred,
                                   float* est_depth, float* est_dens, int64_t* est_idx,
                                   float* depth_coding, const float* ray_intrinsics,
                                   int ray_per_view, float* opacity, float* depth_scale,
                                   float* est_ray_depth, float* ray_depth_coding, float near,
                                   float interval, int raw, int V, int D, int H, int W, int T,
                                   void* stream) {
  if (int e = check_topk("depth_topk_fwd", V, D, H, W, T)) return e;
  if (!cost_out || !est_depth || !est_dens)
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_fwd: null pointer");
  if (!ray_intrinsics && (depth_scale || est_ray_depth || ray_depth_coding))
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_fwd: ray outputs need ray_intrinsics");
  return topk_fwd("depth_topk_fwd", cost_out, s_v, s_c, s_d, s_p, nullptr, nullptr, near, interval,
                  prob_volume, off_pred, est_depth, est_dens, est_idx, depth_coding, ray_intrinsics,
                  ray_per_view, opacity, depth_scale, est_ray_depth, ray_depth_coding, raw, V, D, H, W, T,
                  stream);
}

extern "C" int mvsd_depth_topk_bwd(const float* cost_out, int64_t s_v, int64_t s_c, int64_t s_d,
                                   int64_t s_p, const int64_t* est_idx,
                                   const float* g_prob_volume, const float* g_off_pred,
                                   const float* g_est_depth, const float* g_est_dens,
                                   const float* g_depth_coding, const float* ray_intrinsics,
                                   int ray_per_view, const float* g_est_ray_depth,
                                   const float* g_ray_depth_coding, float* g_cost_out, float near,
                                   float interval, int raw, int V, int D, int H, int W, int T,
                                   void* stream) {
  if (int e = check_topk("depth_topk_bwd", V, D, H, W, T)) return e;
  if (!cost_out || !est_idx || !g_cost_out)
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_bwd: null pointer");
  if (!ray_intrinsics && (g_est_ray_depth || g_ray_depth_coding))
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_bwd: ray gradients need ray_intrinsics");
  return topk_bwd("depth_topk_bwd", cost_out, s_v, s_c, s_d, s_p, est_idx, nullptr, nullptr, near, interval,
                  g_prob_volume, g_off_pred, g_est_depth, g_est_dens, g_depth_coding, ray_intrinsics,
                  ray_per_view, g_est_ray_depth, g_ray_depth_coding, g_cost_out, nullptr, nullptr, raw, V, D,
                  H, W, T, stream);
}

extern "C" int mvsd_depth_topk_fwd_px(const float* cost_out, int64_t s_v, int64_t s_c, int64_t s_d,
                                      int64_t s_p, const float* depth_values, const float* interval_map,
                                      float interval, float* prob_volume, float* off_pred, float* est_depth,
                                      float* est_dens, int64_t* est_idx, float* depth_coding,
                                      const float* ray_intrinsics, int ray_per_view, float* opacity,
                                      float* depth_scale, float* est_ray_depth, float* ray_depth_coding,
                                      int raw, int V, int D, int H, int W, int T, void* stream) {
  if (int e = check_topk("depth_topk_fwd_px", V, D, H, W, T)) return e;
  if (!cost_out || !depth_values || !est_depth || !est_dens)
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_fwd_px: null pointer");
  if (!ray_intrinsics && (depth_scale || est_ray_depth || ray_depth_coding))
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_fwd_px: ray outputs need ray_intrinsics");
  return topk_fwd("depth_topk_fwd_px", cost_out, s_v, s_c, s_d, s_p, depth_values, interval_map, 0.f,
                  interval, prob_volume, off_pred, est_depth, est_dens, est_idx, depth_coding, ray_intrinsics,
                  ray_per_view, opacity, depth_scale, est_ray_depth, ray_depth_coding, raw, V, D, H, W, T,
                  stream);
}

extern "C" int mvsd_depth_topk_bwd_px(const float* cost_out, int64_t s_v, int64_t s_c, int64_t s_d,
                                      int64_t s_p, const int64_t* est_idx, const float* depth_values,
                                      const float* interval_map, float interval, const float* g_prob_volume,
                                      const float* g_off_pred, const float* g_est_depth,
                                      const float* g_est_dens, const float* g_depth_coding,
                                      const float* ray_intrinsics, int ray_per_view,
                                      const float* g_est_ray_depth, const float* g_ray_depth_coding,
                                      float* g_cost_out, float* g_depth_values, float* g_interval_map,
                                      int raw, int V, int D, int H, int W, int T, void* stream) {
  if (int e = check_topk("depth_topk_bwd_px", V, D, H, W, T)) return e;
  if (!cost_out || !est_idx || !depth_values || !g_cost_out)
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_bwd_px: null pointer");
  if (g_interval_map && !interval_map)
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_bwd_px: g_interval_map needs interval_map");
  if (!ray_intrinsics && (g_est_ray_depth || g_ray_depth_coding))
    return fail(MVSD_ERR_INVALID_ARG, "depth_topk_bwd_px: ray gradients need ray_intrinsics");
  return topk_bwd("depth_topk_bwd_px", cost_out, s_v, s_c, s_d, s_p, est_idx, depth_values, interval_map, 0.f,
                  interval, g_prob_volume, g_off_pred, g_est_depth, g_est_dens, g_depth_coding, ray_intrinsics,
                  ray_per_view, g_est_ray_depth, g_ray_depth_coding, g_cost_out, g_depth_values, g_interval_map,
                  raw, V, D, H, W, T, stream);
}

extern "C" int mvsd_ray_depth_scale(const float* intrinsics, int per_view, float* depth_scale, int V,
                                    int H, int W, void* stream) {
  if (V <= 0 || H <= 0 || W <= 0) return fail(MVSD_ERR_INVALID_ARG, "ray_depth_scale: non-positive dimension");
  if (V > 65535) return fail(MVSD_ERR_UNSUPPORTED, "ray_depth_scale: V=%d > 65535", V);
  if (!intrinsics || !depth_scale) return fail(MVSD_ERR_INVALID_ARG, "ray_depth_scale: null pointer");
  dim3 grid((H * W + 127) / 128, V);
  ray_depth_scale_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(intrinsics, per_view ? 1 : 0,
                                                                                depth_scale, H * W, W);
  count_launch();
  return check_launch("ray_depth_scale");
}
