// Probabilistic voxel back-projection with fused view aggregation (forward and
// backward), for sm_100a.
//
// Replaces backproject_Weigh (projects/NeRF-Det/nerfdet/mvsdet.py:1372-1492)
// and the aggregation at mvsdet.py:511-515 / :681-682.  The reference runs V*T
// Python iterations of boolean-mask indexing (each a nonzero + host sync),
// materialises a [V,C,Nvox] volume (524 MB at V=20) and then reduces it; here a
// warp owns a voxel, its lanes test 32 views at a time (projection, rounding,
// depth test -- the integer part of the path, reproduced bit for bit), a
// ballot yields the valid views, and the warp gathers only those pixels'
// C-vectors (lanes = channels, 16-byte loads), accumulating in view order --
// a deterministic segmented reduction with no atomics in the forward.
//
// The backward is the scatter the north-star describes: per valid (view,voxel)
// pair one vector RED per 4 channels into the pixel's gradient, and a
// warp-shuffle reduction over C for the weight gradient.
#include "common.cuh"

namespace mvsd {

constexpr int kBpVox = 32;            // voxels per CTA (one 128 B store row per channel)
// Warps per CTA is a template parameter: more warps = fewer voxels per warp, i.e. a
// shorter dependent chain (project -> hypotheses -> ballot -> feature gather) per
// warp and higher occupancy; ncu showed the 8-warp / 4-voxels-per-warp form waiting
// on exactly that chain (long-scoreboard 4.8-11.9 per issue at 23% occupancy).
// 16 warps (2 voxels per warp) measured best: 52 -> 37 us fwd, 65 -> 46 us bwd.
constexpr int kTileStride = 132;      // floats per voxel row of the transpose tile

struct BpParams {
  const void* feat;
  const float* points; const float* proj; const float* depth; const float* prob;
  int64_t sv, sy, sx, st;
  float vs_z;
  float* out; int32_t* count; uint8_t* valid; float* weight;
  const float* g_out; const int32_t* count_in; float* g_feat; float* g_pn;
  long long* g_feat_q; long long* g_pn_q;      // deterministic form: 64-bit fixed-point accumulators
  int V, C, h, w, T, N, feat_h, feat_w;
};

struct LaneHit {
  int foff;       // (y*feat_w + x), pixel offset inside the allocated map
  int x, y, jstar;
  float weight;
  bool valid;
};

__device__ __forceinline__ LaneHit lane_test(const BpParams& p, int vi, float X, float Y, float Z) {
  LaneHit r;
  r.foff = 0; r.x = 0; r.y = 0; r.jstar = -1; r.weight = 0.f; r.valid = false;
  if (vi < p.V) {
    float P[12];
#pragma unroll
    for (int t = 0; t < 12; ++t) P[t] = __ldg(p.proj + (size_t)vi * 12 + t);
    VoxelHit hit = test_voxel<MVSD_MAX_T>(P, X, Y, Z, p.depth + vi * p.sv, p.prob + vi * p.sv,
                                          p.sy, p.sx, p.st, p.vs_z, p.h, p.w, p.T);
    r.valid = hit.valid;
    r.weight = hit.weight;
    r.jstar = hit.jstar;
    r.x = hit.x; r.y = hit.y;
    r.foff = hit.y * p.feat_w + hit.x;
  }
  return r;
}

// ---------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------
// PAIR (V <= 16, the view-sharded ranks): the projection + depth tests of the warp's TWO voxels run in one
// pass, views of voxel 0 on lanes 0-15 and of voxel 1 on lanes 16-31 -- with few views per rank the kernel is
// all test latency and half of the lanes were idle.  Same gather order (views ascending): same bits.
template <typename TIn, int G, int MODE, bool CFIRST, int kBpWarps, bool PAIR = false>
__global__ void __launch_bounds__(kBpWarps * 32) backproject_fwd_kernel(const BpParams p) {
  __shared__ float s_tile[CFIRST ? kBpVox * kTileStride : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int C = p.C, N = p.N;
  const TIn* feat = static_cast<const TIn*>(p.feat);
  const size_t map = (size_t)p.feat_h * p.feat_w;
  constexpr int VPW = kBpVox / kBpWarps;       // voxels per warp
  static_assert(!PAIR || (VPW == 2 && MODE != MVSD_BP_PER_VIEW), "pair form: two voxels per warp, aggregated modes");
  float4 res[VPW][G];

  if constexpr (PAIR) {
    const int half = lane >> 4, vi = lane & 15;
    const int ul = blockIdx.x * kBpVox + warp * VPW + half;          // this lane's voxel
#pragma unroll
    for (int i = 0; i < VPW; ++i)
#pragma unroll
      for (int g = 0; g < G; ++g) res[i][g] = make_float4(0.f, 0.f, 0.f, 0.f);
    LaneHit hit;
    hit.foff = 0; hit.x = 0; hit.y = 0; hit.jstar = -1; hit.weight = 0.f; hit.valid = false;
    if (ul < N && vi < p.V) {
      const float X = __ldg(p.points + ul), Y = __ldg(p.points + N + ul), Z = __ldg(p.points + 2 * (size_t)N + ul);
      hit = lane_test(p, vi, X, Y, Z);
      if (p.valid) p.valid[(size_t)vi * N + ul] = hit.valid ? 1 : 0;
      if (p.weight) p.weight[(size_t)vi * N + ul] = hit.weight;
    }
    const unsigned both = __ballot_sync(0xffffffffu, hit.valid);
#pragma unroll
    for (int i = 0; i < VPW; ++i) {
      const int u = blockIdx.x * kBpVox + warp * VPW + i;
      unsigned mask = (both >> (16 * i)) & 0xffffu;
      const int cnt = __popc(mask);
      while (mask) {
        const int vs = __ffs(mask) - 1;
        mask &= mask - 1;
        const int foff = __shfl_sync(0xffffffffu, hit.foff, vs + 16 * i);
        const float wgt = __shfl_sync(0xffffffffu, hit.weight, vs + 16 * i);
        const TIn* f = feat + ((size_t)vs * map + foff) * C + 4 * lane;
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (128 * g + 4 * lane >= C) continue;
          float4 a = Io<TIn>::ld(f + 128 * g);
          a.x = __fmul_rn(a.x, wgt); a.y = __fmul_rn(a.y, wgt);
          a.z = __fmul_rn(a.z, wgt); a.w = __fmul_rn(a.w, wgt);
          res[i][g].x = __fadd_rn(res[i][g].x, a.x); res[i][g].y = __fadd_rn(res[i][g].y, a.y);
          res[i][g].z = __fadd_rn(res[i][g].z, a.z); res[i][g].w = __fadd_rn(res[i][g].w, a.w);
        }
      }
      if (u >= N) continue;
      if (lane == 0 && p.count) p.count[u] = cnt;
      if (MODE == MVSD_BP_MEAN) {
        const float den = __fadd_rn((float)cnt, 1e-8f);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (cnt == 0) {
            res[i][g] = make_float4(0.f, 0.f, 0.f, 0.f);
          } else {
            res[i][g].x = __fdiv_rn(res[i][g].x, den); res[i][g].y = __fdiv_rn(res[i][g].y, den);
            res[i][g].z = __fdiv_rn(res[i][g].z, den); res[i][g].w = __fdiv_rn(res[i][g].w, den);
          }
        }
      }
      if (!CFIRST) {
#pragma unroll
        for (int g = 0; g < G; ++g)
          if (128 * g + 4 * lane < C)
            Io<float>::st(p.out + (size_t)u * C + 128 * g + 4 * lane, res[i][g]);
      }
    }
  } else {
#pragma unroll
  for (int i = 0; i < VPW; ++i) {
    const int u = blockIdx.x * kBpVox + warp * VPW + i;
#pragma unroll
    for (int g = 0; g < G; ++g) res[i][g] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (u >= N) continue;
    const float X = __ldg(p.points + u), Y = __ldg(p.points + N + u), Z = __ldg(p.points + 2 * (size_t)N + u);
    int cnt = 0;
    for (int vb = 0; vb < p.V; vb += 32) {
      const int vi = vb + lane;
      const LaneHit hit = lane_test(p, vi, X, Y, Z);
      if (vi < p.V) {
        if (p.valid) p.valid[(size_t)vi * N + u] = hit.valid ? 1 : 0;
        if (p.weight) p.weight[(size_t)vi * N + u] = hit.weight;
      }
      unsigned mask = __ballot_sync(0xffffffffu, hit.valid);
      cnt += __popc(mask);
      while (mask) {
        const int src = __ffs(mask) - 1;
        mask &= mask - 1;
        const int foff = __shfl_sync(0xffffffffu, hit.foff, src);
        const float wgt = __shfl_sync(0xffffffffu, hit.weight, src);
        const int vs = vb + src;
        const TIn* f = feat + ((size_t)vs * map + foff) * C + 4 * lane;
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (128 * g + 4 * lane >= C) continue;
          float4 a = Io<TIn>::ld(f + 128 * g);
          // volume = feature * weight (mvsdet.py:1459), then summed over views
          a.x = __fmul_rn(a.x, wgt); a.y = __fmul_rn(a.y, wgt);
          a.z = __fmul_rn(a.z, wgt); a.w = __fmul_rn(a.w, wgt);
          if (MODE == MVSD_BP_PER_VIEW) {
            Io<float>::st(p.out + ((size_t)vs * N + u) * C + 128 * g + 4 * lane, a);
          } else {
            res[i][g].x = __fadd_rn(res[i][g].x, a.x); res[i][g].y = __fadd_rn(res[i][g].y, a.y);
            res[i][g].z = __fadd_rn(res[i][g].z, a.z); res[i][g].w = __fadd_rn(res[i][g].w, a.w);
          }
        }
      }
    }
    if (MODE != MVSD_BP_PER_VIEW) {
      if (lane == 0 && p.count) p.count[u] = cnt;
      if (MODE == MVSD_BP_MEAN) {
        // sum / (count + 1e-8), zero where count == 0 (mvsdet.py:514-515)
        const float den = __fadd_rn((float)cnt, 1e-8f);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (cnt == 0) {
            res[i][g] = make_float4(0.f, 0.f, 0.f, 0.f);
          } else {
            res[i][g].x = __fdiv_rn(res[i][g].x, den); res[i][g].y = __fdiv_rn(res[i][g].y, den);
            res[i][g].z = __fdiv_rn(res[i][g].z, den); res[i][g].w = __fdiv_rn(res[i][g].w, den);
          }
        }
      }
      if (!CFIRST) {
#pragma unroll
        for (int g = 0; g < G; ++g)
          if (128 * g + 4 * lane < C)
            Io<float>::st(p.out + (size_t)u * C + 128 * g + 4 * lane, res[i][g]);
      }
    }
  }
  }

  if (MODE != MVSD_BP_PER_VIEW && CFIRST) {
    // [32 voxels][C] -> out[c*N + u]: stage 128 channels at a time so that each
    // store instruction writes 32 consecutive voxels of one channel (128 B).
    const int u0 = blockIdx.x * kBpVox;
#pragma unroll
    for (int g = 0; g < G; ++g) {
      __syncthreads();
#pragma unroll
      for (int i = 0; i < VPW; ++i)
        *reinterpret_cast<float4*>(&s_tile[(warp * VPW + i) * kTileStride + 4 * lane]) = res[i][g];
      __syncthreads();
      for (int cl = warp; cl < 128; cl += kBpWarps) {
        const int c = 128 * g + cl;
        if (c < C && u0 + lane < N) p.out[(size_t)c * N + u0 + lane] = s_tile[lane * kTileStride + cl];
      }
    }
  }
}

// ---------------------------------------------------------------------------
// backward (SURVEY.md Appendix A.4)
//   g_vol[i,:,u] = MEAN: g_out[:,u] / (count_u + 1e-8) (0 if count_u == 0)
//                  SUM:  g_out[:,u]       PER_VIEW: g_out[i,u,:]
//   dL/dfeat[i,y,x,:] += weight * g_vol ;  dL/dweight = sum_c g_vol[c] * feat[c]
//   dL/dpn[i,y,x,j*]  += dL/dweight  (j* = arg max routed by torch.max)
// ---------------------------------------------------------------------------
template <typename TIn, int G, int MODE, bool CFIRST, int kBpWarps, bool DET = false>
__global__ void __launch_bounds__(kBpWarps * 32) backproject_bwd_kernel(const BpParams p) {
  __shared__ float s_tile[CFIRST ? kBpVox * kTileStride : 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int C = p.C, N = p.N;
  const TIn* feat = static_cast<const TIn*>(p.feat);
  const size_t map = (size_t)p.feat_h * p.feat_w;
  constexpr int VPW = kBpVox / kBpWarps;
  float4 gv[VPW][G];
  const int u0 = blockIdx.x * kBpVox;

  if (MODE != MVSD_BP_PER_VIEW) {
    if (CFIRST) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
        __syncthreads();
        for (int cl = warp; cl < 128; cl += kBpWarps) {
          const int c = 128 * g + cl;
          s_tile[lane * kTileStride + cl] =
              (c < C && u0 + lane < N) ? __ldg(p.g_out + (size_t)c * N + u0 + lane) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < VPW; ++i)
          gv[i][g] = *reinterpret_cast<const float4*>(&s_tile[(warp * VPW + i) * kTileStride + 4 * lane]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < VPW; ++i) {
        const int u = u0 + warp * VPW + i;
#pragma unroll
        for (int g = 0; g < G; ++g)
          gv[i][g] = (u < N && 128 * g + 4 * lane < C)
                         ? Io<float>::ld(p.g_out + (size_t)u * C + 128 * g + 4 * lane)
                         : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  }

#pragma unroll
  for (int i = 0; i < VPW; ++i) {
    const int u = u0 + warp * VPW + i;
    if (u >= N) continue;
    if (MODE == MVSD_BP_MEAN) {
      const int cnt = __ldg(p.count_in + u);
      if (cnt == 0) continue;                        // zero-filled voxel: no gradient
      const float den = __fadd_rn((float)cnt, 1e-8f);
#pragma unroll
      for (int g = 0; g < G; ++g) {
        gv[i][g].x = __fdiv_rn(gv[i][g].x, den); gv[i][g].y = __fdiv_rn(gv[i][g].y, den);
        gv[i][g].z = __fdiv_rn(gv[i][g].z, den); gv[i][g].w = __fdiv_rn(gv[i][g].w, den);
      }
    }
    const float X = __ldg(p.points + u), Y = __ldg(p.points + N + u), Z = __ldg(p.points + 2 * (size_t)N + u);
    for (int vb = 0; vb < p.V; vb += 32) {
      const LaneHit hit = lane_test(p, vb + lane, X, Y, Z);
      unsigned mask = __ballot_sync(0xffffffffu, hit.valid);
      while (mask) {
        const int src = __ffs(mask) - 1;
        mask &= mask - 1;
        const int foff = __shfl_sync(0xffffffffu, hit.foff, src);
        const float wgt = __shfl_sync(0xffffffffu, hit.weight, src);
        const int vs = vb + src;
        const size_t fo = ((size_t)vs * map + foff) * C + 4 * lane;
        float dot = 0.f;
#pragma unroll
        for (int g = 0; g < G; ++g) {
          if (128 * g + 4 * lane >= C) continue;
          float4 gg;
          if (MODE == MVSD_BP_PER_VIEW)
            gg = Io<float>::ld(p.g_out + ((size_t)vs * N + u) * C + 128 * g + 4 * lane);
          else
            gg = gv[i][g];
          const float4 f = Io<TIn>::ld(feat + fo + 128 * g);
          dot = fmaf(gg.x, f.x, dot); dot = fmaf(gg.y, f.y, dot);
          dot = fmaf(gg.z, f.z, dot); dot = fmaf(gg.w, f.w, dot);
          const float4 contrib = make_float4(gg.x * wgt, gg.y * wgt, gg.z * wgt, gg.w * wgt);
          if (DET) red_add_fixed4(p.g_feat_q + fo + 128 * g, contrib);
          else red_add_f32x4(p.g_feat + fo + 128 * g, contrib);
        }
        dot = warp_sum(dot);
        if (lane == src && hit.jstar >= 0) {
          const int64_t po = vs * p.sv + hit.y * p.sy + hit.x * p.sx + hit.jstar * p.st;
          if (DET) { if (p.g_pn_q) red_add_fixed(p.g_pn_q + po, dot); }
          else if (p.g_pn) atomicAdd(p.g_pn + po, dot);
        }
      }
    }
  }
}

// pn = prob / sum_T prob  ->  g_prob_m = g_pn_m / S - (sum_j g_pn_j p_j) / S^2
__global__ void prob_norm_bwd_kernel(const float* __restrict__ prob, const float* __restrict__ g_pn,
                                     float* __restrict__ g_prob, int64_t sv, int64_t sy, int64_t sx,
                                     int64_t st, int V, int h, int w, int T) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= V * h * w) return;
  const int x = idx % w, y = (idx / w) % h, v = idx / (w * h);
  const int64_t base = v * sv + y * sy + x * sx;
  float S = 0.f, dot = 0.f;
  for (int j = 0; j < T; ++j) {
    const float pj = prob[base + j * st];
    S += pj;
    dot = fmaf(g_pn[base + j * st], pj, dot);
  }
  const float invS = 1.0f / S;
  for (int j = 0; j < T; ++j)
    g_prob[base + j * st] = (g_pn[base + j * st] - dot * invS) * invS;
}

__global__ void voxel_normalize_kernel(const float* __restrict__ sum, const int32_t* __restrict__ count,
                                       float* __restrict__ out, int cfirst, int C, int N) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)C * N) return;
  const int u = cfirst ? (int)(idx % N) : (int)(idx / C);
  const int cnt = count[u];
  out[idx] = cnt == 0 ? 0.f : __fdiv_rn(sum[idx], __fadd_rn((float)cnt, 1e-8f));
}

// ---------------------------------------------------------------------------
// dispatch
// ---------------------------------------------------------------------------
template <typename TIn, int G, bool BWD, int WARPS>
static int launch_bp_warps(const BpParams& p, int mode, bool cfirst, cudaStream_t st) {
  dim3 grid((p.N + kBpVox - 1) / kBpVox);
#define MVSD_BP_LAUNCH(M, CF)                                                                 \
  do {                                                                                        \
    if (BWD) backproject_bwd_kernel<TIn, G, M, CF, WARPS><<<grid, WARPS * 32, 0, st>>>(p);    \
    else if constexpr (M != MVSD_BP_PER_VIEW && kBpVox / WARPS == 2) {                        \
      if (p.V <= 16) backproject_fwd_kernel<TIn, G, M, CF, WARPS, true><<<grid, WARPS * 32, 0, st>>>(p); \
      else backproject_fwd_kernel<TIn, G, M, CF, WARPS><<<grid, WARPS * 32, 0, st>>>(p);      \
    } else backproject_fwd_kernel<TIn, G, M, CF, WARPS><<<grid, WARPS * 32, 0, st>>>(p);      \
  } while (0)
  if (mode == MVSD_BP_PER_VIEW) MVSD_BP_LAUNCH(MVSD_BP_PER_VIEW, false);
  else if (mode == MVSD_BP_MEAN && cfirst) MVSD_BP_LAUNCH(MVSD_BP_MEAN, true);
  else if (mode == MVSD_BP_MEAN) MVSD_BP_LAUNCH(MVSD_BP_MEAN, false);
  else if (cfirst) MVSD_BP_LAUNCH(MVSD_BP_SUM, true);
  else MVSD_BP_LAUNCH(MVSD_BP_SUM, false);
#undef MVSD_BP_LAUNCH
  count_launch();
  return check_launch(BWD ? "backproject_bwd" : "backproject_fwd");
}

template <typename TIn, int G, bool BWD>
static int launch_bp_mode(const BpParams& p, int mode, bool cfirst, cudaStream_t st) {
  // 16 warps per CTA: measured best on B200 (fwd 37 us, bwd 46 us; 8 and 32 warps were slower)
  return launch_bp_warps<TIn, G, BWD, 16>(p, mode, cfirst, st);
}

template <bool BWD>
static int launch_bp(const BpParams& p, int dtype, int mode, bool cfirst, cudaStream_t st) {
  const int G = (p.C + 127) / 128;
  if (dtype == MVSD_F32) {
    if (G == 1) return launch_bp_mode<float, 1, BWD>(p, mode, cfirst, st);
    if (G == 2) return launch_bp_mode<float, 2, BWD>(p, mode, cfirst, st);
    return launch_bp_mode<float, 4, BWD>(p, mode, cfirst, st);
  }
  if (dtype == MVSD_BF16) {
    if (G == 1) return launch_bp_mode<__nv_bfloat16, 1, BWD>(p, mode, cfirst, st);
    if (G == 2) return launch_bp_mode<__nv_bfloat16, 2, BWD>(p, mode, cfirst, st);
    return launch_bp_mode<__nv_bfloat16, 4, BWD>(p, mode, cfirst, st);
  }
  return fail(MVSD_ERR_INVALID_ARG, "backproject: bad dtype");
}

static int check_bp(const char* who, int V, int C, int h, int w, int T, int N, int feat_h,
                    int feat_w, int mode, int layout) {
  if (V <= 0 || C <= 0 || h <= 0 || w <= 0 || T <= 0 || N <= 0)
    return fail(MVSD_ERR_INVALID_ARG, "%s: non-positive dimension", who);
  if (feat_h < h || feat_w < w)
    return fail(MVSD_ERR_INVALID_ARG, "%s: crop [%d,%d] exceeds the map [%d,%d]", who, h, w, feat_h, feat_w);
  if (C % 4 != 0 || C > MVSD_MAX_C)
    return fail(MVSD_ERR_UNSUPPORTED, "%s: C=%d must be a multiple of 4 and <= %d", who, C, MVSD_MAX_C);
  if (T > MVSD_MAX_T) return fail(MVSD_ERR_UNSUPPORTED, "%s: T=%d > %d", who, T, MVSD_MAX_T);
  if (mode < MVSD_BP_MEAN || mode > MVSD_BP_PER_VIEW)
    return fail(MVSD_ERR_INVALID_ARG, "%s: bad mode %d", who, mode);
  if (layout != MVSD_CHANNELS_LAST && layout != MVSD_CHANNELS_FIRST)
    return fail(MVSD_ERR_INVALID_ARG, "%s: bad layout %d", who, layout);
  if (mode == MVSD_BP_PER_VIEW && layout != MVSD_CHANNELS_LAST)
    return fail(MVSD_ERR_UNSUPPORTED, "%s: per-view volumes are channels-last only", who);
  return MVSD_OK;
}

}  // namespace mvsd

using namespace mvsd;

extern "C" int mvsd_backproject_fwd(const void* feat, int feat_dtype, int feat_h, int feat_w,
                                    const float* points, const float* projection,
                                    const float* depth, const float* prob, int64_t dp_sv,
                                    int64_t dp_sy, int64_t dp_sx, int64_t dp_st, float vs_z,
                                    int mode, float* out, int out_layout, int32_t* count,
                                    uint8_t* valid, float* weight, int V, int C, int h, int w,
                                    int T, int N, void* stream) {
  if (int e = check_bp("backproject_fwd", V, C, h, w, T, N, feat_h, feat_w, mode, out_layout)) return e;
  if (!feat || !points || !projection || !depth || !prob || !out)
    return fail(MVSD_ERR_INVALID_ARG, "backproject_fwd: null pointer");
  if (mode != MVSD_BP_PER_VIEW && !count)
    return fail(MVSD_ERR_INVALID_ARG, "backproject_fwd: count is required in MEAN/SUM mode");
  BpParams p{};
  p.feat = feat; p.points = points; p.proj = projection; p.depth = depth; p.prob = prob;
  p.sv = dp_sv; p.sy = dp_sy; p.sx = dp_sx; p.st = dp_st; p.vs_z = vs_z;
  p.out = out; p.count = count; p.valid = valid; p.weight = weight;
  p.V = V; p.C = C; p.h = h; p.w = w; p.T = T; p.N = N; p.feat_h = feat_h; p.feat_w = feat_w;
  return launch_bp<false>(p, feat_dtype, mode, out_layout == MVSD_CHANNELS_FIRST,
                          static_cast<cudaStream_t>(stream));
}

extern "C" int mvsd_backproject_bwd(const float* g_out, int g_layout, int mode,
                                    const int32_t* count, const void* feat, int feat_dtype,
                                    int feat_h, int feat_w, const float* points,
                                    const float* projection, const float* depth, const float* prob,
                                    int64_t dp_sv, int64_t dp_sy, int64_t dp_sx, int64_t dp_st,
                                    float vs_z, float* g_feat, float* g_pn, int V, int C, int h,
                                    int w, int T, int N, void* stream) {
  if (int e = check_bp("backproject_bwd", V, C, h, w, T, N, feat_h, feat_w, mode, g_layout)) return e;
  if (!g_out || !feat || !points || !projection || !depth || !prob || !g_feat)
    return fail(MVSD_ERR_INVALID_ARG, "backproject_bwd: null pointer");
  if (mode == MVSD_BP_MEAN && !count)
    return fail(MVSD_ERR_INVALID_ARG, "backproject_bwd: count is required in MEAN mode");
  BpParams p{};
  p.feat = feat; p.points = points; p.proj = projection; p.depth = depth; p.prob = prob;
  p.sv = dp_sv; p.sy = dp_sy; p.sx = dp_sx; p.st = dp_st; p.vs_z = vs_z;
  p.g_out = g_out; p.count_in = count; p.g_feat = g_feat; p.g_pn = g_pn;
  p.V = V; p.C = C; p.h = h; p.w = w; p.T = T; p.N = N; p.feat_h = feat_h; p.feat_w = feat_w;
  return launch_bp<true>(p, feat_dtype, mode, g_layout == MVSD_CHANNELS_FIRST,
                         static_cast<cudaStream_t>(stream));
}

// Deterministic form of the MEAN-mode backward: the same kernel with 64-bit fixed-point integer REDs
// (common.cuh) into g_feat_q (nhwc, extent of feat) and g_pn_q (strides of prob).
template <typename TIn, int G>
static int launch_bp_bwd_det(const BpParams& p, bool cfirst, cudaStream_t st) {
  dim3 grid((p.N + kBpVox - 1) / kBpVox);
  if (cfirst) backproject_bwd_kernel<TIn, G, MVSD_BP_MEAN, true, 16, true><<<grid, 16 * 32, 0, st>>>(p);
  else backproject_bwd_kernel<TIn, G, MVSD_BP_MEAN, false, 16, true><<<grid, 16 * 32, 0, st>>>(p);
  count_launch();
  return check_launch("backproject_bwd_det");
}

extern "C" int mvsd_backproject_bwd_det(const float* g_out, int g_layout, const int32_t* count,
                                        const void* feat, int feat_dtype, int feat_h, int feat_w,
                                        const float* points, const float* projection, const float* depth,
                                        const float* prob, int64_t dp_sv, int64_t dp_sy, int64_t dp_sx,
                                        int64_t dp_st, float vs_z, int64_t* g_feat_q, int64_t* g_pn_q, int V,
                                        int C, int h, int w, int T, int N, void* stream) {
  if (int e = check_bp("backproject_bwd_det", V, C, h, w, T, N, feat_h, feat_w, MVSD_BP_MEAN, g_layout)) return e;
  if (!g_out || !feat || !points || !projection || !depth || !prob || !g_feat_q || !count)
    return fail(MVSD_ERR_INVALID_ARG, "backproject_bwd_det: null pointer");
  BpParams p{};
  p.feat = feat; p.points = points; p.proj = projection; p.depth = depth; p.prob = prob;
  p.sv = dp_sv; p.sy = dp_sy; p.sx = dp_sx; p.st = dp_st; p.vs_z = vs_z;
  p.g_out = g_out; p.count_in = count;
  p.g_feat_q = reinterpret_cast<long long*>(g_feat_q); p.g_pn_q = reinterpret_cast<long long*>(g_pn_q);
  p.V = V; p.C = C; p.h = h; p.w = w; p.T = T; p.N = N; p.feat_h = feat_h; p.feat_w = feat_w;
  const bool cfirst = g_layout == MVSD_CHANNELS_FIRST;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int G = (C + 127) / 128;
  if (feat_dtype == MVSD_F32) {
    if (G == 1) return launch_bp_bwd_det<float, 1>(p, cfirst, st);
    if (G == 2) return launch_bp_bwd_det<float, 2>(p, cfirst, st);
    return launch_bp_bwd_det<float, 4>(p, cfirst, st);
  }
  if (feat_dtype == MVSD_BF16) {
    if (G == 1) return launch_bp_bwd_det<__nv_bfloat16, 1>(p, cfirst, st);
    if (G == 2) return launch_bp_bwd_det<__nv_bfloat16, 2>(p, cfirst, st);
    return launch_bp_bwd_det<__nv_bfloat16, 4>(p, cfirst, st);
  }
  return fail(MVSD_ERR_INVALID_ARG, "backproject_bwd_det: bad dtype");
}

// Deterministic form of the SUM and PER_VIEW backwards (the MEAN mode stays with mvsd_backproject_bwd_det):
// SUM in both volume layouts, PER_VIEW channels-last only, as in the fp32 form.
template <typename TIn, int G>
static int launch_bp_bwd_det_mode(const BpParams& p, int mode, bool cfirst, cudaStream_t st) {
  dim3 grid((p.N + kBpVox - 1) / kBpVox);
  if (mode == MVSD_BP_PER_VIEW)
    backproject_bwd_kernel<TIn, G, MVSD_BP_PER_VIEW, false, 16, true><<<grid, 16 * 32, 0, st>>>(p);
  else if (cfirst) backproject_bwd_kernel<TIn, G, MVSD_BP_SUM, true, 16, true><<<grid, 16 * 32, 0, st>>>(p);
  else backproject_bwd_kernel<TIn, G, MVSD_BP_SUM, false, 16, true><<<grid, 16 * 32, 0, st>>>(p);
  count_launch();
  return check_launch("backproject_bwd_det_mode");
}

extern "C" int mvsd_backproject_bwd_det_mode(const float* g_out, int g_layout, int mode,
                                             const int32_t* count, const void* feat, int feat_dtype,
                                             int feat_h, int feat_w, const float* points,
                                             const float* projection, const float* depth, const float* prob,
                                             int64_t dp_sv, int64_t dp_sy, int64_t dp_sx, int64_t dp_st,
                                             float vs_z, int64_t* g_feat_q, int64_t* g_pn_q, int V, int C,
                                             int h, int w, int T, int N, void* stream) {
  const char* who = "backproject_bwd_det_mode";
  if (int e = check_bp(who, V, C, h, w, T, N, feat_h, feat_w, mode, g_layout)) return e;
  if (!g_out || !feat || !points || !projection || !depth || !prob || !g_feat_q)
    return fail(MVSD_ERR_INVALID_ARG, "%s: null pointer", who);
  if (mode == MVSD_BP_MEAN)
    return fail(MVSD_ERR_UNSUPPORTED, "%s: the MEAN mode's deterministic backward is mvsd_backproject_bwd_det", who);
  BpParams p{};
  p.feat = feat; p.points = points; p.proj = projection; p.depth = depth; p.prob = prob;
  p.sv = dp_sv; p.sy = dp_sy; p.sx = dp_sx; p.st = dp_st; p.vs_z = vs_z;
  p.g_out = g_out; p.count_in = count;
  p.g_feat_q = reinterpret_cast<long long*>(g_feat_q); p.g_pn_q = reinterpret_cast<long long*>(g_pn_q);
  p.V = V; p.C = C; p.h = h; p.w = w; p.T = T; p.N = N; p.feat_h = feat_h; p.feat_w = feat_w;
  const bool cfirst = g_layout == MVSD_CHANNELS_FIRST;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int G = (C + 127) / 128;
  if (feat_dtype == MVSD_F32) {
    if (G == 1) return launch_bp_bwd_det_mode<float, 1>(p, mode, cfirst, st);
    if (G == 2) return launch_bp_bwd_det_mode<float, 2>(p, mode, cfirst, st);
    return launch_bp_bwd_det_mode<float, 4>(p, mode, cfirst, st);
  }
  if (feat_dtype == MVSD_BF16) {
    if (G == 1) return launch_bp_bwd_det_mode<__nv_bfloat16, 1>(p, mode, cfirst, st);
    if (G == 2) return launch_bp_bwd_det_mode<__nv_bfloat16, 2>(p, mode, cfirst, st);
    return launch_bp_bwd_det_mode<__nv_bfloat16, 4>(p, mode, cfirst, st);
  }
  return fail(MVSD_ERR_INVALID_ARG, "%s: bad dtype", who);
}

extern "C" int mvsd_prob_norm_bwd(const float* prob, const float* g_pn, float* g_prob,
                                  int64_t dp_sv, int64_t dp_sy, int64_t dp_sx, int64_t dp_st,
                                  int V, int h, int w, int T, void* stream) {
  if (V <= 0 || h <= 0 || w <= 0 || T <= 0)
    return fail(MVSD_ERR_INVALID_ARG, "prob_norm_bwd: non-positive dimension");
  if (!prob || !g_pn || !g_prob) return fail(MVSD_ERR_INVALID_ARG, "prob_norm_bwd: null pointer");
  const int total = V * h * w;
  prob_norm_bwd_kernel<<<(total + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      prob, g_pn, g_prob, dp_sv, dp_sy, dp_sx, dp_st, V, h, w, T);
  count_launch();
  return check_launch("prob_norm_bwd");
}

extern "C" int mvsd_voxel_normalize(const float* sum, const int32_t* count, float* out, int layout,
                                    int C, int N, void* stream) {
  if (C <= 0 || N <= 0) return fail(MVSD_ERR_INVALID_ARG, "voxel_normalize: non-positive dimension");
  if (!sum || !count || !out) return fail(MVSD_ERR_INVALID_ARG, "voxel_normalize: null pointer");
  const size_t total = (size_t)C * N;
  voxel_normalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      sum, count, out, layout == MVSD_CHANNELS_FIRST ? 1 : 0, C, N);
  count_launch();
  return check_launch("voxel_normalize");
}
