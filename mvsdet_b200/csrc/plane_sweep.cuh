// Shared pieces of the plane-sweep kernels (forward: plane_sweep_fwd.cu,
// backward: plane_sweep_bwd.cu), sm_100a.
//
// Replaces projects/NeRF-Det/nerfdet/mvsdet.py:439-467 and
// mvs_models/module.py:105-146 of the reference: instead of materialising the
// repeated reference volume, k warped [V,C,D,H,W] volumes, their squares and
// running sums (~30 passes over 1.18 GB tensors), one kernel gathers the
// bilinear taps of the k neighbours and writes the variance once.
//
// Work decomposition.  Features are channels-last ([V,H,W,C]), so a bilinear
// tap is a contiguous C-vector.  A warp owns one pixel of one reference view
// for a slice of 128*G channels (lane l <-> channels slice*128G + 128g + 4l..+3
// for g < G: 16-byte vectors, every request a coalesced 512 bytes) and walks
// the D planes; the reference vector stays in registers for all planes.
//   * The sample geometry (homography, divides, floor, tap weights) is
//     warp-uniform; it is computed ONCE per (pixel, plane, neighbour) with one
//     lane per sample -- 32 samples per pass -- parked in shared memory as
//     pre-multiplied 32-bit element offsets plus four weights, and re-read as a
//     broadcast: the inner loop is one IMAD.WIDE per tap address, vector loads
//     and FMAs.
//   * The 8 warps of a CTA cover a 4x2 pixel patch, so the bilinear overlap of
//     neighbouring pixels is served by L1, the rest by L2 (the whole feature
//     tensor, 49-98 MB, is L2-resident on B200's 126 MB L2).
//   * The variance is written once with evict-first streaming stores.
// A run-based variant (8-pixel runs with a register tap-column cache and
// merged REDs) was measured slower on B200 (register pressure -> 8 warps/SM,
// see DESIGN.md "what was tried"); it is in the git history.
//
// HBM-bound by design (SURVEY.md section 0): no contraction, no tensor cores.
#pragma once
#include "common.cuh"

namespace mvsd {

constexpr int kSweepWarps = 8;
constexpr int kSweepThreads = kSweepWarps * 32;
constexpr int kPatchW = 4, kPatchH = 2;    // pixel patch of a CTA (one warp per pixel)
constexpr int kSlots = 32;                 // sample slots per geometry pass (one per lane)

struct SweepParams {
  const void* feat;        // nhwc features
  const int32_t* nbr;      // [V,k] or nullptr (warp-only: source = same index)
  const float* hom;        // [V,k,12]
  const float* depth;      // [V,D], or [V,D,H,W] when depth_per_pixel
  void* out;               // fwd output [V,D,H,W,C]
  const void* g_out;       // bwd upstream gradient, same layout
  float* g_feat;           // bwd: nhwc fp32, accumulated with RED
  long long* g_feat_q;     // bwd, deterministic form: nhwc 64-bit fixed point (common.cuh), integer REDs
  int V, C, D, H, W, k;
  int ref_begin;           // feat index of reference view 0 (view sharding)
  int n_feat;              // views held by feat: neighbour ids outside [0, n_feat) give no sample
  int depth_per_pixel;     // homo_warping's [B,D,H,W] depth_values branch (module.py:130-133)
  int tiles_x, tiles_y, slices;
  // group-wise correlation backward through the run kernel (group_corr.cu): g_out is the gradient of the
  // cost volumes [V,k,D,H,W,corr_groups]; a channel's group is channel >> corr_cg_shift
  int corr_groups, corr_cg_shift;
  float corr_inv_cg;
};

struct SweepCoord {
  int v, x, y, c0;
  bool ok;
};

template <int G>
__device__ __forceinline__ SweepCoord sweep_coord(const SweepParams& p, int warp, int lane) {
  SweepCoord c;
  int t = blockIdx.x;
  const int tx = t % p.tiles_x; t /= p.tiles_x;
  const int ty = t % p.tiles_y; t /= p.tiles_y;
  const int slice = t % p.slices;
  c.v = t / p.slices;
  c.x = tx * kPatchW + (warp % kPatchW);
  c.y = ty * kPatchH + (warp / kPatchW);
  c.ok = c.x < p.W && c.y < p.H;
  c.c0 = slice * 128 * G + 4 * lane;
  return c;
}

// A neighbour id outside the feature tensor (stale or un-rebased ids against a compact / sliced
// buffer) must neither be read nor -- in the backward -- be the target of a RED: such a
// neighbour simply contributes no sample, like a warp that lands outside the map.  The lane that
// computes a sample loads its neighbour's id TOGETHER with the homography (independent loads, one
// wait) and replaces the plane depth by NaN when the id is unusable: q = r * NaN + t is NaN ->
// "no sample" through the code path that already exists.  One select, no branch on the loaded id
// (a branch serialised the loads and cost the forward 6 %; a mask handed over through shared
// memory put the id load in front of the fill, same cost).
__device__ __forceinline__ int nbr_id_for_check(const SweepParams& p, int v, int j) {
  return p.nbr ? __ldg(p.nbr + (size_t)v * p.k + j) : 0;      // stand-alone warp: no ids, always usable
}
__device__ __forceinline__ float depth_or_nan(float depth, int n, int n_feat) {
  return (unsigned)n < (unsigned)n_feat ? depth : __int_as_float(0x7fc00000);
}

// Depth of plane d at pixel (x, y) of reference view v: the per-view planes [V,D], or with
// PER_PIXEL_DEPTH homo_warping's per-pixel hypotheses [V,D,H,W] (module.py:130-133).
template <bool PER_PIXEL_DEPTH>
__device__ __forceinline__ float plane_depth(const SweepParams& p, int v, int d, int x, int y) {
  const size_t di = (size_t)v * p.D + d;
  return PER_PIXEL_DEPTH ? __ldg(p.depth + (di * p.H + y) * p.W + x) : __ldg(p.depth + di);
}

// Which depth_values form a kernel's fill reads.  The fused kernels are compiled per form (the
// per-pixel ones serve the *_px entry points): as a run-time select inside the per-view kernels'
// fill it cost the forward sweep 6 % (measured: 0.291 vs 0.273 ms).  Only the stand-alone warp
// selects at run time, from p.depth_per_pixel.
enum DepthForm { kDepthPlanes, kDepthPixels, kDepthEither };

// One pass of sample geometry for this warp's pixel: lane s computes the sample
// of (plane d0 + s / k, neighbour s % k).
template <int DEPTH = kDepthPlanes>
__device__ __forceinline__ void fill_samples(WarpSample* tab, const SweepParams& p,
                                             const SweepCoord& c, int d0, int dc, int lane) {
  const int k = p.k;
  if (lane < dc * k) {
    const int dd = lane / k, j = lane - dd * k;
    const int d = d0 + dd;
    WarpSample s;
    s.w00 = s.w01 = s.w10 = s.w11 = 0.f;
    s.p00 = s.p01 = s.p10 = s.p11 = kNoSample;
    if (d < p.D) {
      const float* m = p.hom + ((size_t)c.v * k + j) * 12;
      const int n = nbr_id_for_check(p, c.v, j);
      float mm[12];
#pragma unroll
      for (int t = 0; t < 12; ++t) mm[t] = __ldg(m + t);
      const size_t di = (size_t)c.v * p.D + d;
      const bool per_pixel = DEPTH == kDepthPixels || (DEPTH == kDepthEither && p.depth_per_pixel);
      const float depth = per_pixel ? __ldg(p.depth + (di * p.H + c.y) * p.W + c.x) : __ldg(p.depth + di);
      s = make_warp_sample(mm, (float)c.x, (float)c.y, depth_or_nan(depth, n, p.n_feat), p.H, p.W, p.C);
    }
    tab[lane] = s;
  }
}

__device__ __forceinline__ float4 f4zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4scale(float4 a, float s) {
  return make_float4(a.x * s, a.y * s, a.z * s, a.w * s);
}
__device__ __forceinline__ float4 f4add(float4 a, float4 b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float4 f4sub(float4 a, float4 b) {
  return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w);
}
__device__ __forceinline__ float4 f4mul(float4 a, float4 b) {
  return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w);
}
__device__ __forceinline__ float4 f4fma(float4 a, float s, float4 c) {
  return make_float4(fmaf(a.x, s, c.x), fmaf(a.y, s, c.y), fmaf(a.z, s, c.z), fmaf(a.w, s, c.w));
}
__device__ __forceinline__ float4 f4fma(float4 a, float4 b, float4 c) {
  return make_float4(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z),
                     fmaf(a.w, b.w, c.w));
}

// ---- packed fp32 pairs (sm_100 FFMA2 / FMUL2 / FADD2) -----------------------
// ncu shows both sweep kernels bound by instruction issue (fwd: 81% issue-active),
// not by a memory pipe; Blackwell's f32x2 arithmetic halves the math instruction
// count.  Each lane's 4 channels live in two 64-bit register pairs.  Same fp32
// rounding per element as the scalar ops (fma.rn / mul.rn / add.rn).
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float a, float b) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void upk2(u64 v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
  u64 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
  u64 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
  u64 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ u64 sub2(u64 a, u64 b) {
  u64 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

struct P4 {               // 4 consecutive channels as two f32x2 pairs
  u64 lo, hi;
};
__device__ __forceinline__ P4 p4zero() { return P4{0ull, 0ull}; }
__device__ __forceinline__ P4 p4from(float4 v) { return P4{pk2(v.x, v.y), pk2(v.z, v.w)}; }
__device__ __forceinline__ P4 p4from(uint2 r) {       // 4 x bf16
  return P4{pk2(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u)),
            pk2(__uint_as_float(r.y << 16), __uint_as_float(r.y & 0xffff0000u))};
}
__device__ __forceinline__ float4 p4to(P4 a) {
  float4 v;
  upk2(a.lo, v.x, v.y);
  upk2(a.hi, v.z, v.w);
  return v;
}
__device__ __forceinline__ P4 p4scale(P4 a, u64 s) { return P4{mul2(a.lo, s), mul2(a.hi, s)}; }
__device__ __forceinline__ P4 p4add(P4 a, P4 b) { return P4{add2(a.lo, b.lo), add2(a.hi, b.hi)}; }
__device__ __forceinline__ P4 p4sub(P4 a, P4 b) { return P4{sub2(a.lo, b.lo), sub2(a.hi, b.hi)}; }
__device__ __forceinline__ P4 p4mul(P4 a, P4 b) { return P4{mul2(a.lo, b.lo), mul2(a.hi, b.hi)}; }
__device__ __forceinline__ P4 p4fma(P4 a, u64 s, P4 c) {
  return P4{fma2(a.lo, s, c.lo), fma2(a.hi, s, c.hi)};
}
__device__ __forceinline__ P4 p4fma(P4 a, P4 b, P4 c) {
  return P4{fma2(a.lo, b.lo, c.lo), fma2(a.hi, b.hi, c.hi)};
}

// ---- tensor memory as a warp-private fp32 accumulator file --------------------
// 32x32b shape: lane l of warp w touches TMEM lane 32*(w%4)+l, 4 consecutive
// columns per access; the column index is a run-time value.  Used for per-pixel
// gradient accumulators that must persist across the plane loop (512 B per pixel
// per 128 channels) without costing registers or shared memory (= L1 capacity).
// tools/tmem_probe.cu verifies this usage on the GPU.
__device__ __forceinline__ void tmem_st4(uint32_t taddr, P4 v) {
  float a, b, c, d;
  upk2(v.lo, a, b);
  upk2(v.hi, c, d);
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               :: "r"(taddr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ P4 tmem_ld4(uint32_t taddr) {
  float a, b, c, d;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=f"(a), "=f"(b), "=f"(c), "=f"(d) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  return P4{pk2(a, b), pk2(c, d)};
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// One warp allocates COLS columns for the CTA and publishes the base through smem;
// every thread of the CTA must call both functions (they contain CTA barriers).
template <int COLS>
__device__ __forceinline__ uint32_t tmem_alloc_cta(uint32_t* s_base, int warp) {
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"((uint32_t)__cvta_generic_to_shared(s_base)), "n"(COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  return *s_base + ((uint32_t)((warp & 3) * 32) << 16);     // this warp's lane quarter
}
template <int COLS>
__device__ __forceinline__ void tmem_free_cta(uint32_t* s_base, int warp) {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(*s_base), "n"(COLS) : "memory");
}

// raw (un-converted) 4-channel loads, so the bf16 -> fp32 shift/mask lands next
// to the packed arithmetic that consumes it
template <typename T> struct Raw;
template <> struct Raw<float> {
  typedef float4 type;
  static __device__ __forceinline__ float4 ld(const float* p) {
    return __ldg(reinterpret_cast<const float4*>(p));
  }
  static __device__ __forceinline__ float4 ld_stream(const float* p) {
    return __ldcs(reinterpret_cast<const float4*>(p));
  }
  // read-once stream that must not displace the gathered taps from L1
  static __device__ __forceinline__ float4 ld_stream_na(const float* p) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
  }
  static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
};
template <> struct Raw<__nv_bfloat16> {
  typedef uint2 type;
  static __device__ __forceinline__ uint2 ld(const __nv_bfloat16* p) {
    return __ldg(reinterpret_cast<const uint2*>(p));
  }
  static __device__ __forceinline__ uint2 ld_stream(const __nv_bfloat16* p) {
    return __ldcs(reinterpret_cast<const uint2*>(p));
  }
  static __device__ __forceinline__ uint2 ld_stream_na(const __nv_bfloat16* p) {
    uint2 v;
    asm volatile("ld.global.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    return v;
  }
  static __device__ __forceinline__ uint2 zero() { return make_uint2(0u, 0u); }
};

// 64-bit address = base + 32-bit unsigned element offset: one IMAD.WIDE.U32.
template <typename T>
__device__ __forceinline__ const T* at(const T* base, unsigned off) {
  return reinterpret_cast<const T*>(reinterpret_cast<const char*>(base) +
                                    (unsigned long long)off * sizeof(T));
}
template <typename T>
__device__ __forceinline__ T* at(T* base, unsigned off) {
  return reinterpret_cast<T*>(reinterpret_cast<char*>(base) + (unsigned long long)off * sizeof(T));
}

// lane-activity of channel group g of this warp's slice
template <bool FULL>
__device__ __forceinline__ bool group_on(int c0, int g, int C) {
  return FULL || (c0 + 128 * g < C);
}

// The bilinear sample of one neighbour: nw*w00 + ne*w01 + sw*w10 + se*w11, the
// order ATen's sampler uses.  All 4*G loads are issued before the first FMA.
template <typename TIn, int G, bool FULL>
__device__ __forceinline__ void gather_taps(const TIn* __restrict__ src, const WarpSample& s,
                                            int c0, int C, float4 (&wv)[G]) {
  const TIn* a00 = at(src, s.p00);
  const TIn* a01 = at(src, s.p01);
  const TIn* a10 = at(src, s.p10);
  const TIn* a11 = at(src, s.p11);
  float4 t00[G], t01[G], t10[G], t11[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    if (group_on<FULL>(c0, g, C)) {
      t00[g] = Io<TIn>::ld(a00 + 128 * g);
      t01[g] = Io<TIn>::ld(a01 + 128 * g);
      t10[g] = Io<TIn>::ld(a10 + 128 * g);
      t11[g] = Io<TIn>::ld(a11 + 128 * g);
    } else {
      t00[g] = t01[g] = t10[g] = t11[g] = f4zero();
    }
  }
#pragma unroll
  for (int g = 0; g < G; ++g) {
    float4 w = f4scale(t00[g], s.w00);
    w = f4fma(t01[g], s.w01, w);
    w = f4fma(t10[g], s.w10, w);
    wv[g] = f4fma(t11[g], s.w11, w);
  }
}

// Packed variant of gather_taps: same tap order, FMUL2 / FFMA2.
template <typename TIn, int G, bool FULL>
__device__ __forceinline__ void gather_taps_p(const TIn* __restrict__ src, const WarpSample& s,
                                              int c0, int C, P4 (&wv)[G]) {
  const TIn* a00 = at(src, s.p00);
  const TIn* a01 = at(src, s.p01);
  const TIn* a10 = at(src, s.p10);
  const TIn* a11 = at(src, s.p11);
  typename Raw<TIn>::type t00[G], t01[G], t10[G], t11[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    if (group_on<FULL>(c0, g, C)) {
      t00[g] = Raw<TIn>::ld(a00 + 128 * g);
      t01[g] = Raw<TIn>::ld(a01 + 128 * g);
      t10[g] = Raw<TIn>::ld(a10 + 128 * g);
      t11[g] = Raw<TIn>::ld(a11 + 128 * g);
    } else {
      t00[g] = t01[g] = t10[g] = t11[g] = Raw<TIn>::zero();
    }
  }
  const u64 w00 = pk2(s.w00, s.w00), w01 = pk2(s.w01, s.w01);
  const u64 w10 = pk2(s.w10, s.w10), w11 = pk2(s.w11, s.w11);
#pragma unroll
  for (int g = 0; g < G; ++g) {
    P4 w = p4scale(p4from(t00[g]), w00);
    w = p4fma(p4from(t01[g]), w01, w);
    w = p4fma(p4from(t10[g]), w10, w);
    wv[g] = p4fma(p4from(t11[g]), w11, w);
  }
}

// Split form of gather_taps_p: issue the 4*G loads of a sample (no use), blend
// later -- lets a kernel put the loads of BOTH neighbours (and of the next pixel)
// in flight before the first dependent instruction.  ncu on the fused kernels
// showed ~3 serialized L2 round trips per pixel (long-scoreboard 4.5 / issue).
template <typename TIn, int G>
struct RawTaps {
  typename Raw<TIn>::type t00[G], t01[G], t10[G], t11[G];
};
template <typename TIn, int G, bool FULL>
__device__ __forceinline__ void load_taps(const TIn* __restrict__ src, const WarpSample& s, int c0,
                                          int C, RawTaps<TIn, G>& r) {
  const TIn* a00 = at(src, s.p00);
  const TIn* a01 = at(src, s.p01);
  const TIn* a10 = at(src, s.p10);
  const TIn* a11 = at(src, s.p11);
#pragma unroll
  for (int g = 0; g < G; ++g) {
    if (group_on<FULL>(c0, g, C)) {
      r.t00[g] = Raw<TIn>::ld(a00 + 128 * g);
      r.t01[g] = Raw<TIn>::ld(a01 + 128 * g);
      r.t10[g] = Raw<TIn>::ld(a10 + 128 * g);
      r.t11[g] = Raw<TIn>::ld(a11 + 128 * g);
    } else {
      r.t00[g] = r.t01[g] = r.t10[g] = r.t11[g] = Raw<TIn>::zero();
    }
  }
}
template <typename TIn, int G>
__device__ __forceinline__ void blend_taps(const RawTaps<TIn, G>& r, const WarpSample& s, P4 (&wv)[G]) {
  const u64 w00 = pk2(s.w00, s.w00), w01 = pk2(s.w01, s.w01);
  const u64 w10 = pk2(s.w10, s.w10), w11 = pk2(s.w11, s.w11);
#pragma unroll
  for (int g = 0; g < G; ++g) {
    P4 w = p4scale(p4from(r.t00[g]), w00);
    w = p4fma(p4from(r.t01[g]), w01, w);
    w = p4fma(p4from(r.t10[g]), w10, w);
    wv[g] = p4fma(p4from(r.t11[g]), w11, w);
  }
}

// host-side helpers shared by the two translation units
int sweep_check(const char* who, int V, int C, int D, int H, int W, int k, int layout);
bool sweep_grid(SweepParams& p, int G, dim3& grid);
int sweep_groups(int C);

}  // namespace mvsd
