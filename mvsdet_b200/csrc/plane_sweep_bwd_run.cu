// Plane-sweep backward, run-merging kernels (the product backward for k in {1, 2}).
//
// ncu on the pixel-per-warp backward (plane_sweep_bwd.cu, kept as the generic fallback)
// shows it bound by RED traffic leaving the SM: every (pixel, plane, neighbour) emits four
// 1 KB vector REDs (5.46 GB per scene against a measured 5.7 TB/s ceiling).  Here a warp
// walks a horizontal run of kRun pixels of one row (planes in the outer loop) and keeps the
// contribution to the RIGHT tap column pending in registers: when the next pixel's LEFT
// column is the same source pixel (source position advanced by exactly one -- the common
// case between pose-space neighbours) the two contributions leave as ONE RED; when the
// source position did not advance the right column absorbs the next one.  The four warps
// of a CTA own four consecutive rows and hand the shared tap row to each other through a
// shared-memory queue (sweep_bwd_runs).  RED payload 5.46 -> 3.61 (columns) -> 2.71 GB.
// The per-pixel reference gradient (a sum over planes) lives in tensor memory.
//
// Two kernels are built, one per feature dtype:
//   sweep_bwd_runs   row hand-off + software-pipelined loads; bf16 features
//   sweep_bwd_runq   lean column-merging kernel without hand-off; fp32 features
//                    (the pipelined kernel spills with 80 raw-load registers per pixel)
// The measured-and-dropped variants (scalar math, shared-memory accumulators, block / row-block
// merging, deeper queues, L1 prefetch, pending taps in TMEM at 4 CTAs/SM, 128-channel warps at
// 4-5 CTAs/SM, producer / consumer warp specialisation over a shared-memory ring) are in the git
// history, DESIGN.md section 5/8 and profiles/r02_bwd_experiments.md; they are not shipped.
#include "plane_sweep.cuh"

namespace mvsd {

constexpr int kRun = 8;                    // pixels per warp run
constexpr int kRunQMinBlocks = 3;          // CTAs per SM the kernels are compiled for (168 registers)
constexpr int kRunRows = 4;                // rows (= warps) per CTA
constexpr int kRunThreads = kRunRows * 32;
constexpr unsigned kNoTap = 0xfffffffeu;   // "nothing pending"

struct RunCoord {
  int v, y, x0, npix, c0;
};

template <int G>
__device__ __forceinline__ RunCoord run_coord(const SweepParams& p, int warp, int lane) {
  RunCoord c;
  int t = blockIdx.x;
  const int xr = t % p.tiles_x; t /= p.tiles_x;
  const int yt = t % p.tiles_y; t /= p.tiles_y;
  const int slice = t % p.slices;
  c.v = t / p.slices;
  c.y = yt * kRunRows + warp;
  c.x0 = xr * kRun;
  c.npix = min(kRun, p.W - c.x0);
  c.c0 = slice * 128 * G + 4 * lane;
  return c;
}

// lane s -> sample (plane d0 + s / (kRun*k), pixel x0 + (s % (kRun*k)) / k, neighbour s % k)
// PX: per-pixel depth hypotheses [V,D,H,W] (the *_px entry points), in every run kernel below
template <bool PX>
__device__ __forceinline__ void fill_run_samples(WarpSample* tab, const SweepParams& p,
                                                 const RunCoord& c, int d0, int ppf, int lane) {
  const int k = p.k, spp = kRun * k;
  if (lane < ppf * spp) {
    const int dd = lane / spp, rem = lane - dd * spp;
    const int i = rem / k, j = rem - i * k;
    const int d = d0 + dd;
    WarpSample s;
    s.w00 = s.w01 = s.w10 = s.w11 = 0.f;
    s.p00 = s.p01 = s.p10 = s.p11 = kNoSample;
    if (d < p.D && i < c.npix) {
      const float* m = p.hom + ((size_t)c.v * k + j) * 12;
      const int n = nbr_id_for_check(p, c.v, j);
      float mm[12];
#pragma unroll
      for (int t = 0; t < 12; ++t) mm[t] = __ldg(m + t);
      s = make_warp_sample(mm, (float)(c.x0 + i), (float)c.y,
                           depth_or_nan(plane_depth<PX>(p, c.v, d, c.x0 + i, c.y), n, p.n_feat), p.H, p.W, p.C);
    }
    tab[lane] = s;
  }
}


__device__ __forceinline__ void red_add_p4(float* p, P4 v) {
  float a, b, c, d;
  upk2(v.lo, a, b);
  upk2(v.hi, c, d);
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};"
               :: "l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__device__ __forceinline__ void prefetch_l2(const void* p, unsigned bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(p), "r"(bytes) : "memory");
}

template <int G, bool FULL>
__device__ __forceinline__ void red_group_p(float* dst, unsigned off, const P4 (&v)[G], int c0,
                                            int C) {
  float* a = at(dst, off);
#pragma unroll
  for (int g = 0; g < G; ++g)
    if (group_on<FULL>(c0, g, C)) red_add_p4(a + 128 * g, v[g]);
}

template <int G, bool FULL>
__device__ __forceinline__ void flush_open_p(float* dst, unsigned& id, const P4 (&acc)[G], int c0,
                                             int C) {
  if (id != kNoTap) red_group_p<G, FULL>(dst, id, acc, c0, C);
  id = kNoTap;
}

constexpr int kPrefetchPlanes = 2;

// ---------------------------------------------------------------------------
// Lean kernel.  ncu's per-instruction counts on the first packed run kernel: 335 warp instructions per pixel-plane of which 81 are register moves
// (MOV / IMAD.MOV / CS2R at the joins of "zero, then blend if the sample is valid" and of
// the merge-or-flush branches) and 63 are control flow.  Same algorithm, restructured so
// that nothing is merged at a join:
//   * the pixel body is instantiated per validity pattern of the two samples (a
//     warp-uniform 4-way branch): an absent sample has no loads, no blend, no zeroed
//     vector and leaves the pending taps alone (a later mismatch or the end of the run
//     flushes them);
//   * the scatter keeps one invariant -- "the pending accumulator is zero unless it
//     matches the next left tap" -- so the mismatch arm only issues a RED and zeroes the
//     pending registers in place, and the left tap is always fma(gw, w_left, pending).
// ---------------------------------------------------------------------------
template <int KMAX, int G>
struct RunPending {
  P4 top[KMAX][G], bot[KMAX][G];
  unsigned id_top[KMAX], id_bot[KMAX];
};

template <int G, bool FULL>
__device__ __forceinline__ void side_q(float* dst, const P4 (&gw)[G], float w_left, float w_right,
                                       unsigned p_left, unsigned p_right, unsigned& open_id,
                                       P4 (&open)[G], int c0, int C) {
  const u64 wl = pk2(w_left, w_left), wr = pk2(w_right, w_right);
  P4 a[G];
  if (open_id == p_left) {                 // source x advanced by one: pending + left leave as one RED
#pragma unroll
    for (int g = 0; g < G; ++g) a[g] = p4fma(gw[g], wl, open[g]);
    red_group_p<G, FULL>(dst, p_left, a, c0, C);
#pragma unroll
    for (int g = 0; g < G; ++g) open[g] = p4scale(gw[g], wr);
    open_id = w_right != 0.f ? p_right : kNoTap;
  } else if (open_id == p_right && w_right != 0.f) {   // source x did not advance: right joins the pending tap
#pragma unroll
    for (int g = 0; g < G; ++g) open[g] = p4fma(gw[g], wr, open[g]);
    if (w_left != 0.f) {
#pragma unroll
      for (int g = 0; g < G; ++g) a[g] = p4scale(gw[g], wl);
      red_group_p<G, FULL>(dst, p_left, a, c0, C);
    }
  } else {
    if (open_id != kNoTap) red_group_p<G, FULL>(dst, open_id, open, c0, C);
    if (w_left != 0.f) {
#pragma unroll
      for (int g = 0; g < G; ++g) a[g] = p4scale(gw[g], wl);
      red_group_p<G, FULL>(dst, p_left, a, c0, C);
    }
#pragma unroll
    for (int g = 0; g < G; ++g) open[g] = p4scale(gw[g], wr);
    open_id = w_right != 0.f ? p_right : kNoTap;
  }
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned long long* b, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(b)), "r"(count) : "memory");
}
// side_q for pre-weighted contributions (left / right vectors), used by the receiving
// side of a hand-off.
template <int G, bool FULL>
__device__ __forceinline__ void side_c(float* dst, const P4 (&cl)[G], const P4 (&cr)[G], bool nz_left,
                                       bool nz_right, unsigned p_left, unsigned p_right,
                                       unsigned& open_id, P4 (&open)[G], int c0, int C) {
  P4 a[G];
  if (open_id == p_left) {
#pragma unroll
    for (int g = 0; g < G; ++g) a[g] = p4add(cl[g], open[g]);
    red_group_p<G, FULL>(dst, p_left, a, c0, C);
#pragma unroll
    for (int g = 0; g < G; ++g) open[g] = cr[g];
    open_id = nz_right ? p_right : kNoTap;
  } else if (open_id == p_right && nz_right) {
#pragma unroll
    for (int g = 0; g < G; ++g) open[g] = p4add(cr[g], open[g]);
    if (nz_left) red_group_p<G, FULL>(dst, p_left, cl, c0, C);
  } else {
    if (open_id != kNoTap) red_group_p<G, FULL>(dst, open_id, open, c0, C);
    if (nz_left) red_group_p<G, FULL>(dst, p_left, cl, c0, C);
#pragma unroll
    for (int g = 0; g < G; ++g) open[g] = cr[g];
    open_id = nz_right ? p_right : kNoTap;
  }
}

template <typename TIn, typename TG, int KMAX, int G, bool FULL, bool V0, bool V1>
__device__ __forceinline__ void pixel_q(RunPending<KMAX, G>& pend, const WarpSample& s0,
                                        const WarpSample& s1, const TG* __restrict__ gp,
                                        const TIn* __restrict__ rp, const TIn* const (&nsrc)[KMAX],
                                        float* const (&ndst)[KMAX], uint32_t taddr, u64 inv_n2,
                                        u64 two_inv_n2, int c0, int C) {
  typename Raw<TG>::type graw[G];
  typename Raw<TIn>::type rraw[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const bool on = group_on<FULL>(c0, g, C);
    graw[g] = on ? Raw<TG>::ld_stream_na(gp + 128 * g) : Raw<TG>::zero();
    rraw[g] = on ? Raw<TIn>::ld(rp + 128 * g) : Raw<TIn>::zero();
  }
  RawTaps<TIn, G> t0, t1;
  if (V0) load_taps<TIn, G, FULL>(nsrc[0], s0, c0, C, t0);
  if (V1) load_taps<TIn, G, FULL>(nsrc[KMAX - 1], s1, c0, C, t1);
  P4 w0[G], w1[G], gw0[G], gw1[G];
  if (V0) blend_taps<TIn, G>(t0, s0, w0);
  if (V1) blend_taps<TIn, G>(t1, s1, w1);
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const P4 ref = p4from(rraw[g]);
    P4 mu = ref;
    if (V0) mu = p4add(mu, w0[g]);
    if (V1) mu = p4add(mu, w1[g]);
    mu = p4scale(mu, inv_n2);
    const P4 gv = p4scale(p4from(graw[g]), two_inv_n2);
    const uint32_t ta = taddr + 4u * (uint32_t)g;
    tmem_st4(ta, p4fma(gv, p4sub(ref, mu), tmem_ld4(ta)));
    if (V0) gw0[g] = p4mul(gv, p4sub(w0[g], mu));
    if (V1) gw1[g] = p4mul(gv, p4sub(w1[g], mu));
  }
  if (V0) {
    side_q<G, FULL>(ndst[0], gw0, s0.w00, s0.w01, s0.p00, s0.p01, pend.id_top[0], pend.top[0], c0, C);
    side_q<G, FULL>(ndst[0], gw0, s0.w10, s0.w11, s0.p10, s0.p11, pend.id_bot[0], pend.bot[0], c0, C);
  }
  if (V1) {
    constexpr int J = KMAX - 1;
    side_q<G, FULL>(ndst[J], gw1, s1.w00, s1.w01, s1.p00, s1.p01, pend.id_top[J], pend.top[J], c0, C);
    side_q<G, FULL>(ndst[J], gw1, s1.w10, s1.w11, s1.p10, s1.p11, pend.id_bot[J], pend.bot[J], c0, C);
  }
}

// requires p.k == KMAX (the launcher instantiates KMAX = k for k in {1, 2})
template <typename TIn, typename TG, int KMAX, int G, bool FULL, int MINB, bool PX = false>
__global__ void __launch_bounds__(kRunThreads, MINB) sweep_bwd_runq_kernel(const SweepParams p) {
  constexpr int kCols = kRun * G * 4;
  __shared__ WarpSample s_tab[kRunRows][32];
  __shared__ uint32_t s_tmem;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const RunCoord c = run_coord<G>(p, warp, lane);
  const uint32_t tbase = tmem_alloc_cta<kCols>(&s_tmem, warp);
  if (c.y < p.H) {
    const int C = p.C, HW = p.H * p.W;
    const TIn* feat = static_cast<const TIn*>(p.feat);
    const size_t ref_off = ((size_t)(c.v + p.ref_begin) * HW + (size_t)c.y * p.W + c.x0) * C + c.c0;
    const TIn* ref_row = feat + ref_off;
    const size_t plane_stride = (size_t)HW * C;
    const TG* g_d = static_cast<const TG*>(p.g_out) + ((size_t)c.v * p.D * HW + (size_t)c.y * p.W + c.x0) * C + c.c0;
    const bool one_chunk = p.slices == 1;
    const unsigned pf_bytes = (unsigned)((one_chunk ? (size_t)c.npix * C : (size_t)min(128 * G, C - (c.c0 - 4 * lane))) *
                                         sizeof(TG)) & ~15u;
    const TG* pf_base = g_d - 4 * lane;
    const bool pf_ok = pf_bytes >= 16 && (reinterpret_cast<uintptr_t>(pf_base) & 15) == 0 &&
                       ((plane_stride * sizeof(TG)) & 15) == 0;
    auto prefetch_plane = [&](int d) {
      if (!pf_ok || d >= p.D) return;
      const TG* q = pf_base + (size_t)d * plane_stride;
      if (one_chunk) {
        if (lane == 0) prefetch_l2(q, pf_bytes);
      } else if (lane < c.npix) {
        prefetch_l2(q + (size_t)lane * C, pf_bytes);
      }
    };
#pragma unroll
    for (int d = 0; d < kPrefetchPlanes; ++d) prefetch_plane(d);

    const TIn* nsrc[KMAX];
    float* ndst[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
      const int n = __ldg(p.nbr + (size_t)c.v * KMAX + j);
      nsrc[j] = feat + (size_t)n * HW * C + c.c0;
      ndst[j] = p.g_feat + (size_t)n * HW * C + c.c0;
      asm volatile("" : "+l"(nsrc[j]), "+l"(ndst[j]));
    }
    const float inv_n = 1.0f / (float)(KMAX + 1);
    const u64 inv_n2 = pk2(inv_n, inv_n);
    const u64 two_inv_n2 = pk2(2.0f * inv_n, 2.0f * inv_n);
    constexpr int spp = kRun * KMAX;
    constexpr int ppf = 32 / spp > 0 ? 32 / spp : 1;

#pragma unroll
    for (int q = 0; q < kRun * G; ++q) tmem_st4(tbase + 4u * (uint32_t)q, p4zero());
    tmem_wait_st();

    for (int d0 = 0; d0 < p.D; d0 += ppf) {
      __syncwarp();
      fill_run_samples<PX>(s_tab[warp], p, c, d0, ppf, lane);
      __syncwarp();
      const int dend = min(p.D, d0 + ppf);
      for (int d = d0; d < dend; ++d) {
        prefetch_plane(d + kPrefetchPlanes);
        tmem_wait_st();
        RunPending<KMAX, G> pend;
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
          pend.id_top[j] = pend.id_bot[j] = kNoTap;
#pragma unroll
          for (int g = 0; g < G; ++g) pend.top[j][g] = pend.bot[j][g] = p4zero();
        }
        const WarpSample* tab = s_tab[warp] + (d - d0) * spp;
#pragma unroll 1
        for (int i = 0; i < c.npix; ++i) {
          const WarpSample s0 = tab[i * KMAX];
          const WarpSample s1 = tab[i * KMAX + (KMAX - 1)];
          const bool v0 = s0.p00 != kNoSample;
          const bool v1 = KMAX == 2 && s1.p00 != kNoSample;
          const TG* gp = g_d + i * C;
          const TIn* rp = ref_row + i * C;
          const uint32_t ta = tbase + 4u * (uint32_t)(i * G);
          if (v0 && v1)
            pixel_q<TIn, TG, KMAX, G, FULL, true, true>(pend, s0, s1, gp, rp, nsrc, ndst, ta, inv_n2, two_inv_n2, c.c0, C);
          else if (v0)
            pixel_q<TIn, TG, KMAX, G, FULL, true, false>(pend, s0, s1, gp, rp, nsrc, ndst, ta, inv_n2, two_inv_n2, c.c0, C);
          else if (v1)
            pixel_q<TIn, TG, KMAX, G, FULL, false, true>(pend, s0, s1, gp, rp, nsrc, ndst, ta, inv_n2, two_inv_n2, c.c0, C);
          else
            pixel_q<TIn, TG, KMAX, G, FULL, false, false>(pend, s0, s1, gp, rp, nsrc, ndst, ta, inv_n2, two_inv_n2, c.c0, C);
        }
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
          flush_open_p<G, FULL>(ndst[j], pend.id_top[j], pend.top[j], c.c0, C);
          flush_open_p<G, FULL>(ndst[j], pend.id_bot[j], pend.bot[j], c.c0, C);
        }
        g_d += plane_stride;
      }
    }
    tmem_wait_st();
    float* dst = p.g_feat + ref_off;
    for (int i = 0; i < c.npix; ++i) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const P4 acc = tmem_ld4(tbase + 4u * (uint32_t)(i * G + g));
        if (group_on<FULL>(c.c0, g, C)) red_add_p4(dst + i * C + 128 * g, acc);
      }
    }
  }
  tmem_free_cta<kCols>(&s_tmem, warp);
}

// ---------------------------------------------------------------------------
// Software-pipelined loads.  ncu's per-warp picture of the lean kernel: ~2260 cycles per
// pixel-plane = one L2 round trip for the 20 loads of the pixel (all issued together, ~1000+
// cycles under the RED traffic) followed by ~240 dependent-ish instructions at ~4 cycles each,
// with only 3 warps per scheduler to overlap the two.  An L1 prefetch of the next pixel hides
// the round trip but doubles the L1 tag traffic and is slower (measured twice).  Instead the
// loads of the NEXT pixel are issued into the raw-load registers as soon as the blend has
// consumed the current ones, i.e. before the variance algebra, the tensor-memory update and
// the scatter: the same registers, no extra L1 traffic.
// ---------------------------------------------------------------------------
template <typename TIn, typename TG, int G>
struct PixelRaw {
  typename Raw<TG>::type g[G];
  typename Raw<TIn>::type r[G];
  RawTaps<TIn, G> t0, t1;
};

// MODE 0: variance backward, gp -> this pixel-plane's dL/dvariance vector.  MODE 1: group-wise
// correlation backward (group_corr.cu), gp -> the pixel-plane's corr_groups gradients of neighbour 0
// (neighbour 1 is corr_nstride floats further); the lane's 2 x G group values travel in raw.g[0] as
// (nbr 0 group of g = 0, g = 1, nbr 1 group of g = 0, g = 1), already divided by the group width.
template <typename TIn, typename TG, int KMAX, int G, bool FULL, int MODE>
__device__ __forceinline__ void issue_pixel_loads(PixelRaw<TIn, TG, G>& raw, const WarpSample* smp,
                                                  const TG* __restrict__ gp, const TIn* __restrict__ rp,
                                                  const TIn* const (&nsrc)[KMAX], int c0, int C,
                                                  const SweepParams& p) {
  if constexpr (MODE == 1) {
    const size_t nstride = (size_t)p.D * p.H * p.W * p.corr_groups;
    const float* gq = reinterpret_cast<const float*>(gp);
    float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const bool on = group_on<FULL>(c0, g, C);
      raw.r[g] = on ? Raw<TIn>::ld(rp + 128 * g) : Raw<TIn>::zero();
      if (on) {
        const int grp = (c0 + 128 * g) >> p.corr_cg_shift;
        v[g] = __ldg(gq + grp) * p.corr_inv_cg;
        v[2 + g] = __ldg(gq + nstride + grp) * p.corr_inv_cg;
      }
    }
    raw.g[0] = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int g = 0; g < G; ++g) {
      const bool on = group_on<FULL>(c0, g, C);
      raw.g[g] = on ? Raw<TG>::ld_stream_na(gp + 128 * g) : Raw<TG>::zero();
      raw.r[g] = on ? Raw<TIn>::ld(rp + 128 * g) : Raw<TIn>::zero();
    }
  }
  // only the four tap offsets are needed to issue the loads: the second 16 bytes of a sample
  WarpSample a;
  const uint4 q0 = reinterpret_cast<const uint4*>(smp)[1];
  a.p00 = q0.x; a.p01 = q0.y; a.p10 = q0.z; a.p11 = q0.w;
  if (q0.x != kNoSample) load_taps<TIn, G, FULL>(nsrc[0], a, c0, C, raw.t0);
  if (KMAX == 2) {
    const uint4 q1 = reinterpret_cast<const uint4*>(smp + (KMAX - 1))[1];
    a.p00 = q1.x; a.p01 = q1.y; a.p10 = q1.z; a.p11 = q1.w;
    if (q1.x != kNoSample) load_taps<TIn, G, FULL>(nsrc[KMAX - 1], a, c0, C, raw.t1);
  }
}

// ---------------------------------------------------------------------------
// Row hand-off with the decisions taken at table-fill time.  The four warps of a CTA own
// four consecutive rows of the same 8-pixel run; the bottom taps of row r and the top taps
// of row r+1 are usually the same two source pixels.  The lane that computes a sample also
// computes the samples of the two adjacent rows (same function, same inputs: the same bits
// the other warp gets) and stores the outcome as four flag bits next to the sample; a warp
// then reads only its own table, the per-pixel decision is a byte load, and the only
// coupling left between the warps of a CTA is the hand-off queue itself.
// With per-pixel depth (PX) the adjacent rows' samples are computed with THEIR pixels' depths,
// (x, y+1) and (x, y-1): exactly the bits the other warp computes for its own row.  The depth of
// this row would hand a weighted vector to a row that does not have that tap wherever the depth
// changes between rows.
// ---------------------------------------------------------------------------
constexpr unsigned kHoSend = 1u, kHoRecv = 2u, kHoNzLeft = 4u, kHoNzRight = 8u;

template <bool PX>
__device__ __forceinline__ void fill_run_samples_ho(WarpSample* tab, unsigned char* flg,
                                                    const SweepParams& p, const RunCoord& c, int d0,
                                                    int ppf, int lane, bool has_up, bool has_dn) {
  const int k = p.k, spp = kRun * k;
  if (lane < ppf * spp) {
    const int dd = lane / spp, rem = lane - dd * spp;
    const int i = rem / k, j = rem - i * k;
    const int d = d0 + dd;
    WarpSample s;
    s.w00 = s.w01 = s.w10 = s.w11 = 0.f;
    s.p00 = s.p01 = s.p10 = s.p11 = kNoSample;
    unsigned f = 0u;
    if (d < p.D && i < c.npix) {
      const float* m = p.hom + ((size_t)c.v * k + j) * 12;
      const int n = nbr_id_for_check(p, c.v, j);
      float mm[12];
#pragma unroll
      for (int t = 0; t < 12; ++t) mm[t] = __ldg(m + t);
      const float depth = depth_or_nan(plane_depth<PX>(p, c.v, d, c.x0 + i, c.y), n, p.n_feat);
      const float x = (float)(c.x0 + i);
      s = make_warp_sample(mm, x, (float)c.y, depth, p.H, p.W, p.C);
      if (s.p00 != kNoSample) {
        if (has_dn) {
          const float depth_dn = PX ? depth_or_nan(plane_depth<PX>(p, c.v, d, c.x0 + i, c.y + 1), n, p.n_feat) : depth;
          const WarpSample dn = make_warp_sample(mm, x, (float)(c.y + 1), depth_dn, p.H, p.W, p.C);
          if (dn.p00 != kNoSample && dn.p00 == s.p10 && dn.p01 == s.p11) f |= kHoSend;
        }
        if (has_up) {
          const float depth_up = PX ? depth_or_nan(plane_depth<PX>(p, c.v, d, c.x0 + i, c.y - 1), n, p.n_feat) : depth;
          const WarpSample up = make_warp_sample(mm, x, (float)(c.y - 1), depth_up, p.H, p.W, p.C);
          if (up.p00 != kNoSample && up.p10 == s.p00 && up.p11 == s.p01) {
            f |= kHoRecv;
            if (s.w00 != 0.f || up.w10 != 0.f) f |= kHoNzLeft;
            if (s.w01 != 0.f || up.w11 != 0.f) f |= kHoNzRight;
          }
        }
      }
    }
    tab[lane] = s;
    flg[lane] = (unsigned char)f;
  }
}


// shared-memory bytes of the hand-off queues: NSTG stages of (left, right) weighted vectors per
// (row boundary, neighbour), lane-private 16-byte columns
template <int KMAX, int G, int NSTG>
constexpr size_t run_slot_bytes() { return (size_t)2 * G * 512 * (kRunRows - 1) * KMAX * NSTG; }

// ---------------------------------------------------------------------------
// Hand-off kernel with software-pipelined loads (default for bf16 features) on a register diet:
// the hand-off queues are addressed with 32-bit shared-space addresses computed from two bases,
// the sample of a pixel is re-read from the table where it is used (weights at the blend,
// weights + offsets at the scatter) instead of living in 16 registers across the loads of the
// next pixel, and the per-pixel decisions stay packed in their flag byte (168 registers, 24 B
// of spills outside the pixel bodies).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive_a(unsigned a) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(a) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(unsigned a, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" :: "r"(a), "r"(parity) : "memory");
}
__device__ __forceinline__ void sts_p4(unsigned a, P4 v) {
  asm volatile("st.shared.v2.b64 [%0], {%1, %2};" :: "r"(a), "l"(v.lo), "l"(v.hi) : "memory");
}
__device__ __forceinline__ P4 lds_p4(unsigned a) {
  P4 v;
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(v.lo), "=l"(v.hi) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ float4 lds_f4(unsigned a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint4 lds_u4(unsigned a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ unsigned lds_u32(unsigned a) {
  unsigned v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ unsigned lds_u8(unsigned a) {
  unsigned v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}

template <int KMAX>
struct HoLite {
  unsigned slot_out, slot_in;    // shared address of (boundary below / above, neighbour 0, stage 0), this lane's column
  unsigned bar_out, bar_in;      // shared address of the boundary's first {full, empty} barrier pair
  unsigned h_out[KMAX], h_in[KMAX];
};

// one neighbour (J) of one pixel: wq = (w00, w01, w10, w11), oq = (p00, p01, p10, p11)
template <int G, bool FULL, int NSTG, int J, int KMAX>
__device__ __forceinline__ void scatter_hl(float* dst, const P4 (&gw)[G], float4 wq, uint4 oq,
                                           unsigned& id_top, P4 (&top)[G], unsigned& id_bot,
                                           P4 (&bot)[G], unsigned flags, HoLite<KMAX>& ho, int c0, int C) {
  static_assert((NSTG & (NSTG - 1)) == 0, "stage count must be a power of two");
  constexpr unsigned kVec = 512u;                     // 32 lanes x 16 bytes
  constexpr unsigned kSlot = 2u * G * kVec;           // left + right weighted vectors
  constexpr unsigned jslot = (unsigned)J * NSTG * kSlot, jbar = (unsigned)J * NSTG * 16u;
  if (flags & kHoSend) {
    const unsigned h = ho.h_out[J]++;
    const unsigned stg = h & (unsigned)(NSTG - 1), ph = (h / (unsigned)NSTG) & 1u;
    const unsigned bar = ho.bar_out + jbar + stg * 16u;
    mbar_wait_a(bar + 8u, ph ^ 1u);                   // slot empty
    const unsigned a = ho.slot_out + jslot + stg * kSlot;
    const u64 w10 = pk2(wq.z, wq.z), w11 = pk2(wq.w, wq.w);
#pragma unroll
    for (int g = 0; g < G; ++g) {
      sts_p4(a + (unsigned)g * kVec, p4scale(gw[g], w10));
      sts_p4(a + (unsigned)(G + g) * kVec, p4scale(gw[g], w11));
    }
    mbar_arrive_a(bar);                               // slot full
  } else {
    side_q<G, FULL>(dst, gw, wq.z, wq.w, oq.z, oq.w, id_bot, bot, c0, C);
  }
  if (flags & kHoRecv) {
    const unsigned h = ho.h_in[J]++;
    const unsigned stg = h & (unsigned)(NSTG - 1), ph = (h / (unsigned)NSTG) & 1u;
    const unsigned bar = ho.bar_in + jbar + stg * 16u;
    mbar_wait_a(bar, ph);
    const unsigned a = ho.slot_in + jslot + stg * kSlot;
    P4 cl[G], cr[G];
#pragma unroll
    for (int g = 0; g < G; ++g) {
      cl[g] = lds_p4(a + (unsigned)g * kVec);
      cr[g] = lds_p4(a + (unsigned)(G + g) * kVec);
    }
    mbar_arrive_a(bar + 8u);
    const u64 w00 = pk2(wq.x, wq.x), w01 = pk2(wq.y, wq.y);
#pragma unroll
    for (int g = 0; g < G; ++g) {
      cl[g] = p4fma(gw[g], w00, cl[g]);
      cr[g] = p4fma(gw[g], w01, cr[g]);
    }
    side_c<G, FULL>(dst, cl, cr, (flags & kHoNzLeft) != 0u, (flags & kHoNzRight) != 0u, oq.x, oq.y,
                    id_top, top, c0, C);
  } else {
    side_q<G, FULL>(dst, gw, wq.x, wq.y, oq.x, oq.y, id_top, top, c0, C);
  }
}

template <typename TIn, int G>
__device__ __forceinline__ void blend_taps_w(const RawTaps<TIn, G>& r, float4 wq, P4 (&wv)[G]) {
  WarpSample s;
  s.w00 = wq.x; s.w01 = wq.y; s.w10 = wq.z; s.w11 = wq.w;
  blend_taps<TIn, G>(r, s, wv);
}

// sa: shared address of this pixel's first sample (32 bytes per sample)
template <typename TIn, typename TG, int KMAX, int G, bool FULL, int NSTG, bool V0, bool V1, int MODE>
__device__ __forceinline__ void pixel_q3(RunPending<KMAX, G>& pend, PixelRaw<TIn, TG, G>& raw, unsigned sa,
                                         unsigned flags0, unsigned flags1, bool has_next,
                                         const WarpSample* smp_next, const TG* __restrict__ gp_next,
                                         const TIn* __restrict__ rp_next, const TIn* const (&nsrc)[KMAX],
                                         float* const (&ndst)[KMAX], uint32_t taddr, u64 inv_n2,
                                         u64 two_inv_n2, int c0, int C, HoLite<KMAX>& ho, const SweepParams& p) {
  constexpr unsigned kS1 = 32u * (KMAX - 1);
  P4 w0[G], w1[G], gw0[G], gw1[G], ref[G], gv[G];
  if (V0) blend_taps_w<TIn, G>(raw.t0, lds_f4(sa), w0);
  if (V1) blend_taps_w<TIn, G>(raw.t1, lds_f4(sa + kS1), w1);
  if constexpr (MODE == 1) {
    // group-wise correlation: d ref += gq_0 w_0 + gq_1 w_1 ; d w_j = gq_j ref (gq: the group's gradient / width)
    u64 q0[G], q1[G];
    {
      const float qv[4] = {raw.g[0].x, raw.g[0].y, raw.g[0].z, raw.g[0].w};
#pragma unroll
      for (int g = 0; g < G; ++g) {
        ref[g] = p4from(raw.r[g]);
        q0[g] = pk2(qv[g], qv[g]);
        q1[g] = pk2(qv[2 + g], qv[2 + g]);
      }
    }
    if (has_next) issue_pixel_loads<TIn, TG, KMAX, G, FULL, MODE>(raw, smp_next, gp_next, rp_next, nsrc, c0, C, p);
    if (V0 || V1) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const uint32_t ta = taddr + 4u * (uint32_t)g;
        P4 acc = tmem_ld4(ta);
        if (V0) acc = p4fma(w0[g], q0[g], acc);
        if (V1) acc = p4fma(w1[g], q1[g], acc);
        tmem_st4(ta, acc);
        if (V0) gw0[g] = p4scale(ref[g], q0[g]);
        if (V1) gw1[g] = p4scale(ref[g], q1[g]);
      }
    }
  } else {
#pragma unroll
    for (int g = 0; g < G; ++g) {
      ref[g] = p4from(raw.r[g]);
      gv[g] = p4scale(p4from(raw.g[g]), two_inv_n2);
    }
    if (has_next) issue_pixel_loads<TIn, TG, KMAX, G, FULL, MODE>(raw, smp_next, gp_next, rp_next, nsrc, c0, C, p);
#pragma unroll
    for (int g = 0; g < G; ++g) {
      P4 mu = ref[g];
      if (V0) mu = p4add(mu, w0[g]);
      if (V1) mu = p4add(mu, w1[g]);
      mu = p4scale(mu, inv_n2);
      const uint32_t ta = taddr + 4u * (uint32_t)g;
      tmem_st4(ta, p4fma(gv[g], p4sub(ref[g], mu), tmem_ld4(ta)));
      if (V0) gw0[g] = p4mul(gv[g], p4sub(w0[g], mu));
      if (V1) gw1[g] = p4mul(gv[g], p4sub(w1[g], mu));
    }
  }
  if (V0)
    scatter_hl<G, FULL, NSTG, 0, KMAX>(ndst[0], gw0, lds_f4(sa), lds_u4(sa + 16u), pend.id_top[0], pend.top[0],
                                       pend.id_bot[0], pend.bot[0], flags0, ho, c0, C);
  if (V1)
    scatter_hl<G, FULL, NSTG, KMAX - 1, KMAX>(ndst[KMAX - 1], gw1, lds_f4(sa + kS1), lds_u4(sa + kS1 + 16u),
                                              pend.id_top[KMAX - 1], pend.top[KMAX - 1], pend.id_bot[KMAX - 1],
                                              pend.bot[KMAX - 1], flags1, ho, c0, C);
}

// requires p.k == KMAX
template <typename TIn, typename TG, int KMAX, int G, bool FULL, int MINB, int NSTG, int MODE = 0, bool PX = false>
__global__ void __launch_bounds__(kRunThreads, MINB) sweep_bwd_runs_kernel(const SweepParams p) {
  static_assert(MODE == 0 || (KMAX == 2 && sizeof(TG) == 4), "correlation mode: two neighbours, fp32 gradients");
  constexpr int kCols = kRun * G * 4;
  constexpr unsigned kSlot = 2u * G * 512u;
  extern __shared__ __align__(16) unsigned char s_dyn[];          // [kRunRows - 1][KMAX][NSTG] slots
  // two table buffers per warp: while the planes of one are processed the other already holds the
  // next planes, so the load pipeline never drains at a table refill
  __shared__ WarpSample s_tab[kRunRows][2][32];
  __shared__ unsigned char s_flg[kRunRows][2][32];
  __shared__ __align__(8) unsigned long long s_bar[kRunRows - 1][KMAX][NSTG][2];   // {full, empty}
  __shared__ uint32_t s_tmem;
  static_assert(sizeof(WarpSample) == 32, "sample table stride");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const RunCoord c = run_coord<G>(p, warp, lane);
  if (threadIdx.x < (kRunRows - 1) * KMAX * NSTG * 2) {
    mbar_init(&s_bar[0][0][0][0] + threadIdx.x, 32);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const uint32_t tbase = tmem_alloc_cta<kCols>(&s_tmem, warp);     // contains the CTA barriers
  if (c.y < p.H) {
    const int C = p.C, HW = p.H * p.W;
    const TIn* feat = static_cast<const TIn*>(p.feat);
    const size_t ref_off = ((size_t)(c.v + p.ref_begin) * HW + (size_t)c.y * p.W + c.x0) * C + c.c0;
    const TIn* ref_row = feat + ref_off;
    // MODE 1: the upstream gradient is [V,k,D,H,W,groups]; gpix / plane_stride are its pixel / plane strides
    const int gpix = MODE == 1 ? p.corr_groups : C;
    const size_t plane_stride = MODE == 1 ? (size_t)HW * p.corr_groups : (size_t)HW * C;
    const TG* g_d = MODE == 1
        ? static_cast<const TG*>(p.g_out) + ((size_t)c.v * KMAX * p.D * HW + (size_t)c.y * p.W + c.x0) * p.corr_groups
        : static_cast<const TG*>(p.g_out) + ((size_t)c.v * p.D * HW + (size_t)c.y * p.W + c.x0) * C + c.c0;
    const bool one_chunk = p.slices == 1;
    const unsigned pf_bytes = (unsigned)((one_chunk ? (size_t)c.npix * C : (size_t)min(128 * G, C - (c.c0 - 4 * lane))) *
                                         sizeof(TG)) & ~15u;
    const TG* pf_base = g_d - 4 * lane;
    const bool pf_ok = MODE == 0 && pf_bytes >= 16 && (reinterpret_cast<uintptr_t>(pf_base) & 15) == 0 &&
                       ((plane_stride * sizeof(TG)) & 15) == 0;       // the correlation gradient is small: no L2 prefetch
    auto prefetch_plane = [&](int d) {
      if (!pf_ok || d >= p.D) return;
      const TG* q = pf_base + (size_t)d * plane_stride;
      if (one_chunk) {
        if (lane == 0) prefetch_l2(q, pf_bytes);
      } else if (lane < c.npix) {
        prefetch_l2(q + (size_t)lane * C, pf_bytes);
      }
    };
#pragma unroll
    for (int d = 0; d < kPrefetchPlanes; ++d) prefetch_plane(d);

    const TIn* nsrc[KMAX];
    float* ndst[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
      const int n = __ldg(p.nbr + (size_t)c.v * KMAX + j);
      nsrc[j] = feat + (size_t)n * HW * C + c.c0;
      ndst[j] = p.g_feat + (size_t)n * HW * C + c.c0;
      asm volatile("" : "+l"(nsrc[j]), "+l"(ndst[j]));
    }
    const float inv_n = 1.0f / (float)(KMAX + 1);
    const u64 inv_n2 = pk2(inv_n, inv_n);
    const u64 two_inv_n2 = pk2(2.0f * inv_n, 2.0f * inv_n);
    constexpr int spp = kRun * KMAX;
    constexpr int ppf = 32 / spp > 0 ? 32 / spp : 1;
    const bool has_up = warp > 0;
    const bool has_dn = warp + 1 < kRunRows && c.y + 1 < p.H;
    const int bo = min(warp, kRunRows - 2), bi = max(warp - 1, 0);     // boundary below / above this row
    HoLite<KMAX> ho;
    ho.slot_out = smem_u32(s_dyn) + (unsigned)(bo * KMAX * NSTG) * kSlot + (unsigned)lane * 16u;
    ho.slot_in = smem_u32(s_dyn) + (unsigned)(bi * KMAX * NSTG) * kSlot + (unsigned)lane * 16u;
    ho.bar_out = smem_u32(&s_bar[bo][0][0][0]);
    ho.bar_in = smem_u32(&s_bar[bi][0][0][0]);
#pragma unroll
    for (int j = 0; j < KMAX; ++j) ho.h_out[j] = ho.h_in[j] = 0u;
    const unsigned tab_a = smem_u32(s_tab[warp][0]), flg_a = smem_u32(s_flg[warp][0]);

#pragma unroll
    for (int q = 0; q < kRun * G; ++q) tmem_st4(tbase + 4u * (uint32_t)q, p4zero());
    tmem_wait_st();

    PixelRaw<TIn, TG, G> raw;
    fill_run_samples_ho<PX>(s_tab[warp][0], s_flg[warp][0], p, c, 0, ppf, lane, has_up, has_dn);
    if (ppf < p.D) fill_run_samples_ho<PX>(s_tab[warp][1], s_flg[warp][1], p, c, ppf, ppf, lane, has_up, has_dn);
    __syncwarp();
    // pipeline prologue: first pixel of the first plane
    issue_pixel_loads<TIn, TG, KMAX, G, FULL, MODE>(raw, s_tab[warp][0], g_d, ref_row, nsrc, c.c0, C, p);
    int buf = 0;
    for (int d0 = 0; d0 < p.D; d0 += ppf, buf ^= 1) {
      const int dend = min(p.D, d0 + ppf);
      const bool more_fills = d0 + ppf < p.D;
      for (int d = d0; d < dend; ++d) {
        prefetch_plane(d + kPrefetchPlanes);
        tmem_wait_st();
        RunPending<KMAX, G> pend;
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
          pend.id_top[j] = pend.id_bot[j] = kNoTap;
#pragma unroll
          for (int g = 0; g < G; ++g) pend.top[j][g] = pend.bot[j][g] = p4zero();
        }
        const int toff = buf * 32 + (d - d0) * spp;
        const WarpSample* tab = s_tab[warp][0] + toff;
        const bool last_plane = d + 1 >= dend;
        const bool more_planes = !last_plane || more_fills;
        // first sample of the next plane: next rows of this buffer, or the other buffer
        const WarpSample* tab_next = last_plane ? s_tab[warp][buf ^ 1] : tab + spp;
#pragma unroll 1
        for (int i = 0; i < c.npix; ++i) {
          const unsigned si = (unsigned)(toff + i * KMAX);
          const unsigned sa = tab_a + si * 32u;
          const bool v0 = lds_u32(sa + 16u) != kNoSample;
          const bool v1 = KMAX == 2 && lds_u32(sa + 32u * (KMAX - 1) + 16u) != kNoSample;
          const unsigned f0 = lds_u8(flg_a + si);
          const unsigned f1 = KMAX == 2 ? lds_u8(flg_a + si + (KMAX - 1)) : 0u;
          const bool in_run = i + 1 < c.npix;
          const bool has_next = in_run || more_planes;
          const WarpSample* smp_next = in_run ? tab + (i + 1) * KMAX : tab_next;
          const TG* gp_next = in_run ? g_d + (i + 1) * gpix : g_d + plane_stride;
          const TIn* rp_next = in_run ? ref_row + (i + 1) * C : ref_row;
          const uint32_t ta = tbase + 4u * (uint32_t)(i * G);
          if (v0 && v1)
            pixel_q3<TIn, TG, KMAX, G, FULL, NSTG, true, true, MODE>(pend, raw, sa, f0, f1, has_next, smp_next, gp_next, rp_next, nsrc, ndst, ta, inv_n2, two_inv_n2, c.c0, C, ho, p);
          else if (v0)
            pixel_q3<TIn, TG, KMAX, G, FULL, NSTG, true, false, MODE>(pend, raw, sa, f0, f1, has_next, smp_next, gp_next, rp_next, nsrc, ndst, ta, inv_n2, two_inv_n2, c.c0, C, ho, p);
          else if (v1)
            pixel_q3<TIn, TG, KMAX, G, FULL, NSTG, false, true, MODE>(pend, raw, sa, f0, f1, has_next, smp_next, gp_next, rp_next, nsrc, ndst, ta, inv_n2, two_inv_n2, c.c0, C, ho, p);
          else
            pixel_q3<TIn, TG, KMAX, G, FULL, NSTG, false, false, MODE>(pend, raw, sa, f0, f1, has_next, smp_next, gp_next, rp_next, nsrc, ndst, ta, inv_n2, two_inv_n2, c.c0, C, ho, p);
        }
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
          flush_open_p<G, FULL>(ndst[j], pend.id_top[j], pend.top[j], c.c0, C);
          flush_open_p<G, FULL>(ndst[j], pend.id_bot[j], pend.bot[j], c.c0, C);
        }
        g_d += plane_stride;
      }
      // this buffer's planes are done (the loads already in flight read the other buffer): refill it
      __syncwarp();
      if (d0 + 2 * ppf < p.D)
        fill_run_samples_ho<PX>(s_tab[warp][buf], s_flg[warp][buf], p, c, d0 + 2 * ppf, ppf, lane, has_up, has_dn);
      __syncwarp();
    }
    tmem_wait_st();
    float* dst = p.g_feat + ref_off;
    for (int i = 0; i < c.npix; ++i) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
        const P4 acc = tmem_ld4(tbase + 4u * (uint32_t)(i * G + g));
        if (group_on<FULL>(c.c0, g, C)) red_add_p4(dst + i * C + 128 * g, acc);
      }
    }
  }
  tmem_free_cta<kCols>(&s_tmem, warp);
}

// k in {1,2} only (k*kRun <= 32 samples per plane); other k use the pixel kernel.
// One run kernel is built per feature dtype: the hand-off kernel for bf16 features, the lean
// kernel for fp32 features -- with fp32 features the raw loads of a pixel are 80 registers
// instead of 44 and the pipelined kernel spills (ptxas: 160 B of stack).
template <typename TIn, typename TG, bool PX>
static int launch_bwd_run_t(SweepParams& p, cudaStream_t st) {
  const int G = sweep_groups(p.C);
  p.tiles_x = (p.W + kRun - 1) / kRun;
  p.tiles_y = (p.H + kRunRows - 1) / kRunRows;
  p.slices = (p.C + 128 * G - 1) / (128 * G);
  const long long blocks = (long long)p.V * p.slices * p.tiles_y * p.tiles_x;
  if (blocks > 2147483647LL) return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_bwd: grid too large");
  dim3 grid((unsigned)blocks);
  const bool full = p.C % (128 * G) == 0;
#define MVSD_RUN(KM, GG, FU)                                                                \
  do {                                                                                      \
    if constexpr (sizeof(TIn) == 2) {                                                       \
      auto kern = sweep_bwd_runs_kernel<TIn, TG, KM, GG, FU, kRunQMinBlocks, 2, 0, PX>;     \
      constexpr size_t dyn = run_slot_bytes<KM, GG, 2>();                                   \
      static bool attr_set = false;                                                         \
      if (!attr_set) {                                                                      \
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);  \
        attr_set = true;                                                                    \
      }                                                                                     \
      kern<<<grid, kRunThreads, dyn, st>>>(p);                                              \
    } else {                                                                                \
      sweep_bwd_runq_kernel<TIn, TG, KM, GG, FU, kRunQMinBlocks, PX><<<grid, kRunThreads, 0, st>>>(p); \
    }                                                                                       \
  } while (0)
  if (p.k == 1) {
    if (G == 2) { if (full) MVSD_RUN(1, 2, true); else MVSD_RUN(1, 2, false); }
    else { if (full) MVSD_RUN(1, 1, true); else MVSD_RUN(1, 1, false); }
  } else {
    if (G == 2) { if (full) MVSD_RUN(2, 2, true); else MVSD_RUN(2, 2, false); }
    else { if (full) MVSD_RUN(2, 1, true); else MVSD_RUN(2, 1, false); }
  }
#undef MVSD_RUN
  count_launch();
  return check_launch("plane_sweep_bwd(run)");
}

// Group-wise correlation backward (group_corr.cu) through the hand-off kernel: bf16 features, k = 2.
// Returns -1 when this configuration is not built (the caller falls back to its pixel kernel).
template <bool PX>
static int launch_bwd_run_corr_t(SweepParams& p, cudaStream_t st) {
  typedef __nv_bfloat16 TIn;
  const int G = sweep_groups(p.C);
  p.tiles_x = (p.W + kRun - 1) / kRun;
  p.tiles_y = (p.H + kRunRows - 1) / kRunRows;
  p.slices = (p.C + 128 * G - 1) / (128 * G);
  const long long blocks = (long long)p.V * p.slices * p.tiles_y * p.tiles_x;
  if (blocks > 2147483647LL) return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_groupcorr_bwd: grid too large");
  dim3 grid((unsigned)blocks);
  const bool full = p.C % (128 * G) == 0;
#define MVSD_RUNC(GG, FU)                                                                   \
  do {                                                                                      \
    auto kern = sweep_bwd_runs_kernel<TIn, float, 2, GG, FU, kRunQMinBlocks, 2, 1, PX>;     \
    constexpr size_t dyn = run_slot_bytes<2, GG, 2>();                                      \
    static bool attr_set = false;                                                           \
    if (!attr_set) {                                                                        \
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);    \
      attr_set = true;                                                                      \
    }                                                                                       \
    kern<<<grid, kRunThreads, dyn, st>>>(p);                                                \
  } while (0)
  if (G == 2) { if (full) MVSD_RUNC(2, true); else MVSD_RUNC(2, false); }
  else { if (full) MVSD_RUNC(1, true); else MVSD_RUNC(1, false); }
#undef MVSD_RUNC
  count_launch();
  return check_launch("plane_sweep_groupcorr_bwd(run)");
}

int launch_bwd_run_corr(SweepParams& p, int feat_dtype, cudaStream_t st) {
  if (feat_dtype != MVSD_BF16 || p.k != 2) return -1;
  return p.depth_per_pixel ? launch_bwd_run_corr_t<true>(p, st) : launch_bwd_run_corr_t<false>(p, st);
}

template <bool PX>
static int launch_bwd_run_px(SweepParams& p, int feat_dtype, int g_dtype, cudaStream_t st) {
  if (feat_dtype == MVSD_F32 && g_dtype == MVSD_F32) return launch_bwd_run_t<float, float, PX>(p, st);
  if (feat_dtype == MVSD_BF16 && g_dtype == MVSD_BF16)
    return launch_bwd_run_t<__nv_bfloat16, __nv_bfloat16, PX>(p, st);
  if (feat_dtype == MVSD_BF16 && g_dtype == MVSD_F32)
    return launch_bwd_run_t<__nv_bfloat16, float, PX>(p, st);
  return fail(MVSD_ERR_UNSUPPORTED, "plane_sweep_bwd: dtype combination not built");
}

int launch_bwd_run(SweepParams& p, int feat_dtype, int g_dtype, cudaStream_t st) {
  return p.depth_per_pixel ? launch_bwd_run_px<true>(p, feat_dtype, g_dtype, st)
                           : launch_bwd_run_px<false>(p, feat_dtype, g_dtype, st);
}

}  // namespace mvsd
