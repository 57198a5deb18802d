// Voxel-volume combine of a view-sharded scene over NVLink peer memory.
//
// After the local back-projection every rank holds partial per-voxel feature sums and
// valid counts for its reference views (mvsdet.py:1458-1460 per view); the reference then
// sums over views and divides by the count (mvsdet.py:511-515, :681-682).  Across ranks
// that is sum-all-reduce + normalise.  Instead of NCCL all-reduce + a normalise kernel
// (three passes over 26 MB and a latency-bound collective), ONE kernel does the
// reduce-scatter, the normalisation and the all-gather over peer pointers:
//   rank r owns the r-th 1/G of the flat [C*N] volume; for each owned float4 it loads the
//   partial from every peer (NVLink P2P loads, rank order -> identical bits on every
//   rank), divides by the reduced count and stores the result into EVERY peer's output
//   buffer (P2P stores).  Per rank: (G-1)/G * 26 MB in and out over NVLink, nothing
//   through HBM twice.
// The caller brackets the kernel with two cross-rank barriers (partials complete /
// results delivered); buffers come from torch's symmetric-memory allocator.
#include "common.cuh"

namespace mvsd {
namespace {

constexpr int kMaxPeers = 16;

struct P2PParams {
  const float* const* part;     // device array [world]: peers' partial buffers ([total] fp32 sums, then [N] int32 counts)
  float* const* out;            // device array [world]: peers' result buffers (same layout)
  int32_t* count_local;         // [N] reduced counts (also written to this rank's out tail)
  int world, rank, cfirst, C, N;
};

__device__ __forceinline__ float4 ld_peer4(const float* p) {       // never from a stale L1 line
  return __ldcv(reinterpret_cast<const float4*>(p));
}

// every rank reduces ALL counts (N * world 4-byte loads: 0.1 MB per peer)
__global__ void p2p_count_kernel(const P2PParams p) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= p.N) return;
  const size_t total = (size_t)p.C * p.N;
  int cnt = 0;
  for (int q = 0; q < p.world; ++q)
    cnt += __ldcv(reinterpret_cast<const int32_t*>(p.part[q] + total) + u);
  p.count_local[u] = cnt;
  reinterpret_cast<int32_t*>(p.out[p.rank] + total)[u] = cnt;
}

template <int WORLD>            // 0 = run-time world size
__global__ void __launch_bounds__(256) p2p_reduce_kernel(const P2PParams p) {
  const size_t total4 = ((size_t)p.C * p.N) >> 2;                // float4 elements (C*N % 4 == 0)
  const int world = WORLD ? WORLD : p.world;
  const size_t chunk = (total4 + world - 1) / world;
  const size_t begin = chunk * p.rank, end = min(total4, begin + chunk);
  const float* part[kMaxPeers];
  float* out[kMaxPeers];
#pragma unroll
  for (int q = 0; q < (WORLD ? WORLD : kMaxPeers); ++q) {
    if (q < world) {
      part[q] = p.part[q];
      out[q] = p.out[q];
    }
  }
  for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < end;
       i += (size_t)gridDim.x * blockDim.x) {
    const size_t e = i << 2;
    float4 s = ld_peer4(part[0] + e);
#pragma unroll
    for (int q = 1; q < (WORLD ? WORLD : kMaxPeers); ++q) {
      if (q < world) {
        const float4 t = ld_peer4(part[q] + e);
        s.x = __fadd_rn(s.x, t.x); s.y = __fadd_rn(s.y, t.y);
        s.z = __fadd_rn(s.z, t.z); s.w = __fadd_rn(s.w, t.w);
      }
    }
    int c0, c1, c2, c3;
    if (p.cfirst) {                                              // [C][N]: four consecutive voxels
      const int u = (int)(e % (size_t)p.N);
      const int4 c = *reinterpret_cast<const int4*>(p.count_local + u);
      c0 = c.x; c1 = c.y; c2 = c.z; c3 = c.w;
    } else {                                                     // [N][C]: one voxel, four channels
      c0 = c1 = c2 = c3 = p.count_local[e / (size_t)p.C];
    }
    // sum / (count + 1e-8), zero where count == 0 (mvsdet.py:514-515)
    float4 m;
    m.x = c0 ? __fdiv_rn(s.x, __fadd_rn((float)c0, 1e-8f)) : 0.f;
    m.y = c1 ? __fdiv_rn(s.y, __fadd_rn((float)c1, 1e-8f)) : 0.f;
    m.z = c2 ? __fdiv_rn(s.z, __fadd_rn((float)c2, 1e-8f)) : 0.f;
    m.w = c3 ? __fdiv_rn(s.w, __fadd_rn((float)c3, 1e-8f)) : 0.f;
#pragma unroll
    for (int q = 0; q < (WORLD ? WORLD : kMaxPeers); ++q)
      if (q < world) *reinterpret_cast<float4*>(out[q] + e) = m;
  }
}

// Backward of a view-sharded scene: a rank's plane-sweep backward scatters into the gradient maps
// of its block views AND of its halo views (neighbours owned by other ranks).  The owner of a view
// adds the halo contributions of its peers to its own map: one pull kernel over NVLink peer
// pointers, one CTA column per (owned view, 16-byte chunk), sources in table order -> the same
// summation order on every run (deterministic).  pulls: CSR over the owned views --
// offs[d] .. offs[d+1] index (src_rank, src_local_view) pairs.
// The element type is fp32 (mvsd_halo_reduce_p2p) or the 64-bit fixed point of the *_det scatter
// backwards (mvsd_halo_reduce_p2p_fixed, common.cuh), whose integer adds make the owner's sum
// independent of how the views were split over the ranks.  Both move 16 bytes per peer load.
template <typename T>
struct HaloParams {
  T* const* g;                // device array [world]: peers' gradient buffers [V_local][view_elems]
  const int32_t* offs;        // [n_own + 1]
  const int32_t* src;         // [n_pull][2]
  int rank, n_own;
  size_t view_elems;          // H*W*C, multiple of 4
};

template <typename T> struct HaloVec;
template <> struct HaloVec<float> {                 // one float4
  using V16 = float4;
  static constexpr int kElems = 4;
  static __device__ __forceinline__ float4 ld_peer(const float* p) { return ld_peer4(p); }
  static __device__ __forceinline__ float4 add(float4 s, float4 t) {
    s.x = __fadd_rn(s.x, t.x); s.y = __fadd_rn(s.y, t.y);
    s.z = __fadd_rn(s.z, t.z); s.w = __fadd_rn(s.w, t.w);
    return s;
  }
};
template <> struct HaloVec<long long> {             // two long long
  using V16 = longlong2;
  static constexpr int kElems = 2;
  static __device__ __forceinline__ longlong2 ld_peer(const long long* p) {
    return __ldcv(reinterpret_cast<const longlong2*>(p));
  }
  static __device__ __forceinline__ longlong2 add(longlong2 s, longlong2 t) {
    // two's-complement wrap-around: exact whenever the true sum fits, whatever the order
    s.x = (long long)((unsigned long long)s.x + (unsigned long long)t.x);
    s.y = (long long)((unsigned long long)s.y + (unsigned long long)t.y);
    return s;
  }
};

template <typename T>
__global__ void __launch_bounds__(256) halo_reduce_kernel(const HaloParams<T> p) {
  using Vec = HaloVec<T>;
  using V16 = typename Vec::V16;
  constexpr int kE = Vec::kElems;
  const int d = blockIdx.y;
  const int b = p.offs[d], e = p.offs[d + 1];
  if (b == e) return;
  T* mine = p.g[p.rank] + (size_t)d * p.view_elems;
  const size_t nv = p.view_elems / kE;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (size_t)gridDim.x * blockDim.x) {
    V16 s = *reinterpret_cast<const V16*>(mine + i * kE);
    for (int q = b; q < e; ++q) {
      const T* peer = p.g[p.src[2 * q]] + (size_t)p.src[2 * q + 1] * p.view_elems;
      s = Vec::add(s, Vec::ld_peer(peer + i * kE));
    }
    *reinterpret_cast<V16*>(mine + i * kE) = s;
  }
}

// Forward of a view-sharded scene from each rank's own feature maps: every rank packs the views it owns
// into rows [0, n_own) of its peer-mapped buffer; after a cross-rank barrier it copies its halo views (the
// neighbours of its reference views that other ranks own) from their owners into rows n_own + j.  The rows
// are opaque bytes (bf16 or fp32 channels-last maps), moved in 16-byte vectors, or in 8-byte ones when a row
// is not a multiple of 16 bytes (bf16 with H*W odd and C % 8 == 4: rows packed back to back then start
// 8-byte aligned).  src[2j], src[2j+1] = (owner rank, row in the owner's buffer) of halo row j.
struct GatherParams {
  char* const* feat;          // device array [world]: peers' packed buffers [V_local][view_bytes]
  const int32_t* src;         // [n_halo][2]
  int rank, n_own;
  size_t view_bytes;
};

template <typename V>           // uint4 or uint2
__global__ void __launch_bounds__(256) halo_gather_kernel(const GatherParams p) {
  const int j = blockIdx.y;
  const V* peer = reinterpret_cast<const V*>(p.feat[p.src[2 * j]] + (size_t)p.src[2 * j + 1] * p.view_bytes);
  V* mine = reinterpret_cast<V*>(p.feat[p.rank] + (size_t)(p.n_own + j) * p.view_bytes);
  const size_t nv = p.view_bytes / sizeof(V);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (size_t)gridDim.x * blockDim.x)
    mine[i] = __ldcv(peer + i);                                  // never from a stale L1 line
}

// the rules and the grid both halo kernels follow: at most kMaxPeers ranks, one CTA column per row of
// this rank they write, at most 64 CTAs (of 256 threads, one vector each) across a row
int check_world(const char* who, int world, int rank) {
  if (world < 1 || world > kMaxPeers || rank < 0 || rank >= world)
    return fail(MVSD_ERR_INVALID_ARG, "%s: bad world/rank (%d/%d)", who, rank, world);
  return MVSD_OK;
}

dim3 halo_grid(size_t vecs_per_row, int rows) {
  const size_t want = (vecs_per_row + 255) / 256;
  return dim3((unsigned)(want < 64 ? want : 64), (unsigned)rows);
}

template <typename T>
int halo_reduce(const char* who, void* const* g_ptrs, const int32_t* pull_offsets, const int32_t* pull_sources,
                int world, int rank, int n_own, int64_t view_elems, void* stream) {
  if (!g_ptrs || !pull_offsets || !pull_sources)
    return fail(MVSD_ERR_INVALID_ARG, "%s: null pointer", who);
  if (int e = check_world(who, world, rank)) return e;
  if (n_own <= 0 || n_own > 65535 || view_elems <= 0 || (view_elems & 3))
    return fail(MVSD_ERR_INVALID_ARG, "%s: bad view count / size", who);
  HaloParams<T> p;
  p.g = reinterpret_cast<T* const*>(g_ptrs);
  p.offs = pull_offsets; p.src = pull_sources; p.rank = rank; p.n_own = n_own;
  p.view_elems = (size_t)view_elems;
  const dim3 grid = halo_grid((size_t)view_elems / HaloVec<T>::kElems, n_own);
  halo_reduce_kernel<T><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  count_launch();
  return check_launch(who);
}

}  // namespace
}  // namespace mvsd

using namespace mvsd;

extern "C" int mvsd_halo_reduce_p2p(void* const* g_ptrs, const int32_t* pull_offsets,
                                    const int32_t* pull_sources, int world, int rank, int n_own,
                                    int64_t view_elems, void* stream) {
  return halo_reduce<float>("halo_reduce_p2p", g_ptrs, pull_offsets, pull_sources, world, rank, n_own,
                            view_elems, stream);
}

extern "C" int mvsd_halo_reduce_p2p_fixed(void* const* g_ptrs, const int32_t* pull_offsets,
                                          const int32_t* pull_sources, int world, int rank, int n_own,
                                          int64_t view_elems, void* stream) {
  return halo_reduce<long long>("halo_reduce_p2p_fixed", g_ptrs, pull_offsets, pull_sources, world, rank,
                                n_own, view_elems, stream);
}

extern "C" int mvsd_halo_gather_p2p(void* const* feat_ptrs, const int32_t* gather_sources, int world, int rank,
                                    int n_own, int n_halo, int64_t view_bytes, void* stream) {
  const char* who = "halo_gather_p2p";
  if (!feat_ptrs || !gather_sources)
    return fail(MVSD_ERR_INVALID_ARG, "%s: null pointer", who);
  if (int e = check_world(who, world, rank)) return e;
  if (n_own <= 0 || n_own > 65535 || n_halo <= 0 || n_halo > 65535 || view_bytes <= 0 || (view_bytes & 7))
    return fail(MVSD_ERR_INVALID_ARG, "%s: bad view count / size", who);
  GatherParams p;
  p.feat = reinterpret_cast<char* const*>(feat_ptrs);
  p.src = gather_sources; p.rank = rank; p.n_own = n_own;
  p.view_bytes = (size_t)view_bytes;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (view_bytes & 15)
    halo_gather_kernel<uint2><<<halo_grid((size_t)view_bytes / 8, n_halo), 256, 0, st>>>(p);
  else
    halo_gather_kernel<uint4><<<halo_grid((size_t)view_bytes / 16, n_halo), 256, 0, st>>>(p);
  count_launch();
  return check_launch(who);
}

extern "C" int mvsd_voxel_reduce_p2p(const void* const* part_ptrs, void* const* out_ptrs,
                                     int32_t* count_local, int world, int rank, int layout, int C,
                                     int N, void* stream) {
  if (!part_ptrs || !out_ptrs || !count_local)
    return fail(MVSD_ERR_INVALID_ARG, "voxel_reduce_p2p: null pointer");
  if (world < 1 || world > kMaxPeers || rank < 0 || rank >= world)
    return fail(MVSD_ERR_INVALID_ARG, "voxel_reduce_p2p: bad world/rank (%d/%d, at most %d peers)", rank,
                world, kMaxPeers);
  if (C <= 0 || N <= 0 || (C % 4) || (N % 4))
    return fail(MVSD_ERR_UNSUPPORTED, "voxel_reduce_p2p: C and N must be positive multiples of 4");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  P2PParams p;
  p.part = reinterpret_cast<const float* const*>(part_ptrs);
  p.out = reinterpret_cast<float* const*>(out_ptrs);
  p.count_local = count_local;
  p.world = world; p.rank = rank; p.cfirst = layout == MVSD_CHANNELS_FIRST ? 1 : 0; p.C = C; p.N = N;
  p2p_count_kernel<<<(N + 255) / 256, 256, 0, st>>>(p);
  count_launch();
  if (int e = check_launch("voxel_reduce_p2p(count)")) return e;
  // 148 SMs x 2 CTAs of 256 threads, each thread ~4 float4 per peer in flight: enough peer loads to
  // cover the NVLink round trip without taking every SM slot from a sweep that runs concurrently
  const size_t total4 = ((size_t)C * N) >> 2;
  const size_t chunk = (total4 + world - 1) / world;
  const size_t want = (chunk + 255) / 256;
  const unsigned blocks = (unsigned)(want < 148 * 2 ? (want ? want : 1) : 148 * 2);
  switch (world) {
    case 2: p2p_reduce_kernel<2><<<blocks, 256, 0, st>>>(p); break;
    case 4: p2p_reduce_kernel<4><<<blocks, 256, 0, st>>>(p); break;
    case 8: p2p_reduce_kernel<8><<<blocks, 256, 0, st>>>(p); break;
    default: p2p_reduce_kernel<0><<<blocks, 256, 0, st>>>(p); break;
  }
  count_launch();
  return check_launch("voxel_reduce_p2p");
}
