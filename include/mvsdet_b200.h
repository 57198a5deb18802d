/*
 * mvsdet_b200 -- C ABI of the B200-native MVSDet hot path.
 *
 * The reference (Pixie8888/MVSDet) has NO native/FFI boundary on this path: the
 * plane sweep, depth top-k and voxel back-projection are plain PyTorch calls
 * inlined in MVSDet.extract_feat (projects/NeRF-Det/nerfdet/mvsdet.py:430-515).
 * The boundary below is therefore the one a maintainer would bind from that
 * Python code (ctypes stub in INTEGRATION.md); every entry point names the
 * reference lines whose work it replaces.
 *
 * Conventions (all entry points):
 *   - plain C, no torch / CUDA types in the signatures; `stream` is a
 *     cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch's caching
 *     allocator); the library never allocates, frees or synchronises, so every
 *     call is re-entrant and capturable in a CUDA graph;
 *   - return value: MVSD_OK (0) or a non-zero mvsd_status; nothing is thrown
 *     across the ABI.  mvsd_last_error() gives a human-readable message for the
 *     calling thread's last failure;
 *   - there is no CPU fallback: without a CUDA device every compute entry
 *     point returns MVSD_ERR_CUDA.
 *
 * Layouts.  "nhwc" feature maps are [V][H][W][C] with C fastest, i.e. a
 * torch tensor of logical shape [V,C,H,W] in torch.channels_last memory
 * format.  Volumes with layout MVSD_CHANNELS_LAST are [V][D][H][W][C]
 * (torch.channels_last_3d of logical [V,C,D,H,W]).  C must be a multiple of 4
 * and at most 512.  Accumulation is always fp32 (64-bit fixed point in the
 * bit-reproducible *_det forms of the scatter backwards).
 *
 * Additive symbols (no ABI version change; every earlier signature is unchanged):
 *   mvsd_plane_sweep_fwd_px, mvsd_plane_sweep_bwd_px, mvsd_plane_sweep_bwd_det_px,
 *   mvsd_plane_sweep_groupcorr_fwd_px, mvsd_plane_sweep_groupcorr_bwd_px --
 *   the fused sweeps with per-pixel depth hypotheses;
 *   mvsd_depth_topk_fwd_px, mvsd_depth_topk_bwd_px -- the top-k epilogue over
 *   per-pixel depth hypotheses;
 *   mvsd_plane_sweep_groupcorr_bwd_det, mvsd_plane_sweep_groupcorr_bwd_det_px --
 *   the deterministic group-correlation backward;
 *   mvsd_homo_warp_bwd_det, mvsd_backproject_bwd_det_mode -- the deterministic
 *   backwards of the stand-alone warp and of the SUM / PER_VIEW back-projection;
 *   mvsd_halo_reduce_p2p_fixed -- the halo pull of a view-sharded scene over the
 *   64-bit fixed-point accumulators of the deterministic backwards.
 */
#ifndef MVSDET_B200_H_
#define MVSDET_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVSD_ABI_VERSION 3

typedef enum {
  MVSD_OK = 0,
  MVSD_ERR_INVALID_ARG = 1,   /* null pointer, non-positive dim, bad enum      */
  MVSD_ERR_UNSUPPORTED = 2,   /* legal request outside the compiled envelope  */
  MVSD_ERR_CUDA = 3           /* launch / device error (no device, bad ptr..) */
} mvsd_status;

typedef enum { MVSD_F32 = 0, MVSD_BF16 = 1 } mvsd_dtype;
typedef enum { MVSD_CHANNELS_LAST = 0, MVSD_CHANNELS_FIRST = 1 } mvsd_layout;
typedef enum {
  MVSD_BP_MEAN = 0,      /* sum over views / (count + 1e-8), 0 where count==0 */
  MVSD_BP_SUM = 1,       /* partial sums + counts (view-sharded multi-GPU)    */
  MVSD_BP_PER_VIEW = 2   /* un-aggregated per-view volume (reference API)     */
} mvsd_bp_mode;

/* ---- library info ------------------------------------------------------ */
int mvsd_abi_version(void);
const char* mvsd_build_info(void);          /* "sm_100a, nvcc 12.9, ..."     */
const char* mvsd_status_string(int status);
const char* mvsd_last_error(void);          /* thread-local, never NULL      */
/* TEST HOOK, not part of the drop-in contract and never called on the product
 * path (the host layer, bench.py and smoke() do not use it): selects which of
 * the built plane-sweep backward kernels serves k in {1,2} so the parity tests
 * can exercise both.  key 5: 0 = default (run-merging kernels: row hand-off
 * for bf16 features, lean kernel for fp32 features), 1 = the generic
 * pixel-per-warp kernel that otherwise serves k = 3, 4.  Results agree to fp32
 * summation order.  Process-wide atomic; returns the previous value, or -1 for
 * an unknown key (keys 0..7; only 5 is read).                                */
int mvsd_set_tuning(int key, int value);
/* Number of kernel launches issued through this library by the calling
 * process since load (bench.py's gpu_launches counter).                      */
int64_t mvsd_launch_count(void);

/* ---- layout helpers ----------------------------------------------------- */
/* [V,C,H,W] fp32 contiguous (what the reference's FPN emits, mvsdet.py:373-376)
 * -> nhwc of dst_dtype. */
int mvsd_pack_nchw_to_nhwc(const float* src, void* dst, int dst_dtype,
                           int V, int C, int H, int W, void* stream);
/* nhwc fp32 -> [V,C,H,W] fp32; accumulate != 0 adds into dst. */
int mvsd_unpack_nhwc_to_nchw(const float* src, float* dst, int accumulate,
                             int V, int C, int H, int W, void* stream);

/* ---- a1, a2, a8: per-scene camera geometry in one launch ----------------- *
 * Replaces, per scene, mvsdet.py:43-104 + :432-434 (nearest-pose ids),
 * :249-264 (collect_proj), mvs_models/module.py:116-118 (src_proj @
 * inverse(ref_proj)) and :1124-1156 (_compute_projection).  The HOST keeps two
 * ATen calls whose bits the variance volume depends on (DESIGN.md 6a):
 * ref_proj = K_feat @ w2c and inverse(ref_proj); everything else is here.
 *   w2c       [V,4,4] fp32 world-to-camera extrinsics (img_meta lidar2img)
 *   k_feat    [4,4] (per_view_k = 0) or [V,4,4] (per_view_k = 1) fp32
 *             feature-level intrinsics: rows 0-1 already divided by
 *             ratio = ori_h / (img_h / stride) (mvsdet.py:422-428)
 *   ref_proj  [V,4,4] fp32, inv_ref [V,4,4] fp32 = inverse(ref_proj)
 *   k         neighbours per view, <= min(4, V-1) (reference: min(2, V-1))
 *   ref_begin, n_ref   reference views [ref_begin, ref_begin+n_ref) whose rows
 *             are produced (view sharding; 0, V for a whole scene)
 * Outputs (device): nbr_ids [n_ref,k] int32 (nearest first, self excluded,
 * indices into the V views), hom [n_ref,k,12] fp32, projection [n_ref,3,4].
 * V <= 1024.  Rounding reproduces ATen's CPU matmul kernels (csrc/scene_setup.cu). */
int mvsd_scene_setup(const float* w2c, const float* k_feat, int per_view_k,
                     const float* ref_proj, const float* inv_ref,
                     int32_t* nbr_ids, float* hom, float* projection,
                     int V, int k, int ref_begin, int n_ref, void* stream);

/* ---- a3+a4: fused plane-sweep variance ---------------------------------- *
 * Replaces mvsdet.py:439-467 (ref_volume repeat, k x homo_warping
 * [mvs_models/module.py:105-146], sum / square-sum, variance).
 *   feat     nhwc [V,H,W,C] of feat_dtype
 *   nbr_ids  [V,k] int32, neighbour view of each reference view (mvsdet.py:432-434)
 *   hom      [V,k,12] fp32: rows of rot (9) then trans (3) of
 *            P_nbr @ inverse(P_ref) (module.py:116-118)
 *   depth_values [V,D] fp32 (mvsdet.py:450)
 *   out      variance, [V,D,H,W,C] (MVSD_CHANNELS_LAST) of out_dtype
 * k may be 0..4 (k=0: a single view, variance is exactly 0).
 * View sharding: V counts the REFERENCE views of this call; reference view v
 * reads feat[ref_begin + v] while nbr_ids index feat directly, so a rank can
 * sweep a slice [ref_begin, ref_begin+V) of a scene whose feature maps are all
 * resident (ref_begin = 0 for a whole scene).
 * n_feat_views = number of views feat holds: ref_begin + V must not exceed it
 * (MVSD_ERR_INVALID_ARG), and a neighbour id outside [0, n_feat_views) is never
 * dereferenced -- that neighbour contributes no sample (forward) and receives
 * no gradient (backward), like a warp that falls outside the map.            */
int mvsd_plane_sweep_fwd(const void* feat, int feat_dtype,
                         const int32_t* nbr_ids, const float* hom,
                         const float* depth_values,
                         void* out, int out_dtype, int out_layout,
                         int V, int C, int D, int H, int W, int k, int ref_begin,
                         int n_feat_views, void* stream);
/* Backward of the above (what autograd computes through mvsdet.py:439-467):
 *   g_out   dL/dvariance, same layout as `out`, of g_dtype
 *   g_feat  nhwc fp32, same extent as feat; contributions are ADDED (caller
 *           zero-fills). */
int mvsd_plane_sweep_bwd(const void* g_out, int g_dtype, int g_layout,
                         const void* feat, int feat_dtype,
                         const int32_t* nbr_ids, const float* hom,
                         const float* depth_values, float* g_feat,
                         int V, int C, int D, int H, int W, int k, int ref_begin,
                         int n_feat_views, void* stream);

/* Deterministic form of mvsd_plane_sweep_bwd (bit-reproducible gradients): the
 * contributions are added as signed 64-bit fixed point with 32 fractional bits
 * (integer REDs are order-independent; resolution 2.3e-10, |values| < 2^31) into
 * g_feat_q (nhwc int64, extent of feat, caller zero-fills); mvsd_fixed_to_float
 * converts the sums back (n elements, one rounding each).  Un-merged pixel-per-warp
 * scatter with scalar 64-bit REDs: ~8x the time of mvsd_plane_sweep_bwd (a whole
 * scene forward + backward: 7.3 ms instead of 1.2 ms).  Opt-in reproducibility mode;
 * not the benchmarked path. */
int mvsd_plane_sweep_bwd_det(const void* g_out, int g_dtype, int g_layout,
                             const void* feat, int feat_dtype,
                             const int32_t* nbr_ids, const float* hom,
                             const float* depth_values, int64_t* g_feat_q,
                             int V, int C, int D, int H, int W, int k, int ref_begin,
                             int n_feat_views, void* stream);
int mvsd_fixed_to_float(const int64_t* src, float* dst, int64_t n, void* stream);

/* Per-pixel depth hypotheses: homo_warping's [B,D,H,W] depth_values branch
 * (mvs_models/module.py:130-133) in the fused sweep, e.g. a narrow second sweep
 * around the hypotheses of mvsd_depth_topk_fwd.  Same arguments and semantics as
 * mvsd_plane_sweep_fwd / _bwd / _bwd_det, except that depth_values is
 * [V,D,H,W] fp32 contiguous: plane d of pixel (x, y) of reference view v lies at
 * depth_values[((v*D + d)*H + y)*W + x].  A NaN depth gives no sample.  A map
 * that is constant per (v, d) gives the bits of the per-view call (forward and
 * deterministic backward; the fp32-RED backward to summation order). */
int mvsd_plane_sweep_fwd_px(const void* feat, int feat_dtype,
                            const int32_t* nbr_ids, const float* hom,
                            const float* depth_values,
                            void* out, int out_dtype, int out_layout,
                            int V, int C, int D, int H, int W, int k, int ref_begin,
                            int n_feat_views, void* stream);
int mvsd_plane_sweep_bwd_px(const void* g_out, int g_dtype, int g_layout,
                            const void* feat, int feat_dtype,
                            const int32_t* nbr_ids, const float* hom,
                            const float* depth_values, float* g_feat,
                            int V, int C, int D, int H, int W, int k, int ref_begin,
                            int n_feat_views, void* stream);
int mvsd_plane_sweep_bwd_det_px(const void* g_out, int g_dtype, int g_layout,
                                const void* feat, int feat_dtype,
                                const int32_t* nbr_ids, const float* hom,
                                const float* depth_values, int64_t* g_feat_q,
                                int V, int C, int D, int H, int W, int k, int ref_begin,
                                int n_feat_views, void* stream);

/* ---- f4: group-wise correlation cost volume over the same sweep ----------- *
 * The optional cost volume of SURVEY.md 8(f) rank 4; in the reference it is the
 * inline arithmetic of mvs_models/lss_fpn.py:485-506 (a branch no shipped config
 * reaches), here with MVSDet's own warp (mvs_models/module.py:105-146):
 *   out[v,j,d,y,x,g] = mean_{c in group g} feat[ref_begin+v,y,x,c] * warped_j[v,c,d,y,x]
 * for neighbour j = 0..k-1 and num_groups contiguous channel groups of
 * C / num_groups channels (4, 8, 16, 32, 64 or 128 per group).
 *   out   [V,k,D,H,W,num_groups] fp32 (groups innermost); a sample with all four
 *         taps outside the map gives 0.  feat, nbr_ids, hom, depth_values,
 *         ref_begin, n_feat_views: as for mvsd_plane_sweep_fwd; k >= 1.
 * Backward: g_out has out's layout; g_feat (nhwc fp32, extent of feat) is ADDED to. */
int mvsd_plane_sweep_groupcorr_fwd(const void* feat, int feat_dtype,
                                   const int32_t* nbr_ids, const float* hom,
                                   const float* depth_values, float* out,
                                   int V, int C, int D, int H, int W, int k, int num_groups,
                                   int ref_begin, int n_feat_views, void* stream);
int mvsd_plane_sweep_groupcorr_bwd(const float* g_out, const void* feat, int feat_dtype,
                                   const int32_t* nbr_ids, const float* hom,
                                   const float* depth_values, float* g_feat,
                                   int V, int C, int D, int H, int W, int k, int num_groups,
                                   int ref_begin, int n_feat_views, void* stream);
/* The same with per-pixel depth hypotheses [V,D,H,W] fp32 contiguous
 * (mvs_models/module.py:130-133; layout as for mvsd_plane_sweep_fwd_px). */
int mvsd_plane_sweep_groupcorr_fwd_px(const void* feat, int feat_dtype,
                                      const int32_t* nbr_ids, const float* hom,
                                      const float* depth_values, float* out,
                                      int V, int C, int D, int H, int W, int k, int num_groups,
                                      int ref_begin, int n_feat_views, void* stream);
int mvsd_plane_sweep_groupcorr_bwd_px(const float* g_out, const void* feat, int feat_dtype,
                                      const int32_t* nbr_ids, const float* hom,
                                      const float* depth_values, float* g_feat,
                                      int V, int C, int D, int H, int W, int k, int num_groups,
                                      int ref_begin, int n_feat_views, void* stream);
/* Deterministic form of mvsd_plane_sweep_groupcorr_bwd / _bwd_px (bit-reproducible
 * gradients), as mvsd_plane_sweep_bwd_det is for the variance: same arguments and
 * checks, except that the contributions are added as signed 64-bit fixed point with
 * 32 fractional bits (resolution 2.3e-10, |values| < 2^31; integer REDs are
 * order-independent) into g_feat_q (nhwc int64, extent of feat, caller zero-fills);
 * mvsd_fixed_to_float converts the sums back.  Always the un-merged pixel-per-warp
 * scatter with scalar 64-bit REDs: opt-in reproducibility mode, not the fast path. */
int mvsd_plane_sweep_groupcorr_bwd_det(const float* g_out, const void* feat, int feat_dtype,
                                       const int32_t* nbr_ids, const float* hom,
                                       const float* depth_values, int64_t* g_feat_q,
                                       int V, int C, int D, int H, int W, int k, int num_groups,
                                       int ref_begin, int n_feat_views, void* stream);
int mvsd_plane_sweep_groupcorr_bwd_det_px(const float* g_out, const void* feat, int feat_dtype,
                                          const int32_t* nbr_ids, const float* hom,
                                          const float* depth_values, int64_t* g_feat_q,
                                          int V, int C, int D, int H, int W, int k, int num_groups,
                                          int ref_begin, int n_feat_views, void* stream);

/* ---- a3 alone: homo_warping (mvs_models/module.py:105-146) --------------- *
 *   src  nhwc [B,H,W,C]; hom [B,12]; out [B,D,H,W,C];
 *   depth_values [B,D], or per-pixel [B,D,H,W] when depth_per_pixel != 0
 *   (module.py:130-133; MVSDet itself only uses the [B,D] form).             */
int mvsd_homo_warp_fwd(const void* src, int src_dtype, const float* hom,
                       const float* depth_values, void* out, int out_dtype,
                       int out_layout, int B, int C, int D, int H, int W,
                       int depth_per_pixel, void* stream);
int mvsd_homo_warp_bwd(const void* g_out, int g_dtype, int g_layout,
                       const float* hom, const float* depth_values,
                       float* g_src, int B, int C, int D, int H, int W,
                       int depth_per_pixel, void* stream);
/* Deterministic form of mvsd_homo_warp_bwd (bit-reproducible gradients): same arguments
 * and checks (messages name mvsd_homo_warp_bwd_det), both depth forms, fp32 or bf16
 * g_out, except that the contributions are added as signed 64-bit fixed point with 32
 * fractional bits (resolution 2.3e-10, |values| < 2^31; integer REDs are
 * order-independent) into g_src_q (nhwc int64, extent of src, caller zero-fills);
 * mvsd_fixed_to_float converts the sums back. */
int mvsd_homo_warp_bwd_det(const void* g_out, int g_dtype, int g_layout,
                           const float* hom, const float* depth_values,
                           int64_t* g_src_q, int B, int C, int D, int H, int W,
                           int depth_per_pixel, void* stream);

/* ---- a5-a7: softmax / sigmoid / top-k / depth expectation ---------------- *
 * Replaces mvsdet.py:470-482, sample_depth_prob (:266-283) and
 * compute_avg_depth (:298-317).
 *   cost_out  the cost-regularisation output, logical [V,2,D,H,W]; element
 *             strides s_v, s_c, s_d, s_p (pixel) let it be NCDHW-contiguous
 *             (s_c=D*H*W, s_d=H*W, s_p=1) or channels_last_3d (s_c=1,
 *             s_d=2*H*W, s_p=2)
 *   prob_volume, off_pred  [V,D,H,W] fp32 (either may be NULL)
 *   est_depth, est_dens    [V,T,H,W] fp32;  est_idx [V,T,H,W] int64
 *   depth_coding           [V,H,W] fp32 (may be NULL)
 * Top-k order: descending probability, ties -> lowest plane index first.
 * A pixel with NaN probabilities gets the lowest planes not yet taken (indices
 * stay distinct).  depth_coding is summed in plane order (the reference sums
 * in probability-sorted order): equal to fp32 summation rounding, ~1e-6.
 * raw != 0: channel 0 of cost_out already holds probabilities and channel 1
 * offsets in [0,1] (the stand-alone sample_depth_prob / compute_avg_depth API);
 * softmax / sigmoid are skipped, forward and backward.
 * NVS-branch epilogue (all optional, NULL = skip):
 *   ray_intrinsics  [4,4] or (ray_per_view) [V,4,4] feature-level intrinsics
 *   opacity         [V,H,W] = max_d prob_volume            (mvsdet.py:579)
 *   depth_scale     [V,H,W] z of the unit ray through each pixel
 *                   (compute_depth_scale[_MultiIntrin], mvsdet.py:1158-1218)
 *   est_ray_depth   [V,T,H,W] = est_depth / (depth_scale + 1e-8)     (:494)
 *   ray_depth_coding [V,H,W]  = depth_coding / (depth_scale + 1e-8)  (:583)   */
int mvsd_depth_topk_fwd(const float* cost_out, int64_t s_v, int64_t s_c,
                        int64_t s_d, int64_t s_p,
                        float* prob_volume, float* off_pred, float* est_depth,
                        float* est_dens, int64_t* est_idx, float* depth_coding,
                        const float* ray_intrinsics, int ray_per_view,
                        float* opacity, float* depth_scale, float* est_ray_depth,
                        float* ray_depth_coding,
                        float near, float interval, int raw,
                        int V, int D, int H, int W, int T, void* stream);
/* Backward: any of the upstream gradients may be NULL (treated as 0).
 *   g_cost_out  [V,2,D,H,W] fp32 contiguous, fully overwritten.              */
int mvsd_depth_topk_bwd(const float* cost_out, int64_t s_v, int64_t s_c,
                        int64_t s_d, int64_t s_p, const int64_t* est_idx,
                        const float* g_prob_volume, const float* g_off_pred,
                        const float* g_est_depth, const float* g_est_dens,
                        const float* g_depth_coding,
                        const float* ray_intrinsics, int ray_per_view,
                        const float* g_est_ray_depth, const float* g_ray_depth_coding,
                        float* g_cost_out,
                        float near, float interval, int raw,
                        int V, int D, int H, int W, int T, void* stream);
/* The top-k epilogue over per-pixel depth hypotheses, e.g. the fine cost volume
 * of a second sweep around est_depth (mvsd_plane_sweep_fwd_px).  Arguments as
 * mvsd_depth_topk_fwd / _bwd, except that the planes d*interval + near are
 * replaced by
 *   depth_values  [V,D,H,W] fp32 contiguous (required): z_d of each pixel, in
 *                 any order along D (est_idx indexes this axis)
 *   interval_map  [V,H,W] fp32 contiguous offset scale I per pixel, or NULL:
 *                 I = interval
 * depth_d = z_d + off_d*I (two roundings).  Selection, NaN rule, expectation
 * order and NVS epilogue are those of mvsd_depth_topk_fwd; a NaN z_d propagates
 * into the depths that use it.  Planes z_d = fl(fl(d*interval) + near) with
 * I = interval (scalar or constant map) give the per-view call's bits, forward
 * and g_cost_out.
 * Backward, in addition to g_cost_out (both optional, fully overwritten):
 *   g_depth_values [V,D,H,W]  dL/dz_d = g_coding*p_d + sum_t [d == idx_t] g_est_depth_t
 *   g_interval_map [V,H,W]    dL/dI = g_coding*sum_d p_d off_d + sum_t g_est_depth_t off_idx_t
 *                             (requires interval_map)
 * where g_coding and g_est_depth include the ray-depth terms. */
int mvsd_depth_topk_fwd_px(const float* cost_out, int64_t s_v, int64_t s_c,
                           int64_t s_d, int64_t s_p,
                           const float* depth_values, const float* interval_map, float interval,
                           float* prob_volume, float* off_pred, float* est_depth,
                           float* est_dens, int64_t* est_idx, float* depth_coding,
                           const float* ray_intrinsics, int ray_per_view,
                           float* opacity, float* depth_scale, float* est_ray_depth,
                           float* ray_depth_coding,
                           int raw, int V, int D, int H, int W, int T, void* stream);
int mvsd_depth_topk_bwd_px(const float* cost_out, int64_t s_v, int64_t s_c,
                           int64_t s_d, int64_t s_p, const int64_t* est_idx,
                           const float* depth_values, const float* interval_map, float interval,
                           const float* g_prob_volume, const float* g_off_pred,
                           const float* g_est_depth, const float* g_est_dens,
                           const float* g_depth_coding,
                           const float* ray_intrinsics, int ray_per_view,
                           const float* g_est_ray_depth, const float* g_ray_depth_coding,
                           float* g_cost_out, float* g_depth_values, float* g_interval_map,
                           int raw, int V, int D, int H, int W, int T, void* stream);

/* compute_depth_scale / compute_depth_scale_MultiIntrin alone (mvsdet.py:1158-1218):
 * depth_scale [V,H,W] from [4,4] or (per_view) [V,4,4] feature-level intrinsics. */
int mvsd_ray_depth_scale(const float* intrinsics, int per_view, float* depth_scale,
                         int V, int H, int W, void* stream);
/* process_rgb_raw (mvsdet.py:319-333): bilinear 1/4 down-sampling
 * (align_corners=False) of rgb [V,3,H,W] fp32 for the views src_ids [n_ids]
 * int64 (NULL = views 0..n_ids-1), cropped to [h,w], written as [n_ids,h*w,3]. */
int mvsd_rgb_downsample4(const float* rgb, const int64_t* src_ids, int n_ids, float* out,
                         int V, int H, int W, int h, int w, void* stream);

/* ---- a10+a11: probabilistic voxel back-projection ------------------------ *
 * Replaces backproject_Weigh (mvsdet.py:1372-1492) and the view aggregation
 * (mvsdet.py:511-515, :681-682).
 *   feat        nhwc [V,feat_h,feat_w,C] of feat_dtype; only rows < h and
 *               columns < w are addressed (the reference crops, mvsdet.py:499)
 *   points      [3,N] fp32 voxel centres (get_points, mvsdet.py:1316-1327)
 *   projection  [V,3,4] fp32 (_compute_projection, mvsdet.py:1124-1156)
 *   depth, prob hypotheses of logical shape [V,h,w,T] addressed with element
 *               strides dp_sv, dp_sy, dp_sx, dp_st (same strides for both)
 *   vs_z        voxel_size[2] (depth-test half width, mvsdet.py:1407-1408)
 *   mode        mvsd_bp_mode
 *   out         MEAN/SUM: [N,C] (MVSD_CHANNELS_LAST) or [C,N] (CHANNELS_FIRST)
 *               PER_VIEW: [V,N,C], caller zero-fills
 *   count       [N] int32, number of valid views per voxel (MEAN/SUM; may be
 *               NULL in PER_VIEW)
 *   valid       [V,N] uint8 per-view mask (may be NULL)
 *   weight      [V,N] fp32 per-view weight (may be NULL)                      */
int mvsd_backproject_fwd(const void* feat, int feat_dtype, int feat_h, int feat_w,
                         const float* points, const float* projection,
                         const float* depth, const float* prob,
                         int64_t dp_sv, int64_t dp_sy, int64_t dp_sx, int64_t dp_st,
                         float vs_z, int mode, float* out, int out_layout,
                         int32_t* count, uint8_t* valid, float* weight,
                         int V, int C, int h, int w, int T, int N, void* stream);
/* Backward.
 *   g_out   MEAN/SUM: dL/dout, same layout as out; PER_VIEW: [V,N,C]
 *   count   MEAN: the forward's count (s_u = 1/(count+1e-8)); else NULL
 *   g_feat  nhwc fp32 [V,feat_h,feat_w,C], ADDED into
 *   g_pn    dL/d(normalised hypothesis probability), same strides as prob,
 *           ADDED into (caller zero-fills); feed to mvsd_prob_norm_bwd.       */
int mvsd_backproject_bwd(const float* g_out, int g_layout, int mode,
                         const int32_t* count,
                         const void* feat, int feat_dtype, int feat_h, int feat_w,
                         const float* points, const float* projection,
                         const float* depth, const float* prob,
                         int64_t dp_sv, int64_t dp_sy, int64_t dp_sx, int64_t dp_st,
                         float vs_z, float* g_feat, float* g_pn,
                         int V, int C, int h, int w, int T, int N, void* stream);
/* pn = prob / sum_T prob (mvsdet.py:1395-1396) backward: g_pn -> g_prob, all
 * three addressed with the dp_* strides; overwrites g_prob on the [h,w] crop. */
/* Deterministic form of mvsd_backproject_bwd, MVSD_BP_MEAN only: g_feat_q / g_pn_q are
 * 64-bit fixed-point accumulators (see mvsd_plane_sweep_bwd_det; g_pn_q has prob's
 * strides and may be NULL); convert with mvsd_fixed_to_float before mvsd_prob_norm_bwd. */
int mvsd_backproject_bwd_det(const float* g_out, int g_layout, const int32_t* count,
                             const void* feat, int feat_dtype, int feat_h, int feat_w,
                             const float* points, const float* projection,
                             const float* depth, const float* prob,
                             int64_t dp_sv, int64_t dp_sy, int64_t dp_sx, int64_t dp_st,
                             float vs_z, int64_t* g_feat_q, int64_t* g_pn_q,
                             int V, int C, int h, int w, int T, int N, void* stream);
/* Deterministic form of mvsd_backproject_bwd for MVSD_BP_SUM (either layout) and
 * MVSD_BP_PER_VIEW (channels-last): same arguments and checks (messages name
 * mvsd_backproject_bwd_det_mode; count is unused), except that g_feat_q (nhwc int64,
 * extent of feat) and g_pn_q (int64, prob's strides, may be NULL) take the
 * contributions as signed 64-bit fixed point with 32 fractional bits (resolution
 * 2.3e-10, |values| < 2^31; integer REDs are order-independent); the caller
 * zero-fills both and converts them with mvsd_fixed_to_float.  MVSD_BP_MEAN is
 * MVSD_ERR_UNSUPPORTED here: its deterministic form is mvsd_backproject_bwd_det. */
int mvsd_backproject_bwd_det_mode(const float* g_out, int g_layout, int mode,
                                  const int32_t* count,
                                  const void* feat, int feat_dtype, int feat_h, int feat_w,
                                  const float* points, const float* projection,
                                  const float* depth, const float* prob,
                                  int64_t dp_sv, int64_t dp_sy, int64_t dp_sx, int64_t dp_st,
                                  float vs_z, int64_t* g_feat_q, int64_t* g_pn_q,
                                  int V, int C, int h, int w, int T, int N, void* stream);
int mvsd_prob_norm_bwd(const float* prob, const float* g_pn, float* g_prob,
                       int64_t dp_sv, int64_t dp_sy, int64_t dp_sx, int64_t dp_st,
                       int V, int h, int w, int T, void* stream);
/* After an all-reduce of SUM partials: out = count ? sum/(count+1e-8) : 0.
 * In place is allowed (out == sum).                                           */
int mvsd_voxel_normalize(const float* sum, const int32_t* count, float* out,
                         int layout, int C, int N, void* stream);

/* View-sharded scene (reference views split over `world` GPUs of one NVLink domain):
 * the sum over views of mvsdet.py:511-515 / :681-682 across ranks, fused with the
 * normalisation, over peer memory instead of an all-reduce.  part_ptrs / out_ptrs are
 * DEVICE arrays of `world` peer pointers (e.g. torch symmetric memory
 * buffer_ptrs_dev): each peer buffer is [C*N] fp32 (partial sums in `layout`) followed
 * by [N] int32 (partial valid counts); the result buffers get [C*N] fp32 volume_mean
 * followed by [N] int32 counts, identical bits on every rank.  The caller puts a
 * cross-rank barrier before (all partials written) and after (all results delivered)
 * this call.  count_local: [N] int32 scratch on this rank.                         */
int mvsd_voxel_reduce_p2p(const void* const* part_ptrs, void* const* out_ptrs,
                          int32_t* count_local, int world, int rank, int layout, int C, int N,
                          void* stream);

/* Backward of a view-sharded scene: the owner of each reference view adds the gradient
 * contributions its peers accumulated for that view as a HALO (neighbour) view
 * (mvsd_plane_sweep_bwd scatters into block + halo maps).  g_ptrs: DEVICE array of `world`
 * peer pointers to the ranks' fp32 gradient buffers [V_local][view_elems] (block views
 * first).  CSR pull table of this rank: owned view d receives sources
 * pull_sources[2*q] = peer rank, pull_sources[2*q+1] = view index in that peer's buffer, for
 * q in [pull_offsets[d], pull_offsets[d+1]).  Deterministic (table order).  The caller puts
 * a cross-rank barrier before (all backward kernels done) and after (before the buffers are
 * zeroed again) this call.                                                              */
int mvsd_halo_reduce_p2p(void* const* g_ptrs, const int32_t* pull_offsets,
                         const int32_t* pull_sources, int world, int rank, int n_own,
                         int64_t view_elems, void* stream);
/* The same pull over the int64 fixed-point accumulators of the deterministic backwards
 * (mvsd_plane_sweep_bwd_det, mvsd_backproject_bwd_det; 32 fractional bits): same arguments,
 * checks and grid (messages name halo_reduce_p2p_fixed), except that the peer buffers are
 * int64 [V_local][view_elems] and the owner adds its peers' rows with integer adds.  Integer
 * addition does not depend on order, so after mvsd_fixed_to_float the owned rows are the bits
 * of the single-GPU deterministic gradient, whatever the number of ranks and the split.     */
int mvsd_halo_reduce_p2p_fixed(void* const* g_ptrs, const int32_t* pull_offsets,
                               const int32_t* pull_sources, int world, int rank, int n_own,
                               int64_t view_elems, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* MVSDET_B200_H_ */
