/*
 * vtgs.h -- C ABI of the B200-native differentiable Gaussian-splatting hot path.
 *
 * This is the drop-in boundary for the one path VTGaussian-SLAM spends its time in:
 * the rasteriser binding that the reference imports as the pip module
 * `diff_gaussian_rasterization` (reference requirements.txt:18; import sites
 * src/vtgaussian_slam.py:38, utils/recon_helpers.py:2, utils/eval_helpers.py:17) and
 * calls at src/vtgaussian_slam.py:461,466,747 and utils/eval_helpers.py:240,247,431,443.
 * That module's pybind layer exports `_C.rasterize_gaussians`,
 * `_C.rasterize_gaussians_backward` and `_C.mark_visible`; the three entry points
 * vtgs_forward / vtgs_backward / vtgs_mark_visible below are what a maintainer binds in
 * their place (see INTEGRATION.md).  The fused entry points further down replace the
 * pure-PyTorch work the reference wraps around every rasteriser call
 * (utils/slam_helpers.py:127-160,217-234,255-287,323-385; src/vtgaussian_slam.py:407-689,
 * 180-187) with single launches.
 *
 * Rules of the ABI
 *   - plain C: raw device pointers, sizes, PODs.  No torch / C++ types, no exceptions.
 *   - every function returns 0 on success, a negative VTGS_E_* code otherwise;
 *     vtgs_last_error() returns a thread-local message for the last failure.
 *   - every function only enqueues work on `stream` (a cudaStream_t passed as void*);
 *     nothing synchronises the device or the host, so call sequences are CUDA-graph
 *     capturable.  The number of (tile, Gaussian) pairs R is never read back by the
 *     library: the caller provides `pair_capacity` slots and polls
 *     VtgsCounters.overflow when convenient.
 *   - all arrays are caller-owned device memory, fp32/int32 contiguous, layouts as the
 *     reference passes them (AoS [N,3] / [N,4] / [C,H,W]).
 *   - re-entrant per (VtgsBuffers, stream); no hidden global state.
 */
#ifndef VTGS_H_
#define VTGS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VTGS_API __attribute__((visibility("default")))
#else
#define VTGS_API
#endif

#define VTGS_ABI_VERSION 4

/* ---- named constants of the splatting arithmetic (SURVEY.md Appendix A.0) ---------- */
#define VTGS_TILE            16          /* BLOCK_X = BLOCK_Y                          */
#define VTGS_NEAR_CULL       0.2f        /* cull p_view.z <= 0.2                       */
#define VTGS_FRUSTUM_MULT    1.3f        /* clamp of t.x/t.z in the EWA Jacobian       */
#define VTGS_LOWPASS         0.3f        /* screen-space dilation                      */
#define VTGS_LAMBDA_FLOOR    0.1f
#define VTGS_ALPHA_MAX       0.99f
#define VTGS_ALPHA_MIN       (1.0f / 255.0f)
#define VTGS_T_MIN           0.0001f
#define VTGS_EPS_W           0.0000001f
#define VTGS_RADIUS_SIGMA_MULT_DEFAULT 3.0f   /* the fork's "smallerGSradii" delta is
                                                  unknown offline: runtime parameter   */

/* ---- error codes -------------------------------------------------------------------- */
#define VTGS_OK               0
#define VTGS_E_INVALID       -1          /* bad argument                               */
#define VTGS_E_CUDA          -2          /* a CUDA runtime call failed                 */
#define VTGS_E_UNSUPPORTED   -3          /* e.g. SH colours, cov3D_precomp             */

/*
 * Camera / raster settings.  Mirrors GaussianRasterizationSettings as built by
 * setup_camera (reference utils/recon_helpers.py:14-26): matrices are the flat
 * row-vector-convention arrays the reference passes (viewmatrix = w2c^T, projmatrix =
 * (proj*w2c)^T), i.e. p_view.x = m[0]x + m[4]y + m[8]z + m[12].
 * tile_row_begin/end select a band of 16-px tile rows (multi-GPU tracking shards the
 * image by tile bands); 0,0 means "all rows".
 */
typedef struct VtgsCamera {
    int32_t image_width;
    int32_t image_height;
    float   tanfovx;
    float   tanfovy;
    float   viewmatrix[16];
    float   projmatrix[16];
    float   bg[3];
    float   scale_modifier;
    float   radius_sigma_mult;
    int32_t tile_row_begin;
    int32_t tile_row_end;
} VtgsCamera;

/* Device-side counters; the library writes them, the caller may read them lazily. */
typedef struct VtgsCounters {
    uint32_t num_rendered;      /* R = sum of tiles_touched (before clamping)           */
    uint32_t overflow;          /* 1 if R > pair_capacity (results are then truncated)  */
    uint32_t max_tile_pairs;    /* longest per-tile list                                */
    uint32_t reserved0;
    /* pose of the fused path, written by the library each fused forward (device-resident so
     * that a captured CUDA graph follows the optimiser): p_cam = pose_R * p + pose_t        */
    float    pose_R[9];
    float    pose_t[3];
    float    pose_q[4];         /* cam quaternion after F.normalize (once)                  */
    float    pose_qnorm[2];     /* |q_unnorm|, |F.normalize(q)| (the two normalisations)    */
    float    reserved1[10];
} VtgsCounters;

/*
 * Workspace handed to forward and kept alive by the caller until backward (the
 * equivalent of the reference binding's geomBuffer / binningBuffer / imgBuffer).
 * Sizes come from vtgs_workspace_query.
 */
typedef struct VtgsBuffers {
    void*         geom;           /* N records of VTGS_GEOM_RECORD_BYTES                  */
    uint32_t*     tiles_touched;  /* [N]                                                   */
    uint32_t*     tile_counts;    /* [tiles + 3]  scratch (zeroed by forward); word [tiles] counts band_cand, [tiles + 1] and
                                     [tiles + 2] hold the bit patterns of max |colour| of the rendered Gaussians and of
                                     max |dL/dpixel| (the scales of the deterministic gradient accumulation)          */
    uint32_t*     tile_ranges;    /* [tiles][2] = {begin, end} into point_list             */
    uint64_t*     pair_keys;      /* [pair_capacity] depth_bits<<32 | gaussian id<<8 | region mask */
    uint32_t*     point_list;     /* [pair_capacity] sorted Gaussian ids                   */
    float*        final_T;        /* [H*W]                                                 */
    uint32_t*     n_contrib;      /* [H*W]                                                 */
    float*        grad_geom;      /* [N][VTGS_GRAD_GEOM_FLOATS] scratch of backward; must be zero on
                                     entry to a backward and is left zeroed by it          */
    VtgsCounters* counters;       /* 1                                                     */
    void*         region_pairs;   /* [8 * pair_capacity] uint32x2 {Gaussian id, 1-based position in the tile
                                     list}: per-tile, per-8x4-pixel-region lists built by the sort kernel  */
    uint32_t*     region_cnt;     /* [tiles][8] length of each region list                 */
    uint32_t*     region_masks;   /* [8 * (pair_capacity + 32 tiles)] per (region, group of 32 splats, pixel
                                     lane): bit e = splat e of the group was blended into that pixel.  Written
                                     by the forward blend, consumed by the backward blend               */
    uint32_t*     region_done;    /* [tiles][8] groups of each region list the forward walked before every
                                     pixel of the region had saturated                                   */
    uint64_t      pair_capacity;
    uint8_t*      band_flags;     /* [ceil(N / 256)] optional (may be NULL).  Fused path with a tile-row band: per
                                     iteration the forward marks the 256-Gaussian blocks that can reach the band at the
                                     current pose; preprocess, scatter and backward-preprocess skip the others, so a
                                     rank's per-Gaussian work follows its band instead of N                        */
    uint32_t*     band_cand;      /* [ceil(N / 256)] optional, with band_flags: the marked blocks as a compact list (its
                                     length lives in tile_counts[tiles], zeroed with the counts)                  */
    uint32_t*     tile_order;     /* [tiles] optional (may be NULL).  The tile scan leaves the tiles of the render in
                                     descending order of list length; the sort and blend kernels take their tile from it,
                                     so the longest lists are started first (longest-processing-time-first scheduling of
                                     the blocks: the tail of a launch is filled with short tiles)                   */
    uint32_t      flags;          /* VTGS_BUF_*                                                                       */
    uint32_t      reserved;
} VtgsBuffers;

/* VtgsBuffers.flags.  VTGS_BUF_DETERMINISTIC: the backward blend splits every per-(region, splat) partial sum into a
 * coarse and a fine part on per-Gaussian power-of-two grids before the fp32 `red.global.add` into grad_geom.  Sums of
 * grid multiples that stay below 2^24 grid steps are EXACT in fp32, hence independent of the order in which the tiles'
 * warps arrive: every gradient of the backward is then bitwise reproducible run to run and across ranks, with the same
 * number of memory operations as without the flag.  The grids come from rigorous bounds of the sums (max |dL/dpixel| and
 * max |colour| measured on the device, the splat's opacity / conic / extent / tile count), so the exactness conditions
 * cannot be violated; 22 + (21 - log2 tiles) bits lie below the bound.  Upstream: float atomics in arbitrary order. */
#define VTGS_BUF_DETERMINISTIC 1u

#define VTGS_GEOM_RECORD_BYTES 64
#define VTGS_GRAD_GEOM_FLOATS  32   /* records of 16 floats without, 32 (20 used) with VTGS_BUF_DETERMINISTIC */

typedef struct VtgsWorkspaceSizes {
    uint64_t geom_bytes;
    uint64_t tiles_touched_bytes;
    uint64_t tile_counts_bytes;
    uint64_t tile_ranges_bytes;
    uint64_t pair_keys_bytes;
    uint64_t point_list_bytes;
    uint64_t final_T_bytes;
    uint64_t n_contrib_bytes;
    uint64_t grad_geom_bytes;
    uint64_t counters_bytes;
    uint64_t region_pairs_bytes;
    uint64_t region_cnt_bytes;
    uint64_t region_masks_bytes;
    uint64_t region_done_bytes;
    uint64_t band_flags_bytes;
    uint64_t band_cand_bytes;
    uint64_t tile_order_bytes;
    uint32_t tiles_x;
    uint32_t tiles_y;
} VtgsWorkspaceSizes;

/* ---- library ------------------------------------------------------------------------ */
VTGS_API int         vtgs_abi_version(void);
VTGS_API const char* vtgs_last_error(void);
VTGS_API const char* vtgs_build_info(void);        /* arch / flags the library was built with     */

VTGS_API int vtgs_workspace_query(int32_t image_width, int32_t image_height, int64_t num_gaussians,
                         uint64_t pair_capacity, VtgsWorkspaceSizes* sizes);

/*
 * Forward: replaces _C.rasterize_gaussians (K1..K5 of SURVEY.md section 2.3), the call behind the reference's
 * `Renderer(raster_settings=curr_data['cam'])(**rendervar)` (src/vtgaussian_slam.py:461, :466, :747;
 * utils/eval_helpers.py:240, :247, :431, :443, :728, :733; settings built at utils/recon_helpers.py:14-26).
 * num_gaussians < 2^32 (32-bit Gaussian ids, as in the reference's keys; below 2^24 the low key byte also carries the
 * splat's region mask, from 2^24 on it is re-derived from the record): VTGS_E_UNSUPPORTED beyond.
 *   means3D[N,3] scales[N,3] rotations[N,4] opacities[N] colors[N,3]  ->
 *   out_color[3,H,W]  out_depth[H,W]  radii[N]
 * Colours are precomputed (the reference never passes SHs: sh_degree = 0).
 */
VTGS_API int vtgs_forward(const VtgsCamera* cam, int64_t num_gaussians,
                 const float* means3D, const float* scales, const float* rotations,
                 const float* opacities, const float* colors,
                 float* out_color, float* out_depth, int32_t* radii,
                 VtgsBuffers* buf, void* stream);

/*
 * Backward: replaces _C.rasterize_gaussians_backward (K6, K7), reached from the reference's `loss.backward()`
 * (src/vtgaussian_slam.py:1889 tracking, :2686 mapping) through the rasteriser's autograd Function.
 *   dL_dout_color[3,H,W] + the forward's inputs and buffers ->
 *   dL_dmeans2D[N,3] (z = 0), dL_dcolors[N,3], dL_dopacity[N], dL_dmeans3D[N,3],
 *   dL_dscales[N,3], dL_drotations[N,4].  No gradient flows through out_depth or radii
 *   (as in the reference's "-w-depth" rasteriser).
 */
VTGS_API int vtgs_backward(const VtgsCamera* cam, int64_t num_gaussians,
                  const float* means3D, const float* scales, const float* rotations,
                  const float* opacities, const float* colors,
                  const float* dL_dout_color,
                  float* dL_dmeans2D, float* dL_dcolors, float* dL_dopacity,
                  float* dL_dmeans3D, float* dL_dscales, float* dL_drotations,
                  VtgsBuffers* buf, void* stream);

/* Replaces _C.mark_visible (upstream GaussianRasterizer.markVisible; not called by the reference, kept for the
 * drop-in surface): present[i] = (p_view.z > near cull). */
VTGS_API int vtgs_mark_visible(const VtgsCamera* cam, int64_t num_gaussians, const float* means3D,
                      uint8_t* present, void* stream);

/*
 * Parity/debug view of the binning stage in the reference's own representation:
 * point_list_keys[R] = (tile_id << 32) | float_bits(depth) in sorted order, as
 * cub::DeviceRadixSort leaves them in the reference's binningBuffer.
 */
VTGS_API int vtgs_export_sorted_keys(const VtgsCamera* cam, int64_t num_gaussians, const VtgsBuffers* buf,
                            uint64_t* keys_out, uint64_t keys_capacity, void* stream);

/* Geometry the forward computed, unpacked for parity checks:
 * means2D[N,2], depths[N], conic_opacity[N,4]. Any pointer may be NULL. */
VTGS_API int vtgs_export_geometry(int64_t num_gaussians, const VtgsBuffers* buf,
                         float* means2D, float* depths, float* conic_opacity, void* stream);

/* ===================================================================================== *
 *  Fused view-tied path (what get_loss + backward + Adam do per iteration)              *
 * ===================================================================================== */

/*
 * View-tied Gaussian parameters exactly as the reference's `params` dict stores them
 * (src/vtgaussian_slam.py:132-177): means3D[N,3], rgb_colors[N,3],
 * unnorm_rotations[N,4], logit_opacities[N,1], log_scales[N,1] (isotropic) or [N,3].
 */
typedef struct VtgsParams {
    const float* means3D;
    const float* rgb_colors;
    const float* unnorm_rotations;
    const float* logit_opacities;
    const float* log_scales;
    int32_t      log_scales_dim;   /* 1 (isotropic) or 3 */
    int32_t      pad_;
    int64_t      num_gaussians;
} VtgsParams;

/* Camera pose of the frame being rendered: the slices params['cam_unnorm_rots'][0,:,t]
 * and params['cam_trans'][0,:,t] (device pointers to 4 and 3 floats, any stride-1). */
typedef struct VtgsPose {
    const float* cam_unnorm_rot;   /* [4] (w,x,y,z), un-normalised, device                 */
    const float* cam_trans;        /* [3] device                                            */
    float        depth_row[4];     /* third row of curr_data['w2c'] used by
                                      get_depth_and_silhouette (utils/slam_helpers.py:217-234);
                                      {0,0,1,0} for the reference's relative poses          */
} VtgsPose;

/*
 * Fused forward for one view: transform_to_frame + transformed_params2rendervar +
 * transformed_params2depthplussilhouette + both rasteriser passes of get_loss
 * (src/vtgaussian_slam.py:432-466) as ONE six-channel pass.
 *   out_image7[7,H,W] = {r, g, b, depth, silhouette, depth^2, <unused>}: channel order
 *   is im[0..2] then depth_sil[0..2] of the reference.  Only 6 planes are written.
 *   radii[N] as the RGB pass would return them.
 *   With a tile-row band (VtgsCamera.tile_row_begin/end) only the band's rows of the planes are written and
 *   radii[i] is only guaranteed for Gaussians that touch the band (others may be reported as 0: they are
 *   rejected by a cheap conservative bound before the full projection).
 */
VTGS_API int vtgs_fused_forward(const VtgsCamera* cam, const VtgsParams* params, const VtgsPose* pose,
                       float* out_image6, int32_t* radii, VtgsBuffers* buf, void* stream);

/*
 * Tracking / mapping loss of get_loss (src/vtgaussian_slam.py:513-612,678-679) evaluated
 * on the six rendered planes against the frame, producing the scalar terms and
 * dL/d(image6) in place of autograd.
 *   mode 0: tracking   losses = sum|d|[mask] (depth), sum|rgb diff|[mask] (im)
 *   mode 1: mapping    losses = mean|d|[depth>0] (depth), 0.8*L1mean + 0.2*(1-SSIM) (im)
 * loss_terms[8] = {loss, w_im*im, w_depth*depth, mask_count, l1_im, ssim, depth_l1_mean, 0}.
 */
typedef struct VtgsLossConfig {
    int32_t mode;                   /* 0 tracking, 1 mapping                              */
    int32_t use_sil_for_loss;
    int32_t ignore_outlier_depth;   /* tracking: also mask |gt - d| (gt > 0) >= 50 * its median over the frame
                                       (reference src/vtgaussian_slam.py:525-528; exact lower median as
                                       torch.median, four 8-bit radix-select passes on the device).  With a tile-row
                                       band the median is a frame-wide quantity: pass `median_state` computed with
                                       vtgs_median_hist / an all-reduce / vtgs_median_pick (UNSUPPORTED otherwise)  */
    int32_t use_l1;
    float   sil_thres;
    float   w_im;
    float   w_depth;
    float   far_depth_thres;        /* <= 0: disabled                                     */
    const uint8_t* pixel_mask;      /* optional [H,W] bytes, tracking: pixels with 0 are masked out (the reference's
                                       overlap-visibility mask, :536-583, computed by the caller); NULL: none */
    const float*   sil_thres_dev;   /* optional device float: overrides sil_thres (the Replica threshold chosen on the
                                       device by vtgs_sil_select, so that a captured iteration follows it); NULL: none */
    const uint32_t* median_state;   /* optional: a finished radix-select state (vtgs_median_pick after pass 3), used
                                       instead of running the four passes inside vtgs_loss; NULL: none            */
} VtgsLossConfig;

VTGS_API int vtgs_loss(const VtgsCamera* cam, const VtgsLossConfig* cfg,
              const float* image6, const float* gt_rgb, const float* gt_depth,
              float* dL_dimage6 /* [4,H,W]: r,g,b,depth */, float* loss_terms /* [8] */,
              float* scratch /* vtgs_loss_scratch_floats() floats */, void* stream);
VTGS_API uint64_t vtgs_loss_scratch_floats(int32_t image_width, int32_t image_height, int32_t mode);

/*
 * Frame-wide median of depth_error = |gt - d| (gt > 0) (reference src/vtgaussian_slam.py:525-527, :757-758) by radix
 * select, in a form that shards: per pass, every rank histograms ITS rows (vtgs_median_hist, cam carries the tile-row
 * band), the first VTGS_MEDIAN_SUMMABLE_WORDS words of `state` are all-reduced (SUM, integers), and every rank picks the
 * same bin (vtgs_median_pick).  After pass 3 the state holds the median's bit pattern (NaN if any value was NaN, as
 * torch.median).  `state`: VTGS_MEDIAN_STATE_WORDS uint32, zero before pass 0.
 */
#define VTGS_MEDIAN_STATE_WORDS    264
#define VTGS_MEDIAN_SUMMABLE_WORDS 257
VTGS_API int vtgs_median_hist(const VtgsCamera* cam, const float* depth_plane, const float* gt_depth, int32_t pass,
                              uint32_t* state, void* stream);
VTGS_API int vtgs_median_pick(int64_t num_pixels_total, int32_t pass, uint32_t* state, void* stream);

/*
 * Replica's iteration-0 silhouette-threshold search (reference src/vtgaussian_slam.py:472-510): for the five
 * thresholds {0.990, 0.993, 0.995, 0.997, 0.999} the masked colour MSE over (silhouette > thr & depth > 0).
 *   vtgs_sil_ladder: sums10 = {sum of squared colour differences [5], masked pixel counts [5]} over the camera's
 *                    tile-row band (all-reduce the ten floats when the frame is sharded); scratch: the loss scratch;
 *   vtgs_sil_select: mse_i = sum_i / (3 count_i); *sil_thres_dev = the threshold of the smallest (first on ties,
 *                    index 0 if no pixel passes), *min_mse_dev = that MSE.
 */
VTGS_API int vtgs_sil_ladder(const VtgsCamera* cam, const float* image6, const float* gt_rgb, const float* gt_depth,
                             float* sums10, float* scratch, void* stream);
VTGS_API int vtgs_sil_select(const float* sums10, float* sil_thres_dev, float* min_mse_dev, void* stream);

/*
 * Non-presence mask of the reference's silhouette-driven Gaussian addition (add_new_gaussians_base_frame,
 * src/vtgaussian_slam.py:747-760) from a forward-only fused render:
 *   mask = (silhouette < sil_thres) | ((depth > gt) & (|gt - depth| (gt > 0) > 50 median))
 * median_state: a finished radix-select state of the same render (vtgs_median_hist / vtgs_median_pick).
 * mask_out[H,W] bytes; *count_dev (optional) receives the number of set pixels.
 */
VTGS_API int vtgs_nonpresence_mask(const VtgsCamera* cam, const float* image6, const float* gt_depth, float sil_thres,
                                   const uint32_t* median_state, uint8_t* mask_out, uint32_t* count_dev, void* stream);

/*
 * Fused backward: K6 + K7 + the autograd chain through get_depth_and_silhouette,
 * the activations and transform_to_frame.
 *   want_gaussian_grads: write dL/d{means3D, rgb_colors, unnorm_rotations,
 *       logit_opacities, log_scales} (mapping) -- any pointer may be NULL to skip it.
 *   want_pose_grads: reduce dL/d(cam_unnorm_rot)[4] and dL/d(cam_trans)[3] (tracking / BA).
 *   dL_dmeans2D[N,3] (optional) is what means2D.grad exposes in the reference.
 */
typedef struct VtgsParamGrads {
    float* means3D;
    float* rgb_colors;
    float* unnorm_rotations;
    float* logit_opacities;
    float* log_scales;
    float* means2D;
    float* cam_unnorm_rot;   /* [4] */
    float* cam_trans;        /* [3] */
    float* pose_scratch;     /* vtgs_pose_scratch_floats(N) floats                        */
    const float* pose_scale; /* optional device scalar: the pose gradient is multiplied by it (the incoming dL/dloss of
                                an autograd backward), saving the caller two launches                          */
    const float* dL_abs_bound; /* optional device scalar >= max |dL_dimage4| (VTGS_BUF_DETERMINISTIC only: the grids of
                                the order-independent sums derive from it; NULL = measured by one more pass over
                                dL_dimage4).  vtgs_loss in tracking mode leaves max(w_im, w_depth) in loss_terms[6]. */
} VtgsParamGrads;

VTGS_API uint64_t vtgs_pose_scratch_floats(int64_t num_gaussians);

VTGS_API int vtgs_fused_backward(const VtgsCamera* cam, const VtgsParams* params, const VtgsPose* pose,
                        const float* dL_dimage4 /* [4,H,W]: r,g,b,depth */,
                        int32_t accumulate /* 0: overwrite grads, 1: += (multi-keyframe) */,
                        VtgsParamGrads* grads, VtgsBuffers* buf, void* stream);

/*
 * One reference tracking iteration's render work in ONE call: get_loss(tracking=True) followed by loss.backward()
 * (reference src/vtgaussian_slam.py:1886-1889, get_loss :407-689) = vtgs_fused_forward, vtgs_loss (tracking mode),
 * vtgs_fused_backward to the 7 pose numbers (grads->cam_unnorm_rot / cam_trans; Gaussian-parameter pointers may be set as
 * well) and, when max_2D_radius != NULL, vtgs_book_radii -- the same kernels in the same order on `stream`.  A caller
 * that steps from a host loop (one Python / FFI crossing per iteration) is otherwise paced by its four crossings.
 */
VTGS_API int vtgs_fused_tracking_step(const VtgsCamera* cam, const VtgsParams* params, const VtgsPose* pose,
                        const VtgsLossConfig* cfg, const float* gt_rgb, const float* gt_depth,
                        float* out_image6, int32_t* radii, float* dL_dimage4, float* loss_terms, float* loss_scratch,
                        VtgsParamGrads* grads, float* max_2D_radius /* may be NULL */, uint8_t* seen /* may be NULL */,
                        VtgsBuffers* buf, void* stream);

/*
 * Adam exactly as torch.optim.Adam(betas=(0.9,0.999), eps, weight_decay=0) applies it to
 * one tensor (reference src/vtgaussian_slam.py:180-187): step is the 1-based step count
 * read from *step_dev (device int32, incremented by the caller via vtgs_adam_tick or kept
 * on the host and passed in `step` when step_dev == NULL).
 */
VTGS_API int vtgs_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
              float lr, float beta1, float beta2, float eps, int32_t step,
              const int32_t* step_dev, void* stream);

/*
 * Keyframe-sharded mapping step over NVLink peer memory (one process per GPU; reference: the optimizer.step() after the
 * summed keyframe losses, src/vtgaussian_slam.py:2686-2694, when the keyframes of a mapping iteration are split over
 * the ranks): reduce-scatter of the gradients + Adam + all-gather of the parameters in ONE kernel.
 *   peer_bases[world]  HOST array: base address, in THIS process, of every rank's symmetric block (rank order); every
 *                      block holds the flat parameters at float offset param_off, the rank's flat gradients at grad_off
 *                      (n floats each, n % 4 == 0, 16-byte aligned) and the rank's loss at loss_off
 *   multicast_base     0, or the address of the blocks' NVLS multicast object: the gradients are then reduced inside the
 *                      NVSwitch (multimem.ld_reduce) and the parameters broadcast by it (multimem.st); the order of
 *                      that in-switch sum is the hardware's
 *   exp_avg, exp_avg_sq  THIS rank's slice of the moments: ceil(n / 4 / world) * 4 floats each
 *   seg_end / lr [nseg <= 4]  the flat vector is nseg tensors laid end to end: tensor s ends at element seg_end[s]
 *   step_dev           device int32: 1-based step count;   loss_out: device float, receives the summed loss
 * Rank r sums slice r of all ranks' gradients in rank order (fixed order), updates it with torch.optim.Adam's rule and
 * stores the new parameters into every rank's block.  The caller must run a cross-device barrier before the call
 * (every rank's gradients are complete) and after it (every rank's parameters have landed).  world <= 8.
 */
VTGS_API int vtgs_sharded_adam(int32_t world, int32_t rank, const uint64_t* peer_bases, uint64_t multicast_base, int64_t param_off, int64_t grad_off,
                       int64_t loss_off, float* exp_avg, float* exp_avg_sq, int64_t n, int32_t nseg, const int64_t* seg_end,
                       const float* lr, float beta1, float beta2, float eps, const int32_t* step_dev, float* loss_out,
                       void* stream);

/*
 * Re-tie a section's view-tied Gaussians to its optimised pose (reference src/vtgaussian_slam.py:2706-2727):
 * means3D[i] <- inv([R(q)|t]) * (w2c_old * means3D[i]) for i in [0, n).  w2c_old: 12 HOST floats (rows of the 3x4
 * matrix the section was tied to); q = cam_unnorm_rot[4], t = cam_trans[3] on the DEVICE (the just-stepped pose).
 */
VTGS_API int vtgs_retie(float* means3D, int64_t n, const float* w2c_old, const float* cam_unnorm_rot,
                        const float* cam_trans, void* stream);

/* The same with the OLD pose given as device quaternion / translation (e.g. a copy taken before the optimiser step):
 * nothing crosses to the host, so a mapping iteration with bundle adjustment stays free of synchronisation. */
VTGS_API int vtgs_retie_dev(float* means3D, int64_t n, const float* old_unnorm_rot, const float* old_trans,
                            const float* cam_unnorm_rot, const float* cam_trans, void* stream);

/*
 * The re-ties of a keyframe-sharded bundle-adjustment iteration, every rank's in one launch and without a host round
 * trip.  Each rank writes one record per keyframe whose pose it stepped into its table of records_per_rank records:
 *   words  0-3   int32 valid (0 = empty slot), id (the keyframe's frame index), n_last (rows to re-tie, 0 = none), reserved
 *   words  4-10  float old_q[4], old_t[3]: the pose before the step
 *   words 11-17  float new_q[4], new_t[3]: the pose after the step
 *   words 18-19  pad (a record is VTGS_BA_RECORD_WORDS words; tables are 16-byte aligned)
 *   table_bases[world]  HOST array: device address, in THIS process, of rank r's table (a peer mapping, or a local copy)
 *   means3D[n_rows, 3]  re-tied in place
 *   table_out           NULL, or [world * records_per_rank * VTGS_BA_RECORD_WORDS] words: receives the tables in rank order
 * For every rank r, then every slot s, in that order, a record with valid != 0 and n_last > 0 re-ties the rows
 * [n_rows - min(n_last, n_rows), n_rows) exactly as vtgs_retie_dev(old -> new) does.  A row covered by several records goes
 * through them in (rank, slot) order, so one call gives the bits of the same sequence of vtgs_retie_dev calls.  world <= 8.
 */
#define VTGS_BA_RECORD_WORDS 20
VTGS_API int vtgs_retie_records(int32_t world, const uint64_t* table_bases, int32_t records_per_rank, float* means3D,
                                int64_t n_rows, uint32_t* table_out, void* stream);

/*
 * Tracking pose update in one launch: the reference's `optimizer.step()` on the frame's pose slices
 * (src/vtgaussian_slam.py:1890, Adam betas (0.9, 0.999)) plus its best-candidate bookkeeping (:1961-1970).
 *   msg[16]        = {dL/dq[4], dL/dt[3], pad, loss_terms[8]}  (the all-reduced message of an iteration)
 *   adam_state[14] = {m_q[4], v_q[4], m_t[3], v_t[3]};  *step_dev is incremented
 *   best[8]        = {best_metric, best_q[4], best_t[3]}: a candidate pose is kept if this iteration's metric is smaller
 *   flags: VTGS_TRACK_BOOK_POST_STEP  book the pose AFTER this step (what the reference does: it clones the pose after
 *                                     optimizer.step() against the loss computed before it, :1888-1970); without it the
 *                                     pose the loss was evaluated at is booked;
 *          VTGS_TRACK_CALLER_METRIC   rank candidates by msg[15] (a caller-supplied metric, e.g. the reference's
 *                                     point-to-plane distance `choose_metric`) instead of the loss msg[8].
 */
#define VTGS_TRACK_BOOK_POST_STEP 1
#define VTGS_TRACK_CALLER_METRIC  2
VTGS_API int vtgs_tracking_update(float* cam_unnorm_rot, float* cam_trans, const float* msg, float* adam_state,
                                  int32_t* step_dev, float* best, float lr_rot, float lr_trans, float eps, int32_t flags,
                                  void* stream);

/*
 * Per-frame evaluation metrics of the reference's `eval` (utils/eval_helpers.py:431-477) on a fused six-plane render:
 * valid = gt_depth > 0, presence = silhouette > sil_thres; the images are weighted by valid (and by presence when
 * use_presence != 0: the reference's `mapping_iters == 0 and not add_new_gaussians` configuration).
 *   out8 (device) = {sum sq err r, g, b, sum |depth - gt| (masked), valid count, PSNR (mean over channels of
 *                    20 log10(1 / sqrt(mse_c)), mse over ALL pixels as calc_psnr does), depth L1, depth "RMSE" (the
 *                    reference takes sqrt(x^2) per pixel, i.e. the same number as the L1)}
 *   scratch: vtgs_eval_scratch_floats() floats.  One launch, fixed-order reduction.
 */
VTGS_API uint64_t vtgs_eval_scratch_floats(void);
VTGS_API int vtgs_eval_metrics(const VtgsCamera* cam, const float* image6, const float* gt_rgb, const float* gt_depth,
                               float sil_thres, int32_t use_presence, float* out8, float* scratch, void* stream);

/*
 * Device point-to-plane metric: the reference's compute_point2plane_dist (src/vtgaussian_slam.py:1070-1155, called
 * inside the tracking loop at :1929 / :1956) without its CPU round trips (kornia normals -> numpy -> Open3D KD-tree).
 * vtgs_p2p_prepare: one frame's depth[H,W] (device) -> world points pts[H*W,3] (get_pointcloud, factor 1), optional
 *   world normals nrm[H*W,3] (kornia depth_to_normals, rotated as trans_normal_c2w does; NULL to skip) and
 *   valid[H*W] = depth > 0 [& mask] [& inside the other frame's view: get_frustum_mask when other_w2c12 != NULL].
 *   intr4 = {fx, fy, cx, cy}, c2w12 / other_w2c12 = rows of 3x4 matrices; all three on the HOST.
 * vtgs_p2p_match: for every valid source point the nearest valid target point within max_dist (Open3D
 *   evaluate_registration's correspondence set, threshold 0.02 in the reference) through a uniform hash grid
 *   (table: table_size int32, a power of two; next: n_tgt int32; both device scratch);
 *   out_dist[n_src] = n_target . (p_source - p_target), NaN where there is no correspondence; out_idx (optional) the
 *   target index or -1.  The caller reduces out_dist (sum of squares / max / top-100 mean: `p2p_method`).
 */
VTGS_API int vtgs_p2p_prepare(int32_t W, int32_t H, const float* intr4, const float* c2w12, const float* other_w2c12,
                              const float* depth, const uint8_t* mask, float* pts, float* nrm, uint8_t* valid, void* stream);
VTGS_API int vtgs_p2p_match(int64_t n_tgt, const float* tgt_pts, const float* tgt_nrm, const uint8_t* tgt_valid,
                            int64_t n_src, const float* src_pts, const uint8_t* src_valid, float max_dist,
                            int32_t* table, int64_t table_size, int32_t* next, float* out_dist, int32_t* out_idx, void* stream);

/*
 * Frame conversion on the device (SURVEY 8(f) N2): the raw decoded frame -- colour uint8 [src_h, src_w, 3], depth uint16
 * [src_h, src_w] -- to the planes the loop consumes, im[3, dst_h, dst_w] float32 in [0, 1] and depth[dst_h, dst_w] float32
 * metres, as the reference's loader produces them on the CPU (datasets/gradslam_datasets/basedataset.py:215-272: colour
 * through cv2.resize INTER_LINEAR as float64, depth through INTER_NEAREST then / png_depth_scale; then
 * src/vtgaussian_slam.py:201-202).  Either pair of pointers may be NULL.  All pointers are device pointers.
 */
VTGS_API int vtgs_frame_convert(int32_t src_w, int32_t src_h, int32_t dst_w, int32_t dst_h, const uint8_t* rgb_hwc,
                                const uint16_t* depth_u16, double png_depth_scale, float* im_chw, float* depth_out, void* stream);

/*
 * Radius bookkeeping of get_loss (reference src/vtgaussian_slam.py:681-683) in one launch:
 *   seen[i] = radii[i] > 0;  max_2D_radius[i] = max(max_2D_radius[i], radii[i])   (radii >= 0, so unseen entries keep theirs)
 * radii: int32 [n] as the forward wrote them; max_2D_radius: float [n] in place; seen: 1 byte per Gaussian (torch.bool).
 */
VTGS_API int vtgs_book_radii(int64_t n, const int32_t* radii, float* max_2D_radius, uint8_t* seen, void* stream);

/* FP32 FMA throughput probe (bench.py's measured FP32 peak): every thread of a full grid runs `iters` dependent-free
 * FFMA octets; FLOP = 2 * 8 * iters * threads, threads = *threads_out.  sink: one device float (keeps the work alive). */
VTGS_API int vtgs_ffma_probe(int64_t iters, float* sink, uint64_t* threads_out, void* stream);

/*
 * Optional per-kernel timing for bench.py's roofline: while enabled, every kernel launch of
 * the library is bracketed by CUDA events on its launching stream.  vtgs_profile_summary
 * synchronises those events and writes one line per kernel: "<name> <launches> <total_ms>".
 * Not capturable in a CUDA graph; off by default (zero overhead).
 */
VTGS_API int vtgs_profile_enable(int32_t on);
VTGS_API int vtgs_profile_summary(char* buf, uint64_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* VTGS_H_ */
