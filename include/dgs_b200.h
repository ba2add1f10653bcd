/*
 * dgs_b200.h -- C-ABI of libdgs_b200.so, the B200-native (sm_100a) blurry-view
 * Gaussian-splatting rasterizer.  Every entry point is `extern "C"`, takes plain
 * device pointers + sizes + a cudaStream_t (passed as void*), returns 0 on success
 * or a negative dgs_status whose text is available from dgs_last_error().
 *
 * What each entry point replaces in the reference (taekkii/deblurgs):
 *   dgs_forward / dgs_backward
 *       pybind `rasterize_gaussians` / `rasterize_gaussians_backward`
 *       (submodules/diff-gaussian-rasterization/ext.cpp:15-19, rasterize_points.cu:35-218)
 *       = CudaRasterizer::Rasterizer::forward / backward
 *       (cuda_rasterizer/rasterizer.h:31-95, rasterizer_impl.cu:198-463)
 *   dgs_blur_forward / dgs_blur_backward
 *       the Python loop `for cam in subframe_cams: render(cam, gaussians, bg)` + stack + mean
 *       of CameraMotionModule.query (scene/motion.py:138-150) and the F autograd backward
 *       calls it induces (diff_gaussian_rasterization/__init__.py:111-170)
 *   dgs_pose_forward / dgs_pose_backward
 *       BezierModel.forward (scene/bezier.py:54-83), se3_exp_map
 *       (utils/pytorch3d_functions.py:373-457), _c2w_to_minicam (scene/motion.py:258-294),
 *       MiniCam.__init__ (scene/cameras.py:63-74) and their autograd
 *   dgs_mark_visible        pybind `mark_visible` (ext.cpp:18, rasterizer_impl.cu:54-66,141-153)
 *   dgs_knn_mean_dist2      `distCUDA2` (submodules/simple-knn/spatial.cu:15-26, simple_knn.cu:185-221)
 *
 * Memory ownership follows the reference (rasterize_points.cu:27-33,80-82): the caller
 * owns every buffer; the library asks for its three opaque state buffers through resize
 * callbacks and hands them back for the backward pass.
 *
 * Matrix convention = the reference's: `viewmatrix`/`projmatrix` are the row-major torch
 * tensors world_view_transform / full_proj_transform, i.e. element [4*col + row] of the
 * mathematical matrix (cuda_rasterizer/auxiliary.h:58-77).
 */
#ifndef DGS_B200_H_INCLUDED
#define DGS_B200_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum dgs_status {
    DGS_OK = 0,
    DGS_ERR_INVALID_ARGUMENT = -1,
    DGS_ERR_CUDA = -2,
    DGS_ERR_ALLOC = -3,
    DGS_ERR_UNSUPPORTED = -4
} dgs_status;

/* Resize callback: must return a device pointer to at least `bytes` bytes, 128-B aligned,
 * that stays valid until the matching backward has run.  (Reference: the three
 * std::function<char*(size_t)> of Rasterizer::forward, rasterizer.h:32-34.) */
typedef char* (*dgs_alloc_fn)(void* ctx, size_t bytes);

/* Library / build introspection. */
const char* dgs_last_error(void);
int dgs_version(void);            /* 100 * major + minor */
int dgs_compiled_arch(void);      /* 1000 for sm_100a */

/*
 * Batched forward: F sub-frames of one blurry view over the same P Gaussians.
 *   view/proj   [F,16]   campos [F,3]   (device, fp32)
 *   out_color   [F,3,H,W]   out_depth [F,1,H,W]   radii [F,P] int32
 *   out_blur    [3,H,W] or NULL: (1/F_total) * sum_s out_color[s]   (F_total = blur_denominator,
 *               so a rank that renders a shard of the sub-frames produces its partial mean)
 * Optional inputs follow the reference: exactly one of shs / colors_precomp and exactly one
 * of (scales, rotations) / cov3D_precomp is non-NULL.  sh_degree = active degree D (0..3),
 * sh_coeffs = M (allocated coefficients per Gaussian, >= (D+1)^2).
 * Returns the total number of (Gaussian, tile) duplicates over all F sub-frames in
 * *num_rendered (the reference's per-sub-frame `num_rendered`, summed).
 */
int dgs_blur_forward(
    dgs_alloc_fn geom_alloc, void* geom_ctx,
    dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t* num_rendered, void* stream);

/*
 * The same forward without a host synchronisation.  dgs_blur_forward has to learn the number of duplicates D
 * on the host before it can size the binning buffer (one cudaStreamSynchronize per view; the reference does
 * one per sub-frame, rasterizer_impl.cu:287).  Here the caller supplies `binning_capacity` = the number of
 * duplicates it expects at most (e.g. 1.25 x the previous step's num_rendered); the buffer is sized from it,
 * every kernel of the view is enqueued at once and D stays on the device.
 *   num_rendered != NULL: after enqueuing, the host waits for a 24-byte status read-back that was issued right
 *       after the scan stage (the GPU is busy with the blend meanwhile) and, if D exceeded the capacity, re-runs
 *       the tile sort and the blend with the exact size: results are always complete, *num_rendered = D.
 *   num_rendered == NULL: nothing is waited for (the call can be captured in a CUDA graph).  If D exceeds the
 *       capacity the tile sort is skipped (all lists empty: background only); dgs_blur_forward_status reports
 *       D and the overflow flag so that the caller can replay with a larger capacity.
 * binning_capacity == 0 behaves like dgs_blur_forward.  The backward needs no D: pass num_rendered = -1.
 */
int dgs_blur_forward_hint(
    dgs_alloc_fn geom_alloc, void* geom_ctx,
    dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t binning_capacity, int64_t* num_rendered, void* stream);
/* D and the overflow flag of a forward call, read from its geometry buffer (synchronises the stream). */
int dgs_blur_forward_status(const char* geom_buffer, int P, int F, int64_t* num_rendered, int* overflow,
                            void* stream);
/* Byte offset, from the 128-B aligned start of the geometry buffer, of the 24-byte status record
 * { uint64 num_rendered; uint64 padded; uint32 overflow; uint32 n_chunks } -- for callers that copy it themselves
 * (e.g. as a memcpy node of a captured CUDA graph). */
size_t dgs_blur_forward_status_offset(int P, int F);

/*
 * Batched backward.  dL_dpix [F,3,H,W], dL_dpixdepth [F,1,H,W] (either may be NULL = zeros);
 * dL_dblur [3,H,W] or NULL: gradient of the blurred image, folded in as dL_dpix[s] += dL_dblur /
 * blur_denominator for every sub-frame (the backward of the mean, without materialising [F,3,H,W]).
 * Gaussian gradients are SUMMED over the F sub-frames and written (not accumulated):
 *   dL_dmeans3D [P,3] dL_dsh [P,M,3] dL_dopacity [P,1] dL_dscales [P,3] dL_drotations [P,4]
 *   dL_dcolors_precomp [P,3] dL_dcov3D_precomp [P,6]   (only with the matching precomp input)
 * Per-sub-frame outputs:
 *   dL_dmeans2D [F,P,3] (x,y = gradient w.r.t. NDC, z = 0; reference backward.cu:628-629) or NULL
 *   dL_dviewmatrix [F,16], dL_dprojmatrix [F,16]  (reference quirks reproduced, SURVEY 8a B2/B3)
 * densify_stats [P,3] or NULL: per Gaussian (sum over its visible sub-frames of |dL_dmeans2D.xy|, number of
 * sub-frames in which it is visible, max screen radius) -- the quantities the reference's training loop
 * accumulates per sub-frame (train.py:188-193, scene/gaussian_model.py:456-458), produced in the same pass.
 * `scratch` must hold dgs_blur_backward_scratch_bytes(P,F) bytes; contents undefined on return.
 */
size_t dgs_blur_backward_scratch_bytes(int P, int F);

int dgs_blur_backward(
    int P, int F, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth, const float* dL_dblur, float blur_denominator,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, float* densify_stats, void* stream);

/*
 * The batched backward in pieces, so that a caller can overlap a collective with it: `stages` is a bit set of
 *   DGS_BWD_BLEND      scratch clear + tile-blend backward (all sub-frames)
 *   DGS_BWD_GAUSSIANS  per-Gaussian backward for the Gaussians [g_begin, g_end): their rows of every Gaussian
 *                      gradient (and of dL_dmeans2D / densify_stats) are final when it completes, so e.g. an NCCL
 *                      all-reduce of those rows can run while the next range is computed
 *   DGS_BWD_FINISH     view / projection-matrix gradients (accumulated over all ranges) -> dL_dviewmatrix / dL_dprojmatrix
 * Call BLEND once, GAUSSIANS for ranges that cover [0, P) in any order, FINISH last, all with the same arguments
 * and scratch on the same stream.  dgs_blur_backward = all three over [0, P).
 */
#define DGS_BWD_BLEND 1
#define DGS_BWD_GAUSSIANS 2
#define DGS_BWD_FINISH 4
#define DGS_BWD_ALL 7
int dgs_blur_backward_range(
    int P, int F, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth, const float* dL_dblur, float blur_denominator,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, float* densify_stats,
    int64_t g_begin, int64_t g_end, int stages, void* stream);

/*
 * Antialiased rendering (Mip-Splatting's screen-space filter, DESIGN.md section 3).  Every projected 2-D covariance
 * is dilated by 0.3 px^2 on its diagonal; with antialiasing = 1 the opacity a Gaussian blends with is scaled by
 * rho = sqrt(max(det0 / det, 2.5e-5)) (det0, det: determinants before and after the dilation), so that a Gaussian
 * narrower than a pixel keeps its integrated weight instead of rendering wider and more opaque.  Radii, tile
 * rectangles, depth keys, sorted lists and conics are the same as with antialiasing = 0.
 * Arguments are those of dgs_blur_forward_hint / dgs_blur_backward_range plus `antialiasing` (0 or 1; any other
 * value fails with DGS_ERR_INVALID_ARGUMENT before any device work).  With 0 they are those two entry points.
 * A backward must be called with the antialiasing value of the forward that filled its state buffers.
 */
int dgs_blur_forward_aa(
    dgs_alloc_fn geom_alloc, void* geom_ctx,
    dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t binning_capacity, int64_t* num_rendered, int antialiasing, void* stream);
int dgs_blur_backward_range_aa(
    int P, int F, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth, const float* dL_dblur, float blur_denominator,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, float* densify_stats,
    int64_t g_begin, int64_t g_end, int stages, int antialiasing, void* stream);

/*
 * Contribution scores (DESIGN.md section 3).  dgs_blur_forward_aa plus, for every Gaussian g, over every pixel of every
 * sub-frame where the blend actually used it, with its blending weight w = alpha * T (the weight of its colour term):
 *   contrib_wsum[g] += sum of round(w * DGS_CONTRIB_SCALE)     (fixed point: at most 2^-27 error per blended pixel)
 *   contrib_wmax[g]  = max(contrib_wmax[g], bits of max w)     (float bits: non-negative floats order like their bits)
 * Both are device arrays of [P], ACCUMULATED into: zero them before the first call (wmax = 0 is the float 0).  Integer
 * sums and maxima do not depend on the order of the additions, so the scores are the same bits on every run and for
 * any batching of the sub-frames.  Images, depths, radii and every state buffer are exactly those of
 * dgs_blur_forward_aa (a following dgs_blur_backward_range_aa is valid as usual).
 * A speculative call (binning_capacity > 0) whose hint is too small blends empty lists first, which adds nothing;
 * with num_rendered != NULL the blend is re-run with the exact size and adds the scores once, with num_rendered == NULL
 * (nothing waited for) such an overflowed call adds nothing at all -- dgs_blur_forward_status reports it.
 * NULL score pointers with P > 0 and F > 0, or an antialiasing value other than 0 / 1, fail with
 * DGS_ERR_INVALID_ARGUMENT before any device work.
 */
#define DGS_CONTRIB_SCALE (1 << 26)
int dgs_blur_forward_contrib(
    dgs_alloc_fn geom_alloc, void* geom_ctx,
    dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int F, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    float* out_blur, float blur_denominator,
    int64_t binning_capacity, int64_t* num_rendered, int antialiasing,
    uint64_t* contrib_wsum, uint32_t* contrib_wmax, void* stream);

/* Single-view pair: the reference's rasterize_gaussians / rasterize_gaussians_backward
 * (same argument meaning; F = 1 instance of the batched pair). */
int dgs_forward(
    dgs_alloc_fn geom_alloc, void* geom_ctx,
    dgs_alloc_fn binning_alloc, void* binning_ctx,
    dgs_alloc_fn image_alloc, void* image_ctx,
    int P, int sh_degree, int sh_coeffs,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far,
    int prefiltered, int use_sigmoid,
    float* out_color, float* out_depth, int* radii,
    int64_t* num_rendered, void* stream);

int dgs_backward(
    int P, int sh_degree, int sh_coeffs, int64_t num_rendered,
    const float* background, int width, int height,
    const float* means3D, const float* shs, const float* colors_precomp,
    const float* opacities, const float* scales, float scale_modifier,
    const float* rotations, const float* cov3D_precomp,
    const float* viewmatrix, const float* projmatrix, const float* campos,
    float tan_fovx, float tan_fovy, float z_near, float z_far, int use_sigmoid,
    const int* radii,
    const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
    const float* dL_dpix, const float* dL_dpixdepth,
    char* scratch,
    float* dL_dmeans2D, float* dL_dmeans3D, float* dL_dsh, float* dL_dopacity,
    float* dL_dscales, float* dL_drotations, float* dL_dcolors_precomp, float* dL_dcov3D_precomp,
    float* dL_dviewmatrix, float* dL_dprojmatrix, void* stream);

/*
 * Debug/parity accessors: decode the opaque state buffers of a forward call into the
 * reference's per-sub-frame quantities (GeometryState / BinningState / ImageState,
 * rasterizer_impl.h:31-63).  All outputs optional (NULL = skip).
 *   depths [F,P] means2D [F,P,2] conic_opacity [F,P,4] rgb [F,P,3] clamped [F,P,3]
 *   tiles_touched [F,P] u32   point_offsets [F,P] u32 (per sub-frame: inclusive scan of tiles_touched taken
 *   in the library's depth-sorted order; element [s][P-1] is the sub-frame's num_rendered)
 */
int dgs_debug_geometry(const char* geom_buffer, int P, int F,
                       float* depths, float* means2D, float* conic_opacity, float* rgb,
                       float* clamped, uint32_t* tiles_touched, uint32_t* point_offsets,
                       void* stream);
/*   keys [D] u64 (batched key of every sorted list entry: sub-frame | tile | depth bits; the library sorts in two
 *   stages -- Gaussians by depth, then the generated duplicates by tile inside each sub-frame's segment -- so
 *   the 64-bit key is rebuilt here from the entry's position and depth), point_list [D] u32, both compacted
 *   (the library pads every sub-frame's list to a multiple of 2048); ranges [F,tiles,2] u32 = positions in
 *   that compacted list */
int dgs_debug_binning(const char* geom_buffer, const char* binning_buffer, const char* image_buffer, int P, int F,
                      int width, int height, int64_t num_rendered, uint64_t* keys, uint32_t* point_list,
                      uint32_t* ranges, void* stream);
/*   final_T [F,H,W], n_contrib [F,H,W] u32 */
int dgs_debug_image(const char* image_buffer, int F, int width, int height,
                    float* final_T, uint32_t* n_contrib, void* stream);
/* The library's segmented LSD radix sort on its own (test hook): keys [nseg][len] u32 sorted on their low
 * key_bits bits inside every segment, stable; keys_sorted / index_sorted [nseg][len] (either may be NULL).
 * scratch: dgs_debug_sort_scratch_bytes(nseg, len). */
size_t dgs_debug_sort_scratch_bytes(int nseg, int64_t len);
int dgs_debug_sort(int nseg, int64_t len, int key_bits, const uint32_t* keys, uint32_t* keys_sorted,
                   uint32_t* index_sorted, char* scratch, void* stream);
/* Number of key bits used for the tile id and the sub-frame id of the batched sort key. */
int dgs_key_bits(int width, int height, int F, int* tile_bits, int* subframe_bits);

/*
 * Measurement hooks (used by bench.py; no effect on results).
 * dgs_profile_enable(1): every stage of the calls above is bracketed by a CUDA event pair on the
 * caller's stream.  dgs_profile_read synchronises those events and returns accumulated milliseconds
 * and call counts per stage (names from dgs_profile_stage_name).  dgs_launch_count = number of
 * kernels of THIS library launched so far (every kernel on the path is the library's own).
 * dgs_debug_workload replays the compositing loop and writes {E, K, E_b} (SURVEY.md 8d: list entries
 * evaluated, entries that contributed, entries replayed by the backward) to out_dev[3] (device).
 */
/* Measured FP32 FMA throughput of the current device in TFLOP/s (a register-resident FMA kernel, best of 6 short
 * runs; ~10 ms): the denominator of the issue-bound blend kernels' roofline.  implied_sm_mhz (optional) = the SM
 * clock that rate corresponds to at 128 FMA lanes per SM. */
int dgs_measure_fp32_peak(double* tflops, double* implied_sm_mhz, void* stream);
int dgs_profile_enable(int on);
int dgs_profile_num_stages(void);
const char* dgs_profile_stage_name(int i);
int dgs_profile_read(double* ms, int64_t* calls, int n, int reset);
int64_t dgs_launch_count(int reset);
int dgs_debug_workload(const char* geom_buffer, const char* binning_buffer, const char* image_buffer,
                       int P, int F, int width, int height, int64_t num_rendered, uint64_t* out_dev,
                       void* stream);

/*
 * Sub-frame poses from Bezier control points in se(3) (curve_type == "se3").
 *   ctrl_trans, ctrl_rot [C+1,3] fp32 (control point k weighted by binom(C,k) t^(C-k) (1-t)^k)
 *   nu [F] fp32 in [0,1];  proj_t [16] = the reference camera's `projection_matrix`
 *   (getProjectionMatrix(...).T, row-major)
 * Outputs: viewmatrix [F,16], projmatrix [F,16], campos [F,3] (fp32), and `jacobian`
 * [F, 35, 7] fp64: d(view 16 | proj 16 | campos 3)/d(se3 6-vector u|omega, nu) in the
 * reference's autograd semantics (campos rows are zero: the reference gives no gradient).
 */
int dgs_pose_forward(int F, int curve_order,
                     const float* ctrl_trans, const float* ctrl_rot, const float* nu,
                     const float* proj_t,
                     float* viewmatrix, float* projmatrix, float* campos,
                     double* jacobian, void* stream);
/*   dL_dctrl_trans, dL_dctrl_rot [C+1,3] fp32, dL_dnu [F] fp32 (written, not accumulated) */
int dgs_pose_backward(int F, int curve_order,
                      const float* ctrl_trans, const float* ctrl_rot, const float* nu,
                      const double* jacobian,
                      const float* dL_dviewmatrix, const float* dL_dprojmatrix,
                      float* dL_dctrl_trans, float* dL_dctrl_rot, float* dL_dnu, void* stream);

/*
 * Fused photometric loss of the blurry-view step (reference: train.py:147-163, utils/loss_utils.py:17-18,
 * 80-93):  loss = mean|blurred - gt| + lambda_t_smooth * mean|subframes[1:] - subframes[:-1]|.
 *   subframes [F, chw], blurred [chw], gt [chw] (chw = 3*H*W), loss_out [3] = (loss, l1, smoothness),
 *   scratch [2] doubles.  Backward: grad_out = device pointer to dL/dloss (NULL = 1), writes
 *   dL_dblurred [chw] and dL_dsubframes [F, chw].  With lambda_t_smooth == 0 `subframes` / `dL_dsubframes`
 *   may be NULL: the stack is then neither read nor given a gradient.
 */
int dgs_blur_loss_forward(int F, int64_t chw, const float* subframes, const float* blurred, const float* gt,
                          float lambda_t_smooth, float* loss_out, double* scratch, void* stream);
int dgs_blur_loss_backward(int F, int64_t chw, const float* subframes, const float* blurred, const float* gt,
                           float lambda_t_smooth, const float* grad_out, float* dL_dblurred,
                           float* dL_dsubframes, void* stream);

/*
 * The two regularisers of the reference's training loss (train.py:150-163):
 *   tv_loss  (utils/loss_utils.py:66-78)  x [planes, H, W] (planes = B*C): mean of squared vertical differences +
 *            mean of squared horizontal differences; the depth smoothness term lambda_depth_tv * tv_loss(depths)
 *   hinge_l2 (utils/loss_utils.py:95-104) mean of x^2 where x <= 0 and (x-1)^2 where x >= 1; applied to the raw
 *            opacities (lambda_hinge * hinge_l2(_opacity))
 * loss_out [1] float, scratch [2] doubles; backward: grad_out = device pointer to dL/dloss (NULL = 1), dL_dx written.
 */
int dgs_tv_loss_forward(int64_t planes, int H, int W, const float* x, float* loss_out, double* scratch, void* stream);
int dgs_tv_loss_backward(int64_t planes, int H, int W, const float* x, const float* grad_out, float* dL_dx, void* stream);
int dgs_hinge_l2_forward(int64_t n, const float* x, float* loss_out, double* scratch, void* stream);
int dgs_hinge_l2_backward(int64_t n, const float* x, const float* grad_out, float* dL_dx, void* stream);

/*
 * SSIM (3DGS utils/loss_utils.py `ssim`, window 11, sigma 1.5, zero padding, C1 = 0.01^2, C2 = 0.03^2) of two
 * [N, C, H, W] fp32 stacks, N * C <= 65535.
 *   forward:  ssim_out [1 + N] = (mean over all N*C*H*W map values, mean of image 0, ..., mean of image N-1);
 *             scratch = dgs_ssim_scratch_bytes(N, C, H, W) bytes (one double per 32x16 tile of every plane; 0 for an
 *             invalid size).  The partial sums are reduced in a fixed order: the result does not vary between calls.
 *             maps [3, N, C, H, W] (or NULL when no gradient is wanted) receives dS/dmu1, dS/dsigma1^2, dS/dsigma12.
 *   backward: dL_dimg1 [N, C, H, W] written from the forward's maps; img2 is a constant.  grad_out = device pointer
 *             to dL/dssim (NULL = 1): one value (per_image == 0, the overall mean) or N values (per_image != 0).
 * No allocation and no host synchronisation inside: both calls can be captured in a CUDA graph.
 */
size_t dgs_ssim_scratch_bytes(int N, int C, int H, int W);
int dgs_ssim_forward(int N, int C, int H, int W, const float* img1, const float* img2, float* ssim_out,
                     double* scratch, float* maps, void* stream);
int dgs_ssim_backward(int N, int C, int H, int W, const float* img1, const float* img2, const float* maps,
                      const float* grad_out, int per_image, float* dL_dimg1, void* stream);

/*
 * Gaussian parameter store, the steps either side of the rasterizer (SURVEY.md 8f rank 3).
 *
 * dgs_activate_forward replaces the four getters `render` reads -- get_features (cat of _features_dc
 * [P,1,3] and _features_rest [P,M-1,3]), get_scaling (exp + scale_lb; isotropic != 0: column 0 expanded),
 * get_rotation (F.normalize, eps 1e-12), get_opacity (clamp to [0,1]) -- scene/gaussian_model.py:114-137,
 * scene/gaussian_activation.py:29-52; one launch per blurry view instead of ~8 torch launches per
 * sub-frame.  dgs_activate_backward is its chain rule; incoming gradients may be NULL (= zero), every
 * outgoing gradient is written (not accumulated).
 */
int dgs_activate_forward(int P, int sh_coeffs, const float* features_dc, const float* features_rest,
                         const float* scaling, const float* rotation, const float* opacity,
                         float scale_lower_bound, int isotropic,
                         float* shs, float* scales, float* rotations, float* opacities, void* stream);
int dgs_activate_backward(int P, int sh_coeffs, const float* scaling, const float* rotation, const float* opacity,
                          int isotropic, const float* dL_dshs, const float* dL_dscales, const float* dL_drotations,
                          const float* dL_dopacities, float* dL_dfeatures_dc, float* dL_dfeatures_rest,
                          float* dL_dscaling, float* dL_drotation, float* dL_dopacity, void* stream);

/*
 * Mip-Splatting's 3-D smoothing filter (Yu et al., CVPR 2024; reference: mip-splatting scene/gaussian_model.py).
 *
 * dgs_filter3d_depth restates the sweep of `compute_3D_filter` for n_cams cameras that share one set of intrinsics:
 * viewmatrices [n_cams, 16] are world_view_transform (row-vector layout, p = [x, 1] . V).  For every Gaussian and
 * camera, with z = p.z, z' = max(z, 0.001), u = p.x / z' * focal_x + width / 2, v = p.y / z' * focal_y + height / 2,
 * the camera sees the Gaussian iff z > z_near and -0.15 width <= u <= 1.15 width and -0.15 height <= v <= 1.15 height.
 * min_depth [P] (device, initialised by the caller, e.g. to +inf) is min-combined with the smallest z of the cameras
 * that see each Gaussian.  A float min is exact, so successive calls compose over views and camera chunks and the
 * result is bit-identical for any order or split of the same cameras.  The finalisation (filter = d_min / max focal
 * * sqrt(0.2), unseen Gaussians at the largest finite d_min) is the caller's (deblurgs_b200/filter3d.py).
 * Rejected before any device work: P < 0, n_cams < 0, a focal length or image size <= 0, and NULL pointers when
 * P > 0 and n_cams > 0.
 *
 * dgs_activate_forward_filter3d: dgs_activate_forward with the filter of `get_scaling_with_3D_filter` /
 * `get_opacity_with_3D_filter` applied, f = filter3d[g] (device, [P], a constant without gradient):
 *   scales'_i = sqrt(s_i^2 + f^2),  opacity' = clamp(opacity, 0, 1) * r_0 * r_1 * r_2,  r_i = s_i / scales'_i,
 * where s = exp(scaling) + scale_lower_bound.  The product of per-axis ratios equals Mip-Splatting's
 * sqrt(det1 / det2) and does not underflow for s < ~1e-7 as prod(s_i^2) does in fp32.
 * dgs_activate_backward_filter3d is its chain rule; it needs the forward's scale_lower_bound (the plain backward
 * does not).  A NULL filter3d is rejected.  The plain entry points are the same implementation without the filter.
 */
int dgs_filter3d_depth(int64_t P, const float* means3D, int n_cams, const float* viewmatrices, float focal_x,
                       float focal_y, int width, int height, float z_near, float* min_depth, void* stream);
int dgs_activate_forward_filter3d(int P, int sh_coeffs, const float* features_dc, const float* features_rest,
                                  const float* scaling, const float* rotation, const float* opacity,
                                  float scale_lower_bound, int isotropic, float* shs, float* scales, float* rotations,
                                  float* opacities, const float* filter3d, void* stream);
int dgs_activate_backward_filter3d(int P, int sh_coeffs, const float* scaling, const float* rotation,
                                   const float* opacity, int isotropic, const float* dL_dshs, const float* dL_dscales,
                                   const float* dL_drotations, const float* dL_dopacities, float* dL_dfeatures_dc,
                                   float* dL_dfeatures_rest, float* dL_dscaling, float* dL_drotation,
                                   float* dL_dopacity, float scale_lower_bound, const float* filter3d, void* stream);

/*
 * One Adam step over up to DGS_ADAM_MAX_TENSORS parameter tensors in a single launch: the reference's
 * `torch.optim.Adam(l, lr=0.0, eps=1e-15)` with one parameter per group and per-group learning rates
 * (scene/gaussian_model.py:175-190, train.py:204-208; amsgrad / weight decay / maximize off).
 * HOST arrays of n_tensors entries: device pointers params/grads/exp_avg/exp_avg_sq, numel, lr, and the
 * 1-based step count of each tensor AFTER this update.  clip_grad_value > 0 clamps each gradient element
 * to [-clip, clip] on the fly (torch.nn.utils.clip_grad_value_, train.py:204-205; the stored gradient is
 * left untouched).
 */
#define DGS_ADAM_MAX_TENSORS 8
int dgs_adam_step(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                  float* const* exp_avg_sq, const int64_t* numel, const double* lr, const int64_t* step,
                  double beta1, double beta2, double eps, double clip_grad_value, void* stream);

/*
 * Densify / prune on the parameter store (reference: scene/gaussian_model.py:300-454: prune_points,
 * cat_tensors_to_optimizer / densification_postfix, densify_and_clone, densify_and_split): every per-Gaussian
 * tensor is rebuilt as out[r] = in[src_rows[r]] in ONE launch -- up to DGS_GATHER_MAX_TENSORS tensors (the 6 raw
 * parameters, their 12 Adam moments, the 3 densification statistics), width[k] floats per row.  Tensors with
 * zero_new[k] != 0 (the Adam moments) get zeros in the rows where carry[r] == 0 (the appended Gaussians).
 * HOST arrays of n_tensors entries (device pointers inside); src_rows [n_out] int64 and carry [n_out] uint8 (or NULL
 * = every row carries) on the device.
 */
#define DGS_GATHER_MAX_TENSORS 24
int dgs_rows_gather(int n_tensors, const float* const* in, float* const* out, const int* width, const int* zero_new,
                    int64_t n_out, const int64_t* src_rows, const uint8_t* carry, void* stream);

/*
 * 3DGS-MCMC densification (Kheradmand et al., NeurIPS 2024) on the parameter store, in place.
 *
 * dgs_mcmc_relocate moves n Gaussians: entry r copies source row src_rows[r] into destination row dst_rows[r] and
 * splits the source's opacity and scale between the 1 + (copies) Gaussians that now share it, keeping the rendered
 * image unchanged to first order.  ratio[r] = N = 1 + (number of entries with the same source), clamped to [1, 51]:
 *   o  = clamp(opacity[src], 0, 1)                 (the raw opacity is the activated one: the activation is a clamp)
 *   o' = 1 - (1 - o)^(1/N), stored clamped to [0.005, 1 - 2^-23] (the lower bound is the smallest float above 0.005:
 *        a relocated Gaussian never counts as dead by the rule opacity <= 0.005); c uses the unclamped o'
 *   c  = o / D(o', N),  D = sum_{j=1..N} (-1)^(j-1) C(N,j) o'^j / sqrt(j)   (fp64; equal to the paper's double sum)
 *   raw scaling' = raw + log(c) when scale_lower_bound == 0, else log(max(c (exp(raw) + lb) - lb, 0.001));
 *   isotropic != 0: every column from column 0, as get_scaling expands it.
 * HOST arrays of n_tensors (<= DGS_GATHER_MAX_TENSORS) entries: device pointers `tensors` (fp32, [P, width[k]],
 * rewritten in place), width[k] and kind[k]:
 *   DGS_RELOCATE_COPY     dst row <- src row                    (xyz, features, rotation, the 3-D filter)
 *   DGS_RELOCATE_OPACITY  dst and src rows <- o'                (exactly one, width 1)
 *   DGS_RELOCATE_SCALING  dst and src rows <- raw scaling'      (exactly one, width 3)
 *   DGS_RELOCATE_ZERO     dst and src rows <- 0                 (Adam moments, densification statistics)
 * dst_rows, src_rows [n] int64 and ratio [n] int32 on the device.  PRECONDITION: the destination rows are distinct
 * and no destination row is a source row (sources are drawn from live Gaussians, destinations are dead or appended
 * ones); entries sharing a source must carry the same ratio.  scratch: dgs_mcmc_relocate_scratch_bytes(n) bytes,
 * 16-B aligned.  Two launches, no allocation, no host synchronisation.
 *
 * dgs_mcmc_noise: the SGLD step after the optimizer, for every Gaussian g < P:
 *   xyz[g] += Sigma eps gate step_scale,  Sigma = R diag(s^2) R^T,  gate = 1 / (1 + exp(-k ((1 - clamp(o,0,1)) - x0)))
 * with s = exp(scaling) + scale_lower_bound (isotropic: column 0), R the rotation of the normalised quaternion
 * (w, x, y, z; norm floored at 1e-12) and eps ~ N(0, I3) drawn in the kernel: Philox4x32-10 with key seed (low word
 * first) and counter (g, step) (low words first), then Box-Muller on the pairs (x0, x1) and (x2, x3) of its output, the
 * uniforms being ((x >> 8) + 0.5) / 2^24.  eps is a pure function of (seed, step, g).
 * dgs_debug_mcmc_normals writes that eps to out [P, 3] (test hook).
 */
#define DGS_RELOCATE_COPY 0
#define DGS_RELOCATE_OPACITY 1
#define DGS_RELOCATE_SCALING 2
#define DGS_RELOCATE_ZERO 3
size_t dgs_mcmc_relocate_scratch_bytes(int64_t n);
int dgs_mcmc_relocate(int n_tensors, float* const* tensors, const int* width, const int* kind, int64_t n,
                      const int64_t* dst_rows, const int64_t* src_rows, const int32_t* ratio, float scale_lower_bound,
                      int isotropic, void* scratch, void* stream);
int dgs_mcmc_noise(int64_t P, float* xyz, const float* scaling, const float* rotation, const float* opacity,
                   float scale_lower_bound, int isotropic, float step_scale, float k, float x0, uint64_t seed,
                   int64_t step, void* stream);
int dgs_debug_mcmc_normals(int64_t P, uint64_t seed, int64_t step, float* out, void* stream);

/* present [P] uint8: 1 iff view-space z > 0.2 (reference in_frustum, auxiliary.h:144-169). */
int dgs_mark_visible(int P, const float* means3D, const float* viewmatrix,
                     const float* projmatrix, uint8_t* present, void* stream);

/* Mean squared distance to the 3 nearest neighbours (exact). scratch: dgs_knn_scratch_bytes(P). */
size_t dgs_knn_scratch_bytes(int P);
int dgs_knn_mean_dist2(int P, const float* points, float* mean_dist2, char* scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DGS_B200_H_INCLUDED */
