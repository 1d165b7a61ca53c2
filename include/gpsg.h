/*
 * gpsg.h -- C ABI of libgpsg_sm100.so: the B200 (sm_100a) splat rasterizer and 1-D stereo
 * correlation sampler behind GPS-Gaussian's hot path.
 *
 * The reference has no native code of its own; its FFI for this path is the pybind surface of
 * two third-party extensions it imports by name:
 *   - `diff_gaussian_rasterization._C`  (reference gaussian_renderer/__init__.py:14; called through
 *      GaussianRasterizer at :51-62)          -> rasterize_gaussians / rasterize_gaussians_backward /
 *                                                mark_visible
 *   - `corr_sampler`                    (reference core/corr.py:5-8; called at :22 and :28)
 *                                             -> forward / backward
 * Each entry point below replaces exactly one of those bound functions; plain pointers and sizes,
 * no torch/ATen types, no exceptions.  All pointers are DEVICE pointers unless marked host.
 * Every function returns 0 on success or a negative GPSG_E_* code; gpsg_last_error() gives the
 * message (thread-local).  All work is enqueued on `stream` (a cudaStream_t) of CUDA device `device`.
 */
#ifndef GPSG_H
#define GPSG_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GPSG_API __attribute__((visibility("default")))
#else
#define GPSG_API
#endif

#define GPSG_OK 0
#define GPSG_E_INVALID (-1)   /* bad argument (shape / null / unsupported combination) */
#define GPSG_E_CUDA (-2)      /* a CUDA runtime call or kernel launch failed */
#define GPSG_E_ALLOC (-3)     /* an allocator callback returned NULL */
#define GPSG_E_CAPACITY (-4)  /* caller-provided workspace too small */

/* Mirrors diff_gaussian_rasterization.GaussianRasterizationSettings -- the 12 fields the reference
 * fills at gaussian_renderer/__init__.py:36-49.  Matrices are the 16 floats of the tensors the
 * reference passes (world_view_transform = W2V^T, full_proj_transform), i.e. the maths matrix is
 * M(r,c) = m[c*4+r].  Passed BY VALUE into kernels, so the tensors may live on host or device
 * (in training they stay in pinned host memory: reference train_stage2.py:155-157). */
typedef struct GpsgRasterSettings {
    int32_t image_height;
    int32_t image_width;
    float tanfovx;
    float tanfovy;
    float bg[3];
    float scale_modifier;
    float viewmatrix[16];
    float projmatrix[16];
    int32_t sh_degree;
    float campos[3];
    int32_t prefiltered;
    int32_t debug;
} GpsgRasterSettings;

/* Scratch allocator, the C form of upstream's `std::function<char*(size_t)>` resize callbacks over
 * torch byte tensors: must return a device pointer to >= `bytes` bytes (256-B aligned), valid until
 * the matching backward call has finished.  Called at most once per buffer per forward. */
typedef void* (*gpsg_alloc_fn)(void* user, size_t bytes);

GPSG_API const char* gpsg_last_error(void);
GPSG_API int gpsg_version(void);

/* ---- replaces _C.rasterize_gaussians (SURVEY.md Appendix A.1-A.5) ---------------------------
 * means3D[P,3] opacities[P] ; exactly one of colors_precomp[P,3] / shs[P,sh_M,3] ; either
 * (scales[P,3], rotations[P,4]) or cov3D_precomp[P,6].  Outputs out_color[3,H,W], radii[P].
 * Scratch comes from the three callbacks (geometry / binning / image state, kept for backward).
 * *num_rendered (HOST) receives the number of (tile,Gaussian) pairs.  One host sync, as upstream. */
GPSG_API int gpsg_rasterize_forward(const GpsgRasterSettings* settings, int device, void* stream, int P, int sh_M,
                           const float* means3D, const float* colors_precomp, const float* shs,
                           const float* opacities, const float* scales, const float* rotations,
                           const float* cov3D_precomp, float* out_color, int32_t* radii,
                           gpsg_alloc_fn geom_alloc, void* geom_user, gpsg_alloc_fn binning_alloc,
                           void* binning_user, gpsg_alloc_fn image_alloc, void* image_user,
                           int32_t* num_rendered);

/* ---- sync-free ("planned") forward: same computation as gpsg_rasterize_forward, but every buffer is provided by the
 * caller up front and there is NO host synchronisation, so the call is CUDA-graph capturable and the CPU can run
 * ahead.  `capacity_pairs` bounds the number of (tile,Gaussian) pairs the binning buffer can hold.  The kernels
 * read the actual pair count from device memory; if it exceeds the capacity (or a tile list exceeds the in-CTA sort
 * limit) they set the overflow word and skip their work: the caller must inspect status[2] once it next
 * synchronises and, if set, retry with a larger capacity / the exact entry point (out_color is then undefined).
 * status (device pointer into image_buf, see gpsg_raster_status_ptr; optionally mirrored to `status_host`, pinned):
 * [0] pairs N, [1] longest tile list, [2] overflow flag.  For gpsg_rasterize_backward pass num_rendered = capacity. */
GPSG_API size_t gpsg_raster_geom_bytes(int P);
GPSG_API size_t gpsg_raster_binning_bytes(int64_t capacity_pairs);
GPSG_API size_t gpsg_raster_image_bytes(int W, int H);
GPSG_API const uint32_t* gpsg_raster_status_ptr(const void* image_buffer, int W, int H);
GPSG_API int gpsg_rasterize_forward_planned(const GpsgRasterSettings* settings, int device, void* stream, int P,
                                            const float* means3D, const float* colors_precomp, const float* opacities,
                                            const float* scales, const float* rotations, const float* cov3D_precomp,
                                            float* out_color, int32_t* radii, void* geom_buffer, void* binning_buffer,
                                            int64_t capacity_pairs, void* image_buffer, uint32_t* status_host);

/* ---- replaces _C.rasterize_gaussians_backward (Appendix A.6-A.8) ----------------------------
 * geom/binning/image buffers are the ones the forward allocated.  All dL_* outputs are written
 * (zero for culled Gaussians); dL_dmeans2D is [P,3] (z unused), dL_dcov3D [P,6] and dL_dsh
 * [P,sh_M,3] may be NULL when not needed.  `workspace` must hold gpsg_rasterize_backward_workspace_bytes(P). */
GPSG_API size_t gpsg_rasterize_backward_workspace_bytes(int P);
GPSG_API int gpsg_rasterize_backward(const GpsgRasterSettings* settings, int device, void* stream, int P, int sh_M,
                            int32_t num_rendered, const float* means3D, const float* colors_precomp,
                            const float* shs, const float* opacities, const float* scales, const float* rotations,
                            const float* cov3D_precomp, const int32_t* radii, const void* geom_buffer,
                            const void* binning_buffer, const void* image_buffer, const float* dL_dout_color,
                            float* dL_dmeans2D, float* dL_dcolors, float* dL_dopacity, float* dL_dmeans3D,
                            float* dL_dcov3D, float* dL_dsh, float* dL_dscales, float* dL_drotations,
                            void* workspace);

/* ---- fused map -> Gaussian ingest: the rasterizer behind lib/GaussianRender.py:5-39 (pts2render) -------------------
 * Instead of boolean-mask gathering (10 `nonzero` host syncs per sample) and concatenating the two source views'
 * pixel-aligned maps into [P,k] tensors, the maps are read in place: per view v in {0,1} (lmain, rmain), with S2 =
 * pixels_per_view:  valid[v][S2] (uint8/bool), xyz[v][S2,3], img[v][3,S2] in [-1,1] (colour = img*0.5+0.5),
 * rot[v][4,S2], scale[v][3,S2], opacity[v][1,S2].  Gaussian index = v*S2 + pixel; invalid pixels are culled.
 * radii has 2*S2 entries.  Results (image, and gradients in map layout) equal the gather+render path. */
GPSG_API int gpsg_rasterize_forward_maps(const GpsgRasterSettings* settings, int device, void* stream, int pixels_per_view,
                                         const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                                         const float* const* rot, const float* const* scale, const float* const* opacity,
                                         float* out_color, int32_t* radii, gpsg_alloc_fn geom_alloc, void* geom_user,
                                         gpsg_alloc_fn binning_alloc, void* binning_user, gpsg_alloc_fn image_alloc,
                                         void* image_user, int32_t* num_rendered);
/* gpsg_rasterize_forward_maps in two halves, for a BATCH of samples with ONE host synchronisation (reference
 * lib/GaussianRender.py:8 loops over the samples; upstream synchronises once per sample to read num_rendered):
 *   _begin : projection, pairs-per-tile counts, tile ranges; allocates the geometry and image buffers through the callbacks
 *            (the caller keeps the pointers they returned) and enqueues a copy of 6 status words into `totals_host`
 *            (pinned host memory).  Does NOT synchronise.
 *   ... the caller synchronises `stream` once after the _begin calls of all samples ...
 *   _finish: sizes and allocates the binning buffer from totals_host, bins, sorts, composites into out_color.
 * Results are identical to gpsg_rasterize_forward_maps; the saved buffers feed gpsg_rasterize_backward_maps unchanged. */
GPSG_API int gpsg_rasterize_forward_maps_begin(const GpsgRasterSettings* settings, int device, void* stream, int pixels_per_view,
                                               const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                                               const float* const* rot, const float* const* scale,
                                               const float* const* opacity, int32_t* radii, gpsg_alloc_fn geom_alloc,
                                               void* geom_user, gpsg_alloc_fn image_alloc, void* image_user,
                                               uint32_t* totals_host /* >= 6 words, pinned */);
GPSG_API int gpsg_rasterize_forward_maps_finish(const GpsgRasterSettings* settings, int device, void* stream, int pixels_per_view,
                                                const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                                                const float* const* rot, const float* const* scale,
                                                const float* const* opacity, float* out_color, int32_t* radii,
                                                void* geom_buffer, void* image_buffer, gpsg_alloc_fn binning_alloc,
                                                void* binning_user, const uint32_t* totals_host, int32_t* num_rendered);

/* sync-free form of gpsg_rasterize_forward_maps (same contract as gpsg_rasterize_forward_planned; geom buffer sized for
 * P = 2*pixels_per_view): the serving loop of test_view_interp.py:39-47 renders many novel cameras from ONE pair's
 * cached maps without gathering them and without a host sync. */
GPSG_API int gpsg_rasterize_forward_maps_planned(const GpsgRasterSettings* settings, int device, void* stream,
                                                 int pixels_per_view, const uint8_t* const* valid, const float* const* xyz,
                                                 const float* const* img, const float* const* rot,
                                                 const float* const* scale, const float* const* opacity, float* out_color,
                                                 int32_t* radii, void* geom_buffer, void* binning_buffer,
                                                 int64_t capacity_pairs, void* image_buffer, uint32_t* status_host);
GPSG_API size_t gpsg_rasterize_backward_maps_workspace_bytes(int pixels_per_view);
GPSG_API int gpsg_rasterize_backward_maps(const GpsgRasterSettings* settings, int device, void* stream, int pixels_per_view,
                                          int32_t num_rendered, const uint8_t* const* valid, const float* const* xyz,
                                          const float* const* img, const float* const* rot, const float* const* scale,
                                          const float* const* opacity, const int32_t* radii, const void* geom_buffer,
                                          const void* binning_buffer, const void* image_buffer, const float* dL_dout_color,
                                          float* const* dL_dxyz, float* const* dL_dimg, float* const* dL_drot,
                                          float* const* dL_dscale, float* const* dL_dopacity, void* workspace);

/* ---- replaces _C.mark_visible : present[P] (uint8) = view-space z > 0.2 ---------------------- */
GPSG_API int gpsg_mark_visible(int device, void* stream, int P, const float* means3D, const float* viewmatrix_host16,
                      uint8_t* present);

/* Introspection of the saved buffers (used by the parity tests: "tile indices bit-exact").
 * Each returns a device pointer INTO the given buffer. */
typedef struct GpsgGeomView {
    const float* depths;         /* [P] */
    const float* means2D;        /* [P,2] */
    const float* conic_opacity;  /* [P,4] */
    const uint32_t* tiles_touched; /* [P] */
    const uint32_t* point_offsets; /* [P] inclusive scan */
} GpsgGeomView;
typedef struct GpsgBinningView {
    const uint64_t* point_list_keys; /* [N] sorted */
    const uint32_t* point_list;      /* [N] sorted Gaussian ids */
} GpsgBinningView;
typedef struct GpsgImageView {
    const float* final_T;       /* [H*W] */
    const uint32_t* n_contrib;  /* [H*W] */
    const uint32_t* ranges;     /* [tiles,2] */
} GpsgImageView;
GPSG_API int gpsg_geom_view(const void* geom_buffer, int P, GpsgGeomView* out);
GPSG_API int gpsg_binning_view(const void* binning_buffer, int64_t num_rendered, GpsgBinningView* out);
GPSG_API int gpsg_image_view(const void* image_buffer, int W, int H, GpsgImageView* out);

/* ---- replaces corr_sampler.forward (reference core/corr.py:22; SURVEY.md Appendix B) ---------
 * volume[B,H,W1,W2] with element strides (sb,sh,sw1; innermost contiguous), dtype 0=fp32 1=fp16;
 * coords: fp32, element (n,y,x) at coords[n*coords_sb + y*W1 + x] (channel 0 of [B,C,H,W1]);
 * out[B,2r+1,H,W1] contiguous, dtype of volume. */
GPSG_API int gpsg_corr_sampler_forward(int device, void* stream, int dtype, int B, int H, int W1, int W2, const void* volume,
                              int64_t sb, int64_t sh, int64_t sw1, const float* coords, int64_t coords_sb,
                              int radius, void* out);
/* ---- replaces corr_sampler.backward (reference core/corr.py:28) -------------------------------
 * grad_out[B,2r+1,H,W1] contiguous -> grad_volume[B,H,W1,W2] contiguous (fully written). */
GPSG_API int gpsg_corr_sampler_backward(int device, void* stream, int dtype, int B, int H, int W1, int W2,
                               const float* coords, int64_t coords_sb, const void* grad_out, int radius,
                               void* grad_volume);

/* ---- fused forms of the correlation block (reference core/corr.py:31-61), used by the mirrored CorrBlockFast1D ----
 * gpsg_corr_build_pyramid: fmap1[B,D,H,W1], fmap2[B,D,H,W2] (contiguous, dtype 0=fp32 1=fp16) ->
 *   vol[l][B,H,W1,W2>>l], l < levels<=4 : einsum/sqrt(D) then avg_pool2d([1,2]) per level, each level rounded to dtype.
 *   fp16 with D%16==0, D<=256, W1%8==0, W2%16==0, W2<=128 and 16-byte aligned pointers runs on tcgen05/TMEM (csrc/corr_tc.cu),
 *   anything else on the FFMA kernel (csrc/corr.cu); same rounding chain, results agree to one fp16 ulp.  The environment
 *   variable GPSG_CORR_BUILD=ffma forces the FFMA kernels (tests compare the two).
 * gpsg_corr_lookup_pyramid_forward: all levels of CorrBlockFast1D.__call__ in one launch -> out[B, levels*(2r+1), H, W1]
 *   (coords: channel 0 of [B,C,H,W1] fp32, level l uses coords / 2^l).  _backward: grad_out -> grad_vol[l] (fully written). */
GPSG_API int gpsg_corr_build_pyramid(int device, void* stream, int dtype, int B, int D, int H, int W1, int W2,
                                     const void* fmap1, const void* fmap2, void* const* vols, int levels);
/* backward of the build w.r.t. the feature maps: grad_vol0[B,H,W1,W2] (pooled levels already folded in) -> d fmap1, d fmap2 */
GPSG_API int gpsg_corr_build_backward(int device, void* stream, int dtype, int B, int D, int H, int W1, int W2,
                                      const void* fmap1, const void* fmap2, const void* grad_vol0, void* dfmap1,
                                      void* dfmap2);
GPSG_API int gpsg_corr_lookup_pyramid_forward(int device, void* stream, int dtype, int B, int H, int W1,
                                              const void* const* vols, const int32_t* widths, int levels,
                                              const float* coords, int64_t coords_sb, int radius, void* out);
GPSG_API int gpsg_corr_lookup_pyramid_backward(int device, void* stream, int dtype, int B, int H, int W1,
                                               void* const* grad_vols, const int32_t* widths, int levels,
                                               const float* coords, int64_t coords_sb, int radius, const void* grad_out);

/* ---- fused unprojection, the producer of the rasterizer's means3D (reference lib/network.py:64-69 -> lib/utils.py:87-119:
 * flow2depth + depth2pc + `depth != 0`).  flow_pred[B,1,S,S], mask[B,C,S,S] (channel 0 used; batch stride in elements),
 * intr[B,3,3], extr[B,extr_rows>=3,4], ref_intr[B,3,3], Tf_x[B]  ->  depth[B,1,S,S], xyz[B,S*S,3], valid[B,S*S] (uint8).
 * Backward: dL_dxyz (and optionally an incoming dL_ddepth) -> dL_dflow[B,1,S,S]. */
GPSG_API int gpsg_unproject_forward(int device, void* stream, int B, int S, const float* flow_pred, const float* mask,
                                    int64_t mask_batch_stride, const float* intr, const float* extr, int extr_rows,
                                    const float* ref_intr, const float* Tf_x, float* depth, float* xyz, uint8_t* valid);
GPSG_API int gpsg_unproject_backward(int device, void* stream, int B, int S, const float* depth, const float* mask,
                                     int64_t mask_batch_stride, const float* intr, const float* extr, int extr_rows,
                                     const float* ref_intr, const float* Tf_x, const float* dL_dxyz,
                                     const float* dL_ddepth, float* dL_dflow);

/* ---- stage-1 validation preview: replaces TaichiRenderBatch.flow2render (reference lib/TaichiRender.py:26-60) ----------
 * Per source view v in {0: lmain, 1: rmain} (pointer arrays of 2, like the *_maps entries): flow_pred[v][B,1,S,S],
 * mask[v] (channel 0 of [B,C,S,S]; mask_batch_stride[v], HOST array of 2, in elements), intr[v][B,3,3],
 * extr[v][B,extr_rows>=3,4], ref_intr[v][B,3,3], Tf_x[v][B], img[v][B,3,S,S] in [-1,1].  novel_calib[B,3,4] = K E of the
 * novel camera.  Each pixel with depth != 0 is unprojected (as gpsg_unproject_forward), projected into the novel camera
 * (x, y pixel coordinates; inv = 1/(z + 1e-8)) and splatted onto pixel (clamp(trunc x), clamp(trunc y)) -- off-screen
 * points land on the border, as upstream -- keeping the point with the largest inv >= 0, the last one in (view, pixel)
 * order on ties.  That is the sequential reading of upstream's racy atomic_max kernel; the result is deterministic.
 * Only samples b < bs are rendered (upstream's Taichi field has bs rows); the others stay background.
 * out_color[B,3,res,res] = the winner's raw img value, -1 where no point landed; out_inv_depth[B,res,res] (optional,
 * may be NULL) = its inv, 0 where none.  Requires S == res, bs <= B and 2*S*S + 1 < 2^32.
 * workspace (>= gpsg_flow2render_workspace_bytes(B, res), 8-byte aligned) holds the z-buffer of 64-bit keys
 * (inv bits << 32 | v*S*S + pixel + 1; 0 = no point), left in place after the call.
 * One memset and two kernel launches; no host synchronisation. */
GPSG_API size_t gpsg_flow2render_workspace_bytes(int B, int res);
GPSG_API int gpsg_flow2render(int device, void* stream, int B, int bs, int S, int res, const float* const* flow_pred,
                              const float* const* mask, const int64_t* mask_batch_stride, const float* const* intr,
                              const float* const* extr, int extr_rows, const float* const* ref_intr,
                              const float* const* Tf_x, const float* const* img, const float* novel_calib,
                              void* workspace, size_t workspace_bytes, float* out_color, float* out_inv_depth);

/* ---- fused photometric loss on the rendered image (SURVEY.md 8f-4) -----------------------------------------------
 * replaces  0.8 * l1_loss(img, gt) + 0.2 * (1 - ssim(img, gt))  (train_stage2.py:70-72; lib/loss.py:35-72: 11x11 Gaussian
 * window sigma 1.5, zero padding, C1 = 0.01^2, C2 = 0.03^2, means over all planes*H*W elements) and its autograd.
 * img, gt: [planes, H, W] fp32 (planes = B*C).  out3 (device float[3]) = { w_l1*L1 + w_ssim*(1-SSIM), L1, SSIM }.
 * dmaps (device float[3*planes*H*W], NULL when no gradient is needed) keeps the per-pixel SSIM partials for the backward,
 * which writes dimg = grad_loss * d(out3[0])/d(img); grad_loss is a DEVICE pointer to one float (NULL = 1). */
GPSG_API size_t gpsg_l1_ssim_workspace_bytes(int planes, int H, int W);
GPSG_API int gpsg_l1_ssim_forward(int device, void* stream, int planes, int H, int W, const float* img, const float* gt,
                                  float w_l1, float w_ssim, float* out3, float* dmaps, void* workspace);
GPSG_API int gpsg_l1_ssim_backward(int device, void* stream, int planes, int H, int W, const float* img, const float* gt,
                                   const float* dmaps, float w_l1, float w_ssim, const float* grad_loss, float* dimg);

/* ---- measurement hooks (used by bench.py; off by default) -----------------------------------
 * When enabled, every stage of the forward/backward is bracketed by CUDA events on the launching stream.
 * gpsg_profile_read() synchronises, then returns for stage i: total_ms[i] (summed over the calls since the last
 * reset), calls[i] and the number of kernel launches[i]; it returns the number of stages (names via
 * gpsg_profile_stage_name) and resets the accumulators.  Process-wide (autograd runs backward nodes on its own thread).  on = 2 counts launches only (no events: nothing is
 * inserted into the streams, for timed regions that should only be counted). */
/* fp16 correlation-volume build / backward: 0 = tcgen05 + TMEM kernels when the shape fits (default), 1 = FFMA kernels.
 * Process-wide switch for comparing the two formulations (tests, bench.py); GPSG_CORR_BUILD=ffma sets the initial value. */
GPSG_API int gpsg_set_corr_build(int mode);
GPSG_API int gpsg_profile_enable(int on);
GPSG_API int gpsg_profile_read(float* total_ms, int32_t* calls, int32_t* launches, int capacity);
GPSG_API const char* gpsg_profile_stage_name(int stage);

#ifdef __cplusplus
}
#endif
#endif /* GPSG_H */
