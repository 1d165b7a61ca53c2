// gpsg_internal.cuh -- shared declarations of libgpsg_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "../../include/gpsg.h"

#define GPSG_TILE_X 16
#define GPSG_TILE_Y 16
#define GPSG_TILE_PIX 256

namespace gpsg {

void set_error(const char* fmt, ...);

#define GPSG_CUDA(expr)                                                                         \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            gpsg::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return GPSG_E_CUDA;                                                                 \
        }                                                                                       \
    } while (0)
#define GPSG_LAUNCH_CHECK() GPSG_CUDA(cudaGetLastError())
#define GPSG_REQUIRE(cond, msg)                                  \
    do {                                                         \
        if (!(cond)) {                                           \
            gpsg::set_error("%s:%d: %s", __FILE__, __LINE__, msg); \
            return GPSG_E_INVALID;                               \
        }                                                        \
    } while (0)

// Camera block passed by value (__grid_constant__) to kernels.
struct Camera {
    float view[16];
    float proj[16];
    float tanfovx, tanfovy, focal_x, focal_y;
    float scale_modifier;
    int W, H, grid_x, grid_y;
    float bg[3];
    float campos[3];
};
Camera make_camera(const GpsgRasterSettings& s);


// ---- where the per-Gaussian inputs / gradients live -------------------------------------------------------------
// AoS mode: the gathered [P,k] tensors the reference passes to GaussianRasterizer (gaussian_renderer/__init__.py:54-62).
// Map mode (S2 > 0): the fused ingest of lib/GaussianRender.py:14-33 -- two pixel-aligned source views with S2 pixels
// each, read in place (xyz[S2,3] AoS, CHW planes for img/rot/scale/opacity, a validity mask); Gaussian i = view*S2 +
// pixel, invalid pixels are culled in-kernel, colours are img*0.5+0.5.  Same relative order as the reference's
// boolean-mask gather + concat, so results are identical.
struct GaussianSrc {
    const float* means3D; const float* scales; const float* rots; const float* opacities; const float* colors;
    const float* cov3D_precomp;
    int S2;
    const uint8_t* valid[2]; const float* xyz[2]; const float* img[2]; const float* rot[2]; const float* scale[2];
    const float* opac[2];
};
struct GaussianGrads {
    float* dmeans3D; float* dscales; float* drots; float* dopacity; float* dcov3D;         // AoS mode
    float* dxyz[2]; float* dimg[2]; float* drot[2]; float* dscale[2]; float* dopac[2];     // map mode
};
#ifdef __CUDACC__
// geometry of Gaussian i; false = not a Gaussian (invalid pixel)
__device__ __forceinline__ bool src_geom(const GaussianSrc& s, int i, float& x, float& y, float& z, float sc[3], float4& q,
                                         float& op) {
    if (s.S2 == 0) {
        const float* m = s.means3D + 3 * (size_t)i;
        x = m[0]; y = m[1]; z = m[2];
        if (!s.cov3D_precomp) {
            const float* sp = s.scales + 3 * (size_t)i;
            sc[0] = sp[0]; sc[1] = sp[1]; sc[2] = sp[2];
            const float* rp = s.rots + 4 * (size_t)i;
            q = ((reinterpret_cast<uintptr_t>(s.rots) & 15) == 0) ? __ldg(reinterpret_cast<const float4*>(rp))
                                                                   : make_float4(rp[0], rp[1], rp[2], rp[3]);
        }
        op = s.opacities[i];
        return true;
    }
    const int v = i >= s.S2 ? 1 : 0, px = i - v * s.S2;
    if (!s.valid[v][px]) return false;
    const float* xyz = s.xyz[v] + 3 * (size_t)px;
    x = xyz[0]; y = xyz[1]; z = xyz[2];
    const size_t S2 = (size_t)s.S2;
    sc[0] = s.scale[v][px]; sc[1] = s.scale[v][S2 + px]; sc[2] = s.scale[v][2 * S2 + px];
    q = make_float4(s.rot[v][px], s.rot[v][S2 + px], s.rot[v][2 * S2 + px], s.rot[v][3 * S2 + px]);
    op = s.opac[v][px];
    return true;
}
__device__ __forceinline__ void src_color(const GaussianSrc& s, uint32_t id, float& r, float& g, float& b) {
    if (s.S2 == 0) { r = s.colors[3 * id]; g = s.colors[3 * id + 1]; b = s.colors[3 * id + 2]; return; }
    const int v = (int)id >= s.S2 ? 1 : 0;
    const size_t px = id - (uint32_t)(v * s.S2), S2 = (size_t)s.S2;
    r = s.img[v][px] * 0.5f + 0.5f; g = s.img[v][S2 + px] * 0.5f + 0.5f; b = s.img[v][2 * S2 + px] * 0.5f + 0.5f;
}
#endif

static inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

// ---- saved-state layouts (carved from the caller-allocated byte buffers) -------------------
struct GeomState {
    float* depths;            // [P]
    float2* means2D;          // [P]
    float4* conic_opacity;    // [P]
    float* rgb;               // [P,3]   (SH path only; colours converted from SH)
    uint8_t* clamped;         // [P,3]   (SH path only)
    uint32_t* tiles_touched;  // [P]
    uint32_t* point_offsets;  // [P]
    void* scan_temp;
    size_t scan_temp_bytes;
    static size_t required(int P, size_t scan_temp_bytes);
    static GeomState carve(void* base, int P, size_t scan_temp_bytes);
};
struct BinningState {
    uint2* bucket;            // [N] tile-bucketed (depth bits, id), unordered inside a tile (aliases keys_unsorted)
    uint64_t* keys_unsorted;  // [N]
    uint32_t* vals_unsorted;  // [N]
    uint64_t* keys;           // [N] sorted (tile<<32 | depth bits)
    uint32_t* vals;           // [N] sorted Gaussian ids ("point_list")
    float4* slabA;            // [N] (x, y, cull half-extent x, y)     sorted, tile-contiguous
    float4* slabB;            // [N] (-0.5*log2e*conic.x, -log2e*conic.y, -0.5*log2e*conic.z, opacity)
    float4* slabC;            // [N] (r, g, b, Gaussian id bits)
    void* sort_temp;
    size_t sort_temp_bytes;
    static size_t required(size_t N, size_t sort_temp_bytes);
    static BinningState carve(void* base, size_t N, size_t sort_temp_bytes);
};
struct ImageState {
    float* final_T;       // [HW]
    uint32_t* n_contrib;  // [HW]
    uint2* ranges;        // [tiles]
    uint32_t* tile_count; // [tiles]  pairs per tile (counted by preprocess)
    uint32_t* tile_cursor;// [tiles]  scatter cursors
    uint32_t* totals;     // [64]     N, max count, overflow flag, #big tiles, preprocess CTA ticket (see tile_scan.cuh)
    uint32_t* big_tiles;  // [tiles]  ids of tiles with more than kBigTile pairs
    uint32_t* tile_order; // [tiles]  all tile ids, longest list first (tile_scan.cuh): work order of the compositing kernels
    static size_t required(int W, int H);
    static ImageState carve(void* base, int W, int H);
};
size_t scan_temp_bytes(int P);
size_t sort_temp_bytes(size_t N, int end_bit);

// ---- kernel launchers (each enqueues on `stream`) ------------------------------------------
// raster_preprocess.cu  (compiled with -fmad=false: integer outputs follow the oracle's op order)
int launch_preprocess(const Camera& cam, int P, const GaussianSrc& src, int32_t* radii, GeomState g, ImageState im,
                      uint32_t capacity, cudaStream_t stream);   // also runs the tile scan (last CTA)
int launch_mark_visible(int P, const float* means3D, const float* view16_host, uint8_t* present, cudaStream_t stream);
// raster_binning.cu
int run_scan(GeomState g, int P, cudaStream_t stream);
int launch_duplicate(const Camera& cam, int P, const int32_t* radii, GeomState g, BinningState b, cudaStream_t stream);
int run_sort(BinningState b, size_t N, int end_bit, cudaStream_t stream);
int launch_gather_ranges(const Camera& cam, size_t N, const GaussianSrc& src, GeomState g, BinningState b, ImageState im,
                         cudaStream_t stream);
// tile-bucket path (default): counts -> ranges, bucket scatter, per-tile in-CTA sort fused with the slab gather
constexpr uint32_t kMaxTileSort = 4096;  // largest tile list the in-CTA sort handles (256 thr x 16 keys); beyond: radix path
int launch_tile_scan(const Camera& cam, ImageState im, uint32_t capacity /*0 = unbounded*/, cudaStream_t stream);
int launch_bucket_scatter(const Camera& cam, int P, const int32_t* radii, GeomState g, BinningState b, ImageState im,
                          cudaStream_t stream);
int launch_tile_sort_gather(const Camera& cam, int P, uint32_t max_count, const GaussianSrc& src, GeomState g,
                            BinningState b, ImageState im, cudaStream_t stream);
// raster_render.cu
int launch_render_forward(const Camera& cam, BinningState b, ImageState im, float* out_color, cudaStream_t stream);
// raster_backward.cu
// grad_acc: [P] rows of 3 x float4 (12 floats, zero-initialised by the caller) -- the packed accumulator of the
// compositing backward: (S s dx, S s dy, S s dx^2, S s dx dy | S s dy^2, S s, S w g_r, S w g_g | S w g_b, -, -, -)
int launch_render_backward(const Camera& cam, BinningState b, ImageState im, const float* dL_dpix, float4* grad_acc,
                           cudaStream_t stream);
int launch_preprocess_backward(const Camera& cam, int P, const GaussianSrc& src, const int32_t* radii,
                               const float4* conic_opacity, const float4* grad_acc, float* dL_dmeans2D /* out [P,3] */,
                               float* dL_dcolors /* out [P,3] or NULL */, const GaussianGrads& out, cudaStream_t stream);
// sh.cu
int launch_sh_forward(int P, int deg, int M, const float* campos3, const float* means3D, const float* shs,
                      const int32_t* radii, float* rgb, uint8_t* clamped, cudaStream_t stream);
int launch_sh_backward(int P, int deg, int M, const float* campos3, const float* means3D, const float* shs,
                       const int32_t* radii, const uint8_t* clamped, const float* dL_dcolors, float* dL_dsh,
                       float* dL_dmeans3D, cudaStream_t stream);
// unproject.cu
int launch_unproject_fwd(int B, int S, const float* flow, const float* mask, int64_t mask_bs, const float* intr,
                         const float* extr, int extr_rows, const float* ref_intr, const float* Tf_x, float* depth,
                         float* xyz, uint8_t* valid, cudaStream_t stream);
int launch_unproject_bwd(int B, int S, const float* depth, const float* mask, int64_t mask_bs, const float* intr,
                         const float* extr, int extr_rows, const float* ref_intr, const float* Tf_x,
                         const float* dL_dxyz, const float* dL_ddepth, float* dL_dflow, cudaStream_t stream);
// point_splat.cu (compiled with -fmad=false: the CPU oracle replays its fp32 op order)
struct FlowSplatViews {   // per source view v in {0: lmain, 1: rmain}; passed by value to the kernel
    const float* flow[2]; const float* mask[2]; int64_t mask_bs[2]; const float* intr[2]; const float* extr[2];
    int extr_rows; const float* ref_intr[2]; const float* Tf_x[2]; const float* img[2];
};
int launch_flow2render(int B, int bs, int S, int res, const FlowSplatViews& in, const float* calib, void* zbuf,
                       float* color, float* inv_depth, cudaStream_t stream);
// corr.cu
int corr_build_mode();           // 0 = tcgen05 when possible, 1 = FFMA kernels
void set_corr_build_mode(int m);
int launch_corr_fwd(int dtype, int B, int H, int W1, int W2, const void* vol, int64_t sb, int64_t sh, int64_t sw1,
                    const float* coords, int64_t csb, int r, void* out, cudaStream_t stream);
int launch_corr_bwd(int dtype, int B, int H, int W1, int W2, const float* coords, int64_t csb, const void* gout, int r,
                    void* gvol, cudaStream_t stream);
int launch_corr_build(int dtype, int B, int D, int H, int W1, int W2, const void* f1, const void* f2, void* v0, void* v1,
                      void* v2, void* v3, int levels, cudaStream_t stream);
bool corr_build_tc_supported(int dtype, int D, int W1, int W2, const void* f1, const void* f2, void* const* v, int levels);
int launch_corr_build_tc(int B, int D, int H, int W1, int W2, const void* f1, const void* f2, void* v0, void* v1, void* v2,
                         void* v3, int levels, cudaStream_t stream);
bool corr_build_bwd_tc_supported(int dtype, int D, int W1, int W2, const void* f1, const void* f2, const void* g,
                                 const void* d1, const void* d2);
int launch_corr_build_bwd_tc(int B, int D, int H, int W1, int W2, const void* f1, const void* f2, const void* g, void* df1,
                             void* df2, cudaStream_t stream);
int launch_corr_build_bwd(int dtype, int B, int D, int H, int W1, int W2, const void* f1, const void* f2, const void* g,
                          void* df1, void* df2, cudaStream_t stream);
int launch_corr_lookup_fwd(int dtype, int B, int H, int W1, const void* const* vols, const int* widths, int levels,
                           const float* coords, int64_t csb, int r, void* out, cudaStream_t stream);
int launch_corr_lookup_bwd(int dtype, int B, int H, int W1, void* const* gvols, const int* widths, int levels,
                           const float* coords, int64_t csb, int r, const void* gout, cudaStream_t stream);

size_t l1_ssim_workspace_bytes(int planes, int H, int W);
int launch_l1_ssim_fwd(int planes, int H, int W, const float* img, const float* gt, float w_l1, float w_ssim, float* out3,
                       float* dmaps, void* workspace, cudaStream_t stream);
int launch_l1_ssim_bwd(int planes, int H, int W, const float* img, const float* gt, const float* dmaps, float w_l1,
                       float w_ssim, const float* grad_loss, float* dimg, cudaStream_t stream);

// ---- optional per-stage timing (bench.py); see gpsg_profile_* in gpsg.h ---------------------
enum Stage { ST_PREPROCESS = 0, ST_SCAN, ST_DUPLICATE, ST_SORT, ST_GATHER, ST_TILE_SCAN, ST_SCATTER, ST_TILE_SORT, ST_RENDER_FWD, ST_RENDER_BWD,
             ST_PREPROCESS_BWD, ST_CORR_FWD, ST_CORR_BWD, ST_CORR_BUILD, ST_COUNT };
struct StageTimer {  // RAII: records begin/end events on `stream` when profiling is on
    StageTimer(Stage s, cudaStream_t stream, int launches);
    ~StageTimer();
    Stage stage; cudaStream_t stream; void* slot;
};

}  // namespace gpsg
