// gpsg_capi.cu -- the extern "C" boundary of libgpsg_sm100.so (declared in include/gpsg.h).
// Host-side orchestration only; kernels live in raster_*.cu / corr.cu.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include "gpsg_internal.cuh"

namespace gpsg {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

Camera make_camera(const GpsgRasterSettings& s) {
    Camera c;
    memcpy(c.view, s.viewmatrix, sizeof(c.view));
    memcpy(c.proj, s.projmatrix, sizeof(c.proj));
    c.tanfovx = s.tanfovx;
    c.tanfovy = s.tanfovy;
    c.W = s.image_width;
    c.H = s.image_height;
    c.focal_x = (float)c.W / (2.0f * s.tanfovx);
    c.focal_y = (float)c.H / (2.0f * s.tanfovy);
    c.scale_modifier = s.scale_modifier;
    c.grid_x = (c.W + GPSG_TILE_X - 1) / GPSG_TILE_X;
    c.grid_y = (c.H + GPSG_TILE_Y - 1) / GPSG_TILE_Y;
    for (int k = 0; k < 3; ++k) { c.bg[k] = s.bg[k]; c.campos[k] = s.campos[k]; }
    return c;
}

// ---- buffer layouts -------------------------------------------------------------------------
template <typename T>
static inline T* take(char*& p, size_t count) {
    T* r = reinterpret_cast<T*>(p);
    p += align_up(count * sizeof(T));
    return r;
}

static GeomState carve_geom(char* p, int P, size_t scan_bytes, char** end) {
    GeomState g;
    const size_t n = (size_t)(P > 0 ? P : 1);
    g.depths = take<float>(p, n);
    g.means2D = take<float2>(p, n);
    g.conic_opacity = take<float4>(p, n);
    g.rgb = take<float>(p, 3 * n);
    g.clamped = take<uint8_t>(p, 3 * n);
    g.tiles_touched = take<uint32_t>(p, n);
    g.point_offsets = take<uint32_t>(p, n);
    g.scan_temp = p;
    g.scan_temp_bytes = scan_bytes;
    p += align_up(scan_bytes);
    if (end) *end = p;
    return g;
}
size_t GeomState::required(int P, size_t scan_bytes) {
    char* end = nullptr;
    carve_geom(nullptr, P, scan_bytes, &end);
    return (size_t)(end - (char*)nullptr) + 256;
}
GeomState GeomState::carve(void* base, int P, size_t scan_bytes) {
    return carve_geom((char*)align_up((size_t)base), P, scan_bytes, nullptr);
}

static BinningState carve_binning(char* p, size_t N, size_t sort_bytes, char** end) {
    BinningState b;
    const size_t n = N > 0 ? N : 1;
    b.slabA = take<float4>(p, n);
    b.slabB = take<float4>(p, n);
    b.slabC = take<float4>(p, n);
    b.keys = take<uint64_t>(p, n);
    b.vals = take<uint32_t>(p, n);
    b.keys_unsorted = take<uint64_t>(p, n);
    b.bucket = reinterpret_cast<uint2*>(b.keys_unsorted);   // tile-bucket path: same bytes, never both in use
    b.vals_unsorted = take<uint32_t>(p, n);
    b.sort_temp = p;
    b.sort_temp_bytes = sort_bytes;
    p += align_up(sort_bytes);
    if (end) *end = p;
    return b;
}
size_t BinningState::required(size_t N, size_t sort_bytes) {
    char* end = nullptr;
    carve_binning(nullptr, N, sort_bytes, &end);
    return (size_t)(end - (char*)nullptr) + 256;
}
BinningState BinningState::carve(void* base, size_t N, size_t sort_bytes) {
    return carve_binning((char*)align_up((size_t)base), N, sort_bytes, nullptr);
}

static ImageState carve_image(char* p, int W, int H, char** end) {
    ImageState im;
    const size_t hw = (size_t)W * H;
    const size_t tiles = (size_t)((W + GPSG_TILE_X - 1) / GPSG_TILE_X) * ((H + GPSG_TILE_Y - 1) / GPSG_TILE_Y);
    im.final_T = take<float>(p, hw > 0 ? hw : 1);
    im.n_contrib = take<uint32_t>(p, hw > 0 ? hw : 1);
    im.ranges = take<uint2>(p, tiles > 0 ? tiles : 1);
    im.tile_count = take<uint32_t>(p, tiles > 0 ? tiles : 1);
    im.totals = take<uint32_t>(p, 64);            // directly after tile_count: one memset clears both
    im.tile_cursor = take<uint32_t>(p, tiles > 0 ? tiles : 1);
    im.big_tiles = take<uint32_t>(p, tiles > 0 ? tiles : 1);
    im.tile_order = take<uint32_t>(p, tiles > 0 ? tiles : 1);
    if (end) *end = p;
    return im;
}
size_t ImageState::required(int W, int H) {
    char* end = nullptr;
    carve_image(nullptr, W, H, &end);
    return (size_t)(end - (char*)nullptr) + 256;
}
ImageState ImageState::carve(void* base, int W, int H) { return carve_image((char*)align_up((size_t)base), W, H, nullptr); }


static GaussianSrc aos_src(const float* means3D, const float* scales, const float* rots, const float* opacities,
                           const float* colors, const float* cov3D_precomp) {
    GaussianSrc src;
    memset(&src, 0, sizeof(src));
    src.means3D = means3D; src.scales = scales; src.rots = rots; src.opacities = opacities; src.colors = colors;
    src.cov3D_precomp = cov3D_precomp;
    return src;
}

static int bit_length(uint32_t n) {
    int b = 0;
    while (n) { ++b; n >>= 1; }
    return b;
}

static bool force_radix_binning() {
    static const bool v = [] { const char* e = getenv("GPSG_BINNING"); return e && e[0] == 'r'; }();
    return v;
}

// pinned host slot for the one device->host read of the forward (num_rendered)
static uint32_t* pinned_slot() {
    static thread_local uint32_t* slot = nullptr;
    if (!slot) {
        if (cudaHostAlloc((void**)&slot, 64, cudaHostAllocDefault) != cudaSuccess) slot = nullptr;
    }
    return slot;
}

}  // namespace gpsg


// ---- profiling -------------------------------------------------------------------------------
#include <mutex>
#include <vector>
namespace gpsg {
struct ProfSlot { cudaEvent_t a, b; Stage stage; bool used; };
struct Profiler {
    int on = 0;                      // 0 off, 1 events + launch counts, 2 launch counts only
    std::vector<ProfSlot> slots;
    size_t next = 0;
    int launches[ST_COUNT] = {0};
};
// Process-wide (not thread-local): PyTorch runs autograd backward nodes on its own thread, and the backward launches of a
// training step must land in the same accumulators as the forward launches issued from the caller's thread.
static Profiler g_prof;
static std::mutex g_prof_mu;
static const char* kStageNames[ST_COUNT] = {"preprocess", "scan", "duplicate", "sort", "gather_ranges", "tile_scan",
                                            "bucket_scatter", "tile_sort_gather", "render_forward",
                                            "render_backward", "preprocess_backward", "corr_forward", "corr_backward", "corr_build"};
StageTimer::StageTimer(Stage s, cudaStream_t st, int launches) : stage(s), stream(st), slot(nullptr) {
    if (!g_prof.on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (g_prof.on == 2) { g_prof.launches[s] += launches; return; }
    if (g_prof.next == g_prof.slots.size()) {
        ProfSlot ps; ps.used = false;
        if (cudaEventCreate(&ps.a) != cudaSuccess || cudaEventCreate(&ps.b) != cudaSuccess) return;
        g_prof.slots.push_back(ps);
    }
    ProfSlot* p = &g_prof.slots[g_prof.next++];
    p->stage = s; p->used = true;
    g_prof.launches[s] += launches;
    cudaEventRecord(p->a, stream);
    slot = (void*)(uintptr_t)(g_prof.next);  // index+1 (vector may reallocate)
}
StageTimer::~StageTimer() {
    if (!slot) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    cudaEventRecord(g_prof.slots[(size_t)(uintptr_t)slot - 1].b, stream);
}
}  // namespace gpsg

using namespace gpsg;

extern "C" {

GPSG_API const char* gpsg_last_error(void) { return g_err; }
int gpsg_version(void) { return 100; }

// The exact (one host read) forward in two halves, so that a BATCH of samples needs one host synchronisation in total
// (lib/GaussianRender.py:8 loops over the samples; upstream synchronises once per sample to read num_rendered):
//   begin  : projection + pairs-per-tile counts + tile ranges; enqueues the copy of the status words (N, longest list, ...)
//            into `totals_host` (pinned, >= 6 words).  No synchronisation.
//   finish : (after the caller synchronised the stream once for all samples) sizes the binning buffer from totals_host,
//            bins, sorts and composites.
// `src` says where the Gaussians come from (AoS tensors or maps).
static int forward_exact_begin(const GpsgRasterSettings* s, int device, cudaStream_t stream, int P, const GaussianSrc& src,
                               int32_t* radii, gpsg_alloc_fn geom_alloc, void* geom_user, gpsg_alloc_fn image_alloc,
                               void* image_user, uint32_t* totals_host, void** geom_out, void** image_out) {
    GPSG_CUDA(cudaSetDevice(device));
    const Camera cam = make_camera(*s);
    const size_t scan_bytes = scan_temp_bytes(P);
    void* geom_base = geom_alloc(geom_user, GeomState::required(P, scan_bytes));
    if (!geom_base) { set_error("geometry allocator returned NULL"); return GPSG_E_ALLOC; }
    GeomState g = GeomState::carve(geom_base, P, scan_bytes);
    void* img_base = image_alloc(image_user, ImageState::required(cam.W, cam.H));
    if (!img_base) { set_error("image allocator returned NULL"); return GPSG_E_ALLOC; }
    ImageState im = ImageState::carve(img_base, cam.W, cam.H);
    if (geom_out) *geom_out = geom_base;
    if (image_out) *image_out = img_base;
    int rc = GPSG_OK;
    GPSG_CUDA(cudaMemsetAsync(im.tile_count, 0, (size_t)((char*)(im.totals + 64) - (char*)im.tile_count), stream));
    if (P > 0) {   // projection + pairs-per-tile histogram; its last CTA also scans the histogram into tile ranges
        { StageTimer t(ST_PREPROCESS, stream, 1); rc = launch_preprocess(cam, P, src, radii, g, im, 0u, stream); }
        if (rc) return rc;
        GPSG_CUDA(cudaMemcpyAsync(totals_host, im.totals, 6 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    } else {
        { StageTimer t(ST_TILE_SCAN, stream, 1); rc = launch_tile_scan(cam, im, 0u, stream); }
        if (rc) return rc;
        for (int k = 0; k < 6; ++k) totals_host[k] = 0u;
    }
    return GPSG_OK;
}

static int forward_exact_finish(const GpsgRasterSettings* s, int device, cudaStream_t stream, int P, int sh_M, GaussianSrc src,
                                const float* shs, float* out_color, int32_t* radii, void* geom_base, void* img_base,
                                gpsg_alloc_fn binning_alloc, void* binning_user, const uint32_t* totals_host,
                                int32_t* num_rendered) {
    GPSG_CUDA(cudaSetDevice(device));
    const Camera cam = make_camera(*s);
    GeomState g = GeomState::carve(geom_base, P, scan_temp_bytes(P));
    ImageState im = ImageState::carve(img_base, cam.W, cam.H);
    const int tiles = cam.grid_x * cam.grid_y;
    const uint32_t N = totals_host[0], max_count = totals_host[1];
    GPSG_REQUIRE(totals_host[5] == 0u, "more than 2^31 (tile, Gaussian) pairs: the splats cover (almost) the whole image each -- "
                                       "degenerate scene (32-bit pair offsets, as in the upstream rasterizer)");
    int rc = GPSG_OK;
    if (num_rendered) *num_rendered = (int32_t)N;
    if (shs && P > 0) {   // SH -> RGB for the visible Gaussians (kept in the geometry buffer for the backward)
        rc = launch_sh_forward(P, s->sh_degree, sh_M, s->campos, src.means3D, shs, radii, g.rgb, g.clamped, stream);
        if (rc) return rc;
        src.colors = g.rgb;
    }

    const bool radix_path = max_count > kMaxTileSort || force_radix_binning();
    const int end_bit = 32 + bit_length((uint32_t)tiles);
    const size_t sort_bytes = radix_path ? sort_temp_bytes(N, end_bit) : 0;
    void* bin_base = binning_alloc(binning_user, BinningState::required(N, sort_bytes));
    if (!bin_base) { set_error("binning allocator returned NULL"); return GPSG_E_ALLOC; }
    BinningState b = BinningState::carve(bin_base, N, sort_bytes);

    if (N > 0 && !radix_path) {
        // tile-bucket binning: scatter into per-tile buckets, sort each tile inside one CTA, gather slabs
        { StageTimer t(ST_SCATTER, stream, 1); rc = launch_bucket_scatter(cam, P, radii, g, b, im, stream); }
        if (rc) return rc;
        { StageTimer t(ST_TILE_SORT, stream, max_count > 2048 ? 2 : 1); rc = launch_tile_sort_gather(cam, P, max_count, src, g, b, im, stream); }
        if (rc) return rc;
    } else if (N > 0) {
        // fallback (a tile list too long for the in-CTA sort, or GPSG_BINNING=radix): upstream-style global radix sort
        { StageTimer t(ST_SCAN, stream, 2); rc = run_scan(g, P, stream); }
        if (rc) return rc;
        { StageTimer t(ST_DUPLICATE, stream, 1); rc = launch_duplicate(cam, P, radii, g, b, stream); }
        if (rc) return rc;
        { StageTimer t(ST_SORT, stream, 2 + (end_bit + 7) / 8); rc = run_sort(b, N, end_bit, stream); }
        if (rc) return rc;
        { StageTimer t(ST_GATHER, stream, 1); rc = launch_gather_ranges(cam, N, src, g, b, im, stream); }
        if (rc) return rc;
    }
    { StageTimer t(ST_RENDER_FWD, stream, 1); rc = launch_render_forward(cam, b, im, out_color, stream); }
    if (rc) return rc;
    if (s->debug) GPSG_CUDA(cudaStreamSynchronize(stream));
    return GPSG_OK;
}

static int forward_exact(const GpsgRasterSettings* s, int device, cudaStream_t stream, int P, int sh_M, GaussianSrc src,
                         const float* shs, float* out_color, int32_t* radii, gpsg_alloc_fn geom_alloc, void* geom_user,
                         gpsg_alloc_fn binning_alloc, void* binning_user, gpsg_alloc_fn image_alloc, void* image_user,
                         int32_t* num_rendered) {
    uint32_t* slot = pinned_slot();      // thread-local pinned words for the one device->host read of this forward
    GPSG_REQUIRE(slot != nullptr, "cudaHostAlloc failed");
    void *geom_base = nullptr, *img_base = nullptr;
    int rc = forward_exact_begin(s, device, stream, P, src, radii, geom_alloc, geom_user, image_alloc, image_user, slot,
                                 &geom_base, &img_base);
    if (rc) return rc;
    if (P > 0) GPSG_CUDA(cudaStreamSynchronize(stream));
    return forward_exact_finish(s, device, stream, P, sh_M, src, shs, out_color, radii, geom_base, img_base, binning_alloc,
                                binning_user, slot, num_rendered);
}

int gpsg_rasterize_forward(const GpsgRasterSettings* s, int device, void* stream_, int P, int sh_M,
                           const float* means3D, const float* colors_precomp, const float* shs,
                           const float* opacities, const float* scales, const float* rotations,
                           const float* cov3D_precomp, float* out_color, int32_t* radii, gpsg_alloc_fn geom_alloc,
                           void* geom_user, gpsg_alloc_fn binning_alloc, void* binning_user,
                           gpsg_alloc_fn image_alloc, void* image_user, int32_t* num_rendered) {
    GPSG_REQUIRE(s != nullptr, "settings is NULL");
    GPSG_REQUIRE(P >= 0, "P < 0");
    GPSG_REQUIRE(s->image_width > 0 && s->image_height > 0, "image size must be positive");
    GPSG_REQUIRE(out_color != nullptr, "out_color is NULL");
    GPSG_REQUIRE(geom_alloc && binning_alloc && image_alloc, "allocator callback is NULL");
    if (P > 0) {
        GPSG_REQUIRE(means3D && opacities && radii, "means3D / opacities / radii is NULL");
        GPSG_REQUIRE((colors_precomp != nullptr) != (shs != nullptr),
                     "Please provide excatly one of either SHs or precomputed colors!");
        GPSG_REQUIRE(((scales != nullptr && rotations != nullptr) != (cov3D_precomp != nullptr)),
                     "Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
        if (shs) {
            GPSG_REQUIRE(s->sh_degree >= 0 && s->sh_degree <= 3, "sh_degree must be 0..3");
            GPSG_REQUIRE(sh_M >= (s->sh_degree + 1) * (s->sh_degree + 1), "shs has fewer coefficients than (sh_degree+1)^2");
        }
    }
    return forward_exact(s, device, (cudaStream_t)stream_, P, sh_M,
                         aos_src(means3D, cov3D_precomp ? nullptr : scales, cov3D_precomp ? nullptr : rotations, opacities,
                                 colors_precomp, cov3D_precomp),
                         shs, out_color, radii, geom_alloc, geom_user, binning_alloc, binning_user, image_alloc, image_user,
                         num_rendered);
}

static int check_maps(int S2, const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                      const float* const* rot, const float* const* scale, const float* const* opacity) {
    GPSG_REQUIRE(S2 > 0 && S2 < (1 << 30), "pixels per view must be positive");
    GPSG_REQUIRE(valid && xyz && img && rot && scale && opacity, "map pointer array is NULL");
    for (int v = 0; v < 2; ++v)
        GPSG_REQUIRE(valid[v] && xyz[v] && img[v] && rot[v] && scale[v] && opacity[v], "a source-view map is NULL");
    return GPSG_OK;
}
static GaussianSrc maps_src(int S2, const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                            const float* const* rot, const float* const* scale, const float* const* opacity) {
    GaussianSrc src;
    memset(&src, 0, sizeof(src));
    src.S2 = S2;
    for (int v = 0; v < 2; ++v) {
        src.valid[v] = valid[v]; src.xyz[v] = xyz[v]; src.img[v] = img[v]; src.rot[v] = rot[v]; src.scale[v] = scale[v];
        src.opac[v] = opacity[v];
    }
    return src;
}

int gpsg_rasterize_forward_maps(const GpsgRasterSettings* s, int device, void* stream_, int pixels_per_view,
                                const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                                const float* const* rot, const float* const* scale, const float* const* opacity,
                                float* out_color, int32_t* radii, gpsg_alloc_fn geom_alloc, void* geom_user,
                                gpsg_alloc_fn binning_alloc, void* binning_user, gpsg_alloc_fn image_alloc,
                                void* image_user, int32_t* num_rendered) {
    GPSG_REQUIRE(s != nullptr, "settings is NULL");
    GPSG_REQUIRE(s->image_width > 0 && s->image_height > 0, "image size must be positive");
    GPSG_REQUIRE(out_color && radii, "out_color / radii is NULL");
    GPSG_REQUIRE(geom_alloc && binning_alloc && image_alloc, "allocator callback is NULL");
    int rc = check_maps(pixels_per_view, valid, xyz, img, rot, scale, opacity);
    if (rc) return rc;
    return forward_exact(s, device, (cudaStream_t)stream_, 2 * pixels_per_view, 0,
                         maps_src(pixels_per_view, valid, xyz, img, rot, scale, opacity), nullptr, out_color, radii,
                         geom_alloc, geom_user, binning_alloc, binning_user, image_alloc, image_user, num_rendered);
}

int gpsg_rasterize_forward_maps_begin(const GpsgRasterSettings* s, int device, void* stream_, int pixels_per_view,
                                      const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                                      const float* const* rot, const float* const* scale, const float* const* opacity,
                                      int32_t* radii, gpsg_alloc_fn geom_alloc, void* geom_user, gpsg_alloc_fn image_alloc,
                                      void* image_user, uint32_t* totals_host) {
    GPSG_REQUIRE(s != nullptr, "settings is NULL");
    GPSG_REQUIRE(s->image_width > 0 && s->image_height > 0, "image size must be positive");
    GPSG_REQUIRE(radii && geom_alloc && image_alloc && totals_host, "radii / allocator / totals_host is NULL");
    int rc = check_maps(pixels_per_view, valid, xyz, img, rot, scale, opacity);
    if (rc) return rc;
    return forward_exact_begin(s, device, (cudaStream_t)stream_, 2 * pixels_per_view,
                               maps_src(pixels_per_view, valid, xyz, img, rot, scale, opacity), radii, geom_alloc, geom_user,
                               image_alloc, image_user, totals_host, nullptr, nullptr);
}

int gpsg_rasterize_forward_maps_finish(const GpsgRasterSettings* s, int device, void* stream_, int pixels_per_view,
                                       const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                                       const float* const* rot, const float* const* scale, const float* const* opacity,
                                       float* out_color, int32_t* radii, void* geom_buffer, void* image_buffer,
                                       gpsg_alloc_fn binning_alloc, void* binning_user, const uint32_t* totals_host,
                                       int32_t* num_rendered) {
    GPSG_REQUIRE(s != nullptr, "settings is NULL");
    GPSG_REQUIRE(out_color && radii && geom_buffer && image_buffer && binning_alloc && totals_host, "a required pointer is NULL");
    int rc = check_maps(pixels_per_view, valid, xyz, img, rot, scale, opacity);
    if (rc) return rc;
    return forward_exact_finish(s, device, (cudaStream_t)stream_, 2 * pixels_per_view, 0,
                                maps_src(pixels_per_view, valid, xyz, img, rot, scale, opacity), nullptr, out_color, radii,
                                geom_buffer, image_buffer, binning_alloc, binning_user, totals_host, num_rendered);
}

size_t gpsg_raster_geom_bytes(int P) { return GeomState::required(P > 0 ? P : 0, scan_temp_bytes(P > 0 ? P : 0)); }
size_t gpsg_raster_binning_bytes(int64_t capacity_pairs) { return BinningState::required((size_t)(capacity_pairs > 0 ? capacity_pairs : 0), 0); }
size_t gpsg_raster_image_bytes(int W, int H) { return ImageState::required(W, H); }
const uint32_t* gpsg_raster_status_ptr(const void* image_buffer, int W, int H) {
    if (!image_buffer || W <= 0 || H <= 0) return nullptr;
    return ImageState::carve(const_cast<void*>(image_buffer), W, H).totals;
}

static int forward_planned_common(const GpsgRasterSettings* s, int device, cudaStream_t stream, int P, const GaussianSrc& src,
                                  float* out_color, int32_t* radii, void* geom_buffer, void* binning_buffer,
                                  int64_t capacity_pairs, void* image_buffer, uint32_t* status_host) {
    GPSG_REQUIRE(s != nullptr, "settings is NULL");
    GPSG_REQUIRE(P > 0, "planned forward needs P > 0");
    GPSG_REQUIRE(s->image_width > 0 && s->image_height > 0, "image size must be positive");
    GPSG_REQUIRE(out_color && radii, "out_color / radii is NULL");
    GPSG_REQUIRE(geom_buffer && binning_buffer && image_buffer && capacity_pairs > 0 && capacity_pairs < (1ll << 31),
                 "planned forward: buffers / capacity missing");
    GPSG_CUDA(cudaSetDevice(device));
    const Camera cam = make_camera(*s);
    GeomState g = GeomState::carve(geom_buffer, P, 0);
    ImageState im = ImageState::carve(image_buffer, cam.W, cam.H);
    BinningState b = BinningState::carve(binning_buffer, (size_t)capacity_pairs, 0);
    int rc = GPSG_OK;
    GPSG_CUDA(cudaMemsetAsync(im.tile_count, 0, (size_t)((char*)(im.totals + 64) - (char*)im.tile_count), stream));
    { StageTimer t(ST_PREPROCESS, stream, 1); rc = launch_preprocess(cam, P, src, radii, g, im, (uint32_t)capacity_pairs, stream); }
    if (rc) return rc;
    if (status_host) GPSG_CUDA(cudaMemcpyAsync(status_host, im.totals, 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    { StageTimer t(ST_SCATTER, stream, 1); rc = launch_bucket_scatter(cam, P, radii, g, b, im, stream); }
    if (rc) return rc;
    { StageTimer t(ST_TILE_SORT, stream, 2); rc = launch_tile_sort_gather(cam, P, kMaxTileSort, src, g, b, im, stream); }
    if (rc) return rc;
    { StageTimer t(ST_RENDER_FWD, stream, 1); rc = launch_render_forward(cam, b, im, out_color, stream); }
    return rc;
}

int gpsg_rasterize_forward_planned(const GpsgRasterSettings* s, int device, void* stream_, int P, const float* means3D,
                                   const float* colors_precomp, const float* opacities, const float* scales,
                                   const float* rotations, const float* cov3D_precomp, float* out_color, int32_t* radii,
                                   void* geom_buffer, void* binning_buffer, int64_t capacity_pairs, void* image_buffer,
                                   uint32_t* status_host) {
    GPSG_REQUIRE(means3D && colors_precomp && opacities, "a required pointer is NULL");
    GPSG_REQUIRE(((scales != nullptr && rotations != nullptr) != (cov3D_precomp != nullptr)),
                 "Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
    return forward_planned_common(s, device, (cudaStream_t)stream_, P,
                                  aos_src(means3D, cov3D_precomp ? nullptr : scales, cov3D_precomp ? nullptr : rotations,
                                          opacities, colors_precomp, cov3D_precomp),
                                  out_color, radii, geom_buffer, binning_buffer, capacity_pairs, image_buffer, status_host);
}

int gpsg_rasterize_forward_maps_planned(const GpsgRasterSettings* s, int device, void* stream_, int pixels_per_view,
                                        const uint8_t* const* valid, const float* const* xyz, const float* const* img,
                                        const float* const* rot, const float* const* scale, const float* const* opacity,
                                        float* out_color, int32_t* radii, void* geom_buffer, void* binning_buffer,
                                        int64_t capacity_pairs, void* image_buffer, uint32_t* status_host) {
    int rc = check_maps(pixels_per_view, valid, xyz, img, rot, scale, opacity);
    if (rc) return rc;
    return forward_planned_common(s, device, (cudaStream_t)stream_, 2 * pixels_per_view,
                                  maps_src(pixels_per_view, valid, xyz, img, rot, scale, opacity), out_color, radii,
                                  geom_buffer, binning_buffer, capacity_pairs, image_buffer, status_host);
}

size_t gpsg_rasterize_backward_workspace_bytes(int P) {
    const size_t n = (size_t)(P > 0 ? P : 1);
    return align_up(sizeof(float4) * 3 * n) + align_up(sizeof(float) * 3 * n) + 256;   // packed accumulator rows, dL_dcolors (SH path)
}

static int backward_common(const GpsgRasterSettings* s, int device, cudaStream_t stream, int P, int sh_M,
                           int32_t num_rendered, const GaussianSrc& src, const float* shs, const int32_t* radii,
                           const void* geom_buffer, const void* binning_buffer, const void* image_buffer,
                           const float* dL_dout_color, float* dL_dmeans2D, float* dL_dcolors, float* dL_dsh,
                           const GaussianGrads& out, void* workspace) {
    GPSG_CUDA(cudaSetDevice(device));
    const Camera cam = make_camera(*s);
    BinningState b = BinningState::carve(const_cast<void*>(binning_buffer), (size_t)num_rendered, 0);
    ImageState im = ImageState::carve(const_cast<void*>(image_buffer), cam.W, cam.H);
    GeomState gst = GeomState::carve(const_cast<void*>(geom_buffer), P, 0);
    // one packed accumulator row (3 x float4) per Gaussian: the only buffer that needs zeroing -- the projection backward
    // writes d/dmeans2D and d/dcolours for every Gaussian
    float4* grad_acc = (float4*)align_up((size_t)workspace);
    if (!dL_dcolors && shs) dL_dcolors = (float*)((char*)grad_acc + align_up(sizeof(float4) * 3 * (size_t)P));   // SH path scratch
    GPSG_CUDA(cudaMemsetAsync(grad_acc, 0, sizeof(float4) * 3 * (size_t)P, stream));
    int rc = GPSG_OK;
    if (num_rendered > 0) {
        { StageTimer t(ST_RENDER_BWD, stream, 1); rc = launch_render_backward(cam, b, im, dL_dout_color, grad_acc, stream); }
        if (rc) return rc;
    }
    { StageTimer t(ST_PREPROCESS_BWD, stream, 1);
      rc = launch_preprocess_backward(cam, P, src, radii, gst.conic_opacity, grad_acc, dL_dmeans2D, dL_dcolors, out, stream); }
    if (rc) return rc;
    if (shs) {
        rc = launch_sh_backward(P, s->sh_degree, sh_M, s->campos, src.means3D, shs, radii, gst.clamped, dL_dcolors, dL_dsh,
                                out.dmeans3D, stream);
        if (rc) return rc;
    }
    if (s->debug) GPSG_CUDA(cudaStreamSynchronize(stream));
    return GPSG_OK;
}

int gpsg_rasterize_backward(const GpsgRasterSettings* s, int device, void* stream_, int P, int sh_M,
                            int32_t num_rendered, const float* means3D, const float* colors_precomp, const float* shs,
                            const float* opacities, const float* scales, const float* rotations,
                            const float* cov3D_precomp, const int32_t* radii, const void* geom_buffer,
                            const void* binning_buffer, const void* image_buffer, const float* dL_dout_color,
                            float* dL_dmeans2D, float* dL_dcolors, float* dL_dopacity, float* dL_dmeans3D,
                            float* dL_dcov3D, float* dL_dsh, float* dL_dscales, float* dL_drotations,
                            void* workspace) {
    GPSG_REQUIRE(s != nullptr, "settings is NULL");
    GPSG_REQUIRE(P >= 0 && num_rendered >= 0, "negative size");
    if (P == 0) return GPSG_OK;
    GPSG_REQUIRE(means3D && radii && geom_buffer && binning_buffer && image_buffer && dL_dout_color,
                 "a required input pointer is NULL");
    GPSG_REQUIRE(dL_dmeans2D && dL_dopacity && dL_dmeans3D && workspace, "a required output pointer is NULL");
    GPSG_REQUIRE((shs != nullptr) == (dL_dsh != nullptr), "dL_dsh must be given exactly when shs is");
    GPSG_REQUIRE(shs != nullptr || dL_dcolors != nullptr, "dL_dcolors is NULL");
    GPSG_REQUIRE((scales && rotations) || cov3D_precomp, "need scales+rotations or cov3D_precomp");
    cudaStream_t stream = (cudaStream_t)stream_;
    GaussianGrads out;
    memset(&out, 0, sizeof(out));
    out.dmeans3D = dL_dmeans3D; out.dopacity = dL_dopacity; out.dcov3D = dL_dcov3D;
    out.dscales = cov3D_precomp ? nullptr : dL_dscales;
    out.drots = cov3D_precomp ? nullptr : dL_drotations;
    int rc = backward_common(s, device, stream, P, sh_M, num_rendered,
                             aos_src(means3D, cov3D_precomp ? nullptr : scales, cov3D_precomp ? nullptr : rotations,
                                     opacities, colors_precomp, cov3D_precomp),
                             shs, radii, geom_buffer, binning_buffer, image_buffer, dL_dout_color, dL_dmeans2D, dL_dcolors,
                             dL_dsh, out, workspace);
    if (rc) return rc;
    if (cov3D_precomp) {
        if (dL_dscales) GPSG_CUDA(cudaMemsetAsync(dL_dscales, 0, sizeof(float) * 3 * (size_t)P, stream));
        if (dL_drotations) GPSG_CUDA(cudaMemsetAsync(dL_drotations, 0, sizeof(float) * 4 * (size_t)P, stream));
    }
    return GPSG_OK;
}

size_t gpsg_rasterize_backward_maps_workspace_bytes(int pixels_per_view) {
    const size_t n = (size_t)(pixels_per_view > 0 ? 2 * pixels_per_view : 1);
    return align_up(sizeof(float4) * 3 * n) + align_up(sizeof(float) * 3 * n) + 512;     // accumulator rows + dL_dmeans2D
}

int gpsg_rasterize_backward_maps(const GpsgRasterSettings* s, int device, void* stream_, int pixels_per_view,
                                 int32_t num_rendered, const uint8_t* const* valid, const float* const* xyz,
                                 const float* const* img, const float* const* rot, const float* const* scale,
                                 const float* const* opacity, const int32_t* radii, const void* geom_buffer,
                                 const void* binning_buffer, const void* image_buffer, const float* dL_dout_color,
                                 float* const* dL_dxyz, float* const* dL_dimg, float* const* dL_drot,
                                 float* const* dL_dscale, float* const* dL_dopacity, void* workspace) {
    GPSG_REQUIRE(s != nullptr, "settings is NULL");
    int rc = check_maps(pixels_per_view, valid, xyz, img, rot, scale, opacity);
    if (rc) return rc;
    GPSG_REQUIRE(num_rendered >= 0 && radii && geom_buffer && binning_buffer && image_buffer && dL_dout_color && workspace,
                 "a required input pointer is NULL");
    GPSG_REQUIRE(dL_dxyz && dL_dimg && dL_drot && dL_dscale && dL_dopacity, "gradient pointer array is NULL");
    GaussianGrads out;
    memset(&out, 0, sizeof(out));
    for (int v = 0; v < 2; ++v) {
        GPSG_REQUIRE(dL_dxyz[v] && dL_dimg[v] && dL_drot[v] && dL_dscale[v] && dL_dopacity[v], "a gradient map is NULL");
        out.dxyz[v] = dL_dxyz[v]; out.dimg[v] = dL_dimg[v]; out.drot[v] = dL_drot[v]; out.dscale[v] = dL_dscale[v];
        out.dopac[v] = dL_dopacity[v];
    }
    const int P = 2 * pixels_per_view;
    // workspace: [3 x float4 P accumulator rows][float 3P dL_dmeans2D]
    char* w = (char*)align_up((size_t)workspace);
    float* dmeans2D = (float*)(w + align_up(sizeof(float4) * 3 * (size_t)P));
    return backward_common(s, device, (cudaStream_t)stream_, P, 0, num_rendered,
                           maps_src(pixels_per_view, valid, xyz, img, rot, scale, opacity), nullptr, radii, geom_buffer,
                           binning_buffer, image_buffer, dL_dout_color, dmeans2D, nullptr, nullptr, out, workspace);
}

int gpsg_mark_visible(int device, void* stream_, int P, const float* means3D, const float* viewmatrix_host16,
                      uint8_t* present) {
    GPSG_REQUIRE(P >= 0, "P < 0");
    if (P == 0) return GPSG_OK;
    GPSG_REQUIRE(means3D && viewmatrix_host16 && present, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    return launch_mark_visible(P, means3D, viewmatrix_host16, present, (cudaStream_t)stream_);
}

int gpsg_geom_view(const void* geom_buffer, int P, GpsgGeomView* out) {
    GPSG_REQUIRE(geom_buffer && out, "NULL pointer");
    GeomState g = GeomState::carve(const_cast<void*>(geom_buffer), P, 0);
    out->depths = g.depths;
    out->means2D = reinterpret_cast<const float*>(g.means2D);
    out->conic_opacity = reinterpret_cast<const float*>(g.conic_opacity);
    out->tiles_touched = g.tiles_touched;
    out->point_offsets = g.point_offsets;
    return GPSG_OK;
}
int gpsg_binning_view(const void* binning_buffer, int64_t num_rendered, GpsgBinningView* out) {
    GPSG_REQUIRE(binning_buffer && out && num_rendered >= 0, "bad argument");
    BinningState b = BinningState::carve(const_cast<void*>(binning_buffer), (size_t)num_rendered, 0);
    out->point_list_keys = b.keys;
    out->point_list = b.vals;
    return GPSG_OK;
}
int gpsg_image_view(const void* image_buffer, int W, int H, GpsgImageView* out) {
    GPSG_REQUIRE(image_buffer && out && W > 0 && H > 0, "bad argument");
    ImageState im = ImageState::carve(const_cast<void*>(image_buffer), W, H);
    out->final_T = im.final_T;
    out->n_contrib = im.n_contrib;
    out->ranges = reinterpret_cast<const uint32_t*>(im.ranges);
    return GPSG_OK;
}

int gpsg_corr_sampler_forward(int device, void* stream_, int dtype, int B, int H, int W1, int W2, const void* volume,
                              int64_t sb, int64_t sh, int64_t sw1, const float* coords, int64_t coords_sb, int radius,
                              void* out) {
    GPSG_REQUIRE(dtype == 0 || dtype == 1, "dtype must be 0 (fp32) or 1 (fp16)");
    GPSG_REQUIRE(B >= 0 && H >= 0 && W1 >= 0 && W2 >= 0 && radius >= 0 && radius <= 31, "bad shape / radius");
    if ((int64_t)B * H * W1 == 0) return GPSG_OK;
    GPSG_REQUIRE(volume && coords && out, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    StageTimer t(ST_CORR_FWD, (cudaStream_t)stream_, 1);
    return launch_corr_fwd(dtype, B, H, W1, W2, volume, sb, sh, sw1, coords, coords_sb, radius, out,
                           (cudaStream_t)stream_);
}

int gpsg_corr_sampler_backward(int device, void* stream_, int dtype, int B, int H, int W1, int W2, const float* coords,
                               int64_t coords_sb, const void* grad_out, int radius, void* grad_volume) {
    GPSG_REQUIRE(dtype == 0 || dtype == 1, "dtype must be 0 (fp32) or 1 (fp16)");
    GPSG_REQUIRE(B >= 0 && H >= 0 && W1 >= 0 && W2 >= 0 && radius >= 0 && radius <= 31, "bad shape / radius");
    if ((int64_t)B * H * W1 * W2 == 0) return GPSG_OK;
    GPSG_REQUIRE(coords && grad_out && grad_volume, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    StageTimer t(ST_CORR_BWD, (cudaStream_t)stream_, 1);
    return launch_corr_bwd(dtype, B, H, W1, W2, coords, coords_sb, grad_out, radius, grad_volume,
                           (cudaStream_t)stream_);
}


int gpsg_corr_build_pyramid(int device, void* stream_, int dtype, int B, int D, int H, int W1, int W2, const void* fmap1,
                            const void* fmap2, void* const* vols, int levels) {
    GPSG_REQUIRE(dtype == 0 || dtype == 1, "dtype must be 0 (fp32) or 1 (fp16)");
    GPSG_REQUIRE(B >= 0 && D > 0 && H >= 0 && W1 >= 0 && W2 >= 0 && levels >= 1 && levels <= 4, "bad shape / levels");
    if ((int64_t)B * H * W1 * W2 == 0) return GPSG_OK;
    GPSG_REQUIRE(fmap1 && fmap2 && vols && vols[0], "NULL pointer");
    for (int l = 1; l < levels; ++l) GPSG_REQUIRE(vols[l] != nullptr || (W2 >> l) == 0, "NULL pyramid level");
    GPSG_CUDA(cudaSetDevice(device));
    StageTimer t(ST_CORR_BUILD, (cudaStream_t)stream_, 1);
    return launch_corr_build(dtype, B, D, H, W1, W2, fmap1, fmap2, vols[0], levels > 1 ? vols[1] : nullptr,
                             levels > 2 ? vols[2] : nullptr, levels > 3 ? vols[3] : nullptr, levels, (cudaStream_t)stream_);
}

int gpsg_corr_build_backward(int device, void* stream_, int dtype, int B, int D, int H, int W1, int W2, const void* fmap1,
                             const void* fmap2, const void* grad_vol0, void* dfmap1, void* dfmap2) {
    GPSG_REQUIRE(dtype == 0 || dtype == 1, "dtype must be 0 (fp32) or 1 (fp16)");
    GPSG_REQUIRE(B >= 0 && D > 0 && H >= 0 && W1 >= 0 && W2 >= 0, "bad shape");
    if ((int64_t)B * H * W1 * W2 == 0) return GPSG_OK;
    GPSG_REQUIRE(fmap1 && fmap2 && grad_vol0 && dfmap1 && dfmap2, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    StageTimer t(ST_CORR_BUILD, (cudaStream_t)stream_, 2);
    return launch_corr_build_bwd(dtype, B, D, H, W1, W2, fmap1, fmap2, grad_vol0, dfmap1, dfmap2, (cudaStream_t)stream_);
}

int gpsg_corr_lookup_pyramid_forward(int device, void* stream_, int dtype, int B, int H, int W1, const void* const* vols,
                                     const int32_t* widths, int levels, const float* coords, int64_t coords_sb, int radius,
                                     void* out) {
    GPSG_REQUIRE(dtype == 0 || dtype == 1, "dtype must be 0 (fp32) or 1 (fp16)");
    GPSG_REQUIRE(B >= 0 && H >= 0 && W1 >= 0 && levels >= 1 && levels <= 4 && radius >= 0 && radius <= 31, "bad shape");
    if ((int64_t)B * H * W1 == 0) return GPSG_OK;
    GPSG_REQUIRE(vols && widths && coords && out, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    StageTimer t(ST_CORR_FWD, (cudaStream_t)stream_, 1);
    return launch_corr_lookup_fwd(dtype, B, H, W1, vols, widths, levels, coords, coords_sb, radius, out, (cudaStream_t)stream_);
}

int gpsg_corr_lookup_pyramid_backward(int device, void* stream_, int dtype, int B, int H, int W1, void* const* grad_vols,
                                      const int32_t* widths, int levels, const float* coords, int64_t coords_sb, int radius,
                                      const void* grad_out) {
    GPSG_REQUIRE(dtype == 0 || dtype == 1, "dtype must be 0 (fp32) or 1 (fp16)");
    GPSG_REQUIRE(B >= 0 && H >= 0 && W1 >= 0 && levels >= 1 && levels <= 4 && radius >= 0 && radius <= 31, "bad shape");
    if ((int64_t)B * H * W1 == 0) return GPSG_OK;
    GPSG_REQUIRE(grad_vols && widths && coords && grad_out, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    StageTimer t(ST_CORR_BWD, (cudaStream_t)stream_, 1);
    return launch_corr_lookup_bwd(dtype, B, H, W1, grad_vols, widths, levels, coords, coords_sb, radius, grad_out, (cudaStream_t)stream_);
}

int gpsg_unproject_forward(int device, void* stream_, int B, int S, const float* flow_pred, const float* mask,
                           int64_t mask_batch_stride, const float* intr, const float* extr, int extr_rows,
                           const float* ref_intr, const float* Tf_x, float* depth, float* xyz, uint8_t* valid) {
    GPSG_REQUIRE(B >= 0 && S >= 0 && extr_rows >= 3, "bad shape");
    if ((int64_t)B * S * S == 0) return GPSG_OK;
    GPSG_REQUIRE(flow_pred && mask && intr && extr && ref_intr && Tf_x && depth && xyz && valid, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    return launch_unproject_fwd(B, S, flow_pred, mask, mask_batch_stride, intr, extr, extr_rows, ref_intr, Tf_x, depth, xyz,
                                valid, (cudaStream_t)stream_);
}

int gpsg_unproject_backward(int device, void* stream_, int B, int S, const float* depth, const float* mask,
                            int64_t mask_batch_stride, const float* intr, const float* extr, int extr_rows,
                            const float* ref_intr, const float* Tf_x, const float* dL_dxyz, const float* dL_ddepth,
                            float* dL_dflow) {
    GPSG_REQUIRE(B >= 0 && S >= 0 && extr_rows >= 3, "bad shape");
    if ((int64_t)B * S * S == 0) return GPSG_OK;
    GPSG_REQUIRE(depth && mask && intr && extr && ref_intr && Tf_x && dL_dflow && (dL_dxyz || dL_ddepth), "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    return launch_unproject_bwd(B, S, depth, mask, mask_batch_stride, intr, extr, extr_rows, ref_intr, Tf_x, dL_dxyz,
                                dL_ddepth, dL_dflow, (cudaStream_t)stream_);
}

size_t gpsg_flow2render_workspace_bytes(int B, int res) {
    return (B > 0 && res > 0) ? (size_t)B * res * res * sizeof(unsigned long long) : 0;
}

int gpsg_flow2render(int device, void* stream_, int B, int bs, int S, int res, const float* const* flow_pred,
                     const float* const* mask, const int64_t* mask_batch_stride, const float* const* intr,
                     const float* const* extr, int extr_rows, const float* const* ref_intr, const float* const* Tf_x,
                     const float* const* img, const float* novel_calib, void* workspace, size_t workspace_bytes,
                     float* out_color, float* out_inv_depth) {
    GPSG_REQUIRE(B > 0 && res > 0, "flow2render: empty batch or image");
    GPSG_REQUIRE(bs >= 0 && bs <= B, "flow2render: bs must be in [0, B]");
    GPSG_REQUIRE(S == res, "flow2render: source maps must be res x res");
    GPSG_REQUIRE(2 * (int64_t)S * S + 1 < ((int64_t)1 << 32), "flow2render: 2*S^2 + 1 must fit the 32-bit point id");
    GPSG_REQUIRE(extr_rows >= 3, "flow2render: extr needs >= 3 rows");
    GPSG_REQUIRE(flow_pred && mask && mask_batch_stride && intr && extr && ref_intr && Tf_x && img && novel_calib &&
                 workspace && out_color, "NULL pointer");
    FlowSplatViews in;
    for (int v = 0; v < 2; ++v) {
        GPSG_REQUIRE(flow_pred[v] && mask[v] && intr[v] && extr[v] && ref_intr[v] && Tf_x[v] && img[v],
                     "NULL per-view pointer");
        GPSG_REQUIRE(mask_batch_stride[v] >= (int64_t)S * S, "flow2render: mask batch stride < S^2");
        in.flow[v] = flow_pred[v]; in.mask[v] = mask[v]; in.mask_bs[v] = mask_batch_stride[v]; in.intr[v] = intr[v];
        in.extr[v] = extr[v]; in.ref_intr[v] = ref_intr[v]; in.Tf_x[v] = Tf_x[v]; in.img[v] = img[v];
    }
    in.extr_rows = extr_rows;
    GPSG_REQUIRE(workspace_bytes >= gpsg_flow2render_workspace_bytes(B, res), "flow2render: workspace too small");
    GPSG_REQUIRE(((uintptr_t)workspace & 7) == 0, "flow2render: workspace must be 8-byte aligned");
    GPSG_CUDA(cudaSetDevice(device));
    return launch_flow2render(B, bs, S, res, in, novel_calib, workspace, out_color, out_inv_depth, (cudaStream_t)stream_);
}

size_t gpsg_l1_ssim_workspace_bytes(int planes, int H, int W) {
    return (planes > 0 && H > 0 && W > 0) ? l1_ssim_workspace_bytes(planes, H, W) : 256;
}

int gpsg_l1_ssim_forward(int device, void* stream_, int planes, int H, int W, const float* img, const float* gt, float w_l1,
                         float w_ssim, float* out3, float* dmaps, void* workspace) {
    GPSG_REQUIRE(planes > 0 && H > 0 && W > 0, "l1_ssim: empty image");
    GPSG_REQUIRE(img && gt && out3 && workspace, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    return launch_l1_ssim_fwd(planes, H, W, img, gt, w_l1, w_ssim, out3, dmaps, workspace, (cudaStream_t)stream_);
}

int gpsg_l1_ssim_backward(int device, void* stream_, int planes, int H, int W, const float* img, const float* gt,
                          const float* dmaps, float w_l1, float w_ssim, const float* grad_loss, float* dimg) {
    GPSG_REQUIRE(planes > 0 && H > 0 && W > 0, "l1_ssim: empty image");
    GPSG_REQUIRE(img && gt && dmaps && dimg, "NULL pointer");
    GPSG_CUDA(cudaSetDevice(device));
    return launch_l1_ssim_bwd(planes, H, W, img, gt, dmaps, w_l1, w_ssim, grad_loss, dimg, (cudaStream_t)stream_);
}

int gpsg_set_corr_build(int mode) {
    set_corr_build_mode(mode);
    return GPSG_OK;
}
int gpsg_profile_enable(int on) {
    g_prof.on = on == 2 ? 2 : (on != 0);
    return GPSG_OK;
}
const char* gpsg_profile_stage_name(int stage) { return (stage >= 0 && stage < ST_COUNT) ? kStageNames[stage] : ""; }
int gpsg_profile_read(float* total_ms, int32_t* calls, int32_t* launches, int capacity) {
    GPSG_REQUIRE(total_ms && calls && launches && capacity >= ST_COUNT, "profile_read: capacity < stage count");
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (int i = 0; i < ST_COUNT; ++i) { total_ms[i] = 0.f; calls[i] = 0; launches[i] = g_prof.launches[i]; g_prof.launches[i] = 0; }
    for (size_t k = 0; k < g_prof.next; ++k) {
        ProfSlot& p = g_prof.slots[k];
        if (!p.used) continue;
        GPSG_CUDA(cudaEventSynchronize(p.b));
        float ms = 0.f;
        GPSG_CUDA(cudaEventElapsedTime(&ms, p.a, p.b));
        total_ms[p.stage] += ms; calls[p.stage] += 1; p.used = false;
    }
    g_prof.next = 0;
    return ST_COUNT;
}

}  // extern "C"
