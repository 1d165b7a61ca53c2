// point_splat.cu -- the stage-1 validation preview (reference lib/TaichiRender.py:26-60, TaichiRenderBatch.flow2render):
// both source views' flow maps -> depth -> world points -> novel-view pixel + inverse depth, then a 1-pixel z-buffer
// splat that keeps the nearest point per pixel.  Compiled with -fmad=false so the CPU oracle can replay the fp32 op order.
//
// Upstream runs `ti.atomic_max` on the inverse depth and writes the colour non-atomically afterwards, so two points that
// land on the same pixel race.  Here the sequential reading (views l then r, points in pixel order; a point with
// inv >= current writes its colour) is computed exactly by ONE 64-bit max per point:
//     key = bits(inv) << 32 | (view * S^2 + pixel + 1)
// For inv >= 0 (non-NaN) the float bits order like the values, so the max key is the last point in (view, index) order
// among those with the maximal inverse depth -- which is what the sequential loop leaves behind.  Key 0 = no point.
// Points with inv < 0 (behind the camera) or NaN never draw, as in the sequential loop (depth starts at 0).
//
// One memset (the z-buffer) and two launches, no host synchronisation:
//   flow_splat_kernel     one thread per (sample < bs, view, source pixel): global 64-bit atomicMax into the z-buffer
//   splat_resolve_kernel  one thread per output pixel of all B samples: decode the winner, gather its 3 colour values
#include "gpsg_internal.cuh"
#include "unproject_math.cuh"

namespace gpsg {

__global__ void __launch_bounds__(256) flow_splat_kernel(int bs, int S, int res, FlowSplatViews in,
                                                         const float* __restrict__ calib,
                                                         unsigned long long* __restrict__ zbuf) {
    const int64_t S2 = (int64_t)S * S;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)bs * 2 * S2) return;
    const int b = (int)(idx / (2 * S2));
    const int64_t r = idx - (int64_t)b * 2 * S2;
    const int view = r >= S2 ? 1 : 0;
    const int64_t pix = r - view * S2;
    const int v = (int)(pix / S), u = (int)(pix % S);
    const UnprojCam c = load_cam(in.intr[view], in.extr[view], in.extr_rows, in.ref_intr[view], in.Tf_x[view], b);
    float p[3];
    const float d = unproject_pixel(c, in.flow[view][(size_t)b * S2 + pix],
                                    in.mask[view][(size_t)b * in.mask_bs[view] + pix], u, v, p);
    if (!(d != 0.0f)) return;                                     // valid = depth != 0 (a NaN depth is "valid")
    // perspective (lib/utils.py:121-127) into the novel camera M = K_novel E_novel [3,4]
    const float* M = calib + 12 * (size_t)b;
    float q[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) q[k] = M[4 * k] * p[0] + M[4 * k + 1] * p[1] + M[4 * k + 2] * p[2] + M[4 * k + 3];
    const float x = q[0] / q[2], y = q[1] / q[2];
    const float inv = 1.0f / (q[2] + 1e-8f);                      // lib/TaichiRender.py:44
    if (!(inv >= 0.0f)) return;                                   // behind the camera or NaN: never draws
    // ti.cast(f32 -> i32) then clamp onto the border (off-screen points are NOT dropped upstream)
    const int ix = min(res - 1, max(__float2int_rz(x), 0));
    const int iy = min(res - 1, max(__float2int_rz(y), 0));
    const unsigned long long key = ((unsigned long long)(__float_as_uint(inv) & 0x7fffffffu) << 32) |   // -0 -> +0
                                   (unsigned long long)(uint32_t)(view * S2 + pix + 1);
    unsigned long long* slot = zbuf + ((size_t)b * res + iy) * res + ix;
    // clamped points pile onto the border pixels: skip the atomic when the slot already holds a larger key (slots only grow)
    if (*reinterpret_cast<volatile unsigned long long*>(slot) >= key) return;
    atomicMax(slot, key);
}

__global__ void __launch_bounds__(256) splat_resolve_kernel(int B, int S, int res, const float* __restrict__ img0,
                                                            const float* __restrict__ img1,
                                                            const unsigned long long* __restrict__ zbuf,
                                                            float* __restrict__ color, float* __restrict__ inv_depth) {
    const int64_t R2 = (int64_t)res * res, S2 = (int64_t)S * S;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)B * R2) return;
    const int b = (int)(idx / R2);
    const int64_t pix = idx - (int64_t)b * R2;
    const unsigned long long key = zbuf[idx];
    float rgb[3] = {-1.0f, -1.0f, -1.0f};                         // upstream's background (min_value = -1)
    float inv = 0.0f;
    if (key != 0ull) {
        const int64_t id = (int64_t)(uint32_t)key - 1;
        const int view = id >= S2 ? 1 : 0;
        const float* src = (view ? img1 : img0) + (size_t)b * 3 * S2 + (id - view * S2);
#pragma unroll
        for (int k = 0; k < 3; ++k) rgb[k] = src[k * S2];          // raw img in [-1, 1] (no *0.5+0.5, unlike pts2render)
        inv = __uint_as_float((uint32_t)(key >> 32));
    }
    float* o = color + (size_t)b * 3 * R2 + pix;
#pragma unroll
    for (int k = 0; k < 3; ++k) o[k * R2] = rgb[k];
    if (inv_depth) inv_depth[idx] = inv;
}

int launch_flow2render(int B, int bs, int S, int res, const FlowSplatViews& in, const float* calib, void* zbuf,
                       float* color, float* inv_depth, cudaStream_t stream) {
    const int64_t R2 = (int64_t)res * res, n = (int64_t)bs * 2 * S * S;
    GPSG_CUDA(cudaMemsetAsync(zbuf, 0, (size_t)B * R2 * sizeof(unsigned long long), stream));
    if (n > 0) {
        flow_splat_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(bs, S, res, in, calib,
                                                                           (unsigned long long*)zbuf);
        GPSG_LAUNCH_CHECK();
    }
    splat_resolve_kernel<<<(unsigned)((B * R2 + 255) / 256), 256, 0, stream>>>(B, S, res, in.img[0], in.img[1],
                                                                              (const unsigned long long*)zbuf, color,
                                                                              inv_depth);
    GPSG_LAUNCH_CHECK();
    return GPSG_OK;
}

}  // namespace gpsg
