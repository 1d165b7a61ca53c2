// unproject.cu -- fused flow -> depth -> point cloud, the step right before the rasterizer (SURVEY.md section 8f-3):
// reference lib/utils.py:112-119 (flow2depth) + :87-109 (depth2pc) as called from lib/network.py:64-69
// (flow2gsparms), which is ~12 elementwise / bmm torch kernels with repeat/cat copies over [B,S,S,3].
// One kernel forward (depth, xyz, pts_valid) and one backward (d xyz [+ d depth] -> d flow).  HBM-bound:
// forward reads 8 B and writes 17 B per pixel.
#include "gpsg_internal.cuh"
#include "unproject_math.cuh"

namespace gpsg {

__global__ void __launch_bounds__(256) unproject_forward_kernel(int B, int S, const float* __restrict__ flow,
                                                                const float* __restrict__ mask, int64_t mask_bs,
                                                                const float* __restrict__ intr,
                                                                const float* __restrict__ extr, int extr_rows,
                                                                const float* __restrict__ ref_intr,
                                                                const float* __restrict__ Tf_x,
                                                                float* __restrict__ depth, float* __restrict__ xyz,
                                                                uint8_t* __restrict__ valid) {
    const int64_t S2 = (int64_t)S * S;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)B * S2) return;
    const int b = (int)(idx / S2);
    const int64_t pix = idx - (int64_t)b * S2;
    const int v = (int)(pix / S), u = (int)(pix % S);
    const UnprojCam c = load_cam(intr, extr, extr_rows, ref_intr, Tf_x, b);
    float p[3];
    const float d = unproject_pixel(c, flow[idx], mask[(size_t)b * mask_bs + pix], u, v, p);
    depth[idx] = d;
    valid[idx] = d != 0.0f;
    float* o = xyz + 3 * idx;
#pragma unroll
    for (int k = 0; k < 3; ++k) o[k] = p[k];
}

__global__ void __launch_bounds__(256) unproject_backward_kernel(int B, int S, const float* __restrict__ depth,
                                                                 const float* __restrict__ mask, int64_t mask_bs,
                                                                 const float* __restrict__ intr,
                                                                 const float* __restrict__ extr, int extr_rows,
                                                                 const float* __restrict__ ref_intr,
                                                                 const float* __restrict__ Tf_x,
                                                                 const float* __restrict__ dL_dxyz,
                                                                 const float* __restrict__ dL_ddepth,
                                                                 float* __restrict__ dL_dflow) {
    const int64_t S2 = (int64_t)S * S;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)B * S2) return;
    const int b = (int)(idx / S2);
    const int64_t pix = idx - (int64_t)b * S2;
    const int v = (int)(pix / S), u = (int)(pix % S);
    const UnprojCam c = load_cam(intr, extr, extr_rows, ref_intr, Tf_x, b);
    const float d = depth[idx];
    const float z = 1.0f / (d + 1e-8f);
    float g[3] = {0.f, 0.f, 0.f};
    if (dL_dxyz) { g[0] = dL_dxyz[3 * idx]; g[1] = dL_dxyz[3 * idx + 1]; g[2] = dL_dxyz[3 * idx + 2]; }
    // dL/dp = R g  (xyz = R^T p - R^T t)
    const float gp0 = c.R[0] * g[0] + c.R[1] * g[1] + c.R[2] * g[2];
    const float gp1 = c.R[3] * g[0] + c.R[4] * g[1] + c.R[5] * g[2];
    const float gp2 = c.R[6] * g[0] + c.R[7] * g[1] + c.R[8] * g[2];
    const float dz = gp0 * (((float)u + 0.5f) - c.cx) / c.fx + gp1 * (((float)v + 0.5f) - c.cy) / c.fy + gp2;
    float dd = -dz * z * z;                                   // z = 1/(d + eps)
    if (dL_ddepth) dd += dL_ddepth[idx];
    dL_dflow[idx] = dd * mask[(size_t)b * mask_bs + pix] / c.tfx;   // depth = (flow - offset) * mask / Tf_x
}

int launch_unproject_fwd(int B, int S, const float* flow, const float* mask, int64_t mask_bs, const float* intr,
                         const float* extr, int extr_rows, const float* ref_intr, const float* Tf_x, float* depth,
                         float* xyz, uint8_t* valid, cudaStream_t stream) {
    const int64_t n = (int64_t)B * S * S;
    if (n == 0) return GPSG_OK;
    unproject_forward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(B, S, flow, mask, mask_bs, intr, extr,
                                                                             extr_rows, ref_intr, Tf_x, depth, xyz, valid);
    GPSG_LAUNCH_CHECK();
    return GPSG_OK;
}

int launch_unproject_bwd(int B, int S, const float* depth, const float* mask, int64_t mask_bs, const float* intr,
                         const float* extr, int extr_rows, const float* ref_intr, const float* Tf_x,
                         const float* dL_dxyz, const float* dL_ddepth, float* dL_dflow, cudaStream_t stream) {
    const int64_t n = (int64_t)B * S * S;
    if (n == 0) return GPSG_OK;
    unproject_backward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(B, S, depth, mask, mask_bs, intr, extr,
                                                                              extr_rows, ref_intr, Tf_x, dL_dxyz,
                                                                              dL_ddepth, dL_dflow);
    GPSG_LAUNCH_CHECK();
    return GPSG_OK;
}

}  // namespace gpsg
