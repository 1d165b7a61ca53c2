// unproject_math.cuh -- per-pixel flow -> depth -> world point (reference lib/utils.py:112-119 flow2depth, :87-109
// depth2pc), shared by the fused unprojection (unproject.cu) and the stage-1 preview splat (point_splat.cu).
// Each includer keeps its own compile flags: unproject.cu contracts to FMA, point_splat.cu is built with -fmad=false so
// the CPU oracle (oracle/flow_splat_oracle.c, -ffp-contract=off) can follow its op order bit for bit.
#pragma once
#include <stdint.h>
#include <stddef.h>

namespace gpsg {

// per batch item: K (fx, fy, cx, cy), R (3x3 row-major), t (3), offset = ref_cx - cx, 1/Tf_x sign folded
struct UnprojCam { float fx, fy, cx, cy, R[9], t[3], offset, tfx; };

__device__ __forceinline__ UnprojCam load_cam(const float* intr, const float* extr, int extr_row_stride,
                                              const float* ref_intr, const float* Tf_x, int b) {
    UnprojCam c;
    const float* K = intr + 9 * (size_t)b;
    const float* E = extr + (size_t)b * extr_row_stride * 4;     // [rows>=3, 4]
    c.fx = K[0]; c.fy = K[4]; c.cx = K[2]; c.cy = K[5];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int k = 0; k < 3; ++k) c.R[3 * r + k] = E[4 * r + k];
        c.t[r] = E[4 * r + 3];
    }
    c.offset = ref_intr[9 * (size_t)b + 2] - K[2];
    c.tfx = Tf_x[b];
    return c;
}

// depth of source pixel (u, v) from its flow and mask value, and the world point depth2pc makes of it
// (xyz = R^T p - R^T t, p = ((u+0.5-cx) z / fx, (v+0.5-cy) z / fy, z), z = 1/(depth + 1e-8)).  Returns the depth.
__device__ __forceinline__ float unproject_pixel(const UnprojCam& c, float flow, float mask, int u, int v, float xyz[3]) {
    // flow2depth: depth = -(offset - flow) / Tf_x * mask
    const float disparity = c.offset - flow;
    float d = -disparity / c.tfx;
    d *= mask;
    // depth2pc: inverse-depth parameterisation, pixel centres at +0.5
    const float z = 1.0f / (d + 1e-8f);
    const float px = (((float)u + 0.5f) - c.cx) * z / c.fx;
    const float py = (((float)v + 0.5f) - c.cy) * z / c.fy;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float rp = c.R[k] * px + c.R[3 + k] * py + c.R[6 + k] * z;
        const float rt = c.R[k] * c.t[0] + c.R[3 + k] * c.t[1] + c.R[6 + k] * c.t[2];
        xyz[k] = rp - rt;
    }
    return d;
}

}  // namespace gpsg
