/*
 * flow_splat_oracle.c -- CPU restatement of the stage-1 validation preview (test infrastructure, NOT product code).
 *
 * TaichiRenderBatch.flow2render (reference lib/TaichiRender.py:26-60) as csrc/point_splat.cu computes it:
 *   oracle_flow2render_points  the per-point chain (flow2depth, depth2pc, perspective into the novel camera, inverse
 *                              depth) in the kernel's op order.  point_splat.cu is built with -fmad=false and this file
 *                              with -ffp-contract=off, so the f32 build reproduces the kernel's points bit for bit.
 *   oracle_splat_seq           the sequential reading of the Taichi kernel render_respective_color (:12-23) over V views
 *                              in order on ONE depth / colour state, recording each pixel's winning point.
 * ti.cast(f32 -> i32) of NaN / out-of-range values is undefined; it is taken as CUDA's saturating cvt.rzi.s32.f32
 * (NaN -> 0), which is what the kernel does.  oracle/taichi_splat_oracle.c (the one-view throughput baseline) is left
 * as it is; this file is built into its own libraries by oracle/flow_splat_oracle.py.
 */
#include "oracle_real.h"

/* float->int with CUDA semantics (truncate, saturate, NaN->0), as f2i_sat in gpsg_oracle.c */
static inline int splat_f2i(real v) {
    if (v != v) return 0;
    if (v >= (real)2147483647.0) return 2147483647;
    if (v <= (real)-2147483648.0) return (-2147483647 - 1);
    return (int)v;
}

/* V views of points splatted in order onto ONE depth / colour state, samples b < bs only.  The caller initialises
 * depth (0), color (-1) and winner (-1).  pts[V,B,N,6] = (x, y, inv, r, g, b), mask[V,B,N]; winner[B,res,res] (may be
 * NULL) = v*N + i of the point whose colour the pixel holds. */
void SUFFIX(oracle_splat_seq)(int B, int bs, int V, int N, int res, const real* pts, const real* mask, real* depth,
                              real* color, int32_t* winner) {
    for (int b = 0; b < bs; ++b)
        for (int v = 0; v < V; ++v)
            for (int i = 0; i < N; ++i) {
                const size_t pi = ((size_t)v * B + b) * N + i;
                if (mask[pi] < RC(0.5)) continue;
                const real* p = pts + pi * 6;
                int IX = splat_f2i(p[0]), IY = splat_f2i(p[1]);
                IX = IX < 0 ? 0 : (IX > res - 1 ? res - 1 : IX);
                IY = IY < 0 ? 0 : (IY > res - 1 ? res - 1 : IY);
                const size_t q = ((size_t)b * res + IY) * res + IX;
                const real old = depth[q];
                if (p[2] > old) depth[q] = p[2]; /* atomic_max returns the OLD value */
                if (p[2] >= old) {
                    for (int k = 0; k < 3; ++k) color[(((size_t)b * 3 + k) * res + IY) * res + IX] = p[3 + k];
                    if (winner) winner[q] = (int32_t)((size_t)v * N + i);
                }
            }
}

/* flow[2,B,S*S], mask[2,B,S*S] (channel 0), intr / ref_intr [2,B,9], extr [2,B,12] (3 rows), tfx[2,B],
 * img[2,B,3,S*S], calib[B,12] (K E of the novel camera)  ->  pts[2,B,S*S,6] = (x, y, inv, r, g, b) and valid[2,B,S*S]
 * (1 where depth != 0).  Like upstream, an invalid pixel's point is the origin and its colour 0. */
void SUFFIX(oracle_flow2render_points)(int B, int S, const real* flow, const real* mask, const real* intr,
                                       const real* extr, const real* ref_intr, const real* tfx, const real* img,
                                       const real* calib, real* pts, real* valid) {
    const size_t S2 = (size_t)S * S;
    for (int v = 0; v < 2; ++v)
        for (int b = 0; b < B; ++b) {
            const size_t vb = (size_t)v * B + b;
            const real* K = intr + vb * 9;
            const real* E = extr + vb * 12;
            const real* M = calib + (size_t)b * 12;
            const real offset = ref_intr[vb * 9 + 2] - K[2];
            const real tf = tfx[vb];
            for (size_t pix = 0; pix < S2; ++pix) {
                const int u = (int)(pix % S), w = (int)(pix / S);
                /* flow2depth */
                const real disparity = offset - flow[vb * S2 + pix];
                real d = -disparity / tf;
                d *= mask[vb * S2 + pix];
                const int ok = d != RC(0.0);
                /* depth2pc */
                const real z = RC(1.0) / (d + RC(1e-8));
                const real px = (((real)u + RC(0.5)) - K[2]) * z / K[0];
                const real py = (((real)w + RC(0.5)) - K[5]) * z / K[4];
                real xyz[3] = {RC(0.0), RC(0.0), RC(0.0)};
                if (ok)
                    for (int k = 0; k < 3; ++k) {
                        const real rp = E[k] * px + E[4 + k] * py + E[8 + k] * z;
                        const real rt = E[k] * E[3] + E[4 + k] * E[7] + E[8 + k] * E[11];
                        xyz[k] = rp - rt;
                    }
                /* perspective into the novel camera, then inverse depth */
                real q[3];
                for (int k = 0; k < 3; ++k)
                    q[k] = M[4 * k] * xyz[0] + M[4 * k + 1] * xyz[1] + M[4 * k + 2] * xyz[2] + M[4 * k + 3];
                real* o = pts + (vb * S2 + pix) * 6;
                o[0] = q[0] / q[2];
                o[1] = q[1] / q[2];
                o[2] = RC(1.0) / (q[2] + RC(1e-8));
                for (int k = 0; k < 3; ++k) o[3 + k] = ok ? img[(vb * 3 + k) * S2 + pix] : RC(0.0);
                valid[vb * S2 + pix] = ok ? RC(1.0) : RC(0.0);
            }
        }
}
