// resample.cuh — Spacingd -> Orientationd (MONAI 0.5; 127_...FLAIR.py:120-129, utils.py:186-198) as one gather from the
// loaded volume, included by spatial.cu.
//
// MONAI resamples with torch affine_grid + grid_sample (float64, align_corners=False, border padding) and reorients with
// nibabel's apply_orientation (flip, then transpose).  Per output voxel j:
//   1. j -> q, the voxel's index in Spacingd's output grid: q[g] = base[g] + step[g] * j[axis[g]] (an optional window,
//      a flip mask and Orientationd's signed axis permutation, folded together on the host; exact integer arithmetic);
//   2. q -> taps along each source axis k:
//      separable (the transform maps each grid axis to one source axis): mvtb_resample_tap tables (include/mvtb.h) the
//        host computed with torch's own affine_grid on one line of the grid (bit-equal to the full grid's coordinates,
//        so nearest-neighbour labels match torch exactly, ties included);
//      general: the fp64 3x4 matrix evaluated per voxel (clip to [0, n-1], then floor or round half to even); nearest
//        can differ from torch only where torch's coordinate sits on an exact tie;
//   3. nearest: one load; bilinear: eight loads combined in fp32 in source-axis order (independent of the output axis
//      order, so the fused call and Spacingd followed by Orientationd give the same bits).
// One warp per output row (n, j0, j1), lanes along j2; consecutive rows share source rows through L1/L2.
#pragma once
#include <cmath>

#include "mvtb_common.cuh"

namespace mvtb {

struct ResampleDev {
    long long in_vol;          // elements per source volume
    int in_n[3];               // source (H, W, D)
    int in_stride[3];          // (W D, D, 1)
    int s0, s1, s2;            // output shape
    // separable: per SOURCE axis k, the table entry base + step * j[ax]; general: per GRID axis g, q = base + step * j[ax]
    int ax[3], base[3], step[3];
    const mvtb_resample_tap* taps;
    double m[3][4];            // general: source coordinate k = m[k] . (q0, q1, q2, 1)
};

__device__ __forceinline__ int pick3(int a, int j0, int j1, int j2) { return a == 0 ? j0 : (a == 1 ? j1 : j2); }

// fp32 trilinear combination in source-axis order (axis 0 outermost): a, b, c = element offsets of the two taps along
// source axes 0, 1, 2; u, v, w = their weights
__device__ __forceinline__ float trilerp(const float* __restrict__ src, int a0, int a1, float u0, float u1, int b0, int b1, float v0,
                                         float v1, int c0, int c1, float w0, float w1) {
    const float x00 = w0 * __ldg(src + a0 + b0 + c0) + w1 * __ldg(src + a0 + b0 + c1);
    const float x01 = w0 * __ldg(src + a0 + b1 + c0) + w1 * __ldg(src + a0 + b1 + c1);
    const float x10 = w0 * __ldg(src + a1 + b0 + c0) + w1 * __ldg(src + a1 + b0 + c1);
    const float x11 = w0 * __ldg(src + a1 + b1 + c0) + w1 * __ldg(src + a1 + b1 + c1);
    return u0 * (v0 * x00 + v1 * x01) + u1 * (v0 * x10 + v1 * x11);
}

template <bool SEP, bool NEAREST>
__global__ void __launch_bounds__(256)
k_resample(const float* __restrict__ in, float* __restrict__ out, ResampleDev g, long long n_rows_total) {
    const int lane = threadIdx.x & 31;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = wid; r < n_rows_total; r += nw) {
        const long long v = r / ((long long)g.s0 * g.s1);
        const int rem = (int)(r - v * (long long)g.s0 * g.s1);
        const int j0 = rem / g.s1, j1 = rem - j0 * g.s1;
        const float* src = in + v * g.in_vol;
        float* dst = out + r * g.s2;
        for (int j2 = lane; j2 < g.s2; j2 += 32) {
            int i0[3], i1[3];
            float w0[3], w1[3];
            if (SEP) {
                MVTB_UNROLL
                for (int k = 0; k < 3; ++k) {
                    const mvtb_resample_tap t = g.taps[g.base[k] + g.step[k] * pick3(g.ax[k], j0, j1, j2)];
                    i0[k] = t.i0; i1[k] = t.i1; w0[k] = t.w0; w1[k] = t.w1;
                }
            } else {
                double qd[3];
                MVTB_UNROLL
                for (int gg = 0; gg < 3; ++gg) qd[gg] = (double)(g.base[gg] + g.step[gg] * pick3(g.ax[gg], j0, j1, j2));
                MVTB_UNROLL
                for (int k = 0; k < 3; ++k) {
                    double s = fma(g.m[k][0], qd[0], fma(g.m[k][1], qd[1], fma(g.m[k][2], qd[2], g.m[k][3])));
                    s = fmin(fmax(s, 0.0), (double)(g.in_n[k] - 1));           // border padding
                    if (NEAREST) {
                        i0[k] = (int)rint(s);                                   // round half to even, as nearbyint
                    } else {
                        const double f = floor(s);
                        i0[k] = (int)f;
                        i1[k] = i0[k] + 1 < g.in_n[k] ? i0[k] + 1 : i0[k];
                        w0[k] = (float)((f + 1.0) - s);
                        w1[k] = (float)(s - f);
                    }
                }
            }
            float val;
            if (NEAREST) {
                val = __ldg(src + i0[0] * g.in_stride[0] + i0[1] * g.in_stride[1] + i0[2]);
            } else {
                val = trilerp(src, i0[0] * g.in_stride[0], i1[0] * g.in_stride[0], w0[0], w1[0], i0[1] * g.in_stride[1],
                              i1[1] * g.in_stride[1], w0[1], w1[1], i0[2], i1[2], w0[2], w1[2]);
            }
            dst[j2] = val;
        }
    }
}

}  // namespace mvtb
