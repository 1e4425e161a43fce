// bandlimited.cu — the k-space chain when the mask keeps only a small ball of frequencies.
//
// RandFourierDiskMaskd (F:236-252) with the radii the scripts use (r = 9 ... 30; r = 12.5 in the
// 125/126/127 chains) keeps |f_d| <= F = floor(sqrt(thr)) on every axis, i.e. (2F+1)^2 (F+1) of the
// N_h N_w N_d/2 half-spectrum bins (8 125 of 4.5 M for 240x240x155, r = 12.5).  A full FFT computes
// 550x more bins than survive the mask.  This path computes only the surviving ones, as pruned
// DFTs with the symmetric-pair folding  x[h] +- x[N-h]  (cos part / sin part), in three kernels:
//
//   k_bl_fwd_h   x[v][H][W*D] real       -> Y[v][NF][W*D]      streams the volume ONCE from HBM with coalesced
//                                                             loads (cp.async ring); H % 4 == 0: four rows per
//                                                             table row (bandlimited_quad.cuh)
//   k_bl_midw    Y[v][NF][W][D] in place: one CTA per (v, f_h) plane does the W-axis DFT to K = 2F+1 bins, the
//                D-axis DFT, the pointwise stage (mask / in-box spikes / wrap / 1/N) and both ways back
//   k_bl_inv_h   Y                       -> out[v][H][W*D]     writes the volume ONCE; adds out-of-box spikes as
//                                                             plane waves (SURVEY A.4), tracks per-sample min/max
//
// (k_bl_fwd_w -> G[v][NF][K][D], k_bl_mid, k_bl_inv_w are the same W/D stage as three kernels: used when a plane's
// tile would leave fewer than two CTAs per SM, and by tests through MVTB_PATH_BL_SPLIT.)
//
// HBM traffic is the compulsory 8 B/voxel plus ~1 B/voxel of intermediates (Y is NF/H of the
// volume); arithmetic is ~(2F+1) FMA per voxel and direction.  cos/sin rows are read from shared
// memory as 128-bit broadcasts.  Results are the same numbers the general path produces (same
// pointwise stage, pointwise.cuh), to fp32 rounding.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "philox.cuh"
#include "sp_sampler.cuh"
#include "pointwise.cuh"
#include "tc_common.cuh"

namespace mvtb {

int convert_desc(const mvtb_plan* p, const mvtb_chain_desc* u, DescDev* d);                      // kspace_chain.cu
int plan_stage_upload(mvtb_plan* p, const void* src, size_t bytes, void* stream, void** dptr);   // plan.cu

static const int kColThreads = 256;      // H-axis kernels: 256 threads x 2 columns
// columns per thread in the H-axis kernels: 2 while the accumulators fit (NF <= 16), else 1
template <int NF> struct BlCols { static constexpr int CPT = NF > 16 ? 1 : 2; };
static const int kWThreads = 128;        // W-axis kernels
static const int kWParts = 4;            // lanes per (fh, d) column in k_bl_fwd_w
static const int kMidThreads = 256;
static const int kBlChunk = 64;          // volumes per band-limited launch (intermediates: ~4.3 MB per 240x240x155 volume)

struct BlGeom {
    int H, W, D;
    int F;                    // kept |f| <= F on every axis; NF >= F+1 rows of the h half-spectrum
    long long NC;             // W*D
    const float* tabC[3];     // [N][MVTB_BL_FT] cos(2 pi f n / N), axis 0 = D, 1 = W, 2 = H
    const float* tabS[3];
    const cf* twD;            // exp(-2 pi i t / D)
    float scale;              // 1/(H W D)
};

struct PlaneWave { int fh, fw, fd; float amp; };      // signed frequencies, amplitude incl. wrap weight and 1/N
struct BlVol {                                        // per-volume parameters, uploaded once per call
    DescDev d;                                        // pointwise stage (in-box spikes only)
    int npw;
    int pad;
    PlaneWave pw[MVTB_BL_MAX_PW];                     // out-of-box spikes
};

template <int NF> struct BlDims {
    static constexpr int NT = (2 * NF + 3) & ~3;      // floats per table row: (cos f, sin f) pairs, f = 0..NF-1
};

// Packed fp32 pairs: Blackwell's FFMA2 (fma.rn.f32x2) does two FMAs per issued instruction.  Every inner
// loop below is arranged so that one operand pair is (cos f, sin f) straight out of a 128-bit shared load.
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
#ifdef MVTB_EMU
    return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y));
#else
    return __ffma2_rn(a, b, c);
#endif
}

// (cos, sin) rows of one axis for n = 0 .. N/2 into shared memory, NT floats per row
template <int NF>
__device__ __forceinline__ void bl_load_table(float* sc, const float* __restrict__ tabC,
                                              const float* __restrict__ tabS, int N, int tid, int nthr) {
    constexpr int NT = BlDims<NF>::NT;
    const int rows = N / 2 + 1;
    for (int e = tid; e < rows * (NT / 2); e += nthr) {
        const int n = e / (NT / 2), f = e - n * (NT / 2);
        float c = 0.f, s = 0.f;
        if (f < NF) { c = __ldg(tabC + n * MVTB_BL_FT + f); s = __ldg(tabS + n * MVTB_BL_FT + f); }
        sc[2 * e] = c;
        sc[2 * e + 1] = s;
    }
}

template <int NF>
__device__ __forceinline__ void bl_row(const float* __restrict__ row, float2* cs) {
    constexpr int NT = BlDims<NF>::NT;
    const float4* s4 = reinterpret_cast<const float4*>(row);
    MVTB_UNROLL
    for (int i = 0; i < NT / 4; ++i) {
        const float4 v = s4[i];
        if (2 * i < NF) cs[2 * i] = make_float2(v.x, v.y);
        if (2 * i + 1 < NF) cs[2 * i + 1] = make_float2(v.z, v.w);
    }
}

#ifdef MVTB_EMU
__device__ __forceinline__ float ld_stream(const float* p) { return *p; }
__device__ __forceinline__ void st_stream(float* p, float v) { *p = v; }
#else
// the volume is touched exactly once: keep it from displacing the small intermediates in L2
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }
#endif

// ------------------------------------------------------------------ H axis forward: real -> NF complex rows
template <int NF, int CPT>
__global__ void __launch_bounds__(256, 2)
k_bl_fwd_h(const float* __restrict__ x, cf* __restrict__ Y, BlGeom g, int n_cblocks) {
    constexpr int NT = BlDims<NF>::NT, U = 4;
    MVTB_DYN_SMEM(smem_raw);
    float* sc = (float*)smem_raw;
    const int tid = threadIdx.x;
    bl_load_table<NF>(sc, g.tabC[2], g.tabS[2], g.H, tid, blockDim.x);
    __syncthreads();

    const long long vol = blockIdx.x / n_cblocks;
    const long long c0 = (long long)(blockIdx.x - vol * n_cblocks) * (blockDim.x * CPT) + tid;
    const float* xv = x + vol * g.H * g.NC;
    bool ok[CPT];
    long long col[CPT];
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) {
        col[k] = c0 + (long long)k * blockDim.x;
        ok[k] = col[k] < g.NC;
        if (!ok[k]) col[k] = g.NC - 1;                  // clamp: loads stay in bounds, stores are predicated
    }
    float2 acc[CPT][NF];                                // (re, im)
    const int H = g.H;
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) {
        const float x0 = ld_stream(xv + col[k]);
        const float xn = (H & 1) ? 0.f : ld_stream(xv + (long long)(H / 2) * g.NC + col[k]);
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) acc[k][f] = make_float2(x0 + ((f & 1) ? -xn : xn), 0.f);
    }
    const int npair = (H - 1) / 2;
    const float* plo[CPT];
    const float* phi[CPT];
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) { plo[k] = xv + g.NC + col[k]; phi[k] = xv + (long long)(H - 1) * g.NC + col[k]; }
    int h = 1;
    for (; h + U - 1 <= npair; h += U) {                // 2*U*CPT independent coalesced loads in flight
        float a[U][CPT], b[U][CPT];
        MVTB_UNROLL
        for (int u = 0; u < U; ++u) {
            MVTB_UNROLL
            for (int k = 0; k < CPT; ++k) {
                a[u][k] = ld_stream(plo[k] + (long long)u * g.NC);
                b[u][k] = ld_stream(phi[k] - (long long)u * g.NC);
            }
        }
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) { plo[k] += (long long)U * g.NC; phi[k] -= (long long)U * g.NC; }
        MVTB_UNROLL
        for (int u = 0; u < U; ++u) {
            float2 cs[NF];
            bl_row<NF>(sc + (h + u) * NT, cs);
            MVTB_UNROLL
            for (int k = 0; k < CPT; ++k) {
                const float2 eo = make_float2(a[u][k] + b[u][k], b[u][k] - a[u][k]);   // Im -= (a-b) sin
                MVTB_UNROLL
                for (int f = 0; f < NF; ++f) acc[k][f] = fma2(eo, cs[f], acc[k][f]);
            }
        }
    }
    for (; h <= npair; ++h) {
        float2 cs[NF];
        bl_row<NF>(sc + h * NT, cs);
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) {
            const float a = ld_stream(plo[k]), b = ld_stream(phi[k]);
            plo[k] += g.NC; phi[k] -= g.NC;
            const float2 eo = make_float2(a + b, b - a);
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) acc[k][f] = fma2(eo, cs[f], acc[k][f]);
        }
    }
    cf* yv = Y + vol * NF * g.NC;
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) {
        if (ok[k]) {
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) yv[(long long)f * g.NC + col[k]] = acc[k][f];
        }
    }
}

// ------------------------------------------------------------------ W axis forward: Y[NF][W][D] -> G[NF][K][D]
// kWParts lanes share one (fh, d) column (w-pairs interleaved among them, xor-shuffle reduction at the end):
// 4x the threads of a thread-per-column mapping, which this latency-bound kernel needs to fill the machine.
template <int NF>
__global__ void __launch_bounds__(128, (NF > 16 ? 2 : 4))
k_bl_fwd_w(const cf* __restrict__ Y, cf* __restrict__ G, BlGeom g, int n_tblocks) {
    constexpr int NT = BlDims<NF>::NT, PARTS = kWParts;
    MVTB_DYN_SMEM(smem_raw);
    float* sc = (float*)smem_raw;
    const int tid = threadIdx.x;
    bl_load_table<NF>(sc, g.tabC[1], g.tabS[1], g.W, tid, blockDim.x);
    __syncthreads();

    const int W = g.W, D = g.D, K = 2 * g.F + 1;
    const long long vol = blockIdx.x / n_tblocks;
    const int t = (int)(blockIdx.x - vol * n_tblocks) * blockDim.x + tid;
    int q = t / PARTS;                                   // (fh, d)
    const int part = t - q * PARTS;
    const bool valid = q < NF * D;
    if (!valid) q = NF * D - 1;                          // keep the lane in the shuffles
    const int fh = q / D, d = q - fh * D;
    const cf* yv = Y + ((vol * NF + fh) * (long long)W) * D + d;
    // P = sum (a+b) cos, Q = sum (a-b) sin (complex); kept as (P.x, Q.x) and (P.y, Q.y) pairs
    float2 pqx[NF], pqy[NF];
    {
        cf y0 = cmk(0.f, 0.f), yn = cmk(0.f, 0.f);
        if (part == 0) {
            y0 = yv[0];
            if ((W & 1) == 0) yn = yv[(long long)(W / 2) * D];
        }
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) {
            pqx[f] = make_float2((f & 1) ? y0.x - yn.x : y0.x + yn.x, 0.f);
            pqy[f] = make_float2((f & 1) ? y0.y - yn.y : y0.y + yn.y, 0.f);
        }
    }
    const int npair = (W - 1) / 2;
    int w = 1 + part;
    for (; w + PARTS <= npair; w += 2 * PARTS) {         // two pairs (four 8-byte loads) in flight
        const cf a0 = yv[(long long)w * D], b0 = yv[(long long)(W - w) * D];
        const cf a1 = yv[(long long)(w + PARTS) * D], b1 = yv[(long long)(W - w - PARTS) * D];
        float2 cs[NF];
        bl_row<NF>(sc + w * NT, cs);
        float2 ex = make_float2(a0.x + b0.x, a0.x - b0.x), ey = make_float2(a0.y + b0.y, a0.y - b0.y);
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) { pqx[f] = fma2(ex, cs[f], pqx[f]); pqy[f] = fma2(ey, cs[f], pqy[f]); }
        bl_row<NF>(sc + (w + PARTS) * NT, cs);
        ex = make_float2(a1.x + b1.x, a1.x - b1.x);
        ey = make_float2(a1.y + b1.y, a1.y - b1.y);
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) { pqx[f] = fma2(ex, cs[f], pqx[f]); pqy[f] = fma2(ey, cs[f], pqy[f]); }
    }
    for (; w <= npair; w += PARTS) {
        float2 cs[NF];
        bl_row<NF>(sc + w * NT, cs);
        const cf a = yv[(long long)w * D], b = yv[(long long)(W - w) * D];
        const float2 ex = make_float2(a.x + b.x, a.x - b.x), ey = make_float2(a.y + b.y, a.y - b.y);
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) { pqx[f] = fma2(ex, cs[f], pqx[f]); pqy[f] = fma2(ey, cs[f], pqy[f]); }
    }
    MVTB_UNROLL
    for (int f = 0; f < NF; ++f) {
        MVTB_UNROLL
        for (int o = 1; o < PARTS; o <<= 1) {
            pqx[f].x += __shfl_xor_sync(0xffffffffu, pqx[f].x, o);
            pqx[f].y += __shfl_xor_sync(0xffffffffu, pqx[f].y, o);
            pqy[f].x += __shfl_xor_sync(0xffffffffu, pqy[f].x, o);
            pqy[f].y += __shfl_xor_sync(0xffffffffu, pqy[f].y, o);
        }
    }
    // X(+f) = P - iQ, X(-f) = P + iQ;  row j of G holds fw = j - F; the PARTS lanes share the stores
    cf* gv = G + ((vol * NF + fh) * (long long)K) * D + d;
    MVTB_UNROLL
    for (int f = 0; f < NF; ++f) {
        if (valid && f <= g.F && (f % PARTS) == part) {
            gv[(long long)(g.F + f) * D] = cmk(pqx[f].x + pqy[f].y, pqy[f].x - pqx[f].y);
            if (f > 0) gv[(long long)(g.F - f) * D] = cmk(pqx[f].x - pqy[f].y, pqy[f].x + pqx[f].y);
        }
    }
}

// ------------------------------------------------------------------ D axis both ways + pointwise; CTA = (vol, fh)
__global__ void __launch_bounds__(256)
k_bl_mid(cf* __restrict__ G, BlGeom g, int NF, const BlVol* __restrict__ vols, int vol_base, int shared_desc,
         const cf* __restrict__ twkd /* [K][D] exp(-2 pi i (jd-F) d / D) */) {
    MVTB_DYN_SMEM(smem_raw);
    const int D = g.D, K = 2 * g.F + 1, F = g.F;
    cf* sg = (cf*)smem_raw;            // [K][D]   rows of G for this (vol, fh)
    cf* sw = sg + K * D;               // [K][D]   exp(-2 pi i fd d / D), fd = jd - F
    cf* sb = sw + K * D;               // [K][K]   pointwise-processed bins
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int vol = blockIdx.x / NF, fh = blockIdx.x - vol * NF;
    cf* gv = G + ((long long)vol * NF + fh) * K * D;
    for (int e = tid; e < K * D; e += nthr) {
        sg[e] = gv[e];
        sw[e] = __ldg(twkd + e);
    }
    __syncthreads();

    const BlVol& bv = vols[shared_desc ? 0 : vol_base + vol];
    int shape[3];
    shape[0] = g.D; shape[1] = g.W; shape[2] = g.H;
    // B[jw][jd] = sum_d G[jw][d] exp(-2 pi i fd d / D), then the pointwise stage on that bin
    for (int o = tid; o < K * K; o += nthr) {
        const int jw = o / K, jd = o - jw * K;
        const cf* row = sg + jw * D;
        const cf* wr = sw + jd * D;
        cf acc = cmk(0.f, 0.f), acc2 = cmk(0.f, 0.f);
        int d = 0;
        for (; d + 1 < D; d += 2) {
            const cf a = row[d], w = wr[d], a2 = row[d + 1], w2 = wr[d + 1];
            acc.x = fmaf(a.x, w.x, fmaf(-a.y, w.y, acc.x));
            acc.y = fmaf(a.x, w.y, fmaf(a.y, w.x, acc.y));
            acc2.x = fmaf(a2.x, w2.x, fmaf(-a2.y, w2.y, acc2.x));
            acc2.y = fmaf(a2.x, w2.y, fmaf(a2.y, w2.x, acc2.y));
        }
        if (d < D) {
            const cf a = row[d], w = wr[d];
            acc.x = fmaf(a.x, w.x, fmaf(-a.y, w.y, acc.x));
            acc.y = fmaf(a.x, w.y, fmaf(a.y, w.x, acc.y));
        }
        acc = cadd(acc, acc2);
        int ish[3];
        ish[0] = (jd - F) + D / 2;
        ish[1] = (jw - F) + g.W / 2;
        ish[2] = fh + g.H / 2;
        sb[o] = pointwise_bin(bv.d, 3, shape, ish, acc, g.scale);
    }
    __syncthreads();
    // G'[jw][d] = sum_jd B[jw][jd] exp(+2 pi i fd d / D)
    for (int o = tid; o < K * D; o += nthr) {
        const int jw = o / D, d = o - jw * D;
        const cf* brow = sb + jw * K;
        cf acc = cmk(0.f, 0.f);
        for (int jd = 0; jd < K; ++jd) {
            const cf b = brow[jd], w = sw[jd * D + d];           // conj(w) = exp(+...)
            acc.x = fmaf(b.x, w.x, fmaf(b.y, w.y, acc.x));
            acc.y = fmaf(b.y, w.x, fmaf(-b.x, w.y, acc.y));
        }
        gv[o] = acc;
    }
}

// ------------------------------------------------------------------ W axis inverse: G[NF][K][D] -> Y[NF][W][D]
template <int NF>
__global__ void __launch_bounds__(128, (NF > 16 ? 2 : 4))
k_bl_inv_w(const cf* __restrict__ G, cf* __restrict__ Y, BlGeom g, int n_tblocks) {
    constexpr int NT = BlDims<NF>::NT;
    MVTB_DYN_SMEM(smem_raw);
    float* sc = (float*)smem_raw;
    const int tid = threadIdx.x;
    bl_load_table<NF>(sc, g.tabC[1], g.tabS[1], g.W, tid, blockDim.x);
    __syncthreads();

    const int W = g.W, D = g.D, K = 2 * g.F + 1;
    const long long vol = blockIdx.x / n_tblocks;
    const int t = (int)(blockIdx.x - vol * n_tblocks) * blockDim.x + tid;
    if (t >= NF * D) return;
    const int fh = t / D, d = t - fh * D;
    const cf* gv = G + ((vol * NF + fh) * (long long)K) * D + d;
    // S_f = G(+f) + G(-f), T_f = G(+f) - G(-f);  y[w] = P + iQ, y[W-w] = P - iQ,  P = sum S_f cos, Q = sum T_f sin
    // kept as (S.x, T.x) and (S.y, T.y) pairs so that one FFMA2 with (cos, sin) updates (P, Q)
    float2 stx[NF], sty[NF];
    MVTB_UNROLL
    for (int f = 0; f < NF; ++f) {
        stx[f] = make_float2(0.f, 0.f);
        sty[f] = make_float2(0.f, 0.f);
        if (f <= g.F) {
            const cf gp = gv[(long long)(g.F + f) * D];
            const cf gm = f > 0 ? gv[(long long)(g.F - f) * D] : cmk(0.f, 0.f);
            stx[f] = make_float2(gp.x + gm.x, f > 0 ? gp.x - gm.x : 0.f);
            sty[f] = make_float2(gp.y + gm.y, f > 0 ? gp.y - gm.y : 0.f);
        }
    }
    cf* yv = Y + ((vol * NF + fh) * (long long)W) * D + d;
    {
        cf s0 = cmk(0.f, 0.f), sn = cmk(0.f, 0.f);
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) {
            s0.x += stx[f].x; s0.y += sty[f].x;
            sn.x += (f & 1) ? -stx[f].x : stx[f].x;
            sn.y += (f & 1) ? -sty[f].x : sty[f].x;
        }
        yv[0] = s0;
        if ((W & 1) == 0) yv[(long long)(W / 2) * D] = sn;
    }
    const int npair = (W - 1) / 2;
    for (int w = 1; w <= npair; ++w) {
        float2 cs[NF];
        bl_row<NF>(sc + w * NT, cs);
        float2 pqx = make_float2(0.f, 0.f), pqy = make_float2(0.f, 0.f);       // (P.x, Q.x), (P.y, Q.y)
        float2 pqx2 = make_float2(0.f, 0.f), pqy2 = make_float2(0.f, 0.f);
        MVTB_UNROLL
        for (int f = 0; f + 1 < NF; f += 2) {
            pqx = fma2(stx[f], cs[f], pqx); pqy = fma2(sty[f], cs[f], pqy);
            pqx2 = fma2(stx[f + 1], cs[f + 1], pqx2); pqy2 = fma2(sty[f + 1], cs[f + 1], pqy2);
        }
        if (NF & 1) { pqx = fma2(stx[NF - 1], cs[NF - 1], pqx); pqy = fma2(sty[NF - 1], cs[NF - 1], pqy); }
        const float Px = pqx.x + pqx2.x, Qx = pqx.y + pqx2.y, Py = pqy.x + pqy2.x, Qy = pqy.y + pqy2.y;
        yv[(long long)w * D] = cmk(Px - Qy, Py + Qx);
        yv[(long long)(W - w) * D] = cmk(Px + Qy, Py - Qx);
    }
}

// ------------------------------------------------------------------ H axis inverse: Y[NF][W*D] -> real volume
__device__ __forceinline__ void bl_atomic_min(float* addr, float v) {
    v += 0.0f;
    if (v >= 0.f) atomicMin((int*)addr, __float_as_int(v));
    else atomicMax((unsigned*)addr, __float_as_uint(v));
}
__device__ __forceinline__ void bl_atomic_max(float* addr, float v) {
    v += 0.0f;
    if (v >= 0.f) atomicMax((int*)addr, __float_as_int(v));
    else atomicMin((unsigned*)addr, __float_as_uint(v));
}

__device__ __forceinline__ void bl_unit(int f, int n, int N, float* c, float* s) {
    // exp(+2 pi i f n / N) with the integer product reduced mod N first
    long long m = ((long long)f * n) % N;
    if (m < 0) m += N;
    sincospif(2.0f * (float)m / (float)N, s, c);
}

template <int NF, int CPT>
__global__ void __launch_bounds__(256, 2)
k_bl_inv_h(const cf* __restrict__ Y, float* __restrict__ out, BlGeom g, int n_cblocks,
           const BlVol* __restrict__ vols, int vol_base, int shared_desc,
           float* __restrict__ minmax, int vols_per_sample) {
    constexpr int NT = BlDims<NF>::NT;
    MVTB_DYN_SMEM(smem_raw);
    const int H = g.H;
    float* sc = (float*)smem_raw;
    cf* seh = (cf*)(sc + (H / 2 + 1) * NT);             // [MVTB_BL_MAX_PW][H/2+1] exp(+2 pi i fh h / H)
    const int tid = threadIdx.x;
    const int vol = blockIdx.x / n_cblocks;
    const BlVol& bv = vols[shared_desc ? 0 : vol_base + vol];
    const int npw = bv.npw;
    bl_load_table<NF>(sc, g.tabC[2], g.tabS[2], H, tid, blockDim.x);
    for (int e = tid; e < MVTB_BL_MAX_PW * (H / 2 + 1); e += blockDim.x) {
        const int s = e / (H / 2 + 1), h = e - s * (H / 2 + 1);
        float c_ = 0.f, s_ = 0.f;
        if (s < npw) bl_unit(bv.pw[s].fh, h, H, &c_, &s_);
        seh[e] = cmk(c_, s_);
    }
    __syncthreads();

    const long long c0 = (long long)(blockIdx.x - (long long)vol * n_cblocks) * (blockDim.x * CPT) + tid;
    bool ok[CPT];
    long long col[CPT];
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) {
        col[k] = c0 + (long long)k * blockDim.x;
        ok[k] = col[k] < g.NC;
        if (!ok[k]) col[k] = g.NC - 1;                  // duplicates a valid column: harmless for min/max
    }
    float lo = __int_as_float(0x7f800000), hi = __int_as_float((int)0xff800000u);
    float2 y2[CPT][NF];                                 // c_f (Re, Im) of the half-spectrum rows, c_0 = 1, c_f = 2
    float2 E[CPT][MVTB_BL_MAX_PW];                      // plane waves: amp exp(+2 pi i (fw w/W + fd d/D)); 0 if unused
    {
        const cf* yv = Y + (long long)vol * NF * g.NC;
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) {
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                const cf y = yv[(long long)f * g.NC + col[k]];
                const float cfw = f == 0 ? 1.f : 2.f;
                y2[k][f] = make_float2(cfw * y.x, cfw * y.y);
            }
            const int w = (int)(col[k] / g.D), d = (int)(col[k] - (long long)w * g.D);
            MVTB_UNROLL
            for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
                E[k][s] = make_float2(0.f, 0.f);
                if (s < npw) {
                    float cw, sw, cd, sd;
                    bl_unit(bv.pw[s].fw, w, g.W, &cw, &sw);
                    bl_unit(bv.pw[s].fd, d, g.D, &cd, &sd);
                    const float amp = bv.pw[s].amp;
                    E[k][s] = make_float2(amp * (cw * cd - sw * sd), amp * (sw * cd + cw * sd));
                }
            }
        }
    }
    float* ov = out + (long long)vol * H * g.NC;
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) {
        float v0 = 0.f, vn = 0.f;
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) { v0 += y2[k][f].x; vn += (f & 1) ? -y2[k][f].x : y2[k][f].x; }
        MVTB_UNROLL
        for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
            v0 += E[k][s].x;                                    // exp(0) = 1
            if ((H & 1) == 0) {
                const cf eh = seh[s * (H / 2 + 1) + H / 2];
                vn += E[k][s].x * eh.x - E[k][s].y * eh.y;
            }
        }
        lo = fminf(lo, v0); hi = fmaxf(hi, v0);
        if (ok[k]) st_stream(ov + col[k], v0);
        if ((H & 1) == 0) {
            lo = fminf(lo, vn); hi = fmaxf(hi, vn);
            if (ok[k]) st_stream(ov + (long long)(H / 2) * g.NC + col[k], vn);
        }
    }
    const int npair = (H - 1) / 2;
    float* plo[CPT];
    float* phi[CPT];
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) { plo[k] = ov + g.NC + col[k]; phi[k] = ov + (long long)(H - 1) * g.NC + col[k]; }
    for (int h = 1; h <= npair; ++h) {
        float2 cs[NF];
        bl_row<NF>(sc + h * NT, cs);
        float2 eh[MVTB_BL_MAX_PW];
        MVTB_UNROLL
        for (int s = 0; s < MVTB_BL_MAX_PW; ++s) eh[s] = seh[s * (H / 2 + 1) + h];
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) {
            // (P, Q) = sum_f (a_f cos, b_f sin) + plane waves;  out[h] = P - Q, out[H-h] = P + Q
            float2 pq = make_float2(0.f, 0.f), pq2 = make_float2(0.f, 0.f);
            MVTB_UNROLL
            for (int f = 0; f + 1 < NF; f += 2) {
                pq = fma2(y2[k][f], cs[f], pq);
                pq2 = fma2(y2[k][f + 1], cs[f + 1], pq2);
            }
            if (NF & 1) pq = fma2(y2[k][NF - 1], cs[NF - 1], pq);
            MVTB_UNROLL
            for (int s = 0; s < MVTB_BL_MAX_PW; ++s) pq2 = fma2(E[k][s], eh[s], pq2);
            const float P = pq.x + pq2.x, Q = pq.y + pq2.y;
            const float v1 = P - Q, v2 = P + Q;
            lo = fminf(lo, fminf(v1, v2));
            hi = fmaxf(hi, fmaxf(v1, v2));
            if (ok[k]) { st_stream(plo[k], v1); st_stream(phi[k], v2); }
            plo[k] += g.NC;
            phi[k] -= g.NC;
        }
    }
    if (minmax != nullptr) {
        __shared__ float s_lo[32], s_hi[32];
        MVTB_UNROLL
        for (int o = 16; o > 0; o >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        const int lane = tid & 31, wp = tid >> 5, nw = (blockDim.x + 31) >> 5;
        if (lane == 0) { s_lo[wp] = lo; s_hi[wp] = hi; }
        __syncthreads();
        if (wp == 0) {
            lo = lane < nw ? s_lo[lane] : __int_as_float(0x7f800000);
            hi = lane < nw ? s_hi[lane] : __int_as_float((int)0xff800000u);
            MVTB_UNROLL
            for (int o = 16; o > 0; o >>= 1) {
                lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
                hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
            }
            if (lane == 0) {
                float* mm = minmax + 2 * ((vol_base + vol) / vols_per_sample);
                bl_atomic_min(mm, lo);
                bl_atomic_max(mm + 1, hi);
            }
        }
    }
}

#include "bandlimited_quad.cuh"
#include "bandlimited_sp.cuh"
#include "bandlimited_tc.cuh"
#include "bandlimited_tci.cuh"

// ------------------------------------------------------------------ host side
size_t bl_workspace_per_volume(const mvtb_plan* p, int F);

static int isqrt_ll(long long v) {
    long long r = (long long)floor(sqrt((double)v));
    while (r * r > v) --r;
    while ((r + 1) * (r + 1) <= v) ++r;
    return (int)r;
}

static int pick_nf(int need) {
    static const int avail[] = {4, 8, 13, 16, 20, 26, 32};
    for (int a : avail)
        if (need <= a) return a;
    return 0;
}

// can this call take the band-limited path?  fills *F_out
bool bl_eligible(const mvtb_plan* p, const mvtb_chain_desc* desc, int n_desc, int* F_out) {
    if (p->ndim != 3 || p->opt_path == MVTB_PATH_GENERAL || !p->bl_tab) return false;
    const long long thr = desc[0].mask_thresh;
    const int kind = desc[0].mask_kind;
    if (kind != MVTB_MASK_DISK && kind != MVTB_MASK_CENTRED) return false;
    for (int i = 0; i < n_desc; ++i) {
        const mvtb_chain_desc& d = desc[i];
        if (d.mask_kind != kind || d.mask_ndim != 3 || d.inside_off || d.mask_thresh < 0) return false;
        if (d.mask_thresh != thr) return false;
        if (d.wrap_naxes != 0 && d.wrap_naxes != 3) return false;
        if (d.n_spikes < 0 || d.n_spikes > MVTB_MAX_SPIKES) return false;
    }
    // Largest |f| any kept bin (or its mirror, for M_eff) can have on one axis.  Disk: f^2 <= thr.  Centred masks
    // (GibbsNoise, GibbsNoiseLayer) measure from (N-1)/2: the per-axis term is (2f+1)^2 on an even axis, (2f)^2 on
    // an odd one, so |f| <= floor((s+1)/2) resp. floor(s/2) with s = floor(sqrt(thr)).  The pointwise stage applies
    // the exact mask; this only sizes the box of frequencies that are computed at all.
    int F = isqrt_ll(thr);
    if (kind == MVTB_MASK_CENTRED) {
        const bool any_even = !(p->shape[0] & 1) || !(p->shape[1] & 1) || !(p->shape[2] & 1);
        F = any_even ? (F + 1) / 2 : F / 2;
    }
    const int nf = pick_nf(F + 1);
    if (nf == 0) return false;
    if (2 * nf - 1 > p->shape[2] || 2 * F + 1 > p->shape[1] || 2 * F + 1 > p->shape[0]) return false;
    for (int i = 0; i < n_desc; ++i) {                      // at most MVTB_BL_MAX_PW spikes outside the kept box
        int outside = 0;
        for (int s = 0; s < desc[i].n_spikes; ++s) {
            bool in_box = true;
            for (int a = 0; a < 3; ++a) {
                const int n = p->shape[2 - a];              // user order: outermost (H) first
                const int idx = desc[i].spikes[s].idx[a];
                if (idx < 0 || idx >= n) return false;      // let the general path report the error
                if (abs(idx - n / 2) > F) in_box = false;
            }
            if (!in_box) ++outside;
        }
        if (outside > MVTB_BL_MAX_PW) return false;
    }
    *F_out = F;
    return true;
}

size_t bl_workspace_per_volume(const mvtb_plan* p, int F) {
    const int nf = pick_nf(F + 1);
    const size_t W = p->shape[1], D = p->shape[0], K = 2 * (size_t)F + 1;
    return sizeof(cf) * (size_t)nf * (W * D + K * D);
}

// splits one user descriptor into the pointwise part (in-box spikes) and plane waves (the rest)
static int bl_make_vol(const mvtb_plan* p, const BlGeom& g, const mvtb_chain_desc& u, BlVol* out) {
    memset(out, 0, sizeof(*out));
    mvtb_chain_desc inbox = u;
    inbox.n_spikes = 0;
    for (int s = 0; s < u.n_spikes; ++s) {
        const int fh = u.spikes[s].idx[0] - g.H / 2, fw = u.spikes[s].idx[1] - g.W / 2, fd = u.spikes[s].idx[2] - g.D / 2;
        if (abs(fh) <= g.F && abs(fw) <= g.F && abs(fd) <= g.F) {
            inbox.spikes[inbox.n_spikes++] = u.spikes[s];
        } else {
            // that bin is masked to exactly 0, so new = amp * exp(i angle(0)) = amp (F:384-390)
            float a = u.spikes[s].amplitude * g.scale;
            if (u.wrap_naxes == 3)
                for (int ax = 0; ax < 3; ++ax)
                    if (u.spikes[s].idx[ax] & 1) a *= u.wrap_alpha;
            PlaneWave& pw = out->pw[out->npw++];
            pw.fh = fh; pw.fw = fw; pw.fd = fd; pw.amp = a;
        }
    }
    return convert_desc(p, &inbox, &out->d);
}

#ifndef MVTB_EMU
// ---- tensor-core H-axis kernels: tensor map of the volume rows, operand tables
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// x viewed as a 2-D fp32 tensor [rows][cols]; box = box_rows x box_cols; no swizzle; out-of-bounds reads give zeros
static int tc_make_tmap(CUtensorMap* out, const float* base, unsigned long long rows, unsigned long long cols, unsigned box_cols,
                        unsigned box_rows) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult qr;
        MVTB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qr));
        if (!f || qr != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled is not available in this driver"); return MVTB_EUNSUPPORTED; }
        fn = (EncodeTiledFn)f;
    }
    const cuuint64_t gdim[2] = {cols, rows};
    const cuuint64_t gstride[1] = {cols * sizeof(float)};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with %d", (int)r); return MVTB_EUNSUPPORTED; }
    return MVTB_OK;
}
// ---- operand tables
static int nf_slot(int nf) {
    static const int avail[] = {4, 8, 13, 16, 20, 26, 32};
    for (int i = 0; i < 7; ++i)
        if (avail[i] == nf) return i;
    return -1;
}
static float tf32_round(float x) {                        // cvt.rna.tf32.f32 on the host: nearest, ties away, 10 mantissa bits
    uint32_t u;
    memcpy(&u, &x, 4);
    u += 0x1000u;
    u &= 0xffffe000u;
    float r;
    memcpy(&r, &u, 4);
    return r;
}
// B operand of the forward pass, [2][H * N] (hi, lo) in tc::op_offset layout: row 2f = cos(2 pi f h / H), row 2f+1 =
// -sin(2 pi f h / H) (Y = sum_h x e^{-2 pi i f h / H}), rows >= 2 NF zero; computed in double, split for 3xTF32
static int tc_fwd_table(mvtb_plan* p, int NF, int N, const float** out) {
    const int slot = nf_slot(NF);
    if (slot < 0) return MVTB_EUNSUPPORTED;
    if (!p->tc_tab_fwd[slot]) {
        const int H = p->shape[2];
        std::vector<float> t((size_t)2 * H * N, 0.f);
        for (int n = 0; n < 2 * NF; ++n)
            for (int h = 0; h < H; ++h) {
                const long long m = ((long long)(n / 2) * h) % H;
                const double ang = 2.0 * M_PI * (double)m / (double)H;
                const double v = (n & 1) ? -sin(ang) : cos(ang);
                const float hi = tf32_round((float)v), lo = tf32_round((float)(v - (double)hi));
                const size_t o = tc::op_offset(n, h, N) / 4;
                t[o] = hi;
                t[(size_t)H * N + o] = lo;
            }
        MVTB_CUDA(cudaMalloc((void**)&p->tc_tab_fwd[slot], t.size() * sizeof(float)));
        MVTB_CUDA(cudaMemcpy(p->tc_tab_fwd[slot], t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    if (!p->tc_status) {
        MVTB_CUDA(cudaMalloc((void**)&p->tc_status, sizeof(int)));
        MVTB_CUDA(cudaMemset(p->tc_status, 0, sizeof(int)));
    }
    *out = p->tc_tab_fwd[slot];
    return MVTB_OK;
}
// B operand of the inverse pass (bandlimited_tci.cuh), [2][K * H] (hi, lo) in tc::op_offset(row = h, k, rows = H) order:
// column 2f = c_f cos(2 pi f h / H), 2f+1 = -c_f sin(2 pi f h / H), c_0 = 1, c_f = 2; the plane-wave columns
// (k >= 2 NF) are zero here and written per volume by the kernel
static int tc_inv_table(mvtb_plan* p, int NF, int K, const float** out) {
    const int slot = nf_slot(NF);
    if (slot < 0) return MVTB_EUNSUPPORTED;
    if (!p->tc_tab_inv[slot]) {
        const int H = p->shape[2];
        std::vector<float> t((size_t)2 * H * K, 0.f);
        for (int k = 0; k < 2 * NF; ++k)
            for (int h = 0; h < H; ++h) {
                const int f = k / 2;
                const long long m = ((long long)f * h) % H;
                const double ang = 2.0 * M_PI * (double)m / (double)H;
                const double cfw = f == 0 ? 1.0 : 2.0;
                const double v = (k & 1) ? -cfw * sin(ang) : cfw * cos(ang);
                const float hi = tf32_round((float)v), lo = tf32_round((float)(v - (double)hi));
                const size_t o = tc::op_offset(h, k, H) / 4;
                t[o] = hi;
                t[(size_t)H * K + o] = lo;
            }
        MVTB_CUDA(cudaMalloc((void**)&p->tc_tab_inv[slot], t.size() * sizeof(float)));
        MVTB_CUDA(cudaMemcpy(p->tc_tab_inv[slot], t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    if (!p->tc_status) {
        MVTB_CUDA(cudaMalloc((void**)&p->tc_status, sizeof(int)));
        MVTB_CUDA(cudaMemset(p->tc_status, 0, sizeof(int)));
    }
    *out = p->tc_tab_inv[slot];
    return MVTB_OK;
}
#endif

// One period of the fused kernel's work queue (bandlimited_sp.cuh): the A inverse tiles of a sample at times
// 0 .. A-1, merged with the B select tiles of earlier samples at times lag + spread * j / B after their own sample's
// first inverse tile came A earlier (wrapped into the period, `periods back` recorded per entry).
static void is_build_pattern(int A, int B, int lag, int spread, std::vector<unsigned>& pat, int* max_back) {
    struct Ent { double t; unsigned e; };
    std::vector<Ent> v;
    v.reserve((size_t)A + B);
    for (int j = 0; j < A; ++j) v.push_back(Ent{(double)j, (unsigned)j});
    int mb = 0;
    for (int j = 0; j < B; ++j) {
        const double tau = (double)lag + (double)spread * (double)j / (double)B;
        int back = 1 + (int)floor(tau / (double)A);
        if (back > 7) back = 7;
        double tin = tau - (double)(back - 1) * A;
        if (tin > (double)A) tin = (double)A;
        if (back > mb) mb = back;
        v.push_back(Ent{tin + 0.5, MVTB_IS_SELECT | ((unsigned)back << 28) | (unsigned)j});
    }
    std::stable_sort(v.begin(), v.end(), [](const Ent& x, const Ent& y) { return x.t < y.t; });
    pat.resize(v.size());
    for (size_t i = 0; i < v.size(); ++i) pat[i] = v[i].e;
    *max_back = mb;
}

// shared memory of the fused W/D kernel: the [K][K] bins share the front of the buffer with the W table; then the
// [K][D] W-bins (later [K][F + 1] float4, which needs K + 1 columns when D = K) and the [D] twiddles
template <int NF>
static size_t bl_midw_smem(const BlGeom& g, int K) {
    const size_t smem_w = sizeof(float) * (size_t)(g.W / 2 + 1) * BlDims<NF>::NT;
    const size_t bins = sizeof(cf) * (size_t)K * K;
    const size_t cols = g.D > K ? (size_t)g.D : (size_t)K + 1;
    return ((smem_w > bins ? smem_w : bins) + 15) / 16 * 16 + sizeof(cf) * ((size_t)K * cols + g.D);
}

template <int NF>
static int bl_run(mvtb_plan* p, const float* in, float* out, int n_volumes, const mvtb_chain_desc* desc, int n_desc,
                  int F, float* minmax_out, int vols_per_sample, void* stream, SpFuse* sp, const float* pre_abt) {
    BlGeom g;
    g.D = p->shape[0]; g.W = p->shape[1]; g.H = p->shape[2];
    g.F = F;
    g.NC = (long long)g.W * g.D;
    for (int a = 0; a < 3; ++a) {
        g.tabC[a] = p->bl_tab + (size_t)p->bl_off[a];
        g.tabS[a] = g.tabC[a] + (size_t)p->shape[a] * MVTB_BL_FT;
    }
    g.twD = p->ax[0].tw;
    g.scale = (float)(1.0 / ((double)g.H * g.W * g.D));
    constexpr int NT = BlDims<NF>::NT;
    const int K = 2 * F + 1;

    // per-volume parameters -> device (one async copy per call)
    std::vector<BlVol> hv((size_t)n_desc);
    for (int i = 0; i < n_desc; ++i) {
        int rc = bl_make_vol(p, g, desc[i], &hv[i]);
        if (rc != MVTB_OK) return rc;
    }
    // ... followed, only when the three-kernel W/D stage will run, by the [K][D] D-axis twiddle table of k_bl_mid
    // (3 875 double-precision sincos on the host for r = 12.5: ~0.1 ms per call that the fused W/D kernel never reads)
    const size_t vol_bytes = (hv.size() * sizeof(BlVol) + 15) & ~(size_t)15;
    const bool split_mid = !p->opt_fusemid || bl_midw_smem<NF>(g, K) > (size_t)113 * 1024;
    std::vector<unsigned char> hbuf(vol_bytes + (split_mid ? sizeof(cf) * (size_t)K * g.D : 0));
    memcpy(hbuf.data(), hv.data(), hv.size() * sizeof(BlVol));
    if (split_mid) {
        cf* tw = (cf*)(hbuf.data() + vol_bytes);
        for (int jd = 0; jd < K; ++jd)
            for (int d = 0; d < g.D; ++d) {
                long long m = ((long long)(jd - F) * d) % g.D;
                if (m < 0) m += g.D;
                const double ang = -2.0 * M_PI * (double)m / (double)g.D;
                tw[(size_t)jd * g.D + d].x = (float)cos(ang);
                tw[(size_t)jd * g.D + d].y = (float)sin(ang);
            }
    }
    const int shared_desc = n_desc == 1 ? 1 : 0;
    const bool quad = (g.H % 4) == 0 && p->opt_quad;      // four rows per table row (bandlimited_quad.cuh)
    constexpr int CPT = BlCols<NF>::CPT;

    // intermediates are ~NF/H of a volume each: keep up to kBlChunk volumes in flight so that the small
    // W-axis / mid kernels get enough CTAs to fill the machine
    const size_t per_vol = bl_workspace_per_volume(p, F);
    int chunk = n_volumes < kBlChunk ? n_volumes : kBlChunk;

    // ---- fused inverse + salt-and-pepper (bandlimited_sp.cuh): when the two-column quad kernel applies
    const int vps = vols_per_sample;
    bool fuse = sp != nullptr && p->opt_fusesp && sp->p > 0.f && minmax_out != nullptr && quad && CPT == 2 && (g.NC % 2) == 0 &&
                g.NC * (long long)g.H < 0x7fffffffLL && (((uintptr_t)out) & 7) == 0 && g.H / 4 - 1 >= 1 &&
                vps >= 1 && vps <= kBlChunk && n_volumes % vps == 0 &&
                // the select pass must find its sample in L2: beyond ~1.5 samples of 36 MB the lines are gone (tools/l2probe.cu)
                // and the separate pass is faster (4-channel BraTS samples of 143 MB: 9.4 k vs 8.9 k samples/s)
                (size_t)vps * p->vol_real * sizeof(float) <= ((size_t)p->is_max_sample_mb << 20);
    // ---- tensor-core inverse pass (bandlimited_tci.cuh), with the select pass folded into its stores when asked for
    bool tc_inv = false, tc_sel = false, tc_fsel = false;
    size_t smem_tci = 0, smem_bits = 0;
    int tci_stages = 2;
    unsigned long long tc_bps = 0;
#ifndef MVTB_EMU
    {
        constexpr int KT = TciDims<NF>::K;
        // B (hi, lo) + four A stages (hi, lo) when they fit, else two
        const size_t tci_pwt = 0;
        tci_stages = sizeof(float) * ((size_t)2 * KT * g.H + (size_t)8 * 128 * KT) + tci_pwt <= (size_t)220 * 1024 ? 4 : 2;
        smem_tci = sizeof(float) * ((size_t)2 * KT * g.H + (size_t)tci_stages * 2 * 128 * KT) + tci_pwt;
        smem_bits = (size_t)((g.NC + 3) / 4) * 16;
        tc_inv = p->opt_tc && p->opt_tc_inv && g.H % kTciRowsPerWord == 0 && g.H >= 16 && g.H <= 256 && smem_tci <= (size_t)220 * 1024 &&
                 g.NC * (long long)g.H < 0x7fffffffLL && nf_slot(NF) >= 0;
        tc_bps = ((unsigned long long)vps * p->vol_real + MVTB_SP_SPAN - 1) / MVTB_SP_SPAN;
        tc_sel = tc_inv && sp != nullptr && sp->p > 0.f && minmax_out != nullptr && vps >= 1 && vps <= kBlChunk &&
                 n_volumes % vps == 0 && smem_bits <= (size_t)200 * 1024 && tc_bps <= 0x7fffffffull;
        // mode 3 (MVTB_TC_INV=2): the select pass inside the store kernel, sample by sample while its lines are in L2
        tc_fsel = tc_sel && p->opt_tc_inv == 2 && (size_t)vps * p->vol_real * sizeof(float) <= ((size_t)p->is_max_sample_mb << 20);
        if (tc_inv) fuse = false;
    }
#endif
    IsArgs ia;
    memset(&ia, 0, sizeof(ia));
    std::vector<unsigned> pattern;
    int max_back = 0;
    size_t pat_off = 0, tab_off = 0;
    if (fuse) {
        if (p->is_chunk > 0 && p->is_chunk < chunk) chunk = p->is_chunk;
        chunk -= chunk % vps;                             // whole samples per launch
        int HS = p->is_hs;
        if (HS > g.H / 4 - 1) HS = g.H / 4 - 1;
        if (HS < 1) HS = 1;
        ia.HS = HS;
        ia.vps = vps;
        ia.ncb2 = (int)((g.NC / 2 + kColThreads - 1) / kColThreads);
        ia.A = vps * ia.ncb2 * HS;
        ia.n_per_sample = (unsigned long long)vps * p->vol_real;
        const unsigned long long bps = (ia.n_per_sample + MVTB_SP_SPAN - 1) / MVTB_SP_SPAN;   // spans per sample
        const unsigned long long B = (bps + 8 * kIsSpansPerWarp - 1) / (8 * kIsSpansPerWarp);       // select tiles: 8 warps x kIsSpansPerWarp spans
        if (bps > 0x7fffffffull || B >= (1ull << 28) || (unsigned long long)ia.A >= (1ull << 28)) fuse = false;
        else {
            ia.bps = (unsigned)bps;
            ia.stride = sp->stride ? sp->stride : bps;
            const int lag = p->is_lag >= 0 ? p->is_lag : 2 * p->num_sms + 8;
            const int spread = (int)((long long)ia.A * p->is_spread_pct / 100);
            is_build_pattern(ia.A, (int)B, lag, spread, pattern, &max_back);
            ia.period = (int)pattern.size();
            const double l2q = log2(1.0 - (double)sp->p);
            ia.inv_log2q = (l2q < 0.0 && l2q > -1e300) ? (float)(1.0 / l2q) : 0.f;
            ia.seed = sp->seed;
            ia.offset = sp->offset;
            ia.minmax = minmax_out;
            ia.debug = getenv("MVTB_IS_DEBUG") ? atoi(getenv("MVTB_IS_DEBUG")) : 0;
        }
    }
    if (tc_sel) {
        chunk -= chunk % vps;                             // whole samples per launch
        tab_off = hbuf.size();
        hbuf.resize(tab_off + sizeof(unsigned) * MVTB_SP_BLOCK);
        int rct = mvtb_sparse_table(sp->p, (unsigned*)(hbuf.data() + tab_off));
        if (rct != MVTB_OK) return rct;
    }
    if (fuse) {
        pat_off = hbuf.size();
        hbuf.resize(pat_off + sizeof(unsigned) * pattern.size());
        memcpy(hbuf.data() + pat_off, pattern.data(), sizeof(unsigned) * pattern.size());
        tab_off = hbuf.size();
        hbuf.resize(tab_off + sizeof(unsigned) * MVTB_SP_BLOCK);
        int rct = mvtb_sparse_table(sp->p, (unsigned*)(hbuf.data() + tab_off));
        if (rct != MVTB_OK) return rct;
    }
    void* dvp = nullptr;
    int rc = plan_stage_upload(p, hbuf.data(), hbuf.size(), stream, &dvp);
    if (rc != MVTB_OK) return rc;
    const BlVol* dv = (const BlVol*)dvp;
    const cf* dtw = (const cf*)((const unsigned char*)dvp + vol_bytes);
    if (tc_fsel && !p->is_sync) MVTB_CUDA(cudaMalloc((void**)&p->is_sync, sizeof(unsigned) * (size_t)(1 + kBlChunk)));
    if (fuse) {
        ia.pattern = (const unsigned*)((const unsigned char*)dvp + pat_off);
        ia.table = (const unsigned*)((const unsigned char*)dvp + tab_off);
        const size_t need = sizeof(unsigned) * (size_t)(1 + kBlChunk);
        if (!p->is_sync) MVTB_CUDA(cudaMalloc((void**)&p->is_sync, need));
        ia.sync = p->is_sync;
    }
    if (p->bl_ws_bytes < per_vol * (size_t)chunk) {
        if (p->bl_ws) cudaFree(p->bl_ws);                // synchronises with work that may still use it
        p->bl_ws = nullptr;
        p->bl_ws_bytes = 0;
        MVTB_CUDA(cudaMalloc((void**)&p->bl_ws, per_vol * (size_t)chunk));
        p->bl_ws_bytes = per_vol * (size_t)chunk;
    }
    const int cols_per_cta = kColThreads * CPT;
    const int n_cblocks = (int)((g.NC + cols_per_cta - 1) / cols_per_cta);
    const int n_tblocks = (NF * g.D + kWThreads - 1) / kWThreads;
    const int n_tblocks_f = (NF * g.D * kWParts + kWThreads - 1) / kWThreads;
    const size_t smem_h = sizeof(float) * (size_t)(g.H / 2 + 1) * NT;
    const size_t smem_w = sizeof(float) * (size_t)(g.W / 2 + 1) * NT;
    const size_t smem_hi = smem_h + sizeof(cf) * MVTB_BL_MAX_PW * (g.H / 2 + 1);
    const size_t smem_mid = sizeof(cf) * ((size_t)2 * K * g.D + (size_t)K * K);

#ifndef MVTB_EMU
    // Fail loudly, if late: every tensor-core wait is bounded, and a kernel that gives up leaves a code in tc_status.
    // The flag travels to a pinned host word at the end of each call (no synchronisation), so a later call sees it.
    if (p->tc_status_h && *(volatile int*)p->tc_status_h != 0) {
        const int code = *(volatile int*)p->tc_status_h;
        p->opt_tc = 0;
        p->opt_tc_inv = 0;
        *(volatile int*)p->tc_status_h = 0;
        cudaMemsetAsync(p->tc_status, 0, sizeof(int), (cudaStream_t)stream);
        set_error("band-limited path: a tensor-core kernel of an earlier call on this plan gave up on an mbarrier wait (code %d); "
                  "that call's output is invalid; the plan now uses the CUDA-core kernels", code);
        return MVTB_ETIMEOUT;
    }
#endif
    bool tc_used = false;
    for (int v0 = 0; v0 < n_volumes; v0 += chunk) {
        const int nv = n_volumes - v0 < chunk ? n_volumes - v0 : chunk;
        cf* Y = p->bl_ws;
        cf* G = Y + (size_t)chunk * NF * g.NC;
        // intensity prologue map: the cp.async forward kernel applies it as it reads; any other forward kernel gets the
        // chunk mapped into its output slot first (the inverse pass overwrites that slot only after the forward pass)
        const float* src = in + (size_t)v0 * p->vol_real;
        const float* abt_v = pre_abt ? pre_abt + (size_t)3 * v0 : nullptr;
        // the select pass's (hit, coin) bits of this chunk: data-independent, so the kernel can run on the plan's side
        // stream next to the W/D stage (a k_sp_bits CTA and a k_bl_midw CTA fit one SM together), joined before the
        // store pass; or in line when the overlap is off
        bool bits_launched = false;
        auto launch_bits = [&](void* st) -> int {
#ifndef MVTB_EMU
            const int RG = g.H / kTciRowsPerWord;
            const size_t need = sizeof(unsigned) * (size_t)chunk * RG * (size_t)g.NC;
            if (p->tc_bits_bytes < need) {
                if (p->tc_bits) cudaFree(p->tc_bits);
                p->tc_bits = nullptr;
                p->tc_bits_bytes = 0;
                MVTB_CUDA(cudaMalloc((void**)&p->tc_bits, need));
                p->tc_bits_bytes = need;
            }
            ProfScope prof(p, MVTB_K_SP_BITS, st);
            SpBitsArgs sa;
            sa.bits = p->tc_bits;
            sa.H = g.H; sa.NC = (int)g.NC; sa.vps = vps; sa.RG = RG;
            sa.vol_n = (unsigned long long)p->vol_real;
            sa.n_per_sample = (unsigned long long)vps * p->vol_real;
            sa.bps = (unsigned)tc_bps;
            sa.stride = sp->stride ? sp->stride : tc_bps;
            sa.s_base = v0 / vps;
            sa.table = (const unsigned*)((const unsigned char*)dvp + tab_off);
            const double l2q = log2(1.0 - (double)sp->p);
            sa.inv_log2q = (l2q < 0.0 && l2q > -1e300) ? (float)(1.0 / l2q) : 0.f;
            sa.seed = sp->seed;
            sa.offset = sp->offset;
            MVTB_LAUNCH(k_sp_bits, dim3((unsigned)(nv * RG)), dim3(1024), smem_bits, st, sa);
#endif
            (void)st;
            return MVTB_OK;
        };
        bool tc_fwd = false;
#ifndef MVTB_EMU
        const int tcN = (2 * NF + 15) / 16 * 16;
        // TMA boxes / A-operand slots of k stages of 16 rows, k the largest divisor of H / 16 up to kTcMaxBoxStages whose
        // slots (32 k TMEM columns each, at least two) fit beside the six accumulators; the raw ring takes what shared
        // memory is left next to the table, at most kTcMaxRing boxes
        int tc_bs = 1, tc_slots = 0, tc_sets = 2;
        for (int k = 1; k <= kTcMaxBoxStages; ++k)
            if ((g.H / kTcRows) % k == 0 && 6 * tcN + 2 * 32 * k <= 512) tc_bs = k;
        if (tc_bs == 1 && g.H / kTcRows > 1) {                  // six accumulators would leave single-stage slots: one set of three
            int k1 = 1;
            for (int k = 1; k <= kTcMaxBoxStages; ++k)
                if ((g.H / kTcRows) % k == 0 && 3 * tcN + 2 * 32 * k <= 512) k1 = k;
            if (k1 > 1) { tc_sets = 1; tc_bs = k1; }
        }
        tc_slots = (512 - 3 * tc_sets * tcN) / (32 * tc_bs);
        if (tc_slots > kTcMaxSlots) tc_slots = kTcMaxSlots;
        const size_t tc_tab = ((size_t)2 * g.H * tcN * sizeof(float) + 1023) & ~(size_t)1023;
        int tc_ring = (int)(((size_t)220 * 1024 - tc_tab) / ((size_t)tc_bs * kTcRows * 128 * sizeof(float)));
        if (tc_ring > kTcMaxRing) tc_ring = kTcMaxRing;
        if (tc_slots > 0) tc_ring -= tc_ring % tc_slots;          // a multiple of the converter groups (= slots): see the kernel
        const size_t smem_tc = tc_tab + (size_t)tc_ring * tc_bs * kTcRows * 128 * sizeof(float);
        tc_fwd = p->opt_tc && (g.H % kTcRows) == 0 && (g.NC % 4) == 0 && ((((uintptr_t)in) & 15) == 0) && tcN <= 64 &&
                 tc_ring >= 2 && tc_slots >= 2 && g.NC * (long long)g.H < 0x7fffffffLL;
#endif
        {
            ProfScope prof(p, tc_fwd ? MVTB_K_BL_FWD_TC : MVTB_K_BL_FWD_H, stream);
            const int ncb1 = (int)((g.NC + kColThreads - 1) / kColThreads);
#ifndef MVTB_EMU
            if (tc_fwd) {
                // pruned DFT along H as a 3xTF32 GEMM on the tensor cores (bandlimited_tc.cuh)
                TcFwdArgs ta;
                CUtensorMap tmap;
                int rcm = tc_make_tmap(&tmap, src, (unsigned long long)nv * g.H, (unsigned long long)g.NC, 128, tc_bs * kTcRows);
                if (rcm != MVTB_OK) return rcm;
                ta.Y = Y;
                int rct = tc_fwd_table(p, NF, tcN, &ta.tab);
                if (rct != MVTB_OK) return rct;
                ta.H = g.H; ta.NC = (int)g.NC; ta.NF = NF; ta.N = tcN;
                ta.tiles_per_vol = (int)((g.NC + 127) / 128);
                ta.n_tiles = ta.tiles_per_vol * nv;
                ta.box_stages = tc_bs;
                ta.ring_boxes = tc_ring;
                ta.a_slots = tc_slots;
                ta.acc_sets = tc_sets;
                ta.abt = abt_v;                                // the intensity prologue map, applied as the converters read x
                ta.status = p->tc_status;
                ta.prof = nullptr;
                if (getenv("MVTB_TC_PROF")) {                  // measurements: waits and an event timeline of CTA 0, printed at the next call
                    static long long* dprof = nullptr;
                    const size_t np = 256 + 32 * 64;
                    if (!dprof) { MVTB_CUDA(cudaMalloc((void**)&dprof, np * sizeof(long long))); }
                    else {
                        std::vector<long long> h(np);
                        MVTB_CUDA(cudaMemcpy(h.data(), dprof, np * sizeof(long long), cudaMemcpyDeviceToHost));
                        fprintf(stderr, "k_bl_fwd_tc CTA 0: total %lld cycles; waits by warp (codes 1..7):", h[0]);
                        for (int w = 0; w < 27; ++w) { fprintf(stderr, "\n  warp %2d:", w); for (int c = 1; c < 8; ++c) fprintf(stderr, " %10lld", h[w * 8 + c]); }
                        fprintf(stderr, "\n");
                    }
                    MVTB_CUDA(cudaMemset(dprof, 0, np * sizeof(long long)));
                    ta.prof = dprof;
                }
                const unsigned grid = (unsigned)(ta.n_tiles < p->num_sms ? ta.n_tiles : p->num_sms);
                MVTB_LAUNCH(k_bl_fwd_tc, dim3(grid), dim3(kTcFwdThreads), smem_tc, stream, tmap, ta);
                tc_used = true;
            } else
#endif
            {
            const bool h4a = !tc_fwd && quad && NF <= 16 && (g.NC % 4) == 0 && ((((uintptr_t)in) & 15) == 0) && p->opt_async;
            if (abt_v && !h4a) {
                int rca = mvtb_intensity_affine_f32(src, out + (size_t)v0 * p->vol_real, p->vol_real, nv, abt_v, stream);
                if (rca != MVTB_OK) return rca;
                src = out + (size_t)v0 * p->vol_real;
                abt_v = nullptr;
            }
            if (h4a) {
                // cp.async staging ring: bytes in flight no longer limited by registers
                const size_t smem_a = smem_h + sizeof(float) * kBlStages * 1024;
                if (abt_v) { auto kern = k_bl_fwd_h4a<NF, true>; MVTB_LAUNCH(kern, dim3((unsigned)(ncb1 * nv)), dim3(kColThreads), smem_a, stream, src, Y, g, ncb1, abt_v); }
                else { auto kern = k_bl_fwd_h4a<NF, false>; MVTB_LAUNCH(kern, dim3((unsigned)(ncb1 * nv)), dim3(kColThreads), smem_a, stream, src, Y, g, ncb1, abt_v); }
            } else if (quad) {
                // one column per thread, 16 loads in flight, 3 CTAs/SM while the accumulators allow
                auto kern = k_bl_fwd_h4<NF, 1, 4, (NF > 16 ? 2 : 3)>;
                MVTB_LAUNCH(kern, dim3((unsigned)(ncb1 * nv)), dim3(kColThreads), smem_h, stream, src, Y, g, ncb1);
            } else {
                auto kern = k_bl_fwd_h<NF, CPT>;
                MVTB_LAUNCH(kern, dim3((unsigned)(n_cblocks * nv)), dim3(kColThreads), smem_h, stream,
                            src, Y, g, n_cblocks);
            }
            }
        }
#ifndef MVTB_EMU
        if (tc_sel && !tc_fsel && p->opt_bits_overlap) {
            if (!p->side_stream) {
                MVTB_CUDA(cudaStreamCreateWithFlags(&p->side_stream, cudaStreamNonBlocking));
                MVTB_CUDA(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
                MVTB_CUDA(cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming));
            }
            // after the forward pass (whose CTAs fill shared memory: nothing fits next to them), and after the previous
            // chunk's store pass, which read the same buffer
            MVTB_CUDA(cudaEventRecord(p->ev_fork, (cudaStream_t)stream));
            MVTB_CUDA(cudaStreamWaitEvent(p->side_stream, p->ev_fork, 0));
            int rcb = launch_bits((void*)p->side_stream);
            if (rcb != MVTB_OK) return rcb;
            MVTB_CUDA(cudaEventRecord(p->ev_join, p->side_stream));
            bits_launched = true;
        }
#endif
        const size_t smem_mw = bl_midw_smem<NF>(g, K);
        // (k_bl_midw measured with clock64 stamps at its phase boundaries, since removed -- the volatile clock reads cost 32 bytes
        // of spills and a third of the kernel's speed: a CTA spends 50 % in the W-axis forward pass, 13 % in the D axis + pointwise
        // stage, 35 % on the way back.  L2 prefetches of the rows ahead, by every 16th computing thread or by the five threads
        // without a column, made CTA 0's forward pass 2.6x faster and the kernel 8-50 % slower; DESIGN 8.)
        if (!split_mid) {                                                   // at least 2 CTAs per SM
            // W axis forward + D axis + pointwise + W axis back in one kernel per (volume, f_h) plane
            ProfScope prof(p, MVTB_K_BL_MID, stream);
            auto kern = k_bl_midw<NF>;
            MVTB_LAUNCH(kern, dim3((unsigned)(nv * NF)), dim3(160), smem_mw, stream, Y, g, dv, v0, shared_desc);
        } else {
            {
                ProfScope prof(p, MVTB_K_BL_FWD_W, stream);
                auto kern = k_bl_fwd_w<NF>;
                MVTB_LAUNCH(kern, dim3((unsigned)(n_tblocks_f * nv)), dim3(kWThreads), smem_w, stream, (const cf*)Y, G, g, n_tblocks_f);
            }
            {
                ProfScope prof(p, MVTB_K_BL_MID, stream);
                MVTB_LAUNCH(k_bl_mid, dim3((unsigned)(nv * NF)), dim3(kMidThreads), smem_mid, stream, G, g, NF, dv, v0, shared_desc, dtw);
            }
            {
                ProfScope prof(p, MVTB_K_BL_INV_W, stream);
                auto kern = k_bl_inv_w<NF>;
                MVTB_LAUNCH(kern, dim3((unsigned)(n_tblocks * nv)), dim3(kWThreads), smem_w, stream, (const cf*)G, Y, g, n_tblocks);
            }
        }
#ifndef MVTB_EMU
        if (tc_inv) {
            constexpr int KT = TciDims<NF>::K;
            TciArgs ta;
            memset(&ta, 0, sizeof(ta));
            ta.Y = (const float2*)Y;
            ta.out = out + (size_t)v0 * p->vol_real;
            int rct = tc_inv_table(p, NF, KT, &ta.tab);
            if (rct != MVTB_OK) return rct;
            ta.vols = dv; ta.vol_base = v0; ta.shared_desc = shared_desc;
            ta.H = g.H; ta.NC = (int)g.NC; ta.W = g.W; ta.D = g.D;
            ta.tiles_per_vol = (int)((g.NC + 127) / 128);
            ta.n_vols = nv;
            if (ta.tiles_per_vol >= p->num_sms) {         // big volumes: a few at a time, so that B's plane-wave columns last
                ta.par_vols = nv < p->tci_par_vols ? nv : p->tci_par_vols;
                ta.ctas_per_vol = p->num_sms / ta.par_vols;
            } else {
                ta.ctas_per_vol = ta.tiles_per_vol;
                ta.par_vols = p->num_sms / ta.ctas_per_vol;
                if (ta.par_vols > nv) ta.par_vols = nv;
            }
            ta.n_stages = tci_stages;
            ta.vps = minmax_out ? vps : 1;
            ta.minmax = minmax_out;
            ta.status = p->tc_status;
            ta.prof = nullptr;
            static long long* dprof_i = nullptr;
            if (getenv("MVTB_TC_PROF")) {                      // measurements: waits of CTA 0 of each launch, printed at the next call
                const size_t np = 3 * 1024;
                if (!dprof_i) { MVTB_CUDA(cudaMalloc((void**)&dprof_i, np * sizeof(long long))); }
                else {
                    std::vector<long long> h(np);
                    MVTB_CUDA(cudaMemcpy(h.data(), dprof_i, np * sizeof(long long), cudaMemcpyDeviceToHost));
                    for (int k = 0; k < 3; ++k) {
                        const long long* q = h.data() + k * 1024;
                        if (!q[0]) continue;
                        fprintf(stderr, "k_bl_inv_tc launch %d CTA 0: total %lld cycles, %lld tiles; per tile: build[loads landed, stage free, arrived] issue[a_full, d_empty, committed] epi0[mma_done, drained] epi1[mma_done, drained]\n", k, q[0], q[6]);
                        for (int t = 0; t < 40; ++t) {
                            fprintf(stderr, "  tile %2d:", t);
                            for (int e = 0; e < 10; ++e) fprintf(stderr, " %7lld%s", q[64 + 16 * t + e], (e == 2 || e == 5 || e == 7) ? " |" : "");
                            fprintf(stderr, "\n");
                        }
                    }
                }
                MVTB_CUDA(cudaMemset(dprof_i, 0, np * sizeof(long long)));
            }
            if (tc_fsel && ta.tiles_per_vol >= p->num_sms) {          // one volume at a time: what is written must still be in L2 when it is selected
                ta.par_vols = getenv("MVTB_TCI_PVF") ? atoi(getenv("MVTB_TCI_PVF")) : 1;
                if (ta.par_vols > nv) ta.par_vols = nv;
                ta.ctas_per_vol = p->num_sms / ta.par_vols;
            }
            ta.debug = getenv("MVTB_TCI_DEBUG") ? atoi(getenv("MVTB_TCI_DEBUG")) : 0;
            const unsigned grid = (unsigned)(ta.par_vols * ta.ctas_per_vol);
            tc_used = true;
            if (tc_fsel) {
                ProfScope prof(p, MVTB_K_BL_INV_TC, stream);
                const int nsamp = nv / vps;
                MVTB_CUDA(cudaMemsetAsync(p->is_sync, 0, sizeof(unsigned) * (size_t)(1 + nsamp), (cudaStream_t)stream));
                ta.sync = p->is_sync;
                ta.sp_table = (const unsigned*)((const unsigned char*)dvp + tab_off);
                const double l2q = log2(1.0 - (double)sp->p);
                ta.inv_log2q = (l2q < 0.0 && l2q > -1e300) ? (float)(1.0 / l2q) : 0.f;
                ta.seed = sp->seed;
                ta.offset = sp->offset;
                ta.n_per_sample = (unsigned long long)vps * p->vol_real;
                ta.bps = (unsigned)tc_bps;
                ta.stride = sp->stride ? sp->stride : tc_bps;
                ta.s_base = v0 / vps;
                if (dprof_i && getenv("MVTB_TC_PROF")) ta.prof = dprof_i + 2048;
                auto kern = k_bl_inv_tc<NF, 3>;
                MVTB_LAUNCH(kern, dim3(grid), dim3(kTciThreads), smem_tci, stream, ta);
            } else if (tc_sel) {
                {
                    ProfScope prof(p, MVTB_K_BL_MM_TC, stream);
                    auto kern = k_bl_inv_tc<NF, 0>;
                    if (dprof_i && getenv("MVTB_TC_PROF")) ta.prof = dprof_i;
                    MVTB_LAUNCH(kern, dim3(grid), dim3(kTciThreads), smem_tci, stream, ta);
                }
                if (!bits_launched) {
                    int rcb = launch_bits(stream);
                    if (rcb != MVTB_OK) return rcb;
                } else {
                    MVTB_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, p->ev_join, 0));
                }
                {
                    ProfScope prof(p, MVTB_K_BL_INV_TC, stream);
                    ta.bits = p->tc_bits;
                    if (dprof_i && getenv("MVTB_TC_PROF")) ta.prof = dprof_i + 1024;
                    auto kern = k_bl_inv_tc<NF, 2>;
                    MVTB_LAUNCH(kern, dim3(grid), dim3(kTciThreads), smem_tci, stream, ta);
                }
            } else {
                ProfScope prof(p, MVTB_K_BL_INV_TC, stream);
                auto kern = k_bl_inv_tc<NF, 1>;
                MVTB_LAUNCH(kern, dim3(grid), dim3(kTciThreads), smem_tci, stream, ta);
            }
        } else
#endif
        if (fuse) {
            ProfScope prof(p, MVTB_K_BL_INV_SP, stream);
            ia.nsamp = nv / vps;
            ia.s_base = v0 / vps;
            ia.total = (unsigned)((ia.nsamp + max_back) * ia.period);
            MVTB_CUDA(cudaMemsetAsync(ia.sync, 0, sizeof(unsigned) * (size_t)(1 + ia.nsamp), (cudaStream_t)stream));
            const size_t smem_is = smem_hi + sizeof(unsigned) * MVTB_SP_BLOCK;
            unsigned grid = (unsigned)(p->num_sms * 2);
            if (grid > ia.total) grid = ia.total;
            float* o = out + (size_t)v0 * p->vol_real;
            if (p->is_store == 0) { auto kern = k_bl_inv_sp<NF, 0>; MVTB_LAUNCH(kern, dim3(grid), dim3(256), smem_is, stream, (const cf*)Y, o, g, dv, v0, shared_desc, ia); }
            else if (p->is_store == 2) { auto kern = k_bl_inv_sp<NF, 2>; MVTB_LAUNCH(kern, dim3(grid), dim3(256), smem_is, stream, (const cf*)Y, o, g, dv, v0, shared_desc, ia); }
            else { auto kern = k_bl_inv_sp<NF, 1>; MVTB_LAUNCH(kern, dim3(grid), dim3(256), smem_is, stream, (const cf*)Y, o, g, dv, v0, shared_desc, ia); }
        } else {
            ProfScope prof(p, MVTB_K_BL_INV_H, stream);
            if (quad && CPT == 2 && (g.NC % 2) == 0 && g.NC * (long long)g.H < 0x7fffffffLL && (((uintptr_t)out) & 7) == 0) {
                const int ncb2 = (int)((g.NC / 2 + kColThreads - 1) / kColThreads);
                auto kern = k_bl_inv_h4v<NF>;
                MVTB_LAUNCH(kern, dim3((unsigned)(ncb2 * nv)), dim3(kColThreads), smem_hi, stream,
                            (const cf*)Y, out + (size_t)v0 * p->vol_real, g, ncb2, dv, v0, shared_desc,
                            minmax_out, minmax_out ? vols_per_sample : 1);
            } else {
                auto kern = quad ? k_bl_inv_h4<NF, CPT> : k_bl_inv_h<NF, CPT>;
                MVTB_LAUNCH(kern, dim3((unsigned)(n_cblocks * nv)), dim3(kColThreads), smem_hi, stream,
                            (const cf*)Y, out + (size_t)v0 * p->vol_real, g, n_cblocks, dv, v0, shared_desc,
                            minmax_out, minmax_out ? vols_per_sample : 1);
            }
        }
    }
#ifndef MVTB_EMU
    if (tc_used && p->tc_status) {
        if (!p->tc_status_h) {
            MVTB_CUDA(cudaMallocHost((void**)&p->tc_status_h, sizeof(int)));
            *p->tc_status_h = 0;
        }
        MVTB_CUDA(cudaMemcpyAsync(p->tc_status_h, p->tc_status, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    }
#endif
    MVTB_CUDA(cudaGetLastError());
    if (sp) sp->done = fuse || tc_sel;
    return MVTB_OK;
}

int bl_chain(mvtb_plan* p, const float* in, float* out, int n_volumes, const mvtb_chain_desc* desc, int n_desc,
             int F, float* minmax_out, int vols_per_sample, void* stream, void* sp_fuse, const float* pre_abt) {
    SpFuse* sp = (SpFuse*)sp_fuse;
    switch (pick_nf(F + 1)) {
        case 4: return bl_run<4>(p, in, out, n_volumes, desc, n_desc, F, minmax_out, vols_per_sample, stream, sp, pre_abt);
        case 8: return bl_run<8>(p, in, out, n_volumes, desc, n_desc, F, minmax_out, vols_per_sample, stream, sp, pre_abt);
        case 13: return bl_run<13>(p, in, out, n_volumes, desc, n_desc, F, minmax_out, vols_per_sample, stream, sp, pre_abt);
        case 16: return bl_run<16>(p, in, out, n_volumes, desc, n_desc, F, minmax_out, vols_per_sample, stream, sp, pre_abt);
        case 20: return bl_run<20>(p, in, out, n_volumes, desc, n_desc, F, minmax_out, vols_per_sample, stream, sp, pre_abt);
        case 26: return bl_run<26>(p, in, out, n_volumes, desc, n_desc, F, minmax_out, vols_per_sample, stream, sp, pre_abt);
        case 32: return bl_run<32>(p, in, out, n_volumes, desc, n_desc, F, minmax_out, vols_per_sample, stream, sp, pre_abt);
        default: set_error("band-limited path: F=%d not instantiated", F); return MVTB_EUNSUPPORTED;
    }
}

#ifndef MVTB_EMU
template <typename K>
static int bl_big_smem(K kern, int optin) {
    cudaFuncAttributes a;
    MVTB_CUDA(cudaFuncGetAttributes(&a, kern));
    MVTB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)a.sharedSizeBytes));
    return MVTB_OK;
}
template <int NF>
static int bl_configure_nf(int optin) {
    constexpr int CPT = BlCols<NF>::CPT;
    int rc;
    if ((rc = bl_big_smem(k_bl_fwd_h<NF, CPT>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_fwd_w<NF>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_inv_w<NF>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_inv_h<NF, CPT>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_fwd_h4<NF, 1, 4, (NF > 16 ? 2 : 3)>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_inv_h4<NF, CPT>, optin)) != MVTB_OK) return rc;
    if (CPT == 2 && (rc = bl_big_smem(k_bl_inv_h4v<NF>, optin)) != MVTB_OK) return rc;
    if (CPT == 2 && (rc = bl_big_smem(k_bl_fwd_h4a<NF, false>, optin)) != MVTB_OK) return rc;
    if (CPT == 2 && (rc = bl_big_smem(k_bl_fwd_h4a<NF, true>, optin)) != MVTB_OK) return rc;
    if (CPT == 2 && (rc = bl_big_smem(k_bl_inv_sp<NF, 0>, optin)) != MVTB_OK) return rc;
    if (CPT == 2 && (rc = bl_big_smem(k_bl_inv_sp<NF, 1>, optin)) != MVTB_OK) return rc;
    if (CPT == 2 && (rc = bl_big_smem(k_bl_inv_sp<NF, 2>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_inv_tc<NF, 0>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_inv_tc<NF, 1>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_inv_tc<NF, 2>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_inv_tc<NF, 3>, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_midw<NF>, optin)) != MVTB_OK) return rc;
    MVTB_CUDA(cudaFuncSetAttribute(k_bl_midw<NF>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    return MVTB_OK;
}
#endif

int configure_bl_kernels(const mvtb_plan* p) {
#ifndef MVTB_EMU
    cudaDeviceProp prop;
    MVTB_CUDA(cudaGetDeviceProperties(&prop, p->device));
    const int optin = (int)prop.sharedMemPerBlockOptin;
    int rc;
    if ((rc = bl_configure_nf<4>(optin)) != MVTB_OK) return rc;
    if ((rc = bl_configure_nf<8>(optin)) != MVTB_OK) return rc;
    if ((rc = bl_configure_nf<13>(optin)) != MVTB_OK) return rc;
    if ((rc = bl_configure_nf<16>(optin)) != MVTB_OK) return rc;
    if ((rc = bl_configure_nf<20>(optin)) != MVTB_OK) return rc;
    if ((rc = bl_configure_nf<26>(optin)) != MVTB_OK) return rc;
    if ((rc = bl_configure_nf<32>(optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_mid, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_bl_fwd_tc, optin)) != MVTB_OK) return rc;
    if ((rc = bl_big_smem(k_sp_bits, optin)) != MVTB_OK) return rc;
#endif
    (void)p;
    return MVTB_OK;
}

}  // namespace mvtb
