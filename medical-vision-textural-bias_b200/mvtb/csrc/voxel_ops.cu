// voxel_ops.cu — HBM-bound voxel kernels: per-sample min/max, salt-and-pepper select with
// injected uniforms or in-kernel Philox4x32-10 (one uniform per voxel, or the geometric-gap sampler
// whose cost is proportional to p), and the even-axis wraparound fold.
//   SaltAndPepper.salt_and_pepper   F:465-482   (F = source_code/filters_and_operators.py)
//   WrapArtifact.__call__           F:503-515   (image-domain form, SURVEY.md A.3)
#include <math.h>

#include "mvtb_common.cuh"
#include "philox.cuh"
#include "sp_sampler.cuh"
#include "mt19937.cuh"

namespace mvtb {

__device__ __forceinline__ void philox_group(uint64_t seed, uint64_t ctr, float* u4) {
    uint4 c = make_uint4((unsigned)ctr, (unsigned)(ctr >> 32), 0u, 0u);
    uint2 k;
    k.x = (unsigned)seed;
    k.y = (unsigned)(seed >> 32);
    const uint4 r = Philox::run(c, k);
    u4[0] = Philox::to_unit(r.x);
    u4[1] = Philox::to_unit(r.y);
    u4[2] = Philox::to_unit(r.z);
    u4[3] = Philox::to_unit(r.w);
}

__global__ void __launch_bounds__(256) k_philox_uniform(float* __restrict__ out, size_t n, uint64_t seed, uint64_t offset) {
    const size_t ngroups = (n + 3) / 4;
    for (size_t gi = (size_t)blockIdx.x * blockDim.x + threadIdx.x; gi < ngroups; gi += (size_t)gridDim.x * blockDim.x) {
        float u[4];
        philox_group(seed, offset + gi, u);
        for (int l = 0; l < 4; ++l)
            if (gi * 4 + l < n) out[gi * 4 + l] = u[l];
    }
}

// ------------------------------------------------------------------ min / max
__device__ __forceinline__ void atomic_min_f32v(float* addr, float v) {
    v += 0.0f;
    if (v >= 0.f) atomicMin((int*)addr, __float_as_int(v));
    else atomicMax((unsigned*)addr, __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f32v(float* addr, float v) {
    v += 0.0f;
    if (v >= 0.f) atomicMax((int*)addr, __float_as_int(v));
    else atomicMin((unsigned*)addr, __float_as_uint(v));
}

__global__ void k_minmax_reset(float* mm, int n_samples) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_samples) {
        mm[2 * i] = __int_as_float(0x7f800000);
        mm[2 * i + 1] = __int_as_float((int)0xff800000u);
    }
}

// grid = (blocks_per_sample, n_samples)
__global__ void __launch_bounds__(256) k_minmax(const float* __restrict__ in, size_t n_per_sample, float* __restrict__ mm) {
    const float* x = in + (size_t)blockIdx.y * n_per_sample;
    float lo = __int_as_float(0x7f800000), hi = __int_as_float((int)0xff800000u);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool vec = ((((uintptr_t)x) & 15) == 0);
    if (vec) {
        const size_t n4 = n_per_sample / 4;
        const float4* x4 = (const float4*)x;
        for (size_t g = i; g < n4; g += stride) {
            const float4 v = x4[g];
            lo = fminf(fminf(lo, v.x), fminf(v.y, fminf(v.z, v.w)));
            hi = fmaxf(fmaxf(hi, v.x), fmaxf(v.y, fmaxf(v.z, v.w)));
        }
        for (size_t e = n4 * 4 + i; e < n_per_sample; e += stride) { lo = fminf(lo, x[e]); hi = fmaxf(hi, x[e]); }
    } else {
        for (size_t e = i; e < n_per_sample; e += stride) { lo = fminf(lo, x[e]); hi = fmaxf(hi, x[e]); }
    }
    __shared__ float s_lo[32], s_hi[32];
    MVTB_UNROLL
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if (lane == 0) { s_lo[w] = lo; s_hi[w] = hi; }
    __syncthreads();
    if (w == 0) {
        lo = lane < nw ? s_lo[lane] : __int_as_float(0x7f800000);
        hi = lane < nw ? s_hi[lane] : __int_as_float((int)0xff800000u);
        MVTB_UNROLL
        for (int o = 16; o > 0; o >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (lane == 0) {
            atomic_min_f32v(mm + 2 * blockIdx.y, lo);
            atomic_max_f32v(mm + 2 * blockIdx.y + 1, hi);
        }
    }
}

// ------------------------------------------------------------------ salt and pepper
// y = u <= p/2 ? MIN : (u <= p ? MAX : x),  MIN = min/2, MAX = max/2 over the sample (F:476-479).
// Comparisons are fp32 against fp32(p/2), fp32(p), as torch does for `tensor <= python_float`.
template <bool PHILOX>
__global__ void __launch_bounds__(256)
k_salt_pepper(const float* __restrict__ in, float* __restrict__ out, size_t n_per_sample, size_t n_total,
              const float* __restrict__ u, uint64_t seed, uint64_t offset, float p, const float* __restrict__ mm) {
    const float ph = 0.5f * p;
    const size_t ngroups = (n_total + 3) / 4;
    const bool vec = (((uintptr_t)in | (uintptr_t)out | (PHILOX ? 0 : (uintptr_t)u)) & 15) == 0;
    for (size_t gi = (size_t)blockIdx.x * blockDim.x + threadIdx.x; gi < ngroups; gi += (size_t)gridDim.x * blockDim.x) {
        const size_t e0 = gi * 4;
        float uu[4], x[4];
        const bool full = vec && e0 + 3 < n_total;
        if (PHILOX) philox_group(seed, offset + gi, uu);
        if (full) {
            const float4 xv = *(const float4*)(in + e0);
            x[0] = xv.x; x[1] = xv.y; x[2] = xv.z; x[3] = xv.w;
            if (!PHILOX) { const float4 uv = *(const float4*)(u + e0); uu[0] = uv.x; uu[1] = uv.y; uu[2] = uv.z; uu[3] = uv.w; }
        } else {
            for (int l = 0; l < 4; ++l) {
                const bool ok = e0 + l < n_total;
                x[l] = ok ? in[e0 + l] : 0.f;
                if (!PHILOX) uu[l] = ok ? u[e0 + l] : 2.f;
            }
        }
        size_t smp = e0 / n_per_sample;
        size_t next = (smp + 1) * n_per_sample;          // first element of the next sample
        float lo = 0.5f * __ldg(mm + 2 * smp), hi = 0.5f * __ldg(mm + 2 * smp + 1);
        float y[4];
        MVTB_UNROLL
        for (int l = 0; l < 4; ++l) {
            if (e0 + l >= next && e0 + l < n_total) {
                ++smp;
                next += n_per_sample;
                lo = 0.5f * __ldg(mm + 2 * smp);
                hi = 0.5f * __ldg(mm + 2 * smp + 1);
            }
            y[l] = uu[l] <= ph ? lo : (uu[l] <= p ? hi : x[l]);
        }
        if (full) {
            *(float4*)(out + e0) = make_float4(y[0], y[1], y[2], y[3]);
        } else {
            for (int l = 0; l < 4; ++l)
                if (e0 + l < n_total) out[e0 + l] = y[l];
        }
    }
}


// Fast path: every sample is a whole number of 16-byte groups and all buffers are 16-byte aligned.
// grid = (blocks per sample, samples): no index division; 4 independent 128-bit loads in flight per thread.
// INPLACE (in == out): a selected voxel becomes a per-sample constant and an unselected one keeps its value,
// so x is never read and only the selected voxels (a fraction p) are stored.
template <bool PHILOX, bool INPLACE>
__global__ void __launch_bounds__(256)
k_salt_pepper_vec(const float* __restrict__ in, float* __restrict__ out, unsigned groups_per_sample,
                  const float* __restrict__ u, uint64_t seed, uint64_t offset, float p, const float* __restrict__ mm) {
    const float ph = 0.5f * p;
    const unsigned smp = blockIdx.y;
    const float lo = 0.5f * __ldg(mm + 2 * smp), hi = 0.5f * __ldg(mm + 2 * smp + 1);
    const size_t base = (size_t)smp * groups_per_sample;            // first group of this sample
    // integer thresholds on the raw 32-bit Philox words (p, ph in [0,1]; p 2^24 is exact in fp32)
    const unsigned kp = (unsigned)(p * 16777216.0f), kph = (unsigned)(ph * 16777216.0f);
    const unsigned tp = kp >= 16777216u ? 0xffffffffu : ((kp << 8) | 0xffu);
    const unsigned tph = kph >= 16777216u ? 0xffffffffu : ((kph << 8) | 0xffu);
    const float4* in4 = (const float4*)in + base;
    const float4* u4 = PHILOX ? nullptr : (const float4*)u + base;
    float4* out4 = (float4*)out + base;
    const unsigned nthreads = gridDim.x * blockDim.x;
    unsigned gi = blockIdx.x * blockDim.x + threadIdx.x;
    for (; gi < groups_per_sample; gi += 4 * nthreads) {
        float4 xv[4], uv[4];
        MVTB_UNROLL
        for (int k = 0; k < 4; ++k) {
            const unsigned g = gi + k * nthreads;
            if (g < groups_per_sample) {
                if (!INPLACE) xv[k] = in4[g];
                if (!PHILOX) uv[k] = u4[g];
            }
        }
        MVTB_UNROLL
        for (int k = 0; k < 4; ++k) {
            const unsigned g = gi + k * nthreads;
            if (g < groups_per_sample) {
                if (PHILOX && INPLACE) {
                    // u = k 2^-24 with k = r >> 8, so  u <= p  <=>  r <= (floor(p 2^24) << 8 | 0xff): integer compares,
                    // no int->float conversion; bit-identical to the float comparison
                    uint4 c = make_uint4((unsigned)(offset + base + g), (unsigned)((offset + base + g) >> 32), 0u, 0u);
                    uint2 key;
                    key.x = (unsigned)seed;
                    key.y = (unsigned)(seed >> 32);
                    const uint4 r = Philox::run(c, key);
                    float* o = (float*)(out4 + g);
                    if (r.x <= tp) o[0] = r.x <= tph ? lo : hi;
                    if (r.y <= tp) o[1] = r.y <= tph ? lo : hi;
                    if (r.z <= tp) o[2] = r.z <= tph ? lo : hi;
                    if (r.w <= tp) o[3] = r.w <= tph ? lo : hi;
                    continue;
                }
                float uu[4];
                if (PHILOX) philox_group(seed, offset + base + g, uu);
                else { uu[0] = uv[k].x; uu[1] = uv[k].y; uu[2] = uv[k].z; uu[3] = uv[k].w; }
                if (INPLACE) {
                    float* o = (float*)(out4 + g);
                    MVTB_UNROLL
                    for (int l = 0; l < 4; ++l)
                        if (uu[l] <= p) o[l] = uu[l] <= ph ? lo : hi;
                } else {
                    float4 y;
                    y.x = uu[0] <= ph ? lo : (uu[0] <= p ? hi : xv[k].x);
                    y.y = uu[1] <= ph ? lo : (uu[1] <= p ? hi : xv[k].y);
                    y.z = uu[2] <= ph ? lo : (uu[2] <= p ? hi : xv[k].z);
                    y.w = uu[3] <= ph ? lo : (uu[3] <= p ? hi : xv[k].w);
                    out4[g] = y;
                }
            }
        }
    }
}


// ------------------------------------------------------------------ sparse salt and pepper (in place)
// One warp per span of MVTB_SP_SPAN voxels (sp_sampler.cuh).  grid = (spans per sample / warps per CTA, samples).
static const int kSpThreadsSparse = 256;

__global__ void __launch_bounds__(kSpThreadsSparse)
k_salt_pepper_sparse(float* __restrict__ x, unsigned long long n_per_sample, unsigned spans_per_sample,
                     const unsigned* __restrict__ table, float inv_log2q, uint64_t seed, uint64_t offset, uint64_t sample_stride,
                     const float* __restrict__ mm) {
    __shared__ unsigned sT[MVTB_SP_BLOCK];
    __shared__ unsigned short s_stage[kSpThreadsSparse / 32][kSpStageIters * 96];
    for (int e = threadIdx.x; e < MVTB_SP_BLOCK; e += blockDim.x) sT[e] = __ldg(table + e);
    __syncthreads();
    const unsigned smp = blockIdx.y;
    const float lo = 0.5f * __ldg(mm + 2 * smp), hi = 0.5f * __ldg(mm + 2 * smp + 1);
    const unsigned span = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (span >= spans_per_sample) return;                      // whole warps leave together
    uint2 key;
    key.x = (unsigned)seed;
    key.y = (unsigned)(seed >> 32);
    sp_walk_spans<1>(x + (size_t)smp * n_per_sample, n_per_sample, span, spans_per_sample,
                     offset + (uint64_t)smp * sample_stride + span, key, sT, inv_log2q, lo, hi, threadIdx.x & 31,
                     s_stage[threadIdx.x >> 5]);
}

// ------------------------------------------------------------------ wraparound fold (all axes even)
// One thread owns the orbit {h, h+H/2} x {w, w+W/2} x {d, d+D/2}: 8 reads, 8 writes, each
// voxel touched exactly once.  Per axis: (y0, y1) = (c0 x0 + s c1 x1, c0 x1 + s c1 x0).
__global__ void __launch_bounds__(256)
k_wrap_fold(const float* __restrict__ in, float* __restrict__ out, int H, int W, int D, float c0,
            float ch, float cw, float cd, size_t n_orbits_total) {
    const int H2 = H / 2, W2 = W / 2, D2 = D / 2;
    const size_t per_vol = (size_t)H2 * W2 * D2;
    const size_t vol_elems = (size_t)H * W * D;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n_orbits_total; t += (size_t)gridDim.x * blockDim.x) {
        const size_t v = t / per_vol;
        size_t r = t - v * per_vol;
        const int d = (int)(r % D2); r /= D2;
        const int w = (int)(r % W2);
        const int h = (int)(r / W2);
        const float* x = in + v * vol_elems;
        float* y = out + v * vol_elems;
        float val[8];
        MVTB_UNROLL
        for (int q = 0; q < 8; ++q) {
            const int hh = h + ((q >> 2) & 1) * H2, ww = w + ((q >> 1) & 1) * W2, dd = d + (q & 1) * D2;
            val[q] = x[((size_t)hh * W + ww) * D + dd];
        }
        MVTB_UNROLL
        for (int q = 0; q < 8; q += 2) {      // D axis: bit 0
            const float a = val[q], b = val[q + 1];
            val[q] = c0 * a + cd * b; val[q + 1] = c0 * b + cd * a;
        }
        MVTB_UNROLL
        for (int q = 0; q < 8; ++q) if (!(q & 2)) {   // W axis: bit 1
            const float a = val[q], b = val[q + 2];
            val[q] = c0 * a + cw * b; val[q + 2] = c0 * b + cw * a;
        }
        MVTB_UNROLL
        for (int q = 0; q < 4; ++q) {         // H axis: bit 2
            const float a = val[q], b = val[q + 4];
            val[q] = c0 * a + ch * b; val[q + 4] = c0 * b + ch * a;
        }
        MVTB_UNROLL
        for (int q = 0; q < 8; ++q) {
            const int hh = h + ((q >> 2) & 1) * H2, ww = w + ((q >> 1) & 1) * W2, dd = d + (q & 1) * D2;
            y[((size_t)hh * W + ww) * D + dd] = val[q];
        }
    }
}

static unsigned grid_for(size_t work_items, int threads, int cap_blocks) {
    size_t b = (work_items + threads - 1) / threads;
    if (b < 1) b = 1;
    if (b > (size_t)cap_blocks) b = cap_blocks;
    return (unsigned)b;
}

}  // namespace mvtb

using namespace mvtb;

// 148 SMs x 8 resident CTAs of 256 threads
static const int kCapBlocks = 148 * 8;

extern "C" int mvtb_philox_uniform_f32(float* out, size_t n, uint64_t seed, uint64_t offset, void* stream) {
    if (!out && n) { set_error("philox_uniform: null output"); return MVTB_EINVAL; }
    if (n == 0) return MVTB_OK;
    MVTB_LAUNCH(k_philox_uniform, dim3(grid_for((n + 3) / 4, 256, kCapBlocks)), dim3(256), 0, stream, out, n, seed, offset);
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

extern "C" int mvtb_minmax_f32(const float* in, size_t n_per_sample, int n_samples, float* minmax_out, void* stream) {
    if (!in || !minmax_out) { set_error("minmax: null argument"); return MVTB_EINVAL; }
    if (n_samples < 0 || n_per_sample == 0) { set_error("minmax: empty sample (torch's max() raises on an empty tensor too)"); return MVTB_EINVAL; }
    if (n_samples == 0) return MVTB_OK;
    if (n_samples > 65535) { set_error("minmax: n_samples=%d > 65535", n_samples); return MVTB_EUNSUPPORTED; }
    MVTB_LAUNCH(k_minmax_reset, dim3((n_samples + 127) / 128), dim3(128), 0, stream, minmax_out, n_samples);
    int per = kCapBlocks / n_samples;
    if (per < 1) per = 1;
    const unsigned bx = grid_for((n_per_sample + 3) / 4, 256, per);
    MVTB_LAUNCH(k_minmax, dim3(bx, (unsigned)n_samples), dim3(256), 0, stream, in, n_per_sample, minmax_out);
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

extern "C" int mvtb_salt_pepper_f32(const float* in, float* out, size_t n_per_sample, int n_samples,
                                    const float* u, uint64_t seed, uint64_t offset, float p,
                                    const float* minmax, void* stream) {
    if (!in || !out || !minmax) { set_error("salt_pepper: null argument"); return MVTB_EINVAL; }
    if (n_samples < 0) { set_error("salt_pepper: n_samples=%d", n_samples); return MVTB_EINVAL; }
    if (!(p >= 0.f && p <= 1.f)) { set_error("salt_pepper: p=%g outside [0,1] (the caller clamps, F:444)", (double)p); return MVTB_EINVAL; }
    const size_t total = n_per_sample * (size_t)n_samples;
    if (total == 0) return MVTB_OK;
    const bool aligned = ((((uintptr_t)in) | ((uintptr_t)out) | ((uintptr_t)u)) & 15) == 0;
    if (aligned && (n_per_sample & 3) == 0 && n_per_sample / 4 < 0xffffffffull && n_samples <= 65535) {
        const unsigned gps = (unsigned)(n_per_sample / 4);
        int per = kCapBlocks / n_samples;
        if (per < 1) per = 1;
        const unsigned bx = grid_for((gps + 3) / 4, 256, per);
        const bool inplace = in == out;
#define MVTB_SP_LAUNCH(PH, IP)                                                                                      \
        do {                                                                                                        \
            auto kern = k_salt_pepper_vec<PH, IP>;                                                                  \
            MVTB_LAUNCH(kern, dim3(bx, (unsigned)n_samples), dim3(256), 0, stream, in, out, gps, u, seed, offset, p, minmax); \
        } while (0)
        if (u) { if (inplace) MVTB_SP_LAUNCH(false, true); else MVTB_SP_LAUNCH(false, false); }
        else   { if (inplace) MVTB_SP_LAUNCH(true, true);  else MVTB_SP_LAUNCH(true, false); }
#undef MVTB_SP_LAUNCH
        MVTB_CUDA(cudaGetLastError());
        return MVTB_OK;
    }
    const unsigned grid = grid_for((total + 3) / 4, 256, kCapBlocks);
    if (u) {
        auto kern = k_salt_pepper<false>;
        MVTB_LAUNCH(kern, dim3(grid), dim3(256), 0, stream, in, out, n_per_sample, total, u, seed, offset, p, minmax);
    } else {
        auto kern = k_salt_pepper<true>;
        MVTB_LAUNCH(kern, dim3(grid), dim3(256), 0, stream, in, out, n_per_sample, total, u, seed, offset, p, minmax);
    }
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

extern "C" int mvtb_sparse_table(float p, unsigned* table_out) {
    if (!table_out || !(p >= 0.f && p <= 1.f)) { set_error("sparse_table: bad argument"); return MVTB_EINVAL; }
    // T[k] = floor(2^32 (1 - (1-p)^(k+1))), with (1-p)^(k+1) by repeated double multiplication (no libm: the same
    // values on every host, and in the numpy restatement under oracle/)
    const double q = 1.0 - (double)p;
    double t = 1.0;
    for (int k = 0; k < MVTB_SP_BLOCK; ++k) {
        t *= q;
        double v = floor((1.0 - t) * 4294967296.0);
        if (v > 4294967295.0) v = 4294967295.0;
        if (v < 0.0) v = 0.0;
        table_out[k] = (unsigned)v;
    }
    return MVTB_OK;
}

namespace mvtb {
int sparse_sp_launch(float* x, size_t n_per_sample, int n_samples, uint64_t seed, uint64_t offset, float p,
                     const float* minmax, const unsigned* table_dev, void* stream, uint64_t sample_stride) {
    const size_t sps = (n_per_sample + MVTB_SP_SPAN - 1) / MVTB_SP_SPAN;
    if (sample_stride == 0) sample_stride = sps;
    if (sample_stride < sps) {
        set_error("salt_pepper_sparse: sample stride %llu below the %llu spans of a sample", (unsigned long long)sample_stride,
                  (unsigned long long)sps);
        return MVTB_EINVAL;
    }
    if (p == 0.f || n_samples == 0 || n_per_sample == 0) return MVTB_OK;   // T = 0 everywhere: no voxel is ever selected
    if (sps > 0x7fffffffull) { set_error("salt_pepper_sparse: sample too large"); return MVTB_EUNSUPPORTED; }
    const unsigned per_cta = (unsigned)(kSpThreadsSparse / 32);
    const unsigned gx = (unsigned)((sps + per_cta - 1) / per_cta);
    const double l2q = log2(1.0 - (double)p);          // -inf for p = 1: the guess is then 0 and the table decides
    const float inv_log2q = (l2q < 0.0 && l2q > -1e300) ? (float)(1.0 / l2q) : 0.f;
    MVTB_LAUNCH(k_salt_pepper_sparse, dim3(gx, (unsigned)n_samples), dim3(kSpThreadsSparse), 0, stream, x,
                (unsigned long long)n_per_sample, (unsigned)sps, table_dev, inv_log2q, seed, offset, sample_stride, minmax);
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}
}  // namespace mvtb

extern "C" int mvtb_salt_pepper_sparse_f32(float* x, size_t n_per_sample, int n_samples, uint64_t seed, uint64_t offset,
                                           float p, const float* minmax, unsigned* table_dev, void* stream) {
    if (!x || !minmax || !table_dev) { set_error("salt_pepper_sparse: null argument"); return MVTB_EINVAL; }
    if (n_samples < 0 || n_samples > 65535) { set_error("salt_pepper_sparse: n_samples=%d", n_samples); return MVTB_EINVAL; }
    if (!(p >= 0.f && p <= 1.f)) { set_error("salt_pepper_sparse: p=%g outside [0,1]", (double)p); return MVTB_EINVAL; }
    if (n_samples == 0 || n_per_sample == 0) return MVTB_OK;
    unsigned host_table[MVTB_SP_BLOCK];
    int rc = mvtb_sparse_table(p, host_table);
    if (rc != MVTB_OK) return rc;
    // 1 KB table: a pageable async copy is staged by the runtime before this call returns (mvtb_kspace_chain_sp_f32
    // sends its table through the plan's pinned staging ring instead)
    MVTB_CUDA(cudaMemcpyAsync(table_dev, host_table, sizeof(host_table), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return sparse_sp_launch(x, n_per_sample, n_samples, seed, offset, p, minmax, table_dev, stream);
}

extern "C" int mvtb_wrap_fold_f32(const float* in, float* out, int n_volumes, int H, int W, int D, float alpha, void* stream) {
    if (!in || !out) { set_error("wrap_fold: null argument"); return MVTB_EINVAL; }
    if (in == out) { set_error("wrap_fold: in-place is not supported"); return MVTB_EINVAL; }
    if (n_volumes < 0 || H < 1 || W < 1 || D < 1) { set_error("wrap_fold: bad shape"); return MVTB_EINVAL; }
    if ((H | W | D) & 1) { set_error("wrap_fold: odd axis in %dx%dx%d (use the k-space chain)", H, W, D); return MVTB_EUNSUPPORTED; }
    if (n_volumes == 0) return MVTB_OK;
    const float c0 = 0.5f * (1.f + alpha), c1 = 0.5f * (1.f - alpha);
    const float ch = ((H / 2) & 1) ? -c1 : c1, cw = ((W / 2) & 1) ? -c1 : c1, cd = ((D / 2) & 1) ? -c1 : c1;
    const size_t orbits = (size_t)n_volumes * (H / 2) * (W / 2) * (D / 2);
    MVTB_LAUNCH(k_wrap_fold, dim3(grid_for(orbits, 256, kCapBlocks * 4)), dim3(256), 0, stream, in, out, H, W, D, c0, ch, cw, cd, orbits);
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}
