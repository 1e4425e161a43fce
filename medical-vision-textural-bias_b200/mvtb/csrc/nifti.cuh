// nifti.cuh — the decode half of MONAI 0.5's LoadImaged -> AsChannelFirstd (127_...FLAIR.py:117-119), included by
// spatial.cu: the raw NIfTI payload (already on the device, file order) -> channel-first float32.
//
// The file stores voxel (i, j, k, c) at element ((c Z + k) Y + j) X + i; the output is out[c][i][j][k], C-contiguous.
// For each (c, j) that is the transpose of an (Z, X) plane: a 32 x 32 tile goes through shared memory, loads along i and
// stores along k, so both sides are coalesced.  On the way in each element is byte-swapped (big-endian files), converted
// and scaled by the value rule of mvtb/nifti.py:
//   unscaled: float(raw), rounded to nearest even where float32 cannot hold it (32-bit integers, float64);
//   scaled: raw * slope + inter in float32 (8/16-bit integers, float32) or float64 (32-bit integers, float64), the multiply
//   and the add rounded separately (__fmul_rn / __fadd_rn, __dmul_rn / __dadd_rn: never contracted into an FMA), then
//   rounded once to float32.
// Bytes: bitpix / 8 in + 4 out per voxel.
#pragma once

#include "mvtb_common.cuh"

namespace mvtb {

#define MVTB_NIFTI_TILE 32
#define MVTB_NIFTI_ROWS 8

__device__ __forceinline__ uint8_t nifti_bswap(uint8_t v) { return v; }
__device__ __forceinline__ uint16_t nifti_bswap(uint16_t v) { return (uint16_t)((v >> 8) | (v << 8)); }
__device__ __forceinline__ uint32_t nifti_bswap(uint32_t v) {
    return (v >> 24) | ((v >> 8) & 0xff00u) | ((v << 8) & 0xff0000u) | (v << 24);
}
__device__ __forceinline__ uint64_t nifti_bswap(uint64_t v) {
    return ((uint64_t)nifti_bswap((uint32_t)v) << 32) | nifti_bswap((uint32_t)(v >> 32));
}

// the file's element type T, read through the unsigned type U of the same width
template <typename T> struct NiftiBits;
template <> struct NiftiBits<uint8_t> { typedef uint8_t U; };
template <> struct NiftiBits<int8_t> { typedef uint8_t U; };
template <> struct NiftiBits<int16_t> { typedef uint16_t U; };
template <> struct NiftiBits<uint16_t> { typedef uint16_t U; };
template <> struct NiftiBits<int32_t> { typedef uint32_t U; };
template <> struct NiftiBits<uint32_t> { typedef uint32_t U; };
template <> struct NiftiBits<float> { typedef uint32_t U; };
template <> struct NiftiBits<double> { typedef uint64_t U; };

template <typename T> __device__ __forceinline__ T nifti_as(typename NiftiBits<T>::U u) { T v; memcpy(&v, &u, sizeof(T)); return v; }

// unscaled conversion
__device__ __forceinline__ float nifti_f32(uint8_t v) { return (float)v; }
__device__ __forceinline__ float nifti_f32(int8_t v) { return (float)v; }
__device__ __forceinline__ float nifti_f32(int16_t v) { return (float)v; }
__device__ __forceinline__ float nifti_f32(uint16_t v) { return (float)v; }
__device__ __forceinline__ float nifti_f32(int32_t v) { return __int2float_rn(v); }
__device__ __forceinline__ float nifti_f32(uint32_t v) { return __uint2float_rn(v); }
__device__ __forceinline__ float nifti_f32(float v) { return v; }
__device__ __forceinline__ float nifti_f32(double v) { return __double2float_rn(v); }

// scaled conversion in np.result_type(T, float32): float64 for the 32-bit integers and float64, float32 otherwise
template <typename T> struct NiftiWide { static const bool value = false; };
template <> struct NiftiWide<int32_t> { static const bool value = true; };
template <> struct NiftiWide<uint32_t> { static const bool value = true; };
template <> struct NiftiWide<double> { static const bool value = true; };
template <typename T>
__device__ __forceinline__ float nifti_scale(T v, float s32, float i32, double s64, double i64) {
    if (NiftiWide<T>::value) return __double2float_rn(__dadd_rn(__dmul_rn((double)v, s64), i64));
    return __fadd_rn(__fmul_rn((float)v, s32), i32);
}

struct NiftiDev {
    int X, Y, Z;
    long long C;
    int swap, scaled;
    float s32, i32;
    double s64, i64;
};

// grid: x = tiles along i, y = tiles along k, z strides over the C * Y planes; block (32, 8)
template <typename T>
__global__ void __launch_bounds__(MVTB_NIFTI_TILE * MVTB_NIFTI_ROWS)
k_nifti_decode(const T* __restrict__ raw, float* __restrict__ out, NiftiDev g) {
    typedef typename NiftiBits<T>::U U;
    __shared__ float tile[MVTB_NIFTI_TILE][MVTB_NIFTI_TILE + 1];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int i0 = blockIdx.x * MVTB_NIFTI_TILE, k0 = blockIdx.y * MVTB_NIFTI_TILE;
    const long long planes = g.C * g.Y, xyz = (long long)g.X * g.Y * g.Z;
    const U* src = (const U*)raw;
    for (long long p = blockIdx.z; p < planes; p += gridDim.z) {
        const long long c = p / g.Y;
        const int j = (int)(p - c * g.Y);
        // load: element ((c Z + k) Y + j) X + i, lanes along i
        const int i = i0 + tx;
        MVTB_UNROLL
        for (int r = 0; r < MVTB_NIFTI_TILE; r += MVTB_NIFTI_ROWS) {
            const int k = k0 + ty + r;
            if (i < g.X && k < g.Z) {
                U u = __ldg(src + ((c * g.Z + k) * g.Y + j) * (long long)g.X + i);
                if (g.swap) u = nifti_bswap(u);
                const T v = nifti_as<T>(u);
                tile[ty + r][tx] = g.scaled ? nifti_scale(v, g.s32, g.i32, g.s64, g.i64) : nifti_f32(v);
            }
        }
        __syncthreads();
        // store: out[c][i][j][k], lanes along k
        const int k = k0 + tx;
        float* dst = out + c * xyz + j * (long long)g.Z + k;
        MVTB_UNROLL
        for (int r = 0; r < MVTB_NIFTI_TILE; r += MVTB_NIFTI_ROWS) {
            const int ii = i0 + ty + r;
            if (ii < g.X && k < g.Z) dst[(long long)ii * g.Y * g.Z] = tile[tx][ty + r];
        }
        __syncthreads();
    }
}

}  // namespace mvtb
