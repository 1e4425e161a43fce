// spatial.cu — the two index transforms between the resampled volume and the intensity prologue in every training script
// of the reference (10_scripts/127_.../stylized_gibbs12p5_spikes15_wrap0p5_sap0p05_FLAIR.py:130-133):
//     RandSpatialCropd(roi_size=[128, 128, 64], random_size=False)  ->  RandFlipd(prob=0.5, spatial_axis=0)
// (validation: CenterSpatialCropd).  Both are MONAI 0.5 transforms (monai/transforms/croppad/array.py: SpatialCrop,
// CenterSpatialCrop, RandSpatialCrop; spatial/array.py: Flip = np.flip per channel; MONAI is not part of /root/reference,
// oracle/monai_spatial.py restates them).  Crop then flip is one gather:
//     out[c][i][j][k] = in[c][o0 + (f0 ? s0-1-i : i)][o1 + (f1 ? s1-1-j : j)][o2 + (f2 ? s2-1-k : k)]
// 8 B/voxel of the crop, nothing else; the host draws the offsets and the flip in MONAI's order (mvtb/spatial.py).
// The resampling in front of them (Spacingd -> Orientationd) is k_resample (resample.cuh); in front of that, the NIfTI
// payload is decoded to channel-first float32 by k_nifti_decode (nifti.cuh).
#include "mvtb_common.cuh"
#include "nifti.cuh"
#include "resample.cuh"

namespace mvtb {

struct CropGeom {
    int iw, id;            // input W, D (row pitch and plane pitch in elements come from these)
    long long in_chan;     // elements per input channel
    int s0, s1, s2;        // output shape
    int o0, o1, o2;        // first input index kept on each axis
    int flip;              // bit a: spatial axis a is reversed
};

__global__ void __launch_bounds__(256)
k_crop_flip(const float* __restrict__ in, float* __restrict__ out, CropGeom g, long long n_rows_total) {
    // one warp per output row (c, i, j): the row's s2 elements are contiguous on both sides (reversed when axis 2 flips)
    const int lane = threadIdx.x & 31;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = wid; r < n_rows_total; r += nw) {
        const long long c = r / ((long long)g.s0 * g.s1);
        const int rem = (int)(r - c * (long long)g.s0 * g.s1);
        const int i = rem / g.s1, j = rem - i * g.s1;
        const int si = g.o0 + ((g.flip & 1) ? g.s0 - 1 - i : i);
        const int sj = g.o1 + ((g.flip & 2) ? g.s1 - 1 - j : j);
        const float* src = in + c * g.in_chan + ((long long)si * g.iw + sj) * g.id + g.o2;
        float* dst = out + r * g.s2;
        if (g.flip & 4) {
            for (int k = lane; k < g.s2; k += 32) dst[k] = src[g.s2 - 1 - k];
        } else {
            for (int k = lane; k < g.s2; k += 32) dst[k] = src[k];
        }
    }
}

// the same gather for a batch of samples of one shape, each with its own window and flips (device arrays: the training
// loader draws them per sample); sample b reads in + b * in_sample, writes out + b * (C s0 s1 s2)
__global__ void __launch_bounds__(256)
k_crop_flip_batch(const float* __restrict__ in, float* __restrict__ out, CropGeom g, long long rows_per_sample, long long in_sample,
                  const int* __restrict__ offsets, const int* __restrict__ flips, long long n_rows_total) {
    const int lane = threadIdx.x & 31;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long rr = wid; rr < n_rows_total; rr += nw) {
        const long long b = rr / rows_per_sample, r = rr - b * rows_per_sample;
        const int o0 = __ldg(offsets + 3 * b), o1 = __ldg(offsets + 3 * b + 1), o2 = __ldg(offsets + 3 * b + 2), fl = __ldg(flips + b);
        const long long c = r / ((long long)g.s0 * g.s1);
        const int rem = (int)(r - c * (long long)g.s0 * g.s1);
        const int i = rem / g.s1, j = rem - i * g.s1;
        const int si = o0 + ((fl & 1) ? g.s0 - 1 - i : i);
        const int sj = o1 + ((fl & 2) ? g.s1 - 1 - j : j);
        const float* src = in + b * in_sample + c * g.in_chan + ((long long)si * g.iw + sj) * g.id + o2;
        float* dst = out + rr * g.s2;
        if (fl & 4) {
            for (int k = lane; k < g.s2; k += 32) dst[k] = src[g.s2 - 1 - k];
        } else {
            for (int k = lane; k < g.s2; k += 32) dst[k] = src[k];
        }
    }
}

// the same gather from a ragged cache (the training loader's DeviceCache): sample b reads cache entry entry[b], whose
// spatial shape and first element come from the entry tables, so every sample finds its own row and plane pitch; the
// output channels are the entry's channels g.ch[0 .. n_out_ch) (a SelectChanneld folded into the gather)
struct GatherGeom {
    int s0, s1, s2;        // output shape
    int ch[MVTB_GATHER_MAX_CHANNELS];
};

__global__ void __launch_bounds__(256)
k_crop_flip_gather(const float* __restrict__ cache, float* __restrict__ out, GatherGeom g, long long rows_per_sample,
                   const long long* __restrict__ entry_offset, const int* __restrict__ entry_shape, const int* __restrict__ entry,
                   const int* __restrict__ starts, const int* __restrict__ flips, long long n_rows_total) {
    const int lane = threadIdx.x & 31;
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long rr = wid; rr < n_rows_total; rr += nw) {
        const long long b = rr / rows_per_sample, r = rr - b * rows_per_sample;
        const int e = __ldg(entry + b);
        const int iw = __ldg(entry_shape + 3 * e + 1), id = __ldg(entry_shape + 3 * e + 2);
        const long long in_chan = (long long)__ldg(entry_shape + 3 * e) * iw * id;
        const int o0 = __ldg(starts + 3 * b), o1 = __ldg(starts + 3 * b + 1), o2 = __ldg(starts + 3 * b + 2), fl = __ldg(flips + b);
        const int c = (int)(r / ((long long)g.s0 * g.s1));
        const int rem = (int)(r - (long long)c * g.s0 * g.s1);
        const int i = rem / g.s1, j = rem - i * g.s1;
        const int si = o0 + ((fl & 1) ? g.s0 - 1 - i : i);
        const int sj = o1 + ((fl & 2) ? g.s1 - 1 - j : j);
        const float* src = cache + __ldg(entry_offset + e) + g.ch[c] * in_chan + ((long long)si * iw + sj) * id + o2;
        float* dst = out + rr * g.s2;
        if (fl & 4) {
            for (int k = lane; k < g.s2; k += 32) dst[k] = src[g.s2 - 1 - k];
        } else {
            for (int k = lane; k < g.s2; k += 32) dst[k] = src[k];
        }
    }
}

}  // namespace mvtb

using namespace mvtb;

extern "C" int mvtb_crop_flip_gather_f32(const float* cache, float* out, int n_samples, int n_channels_out, const int64_t* entry_offset_dev,
                                         const int32_t* entry_shape_dev, int n_channels_in, const int32_t* channels,
                                         const int32_t* out_shape, const int32_t* entry_dev, const int32_t* starts_dev,
                                         const int32_t* flips_dev, void* stream) {
    if (!cache || !out || !entry_offset_dev || !entry_shape_dev || !out_shape || !entry_dev || !starts_dev || !flips_dev) {
        set_error("crop_flip_gather: null argument");
        return MVTB_EINVAL;
    }
    if (cache == out) { set_error("crop_flip_gather: in-place is not supported"); return MVTB_EINVAL; }
    if (n_samples < 0 || n_channels_out < 0 || n_channels_in < 0) { set_error("crop_flip_gather: negative count"); return MVTB_EINVAL; }
    if (n_channels_out > MVTB_GATHER_MAX_CHANNELS) {
        set_error("crop_flip_gather: %d output channels, at most %d", n_channels_out, MVTB_GATHER_MAX_CHANNELS);
        return MVTB_EINVAL;
    }
    if (!channels && n_channels_out != n_channels_in) {
        set_error("crop_flip_gather: channels = NULL selects all %d channels, not %d", n_channels_in, n_channels_out);
        return MVTB_EINVAL;
    }
    GatherGeom g;
    for (int c = 0; c < MVTB_GATHER_MAX_CHANNELS; ++c) g.ch[c] = 0;
    for (int c = 0; c < n_channels_out; ++c) {
        g.ch[c] = channels ? channels[c] : c;
        if (g.ch[c] < 0 || g.ch[c] >= n_channels_in) {
            set_error("crop_flip_gather: channel %d outside the %d stored channels", g.ch[c], n_channels_in);
            return MVTB_EINVAL;
        }
    }
    for (int a = 0; a < 3; ++a)
        if (out_shape[a] < 1) { set_error("crop_flip_gather: output axis %d has size %d", a, out_shape[a]); return MVTB_EINVAL; }
    g.s0 = out_shape[0]; g.s1 = out_shape[1]; g.s2 = out_shape[2];
    const long long rows_per_sample = (long long)n_channels_out * g.s0 * g.s1;
    const long long rows = rows_per_sample * n_samples;
    if (rows == 0) return MVTB_OK;
    long long blocks = (rows + 7) / 8;                      // 8 warps per CTA
    if (blocks > 148 * 16) blocks = 148 * 16;
    MVTB_LAUNCH(k_crop_flip_gather, dim3((unsigned)blocks), dim3(256), 0, stream, cache, out, g, rows_per_sample,
                (const long long*)entry_offset_dev, (const int*)entry_shape_dev, (const int*)entry_dev, (const int*)starts_dev,
                (const int*)flips_dev, rows);
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

extern "C" int mvtb_crop_flip_f32(const float* in, float* out, int n_channels, const int32_t* in_shape, const int32_t* out_shape,
                                  const int32_t* offset, int flip_axes_mask, void* stream) {
    if (!in || !out || !in_shape || !out_shape || !offset) { set_error("crop_flip: null argument"); return MVTB_EINVAL; }
    if (in == out) { set_error("crop_flip: in-place is not supported"); return MVTB_EINVAL; }
    if (n_channels < 0 || (flip_axes_mask & ~7)) { set_error("crop_flip: bad channel count or flip mask"); return MVTB_EINVAL; }
    for (int a = 0; a < 3; ++a) {
        if (in_shape[a] < 1 || out_shape[a] < 0 || offset[a] < 0 || (long long)offset[a] + out_shape[a] > in_shape[a]) {
            set_error("crop_flip: axis %d: offset %d + size %d does not fit in %d", a, offset[a], out_shape[a], in_shape[a]);
            return MVTB_EINVAL;
        }
    }
    const long long rows = (long long)n_channels * out_shape[0] * out_shape[1];
    if (rows == 0 || out_shape[2] == 0) return MVTB_OK;
    CropGeom g;
    g.iw = in_shape[1]; g.id = in_shape[2];
    g.in_chan = (long long)in_shape[0] * in_shape[1] * in_shape[2];
    g.s0 = out_shape[0]; g.s1 = out_shape[1]; g.s2 = out_shape[2];
    g.o0 = offset[0]; g.o1 = offset[1]; g.o2 = offset[2];
    g.flip = flip_axes_mask;
    long long blocks = (rows + 7) / 8;                      // 8 warps per CTA
    if (blocks > 148 * 16) blocks = 148 * 16;
    MVTB_LAUNCH(k_crop_flip, dim3((unsigned)blocks), dim3(256), 0, stream, in, out, g, rows);
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

// offsets_dev[3 n_samples], flips_dev[n_samples]: int32 on the device; every window must fit (the caller draws them with
// MONAI's bounds, 0 <= o <= N - s); not checked here, the arrays live on the device.
extern "C" int mvtb_crop_flip_batch_f32(const float* in, float* out, int n_samples, int n_channels, const int32_t* in_shape,
                                        const int32_t* out_shape, const int32_t* offsets_dev, const int32_t* flips_dev, void* stream) {
    if (!in || !out || !in_shape || !out_shape || !offsets_dev || !flips_dev) { set_error("crop_flip_batch: null argument"); return MVTB_EINVAL; }
    if (in == out) { set_error("crop_flip_batch: in-place is not supported"); return MVTB_EINVAL; }
    if (n_samples < 0 || n_channels < 0) { set_error("crop_flip_batch: negative count"); return MVTB_EINVAL; }
    for (int a = 0; a < 3; ++a)
        if (in_shape[a] < 1 || out_shape[a] < 0 || out_shape[a] > in_shape[a]) { set_error("crop_flip_batch: axis %d: size %d of %d", a, out_shape[a], in_shape[a]); return MVTB_EINVAL; }
    const long long rows_per_sample = (long long)n_channels * out_shape[0] * out_shape[1];
    const long long rows = rows_per_sample * n_samples;
    if (rows == 0 || out_shape[2] == 0) return MVTB_OK;
    CropGeom g;
    g.iw = in_shape[1]; g.id = in_shape[2];
    g.in_chan = (long long)in_shape[0] * in_shape[1] * in_shape[2];
    g.s0 = out_shape[0]; g.s1 = out_shape[1]; g.s2 = out_shape[2];
    g.o0 = g.o1 = g.o2 = 0; g.flip = 0;
    long long blocks = (rows + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    MVTB_LAUNCH(k_crop_flip_batch, dim3((unsigned)blocks), dim3(256), 0, stream, in, out, g, rows_per_sample, g.in_chan * n_channels,
                offsets_dev, flips_dev, rows);
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

static bool is_perm3(const int32_t* p) {
    return p[0] >= 0 && p[0] < 3 && p[1] >= 0 && p[1] < 3 && p[2] >= 0 && p[2] < 3 && p[0] != p[1] && p[0] != p[2] && p[1] != p[2];
}

extern "C" int mvtb_resample_f32(const float* in, float* out, int n_volumes, const mvtb_resample_geom* geom, void* stream) {
    if (!in || !out || !geom) { set_error("resample: null argument"); return MVTB_EINVAL; }
    if (in == out) { set_error("resample: in-place is not supported"); return MVTB_EINVAL; }
    const mvtb_resample_geom& G = *geom;
    if (n_volumes < 0) { set_error("resample: negative volume count"); return MVTB_EINVAL; }
    if (G.mode != MVTB_RESAMPLE_BILINEAR && G.mode != MVTB_RESAMPLE_NEAREST) { set_error("resample: unknown mode %d", G.mode); return MVTB_EINVAL; }
    for (int a = 0; a < 3; ++a)
        if (G.in_shape[a] < 1 || G.grid_shape[a] < 1 || G.out_shape[a] < 0) {
            set_error("resample: axis %d: source %d, grid %d, output %d", a, G.in_shape[a], G.grid_shape[a], G.out_shape[a]);
            return MVTB_EINVAL;
        }
    if ((long long)G.in_shape[0] * G.in_shape[1] * G.in_shape[2] > 0x7fffffffLL) { set_error("resample: source volume over 2^31 voxels"); return MVTB_EINVAL; }
    if (!is_perm3(G.axis)) { set_error("resample: axis is not a permutation of (0, 1, 2)"); return MVTB_EINVAL; }
    for (int g = 0; g < 3; ++g) {
        const long long n = G.out_shape[G.axis[g]], last = (long long)G.base[g] + (long long)G.step[g] * (n - 1);
        if ((G.step[g] != 1 && G.step[g] != -1) || (n > 0 && (G.base[g] < 0 || G.base[g] >= G.grid_shape[g] || last < 0 || last >= G.grid_shape[g]))) {
            set_error("resample: grid axis %d: base %d step %d over %lld outputs leaves [0, %d)", g, G.base[g], G.step[g], n, G.grid_shape[g]);
            return MVTB_EINVAL;
        }
    }
    ResampleDev d;
    d.in_vol = (long long)G.in_shape[0] * G.in_shape[1] * G.in_shape[2];
    for (int a = 0; a < 3; ++a) d.in_n[a] = G.in_shape[a];
    d.in_stride[0] = G.in_shape[1] * G.in_shape[2]; d.in_stride[1] = G.in_shape[2]; d.in_stride[2] = 1;
    d.s0 = G.out_shape[0]; d.s1 = G.out_shape[1]; d.s2 = G.out_shape[2];
    d.taps = G.taps;
    if (G.taps) {
        if (!is_perm3(G.tap_grid)) { set_error("resample: tap_grid is not a permutation of (0, 1, 2)"); return MVTB_EINVAL; }
        for (int k = 0; k < 3; ++k) {
            const int g = G.tap_grid[k];
            if (G.tap_off[k] < 0 || (long long)G.tap_off[k] + G.grid_shape[g] > G.n_taps) {
                set_error("resample: source axis %d: taps [%d, %d) outside the %d entries", k, G.tap_off[k], G.tap_off[k] + G.grid_shape[g], G.n_taps);
                return MVTB_EINVAL;
            }
            d.ax[k] = G.axis[g]; d.base[k] = G.tap_off[k] + G.base[g]; d.step[k] = G.step[g];
        }
    } else {
        for (int i = 0; i < 12; ++i)
            if (!std::isfinite(G.matrix[i])) { set_error("resample: matrix entry %d is not finite", i); return MVTB_EINVAL; }
        for (int g = 0; g < 3; ++g) { d.ax[g] = G.axis[g]; d.base[g] = G.base[g]; d.step[g] = G.step[g]; }
        for (int k = 0; k < 3; ++k)
            for (int i = 0; i < 4; ++i) d.m[k][i] = G.matrix[4 * k + i];
    }
    const long long rows = (long long)n_volumes * d.s0 * d.s1;
    if (rows == 0 || d.s2 == 0) return MVTB_OK;
    long long blocks = (rows + 7) / 8;                      // one warp per output row, 8 warps per CTA
    if (blocks > 148 * 16) blocks = 148 * 16;
    const bool nearest = G.mode == MVTB_RESAMPLE_NEAREST;
    if (G.taps && nearest) { auto kern = k_resample<true, true>; MVTB_LAUNCH(kern, dim3((unsigned)blocks), dim3(256), 0, stream, in, out, d, rows); }
    else if (G.taps) { auto kern = k_resample<true, false>; MVTB_LAUNCH(kern, dim3((unsigned)blocks), dim3(256), 0, stream, in, out, d, rows); }
    else if (nearest) { auto kern = k_resample<false, true>; MVTB_LAUNCH(kern, dim3((unsigned)blocks), dim3(256), 0, stream, in, out, d, rows); }
    else { auto kern = k_resample<false, false>; MVTB_LAUNCH(kern, dim3((unsigned)blocks), dim3(256), 0, stream, in, out, d, rows); }
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

// NIfTI datatype code -> element bytes (0: not supported)
static int nifti_bytes(int32_t datatype) {
    switch (datatype) {
        case MVTB_NIFTI_UINT8: case MVTB_NIFTI_INT8: return 1;
        case MVTB_NIFTI_INT16: case MVTB_NIFTI_UINT16: return 2;
        case MVTB_NIFTI_INT32: case MVTB_NIFTI_UINT32: case MVTB_NIFTI_FLOAT32: return 4;
        case MVTB_NIFTI_FLOAT64: return 8;
        default: return 0;
    }
}

template <typename T>
static void nifti_launch(const void* raw, float* out, const NiftiDev& d, void* stream) {
    const long long planes = d.C * d.Y;
    const dim3 grid((unsigned)((d.X + MVTB_NIFTI_TILE - 1) / MVTB_NIFTI_TILE), (unsigned)((d.Z + MVTB_NIFTI_TILE - 1) / MVTB_NIFTI_TILE),
                    (unsigned)(planes < 65535 ? planes : 65535));
    auto kern = k_nifti_decode<T>;
    MVTB_LAUNCH(kern, grid, dim3(MVTB_NIFTI_TILE, MVTB_NIFTI_ROWS), 0, stream, (const T*)raw, out, d);
}

extern "C" int mvtb_nifti_decode_f32(const void* raw, float* out, int32_t datatype, int32_t swap_bytes, const int64_t* dims, double slope,
                                     double inter, int32_t scaled, void* stream) {
    if (!raw || !out || !dims) { set_error("nifti_decode: null argument"); return MVTB_EINVAL; }
    if (raw == (const void*)out) { set_error("nifti_decode: in-place is not supported"); return MVTB_EINVAL; }
    const int bytes = nifti_bytes(datatype);
    if (!bytes) { set_error("nifti_decode: NIfTI datatype %d is not supported", datatype); return MVTB_EUNSUPPORTED; }
    if ((uintptr_t)raw % bytes) { set_error("nifti_decode: payload address not aligned to its %d-byte elements", bytes); return MVTB_EINVAL; }
    for (int a = 0; a < 4; ++a)
        if (dims[a] < 1) { set_error("nifti_decode: dims[%d] = %lld", a, (long long)dims[a]); return MVTB_EINVAL; }
    if (dims[0] > 0x7fffffffLL || dims[1] > 0x7fffffffLL || dims[2] > 0x7fffffffLL || dims[0] * dims[1] * dims[2] > 0x7fffffffLL) {
        set_error("nifti_decode: %lld x %lld x %lld voxels per channel, over 2^31", (long long)dims[0], (long long)dims[1], (long long)dims[2]);
        return MVTB_EINVAL;
    }
    NiftiDev d;
    d.X = (int)dims[0]; d.Y = (int)dims[1]; d.Z = (int)dims[2]; d.C = dims[3];
    d.swap = swap_bytes != 0 && bytes > 1;
    d.scaled = scaled != 0;
    d.s32 = (float)slope; d.i32 = (float)inter; d.s64 = slope; d.i64 = inter;
    switch (datatype) {
        case MVTB_NIFTI_UINT8: nifti_launch<uint8_t>(raw, out, d, stream); break;
        case MVTB_NIFTI_INT8: nifti_launch<int8_t>(raw, out, d, stream); break;
        case MVTB_NIFTI_INT16: nifti_launch<int16_t>(raw, out, d, stream); break;
        case MVTB_NIFTI_UINT16: nifti_launch<uint16_t>(raw, out, d, stream); break;
        case MVTB_NIFTI_INT32: nifti_launch<int32_t>(raw, out, d, stream); break;
        case MVTB_NIFTI_UINT32: nifti_launch<uint32_t>(raw, out, d, stream); break;
        case MVTB_NIFTI_FLOAT32: nifti_launch<float>(raw, out, d, stream); break;
        default: nifti_launch<double>(raw, out, d, stream); break;
    }
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}
