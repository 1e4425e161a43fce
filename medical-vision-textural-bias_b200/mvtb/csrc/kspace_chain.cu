// kspace_chain.cu — general fused k-space chain:  out = Re ifftn( W * (M * fftn(x) + spikes) ).
//
// Replaces, in one forward + one inverse transform and with no fftshift copies, complex
// temporaries or materialised masks:
//   RandFourierDiskMaskd.__call__ (F:236-252)   GibbsNoise.__call__ (F:663-705)
//   GibbsNoiseLayer.forward (S:79-116)          RandPlaneWaves_ellipsoid.__call__ (F:370-393)
//   KSpaceSpikeNoise.__call__ (F:906-945)       WrapArtifact.__call__ (F:503-515)
// (F = source_code/filters_and_operators.py, S = source_code/stylization_layers.py.)
//
// Pipeline per chunk of volumes (half-spectrum workspace, last axis R2C by the
// "two real rows = one complex FFT" trick, valid for odd lengths such as 155):
//   k_rows_fwd            real rows -> half-spectrum rows (axis 0)
//   k_axis<FWD>           middle axes, in place, digit-reversed order kept
//   k_axis<MID>           outermost axis: forward, pointwise (mask / spike / wrap / 1/N), inverse
//   k_axis<INV>           middle axes back
//   k_rows_inv            half-spectrum rows -> real rows, fused per-sample min/max
// CTAs are 128 threads, 4-6 per SM; tiles arrive by cp.async; every per-pass constant comes from the plan (PassDev).
// Also here: k_wrap_fold_hw + k_rows_wrap, the wraparound for volumes with even H, W and an odd last axis.
#include <math.h>
#include <string.h>

#include <vector>

#include "fft_device.cuh"

namespace mvtb {

// bandlimited.cu
bool bl_eligible(const mvtb_plan* p, const mvtb_chain_desc* desc, int n_desc, int* F_out);
int bl_chain(mvtb_plan* p, const float* in, float* out, int n_volumes, const mvtb_chain_desc* desc, int n_desc,
             int F, float* minmax_out, int vols_per_sample, void* stream, void* sp_fuse, const float* pre_abt);

// spike_fast.cu
bool spike_fast_eligible(const mvtb_plan* p, const mvtb_chain_desc* desc, int n_desc);
int spike_fast_chain(mvtb_plan* p, const float* in, float* out, int n_volumes, const mvtb_chain_desc* desc, int n_desc,
                     float* minmax_out, int vols_per_sample, void* stream);

int plan_stage_upload(mvtb_plan* p, const void* src, size_t bytes, void* stream, void** dptr);   // plan.cu

enum { AX_FWD = 0, AX_INV = 1, AX_MID = 2, AX_STATS = 3 };
// Small CTAs, many per SM: a CTA is load -> barrier -> stages -> store with nothing overlapping inside it, so the
// loads in flight come from having 4-6 CTAs per SM in different phases (256 threads x 2 CTAs measured 2-3x slower).
static const int kThreads = 128;

struct ChainGeom {
    int ndim;
    int shape[MVTB_MAX_FFT_DIMS];         // axis 0 = last axis
    int nh;
    const int* pos2k[MVTB_MAX_FFT_DIMS];
    float scale;                          // 1 / prod(shape)
};

// ------------------------------------------------------------------ float atomics on (min,max)
__device__ __forceinline__ void atomic_min_f32(float* addr, float v) {
    v += 0.0f;   // -0 -> +0
    if (v >= 0.f) atomicMin((int*)addr, __float_as_int(v));
    else atomicMax((unsigned*)addr, __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f32(float* addr, float v) {
    v += 0.0f;
    if (v >= 0.f) atomicMax((int*)addr, __float_as_int(v));
    else atomicMin((unsigned*)addr, __float_as_uint(v));
}

__global__ void k_minmax_init(float* mm, int n_samples) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_samples) {
        mm[2 * i] = __int_as_float(0x7f800000);
        mm[2 * i + 1] = __int_as_float((int)0xff800000u);
    }
}

// block-wide (min,max) -> one atomic pair; every thread of the block must call it
__device__ __forceinline__ void block_minmax_commit(float lo, float hi, float* mm) {
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
        if (lane == 0) { atomic_min_f32(mm, lo); atomic_max_f32(mm + 1, hi); }
    }
}

// ------------------------------------------------------------------ axis 0: real rows <-> half spectrum
#define MVTB_MINB(MAXR) ((MAXR) <= 5 ? 6 : 4)

template <int MAXR>
__global__ void __launch_bounds__(128, MVTB_MINB(MAXR))
k_rows_fwd(const float* __restrict__ in, cf* __restrict__ ws, AxisDev ax, int nh, int pitch,
           int pairs_per_cta, long long n_rows) {
    MVTB_DYN_SMEM(smem_raw);
    cf* s = (cf*)smem_raw;
    const int n = ax.n, tid = threadIdx.x, nthr = blockDim.x;
    const long long n_pairs = (n_rows + 1) >> 1;
    const long long pair0 = (long long)blockIdx.x * pairs_per_cta;
    long long rem = n_pairs - pair0;
    const int np = rem < pairs_per_cta ? (int)rem : pairs_per_cta;

    // One warp per row pair, no divisions.  The rows go global -> shared as 4-byte asynchronous copies (row a into
    // the real parts, row b into the imaginary parts), all of them in flight at once.
    const int lane = tid & 31, wid = tid >> 5, nw = nthr >> 5;
    for (int rp = wid; rp < np; rp += nw) {
        const long long ra = 2 * (pair0 + rp);
        const float* pa = in + ra * n;
        const bool hasb = ra + 1 < n_rows;
        cf* sr = s + rp * pitch;
        for (int j = lane; j < n; j += 32) {
            cp_async<4>(&sr[j].x, pa + j);
            if (hasb) cp_async<4>(&sr[j].y, pa + n + j);
            else sr[j].y = 0.f;
        }
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    fft_forward<false, MAXR>(ax, s, pitch, 1, np, tid, nthr, ax.generic ? s + (size_t)pairs_per_cta * pitch : nullptr);

    // Z = FFT(a + i b):  A[k] = (Z[k] + conj Z[n-k]) / 2,  B[k] = (Z[k] - conj Z[n-k]) / (2i)
    // lanes own bins (positions looked up once), the warp walks its row pairs
    for (int k = lane; k < nh; k += 32) {
        const int pk = __ldg(ax.k2pos + k), pn = __ldg(ax.k2pos + (k == 0 ? 0 : n - k));
        for (int rp = wid; rp < np; rp += nw) {
            const long long ra = 2 * (pair0 + rp);
            const cf* sr = s + rp * pitch;
            const cf zk = sr[pk], zn = sr[pn];
            cf* wa = ws + ra * nh;
            wa[k] = cmk(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
            if (ra + 1 < n_rows) wa[nh + k] = cmk(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
        }
    }
}

template <int MAXR>
__global__ void __launch_bounds__(128, MVTB_MINB(MAXR))
k_rows_inv(const cf* __restrict__ ws, float* __restrict__ out, AxisDev ax, int nh, int pitch,
           int pairs_per_cta, long long n_rows, float* __restrict__ minmax, long long rows_per_sample,
           long long row_base) {
    MVTB_DYN_SMEM(smem_raw);
    cf* s = (cf*)smem_raw;
    const int n = ax.n, tid = threadIdx.x, nthr = blockDim.x;
    const long long n_pairs = (n_rows + 1) >> 1;
    const long long pair0 = (long long)blockIdx.x * pairs_per_cta;
    long long rem = n_pairs - pair0;
    const int np = rem < pairs_per_cta ? (int)rem : pairs_per_cta;

    // Z[k] = A[k] + i B[k];  Z[n-k] = conj A[k] + i conj B[k]
    const int lane = tid & 31, wid = tid >> 5, nw = nthr >> 5;
    constexpr int KMAX = 8;                      // bins per lane held in registers by the staged variant
    if (nh <= 32 * KMAX && 2 * nh <= pitch) {
        // Stage the two half-spectrum rows of every pair in the pair's own tile row (A at 0.., B at nh..) with
        // asynchronous copies, all in flight at once; then each warp combines its pairs in place: all of a pair's
        // bins are read into registers before any position is written.
        for (int rp = wid; rp < np; rp += nw) {
            const long long ra = 2 * (pair0 + rp);
            const cf* wa = ws + ra * nh;
            cf* sr = s + rp * pitch;
            const bool hasb = ra + 1 < n_rows;
            for (int k = lane; k < nh; k += 32) {
                cp_async<8>(sr + k, wa + k);
                if (hasb) cp_async<8>(sr + nh + k, wa + nh + k);
                else sr[nh + k] = cmk(0.f, 0.f);
            }
        }
        cp_async_commit();
        int pk[KMAX], pn[KMAX];
        MVTB_UNROLL
        for (int i = 0; i < KMAX; ++i) {
            const int k = lane + 32 * i;
            pk[i] = k < nh ? __ldg(ax.k2pos + k) : 0;
            pn[i] = (k < nh && k != 0 && 2 * k != n) ? __ldg(ax.k2pos + (n - k)) : -1;
        }
        cp_async_wait<0>();
        __syncwarp();                            // a pair is staged and combined by the same warp
        for (int rp = wid; rp < np; rp += nw) {
            cf* sr = s + rp * pitch;
            cf A[KMAX], B[KMAX];
            MVTB_UNROLL
            for (int i = 0; i < KMAX; ++i) {
                const int k = lane + 32 * i;
                if (k < nh) { A[i] = sr[k]; B[i] = sr[nh + k]; }
            }
            __syncwarp();
            MVTB_UNROLL
            for (int i = 0; i < KMAX; ++i) {
                const int k = lane + 32 * i;
                if (k < nh) {
                    sr[pk[i]] = cmk(A[i].x - B[i].y, A[i].y + B[i].x);
                    if (pn[i] >= 0) sr[pn[i]] = cmk(A[i].x + B[i].y, B[i].x - A[i].y);
                }
            }
        }
    } else {
        for (int k = lane; k < nh; k += 32) {
            const int pk = __ldg(ax.k2pos + k);
            const bool mirror = k != 0 && 2 * k != n;
            const int pn = mirror ? __ldg(ax.k2pos + (n - k)) : 0;
            MVTB_UNROLL_N(4)
            for (int rp = wid; rp < np; rp += nw) {
                const long long ra = 2 * (pair0 + rp);
                const cf* wa = ws + ra * nh;
                const cf A = wa[k];
                const cf B = (ra + 1 < n_rows) ? wa[nh + k] : cmk(0.f, 0.f);
                cf* sr = s + rp * pitch;
                sr[pk] = cmk(A.x - B.y, A.y + B.x);
                if (mirror) sr[pn] = cmk(A.x + B.y, B.x - A.y);
            }
        }
    }
    __syncthreads();
    fft_inverse<false, MAXR>(ax, s, pitch, 1, np, tid, nthr, ax.generic ? s + (size_t)pairs_per_cta * pitch : nullptr);

    float lo = __int_as_float(0x7f800000), hi = __int_as_float((int)0xff800000u);
    const long long row_first = 2 * pair0;
    long long row_last = row_first + 2 * np - 1;
    if (row_last >= n_rows) row_last = n_rows - 1;
    const bool want_mm = minmax != nullptr;
    const bool uniform = want_mm && ((row_base + row_first) / rows_per_sample == (row_base + row_last) / rows_per_sample);
    for (int rp = wid; rp < np; rp += nw) {
        const long long ra = 2 * (pair0 + rp);
        const bool hasb = ra + 1 < n_rows;
        const cf* sr = s + rp * pitch;
        float* pa = out + ra * n;
        float* ma = nullptr;
        float* mb = nullptr;
        if (want_mm && !uniform) {
            ma = minmax + 2 * ((row_base + ra) / rows_per_sample);
            mb = minmax + 2 * ((row_base + ra + 1) / rows_per_sample);
        }
        for (int j = lane; j < n; j += 32) {
            const cf z = sr[j];
            pa[j] = z.x;
            if (hasb) pa[n + j] = z.y;
            if (want_mm) {
                if (uniform) {
                    lo = fminf(lo, z.x); hi = fmaxf(hi, z.x);
                    if (hasb) { lo = fminf(lo, z.y); hi = fmaxf(hi, z.y); }
                } else {
                    atomic_min_f32(ma, z.x); atomic_max_f32(ma + 1, z.x);
                    if (hasb) { atomic_min_f32(mb, z.y); atomic_max_f32(mb + 1, z.y); }
                }
            }
        }
    }
    if (uniform) block_minmax_commit(lo, hi, minmax + 2 * ((row_base + row_first) / rows_per_sample));
}

// ------------------------------------------------------------------ wraparound with an odd last axis (240 x 240 x 155)
// WrapArtifact (F:503-515) weights the odd fftshift-ed k-space samples of every axis by alpha.  Along an even axis
// that is an image-domain fold (SURVEY A.3); along an odd axis there is no half shift, but the weight depends on
// that axis' frequency alone, so it is a 1-D filter of every row: two real rows = one complex FFT, and because the
// weight is symmetric under f -> -f it applies to the packed spectrum directly -- forward, weight, inverse in one
// kernel, no unpacking.  k_wrap_fold_hw folds H and W first (the two commute).
template <int MAXR>
__global__ void __launch_bounds__(128, MVTB_MINB(MAXR))
k_rows_wrap(const float* in, float* out, AxisDev ax, int pitch, int pairs_per_cta,
            long long n_rows, float alpha) {
    MVTB_DYN_SMEM(smem_raw);
    cf* s = (cf*)smem_raw;
    const int n = ax.n, tid = threadIdx.x, nthr = blockDim.x;
    const long long n_pairs = (n_rows + 1) >> 1;
    const long long pair0 = (long long)blockIdx.x * pairs_per_cta;
    long long rem = n_pairs - pair0;
    const int np = rem < pairs_per_cta ? (int)rem : pairs_per_cta;
    const int lane = tid & 31, wid = tid >> 5, nw = nthr >> 5;
    for (int rp = wid; rp < np; rp += nw) {
        const long long ra = 2 * (pair0 + rp);
        const float* pa = in + ra * n;
        const bool hasb = ra + 1 < n_rows;
        cf* sr = s + rp * pitch;
        for (int j = lane; j < n; j += 32) {
            cp_async<4>(&sr[j].x, pa + j);
            if (hasb) cp_async<4>(&sr[j].y, pa + n + j);
            else sr[j].y = 0.f;
        }
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    cf* scratch = ax.generic ? s + (size_t)pairs_per_cta * pitch : nullptr;
    fft_forward<false, MAXR>(ax, s, pitch, 1, np, tid, nthr, scratch);
    const float inv_n = 1.f / (float)n;
    for (int j = lane; j < n; j += 32) {
        const int i = (__ldg(ax.pos2k + j) + n / 2) % n;             // fftshift-ed index of the bin at position j
        const float wgt = (i & 1) ? alpha * inv_n : inv_n;
        for (int rp = wid; rp < np; rp += nw) {
            cf* e = s + rp * pitch + j;
            *e = cscale(*e, wgt);
        }
    }
    __syncthreads();
    fft_inverse<false, MAXR>(ax, s, pitch, 1, np, tid, nthr, scratch);
    for (int rp = wid; rp < np; rp += nw) {
        const long long ra = 2 * (pair0 + rp);
        const bool hasb = ra + 1 < n_rows;
        const cf* sr = s + rp * pitch;
        float* pa = out + ra * n;
        for (int j = lane; j < n; j += 32) {
            const cf z = sr[j];
            pa[j] = z.x;
            if (hasb) pa[n + j] = z.y;
        }
    }
}

// H and W folds of one orbit {h, h+H/2} x {w, w+W/2} at every d: 4 reads, 4 writes, d contiguous across threads
__global__ void __launch_bounds__(256)
k_wrap_fold_hw(const float* __restrict__ in, float* __restrict__ out, int H, int W, int D, float c0, float ch, float cw,
               size_t n_total) {
    const int H2 = H / 2, W2 = W / 2;
    const size_t per_vol = (size_t)H2 * W2 * D, vol_elems = (size_t)H * W * D;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n_total; t += (size_t)gridDim.x * blockDim.x) {
        const size_t v = t / per_vol;
        size_t r = t - v * per_vol;
        const int d = (int)(r % D); r /= D;
        const int w = (int)(r % W2);
        const int h = (int)(r / W2);
        const float* x = in + v * vol_elems;
        float* y = out + v * vol_elems;
        const size_t o00 = ((size_t)h * W + w) * D + d, o01 = o00 + (size_t)W2 * D;
        const size_t o10 = o00 + (size_t)H2 * W * D, o11 = o10 + (size_t)W2 * D;
        const float a00 = x[o00], a01 = x[o01], a10 = x[o10], a11 = x[o11];
        const float b00 = c0 * a00 + cw * a01, b01 = c0 * a01 + cw * a00;     // W axis
        const float b10 = c0 * a10 + cw * a11, b11 = c0 * a11 + cw * a10;
        y[o00] = c0 * b00 + ch * b10; y[o10] = c0 * b10 + ch * b00;           // H axis
        y[o01] = c0 * b01 + ch * b11; y[o11] = c0 * b11 + ch * b01;
    }
}

// ------------------------------------------------------------------ pointwise k-space stage
__device__ __forceinline__ long long mask_term(int kind, int i, int n) {
    if (kind == MVTB_MASK_UNIFORM) return 0;
    const long long d = kind == MVTB_MASK_DISK ? (long long)(i - n / 2) : (long long)(2 * i - (n - 1));
    return d * d;
}

__device__ __forceinline__ cf spike_value(cf ko, float amp) {
    const float mag = hypotf(ko.x, ko.y);
    if (mag > 0.f) return cmk(amp * (ko.x / mag), amp * (ko.y / mag));
    return cmk(amp, 0.f);   // angle(0) = 0 (F:384, F:928)
}

// Axes >= 1 of the half-spectrum workspace, viewed as [outer][n][inner].
// One CTA owns a tile of T adjacent `inner` columns over the whole axis: shared memory [n][T].
template <int MODE, int MAXR>
__global__ void __launch_bounds__(128, MVTB_MINB(MAXR))
k_axis(cf* __restrict__ ws, AxisDev ax, int axis, long long inner, int T, int ntiles,
       ChainGeom g, const DescDev* __restrict__ dv, int dshared, double* __restrict__ sums) {
    MVTB_DYN_SMEM(smem_raw);
    cf* s = (cf*)smem_raw;
    const int n = ax.n, tid = threadIdx.x, nthr = blockDim.x;
    const long long o = blockIdx.x / ntiles;
    const long long i0 = (long long)(blockIdx.x - o * ntiles) * T;
    cf* base = ws + o * (long long)n * inner + i0;
    int lgT = 0;                           // T is a power of two and nthr % T == 0: a thread always sees the same column
    while ((1 << lgT) < T) ++lgT;
    const int t = tid & (T - 1);
    const bool col_ok = i0 + t < inner;
    const long long gstep = (long long)(nthr >> lgT) * inner;

    // ---- pointwise stage, what depends only on the column (registers), computed before anything is loaded: a tile
    // whose columns the mask removes entirely (all bins of the column and of its mirror lie outside the ball, no
    // spike on it) is zero whatever the data, so it is neither loaded nor transformed -- 40 % of the tiles for
    // GibbsNoise(0.5) on 240 x 240 x 155, 85 % for a disk of radius 40.
    long long qp = 0, qn = 0;
    long long up_off = 0, un_off = 0;      // MVTB_MASK_UNIFORM: offset of the column (and of its mirror) in the uniform field
    long long u_stride = 1;                // ... and the stride of this axis there
    float wgt = g.scale;
    unsigned mpos = 0, mneg = 0;           // per-spike "all lower axes match" bits
    if (MODE == AX_MID) {
        const DescDev& d = dv[dshared ? 0 : (int)o];
        int ish[MVTB_MAX_FFT_DIMS], ineg[MVTB_MAX_FFT_DIMS];
        long long rest = i0 + t;
        {
            const int k0 = (int)(rest % g.nh);
            rest /= g.nh;
            ish[0] = (k0 + g.shape[0] / 2) % g.shape[0];
        }
        for (int b = 1; b < axis; ++b) {
            const int pb = (int)(rest % g.shape[b]);
            rest /= g.shape[b];
            ish[b] = (__ldg(g.pos2k[b] + pb) + g.shape[b] / 2) % g.shape[b];
        }
        for (int b = 0; b < axis; ++b) {
            const int nb = g.shape[b];
            ineg[b] = (2 * (nb / 2) - ish[b] + nb) % nb;
            if (d.mask_kind != MVTB_MASK_NONE && b < d.mask_ndim) {
                qp += mask_term(d.mask_kind, ish[b], nb);
                qn += mask_term(d.mask_kind, ineg[b], nb);
            }
            if (b < d.wrap_naxes && (ish[b] & 1)) wgt *= d.wrap_alpha;
            up_off += (long long)ish[b] * u_stride;
            un_off += (long long)ineg[b] * u_stride;
            u_stride *= nb;
        }
        for (int sI = 0; sI < d.n_spikes; ++sI) {
            bool pm = true, qm = true;
            for (int b = 0; b < axis; ++b) {
                pm = pm && (ish[b] == d.sp[sI].idx[b]);
                qm = qm && (ineg[b] == d.sp[sI].idx[b]);
            }
            mpos |= (pm ? 1u : 0u) << sI;
            mneg |= (qm ? 1u : 0u) << sI;
        }
        bool col_dead = !col_ok;
        if (col_ok && d.mask_kind != MVTB_MASK_NONE && d.mask_kind != MVTB_MASK_UNIFORM && !d.inside_off && (mpos | mneg) == 0u) {
            // smallest term this axis can add: 0, or 1 for a centred mask on an even axis ((2i - (n-1))^2 is odd)
            const long long tmin = (axis < d.mask_ndim && d.mask_kind != MVTB_MASK_DISK && !(n & 1)) ? 1 : 0;
            col_dead = qp + tmin > d.thr && qn + tmin > d.thr;
        }
        __shared__ int s_alive;
        if (tid == 0) s_alive = 0;
        __syncthreads();
        if (!col_dead) s_alive = 1;
        __syncthreads();
        if (!s_alive) {
            if (col_ok) {
                cf* gz = base + (long long)(tid >> lgT) * inner + t;
                for (int e = tid; e < n * T; e += nthr, gz += gstep) *gz = cmk(0.f, 0.f);
            }
            return;
        }
    }

    {   // the whole tile in flight at once: 8-byte asynchronous copies, no registers held
        const cf* gp = base + (long long)(tid >> lgT) * inner + t;
        if (col_ok) {
            for (int e = tid; e < n * T; e += nthr, gp += gstep) cp_async<8>(s + e, gp);
        } else {
            for (int e = tid; e < n * T; e += nthr) s[e] = cmk(0.f, 0.f);
        }
        cp_async_commit();
    }

    cf* scratch = ax.generic ? s + (size_t)n * T : nullptr;

    // ---- pointwise stage, part 1 (while the tile is still in flight): what depends only on the bin along this
    // axis goes into a shared table, what depends only on the column into registers.
    int4* tab = nullptr;                   // per position j: (shifted index, mask term at +f, mask term at -f, odd)
    if (MODE == AX_MID) {
        const DescDev& d = dv[dshared ? 0 : (int)o];
        tab = (int4*)(smem_raw + (((size_t)n * T * sizeof(cf) * (ax.generic ? 2 : 1)) + 15) / 16 * 16);
        const bool masked = d.mask_kind != MVTB_MASK_NONE && axis < d.mask_ndim;
        for (int j = tid; j < n; j += nthr) {
            const int im = (__ldg(ax.pos2k + j) + n / 2) % n;
            const int imn = (2 * (n / 2) - im + n) % n;
            int4 e;
            e.x = im;
            e.y = masked ? (int)mask_term(d.mask_kind, im, n) : 0;      // < (2n)^2 <= 2^30 for any tile that fits
            e.z = masked ? (int)mask_term(d.mask_kind, imn, n) : 0;
            e.w = (axis < d.wrap_naxes && (im & 1)) ? 1 : 0;
            tab[j] = e;
        }
    }
    cp_async_wait<0>();
    __syncthreads();

    if (MODE != AX_INV) fft_forward<true, MAXR>(ax, s, 1, T, T, tid, nthr, scratch);

    if (MODE == AX_MID) {
        const DescDev& d = dv[dshared ? 0 : (int)o];
        // ---- part 2: per bin
        if (col_ok) {
            const bool any_mask = d.mask_kind != MVTB_MASK_NONE;
            const float wodd = wgt * d.wrap_alpha;
            for (int j = tid >> lgT; j < n; j += nthr >> lgT) {
                const int4 e = tab[j];
                float meff = 1.f;
                if (d.mask_kind == MVTB_MASK_UNIFORM) {              // RandZF: keep <=> u > p at the bin, at its mirror
                    const int imn_ = (2 * (n / 2) - e.x + n) % n;
                    const int kp = (__ldg(d.mask_u + up_off + (long long)e.x * u_stride) > d.mask_p ? 1 : 0) ^ d.inside_off;
                    const int kn = (__ldg(d.mask_u + un_off + (long long)imn_ * u_stride) > d.mask_p ? 1 : 0) ^ d.inside_off;
                    meff = 0.5f * (float)(kp + kn);
                } else if (any_mask) {
                    const int kp = (qp + e.y <= d.thr ? 1 : 0) ^ d.inside_off;
                    const int kn = (qn + e.z <= d.thr ? 1 : 0) ^ d.inside_off;
                    meff = 0.5f * (float)(kp + kn);
                }
                const cf K = s[j * T + t];
                cf acc = cscale(K, meff);
                if ((mpos | mneg) != 0u) {
                    const int im = e.x, imn = (2 * (n / 2) - im + n) % n;
                    for (int sI = 0; sI < d.n_spikes; ++sI) {
                        const bool isp = ((mpos >> sI) & 1u) && im == d.sp[sI].idx[axis];
                        const bool isn = ((mneg >> sI) & 1u) && imn == d.sp[sI].idx[axis];
                        if (!isp && !isn) continue;
                        const float ms = d.sp[sI].meff_at_spike;
                        if (isp && isn) {                 // self-conjugate bin: Re(new)
                            const cf ko = cscale(K, ms);
                            const cf nw = spike_value(ko, d.sp[sI].amp);
                            acc.x += nw.x - ko.x;
                            acc.y -= ko.y;
                        } else if (isp) {
                            const cf ko = cscale(K, ms);
                            const cf nw = spike_value(ko, d.sp[sI].amp);
                            acc.x += 0.5f * (nw.x - ko.x);
                            acc.y += 0.5f * (nw.y - ko.y);
                        } else {                          // this bin is -f_s: K(f_s) = conj K here
                            const cf ko = cscale(cconj(K), ms);
                            const cf nw = spike_value(ko, d.sp[sI].amp);
                            acc.x += 0.5f * (nw.x - ko.x);
                            acc.y -= 0.5f * (nw.y - ko.y);
                        }
                    }
                }
                s[j * T + t] = cscale(acc, e.w ? wodd : wgt);
            }
        }
        __syncthreads();
    }

    if (MODE == AX_STATS) {
        double acc = 0.0;
        if (col_ok) {
            const int k0 = (int)((i0 + t) % g.nh);
            const bool self = k0 == 0 || (2 * k0 == g.shape[0]);
            const double wt = self ? 1.0 : 2.0;
            for (int j = tid >> lgT; j < n; j += nthr >> lgT) {
                const cf K = s[j * T + t];
                acc += wt * (double)logf(hypotf(K.x, K.y) + 1e-10f);
            }
        }
        __shared__ double s_acc[32];
        MVTB_UNROLL
        for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
        if ((tid & 31) == 0) s_acc[tid >> 5] = acc;
        __syncthreads();
        if (tid == 0) {
            double tot = 0.0;
            for (int w = 0; w < (nthr + 31) / 32; ++w) tot += s_acc[w];
            atomicAdd(sums + o, tot);
        }
        return;
    }

    if (MODE != AX_FWD) fft_inverse<true, MAXR>(ax, s, 1, T, T, tid, nthr, scratch);

    if (col_ok) {
        cf* gp = base + (long long)(tid >> lgT) * inner + t;
        MVTB_UNROLL_N(4)
        for (int e = tid; e < n * T; e += nthr, gp += gstep) *gp = s[e];
    }
}

// ------------------------------------------------------------------ host side
#ifndef MVTB_EMU
template <typename K>
static int allow_big_smem(K kern, int optin) {
    cudaFuncAttributes a;
    MVTB_CUDA(cudaFuncGetAttributes(&a, kern));
    MVTB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)a.sharedSizeBytes));
    return MVTB_OK;
}
#endif

template <int MAXR>
static int configure_maxr(int optin) {
#ifndef MVTB_EMU
    int rc;
    if ((rc = allow_big_smem(k_rows_fwd<MAXR>, optin)) != MVTB_OK) return rc;
    if ((rc = allow_big_smem(k_rows_inv<MAXR>, optin)) != MVTB_OK) return rc;
    if ((rc = allow_big_smem(k_rows_wrap<MAXR>, optin)) != MVTB_OK) return rc;
    if ((rc = allow_big_smem(k_axis<AX_FWD, MAXR>, optin)) != MVTB_OK) return rc;
    if ((rc = allow_big_smem(k_axis<AX_INV, MAXR>, optin)) != MVTB_OK) return rc;
    if ((rc = allow_big_smem(k_axis<AX_MID, MAXR>, optin)) != MVTB_OK) return rc;
    if ((rc = allow_big_smem(k_axis<AX_STATS, MAXR>, optin)) != MVTB_OK) return rc;
#endif
    (void)optin;
    return MVTB_OK;
}

int configure_chain_kernels(const mvtb_plan* p) {
    int optin = 0;
#ifndef MVTB_EMU
    cudaDeviceProp prop;
    MVTB_CUDA(cudaGetDeviceProperties(&prop, p->device));
    optin = (int)prop.sharedMemPerBlockOptin;
#endif
    (void)p;
    int rc;
    if ((rc = configure_maxr<5>(optin)) != MVTB_OK) return rc;
    if ((rc = configure_maxr<13>(optin)) != MVTB_OK) return rc;
    if ((rc = configure_maxr<31>(optin)) != MVTB_OK) return rc;
    return MVTB_OK;
}

// radix class of an axis: which kernel instantiation can run it
static int axis_maxr(const mvtb_plan* p, int a) {
    int m = 2;
    for (int s = 0; s < p->ax[a].nstage; ++s) m = p->ax[a].radix[s] > m ? p->ax[a].radix[s] : m;
    return m <= 5 ? 5 : (m <= 13 ? 13 : 31);
}

static ChainGeom make_geom(const mvtb_plan* p) {
    ChainGeom g;
    memset(&g, 0, sizeof(g));
    g.ndim = p->ndim;
    g.nh = p->nh;
    double tot = 1.0;
    for (int a = 0; a < p->ndim; ++a) {
        g.shape[a] = p->shape[a];
        g.pos2k[a] = p->ax[a].pos2k;
        tot *= (double)p->shape[a];
    }
    g.scale = (float)(1.0 / tot);
    return g;
}

static bool same_desc(const mvtb_chain_desc& a, const mvtb_chain_desc& b) {
    if (a.mask_kind == MVTB_MASK_UNIFORM || b.mask_kind == MVTB_MASK_UNIFORM) return false;    // every volume has its own field
    if (a.mask_kind != b.mask_kind || a.mask_ndim != b.mask_ndim || a.mask_thresh != b.mask_thresh || a.inside_off != b.inside_off ||
        a.n_spikes != b.n_spikes || a.wrap_naxes != b.wrap_naxes || memcmp(&a.wrap_alpha, &b.wrap_alpha, sizeof(float)) != 0) return false;
    if (a.n_spikes < 0 || a.n_spikes > MVTB_MAX_SPIKES) return false;
    for (int s = 0; s < a.n_spikes; ++s)
        if (memcmp(a.spikes[s].idx, b.spikes[s].idx, sizeof(a.spikes[s].idx)) != 0 ||
            memcmp(&a.spikes[s].amplitude, &b.spikes[s].amplitude, sizeof(float)) != 0) return false;
    return true;
}

// validates one user descriptor against the plan and converts it to the device view
int convert_desc(const mvtb_plan* p, const mvtb_chain_desc* u, DescDev* d) {
    memset(d, 0, sizeof(*d));
    if (u->mask_kind < MVTB_MASK_NONE || u->mask_kind > MVTB_MASK_UNIFORM) { set_error("chain: mask_kind=%d", u->mask_kind); return MVTB_EINVAL; }
    if (u->mask_kind == MVTB_MASK_UNIFORM && !u->mask_u) { set_error("chain: MVTB_MASK_UNIFORM needs mask_u"); return MVTB_EINVAL; }
    if (u->mask_kind == MVTB_MASK_UNIFORM && u->n_spikes > 0) { set_error("chain: spikes cannot be combined with MVTB_MASK_UNIFORM"); return MVTB_EUNSUPPORTED; }
    if (u->mask_kind == MVTB_MASK_UNIFORM && p->lead_drop > 0) { set_error("chain: MVTB_MASK_UNIFORM with leading axes of length 1 is not built"); return MVTB_EUNSUPPORTED; }
    if (u->mask_kind != MVTB_MASK_NONE && u->mask_kind != MVTB_MASK_UNIFORM && (u->mask_ndim < 1 || u->mask_ndim > p->ndim)) { set_error("chain: mask_ndim=%d with ndim_fft=%d", u->mask_ndim, p->ndim); return MVTB_EINVAL; }
    if (u->n_spikes < 0 || u->n_spikes > MVTB_MAX_SPIKES) { set_error("chain: n_spikes=%d (max %d)", u->n_spikes, MVTB_MAX_SPIKES); return MVTB_EUNSUPPORTED; }
    if (u->wrap_naxes < 0 || u->wrap_naxes > p->ndim) { set_error("chain: wrap_naxes=%d", u->wrap_naxes); return MVTB_EINVAL; }
    d->mask_kind = u->mask_kind;
    d->mask_ndim = u->mask_kind == MVTB_MASK_NONE ? 0 : (u->mask_kind == MVTB_MASK_UNIFORM ? p->ndim : u->mask_ndim);
    d->mask_u = u->mask_kind == MVTB_MASK_UNIFORM ? u->mask_u : nullptr;
    d->mask_p = u->mask_p;
    d->thr = u->mask_thresh;
    d->inside_off = u->inside_off ? 1 : 0;
    d->n_spikes = u->n_spikes;
    d->wrap_alpha = u->wrap_alpha;
    d->wrap_naxes = u->wrap_naxes;
    for (int s = 0; s < u->n_spikes; ++s) {
        long long q = 0, qneg = 0;                                 // mask distance of the bin and of its mirror -f_s
        for (int a = 0; a < p->ndim; ++a) {
            const int idx = u->spikes[s].idx[p->ndim - 1 - a];     // user order: outermost first
            const int n = p->shape[a];
            if (idx < 0 || idx >= n) { set_error("chain: spike %d index %d out of bounds for axis of length %d", s, idx, n); return MVTB_EINVAL; }
            d->sp[s].idx[a] = idx;
            if (a < d->mask_ndim) {
                const int ineg = (2 * (n / 2) - idx + n) % n;
                const long long dd = d->mask_kind == MVTB_MASK_DISK ? (long long)(idx - n / 2) : (long long)(2 * idx - (n - 1));
                const long long dn = d->mask_kind == MVTB_MASK_DISK ? (long long)(ineg - n / 2) : (long long)(2 * ineg - (n - 1));
                q += dd * dd;
                qneg += dn * dn;
            }
        }
        d->sp[s].amp = u->spikes[s].amplitude;
        // The mask stage returns a REAL image, whose spectrum at f_s is M_eff(f_s) K (SURVEY A.2); that is the bin the
        // spike stage reads.  A centred mask on an even axis has M(f) != M(-f) on its boundary shell.
        if (d->mask_kind == MVTB_MASK_NONE) d->sp[s].meff_at_spike = 1.f;
        else d->sp[s].meff_at_spike = 0.5f * (float)((((q <= d->thr) ? 1 : 0) ^ d->inside_off) + (((qneg <= d->thr) ? 1 : 0) ^ d->inside_off));
        for (int s2 = 0; s2 < s; ++s2) {
            bool same = true;
            for (int a = 0; a < p->ndim; ++a) same = same && d->sp[s2].idx[a] == d->sp[s].idx[a];
            if (same) { set_error("chain: spikes %d and %d share a location (deduplicate on the host: the last one wins, F:937-938)", s2, s); return MVTB_EINVAL; }
        }
    }
    return MVTB_OK;
}

static int launch_rows_fwd(mvtb_plan* p, const float* in, cf* ws, long long n_rows, void* stream) {
    ProfScope prof(p, MVTB_K_ROWS_FWD, stream);
    const long long n_pairs = (n_rows + 1) / 2;
    const int rp = p->rows_pairs_per_cta;
    const unsigned grid = (unsigned)((n_pairs + rp - 1) / rp);
    const size_t smem = (size_t)rp * p->row_pitch * sizeof(cf) * (p->ax[0].generic ? 2 : 1);
    switch (axis_maxr(p, 0)) {
        case 5: { auto kern = k_rows_fwd<5>; MVTB_LAUNCH(kern, dim3(grid), dim3(kThreads), smem, stream, in, ws, p->ax[0], p->nh, p->row_pitch, rp, n_rows); break; }
        case 13: { auto kern = k_rows_fwd<13>; MVTB_LAUNCH(kern, dim3(grid), dim3(kThreads), smem, stream, in, ws, p->ax[0], p->nh, p->row_pitch, rp, n_rows); break; }
        default: { auto kern = k_rows_fwd<31>; MVTB_LAUNCH(kern, dim3(grid), dim3(kThreads), smem, stream, in, ws, p->ax[0], p->nh, p->row_pitch, rp, n_rows); break; }
    }
    return MVTB_OK;
}

template <int MODE>
static int launch_axis(mvtb_plan* p, cf* ws, int axis, int n_outer_vols, const ChainGeom& g,
                       const DescDev* dv, int dshared, double* sums, void* stream) {
    ProfScope prof(p, MODE == AX_FWD ? MVTB_K_AXIS_FWD : (MODE == AX_INV ? MVTB_K_AXIS_INV : MVTB_K_AXIS_MID), stream);
    long long inner = p->nh;
    for (int b = 1; b < axis; ++b) inner *= p->shape[b];
    long long outer = n_outer_vols;
    for (int b = axis + 1; b < p->ndim; ++b) outer *= p->shape[b];
    const int T = p->axis_tile;
    const long long ntiles = (inner + T - 1) / T;
    const long long blocks = ntiles * outer;
    if (blocks > 0x7fffffffLL) { set_error("chain: grid too large"); return MVTB_EUNSUPPORTED; }
    size_t smem = (size_t)p->shape[axis] * T * sizeof(cf) * (p->ax[axis].generic ? 2 : 1);
    if (MODE == AX_MID) smem = (smem + 15) / 16 * 16 + (size_t)p->shape[axis] * sizeof(int4);   // per-bin table of the pointwise stage
    switch (axis_maxr(p, axis)) {
        case 5: { auto kern = k_axis<MODE, 5>; MVTB_LAUNCH(kern, dim3((unsigned)blocks), dim3(kThreads), smem, stream, ws, p->ax[axis], axis, inner, T, (int)ntiles, g, dv, dshared, sums); break; }
        case 13: { auto kern = k_axis<MODE, 13>; MVTB_LAUNCH(kern, dim3((unsigned)blocks), dim3(kThreads), smem, stream, ws, p->ax[axis], axis, inner, T, (int)ntiles, g, dv, dshared, sums); break; }
        default: { auto kern = k_axis<MODE, 31>; MVTB_LAUNCH(kern, dim3((unsigned)blocks), dim3(kThreads), smem, stream, ws, p->ax[axis], axis, inner, T, (int)ntiles, g, dv, dshared, sums); break; }
    }
    return MVTB_OK;
}

}  // namespace mvtb

using namespace mvtb;

// sp_fuse: null, or bandlimited.cu's SpFuse (the band-limited path may then run the select pass inside its inverse kernel)
// pre_abt: null, or the intensity prologue map per volume (applied on load by the band-limited path, else by its own pass)
static int chain_impl(mvtb_plan* p, const float* in, float* out, int n_volumes,
                      const mvtb_chain_desc* desc, int n_desc,
                      float* minmax_out, int vols_per_sample, void* stream, void* sp_fuse, const float* pre_abt) {
    if (!p || !in || !out || !desc) { set_error("chain: null argument"); return MVTB_EINVAL; }
    if (n_volumes < 0) { set_error("chain: n_volumes=%d", n_volumes); return MVTB_EINVAL; }
    if (n_desc != 1 && n_desc != n_volumes) { set_error("chain: n_desc=%d must be 1 or n_volumes=%d", n_desc, n_volumes); return MVTB_EINVAL; }
    if (minmax_out && vols_per_sample < 1) { set_error("chain: vols_per_sample=%d", vols_per_sample); return MVTB_EINVAL; }
    if (n_volumes == 0) return MVTB_OK;
    MVTB_CUDA(cudaSetDevice(p->device));

    std::vector<mvtb_chain_desc> shifted;
    if (p->lead_drop > 0) {                                // the plan dropped leading length-1 axes: shift the descriptors
        shifted.assign(desc, desc + n_desc);
        for (int i = 0; i < n_desc; ++i) {
            mvtb_chain_desc& d = shifted[i];
            if (d.mask_ndim > p->ndim) d.mask_ndim = p->ndim;
            if (d.wrap_naxes > p->ndim) d.wrap_naxes = p->ndim;
            for (int s = 0; s < d.n_spikes && s < MVTB_MAX_SPIKES; ++s) {
                for (int a = 0; a < p->lead_drop; ++a)
                    if (d.spikes[s].idx[a] != 0) { set_error("chain: spike %d index %d out of bounds for an axis of length 1", s, d.spikes[s].idx[a]); return MVTB_EINVAL; }
                for (int a = 0; a < p->ndim; ++a) d.spikes[s].idx[a] = d.spikes[s].idx[a + p->lead_drop];
            }
        }
        desc = shifted.data();
    }

    // identical per-volume descriptors (one spike location for a whole slice stack, F:982-983) are one descriptor
    if (n_desc > 1) {
        bool same = true;
        for (int v = 1; v < n_desc && same; ++v) same = same_desc(desc[0], desc[v]);
        if (same) n_desc = 1;
    }
    const ChainGeom g = make_geom(p);
    std::vector<DescDev> hdesc((size_t)n_desc);
    for (int v = 0; v < n_desc; ++v) {                 // validate everything before launching anything
        int rc = convert_desc(p, desc + v, &hdesc[v]);
        if (rc != MVTB_OK) return rc;
    }
    long long rows_per_vol = 1;
    for (int a = 1; a < p->ndim; ++a) rows_per_vol *= p->shape[a];

    if (minmax_out) {
        const int n_samples = (n_volumes + vols_per_sample - 1) / vols_per_sample;
        MVTB_LAUNCH(k_minmax_init, dim3((n_samples + 127) / 128), dim3(128), 0, stream, minmax_out, n_samples);
    }

    int blF = 0;
    const bool spike_fast = spike_fast_eligible(p, desc, n_desc);
    const bool bl = !spike_fast && bl_eligible(p, desc, n_desc, &blF);
    if (pre_abt && !bl) {                              // the other paths read a prepared volume: map it into `out` first
        int rc = mvtb_intensity_affine_f32(in, out, p->vol_real, n_volumes, pre_abt, stream);
        if (rc != MVTB_OK) return rc;
        in = out;
    }
    if (spike_fast)
        return spike_fast_chain(p, in, out, n_volumes, desc, n_desc, minmax_out, vols_per_sample, stream);
    if (bl)
        return bl_chain(p, in, out, n_volumes, desc, n_desc, blF, minmax_out, vols_per_sample, stream, sp_fuse, pre_abt);

    const DescDev* ddesc = nullptr;                    // device copy of the converted descriptors, valid on `stream`
    {
        void* dvp = nullptr;
        int rc = plan_stage_upload(p, hdesc.data(), hdesc.size() * sizeof(DescDev), stream, &dvp);
        if (rc != MVTB_OK) return rc;
        ddesc = (const DescDev*)dvp;
    }
    const int mid = p->ndim - 1;
    for (int v0 = 0; v0 < n_volumes; v0 += p->chunk) {
        const int nv = (n_volumes - v0 < p->chunk) ? (n_volumes - v0) : p->chunk;
        const long long n_rows = rows_per_vol * nv;
        int rc = launch_rows_fwd(p, in + (size_t)v0 * p->vol_real, p->ws, n_rows, stream);
        if (rc != MVTB_OK) return rc;
        for (int a = 1; a < mid; ++a) {
            rc = launch_axis<AX_FWD>(p, p->ws, a, nv, g, nullptr, 1, nullptr, stream);
            if (rc != MVTB_OK) return rc;
        }
        rc = launch_axis<AX_MID>(p, p->ws, mid, nv, g, ddesc + (n_desc == 1 ? 0 : v0), n_desc == 1 ? 1 : 0, nullptr, stream);
        if (rc != MVTB_OK) return rc;
        for (int a = mid - 1; a >= 1; --a) {
            rc = launch_axis<AX_INV>(p, p->ws, a, nv, g, nullptr, 1, nullptr, stream);
            if (rc != MVTB_OK) return rc;
        }
        {
            const long long n_pairs = (n_rows + 1) / 2;
            const int rp = p->rows_pairs_per_cta;
            const unsigned grid = (unsigned)((n_pairs + rp - 1) / rp);
            const size_t smem = (size_t)rp * p->row_pitch * sizeof(cf) * (p->ax[0].generic ? 2 : 1);
            const long long rows_per_sample = rows_per_vol * (minmax_out ? vols_per_sample : 1);
            // chunks need not align with samples: the kernel works from the global row number
            ProfScope prof(p, MVTB_K_ROWS_INV, stream);
#define MVTB_ROWS_INV(MAXR)                                                                                   \
            do {                                                                                              \
                auto kern = k_rows_inv<MAXR>;                                                                 \
                MVTB_LAUNCH(kern, dim3(grid), dim3(kThreads), smem, stream, (const cf*)p->ws,                 \
                            out + (size_t)v0 * p->vol_real, p->ax[0], p->nh, p->row_pitch, rp, n_rows,        \
                            minmax_out, rows_per_sample, rows_per_vol * (long long)v0);                       \
            } while (0)
            switch (axis_maxr(p, 0)) {
                case 5: MVTB_ROWS_INV(5); break;
                case 13: MVTB_ROWS_INV(13); break;
                default: MVTB_ROWS_INV(31); break;
            }
#undef MVTB_ROWS_INV
        }
    }
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

extern "C" int mvtb_kspace_chain_f32(mvtb_plan* p, const float* in, float* out, int n_volumes,
                                     const mvtb_chain_desc* desc, int n_desc,
                                     float* minmax_out, int vols_per_sample, void* stream) {
    return chain_impl(p, in, out, n_volumes, desc, n_desc, minmax_out, vols_per_sample, stream, nullptr, nullptr);
}

extern "C" int mvtb_kspace_chain_ex_strided_f32(mvtb_plan* p, const float* in, float* out, int n_volumes,
                                                const mvtb_chain_desc* desc, int n_desc, const float* pre_abt, float* minmax_out,
                                                int vols_per_sample, const mvtb_sp_params* spp, uint64_t sample_stride, void* stream) {
    if (!spp) return chain_impl(p, in, out, n_volumes, desc, n_desc, minmax_out, vols_per_sample, stream, nullptr, pre_abt);
    const float prob = spp->p;
    if (!p || !minmax_out) { set_error("chain_sp: null plan or minmax_out"); return MVTB_EINVAL; }
    if (!(prob >= 0.f && prob <= 1.f)) { set_error("chain_sp: p=%g outside [0,1] (the caller clamps, F:444)", (double)prob); return MVTB_EINVAL; }
    if (vols_per_sample < 1 || n_volumes < 0 || n_volumes % vols_per_sample != 0) {
        set_error("chain_sp: n_volumes=%d is not a whole number of samples of %d volumes", n_volumes, vols_per_sample);
        return MVTB_EINVAL;
    }
    if (n_volumes / vols_per_sample > 65535) { set_error("chain_sp: more than 65535 samples in one call"); return MVTB_EUNSUPPORTED; }
    if (sample_stride && sample_stride < ((unsigned long long)vols_per_sample * p->vol_real + MVTB_SP_SPAN - 1) / MVTB_SP_SPAN) {
        set_error("chain_sp: sample_stride %llu is below a sample's span count", (unsigned long long)sample_stride);
        return MVTB_EINVAL;
    }
    SpFuse sp;
    sp.p = prob; sp.seed = spp->seed; sp.offset = spp->offset; sp.stride = sample_stride; sp.done = false;
    int rc = chain_impl(p, in, out, n_volumes, desc, n_desc, minmax_out, vols_per_sample, stream, &sp, pre_abt);
    if (rc != MVTB_OK || sp.done || prob == 0.f || n_volumes == 0) return rc;
    // any other path: the select pass follows as its own kernel (same Philox counters, same result)
    unsigned host_table[MVTB_SP_BLOCK];
    rc = mvtb_sparse_table(prob, host_table);
    if (rc != MVTB_OK) return rc;
    void* dtab = nullptr;
    rc = plan_stage_upload(p, host_table, sizeof(host_table), stream, &dtab);
    if (rc != MVTB_OK) return rc;
    return sparse_sp_launch(out, (size_t)vols_per_sample * p->vol_real, n_volumes / vols_per_sample, spp->seed, spp->offset, prob,
                            minmax_out, (const unsigned*)dtab, stream, sample_stride);
}

extern "C" int mvtb_kspace_chain_ex_f32(mvtb_plan* p, const float* in, float* out, int n_volumes,
                                        const mvtb_chain_desc* desc, int n_desc, const float* pre_abt, float* minmax_out,
                                        int vols_per_sample, const mvtb_sp_params* spp, void* stream) {
    return mvtb_kspace_chain_ex_strided_f32(p, in, out, n_volumes, desc, n_desc, pre_abt, minmax_out, vols_per_sample, spp, 0, stream);
}

extern "C" int mvtb_kspace_chain_sp_f32(mvtb_plan* p, const float* in, float* out, int n_volumes,
                                        const mvtb_chain_desc* desc, int n_desc, float* minmax_out, int vols_per_sample,
                                        float prob, uint64_t seed, uint64_t offset, void* stream) {
    mvtb_sp_params sp;
    sp.p = prob; sp.seed = seed; sp.offset = offset;
    return mvtb_kspace_chain_ex_f32(p, in, out, n_volumes, desc, n_desc, nullptr, minmax_out, vols_per_sample, &sp, stream);
}

extern "C" int mvtb_kspace_logabs_sum_f32(mvtb_plan* p, const float* in, int n_volumes, double* sums_out, void* stream) {
    if (!p || !in || !sums_out) { set_error("logabs_sum: null argument"); return MVTB_EINVAL; }
    if (n_volumes < 0) { set_error("logabs_sum: n_volumes=%d", n_volumes); return MVTB_EINVAL; }
    if (n_volumes == 0) return MVTB_OK;
    MVTB_CUDA(cudaSetDevice(p->device));
    MVTB_CUDA(cudaMemsetAsync(sums_out, 0, sizeof(double) * (size_t)n_volumes, (cudaStream_t)stream));
    const ChainGeom g = make_geom(p);
    long long rows_per_vol = 1;
    for (int a = 1; a < p->ndim; ++a) rows_per_vol *= p->shape[a];
    const int mid = p->ndim - 1;
    for (int v0 = 0; v0 < n_volumes; v0 += p->chunk) {
        const int nv = (n_volumes - v0 < p->chunk) ? (n_volumes - v0) : p->chunk;
        int rc = launch_rows_fwd(p, in + (size_t)v0 * p->vol_real, p->ws, rows_per_vol * nv, stream);
        if (rc != MVTB_OK) return rc;
        for (int a = 1; a < mid; ++a) {
            rc = launch_axis<AX_FWD>(p, p->ws, a, nv, g, nullptr, 1, nullptr, stream);
            if (rc != MVTB_OK) return rc;
        }
        rc = launch_axis<AX_STATS>(p, p->ws, mid, nv, g, nullptr, 1, sums_out + v0, stream);
        if (rc != MVTB_OK) return rc;
    }
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}

extern "C" int mvtb_wrap_odd_last_f32(mvtb_plan* p, const float* in, float* out, int n_volumes, float alpha, void* stream) {
    if (!p || !in || !out) { set_error("wrap_odd_last: null argument"); return MVTB_EINVAL; }
    if (n_volumes < 0) { set_error("wrap_odd_last: n_volumes=%d", n_volumes); return MVTB_EINVAL; }
    if (in == out) { set_error("wrap_odd_last: in-place is not supported"); return MVTB_EINVAL; }
    if (p->ndim != 3 || p->lead_drop != 0 || (p->shape[1] & 1) || (p->shape[2] & 1)) {
        set_error("wrap_odd_last: needs a 3-D plan with even H and W (use the k-space chain)");
        return MVTB_EUNSUPPORTED;
    }
    if (n_volumes == 0) return MVTB_OK;
    MVTB_CUDA(cudaSetDevice(p->device));
    const int D = p->shape[0], W = p->shape[1], H = p->shape[2];
    const float c0 = 0.5f * (1.f + alpha), c1 = 0.5f * (1.f - alpha);
    const float ch = ((H / 2) & 1) ? -c1 : c1, cw = ((W / 2) & 1) ? -c1 : c1;
    const size_t orbits = (size_t)n_volumes * (H / 2) * (W / 2) * D;
    size_t blocks = (orbits + 255) / 256;
    if (blocks > (size_t)148 * 32) blocks = (size_t)148 * 32;
    MVTB_LAUNCH(k_wrap_fold_hw, dim3((unsigned)blocks), dim3(256), 0, stream, in, out, H, W, D, c0, ch, cw, orbits);
    const long long n_rows = (long long)n_volumes * H * W;
    const long long n_pairs = (n_rows + 1) / 2;
    const int rp = p->rows_pairs_per_cta;
    const unsigned grid = (unsigned)((n_pairs + rp - 1) / rp);
    const size_t smem = (size_t)rp * p->row_pitch * sizeof(cf) * (p->ax[0].generic ? 2 : 1);
    {
        ProfScope prof(p, MVTB_K_ROWS_WRAP, stream);
        switch (axis_maxr(p, 0)) {
            case 5: { auto kern = k_rows_wrap<5>; MVTB_LAUNCH(kern, dim3(grid), dim3(kThreads), smem, stream, (const float*)out, out, p->ax[0], p->row_pitch, rp, n_rows, alpha); break; }
            case 13: { auto kern = k_rows_wrap<13>; MVTB_LAUNCH(kern, dim3(grid), dim3(kThreads), smem, stream, (const float*)out, out, p->ax[0], p->row_pitch, rp, n_rows, alpha); break; }
            default: { auto kern = k_rows_wrap<31>; MVTB_LAUNCH(kern, dim3(grid), dim3(kThreads), smem, stream, (const float*)out, out, p->ax[0], p->row_pitch, rp, n_rows, alpha); break; }
        }
    }
    MVTB_CUDA(cudaGetLastError());
    return MVTB_OK;
}
