// bandlimited_sp.cuh — the H-axis inverse pass and the salt-and-pepper select of the 127 chain as ONE persistent kernel.
//
// SaltAndPepper (F:465-482) writes min/2 and max/2 of its *input*, i.e. of the k-space chain's whole output sample, so
// no corrupted voxel can be written before the last output voxel of the sample exists.  As two kernels over a
// 64-volume chunk the select pass finds its 2.3 GB long gone from the 126 MB L2 and pays 24 MB per volume of 32-byte
// sector read-modify-write in DRAM (6.6 us per volume for ~0 algorithmic bytes).  Here both run from one work queue:
//
//   inverse tile  I(s, j): 512 columns x one part of the H range (k_bl_inv_h4v's arithmetic, bl_inv_h4v_cols) of one
//                          volume of sample s; output rows leave as plain write-back stores (they stay in L2), the
//                          tile's (min, max) go to the sample's atomics, then a release increment of done[s];
//   select tile   S(s, j): 8 spans of 8192 voxels of sample s, one warp each, walked by the geometric-gap sampler
//                          (sp_sampler.cuh: k_salt_pepper_sparse's arithmetic and Philox counters, bit-identical
//                          output), after an acquire read of done[s] shows every inverse tile of the sample finished.
//
// The queue is a periodic sequence built on the host (one period = the inverse tiles of one sample merged with the
// select tiles of earlier samples, `lag` inverse tiles behind and spread over the period), so that by the time a
// select tile is handed out the tiles it depends on were handed out about one wave of CTAs earlier: the wait is an
// acquire load that almost always succeeds at once, and it cannot deadlock -- a waiting CTA only waits for tiles
// that were dequeued before its own, by CTAs that are therefore resident and never wait themselves.
// Included by bandlimited.cu inside namespace mvtb.
#pragma once

#define MVTB_IS_SELECT 0x80000000u
static const int kIsSpansPerWarp = 1;    // spans a warp of a select tile walks at a time (4 interleaved chains measured slower than 1: 14.5 vs 13.4 us)

struct IsArgs {
    unsigned* sync;              // [0] queue head, [1 + s] finished inverse tiles of sample s; zeroed before the launch
    const unsigned* pattern;     // one period: kind << 31 | periods back << 28 | tile index within the sample
    int period;                  // entries per period
    unsigned total;              // queue length = periods * period
    int nsamp;                   // samples in this launch
    int A;                       // inverse tiles per sample = vps * ncb2 * HS
    int vps, ncb2, HS;
    int s_base;                  // index of the launch's first sample in the call (Philox counters, minmax slot)
    const unsigned* table;       // T[k] = floor(2^32 (1 - (1-p)^(k+1))), MVTB_SP_BLOCK entries
    float inv_log2q;
    unsigned long long seed, offset;
    unsigned long long n_per_sample;
    unsigned bps;                // spans of MVTB_SP_SPAN voxels per sample
    unsigned long long stride;   // Philox span counters from one sample to the next (>= bps)
    float* minmax;               // 2 floats per sample of the call
    int debug;                   // measurements: 1 = select tiles do no work, 2 = ... and do not wait, 4 = inverse tiles skip the fences, 8 = hits stored as found
};

#ifdef MVTB_EMU
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) { return *p; }
__device__ __forceinline__ float ld_l2_f32(const float* p) { return *p; }
__device__ __forceinline__ void is_fence() {}
__device__ __forceinline__ void is_sleep() {}
#else
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ld_l2_f32(const float* p) { return __ldcg(p); }
__device__ __forceinline__ void is_fence() { __threadfence(); }
__device__ __forceinline__ void is_sleep() { __nanosleep(200); }
#endif

template <int NF, int STORE>
__global__ void __launch_bounds__(256, 2)
k_bl_inv_sp(const cf* __restrict__ Y, float* __restrict__ out, BlGeom g, const BlVol* __restrict__ vols, int vol_base,
            int shared_desc, IsArgs a) {
    constexpr int NT = BlDims<NF>::NT;
    MVTB_DYN_SMEM(smem_raw);
    const int H = g.H, H2 = H / 2, H4 = H / 4;
    const int NC = (int)g.NC;
    float* sc = (float*)smem_raw;                                   // (cos, sin) rows 0 .. H/2 of the H axis
    cf* seh = (cf*)(sc + (H2 + 1) * NT);                            // plane-wave phases along H of the cached volume
    unsigned* sT = (unsigned*)(seh + MVTB_BL_MAX_PW * (H2 + 1));    // sampler table
    __shared__ unsigned s_item;
    // select tiles: a warp's hits are parked in stream order and leave 32 consecutive hits per store instruction; about half
    // of the select's sectors are no longer in L2 (ncu: 11 MB read + 12 MB extra written per volume) and for those the
    // ordered read-modify-writes keep a DRAM page together: 13.1 instead of 13.5 us per volume (debug & 8 = as found)
    __shared__ unsigned short s_stage[8][kSpStageIters * 96];
    const int tid = threadIdx.x;
    bl_load_table<NF>(sc, g.tabC[2], g.tabS[2], H, tid, blockDim.x);
    for (int e = tid; e < MVTB_SP_BLOCK; e += blockDim.x) sT[e] = __ldg(a.table + e);
    int cached_vol = -1;
    const unsigned long long pol = STORE == 2 ? l2_policy_evict_last() : 0ull;
    const int tiles_per_vol = a.ncb2 * a.HS;
    const int nq = H4 - 1;                                          // quads 1 .. H/4-1
    uint2 key;
    key.x = (unsigned)a.seed;
    key.y = (unsigned)(a.seed >> 32);

    for (;;) {
        __syncthreads();                                            // the previous tile is done with shared memory
        if (tid == 0) s_item = atomicAdd(a.sync, 1u);
        __syncthreads();
        const unsigned t = s_item;
        if (t >= a.total) break;
        const int per = (int)(t / (unsigned)a.period);
        const unsigned e = __ldg(a.pattern + (t - (unsigned)per * (unsigned)a.period));
        const int s = per - (int)((e >> 28) & 7u);
        if (s < 0 || s >= a.nsamp) continue;                        // head and tail of the periodic sequence
        const int j = (int)(e & 0x0fffffffu);
        if (!(e & MVTB_IS_SELECT)) {
            // ---------------------------------------------------------------- inverse tile
            const int vis = j / tiles_per_vol, r = j - vis * tiles_per_vol;
            const int cb = r / a.HS, part = r - cb * a.HS;
            const int vol = s * a.vps + vis;                        // volume within this launch
            const BlVol& bv = vols[shared_desc ? 0 : vol_base + vol];
            if (vol != cached_vol) {
                const int npw = bv.npw;
                for (int i = tid; i < MVTB_BL_MAX_PW * (H2 + 1); i += blockDim.x) {
                    const int sp = i / (H2 + 1), h = i - sp * (H2 + 1);
                    float c_ = 0.f, s_ = 0.f;
                    if (sp < npw) bl_unit32(bv.pw[sp].fh, h, H, &c_, &s_);
                    seh[i] = cmk(c_, s_);
                }
                cached_vol = vol;
                __syncthreads();
            }
            // quads 1 .. nq in HS nearly equal parts; the last (shortest) part also does rows 0, H/2, H/4, 3H/4
            const int base = nq / a.HS, rem = nq - base * a.HS;
            const int q0 = 1 + part * base + (part < rem ? part : rem);
            const int q1 = q0 + base + (part < rem ? 1 : 0);
            int col = (cb * 256 + tid) * 2;
            const bool ok = col < NC;
            if (!ok) col = NC - 2;
            float lo = __int_as_float(0x7f800000), hi = __int_as_float((int)0xff800000u);
            bl_inv_h4v_cols<NF, STORE>(sc, seh, Y + (size_t)vol * NF * NC + col, out + (size_t)vol * H * NC + col, g, bv,
                                       col, ok, q0, q1, part == a.HS - 1, pol, lo, hi);
            if (!(a.debug & 4)) is_fence();                         // this thread's rows are visible device-wide ...
            bl_block_minmax(lo, hi, a.minmax + 2 * (size_t)(a.s_base + s));
            if (tid == 0) {                                         // ... before the tile counts as finished
                is_fence();
                atomicAdd(a.sync + 1 + s, 1u);
            }
        } else {
            // ---------------------------------------------------------------- select tile: 8 warps x kIsSpansPerWarp spans
            if (tid == 0 && !(a.debug & 2))
                while (ld_acquire_u32(a.sync + 1 + s) < (unsigned)a.A) is_sleep();
            __syncthreads();
            if (a.debug & 1) continue;
            const float* mm = a.minmax + 2 * (size_t)(a.s_base + s);
            const float lo = 0.5f * ld_l2_f32(mm), hi = 0.5f * ld_l2_f32(mm + 1);
            const unsigned span = ((unsigned)j * 8u + (unsigned)(tid >> 5)) * kIsSpansPerWarp;
            if (span < a.bps)
                sp_walk_spans<kIsSpansPerWarp>(out + (size_t)s * a.n_per_sample, a.n_per_sample, span, a.bps,
                                               a.offset + (unsigned long long)(a.s_base + s) * a.stride + span, key, sT, a.inv_log2q,
                                               lo, hi, tid & 31, (a.debug & 8) ? nullptr : s_stage[tid >> 5]);
        }
    }
}
