// bandlimited_tci.cuh — the H-axis INVERSE pass of the band-limited path on the tensor cores, and the select pass
// (SaltAndPepper, F:465-482) folded into its stores.
//
// The inverse pruned DFT along H plus the out-of-box spikes' plane waves is one real GEMM per tile of 128 columns:
//
//   out[h, col] = sum_k A[col, k] * B[h, k],   k = (f, re|im) for f < NF, then (plane wave s, re|im), K = 8 ceil((2 NF + 4) / 8)
//   A[col, 2f] = Re Y[f, col], A[col, 2f+1] = Im Y[f, col], A[col, 2NF+2s] = Re E_s(col), A[col, 2NF+2s+1] = Im E_s(col)
//   B[h, 2f] = c_f cos(2 pi f h / H), B[h, 2f+1] = -c_f sin(2 pi f h / H)  (c_0 = 1, c_f = 2: Hermitian half-spectrum),
//   B[h, 2NF+2s] = cos(2 pi fh_s h / H), B[h, 2NF+2s+1] = -sin(2 pi fh_s h / H)
//
// i.e. M = 128 columns, N = H rows, K = 32 for the BraTS chains: 12 tcgen05.mma (kind::tf32, 3xTF32 split, both
// operands in shared memory, one fp32 accumulator of H TMEM columns) per 30 720 voxels, where k_bl_inv_h4v spends ~16
// FFMA-pipe instructions per voxel.  What is left for the SM's threads is ~2 instructions per voxel (tcgen05.ld, the
// store), and that changes how the select pass is best done: SaltAndPepper writes min/2 and max/2 of the whole sample,
// so it cannot be applied before the last voxel exists -- but a pass that only COMPUTES the output and keeps
// (min, max) now costs ~1.5 us per 240x240x155 volume, less than the 24 MB per volume of sector read-modify-write the
// select pass costs after the fact (bandlimited_sp.cuh, DESIGN 3.5).  So the chain runs
//
//   k_bl_inv_tc<NF, 0>   compute only: per-sample (min, max)
//   k_sp_bits            the geometric-gap sampler (sp_sampler.cuh: the same spans, Philox counters and hits as
//                        k_salt_pepper_sparse) leaves 2 bits per voxel (hit, salt|pepper) in the layout the epilogue reads
//   k_bl_inv_tc<NF, 2>   computes the same tile again (bit-identical: same instructions, same operands) and stores
//                        hit ? (coin ? max/2 : min/2) : value -- every output sector is written exactly once.
//
// k_bl_inv_tc<NF, 1> is the plain inverse pass (stores, optional min/max) for mvtb_kspace_chain_f32.
//
// Roles of a CTA (persistent, one per SM): warp 0 issues the MMAs; warps 1-4 / 5-8 build
// the A operand of the even / odd tiles (coalesced reads of Y one tile of their own ahead, plane-wave amplitudes, hi/lo
// split, 16-byte shared stores in core-matrix order) and rewrite B's plane-wave columns when the volume changes; warps
// 9-24 drain the accumulators (two of H columns in TMEM, even / odd tiles; two groups of four warps each, one per half of
// the rows): tcgen05.ld of 16 rows, select, one streaming store per voxel (a warp writes 128 contiguous bytes of a row;
// staging boxes in shared memory + TMA stores were measured 1-2 k cycles per box of 16 rows: slower).  All hand-offs
// are mbarriers with bounded waits.
// GPU only (no emulator build); included by bandlimited.cu inside namespace mvtb.
#pragma once
#ifndef MVTB_EMU
#ifndef MVTB_TCI_SEL_SPANS
#define MVTB_TCI_SEL_SPANS 2
#endif

static const int kTciWarpBuild0 = 1, kTciWarpEpi0 = 9;
static const int kTciEpiGroups = 4;            // (accumulator = tile parity, half of its row groups), 4 warps each
static const int kTciThreads = 32 * (kTciWarpEpi0 + 4 * kTciEpiGroups);
static const int kTciSelSpans = MVTB_TCI_SEL_SPANS;   // mode 3: spans a select warp walks in lock step
static const int kTciPrefetch = 6;             // own tiles (every other tile of the CTA) between an L2 prefetch of Y and its use
static const int kTciRowsPerWord = 16;         // rows of one column whose (hit, coin) bits share a 32-bit word = one tcgen05.ld.x16

template <int NF> struct TciDims {
    static constexpr int K = (2 * NF + 2 * MVTB_BL_MAX_PW + 7) / 8 * 8;
};

struct TciArgs {
    const float2* Y;             // [nvol][NF][NC], scaled, after the W/D stage
    float* out;                  // [nvol][H][NC]
    const float* tab;            // [2][K * H]: B hi, lo in tc::op_offset(row = h, k, rows = H) order; plane-wave columns zero
    const BlVol* vols;
    int vol_base, shared_desc;
    int H, NC, W, D;
    int n_vols, tiles_per_vol;
    int par_vols, ctas_per_vol;  // tile order: par_vols volumes at a time, each volume's tiles strided over ctas_per_vol CTAs (grid = product)
    int n_stages;                // A-operand stages in shared memory: 2 or 4
    int vps;                     // volumes per sample ((min, max) and the select values are per sample)
    float* minmax;               // 2 floats per sample of the call, or null
    const unsigned* bits;        // mode 2: [nvol][H / 16][NC] words, bits 2j, 2j+1 = (hit, coin) of row 16 rg + j
    // mode 3: the select pass inside the kernel (warps 5-8), sample by sample as the counters fill
    unsigned* sync;              // [n_vols / vps] finished (tile, epilogue warp) pairs per sample of the launch; zeroed before the launch
    const unsigned* sp_table;    // sampler table T[k] (MVTB_SP_BLOCK entries)
    float inv_log2q;
    unsigned long long seed, offset, n_per_sample;
    unsigned bps;                // spans per sample
    unsigned long long stride;   // Philox span counters from one sample to the next (>= bps)
    int s_base;                  // index of the launch's first sample in the call
    int debug;                   // MVTB_TCI_DEBUG, measurements: 1 = the select warps wait but do not walk, 2 = no fence before the counters (unsafe)
    int* status;
    long long* prof;             // null, or wait cycles of CTA 0 by warp and barrier kind (MVTB_TC_PROF)
};

struct TciBars {
    unsigned long long a_full[4], mma_done[4], d_empty[2];
};

__device__ __forceinline__ bool tci_wait(unsigned long long* bar, uint32_t parity, volatile int* abort_flag, int* status, int code,
                                         long long* prof) {
    if (prof == nullptr || blockIdx.x != 0) return tc_wait_raw(bar, parity, abort_flag, status, 10 + code);
    const long long t0 = clock64();
    const bool ok = tc_wait_raw(bar, parity, abort_flag, status, 10 + code);
    if ((threadIdx.x & 31) == 0) prof[(threadIdx.x >> 5) * 8 + code] += clock64() - t0;
    return ok;
}

// a * b + c with 32-bit a, b and a 64-bit sum in ONE instruction (IMAD.WIDE.U32); written as C the compiler turns the
// sixteen row addresses of a thread into a chain of 64-bit additions, four instructions per store
__device__ __forceinline__ unsigned long long tci_mad_wide(unsigned a, unsigned b, unsigned long long c) {
    unsigned long long r;
    asm volatile("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(a), "r"(b), "l"(c));   // volatile: not split into a hoisted product + a 64-bit add
    return r;
}

// MODE 0: (min, max) only; 1: store (+ min/max when a.minmax); 2: store with the select applied (reads a.minmax, a.bits);
// 3: store (L2 evict_last) + min/max + per-sample completion counters, and four warps that run the select pass of each
//    sample as soon as it is complete, while its lines are still in L2 (one builder group then feeds the tensor core)
template <int NF, int MODE>
__global__ void __launch_bounds__(kTciThreads, 1)
k_bl_inv_tc(TciArgs a) {
    constexpr int K = TciDims<NF>::K, KS = K / 8;
    extern __shared__ __align__(1024) unsigned char tci_smem[];
    __shared__ TciBars bars;
    __shared__ uint32_t s_tmem;
    __shared__ int s_abort;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int H = a.H, NC = a.NC;
    const size_t tab_floats = (size_t)K * H;
    float* b_hi = (float*)tci_smem;
    float* b_lo = b_hi + tab_floats;
    float* a_st = b_lo + tab_floats;                       // [n_stages][hi | lo][128 * K]
    constexpr int kAFloats = 128 * K;

    for (size_t i = tid; i < 2 * tab_floats / 4; i += blockDim.x) ((float4*)tci_smem)[i] = __ldg((const float4*)a.tab + i);
    __shared__ unsigned s_spT[MODE == 3 ? MVTB_SP_BLOCK : 1];
    if (MODE == 3)
        for (int e = tid; e < MVTB_SP_BLOCK; e += blockDim.x) s_spT[e] = __ldg(a.sp_table + e);
    if (tid == 0) {
        s_abort = 0;
        for (int i = 0; i < 4; ++i) {
            tc::mbar_init(tc::smem_u32(&bars.a_full[i]), 4);
            tc::mbar_init(tc::smem_u32(&bars.mma_done[i]), 1);
        }
        for (int i = 0; i < 2; ++i) tc::mbar_init(tc::smem_u32(&bars.d_empty[i]), 8);
        tc::mbar_init_fence();
    }
    if (warp == 0) tc::tmem_alloc(tc::smem_u32(&s_tmem), 512);
    tc::fence_async_smem();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tmem = s_tmem;
    volatile int* abortp = &s_abort;
    constexpr int NBG = MODE == 3 ? 1 : 2;                 // builder groups
    // This CTA's tiles, in order: volumes pv, pv + P, ...; within a volume the tiles cv, cv + C, ...  The C CTAs of a
    // volume then write adjacent 512-byte row segments at about the same time -- measured with tools/wpat.cu, the
    // DRAM write stream of this pattern runs at 5.4 TB/s against 4.85 TB/s for a contiguous tile range per CTA (and
    // 6.9 TB/s for a linear fill) -- while a volume (B's plane-wave columns) still lasts tiles_per_vol / C tiles.
    const int cv = (int)blockIdx.x % a.ctas_per_vol, pv = (int)blockIdx.x / a.ctas_per_vol;
    const int nt_c = cv < a.tiles_per_vol ? (a.tiles_per_vol - cv + a.ctas_per_vol - 1) / a.ctas_per_vol : 0;
    const int nv_p = pv < a.n_vols ? (a.n_vols - pv + a.par_vols - 1) / a.par_vols : 0;
    const int n_items = nt_c * nv_p;
    const int NST = a.n_stages;
    auto locate = [&](int i, int& vol, int& c0) {
        const int vi = i / nt_c, k = i - vi * nt_c;
        vol = pv + vi * a.par_vols;
        c0 = (cv + k * a.ctas_per_vol) * 128;
    };
    const long long t_start = a.prof ? clock64() : 0;
    // MVTB_TC_PROF: timeline of CTA 0's first 64 tiles, prof[64 + 16 * tile + event] = cycles since the start
#define TCI_EV(tl, ev) do { if (a.prof && blockIdx.x == 0 && (tl) < 40 && lane == 0) a.prof[64 + 16 * (tl) + (ev)] = clock64() - t_start; } while (0)

    if (warp == 0) {
        // ------------------------------------------------------------ MMA issuer: 3 KS MMAs and one commit per tile
        const uint32_t idesc = tc::idesc_tf32(128, H);
        const uint32_t a_chunk = 16u * 128u, b_chunk = (uint32_t)(H / 8) * 128u;
        const uint32_t bh = tc::smem_u32(b_hi), bl = tc::smem_u32(b_lo);
        // In the compute-only pass the waits for tile t + 1 come BEFORE the commit of tile t: a wait issued right after a
        // tcgen05.commit was measured to return ~700 cycles late even on a barrier completed long before (the tile
        // period was issue + that: 2.2 k cycles for 1.3 k of issue).  The store passes keep commit first: there the
        // epilogue is the slow stage and must hear of a finished tile at once.
        bool ready = false;                                              // tile tcount's operands and accumulator are known to be free
        for (unsigned tcount = 0; (int)tcount < n_items && !*abortp; ++tcount) {
            const unsigned st = tcount % (unsigned)NST, ph = (tcount / (unsigned)NST) & 1u;
            const unsigned db = tcount & 1u, dph = (tcount >> 1) & 1u;
            if (!ready) {
                if (!tc_wait_raw(&bars.a_full[st], ph, abortp, a.status, 11)) break;
                TCI_EV(tcount, 3);
                if (!tc_wait_raw(&bars.d_empty[db], dph ^ 1u, abortp, a.status, 12)) break;
                TCI_EV(tcount, 4);
            }
            tc::fence_after_sync();
            if (tc::elect_one()) {
                const uint32_t ah = tc::smem_u32(a_st + (size_t)st * 2 * kAFloats), al = ah + (uint32_t)kAFloats * 4u;
                const uint32_t d = tmem + 256u * db;
                uint32_t acc = 0;
                MVTB_UNROLL
                for (int term = 0; term < 3; ++term) {                  // lo*hi, hi*lo, then hi*hi
                    if (term == 1 && (a.debug & 4)) continue;           // (measurement: two terms only)
                    const uint32_t aa = term == 0 ? al : ah, bb = term == 1 ? bl : bh;
                    MVTB_UNROLL
                    for (int j = 0; j < KS; ++j) {
                        tc::mma_ss(d, tc::smem_desc(aa + (uint32_t)j * 2u * a_chunk, a_chunk, 128u),
                                   tc::smem_desc(bb + (uint32_t)j * 2u * b_chunk, b_chunk, 128u), idesc, acc);
                        acc = 1;
                    }
                }
            }
            __syncwarp();
            ready = false;
            // (not before a volume's first tile: its builders wait for THIS tile to be finished before they touch B)
            if (MODE == 0 && (int)tcount + 1 < n_items && ((int)tcount + 1) % nt_c != 0) {
                const unsigned t1 = tcount + 1;
                if (!tc_wait_raw(&bars.a_full[t1 % (unsigned)NST], (t1 / (unsigned)NST) & 1u, abortp, a.status, 11)) break;
                TCI_EV(t1, 3);
                if (!tc_wait_raw(&bars.d_empty[t1 & 1u], ((t1 >> 1) & 1u) ^ 1u, abortp, a.status, 12)) break;
                TCI_EV(t1, 4);
                ready = true;
            }
            if (tc::elect_one()) tc::mma_commit(tc::smem_u32(&bars.mma_done[st]));
            __syncwarp();
            TCI_EV(tcount, 5);
        }
    } else if (MODE == 3 && warp >= kTciWarpBuild0 + 4 && warp < kTciWarpEpi0) {
        // ------------------------------------------------------------ select warps (mode 3): sample s once all its tiles are stored
        const unsigned gsw = blockIdx.x * 4u + (unsigned)(warp - kTciWarpBuild0 - 4), nsw = gridDim.x * 4u;
        const int n_samp = a.n_vols / a.vps;
        const unsigned expected = (unsigned)a.vps * (unsigned)a.tiles_per_vol * 8u;      // 8 epilogue warps drain a tile
        uint2 key;
        key.x = (unsigned)a.seed;
        key.y = (unsigned)(a.seed >> 32);
        for (int sidx = 0; sidx < n_samp && !*abortp; ++sidx) {
            bool ok = false;
            for (int spin = 0; spin < (1 << 21); ++spin) {                               // bounded: ~1 s
                if (ld_acquire_u32(a.sync + sidx) >= expected) { ok = true; break; }
                if (*abortp) break;
                __nanosleep(500);
            }
            if (!ok) { *abortp = 1; atomicCAS(a.status, 0, 16); break; }
            const float* mm = a.minmax + 2 * (size_t)(a.s_base + sidx);
            const float slo = 0.5f * __ldcg(mm), shi = 0.5f * __ldcg(mm + 1);
            if (a.debug & 1) continue;                                                   // (measurement: no select work)
            // kTciSelSpans spans at a time per warp: the tensor-core inverse leaves the SM's issue slots idle, so the walk is
            // bound by its dependent chains (Philox, table search, prefix sum) and interleaved chains overlap them
            for (unsigned span = gsw * kTciSelSpans; span < a.bps; span += nsw * kTciSelSpans)
                sp_walk_spans<kTciSelSpans>(a.out + (size_t)sidx * a.n_per_sample, a.n_per_sample, span, a.bps,
                                            a.offset + (unsigned long long)(a.s_base + sidx) * a.stride + span, key, s_spT, a.inv_log2q, slo, shi, lane);
        }
    } else if (warp < kTciWarpEpi0) {
        // ------------------------------------------------------------ A builders: group = tile parity, thread = column of the tile
        // This path feeds the tensor core (two groups, one tile each per iteration), so per tile it does only what depends
        // on the tile: tile coordinates advance by addition, the volume's plane-wave parameters sit in registers.  The
        // next tile's Y is requested right AFTER fence.proxy.async -- issued before it, the fence waits for those loads
        // too (3-6 k cycles per tile while the store pass saturates the memory system: MVTB_TC_PROF timeline) -- and is
        // consumed after the wait for the stage, which is where a builder that is ahead spends its time anyway.
        const unsigned grp = (unsigned)(warp - kTciWarpBuild0) >> 2;
        const int m = 32 * ((warp - kTciWarpBuild0) & 3) + lane;
        struct Loc { int k, vi; };
        auto loc_init = [&](int i) { Loc l; l.vi = nt_c ? i / nt_c : 0; l.k = i - l.vi * nt_c; return l; };
        auto loc_adv = [&](Loc& l) { l.k += NBG; while (l.k >= nt_c) { l.k -= nt_c; ++l.vi; } };
        auto loc_vol = [&](const Loc& l) { return pv + l.vi * a.par_vols; };
        auto loc_col = [&](const Loc& l) { int c = (cv + l.k * a.ctas_per_vol) * 128 + m; return c < NC ? c : NC - 1; };   // past the end: computed, never stored
        float2 ynext[NF];
        int pvol = -1, npw = 0, pfh[MVTB_BL_MAX_PW], pfw[MVTB_BL_MAX_PW], pfd[MVTB_BL_MAX_PW];
        float pamp[MVTB_BL_MAX_PW];
        auto load_y = [&](const Loc& l, float2 (&y)[NF]) {
            const float2* yv = a.Y + (size_t)loc_vol(l) * NF * NC + loc_col(l);
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) y[f] = __ldg(yv + (size_t)f * NC);
        };
        auto prefetch_y = [&](const Loc& l) {                            // Y is read once from DRAM: pull the lines into L2 early
            const float2* yv = a.Y + (size_t)loc_vol(l) * NF * NC + loc_col(l);
            if ((m & 15) == 0) {                                         // one prefetch per 128-byte line
                MVTB_UNROLL
                for (int f = 0; f < NF; ++f) asm volatile("prefetch.global.L2 [%0];" ::"l"(yv + (size_t)f * NC));
            }
        };
        // exp(2 pi i f n / N): the product reduced mod N by one float division (exact below 2^24) instead of the integer one
        auto unit = [&](int f, int n, int N, float invN, float& c_, float& s_) {
            const int pr = f * n;
            int q = (int)floorf((float)pr * invN);
            int r = pr - q * N;
            if (r < 0) r += N;
            if (r >= N) r -= N;
            sincospif(2.0f * (float)r / (float)N, &s_, &c_);             // the correctly rounded quotient, as bl_unit32 (r * (1/N) is an ulp worse)
        };
        const float invW = 1.0f / (float)a.W, invD = 1.0f / (float)a.D, invH = 1.0f / (float)H;
        Loc lc = loc_init((int)grp), ln = lc, lp = lc;
        if ((int)grp < n_items) load_y(lc, ynext);
        loc_adv(ln);
        for (int i = 1; i < kTciPrefetch; ++i) {
            loc_adv(lp);
            if ((int)grp + NBG * i < n_items) prefetch_y(lp);
        }
        loc_adv(lp);
        for (int tile = (int)grp; tile < n_items && !*abortp; tile += NBG, loc_adv(lc), loc_adv(ln), loc_adv(lp)) {
            const unsigned tcount = (unsigned)tile, st = tcount % (unsigned)NST, ph = (tcount / (unsigned)NST) & 1u;
            const int vol = loc_vol(lc);
            const bool new_vol = vol != pvol;
            if (new_vol) {
                const BlVol& bv = a.vols[a.shared_desc ? 0 : a.vol_base + vol];
                npw = bv.npw;
                MVTB_UNROLL
                for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
                    pfh[s] = bv.pw[s].fh; pfw[s] = bv.pw[s].fw; pfd[s] = bv.pw[s].fd; pamp[s] = bv.pw[s].amp;
                }
                pvol = vol;
            }
            float ev[2 * MVTB_BL_MAX_PW];
            MVTB_UNROLL
            for (int s = 0; s < 2 * MVTB_BL_MAX_PW; ++s) ev[s] = 0.f;
            if (npw > 0) {
                const int col = loc_col(lc);
                int w = (int)((float)col * invD);                        // col < 2^24: within one of the quotient
                if (w * a.D > col) --w;
                if ((w + 1) * a.D <= col) ++w;
                const int d = col - w * a.D;
                MVTB_UNROLL
                for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
                    if (s < npw) {
                        float cw, sw, cd, sd;
                        unit(pfw[s], w, a.W, invW, cw, sw);
                        unit(pfd[s], d, a.D, invD, cd, sd);
                        ev[2 * s] = pamp[s] * (cw * cd - sw * sd);
                        ev[2 * s + 1] = pamp[s] * (sw * cd + cw * sd);
                    }
                }
            }
            // the stage's previous tile (n_stages tiles ago) has been multiplied
            if (warp == kTciWarpBuild0 + 4 * (int)grp) TCI_EV(tcount, 0);
            if (!tc_wait_raw(&bars.mma_done[st], ph ^ 1u, abortp, a.status, 13)) break;
            if (warp == kTciWarpBuild0 + 4 * (int)grp) TCI_EV(tcount, 1);
            if (lc.k == 0) {
                // B's plane-wave columns belong to the volume and are rewritten by the builders of the CTA's first tile of
                // it (the other group's first tile of the volume is multiplied later: the issuer works in order).  Every
                // earlier MMA must be finished before they change (the tile before this one; MMAs complete in order).
                if (tcount > 0 && !tc_wait_raw(&bars.mma_done[(tcount - 1) % (unsigned)NST], ((tcount - 1) / (unsigned)NST) & 1u, abortp, a.status, 14)) break;
                for (int e = m; e < MVTB_BL_MAX_PW * H; e += 128) {
                    const int s = e / H, h = e - s * H;
                    float c_ = 0.f, s_ = 0.f;
                    if (s < npw) unit(s == 0 ? pfh[0] : pfh[MVTB_BL_MAX_PW - 1], h, H, invH, c_, s_);
                    const float v2[2] = {c_, -s_};
                    MVTB_UNROLL
                    for (int r = 0; r < 2; ++r) {
                        const size_t o = tc::op_offset(h, 2 * NF + 2 * s + r, H) / 4;
                        const float hi = __uint_as_float(__float_as_uint(v2[r]) & 0xffffe000u);
                        b_hi[o] = hi;
                        b_lo[o] = v2[r] - hi;
                    }
                }
            }
            float v[K];
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                v[2 * f] = ynext[f].x;
                v[2 * f + 1] = ynext[f].y;
            }
            MVTB_UNROLL
            for (int k = 2 * NF; k < K; ++k) v[k] = (k - 2 * NF) < 2 * MVTB_BL_MAX_PW ? ev[(k - 2 * NF) < 2 * MVTB_BL_MAX_PW ? k - 2 * NF : 0] : 0.f;
            float* ah = a_st + (size_t)st * 2 * kAFloats;
            float* al = ah + kAFloats;
            MVTB_UNROLL
            for (int c = 0; c < K / 4; ++c) {                            // [k / 4][col / 8][col % 8][4]: 16 bytes per (chunk, column)
                float4 hi, lo;
                hi.x = __uint_as_float(__float_as_uint(v[4 * c]) & 0xffffe000u);     lo.x = v[4 * c] - hi.x;
                hi.y = __uint_as_float(__float_as_uint(v[4 * c + 1]) & 0xffffe000u); lo.y = v[4 * c + 1] - hi.y;
                hi.z = __uint_as_float(__float_as_uint(v[4 * c + 2]) & 0xffffe000u); lo.z = v[4 * c + 2] - hi.z;
                hi.w = __uint_as_float(__float_as_uint(v[4 * c + 3]) & 0xffffe000u); lo.w = v[4 * c + 3] - hi.w;
                *(float4*)(ah + (size_t)c * 512 + (size_t)m * 4) = hi;
                *(float4*)(al + (size_t)c * 512 + (size_t)m * 4) = lo;
            }
            tc::fence_async_smem();                                      // generic-proxy writes -> visible to the MMA unit
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tc::smem_u32(&bars.a_full[st]));
            if (warp == kTciWarpBuild0 + 4 * (int)grp) TCI_EV(tcount, 2);
            if (tile + NBG < n_items) load_y(ln, ynext);                 // lands while the next tile waits for its stage
            if (tile + NBG * kTciPrefetch < n_items) prefetch_y(lp);
        }
    } else {
        // ------------------------------------------------------------ epilogue: group = (tile parity, half of the row groups)
        const unsigned eg = (unsigned)(warp - kTciWarpEpi0) >> 2, grp = eg & 1u, half = eg >> 1;
        const int q = warp & 3;                                          // TMEM lanes 32 q .. 32 q + 31
        const int m = 32 * q + lane;
        const int RG = H / kTciRowsPerWord;
        const int rg_lo = half == 0 ? 0 : (RG + 1) / 2, rg_hi = half == 0 ? (RG + 1) / 2 : RG;
        const unsigned row_bytes = (unsigned)NC * 4u;
        float lo = __int_as_float(0x7f800000), hi = __int_as_float((int)0xff800000u);
        float sel_lo = 0.f, sel_hi = 0.f;
        const bool want_mm = MODE == 0 || MODE == 3 || (MODE == 1 && a.minmax != nullptr);
        const unsigned long long pol = MODE == 3 ? l2_policy_evict_last() : 0ull;
        int cur_sample = -1;
        auto flush_mm = [&]() {
            MVTB_UNROLL
            for (int o = 16; o > 0; o >>= 1) {
                lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
                hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
            }
            if (lane == 0 && lo <= hi) { bl_atomic_min(a.minmax + 2 * (size_t)cur_sample, lo); bl_atomic_max(a.minmax + 2 * (size_t)cur_sample + 1, hi); }
            lo = __int_as_float(0x7f800000); hi = __int_as_float((int)0xff800000u);
        };
        for (int tile = (int)grp; tile < n_items && !*abortp; tile += 2) {
            const unsigned tcount = (unsigned)tile, st = tcount % (unsigned)NST, ph = (tcount / (unsigned)NST) & 1u;
            int vol, c0;
            locate(tile, vol, c0);
            const int sample = (a.vol_base + vol) / a.vps;
            if (sample != cur_sample) {
                if (want_mm && MODE != 3 && cur_sample >= 0) flush_mm();
                if (MODE == 2) {
                    sel_lo = 0.5f * __ldcg(a.minmax + 2 * (size_t)sample);
                    sel_hi = 0.5f * __ldcg(a.minmax + 2 * (size_t)sample + 1);
                }
                cur_sample = sample;
            }
            const int col = c0 + m;
            const bool okc = col < NC;
            unsigned wb[8];                                              // this column's (hit, coin) words, in flight during the wait
            if (MODE == 2) {
                const unsigned* bp = a.bits + ((size_t)vol * RG + rg_lo) * NC + col;
                MVTB_UNROLL
                for (int r = 0; r < 8; ++r) wb[r] = (okc && rg_lo + r < rg_hi) ? __ldg(bp + (size_t)r * NC) : 0u;
            }
            if (!tc_wait_raw(&bars.mma_done[st], ph, abortp, a.status, 15)) break;
            if (q == 0) TCI_EV(tcount, 6 + 2 * (int)half);
            tc::fence_after_sync();
            const uint32_t t0 = tmem + ((uint32_t)(32 * q) << 16) + 256u * grp;
            float* op = a.out + (size_t)vol * H * NC + col;
            MVTB_UNROLL
            for (int r = 0; r < 8; ++r) {
                const int rg = rg_lo + r;
                if (rg >= rg_hi) break;
                uint32_t v[16];
                tc::tmem_ld16(t0 + 16u * (uint32_t)rg, v);
                tc::tmem_ld_wait();
                if (rg == rg_hi - 1) {                                   // this group's part of the accumulator is in registers
                    tc::fence_before_sync();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(tc::smem_u32(&bars.d_empty[grp]));
                }
                if (want_mm && okc) {
                    MVTB_UNROLL
                    for (int j = 0; j < 16; j += 2) {
                        lo = min3(lo, __uint_as_float(v[j]), __uint_as_float(v[j + 1]));
                        hi = max3(hi, __uint_as_float(v[j]), __uint_as_float(v[j + 1]));
                    }
                }
                if (MODE != 0 && okc) {
                    // row addresses as base + (32-bit stride) x (constant row): one IMAD.WIDE each
                    const unsigned long long ob = tci_mad_wide(row_bytes, (unsigned)(rg * 16), (unsigned long long)op);
                    MVTB_UNROLL
                    for (int j = 0; j < 16; ++j) {
                        float x = __uint_as_float(v[j]);
                        if (MODE == 2) {
                            const float sv = (wb[r] & (2u << (2 * j))) ? sel_hi : sel_lo;
                            x = (wb[r] & (1u << (2 * j))) ? sv : x;
                        }
                        float* o = (float*)tci_mad_wide(row_bytes, (unsigned)j, ob);
                        if (MODE == 3) asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(o), "f"(x), "l"(pol) : "memory");
                        else __stcs(o, x);
                    }
                }
            }
            if (q == 0) TCI_EV(tcount, 7 + 2 * (int)half);
            if (MODE == 3) {
                flush_mm();                                              // the tile's (min, max) are in before it counts as stored
                if (!(a.debug & 2)) __threadfence();                     // ... and so are this thread's rows, device-wide
                __syncwarp();
                if (lane == 0) atomicAdd(a.sync + vol / a.vps, 1u);
            }
        }
        if (want_mm && MODE != 3 && cur_sample >= 0) flush_mm();
    }
    tc::fence_before_sync();
    __syncthreads();
    if (a.prof && blockIdx.x == 0 && tid == 0) { a.prof[0] = clock64() - t_start; a.prof[6] = n_items; }
#undef TCI_EV
    if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------ the select pass's coordinates as bits
// One CTA per (volume, group of 16 rows): its 16 NC voxels are a contiguous range of the sample, covered by ~16 NC / 8192
// spans of the sampler; one warp per span walks it (sp_walk_span_cb: k_salt_pepper_sparse's stream) and ORs (hit, coin)
// into the range's NC words in shared memory, which then leave as coalesced stores.  A span that straddles two ranges
// is walked by both CTAs; each keeps the hits inside its own range.
struct SpBitsArgs {
    unsigned* bits;              // [nvol][RG][NC]
    int H, NC, vps, RG;
    unsigned long long vol_n;    // voxels per volume
    unsigned long long n_per_sample;
    unsigned bps;                // spans per sample
    unsigned long long stride;   // Philox span counters from one sample to the next (>= bps)
    int s_base;                  // index of the launch's first sample in the call
    const unsigned* table;
    float inv_log2q;
    unsigned long long seed, offset;
};

__global__ void __launch_bounds__(1024, 1)
k_sp_bits(SpBitsArgs a) {
    extern __shared__ __align__(16) unsigned char spb_smem[];
    unsigned* sw = (unsigned*)spb_smem;                    // NC words (padded to a multiple of 4)
    __shared__ unsigned sT[MVTB_SP_BLOCK];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int NC = a.NC, NC4 = (NC + 3) / 4;
    for (int e = tid; e < MVTB_SP_BLOCK; e += blockDim.x) sT[e] = __ldg(a.table + e);
    for (int i = tid; i < NC4; i += blockDim.x) ((uint4*)sw)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    const int rg = blockIdx.x % a.RG, vol = blockIdx.x / a.RG;           // volume within the launch
    const int s = vol / a.vps, vin = vol - s * a.vps;
    const unsigned long long r0 = (unsigned long long)vin * a.vol_n + (unsigned long long)rg * kTciRowsPerWord * NC;
    const unsigned r_len = (unsigned)kTciRowsPerWord * (unsigned)NC;
    const unsigned sp0 = (unsigned)(r0 / MVTB_SP_SPAN), sp1 = (unsigned)((r0 + r_len - 1) / MVTB_SP_SPAN);
    uint2 key;
    key.x = (unsigned)a.seed;
    key.y = (unsigned)(a.seed >> 32);
    for (unsigned span = sp0 + (unsigned)warp; span <= sp1; span += (unsigned)nwarps) {
        const unsigned long long j0 = (unsigned long long)span * MVTB_SP_SPAN;
        const int len = (int)((a.n_per_sample - j0) < (unsigned long long)MVTB_SP_SPAN ? (a.n_per_sample - j0) : (unsigned long long)MVTB_SP_SPAN);
        // (row, column) of the span's first voxel relative to the range, rows floor-divided (the first span starts above it)
        const long long rel0 = (long long)j0 - (long long)r0;
        long long row0l = rel0 / NC;
        if (rel0 - row0l * NC < 0) --row0l;
        const int row0 = (int)row0l, col0 = (int)(rel0 - row0l * NC);
        sp_walk_span_cb(len, a.offset + (unsigned long long)(a.s_base + s) * a.stride + span, key, sT, a.inv_log2q, lane,
                        [&](int pos, unsigned coin) {
                            int c = col0 + pos, j = row0;
                            while (c >= NC) { c -= NC; ++j; }
                            if (j >= 0 && j < kTciRowsPerWord) atomicOr(sw + c, (1u | (coin << 1)) << (2 * j));
                        });
    }
    __syncthreads();
    unsigned* dst = a.bits + ((size_t)vol * a.RG + rg) * NC;
    if ((NC & 3) == 0 && ((((size_t)vol * a.RG + rg) * NC) & 3) == 0) {
        for (int i = tid; i < NC4; i += blockDim.x) ((uint4*)dst)[i] = ((const uint4*)sw)[i];
    } else {
        for (int i = tid; i < NC; i += blockDim.x) dst[i] = sw[i];
    }
}
#endif  // MVTB_EMU
