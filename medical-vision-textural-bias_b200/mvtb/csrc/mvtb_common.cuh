// mvtb_common.cuh — shared declarations for the libmvtb kernels (sm_100a).
//
// The sources also compile with g++ -DMVTB_EMU against tests/cuemu/cuemu.h (a debug-only
// fiber emulator used in the GPU-less build container to exercise index arithmetic); every
// difference between the two builds is confined to the MVTB_EMU blocks in this header.
#pragma once
#include <stdint.h>
#include <stddef.h>

#ifdef MVTB_EMU
#include "cuemu.h"
#define MVTB_LAUNCH(kern, grid, block, smem, stream, ...) \
    do { mvtb::count_launch(); cuemu::launch((grid), (block), (smem), [&]() { kern(__VA_ARGS__); }); } while (0)
#define MVTB_DYN_SMEM(name) unsigned char* name = cuemu::g_dyn_smem
#define MVTB_UNROLL
#define MVTB_UNROLL_N(n)
// double-precision intrinsics the emulator lacks (nifti.cuh); volatile keeps g++ from contracting them into an FMA
static inline float __double2float_rn(double d) { return (float)d; }
static inline double __dmul_rn(double a, double b) { volatile double r = a * b; return r; }
static inline double __dadd_rn(double a, double b) { volatile double r = a + b; return r; }
// the jump's shared-memory reduction (mt19937.cuh); blocks run one thread at a time
static inline unsigned atomicXor(unsigned* p, unsigned v) { unsigned o = *p; *p = o ^ v; return o; }
#else
#include <cuda_runtime.h>
#define MVTB_LAUNCH(kern, grid, block, smem, stream, ...) \
    do { mvtb::count_launch(); kern<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__); } while (0)
#define MVTB_DYN_SMEM(name) extern __shared__ __align__(16) unsigned char name[]
#define MVTB_UNROLL _Pragma("unroll")
#define MVTB_STR_(x) #x
#define MVTB_UNROLL_N(n) _Pragma(MVTB_STR_(unroll n))
#endif

#include "../../../include/mvtb.h"

namespace mvtb {

// ---------------------------------------------------------------- error plumbing
void set_error(const char* fmt, ...);
void count_launch();
int cuda_fail(cudaError_t e, const char* what);   // records text, returns (int)e

#define MVTB_CUDA(call)                                         \
    do {                                                        \
        cudaError_t e_ = (call);                                \
        if (e_ != cudaSuccess) return mvtb::cuda_fail(e_, #call); \
    } while (0)

// ---------------------------------------------------------------- complex helpers
typedef float2 cf;
__device__ __forceinline__ cf cmk(float x, float y) { cf r; r.x = x; r.y = y; return r; }
__device__ __forceinline__ cf cadd(cf a, cf b) { return cmk(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ cf csub(cf a, cf b) { return cmk(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ cf cmul(cf a, cf b) { return cmk(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ cf cmulc(cf a, cf b) { return cmk(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); }  // a * conj(b)
__device__ __forceinline__ cf cconj(cf a) { return cmk(a.x, -a.y); }
__device__ __forceinline__ cf cscale(cf a, float s) { return cmk(a.x * s, a.y * s); }
__device__ __forceinline__ cf cmuli(cf a) { return cmk(-a.y, a.x); }    // a * (+i)
__device__ __forceinline__ cf cmulni(cf a) { return cmk(a.y, -a.x); }   // a * (-i)

// ---------------------------------------------------------------- asynchronous global -> shared copies (LDGSTS)
// The bytes a CTA has in flight stop being limited by registers; the emulator copies synchronously.
template <int BYTES>
__device__ __forceinline__ void cp_async(void* smem_dst, const void* gsrc) {
#ifdef MVTB_EMU
    for (int i = 0; i < BYTES; ++i) ((unsigned char*)smem_dst)[i] = ((const unsigned char*)gsrc)[i];
#else
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    if (BYTES == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(d), "l"(gsrc), "n"(BYTES) : "memory");
#endif
}
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) { cp_async<16>(smem_dst, gsrc); }
// the same with the shared-memory address converted once by the caller (32-bit arithmetic in the loop)
#ifdef MVTB_EMU
typedef unsigned char* smem_addr_t;
__device__ __forceinline__ smem_addr_t smem_addr(void* p) { return (unsigned char*)p; }
__device__ __forceinline__ void cp_async16_at(smem_addr_t d, const void* gsrc) { cp_async<16>(d, gsrc); }
#else
typedef unsigned smem_addr_t;
__device__ __forceinline__ smem_addr_t smem_addr(void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16_at(smem_addr_t d, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
#endif
__device__ __forceinline__ void cp_async_commit() {
#ifndef MVTB_EMU
    asm volatile("cp.async.commit_group;" ::: "memory");
#endif
}
template <int N>
__device__ __forceinline__ void cp_async_wait() {
#ifndef MVTB_EMU
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
#endif
}

// ---------------------------------------------------------------- per-axis FFT description
struct DescDev;
// voxel_ops.cu: the geometric-gap sampler on its own (table_dev already holds mvtb_sparse_table(p))
// sample_stride: Philox span counters between consecutive samples, 0 = the sample's own span count
int sparse_sp_launch(float* x, size_t n_per_sample, int n_samples, uint64_t seed, uint64_t offset, float p,
                     const float* minmax, const unsigned* table_dev, void* stream, uint64_t sample_stride = 0);
// salt-and-pepper to run behind the chain (mvtb_kspace_chain_sp_f32); `done` is set by the path that fused it
struct SpFuse {
    float p;
    unsigned long long seed, offset;
    unsigned long long stride;   // Philox span counters from one sample to the next; 0 = the sample's span count
    bool done;
};
#define MVTB_MAX_STAGES 12
// One pass over the shared-memory tile: a radix stage, or two stages fused in registers.  Everything a thread
// needs is precomputed on the host: with 128-thread CTAs a thread runs only a couple of butterflies per pass, so
// per-pass integer divisions would cost as much as the butterflies.
struct PassDev {
    int r1, r2;                  // radices (r2 = 0: single stage)
    int L;                       // block length entering the pass (forward order)
    int m;                       // block length leaving it: L / (r1 * max(r2, 1))
    int per_seq;                 // butterflies per sequence: n / (r1 * max(r2, 1))
    int ts1, ts2;                // twiddle strides n / L and n / (L / r1)
    unsigned magic_m, magic_ps;  // x / m = umulhi(x, magic_m), x / per_seq likewise (unused when the divisor is 1)
};
struct AxisDev {
    int n;                       // axis length
    int nstage;                  // radix stages
    int radix[MVTB_MAX_STAGES];  // forward (DIF) order
    int fuse[MVTB_MAX_STAGES];   // 1: stage s and s+1 run as one register-fused pass (fft_stage2)
    int npass;
    PassDev pass[MVTB_MAX_STAGES];
    int generic;                 // 1: some radix is a prime > 31 (fft_stage_generic: needs a scratch tile)
    const cf* tw;                // tw[t] = exp(-2 pi i t / n), t in [0, n)
    const int* pos2k;            // position after the in-place DIF  ->  frequency bin
    const int* k2pos;            // inverse map
};

// device view of mvtb_chain_desc, prepared on the host
struct SpikeDev {
    int idx[MVTB_MAX_FFT_DIMS];  // shifted index per FFT axis, axis 0 = LAST (contiguous) axis
    float amp;
    float meff_at_spike;         // (M(f_s) + M(-f_s)) / 2 in {0, 1/2, 1}: the weight of that bin after the mask stage
};
struct DescDev {
    int mask_kind, mask_ndim;
    long long thr;
    int inside_off, n_spikes;
    float wrap_alpha;
    int wrap_naxes;
    SpikeDev sp[MVTB_MAX_SPIKES];
    const float* mask_u;         // MVTB_MASK_UNIFORM: the volume's uniform field, full fftshift-ed layout
    float mask_p;
    int pad_;
};

}  // namespace mvtb

#define MVTB_PROF_MAX 2048
#define MVTB_STAGE_SLOTS 4
#define MVTB_BL_FT 36                     // table columns: frequencies 0..35
#define MVTB_BL_MAX_PW 2                  // out-of-box spikes per volume the inverse kernel adds as plane waves
struct mvtb_plan {
    int ndim;                             // FFT rank (2..4) after dropping leading length-1 axes
    int lead_drop;                        // how many leading length-1 FFT axes the caller's shape had
    int shape[MVTB_MAX_FFT_DIMS];         // axis 0 = LAST (contiguous) axis ... axis ndim-1 = outermost
    int nh;                               // shape[0]/2 + 1
    int chunk;                            // volumes in flight
    int device;
    int num_sms;
    size_t vol_real;                      // floats per volume
    size_t vol_half;                      // complex per volume half-spectrum
    mvtb::AxisDev ax[MVTB_MAX_FFT_DIMS];  // device tables
    void* table_mem;                      // one allocation behind all tables
    mvtb::cf* ws;                         // chunk * vol_half complex
    size_t ws_bytes;
    // rows kernels geometry
    int row_pitch;                        // complex slots per row pair in shared memory (odd)
    int rows_pairs_per_cta;
    int axis_tile;                        // columns per CTA in the axis kernels
    // band-limited path (bandlimited.cu): cos/sin tables per axis, [N][MVTB_BL_FT] each
    int opt_path;
    int opt_async;                        // 1: cp.async staging ring in the forward H kernel (MVTB_NO_ASYNC=1 turns it off)
    int opt_fusemid;                      // 1: one kernel for the W axis, D axis and pointwise stage (MVTB_NO_FUSEMID=1: three)
    int opt_quad;                         // 1: use the quad-symmetry H kernels when H % 4 == 0 (tests can turn it off)
    float* bl_tab;
    size_t bl_off[3];
    mvtb::cf* bl_ws;                      // band-limited intermediates (Y, G), grown on demand
    size_t bl_ws_bytes;
    // fused inverse + salt-and-pepper kernel (bandlimited_sp.cuh); the MVTB_IS_* environment variables are for measurements
    int opt_fusesp;                       // 1: mvtb_kspace_chain_sp_f32 runs the select pass inside the inverse kernel (MVTB_NO_FUSESP=1: after it)
    int is_chunk;                         // volumes per launch (0: the band-limited default)
    int is_hs;                            // parts the H range of a column tile is split into
    int is_lag;                           // select tiles trail their sample's inverse tiles by this many tiles (-1: one wave of CTAs)
    int is_spread_pct;                    // ... and are spread over this share of a period
    int is_store;                         // 0 streaming, 1 write-back, 2 write-back + L2 evict_last
    int is_max_sample_mb;                 // samples larger than this take the separate select pass (their lines leave L2 first)
    unsigned* is_sync;                    // queue head + per-sample completion counters
    // tensor-core H-axis kernels (bandlimited_tc.cuh): operand tables per NF (built on first use), failure flag
    int opt_tc;                           // 1: tensor-core forward H pass when the shape allows (MVTB_TC, default 1; MVTB_PATH_BL_TC / _CUDACORE)
    int opt_tc_inv;                       // with opt_tc: the inverse pass too (MVTB_TC_INV, default 0: measured slower than the fused CUDA-core kernel; MVTB_PATH_BL_TC)
    int opt_bits_overlap;                 // k_sp_bits on the plan's side stream, next to the W/D stage (MVTB_BITS_OVERLAP, default 1)
    cudaStream_t side_stream;             // created on first use
    cudaEvent_t ev_fork, ev_join;
    int tci_par_vols;                     // inverse tensor-core pass: volumes in flight at a time (MVTB_TCI_PV, default 4)
    int tc_tma;                           // 1: the forward kernel stages x with TMA tensor-map copies (MVTB_TC_TMA=1); 0: coalesced LDG
    float* tc_tab_fwd[8];                 // by NF slot: [2][H * N] forward table (hi, lo)
    float* tc_tab_inv[8];                 // by NF slot: inverse table
    unsigned* tc_bits;                    // (hit, coin) words of the select pass for one chunk of volumes (bandlimited_tci.cuh)
    size_t tc_bits_bytes;
    int* tc_status;                       // device int: 0, or the code of the bounded wait that expired
    int* tc_status_h;                     // pinned host copy, refreshed (asynchronously) at the end of every call that ran a tensor-core kernel
    // ring of pinned-host / device staging slots for per-call parameter arrays (plan_stage_upload)
    void* stage_h[MVTB_STAGE_SLOTS];
    void* stage_d[MVTB_STAGE_SLOTS];
    size_t stage_cap[MVTB_STAGE_SLOTS];
    cudaEvent_t stage_ev[MVTB_STAGE_SLOTS];
    int stage_next;
    // measurement hooks (mvtb_plan_profile*)
    int profiling;
    int prof_n;
    int prof_kind[MVTB_PROF_MAX];
    cudaEvent_t prof_ev[2 * MVTB_PROF_MAX];
    double prof_ms[MVTB_K_KINDS];
    int prof_cnt[MVTB_K_KINDS];
};

namespace mvtb {
// brackets one launch with events when the plan is recording
struct ProfScope {
    mvtb_plan* p;
    void* stream;
    int slot;
    ProfScope(mvtb_plan* plan, int kind, void* st) : p(plan), stream(st), slot(-1) {
        if (p && p->profiling && p->prof_n < MVTB_PROF_MAX) {
            slot = p->prof_n++;
            p->prof_kind[slot] = kind;
            cudaEventRecord(p->prof_ev[2 * slot], (cudaStream_t)stream);
        }
    }
    ~ProfScope() {
        if (slot >= 0) cudaEventRecord(p->prof_ev[2 * slot + 1], (cudaStream_t)stream);
    }
};
}  // namespace mvtb
