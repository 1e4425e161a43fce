// mt19937.cuh — torch's CPU Mersenne Twister (the stream behind torch.rand on the default generator) on the device,
// and jump-ahead on the host.  Included once, from voxel_ops.cu.
//
// torch.rand(n) in float32 is the sequential MT19937 outputs y mapped to float32((y & 0xFFFFFF) 2^-24).  The generator is
// F2-linear with the degree-19937 characteristic polynomial phi, so the word sequence x[k] obeys x[N + m] = XOR over the
// set bits i of (t^N mod phi) of x[i + m]: a jump of N words is a GF(2) convolution of the first 19937 + 623 words.
//
// Torch layout of a state: the current block W[0..623] of the word sequence z (z[0..623] = W), `next` and `left`.  A
// state as torch leaves it has left = 1 (the next output twists first: z[624]) or left = 625 - next with 1 <= next <= 624
// (the next output is z[next]); pos = left == 1 ? 624 : next is the index in z of the next output.  Below y[m] = z[m + 1]:
// every word of y is a linear function of the 19937-bit state, so y (unlike z, whose z[0] carries 31 free bits) obeys phi.
#include <string.h>

namespace mvtb {
namespace mt {

static const int kN = 624;
static const int kDeg = 19937;
static const int kW64 = 312;                   // 64-bit words of a polynomial of degree < 19937
static const int kY = kDeg + kN - 1;           // words of y a jump reads: y[0 .. 19936 + 623]
// phi = t^19937 + sum t^k over these exponents (135 terms; derived by Berlekamp-Massey in tests/test_mt19937.py)
static const unsigned short kPhiLow[134] = {
    0, 1189, 1416, 1585, 1643, 1870, 2493, 2773, 3000, 3227, 3454, 3681, 3908, 4135, 4362, 4753, 5661, 6337, 6569, 7129,
    7477, 7525, 7583, 7752, 7979, 8206, 9505, 9901, 9969, 10128, 10693, 10761, 10920, 11089, 11147, 11157, 11215, 11321,
    11374, 11384, 11485, 11611, 11712, 11717, 11838, 11881, 11944, 11997, 12277, 12335, 12393, 12504, 12509, 12620, 12673,
    12731, 12736, 12789, 12905, 12958, 12963, 13137, 13185, 13190, 13243, 13301, 13412, 13528, 13533, 13639, 13697, 13760,
    13813, 13866, 14093, 14151, 14209, 14320, 14325, 14436, 14547, 14552, 14605, 14721, 14774, 14779, 14953, 15001, 15006,
    15059, 15117, 15228, 15344, 15349, 15455, 15513, 15576, 15629, 15682, 15909, 15967, 16025, 16136, 16141, 16252, 16363,
    16368, 16421, 16537, 16590, 16595, 16817, 16822, 16875, 16933, 17044, 17160, 17271, 17329, 17445, 17498, 17725, 17783,
    17841, 17952, 18068, 18179, 18237, 18406, 18633, 18691, 18860, 19087, 19314};

__host__ __device__ __forceinline__ uint32_t twist(uint32_t u, uint32_t v) {
    return (((u & 0x80000000u) | (v & 0x7fffffffu)) >> 1) ^ ((v & 1u) ? 0x9908b0dfu : 0u);
}
__host__ __device__ __forceinline__ uint32_t temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    return y ^ (y >> 18);
}
// torch's uniform_real_distribution<float>: 24 random bits times 2^-24 (exact in fp32)
__host__ __device__ __forceinline__ float to_unit(uint32_t y) { return (float)(temper(y) & 0xffffffu) * 5.9604644775390625e-08f; }

// ---------------------------------------------------------------- host: polynomials over GF(2) modulo phi
static inline void xor_at(uint64_t* a, uint64_t w, int bit) {    // a ^= w t^bit
    const int q = bit >> 6, r = bit & 63;
    a[q] ^= w << r;
    if (r) a[q + 1] ^= w >> (64 - r);
}
// a (nw words) mod phi, in place; the words from kW64 on are left zero.  Top down, 64 coefficients at a time:
// t^(19937 + s) = sum_k t^(k + s), which lands strictly below the word being cleared.
static inline void poly_reduce(uint64_t* a, int nw) {
    for (int i = nw - 1; i >= kW64 - 1; --i) {
        uint64_t w = a[i];
        int pos;
        if (i == kW64 - 1) {                    // word 311 holds t^19904 .. t^19967: only bits 33 and up are reduced
            w >>= kDeg - 64 * (kW64 - 1);
            a[i] &= (1ull << (kDeg - 64 * (kW64 - 1))) - 1;
            pos = 0;
        } else {
            a[i] = 0;
            pos = 64 * i - kDeg;
        }
        if (!w) continue;
        for (int k = 0; k < 134; ++k) xor_at(a, w, pos + kPhiLow[k]);
    }
}
static inline uint64_t spread32(uint32_t x) {   // bit i -> bit 2i
    uint64_t v = x;
    v = (v | (v << 16)) & 0x0000ffff0000ffffull;
    v = (v | (v << 8)) & 0x00ff00ff00ff00ffull;
    v = (v | (v << 4)) & 0x0f0f0f0f0f0f0f0full;
    v = (v | (v << 2)) & 0x3333333333333333ull;
    return (v | (v << 1)) & 0x5555555555555555ull;
}
static inline void poly_sqr(uint64_t* a) {
    uint64_t b[2 * kW64];
    for (int j = 0; j < kW64; ++j) {
        b[2 * j] = spread32((uint32_t)a[j]);
        b[2 * j + 1] = spread32((uint32_t)(a[j] >> 32));
    }
    poly_reduce(b, 2 * kW64);
    memcpy(a, b, kW64 * sizeof(uint64_t));
}
// a *= t^k mod phi, in steps of at most 19904 coefficients (a shifted product then fits 2 * kW64 words)
static inline void poly_mul_tk(uint64_t* a, uint64_t k) {
    uint64_t b[2 * kW64];
    while (k) {
        const int s = k > 19904 ? 19904 : (int)k;
        memset(b, 0, sizeof(b));
        for (int j = 0; j < kW64; ++j)
            if (a[j]) xor_at(b, a[j], 64 * j + s);
        poly_reduce(b, 2 * kW64);
        memcpy(a, b, kW64 * sizeof(uint64_t));
        k -= (uint64_t)s;
    }
}
static inline void poly_pow_t(uint64_t e, uint64_t* a) {       // a = t^e mod phi
    memset(a, 0, kW64 * sizeof(uint64_t));
    a[0] = 1;
    for (int b = 63; b >= 0; --b) {
        poly_sqr(a);
        if ((e >> b) & 1) poly_mul_tk(a, 1);
    }
}
static inline void poly_to_words(const uint64_t* a, uint32_t* out) {
    for (int j = 0; j < kW64; ++j) {
        out[2 * j] = (uint32_t)a[j];
        out[2 * j + 1] = (uint32_t)(a[j] >> 32);
    }
}

// ---------------------------------------------------------------- device
static const int kThreads = 256;               // 227 of them run the recurrence
static const int kR = 21;                      // jump outputs per lane: 32 x 21 >= 624, odd so lanes hit distinct banks
static const int kYPad = kY + 32 * kR;         // y in shared memory, zero-padded for the lanes past output 623
static const int kRing = 1024;

// y[0 .. kY) of each segment from 624 consecutive words of its sequence: seed[skip ..] are y's first words
__global__ void __launch_bounds__(kThreads)
k_mt_prefix(const uint32_t* __restrict__ seed, size_t seed_stride, int skip, uint32_t* __restrict__ ybuf) {
    __shared__ uint32_t ring[kRing];
    const uint32_t* w = seed + (size_t)blockIdx.x * seed_stride;
    uint32_t* y = ybuf + (size_t)blockIdx.x * kY;
    for (int j = threadIdx.x; j < kN; j += blockDim.x) {
        ring[j] = w[j];
        if (j >= skip) y[j - skip] = w[j];
    }
    __syncthreads();
    for (int k0 = kN; k0 < kY + skip; k0 += 227) {
        const int k = k0 + (int)threadIdx.x;
        if (threadIdx.x < 227 && k < kY + skip) {
            const uint32_t v = ring[(k - 227) & (kRing - 1)] ^ twist(ring[(k - kN) & (kRing - 1)], ring[(k - kN + 1) & (kRing - 1)]);
            ring[k & (kRing - 1)] = v;
            y[k - skip] = v;
        }
        __syncthreads();
    }
}

// One CTA per (chunk c of this round, segment).  Its first 624 words y[cL .. cL + 623] are the jump of the segment's y by
// table[c] = t^(cL) mod phi; from there the recurrence runs 227 words wide.  Output t of the chunk (global index
// base + cL + t) is y[cL + pos - 1 + t].  With `handoff`, the chunk also writes y[cL + L .. cL + L + 623]: the start of
// the next round's y when c is the round's last chunk.
__global__ void __launch_bounds__(kThreads, 2)
k_mt_chunks(const uint32_t* __restrict__ ybuf, const uint32_t* __restrict__ table, const uint32_t* __restrict__ states,
            size_t state_stride, uint32_t* __restrict__ handoff, float* __restrict__ u, size_t n, size_t L, size_t base,
            int handoff_chunk) {
    MVTB_DYN_SMEM(smem);
    uint32_t* ys = (uint32_t*)smem;             // kYPad
    uint32_t* st = ys + kYPad;                  // 32 * kR
    uint32_t* ring = st + 32 * kR;              // kRing
    const unsigned seg = blockIdx.y, c = blockIdx.x;
    const uint32_t* yg = ybuf + (size_t)seg * kY;
    for (int j = threadIdx.x; j < kYPad; j += blockDim.x) ys[j] = j < kY ? yg[j] : 0u;
    for (int j = threadIdx.x; j < 32 * kR; j += blockDim.x) st[j] = 0u;
    __syncthreads();
    {   // the jump: warp w takes poly words [w * 624 / 8, ...), lane l outputs m = kR l .. kR l + kR - 1
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
        const uint32_t* poly = table + (size_t)c * kN;
        uint32_t acc[kR];
        MVTB_UNROLL
        for (int r = 0; r < kR; ++r) acc[r] = 0u;
        const int m0 = kR * lane;
        for (int pw = warp * kN / nwarps; pw < (warp + 1) * kN / nwarps; ++pw) {
            const uint32_t bits = __ldg(poly + pw);
            if (!bits) continue;
            uint32_t v[32 + kR - 1];
            MVTB_UNROLL
            for (int j = 0; j < 32 + kR - 1; ++j) v[j] = ys[32 * pw + m0 + j];
            MVTB_UNROLL
            for (int j = 0; j < 32; ++j) {
                if ((bits >> j) & 1u) {
                    MVTB_UNROLL
                    for (int r = 0; r < kR; ++r) acc[r] ^= v[j + r];
                }
            }
        }
        MVTB_UNROLL
        for (int r = 0; r < kR; ++r) atomicXor(st + m0 + r, acc[r]);
    }
    __syncthreads();
    const int pos = (int)states[(size_t)seg * state_stride + kN + 1] == 1 ? kN : (int)states[(size_t)seg * state_stride + kN];
    const size_t first = base + (size_t)c * L;  // global index of the chunk's output 0
    const size_t cnt = first + L <= n ? L : n - first;
    float* uo = u + (size_t)seg * n + first;
    const long long out_end = (long long)pos - 1 + (long long)cnt;    // local y index past the chunk's last output
    const long long end = ((int)c == handoff_chunk && out_end < (long long)L + kN) ? (long long)L + kN : out_end;
    for (int j = threadIdx.x; j < kN; j += blockDim.x) {
        const uint32_t v = st[j];
        ring[j] = v;
        if (j >= pos - 1 && j < out_end) uo[j - (pos - 1)] = to_unit(v);
    }
    __syncthreads();
    for (long long j0 = kN; j0 < end; j0 += 227) {
        const long long j = j0 + threadIdx.x;
        if (threadIdx.x < 227 && j < end) {
            const uint32_t v = ring[(j - 227) & (kRing - 1)] ^ twist(ring[(j - kN) & (kRing - 1)], ring[(j - kN + 1) & (kRing - 1)]);
            ring[j & (kRing - 1)] = v;
            if (j < out_end) uo[j - (pos - 1)] = to_unit(v);
            if ((int)c == handoff_chunk && j >= (long long)L) handoff[(size_t)seg * kN + (size_t)(j - (long long)L)] = v;
        }
        __syncthreads();
    }
}

}  // namespace mt
}  // namespace mvtb

// ---------------------------------------------------------------- C entries
extern "C" int mvtb_mt19937_jump_poly(uint64_t n, uint32_t* poly_out) {
    if (!poly_out) { mvtb::set_error("mt19937_jump_poly: null output"); return MVTB_EINVAL; }
    uint64_t a[mvtb::mt::kW64];
    mvtb::mt::poly_pow_t(n, a);
    mvtb::mt::poly_to_words(a, poly_out);
    return MVTB_OK;
}

extern "C" int mvtb_mt19937_chunk_table(uint64_t chunk_len, int n_chunks, uint32_t* table_out) {
    if (!table_out || n_chunks < 1 || chunk_len < (uint64_t)mvtb::mt::kN || chunk_len > (1ull << 40)) {
        mvtb::set_error("mt19937_chunk_table: bad argument (chunk_len=%llu must be in [624, 2^40], n_chunks=%d >= 1)",
                        (unsigned long long)chunk_len, n_chunks);
        return MVTB_EINVAL;
    }
    uint64_t a[mvtb::mt::kW64];
    memset(a, 0, sizeof(a));
    a[0] = 1;
    for (int c = 0; c < n_chunks; ++c) {
        mvtb::mt::poly_to_words(a, table_out + (size_t)c * mvtb::mt::kN);
        if (c + 1 < n_chunks) mvtb::mt::poly_mul_tk(a, chunk_len);
    }
    return MVTB_OK;
}

extern "C" int mvtb_mt19937_advance(const uint32_t* poly, uint64_t n, uint32_t* state, int32_t* next, int32_t* left) {
    using namespace mvtb::mt;
    if (!state || !next || !left) { mvtb::set_error("mt19937_advance: null argument"); return MVTB_EINVAL; }
    const int nx = *next, lf = *left;
    if (!(lf == 1 && nx >= 0 && nx <= kN) && !(nx >= 1 && nx <= kN && lf == kN + 1 - nx)) {
        mvtb::set_error("mt19937_advance: next=%d left=%d is not a state torch leaves (left = 1, or left = 625 - next with "
                        "1 <= next <= 624)", nx, lf);
        return MVTB_EINVAL;
    }
    if (n >= (uint64_t)kN + 1 && !poly) { mvtb::set_error("mt19937_advance: n=%llu needs the jump polynomial",
                                                          (unsigned long long)n); return MVTB_EINVAL; }
    if (n > (1ull << 62)) { mvtb::set_error("mt19937_advance: n=%llu too large", (unsigned long long)n); return MVTB_EINVAL; }
    if (n == 0) return MVTB_OK;
    const uint64_t pos = lf == 1 ? kN : (uint64_t)nx;
    const uint64_t P = pos + n, q = (P - 1) / kN, k = P - kN * q;    // the last draw is z[P - 1], in block q at k - 1
    if (q > 0) {
        // w[j] = z[b + j] for a window starting at b, extended by the recurrence to the new block z[624q .. 624q + 623]
        uint32_t w[3 * kN + 2];                 // at most 624q - b + 624 <= 1871 words
        uint64_t b = 0;
        if (n < (uint64_t)kN + 1) {
            memcpy(w, state, kN * sizeof(uint32_t));
        } else {                                // poly = t^(n - 625): z[n - 624 + m] = y[n - 625 + m] = XOR_i c_i y[i + m]
            uint32_t z[kY + 1];
            memcpy(z, state, kN * sizeof(uint32_t));
            for (int j = kN; j <= kY; ++j) z[j] = z[j - 227] ^ twist(z[j - kN], z[j - kN + 1]);
            uint32_t acc[kN];
            memset(acc, 0, sizeof(acc));
            for (int pw = 0; pw < kN; ++pw) {
                uint32_t bits = poly[pw];
                while (bits) {
                    const int i = 32 * pw + __builtin_ctz(bits);
                    bits &= bits - 1;
                    if (i >= kDeg) break;
                    const uint32_t* src = z + 1 + i;
                    for (int m = 0; m < kN; ++m) acc[m] ^= src[m];
                }
            }
            memcpy(w, acc, sizeof(acc));
            b = n - kN;
        }
        const int hi = (int)(kN * q - b) + kN;  // window words needed
        for (int j = kN; j < hi; ++j) w[j] = w[j - 227] ^ twist(w[j - kN], w[j - kN + 1]);
        memcpy(state, w + (kN * q - b), kN * sizeof(uint32_t));
    }
    *next = (int32_t)k;
    *left = (int32_t)(kN + 1 - k);
    return MVTB_OK;
}

extern "C" size_t mvtb_mt19937_workspace_bytes(int n_segments) {
    return n_segments > 0 ? (size_t)n_segments * (mvtb::mt::kY + mvtb::mt::kN) * sizeof(uint32_t) : 0;
}

extern "C" int mvtb_mt19937_uniform_f32(float* u, size_t n, int n_segments, const uint32_t* states, const uint32_t* table,
                                        uint64_t chunk_len, int n_chunks, void* workspace, void* stream) {
    using namespace mvtb::mt;
    if (n_segments < 0 || n_segments > 65535) { mvtb::set_error("mt19937_uniform: n_segments=%d", n_segments); return MVTB_EINVAL; }
    if (n_chunks < 1 || chunk_len < (uint64_t)kN || chunk_len > (1ull << 40)) {
        mvtb::set_error("mt19937_uniform: chunk_len=%llu must be in [624, 2^40] and n_chunks=%d >= 1",
                        (unsigned long long)chunk_len, n_chunks);
        return MVTB_EINVAL;
    }
    if (n == 0 || n_segments == 0) return MVTB_OK;
    if (!u || !states || !table || !workspace) { mvtb::set_error("mt19937_uniform: null argument"); return MVTB_EINVAL; }
    if (n > (1ull << 40)) { mvtb::set_error("mt19937_uniform: n=%llu too large", (unsigned long long)n); return MVTB_EINVAL; }
    const size_t state_stride = MVTB_MT_STATE_WORDS;
    uint32_t* ybuf = (uint32_t*)workspace;
    uint32_t* hand = ybuf + (size_t)n_segments * kY;
    const size_t smem = (size_t)(kYPad + 32 * kR + kRing) * sizeof(uint32_t);
    MVTB_CUDA(cudaFuncSetAttribute(k_mt_chunks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint64_t nch = (n + chunk_len - 1) / chunk_len;
    const uint64_t rounds = (nch + n_chunks - 1) / n_chunks;
    for (uint64_t r = 0; r < rounds; ++r) {
        if (r == 0)
            MVTB_LAUNCH(k_mt_prefix, dim3((unsigned)n_segments), dim3(kThreads), 0, stream, states, state_stride, 1, ybuf);
        else
            MVTB_LAUNCH(k_mt_prefix, dim3((unsigned)n_segments), dim3(kThreads), 0, stream, (const uint32_t*)hand, (size_t)kN, 0, ybuf);
        const uint64_t c0 = r * (uint64_t)n_chunks;
        const unsigned active = (unsigned)(nch - c0 < (uint64_t)n_chunks ? nch - c0 : (uint64_t)n_chunks);
        const int handoff_chunk = r + 1 < rounds ? n_chunks - 1 : -1;
        MVTB_LAUNCH(k_mt_chunks, dim3(active, (unsigned)n_segments), dim3(kThreads), smem, stream, ybuf, table, states, state_stride,
                    hand, u, n, (size_t)chunk_len, (size_t)(c0 * chunk_len), handoff_chunk);
        MVTB_CUDA(cudaGetLastError());
    }
    return MVTB_OK;
}
