// bandlimited_quad.cuh — H-axis kernels of the band-limited path for H % 4 == 0 (240, 128, 64, ...).
//
// One more level of symmetry than the pair folding: rows h, H-h, H/2-h, H/2+h share
// cos_f(h), sin_f(h) up to signs that depend only on the parity of f:
//     cos_f(H-h) =  cos_f(h)            sin_f(H-h) = -sin_f(h)
//     cos_f(H/2-h) = (-1)^f cos_f(h)    sin_f(H/2-h) = -(-1)^f ... = (-1)^(f+1) (-sin_f(h)) ...
// worked out below.  Four rows are produced / consumed per table row, which halves the FMAs and the
// shared-memory table traffic per voxel relative to k_bl_fwd_h / k_bl_inv_h.  Included by bandlimited.cu.
// (no namespace here: included inside namespace mvtb)
#pragma once

__device__ __forceinline__ float2 add2(float2 a, float2 b) {
#ifdef MVTB_EMU
    return make_float2(a.x + b.x, a.y + b.y);
#else
    return __fadd2_rn(a, b);
#endif
}

// ------------------------------------------------------------------ forward, quads
// a = x[h], b = x[H-h], c = x[H/2-h], d = x[H/2+h]:
//   f even:  re += (a+b+c+d) cos,  im -= (a-b-c+d) sin
//   f odd :  re += (a+b-c-d) cos,  im -= (a-b+c-d) sin
template <int NF, int CPT, int U, int MINB>
__global__ void __launch_bounds__(256, MINB)
k_bl_fwd_h4(const float* __restrict__ x, cf* __restrict__ Y, BlGeom g, int n_cblocks) {
    constexpr int NT = BlDims<NF>::NT;
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
        if (!ok[k]) col[k] = g.NC - 1;
    }
    const int H = g.H, H2 = H / 2, H4 = H / 4;
    float2 acc[CPT][NF];                                // (re, im)
    {
        // rows 0 and H/2 (cos = 1 / (-1)^f, sin = 0), then the pair H/4, 3H/4 with table row H/4
        float2 cs[NF];
        bl_row<NF>(sc + H4 * NT, cs);
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) {
            const float x0 = ld_stream(xv + col[k]);
            const float xn = ld_stream(xv + (long long)H2 * g.NC + col[k]);
            const float a = ld_stream(xv + (long long)H4 * g.NC + col[k]);
            const float b = ld_stream(xv + (long long)(H - H4) * g.NC + col[k]);
            const float2 eo = make_float2(a + b, b - a);
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) acc[k][f] = fma2(eo, cs[f], make_float2(x0 + ((f & 1) ? -xn : xn), 0.f));
        }
    }
    const float* pa[CPT];   // row h        (ascending)
    const float* pb[CPT];   // row H-h      (descending)
    const float* pc[CPT];   // row H/2-h    (descending)
    const float* pd[CPT];   // row H/2+h    (ascending)
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) {
        pa[k] = xv + g.NC + col[k];
        pb[k] = xv + (long long)(H - 1) * g.NC + col[k];
        pc[k] = xv + (long long)(H2 - 1) * g.NC + col[k];
        pd[k] = xv + (long long)(H2 + 1) * g.NC + col[k];
    }
    const int nq = H4 - 1;
    int h = 1;
    for (; h + U - 1 <= nq; h += U) {                   // 4*U*CPT independent coalesced loads in flight
        float a[U][CPT], b[U][CPT], c[U][CPT], d[U][CPT];
        MVTB_UNROLL
        for (int u = 0; u < U; ++u) {
            MVTB_UNROLL
            for (int k = 0; k < CPT; ++k) {
                a[u][k] = ld_stream(pa[k] + (long long)u * g.NC);
                b[u][k] = ld_stream(pb[k] - (long long)u * g.NC);
                c[u][k] = ld_stream(pc[k] - (long long)u * g.NC);
                d[u][k] = ld_stream(pd[k] + (long long)u * g.NC);
            }
        }
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) {
            pa[k] += (long long)U * g.NC; pd[k] += (long long)U * g.NC;
            pb[k] -= (long long)U * g.NC; pc[k] -= (long long)U * g.NC;
        }
        MVTB_UNROLL
        for (int u = 0; u < U; ++u) {
            float2 cs[NF];
            bl_row<NF>(sc + (h + u) * NT, cs);
            MVTB_UNROLL
            for (int k = 0; k < CPT; ++k) {
                const float s1 = a[u][k] + b[u][k], s2 = c[u][k] + d[u][k];
                const float d1 = a[u][k] - b[u][k], d2 = c[u][k] - d[u][k];
                const float2 ev = make_float2(s1 + s2, d2 - d1);        // (ee, -oe),  oe = d1 - d2
                const float2 od = make_float2(s1 - s2, -(d1 + d2));     // (eo, -oo),  oo = d1 + d2
                MVTB_UNROLL
                for (int f = 0; f < NF; ++f) acc[k][f] = fma2((f & 1) ? od : ev, cs[f], acc[k][f]);
            }
        }
    }
    for (; h <= nq; ++h) {
        float2 cs[NF];
        bl_row<NF>(sc + h * NT, cs);
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) {
            const float a = ld_stream(pa[k]), b = ld_stream(pb[k]), c = ld_stream(pc[k]), d = ld_stream(pd[k]);
            pa[k] += g.NC; pd[k] += g.NC; pb[k] -= g.NC; pc[k] -= g.NC;
            const float s1 = a + b, s2 = c + d, d1 = a - b, d2 = c - d;
            const float2 ev = make_float2(s1 + s2, d2 - d1);
            const float2 od = make_float2(s1 - s2, -(d1 + d2));
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) acc[k][f] = fma2((f & 1) ? od : ev, cs[f], acc[k][f]);
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

// ------------------------------------------------------------------ inverse, quads
// With (Pe, Qe) = sum over even f of (a_f cos_f(h), b_f sin_f(h)) and (Po, Qo) over odd f:
//   out[h]     = (Pe+Po) - (Qe+Qo)        out[H-h]   = (Pe+Po) + (Qe+Qo)
//   out[H/2-h] = (Pe-Po) + (Qe-Qo)        out[H/2+h] = (Pe-Po) - (Qe-Qo)
// A plane wave with frequency f_s joins the even or the odd sums according to the parity of f_s.
template <int NF, int CPT>
__global__ void __launch_bounds__(256, 2)
k_bl_inv_h4(const cf* __restrict__ Y, float* __restrict__ out, BlGeom g, int n_cblocks,
            const BlVol* __restrict__ vols, int vol_base, int shared_desc,
            float* __restrict__ minmax, int vols_per_sample) {
    constexpr int NT = BlDims<NF>::NT;
    MVTB_DYN_SMEM(smem_raw);
    const int H = g.H, H2 = H / 2, H4 = H / 4;
    float* sc = (float*)smem_raw;
    cf* seh = (cf*)(sc + (H2 + 1) * NT);                // [MVTB_BL_MAX_PW][H/2+1] exp(+2 pi i fh h / H)
    const int tid = threadIdx.x;
    const int vol = blockIdx.x / n_cblocks;
    const BlVol& bv = vols[shared_desc ? 0 : vol_base + vol];
    const int npw = bv.npw;
    bl_load_table<NF>(sc, g.tabC[2], g.tabS[2], H, tid, blockDim.x);
    for (int e = tid; e < MVTB_BL_MAX_PW * (H2 + 1); e += blockDim.x) {
        const int s = e / (H2 + 1), h = e - s * (H2 + 1);
        float c_ = 0.f, s_ = 0.f;
        if (s < npw) bl_unit(bv.pw[s].fh, h, H, &c_, &s_);
        seh[e] = cmk(c_, s_);
    }
    __syncthreads();
    bool podd[MVTB_BL_MAX_PW];
    MVTB_UNROLL
    for (int s = 0; s < MVTB_BL_MAX_PW; ++s) podd[s] = s < npw && (bv.pw[s].fh & 1);

    const long long c0 = (long long)(blockIdx.x - (long long)vol * n_cblocks) * (blockDim.x * CPT) + tid;
    bool ok[CPT];
    long long col[CPT];
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) {
        col[k] = c0 + (long long)k * blockDim.x;
        ok[k] = col[k] < g.NC;
        if (!ok[k]) col[k] = g.NC - 1;
    }
    float lo = __int_as_float(0x7f800000), hi = __int_as_float((int)0xff800000u);
    float2 y2[CPT][NF];
    float2 E[CPT][MVTB_BL_MAX_PW];
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
    // rows 0, H/2 and the pair H/4, 3H/4
    {
        float2 cs[NF];
        bl_row<NF>(sc + H4 * NT, cs);
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) {
            float v0 = 0.f, vn = 0.f;
            float2 pq = make_float2(0.f, 0.f);
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                v0 += y2[k][f].x;
                vn += (f & 1) ? -y2[k][f].x : y2[k][f].x;
                pq = fma2(y2[k][f], cs[f], pq);
            }
            MVTB_UNROLL
            for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
                const cf e2 = seh[s * (H2 + 1) + H2], e4 = seh[s * (H2 + 1) + H4];
                v0 += E[k][s].x;
                vn += E[k][s].x * e2.x - E[k][s].y * e2.y;
                pq = fma2(E[k][s], e4, pq);
            }
            const float vq = pq.x - pq.y, v3q = pq.x + pq.y;
            lo = fminf(fminf(lo, v0), fminf(vn, fminf(vq, v3q)));
            hi = fmaxf(fmaxf(hi, v0), fmaxf(vn, fmaxf(vq, v3q)));
            if (ok[k]) {
                st_stream(ov + col[k], v0);
                st_stream(ov + (long long)H2 * g.NC + col[k], vn);
                st_stream(ov + (long long)H4 * g.NC + col[k], vq);
                st_stream(ov + (long long)(H - H4) * g.NC + col[k], v3q);
            }
        }
    }
    float* pa[CPT];
    float* pb[CPT];
    float* pc[CPT];
    float* pd[CPT];
    MVTB_UNROLL
    for (int k = 0; k < CPT; ++k) {
        pa[k] = ov + g.NC + col[k];
        pb[k] = ov + (long long)(H - 1) * g.NC + col[k];
        pc[k] = ov + (long long)(H2 - 1) * g.NC + col[k];
        pd[k] = ov + (long long)(H2 + 1) * g.NC + col[k];
    }
    const int nq = H4 - 1;
    for (int h = 1; h <= nq; ++h) {
        float2 cs[NF];
        bl_row<NF>(sc + h * NT, cs);
        float2 eh[MVTB_BL_MAX_PW];
        MVTB_UNROLL
        for (int s = 0; s < MVTB_BL_MAX_PW; ++s) eh[s] = seh[s * (H2 + 1) + h];
        MVTB_UNROLL
        for (int k = 0; k < CPT; ++k) {
            float2 pe = make_float2(0.f, 0.f), po = make_float2(0.f, 0.f);       // (Pe, Qe), (Po, Qo)
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                if (f & 1) po = fma2(y2[k][f], cs[f], po);
                else pe = fma2(y2[k][f], cs[f], pe);
            }
            MVTB_UNROLL
            for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
                if (podd[s]) po = fma2(E[k][s], eh[s], po);
                else pe = fma2(E[k][s], eh[s], pe);
            }
            const float2 sm = add2(pe, po);                                       // (Pe+Po, Qe+Qo)
            const float2 df = add2(pe, make_float2(-po.x, -po.y));                // (Pe-Po, Qe-Qo)
            const float v1 = sm.x - sm.y, v2 = sm.x + sm.y, v3 = df.x + df.y, v4 = df.x - df.y;
            lo = fminf(fminf(lo, fminf(v1, v2)), fminf(v3, v4));
            hi = fmaxf(fmaxf(hi, fmaxf(v1, v2)), fmaxf(v3, v4));
            if (ok[k]) { st_stream(pa[k], v1); st_stream(pb[k], v2); st_stream(pc[k], v3); st_stream(pd[k], v4); }
            pa[k] += g.NC; pd[k] += g.NC;
            pb[k] -= g.NC; pc[k] -= g.NC;
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

// ------------------------------------------------------------------ inverse, quads, two ADJACENT columns per thread
// Same arithmetic as k_bl_inv_h4 for W*D even: the two columns of a thread are neighbours, so the rows of Y
// arrive as one 16-byte load and every output row leaves as one 8-byte store (half the address arithmetic and
// store instructions).  Index math is 32-bit (a volume has < 2^31 voxels; |f| n < 2^31).
__device__ __forceinline__ void bl_unit32(int f, int n, int N, float* c, float* s) {
    int m = (f * n) % N;
    if (m < 0) m += N;
    sincospif(2.0f * (float)m / (float)N, s, c);
}

// How the output rows leave: 0 = streaming (evict-first: the volume is not read again by this library), 1 = plain
// write-back (the fused inverse + select kernel touches the lines again while they are in L2), 2 = plain with an
// L2 evict_last policy.
#ifdef MVTB_EMU
template <int STORE>
__device__ __forceinline__ void st_out2(float* p, float a, float b, unsigned long long) { p[0] = a; p[1] = b; }
__device__ __forceinline__ unsigned long long l2_policy_evict_last() { return 0; }
#else
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
template <int STORE>
__device__ __forceinline__ void st_out2(float* p, float a, float b, unsigned long long pol) {
    if (STORE == 0) __stcs((float2*)p, make_float2(a, b));
    else if (STORE == 1) *(float2*)p = make_float2(a, b);
    else asm volatile("st.global.L2::cache_hint.v2.f32 [%0], {%1, %2}, %3;" ::"l"(p), "f"(a), "f"(b), "l"(pol) : "memory");
}
#endif

__device__ __forceinline__ float min3(float a, float b, float c) { return fminf(fminf(a, b), c); }
__device__ __forceinline__ float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// The rows of quads q0 .. q1-1 (and, when `special`, rows 0, H/2, H/4, 3H/4) of this thread's two adjacent columns.
// sc: (cos, sin) table rows 0 .. H/2; seh: [MVTB_BL_MAX_PW][H/2+1] exp(+2 pi i fh h / H) of this volume's plane waves;
// yv / ov: this thread's first column in the volume's Y rows / output rows.
template <int NF, int STORE>
__device__ __forceinline__ void bl_inv_h4v_cols(const float* __restrict__ sc, const cf* __restrict__ seh, const cf* __restrict__ yv,
                                                float* __restrict__ ov, const BlGeom& g, const BlVol& bv, int col,
                                                bool ok, int q0, int q1, bool special, unsigned long long pol,
                                                float& lo, float& hi) {
    constexpr int NT = BlDims<NF>::NT;
    const int H = g.H, H2 = H / 2, H4 = H / 4;
    const int NC = (int)g.NC;
    const int npw = bv.npw;
    bool podd[MVTB_BL_MAX_PW];
    MVTB_UNROLL
    for (int s = 0; s < MVTB_BL_MAX_PW; ++s) podd[s] = s < npw && (bv.pw[s].fh & 1);
    float2 y2[2][NF];
    float2 E[2][MVTB_BL_MAX_PW];
    MVTB_UNROLL
    for (int f = 0; f < NF; ++f) {
        const float4 y = *reinterpret_cast<const float4*>(yv + (size_t)f * NC);
        const float cfw = f == 0 ? 1.f : 2.f;
        y2[0][f] = make_float2(cfw * y.x, cfw * y.y);
        y2[1][f] = make_float2(cfw * y.z, cfw * y.w);
    }
    MVTB_UNROLL
    for (int k = 0; k < 2; ++k) {
        const int w = (col + k) / g.D, d = (col + k) - w * g.D;
        MVTB_UNROLL
        for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
            E[k][s] = make_float2(0.f, 0.f);
            if (s < npw) {
                float cw, sw, cd, sd;
                bl_unit32(bv.pw[s].fw, w, g.W, &cw, &sw);
                bl_unit32(bv.pw[s].fd, d, g.D, &cd, &sd);
                const float amp = bv.pw[s].amp;
                E[k][s] = make_float2(amp * (cw * cd - sw * sd), amp * (sw * cd + cw * sd));
            }
        }
    }
    if (special) {
        float2 cs[NF];
        bl_row<NF>(sc + H4 * NT, cs);
        float v0[2], vn[2], vq[2], v3q[2];
        MVTB_UNROLL
        for (int k = 0; k < 2; ++k) {
            v0[k] = 0.f; vn[k] = 0.f;
            float2 pq = make_float2(0.f, 0.f);
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                v0[k] += y2[k][f].x;
                vn[k] += (f & 1) ? -y2[k][f].x : y2[k][f].x;
                pq = fma2(y2[k][f], cs[f], pq);
            }
            MVTB_UNROLL
            for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
                const cf e2 = seh[s * (H2 + 1) + H2], e4 = seh[s * (H2 + 1) + H4];
                v0[k] += E[k][s].x;
                vn[k] += E[k][s].x * e2.x - E[k][s].y * e2.y;
                pq = fma2(E[k][s], e4, pq);
            }
            vq[k] = pq.x - pq.y; v3q[k] = pq.x + pq.y;
            lo = fminf(fminf(lo, v0[k]), fminf(vn[k], fminf(vq[k], v3q[k])));
            hi = fmaxf(fmaxf(hi, v0[k]), fmaxf(vn[k], fmaxf(vq[k], v3q[k])));
        }
        if (ok) {
            st_out2<STORE>(ov, v0[0], v0[1], pol);
            st_out2<STORE>(ov + (size_t)H2 * NC, vn[0], vn[1], pol);
            st_out2<STORE>(ov + (size_t)H4 * NC, vq[0], vq[1], pol);
            st_out2<STORE>(ov + (size_t)(H - H4) * NC, v3q[0], v3q[1], pol);
        }
    }
    float* pa = ov + (size_t)q0 * NC;
    float* pb = ov + (size_t)(H - q0) * NC;
    float* pc = ov + (size_t)(H2 - q0) * NC;
    float* pd = ov + (size_t)(H2 + q0) * NC;
    for (int h = q0; h < q1; ++h) {
        float2 cs[NF];
        bl_row<NF>(sc + h * NT, cs);
        float2 eh[MVTB_BL_MAX_PW];
        MVTB_UNROLL
        for (int s = 0; s < MVTB_BL_MAX_PW; ++s) eh[s] = seh[s * (H2 + 1) + h];
        float v1[2], v2[2], v3[2], v4[2];
        MVTB_UNROLL
        for (int k = 0; k < 2; ++k) {
            float2 pe = make_float2(0.f, 0.f), po = make_float2(0.f, 0.f);
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                if (f & 1) po = fma2(y2[k][f], cs[f], po);
                else pe = fma2(y2[k][f], cs[f], pe);
            }
            MVTB_UNROLL
            for (int s = 0; s < MVTB_BL_MAX_PW; ++s) {
                if (podd[s]) po = fma2(E[k][s], eh[s], po);
                else pe = fma2(E[k][s], eh[s], pe);
            }
            const float2 sm = add2(pe, po);
            const float2 df = add2(pe, make_float2(-po.x, -po.y));
            v1[k] = sm.x - sm.y; v2[k] = sm.x + sm.y; v3[k] = df.x + df.y; v4[k] = df.x - df.y;
            lo = min3(lo, fminf(v1[k], v2[k]), fminf(v3[k], v4[k]));
            hi = max3(hi, fmaxf(v1[k], v2[k]), fmaxf(v3[k], v4[k]));
        }
        if (ok) {
            st_out2<STORE>(pa, v1[0], v1[1], pol);
            st_out2<STORE>(pb, v2[0], v2[1], pol);
            st_out2<STORE>(pc, v3[0], v3[1], pol);
            st_out2<STORE>(pd, v4[0], v4[1], pol);
        }
        pa += NC; pd += NC;
        pb -= NC; pc -= NC;
    }
}

// CTA-wide (min, max) -> one ordered-int atomic pair on mm[0], mm[1] by thread 0; every thread passes one __syncthreads
__device__ __forceinline__ void bl_block_minmax(float lo, float hi, float* mm) {
    __shared__ float s_lo[32], s_hi[32];
    const int tid = threadIdx.x;
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
            bl_atomic_min(mm, lo);
            bl_atomic_max(mm + 1, hi);
        }
    }
}

template <int NF>
__global__ void __launch_bounds__(256, 2)
k_bl_inv_h4v(const cf* __restrict__ Y, float* __restrict__ out, BlGeom g, int n_cblocks,
             const BlVol* __restrict__ vols, int vol_base, int shared_desc,
             float* __restrict__ minmax, int vols_per_sample) {
    constexpr int NT = BlDims<NF>::NT;
    MVTB_DYN_SMEM(smem_raw);
    const int H = g.H, H2 = H / 2, H4 = H / 4;
    const int NC = (int)g.NC;
    float* sc = (float*)smem_raw;
    cf* seh = (cf*)(sc + (H2 + 1) * NT);
    const int tid = threadIdx.x;
    const int vol = blockIdx.x / n_cblocks;
    const BlVol& bv = vols[shared_desc ? 0 : vol_base + vol];
    const int npw = bv.npw;
    bl_load_table<NF>(sc, g.tabC[2], g.tabS[2], H, tid, blockDim.x);
    for (int e = tid; e < MVTB_BL_MAX_PW * (H2 + 1); e += blockDim.x) {
        const int s = e / (H2 + 1), h = e - s * (H2 + 1);
        float c_ = 0.f, s_ = 0.f;
        if (s < npw) bl_unit32(bv.pw[s].fh, h, H, &c_, &s_);
        seh[e] = cmk(c_, s_);
    }
    __syncthreads();

    int col = ((blockIdx.x - vol * n_cblocks) * blockDim.x + tid) * 2;
    const bool ok = col < NC;
    if (!ok) col = NC - 2;
    float lo = __int_as_float(0x7f800000), hi = __int_as_float((int)0xff800000u);
    bl_inv_h4v_cols<NF, 0>(sc, seh, Y + (size_t)vol * NF * NC + col, out + (size_t)vol * H * NC + col, g, bv, col, ok,
                           1, H4, true, 0ull, lo, hi);
    if (minmax != nullptr) bl_block_minmax(lo, hi, minmax + 2 * ((vol_base + vol) / vols_per_sample));
}

// ------------------------------------------------------------------ forward, quads, cp.async staging ring
// k_bl_fwd_h4 is bound by load latency: its bytes in flight are limited by registers (16 loads x 24 warps).
// Here the four rows of a quad for the CTA's 256 columns (4 KB) are copied global -> shared with one 16-byte
// cp.async (LDGSTS) per thread, kBlStages quads ahead, so ~28 KB per CTA are in flight without holding
// registers; the threads then read their own column from shared memory.  Needs W*D % 4 == 0 and a 16-byte
// aligned input (else the register-staged kernel runs).
static const int kBlStages = 8;

// cp_async16 / cp_async_commit / cp_async_wait: mvtb_common.cuh

// PRE: the intensity prologue map y = x != 0 ? a x + b : t of the volume (abt[3 vol ..]) is applied to every value read
template <int NF, bool PRE>
__global__ void __launch_bounds__(256, 3)
k_bl_fwd_h4a(const float* __restrict__ x, cf* __restrict__ Y, BlGeom g, int n_cblocks, const float* __restrict__ abt) {
    constexpr int NT = BlDims<NF>::NT, S = kBlStages;
    MVTB_DYN_SMEM(smem_raw);
    const int H = g.H, H2 = H / 2, H4 = H / 4;
    float* sc = (float*)smem_raw;                       // (cos, sin) rows 0 .. H/2
    float* ring = sc + (H2 + 1) * NT;                   // [S][4][256] floats
    const int tid = threadIdx.x;
    const long long vol = blockIdx.x / n_cblocks;
    const long long c0 = (long long)(blockIdx.x - vol * n_cblocks) * 256;
    const float* xv = x + vol * H * g.NC;
    float pa_ = 1.f, pb_ = 0.f, pt_ = 0.f;
    if (PRE) { pa_ = __ldg(abt + 3 * vol); pb_ = __ldg(abt + 3 * vol + 1); pt_ = __ldg(abt + 3 * vol + 2); }
#define MVTB_PRE(v) (PRE ? ((v) != 0.f ? fmaf(pa_, (v), pb_) : pt_) : (v))

    // this thread's 16-byte piece of every stage: row r of the quad, columns c0 + 4 j .. + 3
    const int r = tid >> 6, j = tid & 63;
    const bool piece_ok = c0 + 4 * j < g.NC;
    const float* src0;                                  // row of quad q = 1 for this thread's r
    long long step;                                     // rows advance by +-NC per quad
    if (r == 0)      { src0 = xv + g.NC;                          step = g.NC; }
    else if (r == 1) { src0 = xv + (long long)(H - 1) * g.NC;     step = -g.NC; }
    else if (r == 2) { src0 = xv + (long long)(H2 - 1) * g.NC;    step = -g.NC; }
    else             { src0 = xv + (long long)(H2 + 1) * g.NC;    step = g.NC; }
    src0 += c0 + 4 * j;
    float* dst0 = ring + r * 256 + 4 * j;
    const smem_addr_t dst_base = smem_addr(dst0);       // converted once; the loop does 32-bit slot arithmetic
    const int nq = H4 - 1;
    for (int q = 1; q < S; ++q) {                       // quads 1 .. S-1 in flight before the loop
        if (q <= nq && piece_ok) cp_async16_at(dst_base + (q - 1) * 4096, src0 + (long long)(q - 1) * step);
        cp_async_commit();
    }
    const float* src_next = src0 + (long long)(S - 1) * step;   // row of quad q - 1 + S, advanced every iteration
    int slot = 0;                                               // (q - 1) % S
    bl_load_table<NF>(sc, g.tabC[2], g.tabS[2], H, tid, blockDim.x);

    const long long col = c0 + tid;
    const bool ok = col < g.NC;
    const long long colc = ok ? col : g.NC - 1;
    float2 acc[NF];
    __syncthreads();                                    // table ready
    {
        float2 cs[NF];
        bl_row<NF>(sc + H4 * NT, cs);
        const float x0 = MVTB_PRE(ld_stream(xv + colc));
        const float xn = MVTB_PRE(ld_stream(xv + (long long)H2 * g.NC + colc));
        const float a = MVTB_PRE(ld_stream(xv + (long long)H4 * g.NC + colc));
        const float b = MVTB_PRE(ld_stream(xv + (long long)(H - H4) * g.NC + colc));
        const float2 eo = make_float2(a + b, b - a);
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) acc[f] = fma2(eo, cs[f], make_float2(x0 + ((f & 1) ? -xn : xn), 0.f));
    }
    for (int q = 1; q <= nq; ++q) {
        cp_async_wait<S - 2>();                         // this thread's piece of quad q has landed
        __syncthreads();                                // ... everyone's has, and stage(q-1) is no longer being read
        {
            // refill the stage read in the previous iteration: quad q - 1 + S goes to slot (q - 2) mod S
            const int prev = slot == 0 ? S - 1 : slot - 1;
            if (q - 1 + S <= nq && piece_ok) cp_async16_at(dst_base + prev * 4096, src_next);
            cp_async_commit();
            src_next += step;
        }
        const float* st = ring + slot * 1024 + tid;
        slot = slot + 1 == S ? 0 : slot + 1;
        const float a = MVTB_PRE(st[0]), b = MVTB_PRE(st[256]), c = MVTB_PRE(st[512]), d = MVTB_PRE(st[768]);
        float2 cs[NF];
        bl_row<NF>(sc + q * NT, cs);
        const float s1 = a + b, s2 = c + d, d1 = a - b, d2 = c - d;
        const float2 ev = make_float2(s1 + s2, d2 - d1);
        const float2 od = make_float2(s1 - s2, -(d1 + d2));
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) acc[f] = fma2((f & 1) ? od : ev, cs[f], acc[f]);
    }
    if (ok) {
        cf* yv = Y + vol * NF * g.NC + col;
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) yv[(long long)f * g.NC] = acc[f];
    }
#undef MVTB_PRE
}

// ------------------------------------------------------------------ W axis, D axis and pointwise stage in one kernel
// k_bl_fwd_w + k_bl_mid + k_bl_inv_w for one (volume, f_h) plane per CTA: thread d streams its column of
// Y[f_h][.][d] once (pair folding over w, 16 loads in flight), the 2F+1 W-bins of all columns meet in shared
// memory for the D-axis DFT and the pointwise stage, and the same thread expands its column back and overwrites
// Y in place.  The G workspace and two launches disappear; the plane is read once and written once.
// CTAs per SM: 4 up to NF = 16 (96 registers), 3 at NF = 20, 2 beyond (the 4 NF accumulator registers dominate)
#define MVTB_MIDW_MINB(NF) ((NF) <= 16 ? 4 : ((NF) <= 20 ? 3 : 2))
template <int NF>
__global__ void __launch_bounds__(160, MVTB_MIDW_MINB(NF))
k_bl_midw(cf* __restrict__ Y, BlGeom g, const BlVol* __restrict__ vols, int vol_base, int shared_desc) {
    constexpr int NT = BlDims<NF>::NT, U = 8;
    MVTB_DYN_SMEM(smem_raw);
    const int W = g.W, D = g.D, F = g.F, K = 2 * F + 1;
    // The W table is dead between the two W-axis phases, which is exactly when the [K][K] bins live: they share
    // the front of the buffer and the table is reloaded (from L2) before the way back.
    const size_t sc_bytes = sizeof(float) * (size_t)(W / 2 + 1) * NT, sb_bytes = sizeof(cf) * (size_t)K * K;
    const size_t front = ((sc_bytes > sb_bytes ? sc_bytes : sb_bytes) + 15) / 16 * 16;
    float* sc = (float*)smem_raw;                        // (cos, sin) rows of the W axis, 0 .. W/2
    cf* sb = (cf*)smem_raw;                              // [K][K]  bins after the pointwise stage
    cf* sg = (cf*)(smem_raw + front);                    // [K][D]  W-bins of every column
    // the way back reuses sg as [K][F + 1] float4 = K (K + 1) cf, one row more than [K][D] holds when D = K
    cf* st = sg + (size_t)K * (D > K ? D : K + 1);       // [D]     exp(-2 pi i t / D)
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int vol = blockIdx.x / NF, fh = blockIdx.x - vol * NF;
    bl_load_table<NF>(sc, g.tabC[1], g.tabS[1], W, tid, nthr);
    for (int e = tid; e < D; e += nthr) st[e] = __ldg(g.twD + e);
    __syncthreads();
    cf* yplane = Y + ((size_t)vol * NF + fh) * (size_t)W * D;
    const int npair = (W - 1) / 2;

    // ---- forward along W: column d -> sg[F +- f][d]
    for (int d = tid; d < D; d += nthr) {
        const cf* yv = yplane + d;
        float2 pqx[NF], pqy[NF];
        {
            const cf y0 = yv[0];
            const cf yn = (W & 1) ? cmk(0.f, 0.f) : yv[(size_t)(W / 2) * D];
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                pqx[f] = make_float2((f & 1) ? y0.x - yn.x : y0.x + yn.x, 0.f);
                pqy[f] = make_float2((f & 1) ? y0.y - yn.y : y0.y + yn.y, 0.f);
            }
        }
        int w = 1;
        for (; w + U - 1 <= npair; w += U) {
            cf a[U], b[U];
            MVTB_UNROLL
            for (int u = 0; u < U; ++u) { a[u] = yv[(size_t)(w + u) * D]; b[u] = yv[(size_t)(W - w - u) * D]; }
            MVTB_UNROLL
            for (int u = 0; u < U; ++u) {
                float2 cs[NF];
                bl_row<NF>(sc + (w + u) * NT, cs);
                const float2 ex = make_float2(a[u].x + b[u].x, a[u].x - b[u].x);
                const float2 ey = make_float2(a[u].y + b[u].y, a[u].y - b[u].y);
                MVTB_UNROLL
                for (int f = 0; f < NF; ++f) { pqx[f] = fma2(ex, cs[f], pqx[f]); pqy[f] = fma2(ey, cs[f], pqy[f]); }
            }
        }
        for (; w <= npair; ++w) {
            float2 cs[NF];
            bl_row<NF>(sc + w * NT, cs);
            const cf a = yv[(size_t)w * D], b = yv[(size_t)(W - w) * D];
            const float2 ex = make_float2(a.x + b.x, a.x - b.x), ey = make_float2(a.y + b.y, a.y - b.y);
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) { pqx[f] = fma2(ex, cs[f], pqx[f]); pqy[f] = fma2(ey, cs[f], pqy[f]); }
        }
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) {
            if (f <= F) {                                // X(+f) = P - iQ, X(-f) = P + iQ
                sg[(F + f) * D + d] = cmk(pqx[f].x + pqy[f].y, pqy[f].x - pqx[f].y);
                if (f > 0) sg[(F - f) * D + d] = cmk(pqx[f].x - pqy[f].y, pqy[f].x + pqx[f].y);
            }
        }
    }
    __syncthreads();

    // ---- D axis forward, pair-folded like the other axes: with e = G[d] + G[D-d], o = G[d] - G[D-d] (in place),
    //   B(+-fd) = G[0] (+ G[D/2] (-1)^fd) + P -+ iQ,   P = sum_d e cos(2 pi fd d / D),  Q = sum_d o sin(2 pi fd d / D)
    const int dpairs = (D - 1) / 2;
    for (int o = tid; o < K * dpairs; o += nthr) {
        const int jw = o / dpairs, dd = o - jw * dpairs + 1;
        cf* row = sg + jw * D;
        const cf a = row[dd], b = row[D - dd];
        row[dd] = cadd(a, b);
        row[D - dd] = csub(a, b);
    }
    __syncthreads();
    {
        const BlVol& bv = vols[shared_desc ? 0 : vol_base + vol];
        int shape[3];
        shape[0] = g.D; shape[1] = g.W; shape[2] = g.H;
        for (int o = tid; o < K * (F + 1); o += nthr) {
            const int jw = o / (F + 1), fd = o - jw * (F + 1);
            const cf* row = sg + jw * D;
            cf P = cmk(0.f, 0.f), Qs = cmk(0.f, 0.f);
            int idx = 0;
            for (int dd = 1; dd <= dpairs; ++dd) {
                idx += fd;
                if (idx >= D) idx -= D;
                const cf e = row[dd], od = row[D - dd], w_ = st[idx];     // w_ = (cos, -sin)
                P.x = fmaf(e.x, w_.x, P.x);
                P.y = fmaf(e.y, w_.x, P.y);
                Qs.x = fmaf(od.x, -w_.y, Qs.x);
                Qs.y = fmaf(od.y, -w_.y, Qs.y);
            }
            cf base = row[0];
            if ((D & 1) == 0) {
                const cf gn = row[D / 2];
                base = (fd & 1) ? csub(base, gn) : cadd(base, gn);
            }
            P = cadd(P, base);
            int ish[3];
            ish[1] = (jw - F) + g.W / 2;
            ish[2] = fh + g.H / 2;
            ish[0] = fd + D / 2;
            sb[jw * K + F + fd] = pointwise_bin(bv.d, 3, shape, ish, cmk(P.x + Qs.y, P.y - Qs.x), g.scale);     // P - iQ
            if (fd > 0) {
                ish[0] = -fd + D / 2;
                sb[jw * K + F - fd] = pointwise_bin(bv.d, 3, shape, ish, cmk(P.x - Qs.y, P.y + Qs.x), g.scale); // P + iQ
            }
        }
    }
    __syncthreads();
    // E = B(+fd) + B(-fd), O = B(+fd) - B(-fd) packed as float4 over the now free G tile: the way back along D is
    //   G'[j][d] = B(0) + sum_fd ( E cos(2 pi fd d / D) + i O sin(2 pi fd d / D) )
    float4* seo = (float4*)sg;                            // [K][F + 1]; entry 0 of a row holds (B(0), 0)
    for (int o = tid; o < K * (F + 1); o += nthr) {
        const int jw = o / (F + 1), fd = o - jw * (F + 1);
        const cf bp = sb[jw * K + F + fd], bm = sb[jw * K + F - fd];
        seo[o] = fd == 0 ? make_float4(bp.x, bp.y, 0.f, 0.f) : make_float4(bp.x + bm.x, bp.y + bm.y, bp.x - bm.x, bp.y - bm.y);
    }
    __syncthreads();
    bl_load_table<NF>(sc, g.tabC[1], g.tabS[1], W, tid, nthr);      // over the bins, which are no longer needed
    __syncthreads();

    // ---- back along D (into registers) and along W (streamed out in place)
    for (int d = tid; d < D; d += nthr) {
        // gp[f] = G'[F + f][d], gm[f] = G'[F - f][d]; the W axis then needs S_f = gp + gm, T_f = gp - gm
        cf gp[NF], gm[NF];
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) {
            gp[f] = cmk(0.f, 0.f);
            gm[f] = cmk(0.f, 0.f);
            if (f <= F) {
                const float4 e0 = seo[(F + f) * (F + 1)], e1 = seo[(F - f) * (F + 1)];
                gp[f] = cmk(e0.x, e0.y);
                gm[f] = cmk(e1.x, e1.y);
            }
        }
        int idx = 0;
        for (int fd = 1; fd <= F; ++fd) {
            idx += d;
            if (idx >= D) idx -= D;
            const cf w_ = st[idx];                        // (cos, -sin) of 2 pi fd d / D
            const float c = w_.x, sn = -w_.y;
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                if (f <= F) {
                    const float4 eo = seo[(F + f) * (F + 1) + fd];
                    gp[f].x = fmaf(eo.x, c, fmaf(-eo.w, sn, gp[f].x));
                    gp[f].y = fmaf(eo.y, c, fmaf(eo.z, sn, gp[f].y));
                    if (f > 0) {
                        const float4 em = seo[(F - f) * (F + 1) + fd];
                        gm[f].x = fmaf(em.x, c, fmaf(-em.w, sn, gm[f].x));
                        gm[f].y = fmaf(em.y, c, fmaf(em.z, sn, gm[f].y));
                    }
                }
            }
        }
        float2 stx[NF], sty[NF];
        MVTB_UNROLL
        for (int f = 0; f < NF; ++f) {
            if (f == 0) { stx[0] = make_float2(gp[0].x, 0.f); sty[0] = make_float2(gp[0].y, 0.f); }
            else { stx[f] = make_float2(gp[f].x + gm[f].x, gp[f].x - gm[f].x); sty[f] = make_float2(gp[f].y + gm[f].y, gp[f].y - gm[f].y); }
        }
        cf* yv = yplane + d;
        {
            cf s0 = cmk(0.f, 0.f), sn = cmk(0.f, 0.f);
            MVTB_UNROLL
            for (int f = 0; f < NF; ++f) {
                s0.x += stx[f].x; s0.y += sty[f].x;
                sn.x += (f & 1) ? -stx[f].x : stx[f].x;
                sn.y += (f & 1) ? -sty[f].x : sty[f].x;
            }
            yv[0] = s0;
            if ((W & 1) == 0) yv[(size_t)(W / 2) * D] = sn;
        }
        for (int w = 1; w <= npair; ++w) {
            float2 cs[NF];
            bl_row<NF>(sc + w * NT, cs);
            float2 pqx = make_float2(0.f, 0.f), pqy = make_float2(0.f, 0.f);
            float2 pqx2 = make_float2(0.f, 0.f), pqy2 = make_float2(0.f, 0.f);
            MVTB_UNROLL
            for (int f = 0; f + 1 < NF; f += 2) {
                pqx = fma2(stx[f], cs[f], pqx); pqy = fma2(sty[f], cs[f], pqy);
                pqx2 = fma2(stx[f + 1], cs[f + 1], pqx2); pqy2 = fma2(sty[f + 1], cs[f + 1], pqy2);
            }
            if (NF & 1) { pqx = fma2(stx[NF - 1], cs[NF - 1], pqx); pqy = fma2(sty[NF - 1], cs[NF - 1], pqy); }
            const float Px = pqx.x + pqx2.x, Qx = pqx.y + pqx2.y, Py = pqy.x + pqy2.x, Qy = pqy.y + pqy2.y;
            yv[(size_t)w * D] = cmk(Px - Qy, Py + Qx);
            yv[(size_t)(W - w) * D] = cmk(Px + Qy, Py - Qx);
        }
    }
}
