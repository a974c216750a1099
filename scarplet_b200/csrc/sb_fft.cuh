// Register-resident Stockham FFT for power-of-two lengths, complex64 or complex128.
//
// One FFT of length N is carried by a group of T = N / E threads; thread t holds
// E = 16 elements x[t + q*T], q = 0..E-1, in registers.  Every stage is a set of
// radix-R butterflies (R <= E, R in {2,4,8,16}) done entirely in registers; between
// stages the data is exchanged through a padded shared-memory buffer.  Input and
// output are both in natural order with the same thread/register layout, so
// global loads and stores are coalesced across the group and no bit reversal is
// ever materialised.  Twiddles come from per-stage tables laid out [u][k] so that
// a warp reads consecutive addresses.
//
// The inverse transform is obtained by swapping real and imaginary parts before
// and after a forward transform (unnormalised).
#pragma once
#include "sb_rt.h"

namespace sbfft {

constexpr int E = 16;  // elements per thread

SB_HOSTDEV int pad_index(int i) { return i + (i >> 4); }
SB_CONSTEXPR int padded_len(int n) { return n + (n >> 4); }

// ---- stage plan -----------------------------------------------------------
// radices for N = 2^k, 128 <= N <= 8192: as many 16s as fit, then the rest.
SB_CONSTEXPR int num_stages(int N) {
    int s = 0;
    while (N > 1) { N = (N >= 16) ? N / 16 : 1; ++s; }
    return s;
}
SB_CONSTEXPR int stage_radix(int N, int s) {
    int r = 16;
    for (int i = 0; i <= s; ++i) { r = (N >= 16) ? 16 : N; N /= r; }
    return r;
}
SB_CONSTEXPR int stage_ns(int N, int s) {   // product of the radices before stage s
    int ns = 1;
    for (int i = 0; i < s; ++i) ns *= stage_radix(N, i);
    return ns;
}
// offset (in elements) of stage s in the twiddle table; stage 0 has no twiddles
SB_CONSTEXPR int twiddle_offset(int N, int s) {
    int off = 0;
    for (int i = 1; i < s; ++i) off += (stage_radix(N, i) - 1) * stage_ns(N, i);
    return off;
}
SB_CONSTEXPR int twiddle_count(int N) { return twiddle_offset(N, num_stages(N)); }

// host: fill the table for length N (float64 sincos, rounded once for complex64)
template <typename R>
inline void fill_twiddles(int N, typename Vec<R>::v2* out) {
    int ns = 1, off = 0;
    for (int s = 0; N > ns; ++s) {
        int rest = N / ns;
        int r = rest >= 16 ? 16 : rest;
        if (s > 0) {
            for (int u = 1; u < r; ++u)
                for (int k = 0; k < ns; ++k) {
                    double a = -2.0 * M_PI * (double)u * (double)k / ((double)ns * (double)r);
                    out[off + (u - 1) * ns + k].x = (R)cos(a);
                    out[off + (u - 1) * ns + k].y = (R)sin(a);
                }
            off += (r - 1) * ns;
        }
        ns *= r;
    }
}

// ---- small DFTs in registers ------------------------------------------------
template <typename C> SB_DEVICE C cadd(C a, C b) { C r; r.x = a.x + b.x; r.y = a.y + b.y; return r; }
template <typename C> SB_DEVICE C csub(C a, C b) { C r; r.x = a.x - b.x; r.y = a.y - b.y; return r; }
template <typename C> SB_DEVICE C cmul(C a, C b) {
    C r; r.x = a.x * b.x - a.y * b.y; r.y = a.x * b.y + a.y * b.x; return r;
}
template <typename C> SB_DEVICE C mul_mi(C a) { C r; r.x = a.y; r.y = -a.x; return r; }   // a * (-i)

// ---- packed FP32 (sm_100a FADD2 / FMUL2 / FFMA2) -------------------------------
// A float2 is one 64-bit register pair; add/mul/fma.f32x2 work on both halves in one issue
// slot, and ptxas folds half swaps, per-half negations and scalar broadcasts of the operands
// into the instruction (R.F32x2.LO_HI, .NP, R.F32), so a complex add is 1 instruction
// instead of 2, a complex multiply 2 instead of 4, and multiplying by -i is free.  The
// butterflies below are written against these helpers; the emulator build and complex128
// use the scalar forms above.
#ifndef SB_EMU
#define SB_F32X2 1
typedef unsigned long long pk_t;
SB_DEVICE pk_t pk(float lo, float hi) { pk_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
SB_DEVICE pk_t pk(float2 a) { return pk(a.x, a.y); }
SB_DEVICE float2 unpk(pk_t v) { float2 r; asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v)); return r; }
SB_DEVICE pk_t add2(pk_t a, pk_t b) { pk_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
SB_DEVICE pk_t mul2(pk_t a, pk_t b) { pk_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
SB_DEVICE pk_t fma2(pk_t a, pk_t b, pk_t c) { pk_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

SB_DEVICE float2 cadd(float2 a, float2 b) { return unpk(add2(pk(a), pk(b))); }
SB_DEVICE float2 csub(float2 a, float2 b) { return unpk(add2(pk(a), pk(-b.x, -b.y))); }
SB_DEVICE float2 cmul(float2 a, float2 b) {
    return unpk(fma2(pk(-a.y, a.x), pk(b.y, b.y), mul2(pk(a), pk(b.x, b.x))));
}
// e + s * r, e - s * r for a real scalar r
SB_DEVICE float2 caxpy(float2 e, float2 s, float r) { return unpk(fma2(pk(s), pk(r, r), pk(e))); }
// a - i a = (a.x + a.y, a.y - a.x);  -(a + i a) = (a.y - a.x, -a.x - a.y)
SB_DEVICE float2 rot_m45(float2 a) { return unpk(add2(pk(a), pk(a.y, -a.x))); }
SB_DEVICE float2 rot_m135(float2 a) { return unpk(add2(pk(a.y, -a.x), pk(-a.x, -a.y))); }
#endif

template <typename R, int RADIX> struct Dft;

template <typename R> struct Dft<R, 2> {
    typedef typename Vec<R>::v2 C;
    SB_DEVICE static void run(C* x) {
        C a = x[0], b = x[1];
        x[0] = cadd(a, b);
        x[1] = csub(a, b);
    }
};

template <typename R> struct Dft<R, 4> {
    typedef typename Vec<R>::v2 C;
    SB_DEVICE static void run(C* x) {
        C t0 = cadd(x[0], x[2]), t1 = csub(x[0], x[2]);
        C t2 = cadd(x[1], x[3]), t3 = mul_mi(csub(x[1], x[3]));
        x[0] = cadd(t0, t2);
        x[2] = csub(t0, t2);
        x[1] = cadd(t1, t3);
        x[3] = csub(t1, t3);
    }
};

template <typename R> struct Dft<R, 8> {
    typedef typename Vec<R>::v2 C;
    SB_DEVICE static void run(C* x) {
        const R h = (R)0.70710678118654752440;
        C e[4] = {x[0], x[2], x[4], x[6]};
        C o[4] = {x[1], x[3], x[5], x[7]};
        Dft<R, 4>::run(e);
        Dft<R, 4>::run(o);
        // o[k] *= W8^k
        o[1] = mk2<R>(h * (o[1].x + o[1].y), h * (o[1].y - o[1].x));
        o[2] = mul_mi(o[2]);
        o[3] = mk2<R>(h * (o[3].y - o[3].x), -h * (o[3].x + o[3].y));
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            x[k] = cadd(e[k], o[k]);
            x[k + 4] = csub(e[k], o[k]);
        }
    }
};

template <typename R> struct Dft<R, 16> {
    typedef typename Vec<R>::v2 C;
    SB_DEVICE static void run(C* x) {
        const R h = (R)0.70710678118654752440;
        const R c1 = (R)0.92387953251128675613;   // cos(pi/8)
        const R s1 = (R)0.38268343236508977173;   // sin(pi/8)
        C e[8], o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { e[k] = x[2 * k]; o[k] = x[2 * k + 1]; }
        Dft<R, 8>::run(e);
        Dft<R, 8>::run(o);
        // o[k] *= W16^k = exp(-i*pi*k/8)
        o[1] = cmul(o[1], mk2<R>(c1, -s1));
        o[2] = mk2<R>(h * (o[2].x + o[2].y), h * (o[2].y - o[2].x));
        o[3] = cmul(o[3], mk2<R>(s1, -c1));
        o[4] = mul_mi(o[4]);
        o[5] = cmul(o[5], mk2<R>(-s1, -c1));
        o[6] = mk2<R>(h * (o[6].y - o[6].x), -h * (o[6].x + o[6].y));
        o[7] = cmul(o[7], mk2<R>(-c1, -s1));
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            x[k] = cadd(e[k], o[k]);
            x[k + 8] = csub(e[k], o[k]);
        }
    }
};

#ifdef SB_F32X2
// float specialisations: the W8 / W16 constant rotations fold into packed FMAs
template <> struct Dft<float, 8> {
    typedef float2 C;
    SB_DEVICE static void run(C* x) {
        const float h = 0.70710678118654752440f;
        C e[4] = {x[0], x[2], x[4], x[6]};
        C o[4] = {x[1], x[3], x[5], x[7]};
        Dft<float, 4>::run(e);
        Dft<float, 4>::run(o);
        const C s1 = rot_m45(o[1]), s3 = rot_m135(o[3]), s2 = mul_mi(o[2]);
        x[0] = cadd(e[0], o[0]);  x[4] = csub(e[0], o[0]);
        x[1] = caxpy(e[1], s1, h);  x[5] = caxpy(e[1], s1, -h);
        x[2] = cadd(e[2], s2);  x[6] = csub(e[2], s2);
        x[3] = caxpy(e[3], s3, h);  x[7] = caxpy(e[3], s3, -h);
    }
};

template <> struct Dft<float, 16> {
    typedef float2 C;
    SB_DEVICE static void run(C* x) {
        const float h = 0.70710678118654752440f;
        const float c1 = 0.92387953251128675613f;   // cos(pi/8)
        const float s1 = 0.38268343236508977173f;   // sin(pi/8)
        C e[8], o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { e[k] = x[2 * k]; o[k] = x[2 * k + 1]; }
        Dft<float, 8>::run(e);
        Dft<float, 8>::run(o);
        // o[k] *= W16^k = exp(-i*pi*k/8); the multiples of pi/4 fold into the final add
        o[1] = cmul(o[1], make_float2(c1, -s1));
        o[3] = cmul(o[3], make_float2(s1, -c1));
        o[5] = cmul(o[5], make_float2(-s1, -c1));
        o[7] = cmul(o[7], make_float2(-c1, -s1));
        const C r2 = rot_m45(o[2]), r6 = rot_m135(o[6]), r4 = mul_mi(o[4]);
        x[0] = cadd(e[0], o[0]);  x[8] = csub(e[0], o[0]);
        x[1] = cadd(e[1], o[1]);  x[9] = csub(e[1], o[1]);
        x[2] = caxpy(e[2], r2, h);  x[10] = caxpy(e[2], r2, -h);
        x[3] = cadd(e[3], o[3]);  x[11] = csub(e[3], o[3]);
        x[4] = cadd(e[4], r4);  x[12] = csub(e[4], r4);
        x[5] = cadd(e[5], o[5]);  x[13] = csub(e[5], o[5]);
        x[6] = caxpy(e[6], r6, h);  x[14] = caxpy(e[6], r6, -h);
        x[7] = cadd(e[7], o[7]);  x[15] = csub(e[7], o[7]);
    }
    // Same transform, outputs as pairs over (k, k + 8): re[k] = (Re x[k], Re x[k + 8]),
    // im[k] likewise -- the form a packed two-pixel epilogue wants.  The last butterfly
    // level e +- s is one FFMA2 per pair with both scalars broadcast: s * (1, -1) + e.
    SB_DEVICE static void run_soa(C* x, pk_t* re, pk_t* im) {
        const float h = 0.70710678118654752440f;
        const float c1 = 0.92387953251128675613f;
        const float s1 = 0.38268343236508977173f;
        C e[8], o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { e[k] = x[2 * k]; o[k] = x[2 * k + 1]; }
        Dft<float, 8>::run(e);
        Dft<float, 8>::run(o);
        o[1] = cmul(o[1], make_float2(c1, -s1));
        o[3] = cmul(o[3], make_float2(s1, -c1));
        o[5] = cmul(o[5], make_float2(-s1, -c1));
        o[7] = cmul(o[7], make_float2(-c1, -s1));
        o[2] = rot_m45(o[2]);
        o[6] = rot_m135(o[6]);
        o[4] = mul_mi(o[4]);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float f = (k == 2 || k == 6) ? h : 1.f;
            const pk_t pm = pk(f, -f);
            re[k] = fma2(pk(o[k].x, o[k].x), pm, pk(e[k].x, e[k].x));
            im[k] = fma2(pk(o[k].y, o[k].y), pm, pk(e[k].y, e[k].y));
        }
    }
};
#endif

// ---- one Stockham stage, split into its four parts ----------------------------
// v[q] = x[t + q*T].  A stage is: fetch the thread's twiddles (global, L1-resident),
// multiply + radix butterflies in registers, scatter to the exchange buffer in the
// order the next stage reads, gather v[q] = sm[t + q*T].  Kernels that pipeline two
// transforms (sb_kernels.cuh, "leapfrog") call the parts; `stage` strings them
// together for the simple one-transform-at-a-time kernels.
constexpr int TW = E - 1;    // twiddle registers a thread needs for one stage (at most)

// SMEM: `tw` is the compact copy of the table in shared memory (copy_ctw; plain loads)
// Twiddle diet (complex64, radix 16): only W^k, W^2k, W^3k, W^4k, W^8k, W^12k are fetched; the
// other nine are one complex product of two of those (1.5 ulp instead of 0.5).  The table
// reads of a stage drop from 15 to 6 per thread -- they share the LSU with the exchange --
// and 18 fewer registers are live across the barrier that follows the fetch.
template <typename R, int RADIX>
SB_CONSTEXPR bool tw_derived(int u) {
#ifdef SB_F32X2
    return sizeof(R) == 4 && RADIX == 16 && !(u <= 4 || u == 8 || u == 12);
#else
    return false;
#endif
}

// Compact copy of the table for shared memory: per stage only the rows that are fetched
// (6 of 15 under the diet), same [row][k] order.
template <typename R>
SB_CONSTEXPR int ctw_rows(int N, int s) {
    const int r = stage_radix(N, s);
    int n = 0;
    for (int u = 1; u < r; ++u) n += (r == 16 ? tw_derived<R, 16>(u) : false) ? 0 : 1;
    return n;
}
template <typename R>
SB_CONSTEXPR int ctw_offset(int N, int s) {
    int off = 0;
    for (int i = 1; i < s; ++i) off += ctw_rows<R>(N, i) * stage_ns(N, i);
    return off;
}
template <typename R> SB_CONSTEXPR int ctw_count(int N) { return ctw_offset<R>(N, num_stages(N)); }
// row of multiplier u in the compact table of a radix-RADIX stage
template <typename R, int RADIX>
SB_CONSTEXPR int ctw_row(int u) {
    int row = 0;
    for (int i = 1; i < u; ++i) row += tw_derived<R, RADIX>(i) ? 0 : 1;
    return row;
}
// all `nthreads` threads of the CTA: dst (shared) <- compact copy of the table `src` (global)
template <int N, typename R>
SB_DEVICE void copy_ctw(typename Vec<R>::v2* dst, const typename Vec<R>::v2* SB_RESTRICT src, int tid, int nthreads) {
#pragma unroll
    for (int s = 1; s < num_stages(N); ++s) {
        const int ns = stage_ns(N, s), r = stage_radix(N, s);
        int row = 0;
        for (int u = 1; u < r; ++u) {
            if (r == 16 && tw_derived<R, 16>(u)) continue;
            for (int k = tid; k < ns; k += nthreads)
                dst[ctw_offset<R>(N, s) + row * ns + k] = sb_ldg(src + twiddle_offset(N, s) + (u - 1) * ns + k);
            ++row;
        }
    }
}

template <int N, int S, typename R, bool SMEM = false>
SB_DEVICE void load_tw(typename Vec<R>::v2 (&w)[TW], int t, const typename Vec<R>::v2* SB_RESTRICT tw) {
    constexpr int T = N / E;
    constexpr int RADIX = stage_radix(N, S);
    constexpr int NS = stage_ns(N, S);
    constexpr int B = E / RADIX;
    constexpr int TWO = twiddle_offset(N, S);
    if (S == 0) return;
#pragma unroll
    for (int m = 0; m < B; ++m) {
        const int k = (t + m * T) & (NS - 1);
#pragma unroll
        for (int u = 1; u < RADIX; ++u) {
            if (tw_derived<R, RADIX>(u)) continue;          // stage_math multiplies it together
            w[(u - 1) * B + m] = SMEM ? tw[ctw_offset<R>(N, S) + ctw_row<R, RADIX>(u) * NS + k]
                                      : ld2(tw + TWO + (u - 1) * NS + k);
        }
    }
}

template <int N, int S, typename R>
SB_DEVICE void stage_math(typename Vec<R>::v2 (&v)[E], const typename Vec<R>::v2 (&w)[TW]) {
    typedef typename Vec<R>::v2 C;
    constexpr int RADIX = stage_radix(N, S);
    constexpr int B = E / RADIX;
#pragma unroll
    for (int m = 0; m < B; ++m) {
        C x[RADIX];
#pragma unroll
        for (int u = 0; u < RADIX; ++u) x[u] = v[m + u * B];
        if (S > 0) {
#pragma unroll
            for (int u = 1; u < RADIX; ++u) {
                if (tw_derived<R, RADIX>(u)) {
                    const int hi = u & ~3, lo = u & 3;       // u = hi + lo, hi in {4, 8, 12}
                    x[u] = cmul(x[u], cmul(w[(hi - 1) * B + m], w[(lo - 1) * B + m]));
                } else {
                    x[u] = cmul(x[u], w[(u - 1) * B + m]);
                }
            }
        }
        Dft<R, RADIX>::run(x);
#pragma unroll
        for (int u = 0; u < RADIX; ++u) v[m + u * B] = x[u];
    }
}

#ifdef SB_F32X2
// Small DFTs with paired outputs: re[k] = (Re X[k], Re X[k + R/2]), im[k] likewise.  The last
// butterfly level e +- f*s is one FFMA2 per pair with both scalars broadcast.
SB_DEVICE void soa_pair(float2 e, float2 s, float f, pk_t& re, pk_t& im) {
    const pk_t pm = pk(f, -f);
    re = fma2(pk(s.x, s.x), pm, pk(e.x, e.x));
    im = fma2(pk(s.y, s.y), pm, pk(e.y, e.y));
}
template <int RADIX> struct DftSoa;
template <> struct DftSoa<2> {
    SB_DEVICE static void run(float2* x, pk_t* re, pk_t* im) { soa_pair(x[0], x[1], 1.f, re[0], im[0]); }
};
template <> struct DftSoa<4> {
    SB_DEVICE static void run(float2* x, pk_t* re, pk_t* im) {
        const float2 t0 = cadd(x[0], x[2]), t1 = csub(x[0], x[2]);
        const float2 t2 = cadd(x[1], x[3]), t3 = mul_mi(csub(x[1], x[3]));
        soa_pair(t0, t2, 1.f, re[0], im[0]);
        soa_pair(t1, t3, 1.f, re[1], im[1]);
    }
};
template <> struct DftSoa<8> {
    SB_DEVICE static void run(float2* x, pk_t* re, pk_t* im) {
        const float h = 0.70710678118654752440f;
        float2 e[4] = {x[0], x[2], x[4], x[6]};
        float2 o[4] = {x[1], x[3], x[5], x[7]};
        Dft<float, 4>::run(e);
        Dft<float, 4>::run(o);
        soa_pair(e[0], o[0], 1.f, re[0], im[0]);
        soa_pair(e[1], rot_m45(o[1]), h, re[1], im[1]);
        soa_pair(e[2], mul_mi(o[2]), 1.f, re[2], im[2]);
        soa_pair(e[3], rot_m135(o[3]), h, re[3], im[3]);
    }
};
template <> struct DftSoa<16> {
    SB_DEVICE static void run(float2* x, pk_t* re, pk_t* im) { Dft<float, 16>::run_soa(x, re, im); }
};

// Last stage of a transform (S > 0) with its outputs paired over (q, q + 8), q = 0..7 -- the
// form the packed two-pixel epilogue of the fit kernel wants.
template <int N, int S>
SB_DEVICE void stage_math_soa(const float2 (&v)[E], const float2 (&w)[TW], pk_t (&re)[8], pk_t (&im)[8]) {
    constexpr int RADIX = stage_radix(N, S);
    constexpr int B = E / RADIX;
    static_assert(S > 0, "stage_math_soa: twiddled stage expected");
#pragma unroll
    for (int m = 0; m < B; ++m) {
        float2 x[RADIX];
        x[0] = v[m];
#pragma unroll
        for (int u = 1; u < RADIX; ++u) {
            if (tw_derived<float, RADIX>(u)) {
                const int hi = u & ~3, lo = u & 3;
                x[u] = cmul(v[m + u * B], cmul(w[(hi - 1) * B + m], w[(lo - 1) * B + m]));
            } else {
                x[u] = cmul(v[m + u * B], w[(u - 1) * B + m]);
            }
        }
        pk_t r[RADIX / 2], i[RADIX / 2];
        DftSoa<RADIX>::run(x, r, i);
#pragma unroll
        for (int u = 0; u < RADIX / 2; ++u) { re[m + u * B] = r[u]; im[m + u * B] = i[u]; }
    }
}
#endif

template <int N, int S, typename R>
SB_DEVICE void stage_store(const typename Vec<R>::v2 (&v)[E], int t, typename Vec<R>::v2* sm) {
    constexpr int T = N / E;
    constexpr int RADIX = stage_radix(N, S);
    constexpr int NS = stage_ns(N, S);
    constexpr int B = E / RADIX;
    // pad_index(base + u*NS) is linear in u (NS is 1 or a multiple of 16): one address per
    // butterfly, the rest are immediate offsets
    static_assert(NS == 1 || NS % 16 == 0, "stage_store: unexpected stage geometry");
    constexpr int STEP = NS == 1 ? 1 : NS + NS / 16;
#pragma unroll
    for (int m = 0; m < B; ++m) {
        const int j = t + m * T;
        const int base = (j / NS) * (NS * RADIX) + (j & (NS - 1));
        typename Vec<R>::v2* p = sm + pad_index(base);
#pragma unroll
        for (int u = 0; u < RADIX; ++u) p[u * STEP] = v[m + u * B];
    }
}

template <int N, typename R>
SB_DEVICE void stage_load(typename Vec<R>::v2 (&v)[E], int t, const typename Vec<R>::v2* sm) {
    constexpr int T = N / E;
    if constexpr (T % 16 == 0) {
        const typename Vec<R>::v2* p = sm + pad_index(t);     // pad_index(t + q*T) = pad_index(t) + q*(T + T/16)
#pragma unroll
        for (int q = 0; q < E; ++q) v[q] = p[q * (T + T / 16)];
    } else {
#pragma unroll
        for (int q = 0; q < E; ++q) v[q] = sm[pad_index(t + q * T)];
    }
}

// First stage (radix 16, no twiddles) when only v[0] and v[15] are non-zero: the
// column transform of a template whose support is shorter than T on either side of
// the origin.  X[u] = v0 + v15 * W16^(-u): 8 constant products instead of a full DFT16.
template <typename R>
SB_DEVICE void stage0_sparse2(typename Vec<R>::v2 (&v)[E]) {
    typedef typename Vec<R>::v2 C;
    const R h = (R)0.70710678118654752440;
    const R c1 = (R)0.92387953251128675613;
    const R s1 = (R)0.38268343236508977173;
    const C a = v[0], b = v[E - 1];
    C p[8];
    const R cx = c1 * b.x, cy = c1 * b.y, sx = s1 * b.x, sy = s1 * b.y, hx = h * b.x, hy = h * b.y;
    p[0] = b;
    p[1] = mk2<R>(cx - sy, cy + sx);
    p[2] = mk2<R>(hx - hy, hx + hy);
    p[3] = mk2<R>(sx - cy, sy + cx);
    p[4] = mk2<R>(-b.y, b.x);
    p[5] = mk2<R>(-sx - cy, cx - sy);
    p[6] = mk2<R>(-hx - hy, hx - hy);
    p[7] = mk2<R>(-cx - sy, sx - cy);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        v[u] = cadd(a, p[u]);
        v[u + 8] = csub(a, p[u]);
    }
}

template <int N, int S, typename R>
SB_DEVICE void stage(typename Vec<R>::v2 (&v)[E], int t, typename Vec<R>::v2* sm,
                     const typename Vec<R>::v2* SB_RESTRICT tw) {
    typedef typename Vec<R>::v2 C;
    constexpr bool LAST = (stage_ns(N, S) * stage_radix(N, S) == N);
    C w[TW];
    load_tw<N, S, R>(w, t, tw);
    stage_math<N, S, R>(v, w);
    if (!LAST) {
        stage_store<N, S, R>(v, t, sm);
        sb_sync();
        stage_load<N, R>(v, t, sm);
        sb_sync();
    }
}

template <int N, typename R, int S = 0>
struct Stages {
    typedef typename Vec<R>::v2 C;
    SB_DEVICE static void run(C (&v)[E], int t, C* sm, const C* SB_RESTRICT tw) {
        stage<N, S, R>(v, t, sm, tw);
        if constexpr (S + 1 < num_stages(N)) Stages<N, R, S + 1>::run(v, t, sm, tw);
    }
};

// Forward FFT whose only non-zero inputs are v[0] and v[15] (a signal supported on fewer than
// T samples either side of the origin): the first radix-16 stage is 8 constant products.
template <int N, typename R>
SB_DEVICE void forward_sparse2(typename Vec<R>::v2 (&v)[E], int t, typename Vec<R>::v2* sm,
                               const typename Vec<R>::v2* SB_RESTRICT tw) {
    static_assert(stage_radix(N, 0) == 16 && num_stages(N) >= 2, "forward_sparse2: N >= 256");
    stage0_sparse2<R>(v);
    stage_store<N, 0, R>(v, t, sm);
    sb_sync();
    stage_load<N, R>(v, t, sm);
    sb_sync();
    Stages<N, R, 1>::run(v, t, sm, tw);
}

// Forward FFT of length N over the group's registers.  `sm` is the group's
// private exchange buffer of padded_len(N) elements.  All threads of the CTA must
// call this together (it contains CTA-wide barriers).
template <int N, typename R>
SB_DEVICE void forward(typename Vec<R>::v2 (&v)[E], int t, typename Vec<R>::v2* sm,
                       const typename Vec<R>::v2* SB_RESTRICT tw) {
    Stages<N, R, 0>::run(v, t, sm, tw);
}

}  // namespace sbfft
