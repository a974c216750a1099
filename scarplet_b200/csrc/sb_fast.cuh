// Pipelined ("leapfrog") versions of the two per-template kernels, complex64 only.
//
// The simple kernels in sb_kernels.cuh run one transform at a time: every exchange
// between radix-16 stages costs two CTA barriers, and the loads that feed a stage
// (twiddles, spectra) are issued right where their values are needed.  ncu showed
// those kernels waiting, not working (46 % of warp stalls on loads, 9 % on barriers,
// issue slots 31 % busy).  Here every thread group carries TWO independent transforms
// a and b that take turns: while a computes a stage in registers, b's data rests in
// its own exchange buffer, and vice versa --
//
//     a.math  a.store | bar | b.math  b.store  a.load  a.twiddles | bar | a.math ...
//
// so there is ONE barrier per exchange, the twiddles and the exchanged data of the
// next stage are already in flight when the barrier opens, and only one transform's
// 16 elements are live in registers at any time.
//
//   k_conv_cols_f  a, b = the two fields (t * curv, M * curv^2) of one spectrum column
//   k_fit_rows_f   a, b = two templates of the batch, same raster row
#pragma once
#include "sb_kernels.cuh"

namespace sb {

using sbfft::TW;
#ifdef SB_EMU
using std::max;
using std::min;
#endif

SB_CONSTEXPR int ilog2(int n) { return n <= 1 ? 0 : 1 + ilog2(n / 2); }

// ---------------------------------------------------------------------------
// leapfrog driver.  Ctx provides, for phase P of stream F (0 = a, 1 = b):
//   twid<P>(w)       fetch the twiddles phase P will use
//   phase<P, F>(v,w) register work of the phase
//   store<P, F>(v)   scatter to the stream's exchange buffer (not after the last phase)
//   load<F>(v)       gather the next phase's elements
//   bar()            barrier over the threads that carry the two transforms
// On entry to Frog<P>: a has finished phase P and stored it, a barrier has passed,
// b holds its phase-P input in vb (and wb).
// ---------------------------------------------------------------------------
template <int P, int K, class Ctx>
struct Frog {
    SB_DEVICE static void run(Ctx& c, float2 (&va)[E], float2 (&vb)[E], float2 (&wa)[TW], float2 (&wb)[TW]) {
        c.template phase<P, 1>(vb, wb);
        if constexpr (P < K - 1) {
            c.template store<P, 1>(vb);
            c.template load<0>(va);
            c.template twid<P + 1>(wa);
            c.bar();
            c.template phase<P + 1, 0>(va, wa);
            if constexpr (P + 1 < K - 1) c.template store<P + 1, 0>(va);
            c.template load<1>(vb);
            c.template twid<P + 1>(wb);
            if constexpr (P + 1 < K - 1) c.bar();
            Frog<P + 1, K, Ctx>::run(c, va, vb, wa, wb);
        }
    }
};

template <int K, class Ctx>
SB_DEVICE void leapfrog(Ctx& c, float2 (&va)[E], float2 (&vb)[E]) {
    float2 wa[TW], wb[TW];
    c.template twid<0>(wa);
    c.template twid<0>(wb);
    c.template phase<0, 0>(va, wa);
    c.template store<0, 0>(va);
    c.bar();
    Frog<0, K, Ctx>::run(c, va, vb, wa, wb);
}

// ---------------------------------------------------------------------------
// k_conv_cols_f<Py, SPARSE>: grid (n_templates, ceil(KX / GP)) -- the template index
// runs fastest, so the CTAs that multiply by the same curvature-spectrum column are
// co-resident and the column comes out of L2 for all but the first of them.
// Phases of one field: forward stages 0..NST-1, the last one fused with the product
// (core.py:359 / :363) and inverse stage 0, then inverse stages 1..NST-1.
// SPARSE: the template support is shorter than T rows on either side of the origin,
// so each thread's only non-zero inputs are elements 0 and 15 (stage0_sparse2).
// ---------------------------------------------------------------------------
// PERSIST (k_conv_cols_p): the spectrum columns are in shared memory and the thread group has
// its own named barrier.
template <int N, bool SPARSE, bool PERSIST = false>
struct ConvCtx {
    static constexpr int NST = sbfft::num_stages(N);
    static constexpr int K = 2 * NST - 1;
    static constexpr int T = N / E;
    int t;
    float2 *smA, *smB;
    const float2* tw;
    const float2 *specA, *specB;      // curvature-spectrum columns of the two fields (+ t)
    float4* dst;                      // gbuf plane of this template (nullptr: inactive group)
    int kx, dly, out_ny, kpitch;
    int bar_id;                       // PERSIST: named barrier of this thread group
    // field a's result waits in its registers (the array handed to leapfrog) for field b
    // (parking it in shared memory instead: +2 %)
    const float2* va_fin;

    SB_DEVICE void bar() const {
        if constexpr (PERSIST) sb_bar(bar_id, T);
        else sb_sync();
    }
    SB_CONSTEXPR static int stage_of(int P) { return P < NST ? P : P - NST + 1; }

    template <int P> SB_DEVICE void twid(float2 (&w)[TW]) {
        sbfft::load_tw<N, stage_of(P), float, PERSIST>(w, t, tw);   // PERSIST: the CTA's shared-memory copy
    }

    template <int P, int F> SB_DEVICE void phase(float2 (&v)[E], const float2 (&w)[TW]) {
        if constexpr (P == 0 && SPARSE) sbfft::stage0_sparse2<float>(v);
        else sbfft::stage_math<N, stage_of(P), float>(v, w);
        if constexpr (P == NST - 1) {
            const float2* spec = F == 0 ? specA : specB;
#pragma unroll
            for (int q = 0; q < E; ++q) {
                const float2 s = PERSIST ? spec[q * T] : sb_ld_stream(spec + q * T);
                const float2 pr = sbfft::cmul(v[q], s);
                v[q] = make_float2(pr.y, pr.x);                  // swap: inverse via forward
            }
            sbfft::stage_math<N, 0, float>(v, w);
        }
        if constexpr (P == K - 1 && F == 1) {
            if (dst) {
                // row m = t + q T lies at gbuf_index(t, kx) + q * T * kpitch (T is even): one pointer,
                // one add per store
                static_assert(kGbufRows == 2 && T % 2 == 0, "row-pair interleave");
                const long step = (long)T * kpitch;
                float4* p = dst + gbuf_index(t, kx, kpitch);
                const int io0 = t + dly;
#pragma unroll
                for (int q = 0; q < E; ++q) {
                    const float2 a = va_fin[q];      // field a's result, still in the caller's registers
                    const float4 out = gbuf_pack<float2, float4>(a, v[q]);
                    if (((io0 + q * T) & (N - 1)) < out_ny) sb_st_stream(p, out);
                    p += step;
                }
            }
        }
    }
    template <int P, int F> SB_DEVICE void store(const float2 (&v)[E]) {
        constexpr int S = (P == NST - 1) ? 0 : stage_of(P);
        sbfft::stage_store<N, S, float>(v, t, F == 0 ? smA : smB);
    }
    template <int F> SB_DEVICE void load(float2 (&v)[E]) { sbfft::stage_load<N, float>(v, t, F == 0 ? smA : smB); }
};

template <int N, bool SPARSE>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), (N / E > 256 ? 1 : 2))
k_conv_cols_f(Geom g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, int angle_base,
              const float4* SB_RESTRICT trt, const float2* SB_RESTRICT fct, float4* SB_RESTRICT gbuf,
              const float2* SB_RESTRICT tw) {
    constexpr int T = N / E;
    constexpr int GP = (T > 256 ? T : 256) / T;
    constexpr int PL = sbfft::padded_len(N);
    const int grp = sb_tid() / T, t = sb_tid() % T;
    const int KX = g.Px / 2 + 1;
    const int p_loc = sb_bx();
    const int kx = sb_by() * GP + grp;
    const bool active = kx < KX;
    const int kxc = active ? kx : 0;
    const Tmpl* p = tmpls + tmpl_base + p_loc;
    const int sy_lo = p->sy_lo, sy_hi = p->sy_hi;
    const int a_loc = p->angle_id - angle_base;

    ConvCtx<N, SPARSE> c;
    c.t = t;
    c.smA = (float2*)sb_shared() + (long)grp * 2 * PL;
    c.smB = c.smA + PL;
    c.tw = tw;
    c.specA = fct + (((long)a_loc * 2) * KX + kxc) * N + t;
    c.specB = c.specA + (long)KX * N;
    c.dst = active ? gbuf + (long)p_loc * N * g.kpitch : nullptr;
    c.kx = kx;
    c.dly = g.dly;
    c.out_ny = g.out_ny;
    c.kpitch = g.kpitch;
    // one 128-byte line of each spectrum column per thread (T lines per column)
    sb_prefetch_l2(c.specA + 15 * t);
    sb_prefetch_l2(c.specB + 15 * t);

    const float4* src = trt + ((long)p_loc * KX + kxc) * g.syp;
    float2 va[E], vb[E];
#pragma unroll
    for (int q = 0; q < E; ++q) {
        va[q] = make_float2(0.f, 0.f);
        vb[q] = make_float2(0.f, 0.f);
        if (SPARSE && q != 0 && q != E - 1) continue;
        const int qy = t + q * T;
        const int s = qy < N / 2 ? qy : qy - N;
        if (active && s >= sy_lo && s <= sy_hi) {
            const float4 w = sb_ld_stream(src + (s - sy_lo));
            va[q] = make_float2(w.x, w.y);
            vb[q] = make_float2(w.z, w.w);
        }
    }
    c.va_fin = va;
    leapfrog<ConvCtx<N, SPARSE>::K>(c, va, vb);     // the last phase of field b writes gbuf
}

// ---------------------------------------------------------------------------
// k_conv_cols_p<Py, SPARSE>: persistent variant, grid (KX), 512 threads = G groups of T.
// A CTA owns one spectrum column kx for the whole batch of templates.  The batch is
// walked in runs of templates that share a search angle: the two curvature-spectrum
// columns of that angle are staged in shared memory ONCE and multiplied into every
// template of the run (k_conv_cols_f fetches them from L2 per template, right where the
// product needs them -- a third of its warp stalls); the twiddles stay in registers
// for the whole batch; the groups take the templates of a run round-robin, each behind
// its own named barrier.
// ---------------------------------------------------------------------------
constexpr int kConvPThreads = 512;
constexpr int kConvPMaxBatch = 64;

template <int N, bool SPARSE>
SB_GLOBAL SB_LAUNCH_BOUNDS(kConvPThreads, 1)
k_conv_cols_p(Geom g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, int cnt, int angle_base,
              const float4* SB_RESTRICT trt, const float2* SB_RESTRICT fct, float4* SB_RESTRICT gbuf,
              const float2* SB_RESTRICT tw) {
    constexpr int T = N / E;
    constexpr int G = kConvPThreads / T;
    constexpr int PL = sbfft::padded_len(N);
    static_assert(T >= 32 && G >= 1, "k_conv_cols_p: one group must be whole warps");
    typedef ConvCtx<N, SPARSE, true> Ctx;
    const int grp = sb_tid() / T, t = sb_tid() % T;
    const int KX = g.Px / 2 + 1;
    const int kx = sb_bx();
    float2* sm = (float2*)sb_shared();
    float2* spec_s = sm + (long)G * 2 * PL;               // [2][N]
    int* s_meta = (int*)(spec_s + 2 * N);                  // [kConvPMaxBatch][4]: sy_lo, sy_hi, angle_id
    float2* tw_s = (float2*)(s_meta + 4 * kConvPMaxBatch);  // compact twiddle table
    sbfft::copy_ctw<N, float>(tw_s, tw, sb_tid(), kConvPThreads);

    for (int i = sb_tid(); i < cnt; i += kConvPThreads) {
        const Tmpl* p = tmpls + tmpl_base + i;
        s_meta[4 * i + 0] = p->sy_lo;
        s_meta[4 * i + 1] = p->sy_hi;
        s_meta[4 * i + 2] = p->angle_id - angle_base;
    }

    Ctx c;
    c.t = t;
    c.smA = sm + (long)grp * 2 * PL;
    c.smB = c.smA + PL;
    c.tw = tw_s;
    c.specA = spec_s + t;
    c.specB = spec_s + N + t;
    c.kx = kx;
    c.dly = g.dly;
    c.out_ny = g.out_ny;
    c.kpitch = g.kpitch;
    c.bar_id = 1 + grp;
    sb_sync();

    int s0 = 0;
#pragma unroll 1
    while (s0 < cnt) {
        const int a_loc = s_meta[4 * s0 + 2];
        int s1 = s0 + 1;
        while (s1 < cnt && s_meta[4 * s1 + 2] == a_loc) ++s1;
        if (s0 > 0) sb_sync();                              // the previous run's products are done
        {
            const float4* src = (const float4*)(fct + (((long)a_loc * 2) * KX + kx) * N);
            const float4* src2 = (const float4*)(fct + (((long)a_loc * 2 + 1) * KX + kx) * N);
            float4* dst = (float4*)spec_s;
            for (int i = sb_tid(); i < N / 2; i += kConvPThreads) {
                dst[i] = sb_ld_stream(src + i);
                dst[N / 2 + i] = sb_ld_stream(src2 + i);
            }
        }
        sb_sync();
        // SPARSE: a thread's only inputs are rows t and t - T of the template column; they are
        // fetched one template ahead, so that their latency hides behind the transform
        float4 in_lo = make_float4(0.f, 0.f, 0.f, 0.f), in_hi = in_lo;
        auto fetch_sparse = [&](int p_loc) {
            const int sy_lo = s_meta[4 * p_loc + 0], sy_hi = s_meta[4 * p_loc + 1];
            const float4* src = trt + ((long)p_loc * KX + kx) * g.syp;
            in_lo = make_float4(0.f, 0.f, 0.f, 0.f);
            in_hi = in_lo;
            if (t >= sy_lo && t <= sy_hi) in_lo = sb_ld_stream(src + (t - sy_lo));
            if (t - T >= sy_lo && t - T <= sy_hi) in_hi = sb_ld_stream(src + (t - T - sy_lo));
        };
        if (SPARSE && s0 + grp < s1) fetch_sparse(s0 + grp);
#pragma unroll 1
        for (int p_loc = s0 + grp; p_loc < s1; p_loc += G) {
            c.dst = gbuf + (long)p_loc * N * g.kpitch;
            float2 va[E], vb[E];
#pragma unroll
            for (int q = 0; q < E; ++q) {
                va[q] = make_float2(0.f, 0.f);
                vb[q] = make_float2(0.f, 0.f);
            }
            if (SPARSE) {
                va[0] = make_float2(in_lo.x, in_lo.y);
                vb[0] = make_float2(in_lo.z, in_lo.w);
                va[E - 1] = make_float2(in_hi.x, in_hi.y);
                vb[E - 1] = make_float2(in_hi.z, in_hi.w);
                if (p_loc + G < s1) fetch_sparse(p_loc + G);
            } else {
                const int sy_lo = s_meta[4 * p_loc + 0], sy_hi = s_meta[4 * p_loc + 1];
                const float4* src = trt + ((long)p_loc * KX + kx) * g.syp;
#pragma unroll
                for (int q = 0; q < E; ++q) {
                    const int qy = t + q * T;
                    const int s = qy < N / 2 ? qy : qy - N;
                    if (s >= sy_lo && s <= sy_hi) {
                        const float4 w = sb_ld_stream(src + (s - sy_lo));
                        va[q] = make_float2(w.x, w.y);
                        vb[q] = make_float2(w.z, w.w);
                    }
                }
            }
            c.va_fin = va;
            leapfrog<Ctx::K>(c, va, vb);                    // the last phase of field b writes gbuf
        }
        s0 = s1;
    }
}

// ---------------------------------------------------------------------------
// Fit kernel (complex64 fast path).  Per template and row: Hermitian-extended inverse row
// FFT of Gt + i Gm (real part xcorr, imaginary part T3), amplitude / SNR (core.py:360-367),
// edge mask (core.py:373-375), optional get_err_mask (core.py:369-371), running best-SNR
// select (core.py:198-243) in registers.  The raw-plane mode of match_template and the
// complex128 pipeline use k_fit_rows (sb_kernels.cuh).
// ---------------------------------------------------------------------------
constexpr int kFitMaxBatch = 64;

// X, T: raw outputs of the inverse transform (xcorr and T3 up to the exact power-of-two
// factors folded into FitT).  snr = |T1 / error| with error = (T3 - xcorr^2 / ts) / n + eps
// (core.py:362-367); the cancellation T3 - xcorr^2 / ts is evaluated with error-free products.
SB_DEVICE void fit_pixel_fast(float X, float T, const FitT& k, float& amp, float& snr) {
    amp = X * k.amp_k;                               // core.py:360
    const float pp = X * X;
    const float pe = fmaf(X, X, -pp);                // X*X = pp + pe exactly
    float num = fmaf(-pp, k.a_hi, T);
    num = fmaf(-pp, k.a_lo, num);
    num = fmaf(-pe, k.a_hi, num);
    const float t1 = pp * k.a_hi;                    // core.py:362
    const float err = fmaf(num, k.inv_n, k.eps_k);   // core.py:366
    snr = fabsf(sb_fdiv_fast(t1, err));              // core.py:367
}

// ---------------------------------------------------------------------------
// Nodata-masked fit (DESIGN.md 11).  Every template of a masked sweep has a companion record
// (t**2 * s2 + i M, same support) whose column pass multiplies by F[U] in both fields, so the
// inverse row transform of its gbuf plane is  D_t * s2 / norm + i D_m / norm  with
// D_t = t**2 (*) U and D_m = M (*) U, the template mass over the missing cells.
// ---------------------------------------------------------------------------
struct FitM {
    double ts;               // sum(t**2) of the template              core.py:356
    double dt_k;             // norm / s2: D_t = dt_k * Re(companion)
    double amp_f;            // xn: amp = X * xn / ts_m
    double a_f;              // xn**2 / tn: the epilogue's a = a_f / ts_m
    float dm_k;              // norm: D_m = dm_k * Im(companion)
    int n;                   // sum(M)
    int need;                // ceil(min_coverage * n): least n_valid of a candidate
    int pad;
};

// k_tmpl_sums has run over the chunk's 2 * cnt records (templates, then their companions)
SB_GLOBAL k_mask_consts(Geom g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, int cnt, double min_coverage,
                        const TSum* SB_RESTRICT sums, FitM* SB_RESTRICT fitm) {
    const int i = sb_bx() * 32 + sb_tid();
    if (i >= cnt) return;
    const Tmpl p = tmpls[tmpl_base + i];
    const double xn = g.norm / p.tscale, tn = g.norm / g.c2_scale;      // powers of two
    FitM m;
    m.ts = sums[i].ts;
    m.dt_k = g.norm / tmpls[tmpl_base + cnt + i].tscale;
    m.amp_f = xn;
    m.a_f = xn * xn / tn;
    m.dm_k = (float)g.norm;
    m.n = (int)rint(sums[i].n_eps);
    m.need = (int)ceil(min_coverage * (double)m.n);
    m.pad = 0;
    fitm[i] = m;
}

// one pixel of the masked fit: X, T raw outputs of the template's transform, d = (Im, Re) of its
// companion's (the transforms leave real and imaginary parts swapped).  Where no missing cell lies
// under M the template's exact constants are used, i.e. the arithmetic of the unmasked fit.
SB_DEVICE void fit_pixel_masked(float X, float T, const FitT& k, const FitM& m, float2 d, float& amp, float& snr) {
    const float miss = rintf(d.x * m.dm_k);                              // rint(D_m)
    if (miss == 0.f) {
        fit_pixel_fast(X, T, k, amp, snr);
        return;
    }
    const float nv = (float)m.n - miss;                                  // n_valid, exact
    if (!(nv >= (float)m.need)) {                                        // below min_coverage: no candidate
        amp = 0.f;
        snr = -1.f;
        return;
    }
    const double its = 1.0 / (m.ts - (double)d.y * m.dt_k);             // 1 / (ts - D_t)
    const float its_hi = (float)its, its_lo = (float)(its - (double)its_hi);
    FitT km = k;
    km.amp_k = (float)((double)its_hi * m.amp_f);
    km.a_hi = (float)((double)its_hi * m.a_f);
    km.a_lo = (float)((double)its_lo * m.a_f);
    km.inv_n = (float)(1.0 / ((double)nv + kEps));
    fit_pixel_fast(X, T, km, amp, snr);
}

// ---------------------------------------------------------------------------
// Fit confidence region (DESIGN.md 14): a second sweep of the same templates against best state 0
// (the first sweep's result) records, per pixel, the templates whose SNR s satisfies s > 0 and
// (double)s >= ratio * (double)best -- their count, the lowest and highest age rank, and a bitmask
// of orientation positions.  Integer atomics: the planes do not depend on the order in which
// sub-streams, batches or launches reach a pixel.
// ---------------------------------------------------------------------------
struct RegionOut {
    const float* best;        // best state 0, addressed by raster row (gi * nx + gj), read only
    int* count;               // planes of the plan's rows, addressed like `best`
    int* rank_lo;
    int* rank_hi;
    unsigned* bits;           // [words][plane]: orientation position p is bit p & 31 of word p >> 5
    const int* age_rank;      // per flat index: rank of its age among the search's ages
    const int* angle_pos;     // per flat index: orientation position
    long plane;               // elements of one plane
    double ratio;
};

template <bool REGION> struct RegionSlot {};
template <> struct RegionSlot<true> { RegionOut rg; };

SB_DEVICE void sb_atomic_add(int* p, int v) {
#ifdef SB_EMU
    __atomic_fetch_add(p, v, __ATOMIC_RELAXED);
#else
    atomicAdd(p, v);
#endif
}
SB_DEVICE void sb_atomic_min(int* p, int v) {
#ifdef SB_EMU
    int cur = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v < cur && !__atomic_compare_exchange_n(p, &cur, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
#else
    atomicMin(p, v);
#endif
}
SB_DEVICE void sb_atomic_max(int* p, int v) {
#ifdef SB_EMU
    int cur = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v > cur && !__atomic_compare_exchange_n(p, &cur, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
#else
    atomicMax(p, v);
#endif
}
SB_DEVICE void sb_atomic_or(unsigned* p, unsigned v) {
#ifdef SB_EMU
    __atomic_fetch_or(p, v, __ATOMIC_RELAXED);
#else
    atomicOr(p, v);
#endif
}

// the pixel's threshold in the running-best registers: the largest float <= ratio * best (so that
// s >= it is implied by (double)s >= ratio * best), +inf where there is no fit (best <= 0 or NaN)
SB_DEVICE float region_threshold(float best, double ratio) {
    if (!(best > 0.f)) return INFINITY;
    const double x = ratio * (double)best;
#ifdef SB_EMU
    float f = (float)x;
    if ((double)f > x) f = std::nextafter(f, -INFINITY);
    return f;
#else
    return __double2float_rd(x);
#endif
}

// ---------------------------------------------------------------------------
// Secondary fit (DESIGN.md 16): a second sweep of the same templates folds into best state 1 only the
// templates whose orientation position is at least min_sep from the position of the pixel's winner
// in best state 0 (the `pos` plane, k_secondary_pos).  An inadmissible candidate is skipped before it
// touches the running best; everything else is the search's fold, so state 1 is the max-fold over
// the admissible templates whatever the batches, sub-streams or launch order.
// ---------------------------------------------------------------------------
constexpr unsigned short kNoPos = 0xffff;          // `pos` of a pixel without a fit: nothing qualifies

struct SecondOut {
    const unsigned short* pos;    // winner's orientation position per pixel, addressed by raster row
    const int* angle_pos;         // per flat index: orientation position
    int n_pos;
    int min_sep;                  // in positions, >= 1
    int periodic;                 // positions 0 .. n_pos - 1 close into a circle
};

template <bool SECOND> struct SecondSlot {};
template <> struct SecondSlot<true> {
    SecondOut sec;
    int tpos;                     // orientation position of the current template
};

// the `pos` plane of a secondary fit from best state 0: the winner's orientation position where
// decode_best sees a hit (SNR > 0, index in range), kNoPos elsewhere (no fit, NaN)
SB_GLOBAL k_secondary_pos(long n, const float* SB_RESTRICT snr, const int* SB_RESTRICT idx,
                          const int* SB_RESTRICT angle_pos, int n_idx, unsigned short* SB_RESTRICT pos) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    const int k = idx[i];
    pos[i] = (snr[i] > 0.f && k >= 0 && k < n_idx) ? (unsigned short)angle_pos[k] : kNoPos;
}

// ---------------------------------------------------------------------------
// Sub-grid fit peak (DESIGN.md 17): a second sweep of the same templates records, at each pixel, the
// largest SNR of each of the four axis neighbours of the winner of best state 0 -- the templates one
// age rank either side at its orientation position, and one position either side at its age rank.
// The running-best registers hold each pixel's winner code (rank << 16 | pos, k_peak_code); every
// template carries the four winner codes it neighbours (`codes`, built on the host with the periodic
// wrap), so the test per pixel is four integer compares.  A hit is an integer atomicMax of the SNR's
// bits (positive floats order as their bits): the planes do not depend on batches, sub-streams or
// launch order.
// ---------------------------------------------------------------------------
constexpr unsigned kNoCode = 0xffffffffu;          // code of a pixel without a fit: it neighbours nothing

struct PeakOut {
    const unsigned* code;     // winner code per pixel, addressed by raster row (gi * nx + gj)
    int* planes;              // [age-][age+][ang-][ang+] float32 SNR bits, addressed like `code`
    const int4* codes;        // per flat index: the winner codes whose age-, age+, ang-, ang+ neighbour
                              // it is (0xfffffffe where there is none: rank 0xffff is nobody's)
    long plane;               // elements of one plane
};

template <bool PEAK> struct PeakSlot {};
template <> struct PeakSlot<true> {
    PeakOut pk;
    int4 tcodes;              // `codes` of the current template
};

// the code plane of a fit peak from best state 0: (age rank << 16) | orientation position of the winner
// where decode_best sees a hit (SNR > 0, index in range), kNoCode elsewhere (no fit, NaN)
SB_GLOBAL k_peak_code(long n, const float* SB_RESTRICT snr, const int* SB_RESTRICT idx,
                      const int* SB_RESTRICT age_rank, const int* SB_RESTRICT angle_pos, int n_idx,
                      unsigned* SB_RESTRICT code) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    const int k = idx[i];
    code[i] = (snr[i] > 0.f && k >= 0 && k < n_idx) ? ((unsigned)age_rank[k] << 16) | (unsigned)angle_pos[k] : kNoCode;
}

// Fit peak (sb_peak_finalize): [amp, age, angle, snr] of best state 0 as k_finalize decodes it, then
// [age_peak, angle_peak, snr_peak, refined] from the winner code and the four neighbour SNRs, by the
// vertex of the parabola through the winner and its two neighbours on each axis (ages on the log10
// axis `lx`, log10 of the sorted ages).  Float64 without contraction (sb_mul ...), so that planes 5..7
// can equal a NumPy restatement bit for bit; only age_peak goes through exp10.  Planes 4..7 are 0
// where the pixel has no fit, [0, 0, NaN, 0] where its SNR is NaN.
SB_GLOBAL k_peak_finalize(long n, long plane, const float* SB_RESTRICT snr, const float* SB_RESTRICT amp,
                          const int* SB_RESTRICT idx, const unsigned* SB_RESTRICT code,
                          const float* SB_RESTRICT nb, const double* SB_RESTRICT age_of,
                          const double* SB_RESTRICT angle_of, int n_idx, const double* SB_RESTRICT lx, int n_ranks,
                          int n_pos, int periodic, double step, double* SB_RESTRICT out8) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    const float s = snr[i];
    double o[4];
    decode_best(s, idx[i], amp + i, age_of, angle_of, n_idx, o);
    double age_pk = 0.0, ang_pk = 0.0, snr_pk = s != s ? (double)s : 0.0, refined = 0.0;
    if (o[3] > 0.0) {
        const double s0 = o[3];
        const unsigned c = code[i];
        const int r = (int)(c >> 16), p = (int)(c & 0xffffu);
        const double am = (double)nb[i], ap = (double)nb[plane + i];
        const double gm = (double)nb[2 * plane + i], gp = (double)nb[3 * plane + i];
        double g_age = 0.0, g_ang = 0.0;
        age_pk = o[1];
        ang_pk = o[2];
        if (r > 0 && r < n_ranks - 1 && am > 0.0 && ap > 0.0) {
            const double dm = sb_sub(s0, am), dp = sb_sub(s0, ap);
            if (sb_add(dm, dp) > 0.0) {
                const double hm = sb_sub(lx[r], lx[r - 1]), hp = sb_sub(lx[r + 1], lx[r]);
                const double num = sb_sub(sb_mul(dm, sb_mul(hp, hp)), sb_mul(dp, sb_mul(hm, hm)));
                const double u = sb_div(num, sb_mul(2.0, sb_add(sb_mul(dm, hp), sb_mul(dp, hm))));
                age_pk = exp10(sb_add(lx[r], u));
                g_age = sb_div(sb_mul(u, num), sb_mul(sb_mul(sb_mul(2.0, hm), hp), sb_add(hm, hp)));
                refined = 1.0;
            }
        }
        if ((periodic ? n_pos >= 3 : (p > 0 && p < n_pos - 1)) && gm > 0.0 && gp > 0.0) {
            const double dm = sb_sub(s0, gm), dp = sb_sub(s0, gp);
            const double sum = sb_add(dm, dp);
            if (sum > 0.0) {
                const double t = sb_sub(dm, dp);
                ang_pk = sb_add(o[2], sb_mul(sb_div(t, sb_mul(2.0, sum)), step));
                g_ang = sb_div(sb_mul(t, t), sb_mul(8.0, sum));
                refined = sb_add(refined, 2.0);
            }
        }
        snr_pk = sb_add(sb_add(s0, g_age), g_ang);
    }
    out8[i] = o[0];
    out8[n + i] = o[1];
    out8[2 * n + i] = o[2];
    out8[3 * n + i] = o[3];
    out8[4 * n + i] = age_pk;
    out8[5 * n + i] = ang_pk;
    out8[6 * n + i] = snr_pk;
    out8[7 * n + i] = refined;
}

// ---------------------------------------------------------------------------
// k_fit_rows_g<Px>: grid (Py / 2 / GP).  The two transforms
// a thread group pipelines are the two raster rows that share every 32-byte sector of the
// interleaved planes (gbuf_index), of ONE template: a thread fetches whole sectors with
// 256-bit loads and feeds one half to each row, so the planes cross the L2 -> SM crossbar
// in full sectors (a one-row kernel uses 16 bytes of every 32 it requests).  The running best keeps
// only the SNR in registers; amplitude and flat index go straight to the best state when a
// pixel improves (rare after the first templates of a sweep).
// ---------------------------------------------------------------------------
// MASKED (k_fit_rows_gm): per template, the companion's row pair runs first (comp) and parks its
// outputs in `park`, every thread in the slots only it reads back; then the template's own.
// REGION (k_fit_rows_gr / _gmr): bsA / bsB hold each pixel's region threshold (region_threshold) and
// never change; a candidate is confirmed in float64 and recorded in the region planes (region_hit).
// SECOND (k_fit_rows_gs / _gms): a candidate the separation rules out (second_ok) is skipped.
// PEAK (k_fit_rows_gp / _gmp): bsA / bsB hold each pixel's winner code (as float bits) and never
// change; a template that neighbours the winner (peak_any) and has SNR > 0 is recorded (peak_hit).
template <int N, bool MASKED = false, bool REGION = false, bool SECOND = false, bool PEAK = false>
struct FitPairCtx : RegionSlot<REGION>, SecondSlot<SECOND>, PeakSlot<PEAK> {
    static constexpr int K = sbfft::num_stages(N);
    static constexpr int T = N / E;
    static constexpr int LOG2T = ilog2(T);
    int t;
    float2 *smA, *smB;
    const float2* tw;
    const float4* pair;               // the template's row pair: element kk of row F at pair[2 * kk + F]
    const FitT* s_fit;
    const FitM* s_fm;                 // MASKED only
    float2* park;                     // MASKED only: [row F][N]
    bool comp;                        // MASKED only: this pass is the companion's
    int slot;
    int giA, giB;                     // raster rows of the two streams
    bool actA, actB;
    int ox, m0, out_nx, nx;
    float* best_amp;
    int* best_idx;
    const int4* cross;                // get_err_mask column ranges per (angle, raster row), or null
    int ny;
    float (&bsA)[E];
    float (&bsB)[E];
    float2 (&vb_in)[E];               // stream b's input, filled together with stream a's
    unsigned chg;                     // bit q (+16 for row B): the pixel's best SNR changed

    SB_DEVICE FitPairCtx(float (&a)[E], float (&b)[E], float2 (&vb)[E]) : bsA(a), bsB(b), vb_in(vb), chg(0u) {}

    SB_DEVICE void bar() const { sb_sync(); }

    template <int P> SB_DEVICE void twid(float2 (&w)[TW]) { sbfft::load_tw<N, P, float, true>(w, t, tw); }

    SB_DEVICE unsigned mask(const FitT& k, int gi, bool act) const {
        if (!act || gi < k.i_lo || gi > k.i_hi) return 0u;
        int jl = k.j_lo, jh = k.j_hi;
        if (k.errmode != 0) {
            // snr[get_err_mask()] = 0 (core.py:369-371): a pixel whose SNR is 0 never wins the
            // fold, so inside a search the mask only narrows the row's candidate columns
            const int4 cr = cross[(long)k.angle_id * ny + gi];
            jl = max(jl, k.errmode == 1 ? cr.x : cr.z);
            jh = min(jh, k.errmode == 1 ? cr.y : cr.w);
        }
        const int lo = max(jl - ox, 0), hi = min(jh - ox, out_nx - 1);
        if (lo > hi) return 0u;
        const int qlo = max((lo - m0 + T - 1) >> LOG2T, 0);
        const int qhi = min((hi - m0) >> LOG2T, E - 1);
        return qlo <= qhi ? ((2u << qhi) - (1u << qlo)) : 0u;
    }

    // X(k) = Gt(k) + i Gm(k) and X(N-k) = conj Gt(k) + i conj Gm(k) come ready (and swapped: inverse
    // via forward) in the element (gbuf_pack)
    SB_DEVICE static float2 herm(const float4 g4, bool direct) {
        return direct ? make_float2(g4.x, g4.y) : make_float2(g4.z, g4.w);
    }

    // REGION: template `idx` has SNR `snr` >= the threshold at pixel `pix` (gi * nx + gj)
    SB_DEVICE void region_hit(long pix, float snr, int idx) const {
        const RegionOut& r = this->rg;
        const float best = r.best[pix];
        if (!(best > 0.f && (double)snr >= r.ratio * (double)best)) return;
        sb_atomic_add(r.count + pix, 1);
        const int rank = r.age_rank[idx];
        sb_atomic_min(r.rank_lo + pix, rank);
        sb_atomic_max(r.rank_hi + pix, rank);
        const int p = r.angle_pos[idx];
        sb_atomic_or(r.bits + (long)(p >> 5) * r.plane + pix, 1u << (p & 31));
    }

    // SECOND: the current template is at least min_sep positions from the winner at pixel `pix`
    SB_DEVICE bool second_ok(long pix) const {
        const SecondOut& s = this->sec;
        const int ps = s.pos[pix];
        if (ps == kNoPos) return false;
        int d = abs(this->tpos - ps);
        if (s.periodic) d = min(d, s.n_pos - d);
        return d >= s.min_sep;
    }

    // PEAK: the current template is an axis neighbour of the winner of code `c`
    SB_DEVICE bool peak_any(unsigned c) const {
        const int4 t = this->tcodes;
        const int v = (int)c;
        return (v == t.x) | (v == t.y) | (v == t.z) | (v == t.w);
    }
    // PEAK: record SNR `snr` > 0 of the current template, a neighbour of code `c`, at pixel `pix`
    SB_DEVICE void peak_hit(long pix, unsigned c, float snr) const {
        const int4 t = this->tcodes;
        const int v = (int)c;
        const int j = v == t.x ? 0 : v == t.y ? 1 : v == t.z ? 2 : 3;
        sb_atomic_max(this->pk.planes + j * this->pk.plane + pix, (int)sb_float_bits(snr));
    }

    template <int F> SB_DEVICE void epilogue(const float2 (&v)[E], float (&bs)[E]) {
        const int gi = F == 0 ? giA : giB;
        const FitT k = s_fit[slot];
        const unsigned mk = mask(k, gi, F == 0 ? actA : actB);
        float* pa = best_amp + ((long)gi * nx + ox);
        int* pi = best_idx + ((long)gi * nx + ox);
#pragma unroll
        for (int q = 0; q < E; ++q) {
            float amp, snr;
            if constexpr (MASKED) fit_pixel_masked(v[q].y, v[q].x, k, s_fm[slot], park[F * N + t + q * T], amp, snr);
            else fit_pixel_fast(v[q].y, v[q].x, k, amp, snr);
            snr = ((mk >> q) & 1u) ? snr : -1.f;              // edge-masked: never wins
            if constexpr (PEAK) {
                const unsigned cq = sb_float_bits(bs[q]);
                if (snr > 0.f && peak_any(cq)) peak_hit((long)gi * nx + ox + ((m0 + q * T) & (N - 1)), cq, snr);
                continue;
            }
            // first maximum wins (core.py:230-240); equal positive SNRs (in float32 mostly the
            // -90 / +90 degree pair) go to the lower flat index, whatever the batch order.
            // (A branch-free select over the 16 pixels was measured 3 % slower: it spills.)
            if (snr >= bs[q] && snr > 0.f) {
                const int jo = (m0 + q * T) & (N - 1);
                if constexpr (REGION) {
                    region_hit((long)gi * nx + ox + jo, snr, k.idx);
                    continue;
                }
                if constexpr (SECOND) {
                    if (!second_ok((long)gi * nx + ox + jo)) continue;
                }
                if (snr > bs[q] || k.idx < pi[jo]) {
                    bs[q] = snr;
                    pa[jo] = amp;
                    pi[jo] = k.idx;
                    chg |= 1u << (q + 16 * F);
                }
            }
        }
    }

#ifdef SB_F32X2
    // Two pixels (q, q + 8) per packed instruction: X = xcorr pair, Tp = T3 pair (fit_pixel_fast).
    // The window mask is applied to the candidate bits, not to the 16 values; improvements
    // (rare after the first templates of a sweep) are resolved after the common path.
    static constexpr bool SOA = K > 1 && !MASKED;
    template <int F> SB_DEVICE void epilogue2(const sbfft::pk_t (&re)[8], const sbfft::pk_t (&im)[8], float (&bs)[E]) {
        using namespace sbfft;
        const int gi = F == 0 ? giA : giB;
        const FitT k = s_fit[slot];
        const unsigned mk = mask(k, gi, F == 0 ? actA : actB);
        float2 snr2[8], amp2[8];
        unsigned cand = 0u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const pk_t X = im[j], Tp = re[j];
            amp2[j] = unpk(mul2(X, pk(k.amp_k, k.amp_k)));                    // core.py:360
            const pk_t pp = mul2(X, X);
            const float2 ppf = unpk(pp);
            const pk_t npp = pk(-ppf.x, -ppf.y);
            const float2 pef = unpk(fma2(X, X, npp));                          // X*X = pp + pe exactly
            pk_t num = fma2(npp, pk(k.a_hi, k.a_hi), Tp);
            num = fma2(npp, pk(k.a_lo, k.a_lo), num);
            num = fma2(pk(-pef.x, -pef.y), pk(k.a_hi, k.a_hi), num);
            const float2 t1 = unpk(mul2(pp, pk(k.a_hi, k.a_hi)));              // core.py:362
            const float2 err = unpk(fma2(num, pk(k.inv_n, k.inv_n), pk(k.eps_k, k.eps_k)));   // core.py:366
            const float s_lo = fabsf(sb_fdiv_fast(t1.x, err.x));               // core.py:367
            const float s_hi = fabsf(sb_fdiv_fast(t1.y, err.y));
            snr2[j] = make_float2(s_lo, s_hi);
            // (a NaN SNR -- NaN in the DEM -- never wins here; k_poison_windows marks those pixels)
            if constexpr (PEAK) {
                cand |= (s_lo > 0.f && peak_any(sb_float_bits(bs[j]))) ? (1u << j) : 0u;
                cand |= (s_hi > 0.f && peak_any(sb_float_bits(bs[j + 8]))) ? (1u << (j + 8)) : 0u;
            } else {
                cand |= (s_lo >= bs[j] && s_lo > 0.f) ? (1u << j) : 0u;
                cand |= (s_hi >= bs[j + 8] && s_hi > 0.f) ? (1u << (j + 8)) : 0u;
            }
        }
        cand &= mk;                                                            // edge-masked: never wins
        if (cand != 0u) {
            float* pa = best_amp + ((long)gi * nx + ox);
            int* pi = best_idx + ((long)gi * nx + ox);
            // first maximum wins (core.py:230-240); equal positive SNRs (in float32 mostly the
            // -90 / +90 degree pair) go to the lower flat index, whatever the batch order
#pragma unroll
            for (int q = 0; q < E; ++q) {
                if ((cand >> q) & 1u) {
                    const float snr = q < 8 ? snr2[q & 7].x : snr2[q & 7].y;
                    const float amp = q < 8 ? amp2[q & 7].x : amp2[q & 7].y;
                    const int jo = (m0 + q * T) & (N - 1);
                    if constexpr (PEAK) {
                        peak_hit((long)gi * nx + ox + jo, sb_float_bits(bs[q]), snr);
                        continue;
                    }
                    if constexpr (REGION) {
                        region_hit((long)gi * nx + ox + jo, snr, k.idx);
                        continue;
                    }
                    if constexpr (SECOND) {
                        if (!second_ok((long)gi * nx + ox + jo)) continue;
                    }
                    if (snr > bs[q] || k.idx < pi[jo]) {
                        bs[q] = snr;
                        pa[jo] = amp;
                        pi[jo] = k.idx;
                        chg |= 1u << (q + 16 * F);
                    }
                }
            }
        }
    }
#else
    static constexpr bool SOA = false;
#endif

    template <int P, int F> SB_DEVICE void phase(float2 (&v)[E], const float2 (&w)[TW]) {
        if constexpr (P == 0 && F == 0) {
#pragma unroll
            for (int q = 0; q < E; ++q) {
                bool direct = q < E / 2;
                int kk = q < E / 2 ? t + q * T : N - (t + q * T);
                if (q == E / 2) { direct = t == 0; kk = direct ? N / 2 : N / 2 - t; }
                float4 ga, gb;
                sb_ld_sector(pair + kGbufRows * kk, ga, gb);
                v[q] = herm(ga, direct);
                vb_in[q] = herm(gb, direct);
            }
        }
#ifdef SB_F32X2
        if constexpr (P == K - 1 && SOA) {
            sbfft::pk_t re[8], im[8];
            sbfft::stage_math_soa<N, P>(v, w, re, im);
            if constexpr (F == 0) epilogue2<0>(re, im, bsA);
            else epilogue2<1>(re, im, bsB);
            return;
        }
#endif
        sbfft::stage_math<N, P, float>(v, w);
        if constexpr (P == K - 1) {
            if constexpr (MASKED) {
                if (comp) {
#pragma unroll
                    for (int q = 0; q < E; ++q) park[F * N + t + q * T] = v[q];
                    return;
                }
            }
            if constexpr (F == 0) epilogue<0>(v, bsA);
            else epilogue<1>(v, bsB);
        }
    }
    template <int P, int F> SB_DEVICE void store(const float2 (&v)[E]) {
        sbfft::stage_store<N, P, float>(v, t, F == 0 ? smA : smB);
    }
    template <int F> SB_DEVICE void load(float2 (&v)[E]) { sbfft::stage_load<N, float>(v, t, F == 0 ? smA : smB); }
};

// shared memory of k_fit_rows_gm beyond k_fit_rows_g's: the batch's FitM, then the park buffers
template <int N>
SB_CONSTEXPR size_t fit_masked_extra_smem() {
    return kFitMaxBatch * sizeof(FitM) + (size_t)((N / E > 256 ? N / E : 256) / (N / E)) * 2 * N * sizeof(float2);
}

template <int N, bool MASKED, bool REGION = false, bool SECOND = false, bool PEAK = false>
SB_DEVICE void fit_rows_g_body(const Geom& g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
                               const FitM* SB_RESTRICT fitm, int comp_off, const float4* SB_RESTRICT gbuf,
                               float* SB_RESTRICT best_snr, float* SB_RESTRICT best_amp, int* best_idx,
                               const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross, long sub_stride,
                               const RegionOut& rg = RegionOut(), const SecondOut& sec = SecondOut(),
                               const PeakOut& pk = PeakOut()) {
    // grid.y > 1 (small rasters, whose row pairs alone do not fill the GPU): the templates of the
    // launch are dealt round-robin to grid.y sub-streams; sub-stream j folds into copy j of the
    // best state (best_* + j * sub_stride; copy 0 is the state itself) and k_best_fold merges the
    // copies after the sweep.
    // `slots` (optional): the `count` batch slots this launch folds -- the templates of one best
    // state (template scale) inside a batch that mixes several; null: slots 0 .. count - 1.
    // best_*: the state's planes, offset so that raster row gi is at gi * nx (row slabs).
    // `cross` (templates with get_err_mask only): per (angle, raster row) the column ranges
    // with xr > 0 (.x .. .y) and xr < 0 (.z .. .w), k_err_cross.
    // REGION: best_* are unused; the thresholds come from rg.best (state 0 for every sub-stream)
    // and nothing writes a best state.
    // SECOND: best_* are state 1's planes; `sec` rules out the templates too close to the winner.
    // PEAK: as REGION, with the winner codes of pk.code and the neighbour planes of `pk`.
    constexpr int T = N / E;
    constexpr int THREADS = T > 256 ? T : 256;
    constexpr int GP = THREADS / T;
    constexpr int PL = sbfft::padded_len(N);
    typedef FitPairCtx<N, MASKED, REGION, SECOND, PEAK> Ctx;
    const int grp = sb_tid() / T, t = sb_tid() % T;
    float2* sm = (float2*)sb_shared();
    FitT* s_fit = (FitT*)(sm + (long)GP * 2 * PL);
    // [kFitMaxBatch] active templates, [kFitMaxBatch] flags (16-byte aligned: the compiler reads
    // them with vector loads), the count -- s_list[2 * kFitMaxBatch] --, [kFitMaxBatch] gbuf slots
    int* s_list = (int*)(s_fit + kFitMaxBatch);
    int* s_flag = s_list + kFitMaxBatch;
    int* s_gslot = s_flag + kFitMaxBatch + 2;
    float2* tw_s = (float2*)(s_gslot + kFitMaxBatch);
    sbfft::copy_ctw<N, float>(tw_s, tw, sb_tid(), THREADS);
    FitM* s_fm = nullptr;
    float2* park = nullptr;
    if constexpr (MASKED) {
        s_fm = (FitM*)(tw_s + sbfft::ctw_count<float>(N));
        park = (float2*)(s_fm + kFitMaxBatch) + (long)grp * 2 * N;
        if (sb_tid() < count) s_fm[sb_tid()] = fitm[slots ? slots[sb_tid()] : sb_tid()];
    }
    const int pairs = g.Py / 2;
    const int pr = min(sb_bx() * GP + grp, pairs - 1);    // row pair of the FFT domain
    const int ioA = (2 * pr + g.dly) & (g.Py - 1), ioB = (2 * pr + 1 + g.dly) & (g.Py - 1);
    const bool actA = sb_bx() * GP + grp < pairs && ioA < g.out_ny;
    const bool actB = sb_bx() * GP + grp < pairs && ioB < g.out_ny;

    // stage the batch's scalars; list the templates whose window meets one of this CTA's rows
    if (sb_tid() < count) {
        const int slot = slots ? slots[sb_tid()] : sb_tid();
        const FitT k = fit[slot];
        s_fit[sb_tid()] = k;
        s_gslot[sb_tid()] = slot;
        int flag = 0;
        for (int r = 0; r < 2 * GP && sb_tid() % sb_nby() == sb_by(); ++r) {
            const int m = 2 * sb_bx() * GP + r;
            const int io = (m + g.dly) & (g.Py - 1);
            if (m < g.Py && io < g.out_ny && g.oy + io >= k.i_lo && g.oy + io <= k.i_hi) flag = 1;
        }
        s_flag[sb_tid()] = flag;
    }
    sb_sync();
    if (sb_tid() < count) {
        int pos = 0;
        for (int i = 0; i < sb_tid(); ++i) pos += s_flag[i];
        if (s_flag[sb_tid()]) s_list[pos] = sb_tid();
        if (sb_tid() == count - 1) s_list[2 * kFitMaxBatch] = pos + s_flag[sb_tid()];
    }
    sb_sync();
    const int n_act = s_list[2 * kFitMaxBatch];

    float bsA[E], bsB[E];
    float2 va[E], vb[E];
    Ctx c(bsA, bsB, vb);
    c.t = t;
    c.smA = sm + (long)grp * 2 * PL;
    c.smB = c.smA + PL;
    c.tw = tw_s;
    c.giA = g.oy + ioA;
    c.giB = g.oy + ioB;
    c.actA = actA;
    c.actB = actB;
    c.ox = g.ox;
    c.m0 = t + g.dlx;
    c.out_nx = g.out_nx;
    c.nx = g.nx;
    c.s_fit = s_fit;
    c.s_fm = s_fm;
    c.park = park;
    c.comp = false;
    if constexpr (SECOND) c.sec = sec;
    if constexpr (REGION) {
        c.rg = rg;
    } else if constexpr (PEAK) {
        c.pk = pk;
    } else {
        best_snr += sb_by() * sub_stride;
        best_amp += sb_by() * sub_stride;
        best_idx += sb_by() * sub_stride;
    }
    c.best_amp = best_amp;
    c.best_idx = best_idx;
    c.cross = cross;
    c.ny = g.ny;
#pragma unroll
    for (int q = 0; q < E; ++q) {
        const int jo = (t + q * T + g.dlx) & (N - 1);
        const bool in = jo < g.out_nx;
        if constexpr (REGION) {
            bsA[q] = (actA && in) ? region_threshold(rg.best[(long)c.giA * g.nx + g.ox + jo], rg.ratio) : INFINITY;
            bsB[q] = (actB && in) ? region_threshold(rg.best[(long)c.giB * g.nx + g.ox + jo], rg.ratio) : INFINITY;
        } else if constexpr (PEAK) {
            bsA[q] = sb_bits_float((actA && in) ? pk.code[(long)c.giA * g.nx + g.ox + jo] : kNoCode);
            bsB[q] = sb_bits_float((actB && in) ? pk.code[(long)c.giB * g.nx + g.ox + jo] : kNoCode);
        } else {
            bsA[q] = (actA && in) ? best_snr[(long)c.giA * g.nx + g.ox + jo] : 0.f;
            bsB[q] = (actB && in) ? best_snr[(long)c.giB * g.nx + g.ox + jo] : 0.f;
        }
    }
    const long row_off = gbuf_index(2 * pr, 0, g.kpitch);
    const long tmpl_pitch = (long)g.Py * g.kpitch;
    // 128-byte lines that hold the row pair (with kGbufRows > 2 they are shared with the
    // neighbouring pairs, whose CTAs run at the same time)
    const int lines = (kGbufRows * (g.Px / 2 + 1) + 7) / 8;
    const long pf_off = gbuf_index(2 * pr - (2 * pr) % kGbufRows, 0, g.kpitch);

#pragma unroll 1
    for (int i = 0; i < n_act; ++i) {
        const int p = s_list[i];
        c.slot = p;
        if constexpr (SECOND) c.tpos = sec.angle_pos[s_fit[p].idx];
        if constexpr (PEAK) c.tcodes = pk.codes[s_fit[p].idx];
        if constexpr (MASKED) {
            // the companion's row pair first (its gbuf plane is comp_off slots further on); no
            // barrier between the two passes, for the reason given below
            c.pair = gbuf + (s_gslot[p] + comp_off) * tmpl_pitch + row_off;
            c.comp = true;
            const float4* nx0 = gbuf + s_gslot[p] * tmpl_pitch + pf_off;
            for (int l = t; l < lines; l += T) sb_prefetch_l2(nx0 + 8 * l);
            leapfrog<Ctx::K>(c, va, vb);
            c.comp = false;
        }
        c.pair = gbuf + s_gslot[p] * tmpl_pitch + row_off;
        if (i + 1 < n_act) {                                // next template's row pair towards L2
            const float4* nx0 = gbuf + (s_gslot[s_list[i + 1]] + (MASKED ? comp_off : 0)) * tmpl_pitch + pf_off;
            for (int l = t; l < lines; l += T) sb_prefetch_l2(nx0 + 8 * l);
        }
        // no barrier between templates: buffer A was last read before the final barrier,
        // buffer B is next written after the coming template's first barrier
        leapfrog<Ctx::K>(c, va, vb);
    }
    if constexpr (!REGION && !PEAK) {
#pragma unroll
        for (int q = 0; q < E; ++q) {
            const int jo = (t + q * T + g.dlx) & (N - 1);
            if ((c.chg >> q) & 1u) best_snr[(long)c.giA * g.nx + g.ox + jo] = bsA[q];
            if ((c.chg >> (q + 16)) & 1u) best_snr[(long)c.giB * g.nx + g.ox + jo] = bsB[q];
        }
    }
}

template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), (N / E > 256 ? 1 : 2))
k_fit_rows_g(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
             const float4* SB_RESTRICT gbuf, float* SB_RESTRICT best_snr, float* SB_RESTRICT best_amp, int* best_idx,
             const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross, long sub_stride) {
    fit_rows_g_body<N, false>(g, count, slots, fit, nullptr, 0, gbuf, best_snr, best_amp, best_idx, tw, cross,
                              sub_stride);
}

// k_fit_rows_g of a masked sweep: `fitm` per batch slot, the companion of slot s in gbuf slot
// s + comp_off.  One CTA per SM (the park buffers), so the kernel may use every register.
template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), 1)
k_fit_rows_gm(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
              const FitM* SB_RESTRICT fitm, int comp_off, const float4* SB_RESTRICT gbuf, float* SB_RESTRICT best_snr,
              float* SB_RESTRICT best_amp, int* best_idx, const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross,
              long sub_stride) {
    fit_rows_g_body<N, true>(g, count, slots, fit, fitm, comp_off, gbuf, best_snr, best_amp, best_idx, tw, cross,
                             sub_stride);
}

// the threshold pass of a fit confidence region (sb_region_sweep): k_fit_rows_g / k_fit_rows_gm with
// the region planes `rg` in place of the best state; grid.y sub-streams all read state 0
template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), (N / E > 256 ? 1 : 2))
k_fit_rows_gr(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
              const float4* SB_RESTRICT gbuf, const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross,
              RegionOut rg) {
    fit_rows_g_body<N, false, true>(g, count, slots, fit, nullptr, 0, gbuf, nullptr, nullptr, nullptr, tw, cross, 0,
                                    rg);
}

template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), 1)
k_fit_rows_gmr(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
               const FitM* SB_RESTRICT fitm, int comp_off, const float4* SB_RESTRICT gbuf,
               const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross, RegionOut rg) {
    fit_rows_g_body<N, true, true>(g, count, slots, fit, fitm, comp_off, gbuf, nullptr, nullptr, nullptr, tw, cross, 0,
                                   rg);
}

// the sweep of a secondary fit (sb_secondary_sweep): k_fit_rows_g / k_fit_rows_gm folding into best
// state 1 (best_*) only the templates `sec` admits at each pixel
template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), (N / E > 256 ? 1 : 2))
k_fit_rows_gs(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
              const float4* SB_RESTRICT gbuf, float* SB_RESTRICT best_snr, float* SB_RESTRICT best_amp, int* best_idx,
              const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross, long sub_stride, SecondOut sec) {
    fit_rows_g_body<N, false, false, true>(g, count, slots, fit, nullptr, 0, gbuf, best_snr, best_amp, best_idx, tw,
                                           cross, sub_stride, RegionOut(), sec);
}

template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), 1)
k_fit_rows_gms(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
               const FitM* SB_RESTRICT fitm, int comp_off, const float4* SB_RESTRICT gbuf, float* SB_RESTRICT best_snr,
               float* SB_RESTRICT best_amp, int* best_idx, const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross,
               long sub_stride, SecondOut sec) {
    fit_rows_g_body<N, true, false, true>(g, count, slots, fit, fitm, comp_off, gbuf, best_snr, best_amp, best_idx, tw,
                                          cross, sub_stride, RegionOut(), sec);
}

// the neighbour pass of a fit peak (sb_peak_sweep): k_fit_rows_g / k_fit_rows_gm recording the axis
// neighbours of each pixel's winner in the planes of `pk`; grid.y sub-streams all read state 0
template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), (N / E > 256 ? 1 : 2))
k_fit_rows_gp(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
              const float4* SB_RESTRICT gbuf, const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross,
              PeakOut pk) {
    fit_rows_g_body<N, false, false, false, true>(g, count, slots, fit, nullptr, 0, gbuf, nullptr, nullptr, nullptr, tw,
                                                  cross, 0, RegionOut(), SecondOut(), pk);
}

template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), 1)
k_fit_rows_gmp(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
               const FitM* SB_RESTRICT fitm, int comp_off, const float4* SB_RESTRICT gbuf,
               const float2* SB_RESTRICT tw, const int4* SB_RESTRICT cross, PeakOut pk) {
    fit_rows_g_body<N, true, false, false, true>(g, count, slots, fit, fitm, comp_off, gbuf, nullptr, nullptr, nullptr,
                                                 tw, cross, 0, RegionOut(), SecondOut(), pk);
}

// Hermitian split (sb_kernels.cuh) of the spectrum parked in natural order in `sm`
template <int N>
SB_DEVICE void split_from_shared(const float2* sm, int t, float4 (&h)[E / 2 + 1]) {
    constexpr int T = N / E;
#pragma unroll
    for (int q = 0; q < E / 2; ++q) {
        const int k = t + q * T;
        const float2 a = sm[sbfft::pad_index(k)];
        const float2 zp = sm[sbfft::pad_index((N - k) & (N - 1))];
        h[q] = make_float4(0.5f * (a.x + zp.x), 0.5f * (a.y - zp.y), 0.5f * (a.y + zp.y), -0.5f * (a.x - zp.x));
    }
    const float2 ny = sm[sbfft::pad_index(N / 2)];
    h[E / 2] = make_float4(ny.x, 0.f, ny.y, 0.f);
}

// ---------------------------------------------------------------------------
// Curvature spectra without one 2-D transform per orientation.  The directional Laplacian is
// linear in the three second differences (dem.py:103-104):
//     curv(a)   = c2 dxx - sc dxy + s2 dyy                      (c2 = cos^2 a, sc = 2 sin a cos a, s2 = sin^2 a)
//     curv(a)^2 = c2^2 dxx^2 + sc^2 dxy^2 + s2^2 dyy^2 - 2 c2 sc dxx dxy + 2 c2 s2 dxx dyy - 2 sc s2 dxy dyy
// and so is the Fourier transform: the spectra of the NINE planes (3 differences, 6 products)
// are computed once per FFT tile (five packed pairs through k_diff_rows_f / k_curv_cols) and
// every orientation's F[curv], F[curv^2] are combinations of them with nine scalars --
// k_combine_spectra, an elementwise pass at HBM speed -- instead of a row kernel and a column
// kernel per orientation.  Plane order (pair pp, field f -> plane 2 pp + f):
//   0 dxx   1 dxy   2 dyy   3 s dxx^2   4 s dxy^2   5 s dyy^2   6 s dxx dxy   7 s dxx dyy   8 s dxy dyy
//   9 U (the nodata plane of a masked search, k_second_differences_m; 0 otherwise)
// (s = c2_scale, the power of two that brings the quadratic planes to the magnitude of the
// linear ones in the packed transforms).
// ---------------------------------------------------------------------------
constexpr int kDiffPairs = 5;
constexpr int kDiffPlanes = 9;

template <int N, bool WITH_U = false>
struct DiffCtx {
    static constexpr int K = sbfft::num_stages(N);
    static constexpr int T = N / E;
    int t;
    float2 *smA, *smB;
    const float2* tw;
    const float4* diffs;               // [pixel][dxx, dxy, dyy, -] float32
    int pp;                            // plane pair
    int oy, ox, ny, nx, need_y_lo, need_x_lo, need_x_hi, split_x, poison;
    int row0;
    float c2_scale;
    int rp;                            // row pair: rows 2 rp (stream a) and 2 rp + 1 (stream b)
    int need_rows;

    SB_DEVICE void bar() const { sb_sync(); }
    template <int P> SB_DEVICE void twid(float2 (&w)[TW]) { sbfft::load_tw<N, P, float>(w, t, tw); }

    SB_DEVICE float2 planes(const float4 d) const {
        const float s = c2_scale;
        switch (pp) {
            case 0: return make_float2(d.x, d.y);
            case 1: return make_float2(d.z, d.x * d.x * s);
            case 2: return make_float2(d.y * d.y * s, d.z * d.z * s);
            case 3: return make_float2(d.x * d.y * s, d.x * d.z * s);
            default: return make_float2(d.y * d.z * s, WITH_U ? d.w : 0.f);     // d.w: U (k_second_differences_m)
        }
    }
    template <int F> SB_DEVICE void fill(float2 (&v)[E]) const {
        const int r = 2 * rp + F;
        const bool active = r < need_rows;
        int gi = wrap(oy + need_y_lo + (active ? r : 0), ny) - row0;
        gi += gi < 0 ? ny : 0;                   // row of the slab
#pragma unroll
        for (int q = 0; q < E; ++q) {
            const int qx = t + q * T;
            const int sx = qx < split_x ? qx : qx - N;
            float2 val = make_float2(0.f, 0.f);
            if (active && sx >= need_x_lo && sx <= need_x_hi) {
                const int gj = wrap_near(ox + sx, nx);
                val = planes(sb_ldg(diffs + (long)gi * nx + gj));
            }
            // a NaN in the DEM reaches every output pixel (dem.py:105 through the reference's fft2)
            if (poison && pp == 0 && r == 0 && qx == 0) val = make_float2(NAN, NAN);
            v[q] = val;
        }
    }
    template <int P, int F> SB_DEVICE void phase(float2 (&v)[E], const float2 (&w)[TW]) {
        sbfft::stage_math<N, P, float>(v, w);
    }
    template <int P, int F> SB_DEVICE void store(const float2 (&v)[E]) {
        sbfft::stage_store<N, P, float>(v, t, F == 0 ? smA : smB);
    }
    template <int F> SB_DEVICE void load(float2 (&v)[E]) { sbfft::stage_load<N, float>(v, t, F == 0 ? smA : smB); }
};

// grid (kDiffPairs, ceil(need_rows / 2 / GP)); output layout as k_curv_rows with the plane
// pair in the place of the orientation: cr[pp][kx][rpitch rows] float4
template <int N, bool WITH_U>
SB_DEVICE void diff_rows_body(const Geom& g, const float4* SB_RESTRICT diffs, float4* SB_RESTRICT cr,
                              const float2* SB_RESTRICT tw) {
    constexpr int T = N / E;
    constexpr int GP = (T > 256 ? T : 256) / T;
    constexpr int PL = sbfft::padded_len(N);
    const int grp = sb_tid() / T, t = sb_tid() % T;
    const int KX = N / 2 + 1;
    DiffCtx<N, WITH_U> c;
    c.t = t;
    c.smA = (float2*)sb_shared() + (long)grp * 2 * PL;
    c.smB = c.smA + PL;
    c.tw = tw;
    c.diffs = diffs;
    c.pp = sb_bx();
    c.oy = g.oy; c.ox = g.ox; c.ny = g.ny; c.nx = g.nx;
    c.need_y_lo = g.need_y_lo; c.need_x_lo = g.need_x_lo; c.need_x_hi = g.need_x_hi;
    c.split_x = g.split_x; c.poison = g.poison; c.c2_scale = (float)g.c2_scale;
    c.row0 = g.row0;
    c.rp = sb_by() * GP + grp;
    c.need_rows = g.need_y_hi - g.need_y_lo + 1;
    float2 va[E], vb[E];
    c.template fill<0>(va);
    c.template fill<1>(vb);
    leapfrog<DiffCtx<N, WITH_U>::K>(c, va, vb);
    sb_sync();                                  // every thread is done with the exchange buffers
#pragma unroll
    for (int q = 0; q < E; ++q) {
        c.smA[sbfft::pad_index(t + q * T)] = va[q];
        c.smB[sbfft::pad_index(t + q * T)] = vb[q];
    }
    sb_sync();
    float4 h0[E / 2 + 1], h1[E / 2 + 1];
    split_from_shared<N>(c.smA, t, h0);
    split_from_shared<N>(c.smB, t, h1);
    if (2 * c.rp < c.need_rows)
        store_row_pair<N, float>(h0, h1, t, cr + (long)c.pp * KX * g.rpitch + 2 * c.rp, g.rpitch);
}

template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), (N / E > 256 ? 1 : 2))
k_diff_rows_f(Geom g, const float4* SB_RESTRICT diffs, float4* SB_RESTRICT cr, const float2* SB_RESTRICT tw) {
    diff_rows_body<N, false>(g, diffs, cr, tw);
}

// masked search: plane 9 = U (the .w lane of k_second_differences_m's output)
template <int N>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), (N / E > 256 ? 1 : 2))
k_diff_rows_fm(Geom g, const float4* SB_RESTRICT diffs, float4* SB_RESTRICT cr, const float2* SB_RESTRICT tw) {
    diff_rows_body<N, true>(g, diffs, cr, tw);
}

// per-orientation coefficients of the nine planes (host: float32 of the float64 cos / sin values)
struct SpecCoef { float c[kDiffPlanes + 3]; };      // padded to 48 bytes

// fct[a][field][kx][ky] = sum_p coef[a][p] * spec9[p][kx][ky] for the orientations a0 .. a0 + na - 1.
// One thread per pair of adjacent ky (float4): nine 16-byte loads, then two 16-byte stores per
// orientation.  n2 = planes' size in float4 units (KX * Py / 2).
SB_GLOBAL k_combine_spectra(long n2, int na, int a0, const SpecCoef* SB_RESTRICT coef, const float4* SB_RESTRICT spec9,
                            float4* SB_RESTRICT fct) {
    SpecCoef* sc = (SpecCoef*)sb_shared();
    for (int i = sb_tid(); i < na * (int)(sizeof(SpecCoef) / 4); i += 256) ((float*)sc)[i] = ((const float*)(coef + a0))[i];
    sb_sync();
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n2) return;
    float4 p[kDiffPlanes];
#pragma unroll
    for (int k = 0; k < kDiffPlanes; ++k) p[k] = sb_ld_stream(spec9 + (long)k * n2 + i);
    // explicit fused multiply-adds in a fixed order: an orientation's spectra must not depend on
    // its position in the batch (the sharded searches are bit-identical to the single-GPU one)
#pragma unroll 1
    for (int a = 0; a < na; ++a) {
        const SpecCoef& w = sc[a];
        float4 A, B;
        A.x = fmaf(w.c[2], p[2].x, fmaf(w.c[1], p[1].x, w.c[0] * p[0].x));
        A.y = fmaf(w.c[2], p[2].y, fmaf(w.c[1], p[1].y, w.c[0] * p[0].y));
        A.z = fmaf(w.c[2], p[2].z, fmaf(w.c[1], p[1].z, w.c[0] * p[0].z));
        A.w = fmaf(w.c[2], p[2].w, fmaf(w.c[1], p[1].w, w.c[0] * p[0].w));
        B.x = w.c[3] * p[3].x; B.y = w.c[3] * p[3].y; B.z = w.c[3] * p[3].z; B.w = w.c[3] * p[3].w;
#pragma unroll
        for (int k = 4; k < kDiffPlanes; ++k) {
            B.x = fmaf(w.c[k], p[k].x, B.x); B.y = fmaf(w.c[k], p[k].y, B.y);
            B.z = fmaf(w.c[k], p[k].z, B.z); B.w = fmaf(w.c[k], p[k].w, B.w);
        }
        sb_st_stream(fct + (long)(2 * a) * n2 + i, A);
        sb_st_stream(fct + (long)(2 * a + 1) * n2 + i, B);
    }
}

// ---------------------------------------------------------------------------
// k_poison_windows: only launched when the DEM holds a NaN (dem.py:105).  Every FFT output is
// NaN then, and compare's arithmetic select (core.py:230-240: 0 * best + 0 * NaN) leaves NaN
// wherever a template is un-masked; the pipelined fit kernels never let a NaN win, so the
// pixels inside the windows of the batch's templates are marked here.  A NaN best SNR then
// loses no later comparison (SURVEY 8a-5).
// ---------------------------------------------------------------------------
SB_GLOBAL k_poison_windows(Geom g, int count, const int* SB_RESTRICT slots, const FitT* SB_RESTRICT fit,
                           float* SB_RESTRICT best_snr) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= (long)g.out_ny * g.out_nx) return;
    const int gi = g.oy + (int)(i / g.out_nx), gj = g.ox + (int)(i % g.out_nx);
    bool hit = false;
    for (int p = 0; p < count && !hit; ++p) {
        const FitT k = fit[slots ? slots[p] : p];
        hit = gi >= k.i_lo && gi <= k.i_hi && gj >= k.j_lo && gj <= k.j_hi;
    }
    if (hit) best_snr[(long)gi * g.nx + gj] = NAN;
}

}  // namespace sb
