// CUDA kernels of the scarplet template-matching hot path (sm_100a).
//
// Schedule (per tile of the raster, FFT domain Py x Px, both powers of two):
//   k_curv_rows   per search angle: directional Laplacian (float64 stencil on the DEM,
//                 dem.py:68-107) -> pack curv + i*curv^2 -> row FFT -> Hermitian split
//   k_curv_cols   per search angle: column FFTs -> F[curv], F[curv^2] half spectra,
//                 stored column-major so the next kernel reads them coalesced
//   k_tmpl_rows   per template: evaluate the windowed template (WindowedTemplate.py:
//                 159-183, 497-520) in float64 on its support box only -> pack
//                 t + i*M -> row FFT -> Hermitian split (stored column-major)
//   k_conv_cols   per template: column FFT of the (sparse) template columns ->
//                 pointwise products with the curvature spectra (core.py:359,363) ->
//                 inverse column FFT
//   k_fit_rows    per batch of templates: inverse row FFT (fftshift folded into the
//                 index map) -> amplitude / SNR (core.py:360-367) -> masks
//                 (core.py:369-375) -> running best-SNR select (core.py:198-243) kept
//                 in registers across the batch
#pragma once
#include "sb_fft.cuh"

namespace sb {

using sbfft::E;

// ---------------------------------------------------------------------------
// parameter blocks (plain data, passed by value or read from global memory)
// ---------------------------------------------------------------------------
struct Geom {
    int ny, nx;              // raster
    int Py, Px;              // FFT domain
    int oy, ox;              // raster index of the tile's first output pixel
    int out_ny, out_nx;      // tile output extent
    int split_y, split_x;    // domain index q maps to signed offset s = q (q < split) or q - P
    int dly, dlx;            // -(n & 1): circular-shift bookkeeping of fftshift + centring
    int need_y_lo, need_y_hi;  // signed offsets of the domain rows that carry curvature
    int need_x_lo, need_x_hi;
    int kpitch;              // pitch (elements) of half-spectrum rows
    int syp;                 // pitch (rows, even) of the per-template support block
    int rpitch;              // pitch (rows, even) of the transposed curvature row spectra
    double dx, dx2, dy2;     // cell size, dx**2, dy**2 as the host computes them
    double norm;             // 1 / (Px * Py)
    double c2_scale;         // power of two: curv**2 is packed as curv**2 * c2_scale next to curv
    int poison;              // the DEM holds a NaN: every FFT domain gets one (the reference's fft2 spans the raster)
    // Row slab (spatial sharding over GPUs, SURVEY 8e): the buffers derived from the DEM hold the
    // `drows` raster rows starting at global row `row0` (periodic in ny), the best state holds
    // the rows starting at `brow0`.  A plan over the whole raster has row0 = brow0 = 0, drows = ny.
    int row0, drows, brow0;
};

// local row of the DEM-derived buffers for global raster row gi (0 <= gi < ny)
SB_DEVICE int slab_row(const Geom& g, int gi) {
    const int li = gi - g.row0;
    return li < 0 ? li + g.ny : li;
}

struct Angle {               // one search orientation (curvature direction)
    double ca, sa, ca2, sa2;  // cos, sin, cos**2, sin**2 of the search angle (host float64)
};

struct Tmpl {                // one (scale, age, angle) template
    double ca, sa;           // cos / sin of the template's alpha = -angle
    double c, d;             // half-widths of the curvature window
    double k0, k1;           // scarp: 2*kt**1.5*sqrt(pi), 4*kt   ricker: pi*f, unused
    double sign;             // -1 for the right-facing upper-break template
    double tscale;           // power of two: t is packed as t * tscale next to M (0/1)
    int kind;                // 0 scarp family, 1 ricker/channel, 2 raster (values from the caller)
    int errmode;             // 0 none, 1 snr=0 where xr<=0, 2 snr=0 where xr>=0
    int sy_lo, sy_hi, sx_lo, sx_hi;   // support box, offsets from (ny//2, nx//2)
    int i_lo, i_hi, j_lo, j_hi;       // un-masked output window (inclusive raster indices)
    int angle_id;            // index into the sweep's angle list
    int idx;                 // flat result index (tie priority and decode key)
    int state;               // best state the template folds into (one per template scale, CHANGELOG.md:20-24)
    int reserved;
};

struct TSum {                // per-template scalars produced by k_tmpl_sums
    double n_eps;            // sum(M) + eps          core.py:350
    double ts;               // sum(t**2)             core.py:356
    double inv_n;            // 1 / n_eps
    double inv_ts;
};

constexpr double kEps = 2.220446049250313e-16;   // np.spacing(1), core.py:339

// per-template scalars of the float32 epilogue of k_fit_rows_g (written by k_tmpl_sums)
// xn = norm / tscale and tn = norm / c2_scale are exact powers of two that undo the packing
// scales and the unnormalised FFTs; they are folded into the constants below (exactly), so
// the epilogue works on the raw transform outputs X = xcorr / xn, T = T3 / tn.
struct FitT {
    float amp_k;             // xn / ts                  amp = X * amp_k            core.py:360
    float a_hi, a_lo;        // xn**2 / (ts * tn) = hi + lo
    float eps_k;             // eps / tn
    float inv_n;
    int i_lo, i_hi, j_lo, j_hi;   // un-masked output window (core.py:373-375)
    int idx;                 // flat result index
    int errmode;             // get_err_mask (core.py:369-371): 0 none, 1 snr = 0 where xr <= 0, 2 where xr >= 0
    int angle_id;            // row of the k_err_cross table
};

// gbuf (the inverse-column planes handed from the column kernel to the row kernel).  With Gt,
// Gm the inverse-column transforms of ft * fc and fm2 * fc2 (core.py:359, 363), an element holds
// the two inputs the inverse ROW transform of X = Gt + i Gm needs from it, ready to use:
//     (Im X(k), Re X(k), Im X(N - k), Re X(N - k)),   X(N - k) = conj Gt(k) + i conj Gm(k)
// (real and imaginary parts swapped: the inverse runs as a forward transform) -- the column
// kernels have both fields in registers when they store, so the Hermitian extension costs the
// row kernel no arithmetic.  Per template, Py domain rows m of kpitch C4 elements, two rows interleaved:
// [m / 2][kx][m & 1].  The column kernel has rows m, m + 1 in adjacent lanes, so a warp
// store fills whole 32-byte sectors (a 16-byte half-sector store runs at 0.9 TB/s on
// B200, a full-sector one at 4.7 TB/s: scratch/ubench_scatter.cu); the row kernel reads
// its row at a 32-byte stride.
constexpr int kGbufRows = 2;      // rows interleaved per spectrum column (power of two, even)
// a, b: the two fields' inverse-column results as the transforms leave them (swapped: (im, re))
template <typename C2, typename C4>
SB_DEVICE C4 gbuf_pack(const C2 a, const C2 b) {
    C4 r;
    r.x = a.x + b.y;      // Im X(k)     = Im Gt + Re Gm
    r.y = a.y - b.x;      // Re X(k)     = Re Gt - Im Gm
    r.z = b.y - a.x;      // Im X(N - k) = Re Gm - Im Gt
    r.w = a.y + b.x;      // Re X(N - k) = Re Gt + Im Gm
    return r;
}

#ifdef SB_F32X2
// the same in two packed adds: (a.x, a.y) + (b.y, -b.x) and (b.y, b.x) + (-a.x, a.y)
template <>
SB_DEVICE float4 gbuf_pack<float2, float4>(const float2 a, const float2 b) {
    const float2 d = sbfft::unpk(sbfft::add2(sbfft::pk(a), sbfft::pk(b.y, -b.x)));
    const float2 m = sbfft::unpk(sbfft::add2(sbfft::pk(b.y, b.x), sbfft::pk(-a.x, a.y)));
    return make_float4(d.x, d.y, m.x, m.y);
}
#endif

SB_DEVICE long gbuf_index(int m, int kx, int kpitch) {
    return ((long)(m / kGbufRows) * kpitch + kx) * kGbufRows + (m % kGbufRows);
}

// periodic index for v in [-2n, 3n): the halo of a tile never reaches further (the support box
// lies inside the raster); four predicated adds instead of an integer division per pixel
SB_DEVICE int wrap_near(int v, int n) {
    v += v < 0 ? n : 0;
    v += v < 0 ? n : 0;
    v -= v >= n ? n : 0;
    v -= v >= n ? n : 0;
    return v;
}

SB_DEVICE int wrap(int v, int n) {
    int r = v % n;
    return r < 0 ? r + n : r;
}

// ---------------------------------------------------------------------------
// directional Laplacian at one raster pixel (dem.py:68-107), float64, no FMA
// ---------------------------------------------------------------------------
SB_DEVICE double zfill(const double* SB_RESTRICT z, long i) {
    double v = sb_ldg(z + i);
    return v != v ? 0.0 : v;            // dem.py:85-86
}

// the three angle-independent second differences (dem.py:88-99); NaN centre -> NaN dxx
struct Diff3 { double dxx, dxy, dyy; };

// gi: raster row (decides the boundary rows of dem.py:90-99); li: the same row's index in `z`,
// which holds `drows` rows (the whole raster, or a row slab with its halo)
SB_DEVICE Diff3 second_differences_at(const double* SB_RESTRICT z, int ny, int nx, int gi, int li, int drows,
                                      int j, double dx, double dx2, double dy2) {
    const long o = (long)li * nx + j;
    const double zc = sb_ldg(z + o);
    Diff3 r;
    r.dxx = 0.0; r.dyy = 0.0; r.dxy = 0.0;
    if (zc != zc) { r.dxx = zc; return r; }         // dem.py:105
    const bool jm = j >= 1, jp = j <= nx - 2;
    const bool im = gi >= 1 && li >= 1, ip = gi <= ny - 2 && li <= drows - 2;
    double zl = 0.0, zu = 0.0;
    if (jm) zl = zfill(z, o - 1);
    if (im) zu = zfill(z, o - nx);
    if (jm && jp) {
        const double zr = zfill(z, o + 1);
        r.dxx = sb_div(sb_sub(sb_sub(zr, zc), sb_sub(zc, zl)), dx2);       // dem.py:95
    }
    if (im && ip) {
        const double zd = zfill(z, o + nx);
        r.dyy = sb_div(sb_sub(sb_sub(zd, zc), sb_sub(zc, zu)), dy2);       // dem.py:99
    }
    if (im && jm) {
        const double zul = zfill(z, o - nx - 1);
        const double g1 = sb_div(sb_sub(zc, zl), dx);                    // dem.py:88
        const double g0 = sb_div(sb_sub(zu, zul), dx);
        r.dxy = sb_div(sb_sub(g1, g0), dx);                              // dem.py:89
    }
    return r;
}

// dem.py:103-104, left to right; a NaN dxx (NaN DEM cell) propagates
SB_DEVICE double combine_curvature(double dxx, double dxy, double dyy, const Angle& a) {
    const double t0 = sb_mul(dxx, a.ca2);
    const double t1 = sb_mul(sb_mul(sb_mul(2.0, dxy), a.sa), a.ca);
    const double t2 = sb_mul(dyy, a.sa2);
    return sb_add(sb_sub(t0, t1), t2);
}

SB_DEVICE double curvature_at(const double* SB_RESTRICT z, int ny, int nx, int gi, int li, int drows, int j,
                              double dx, double dx2, double dy2, const Angle& a) {
    const Diff3 d = second_differences_at(z, ny, nx, gi, li, drows, j, dx, dx2, dy2);
    if (d.dxx != d.dxx) return d.dxx;
    return combine_curvature(d.dxx, d.dxy, d.dyy, a);
}

// the DEM's second differences, computed once per DEM: planes [dxx][dxy][dyy] of ny*nx
// out32: the same three planes rounded to float32, interleaved [pixel][dxx, dxy, dyy, 0], for the
// complex64 pipeline (its curvature is rounded to float32 before the transform anyway)
// `dem` holds raster rows row0 .. row0 + drows - 1 (mod ny); `out` (optional: complex128 pipeline only)
SB_GLOBAL k_second_differences(int ny, int nx, int row0, int drows, const double* SB_RESTRICT dem, double dx,
                               double dx2, double dy2, double* SB_RESTRICT out, float4* SB_RESTRICT out32) {
    const long n = (long)drows * nx;
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    const int li = (int)(i / nx);
    int gi = row0 + li;
    gi -= gi >= ny ? ny : 0;
    const Diff3 d = second_differences_at(dem, ny, nx, gi, li, drows, (int)(i % nx), dx, dx2, dy2);
    if (out) {
        out[i] = d.dxx;
        out[n + i] = d.dxy;
        out[2 * n + i] = d.dyy;
    }
    if (out32) out32[i] = make_float4((float)d.dxx, (float)d.dxy, (float)d.dyy, 0.f);
}

// ---------------------------------------------------------------------------
// Nodata-masked search (sb_plan_set_nodata, SB_NODATA_MASK).  V(p) = 1 when every DEM cell the
// second differences at p depend on (dem.py:88-99, second_differences_at) is finite, U = 1 - V.
// ---------------------------------------------------------------------------
SB_DEVICE bool finite_cell(double v) { return v - v == 0.0; }     // false for NaN and +-Inf

SB_DEVICE bool stencil_finite(const double* SB_RESTRICT z, int ny, int nx, int gi, int li, int drows, int j) {
    const long o = (long)li * nx + j;
    const bool jm = j >= 1, jp = j <= nx - 2;
    const bool im = gi >= 1 && li >= 1, ip = gi <= ny - 2 && li <= drows - 2;
    bool ok = finite_cell(sb_ldg(z + o));
    if (jm && (jp || im)) ok &= finite_cell(sb_ldg(z + o - 1));       // dxx, dxy
    if (jm && jp) ok &= finite_cell(sb_ldg(z + o + 1));               // dxx
    if (im && (ip || jm)) ok &= finite_cell(sb_ldg(z + o - nx));      // dyy, dxy
    if (im && ip) ok &= finite_cell(sb_ldg(z + o + nx));              // dyy
    if (im && jm) ok &= finite_cell(sb_ldg(z + o - nx - 1));          // dxy
    return ok;
}

// k_second_differences for the masked search: out32 = (V dxx, V dxy, V dyy, U)
SB_GLOBAL k_second_differences_m(int ny, int nx, int row0, int drows, const double* SB_RESTRICT dem, double dx,
                                 double dx2, double dy2, float4* SB_RESTRICT out32) {
    const long n = (long)drows * nx;
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    const int li = (int)(i / nx), j = (int)(i % nx);
    int gi = row0 + li;
    gi -= gi >= ny ? ny : 0;
    if (!stencil_finite(dem, ny, nx, gi, li, drows, j)) {
        out32[i] = make_float4(0.f, 0.f, 0.f, 1.f);
        return;
    }
    const Diff3 d = second_differences_at(dem, ny, nx, gi, li, drows, j, dx, dx2, dy2);
    out32[i] = make_float4((float)d.dxx, (float)d.dxy, (float)d.dyy, 0.f);
}

// k_curv_sumsq for the masked search: dxx**2 + dyy**2 summed over the pixels with V = 1 only
SB_GLOBAL k_curv_sumsq_m(int ny, int nx, int row0, int drows, int own_first, int own_rows,
                         const double* SB_RESTRICT dem, double dx, double dx2, double dy2, double* SB_RESTRICT partial) {
    double* sd = (double*)sb_shared();
    const long n = (long)own_rows * nx;
    double acc = 0.0;
    for (long i = (long)sb_bx() * 256 + sb_tid(); i < n; i += (long)sb_nbx() * 256) {
        const int r = own_first + (int)(i / nx), c = (int)(i % nx);
        int gr = row0 + r;
        gr -= gr >= ny ? ny : 0;
        if (!stencil_finite(dem, ny, nx, gr, r, drows, c)) continue;
        const Diff3 d = second_differences_at(dem, ny, nx, gr, r, drows, c, dx, dx2, dy2);
        acc += d.dxx * d.dxx + d.dyy * d.dyy;
    }
    sd[sb_tid()] = acc;
    sb_sync();
    for (int w = 128; w > 0; w >>= 1) {
        if (sb_tid() < w) sd[sb_tid()] += sd[sb_tid() + w];
        sb_sync();
    }
    if (sb_tid() == 0) partial[sb_bx()] = sd[0];
}

// After a masked sweep: a pixel whose own DEM cell is not finite gets no result (initial best
// state in every state).  The plan's best rows are brow0 .. brow0 + brows - 1; state s at s * bn.
SB_GLOBAL k_best_clear_nodata(int ny, int nx, int row0, int brow0, int brows, int n_states, long bn,
                              const double* SB_RESTRICT dem, float* snr, float* amp, int* idx) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= (long)brows * nx) return;
    int li = brow0 + (int)(i / nx) - row0;
    li += li < 0 ? ny : 0;
    if (finite_cell(sb_ldg(dem + (long)li * nx + i % nx))) return;
    for (int s = 0; s < n_states; ++s) {
        snr[s * bn + i] = 0.f;
        amp[s * bn + i] = 0.f;
        idx[s * bn + i] = 0x7fffffff;
    }
}

// ---------------------------------------------------------------------------
// windowed template value at one pixel (float64)
// ---------------------------------------------------------------------------
SB_DEVICE double template_at(const Tmpl& p, double x, double y) {
    const double xr = sb_add(sb_mul(x, p.ca), sb_mul(y, p.sa));          // WindowedTemplate.py:57
    const double yr = sb_add(sb_mul(-x, p.sa), sb_mul(y, p.ca));         // :58
    const bool inside = (fabs(xr) < p.c) && (fabs(yr) < p.d);            // :63
    if (!inside) return 0.0;
    double w;
    if (p.kind == 0) {
        // (-xr / (2 kt^1.5 sqrt(pi))) * exp(-xr^2 / (4 kt))              :177-178
        w = sb_mul(sb_div(-xr, p.k0), exp(sb_div(-sb_mul(xr, xr), p.k1)));
    } else {
        // (1 - 2 u^2) * exp(-u^2), u = pi f xr                            :514-515
        // The Ricker window is as wide as the raster, so the support M = (W != 0) ends
        // where exp(-u^2) underflows to 0.0 in float64: u^2 >= 1075 ln 2 under IEEE
        // round-to-nearest (what glibc / NumPy deliver).  A device exp() may round the
        // last subnormal differently, and one pixel in n is already a 5e-4 SNR error, so
        // the boundary is decided on u^2 itself.
        const double u = sb_mul(p.k0, xr);
        const double u2 = sb_mul(u, u);
        double e = 0.0;
        if (u2 < 745.13321910194122) {
            e = exp(-u2);
            if (e == 0.0) e = 4.9406564584124654e-324;
        }
        w = sb_mul(sb_sub(1.0, sb_mul(2.0, u2)), e);
    }
    return p.sign < 0 ? -w : w;
}

// Hermitian split of the spectrum Z of a packed pair a + i*b of real rows:
// F[a](k) = (Z(k) + conj Z(-k)) / 2,  F[b](k) = (Z(k) - conj Z(-k)) / (2i).
// v holds Z[t + q*T]; writes C4 (F[a], F[b]) for k = 0..N/2 to out[k * stride].
template <int N, typename R>
SB_DEVICE void hermitian_split(const typename Vec<R>::v2 (&v)[E], int t, typename Vec<R>::v2* sm,
                               typename Vec<R>::v4* out, long stride,
                               bool active) {
    typedef typename Vec<R>::v2 C2;
    typedef typename Vec<R>::v4 C4;
    constexpr int T = N / E;
#pragma unroll
    for (int q = 0; q < E; ++q) sm[sbfft::pad_index(t + q * T)] = v[q];
    sb_sync();
#pragma unroll
    for (int q = 0; q < E / 2; ++q) {
        const int k = t + q * T;
        const C2 zp = sm[sbfft::pad_index((N - k) & (N - 1))];
        const C2 a = v[q];
        if (active)
            out[(long)k * stride] = mk4<R>((R)0.5 * (a.x + zp.x), (R)0.5 * (a.y - zp.y),
                                                (R)0.5 * (a.y + zp.y), -(R)0.5 * (a.x - zp.x));
    }
    if (t == 0 && active) {
        const C2 a = v[E / 2];                 // Nyquist, index N/2 = (E/2)*T
        out[(long)(N / 2) * stride] = mk4<R>(a.x, (R)0, a.y, (R)0);
    }
    sb_sync();
}

// The same split into registers: h[q] for k = t + q*T (q < E/2), h[E/2] for k = N/2 (thread 0).
template <int N, typename R>
SB_DEVICE void hermitian_split_regs(const typename Vec<R>::v2 (&v)[E], int t, typename Vec<R>::v2* sm,
                                    typename Vec<R>::v4 (&h)[E / 2 + 1]) {
    typedef typename Vec<R>::v2 C2;
    constexpr int T = N / E;
#pragma unroll
    for (int q = 0; q < E; ++q) sm[sbfft::pad_index(t + q * T)] = v[q];
    sb_sync();
#pragma unroll
    for (int q = 0; q < E / 2; ++q) {
        const int k = t + q * T;
        const C2 zp = sm[sbfft::pad_index((N - k) & (N - 1))];
        const C2 a = v[q];
        h[q] = mk4<R>((R)0.5 * (a.x + zp.x), (R)0.5 * (a.y - zp.y), (R)0.5 * (a.y + zp.y), -(R)0.5 * (a.x - zp.x));
    }
    h[E / 2] = mk4<R>(v[E / 2].x, (R)0, v[E / 2].y, (R)0);      // Nyquist, index N/2 = (E/2)*T
    sb_sync();
}

// Row pair (2p, 2p + 1) of a transposed plane [kx][pitch rows]: both rows' values of one kx
// leave in one store, so the column kernels read their inputs fully coalesced and the row
// kernels write whole sectors (a 16-byte strided store runs at a fifth of the rate).
template <int N, typename R>
SB_DEVICE void store_row_pair(const typename Vec<R>::v4 (&h0)[E / 2 + 1], const typename Vec<R>::v4 (&h1)[E / 2 + 1],
                              int t, typename Vec<R>::v4* out, long pitch) {
    constexpr int T = N / E;
#pragma unroll
    for (int q = 0; q < E / 2; ++q) sb_st_pair(out + (long)(t + q * T) * pitch, h0[q], h1[q]);
    if (t == 0) sb_st_pair(out + (long)(N / 2) * pitch, h0[E / 2], h1[E / 2]);
}

// ---------------------------------------------------------------------------
// k_curv_rows<Px>: grid (n_angles, ceil(need_rows / 2 / GP)), a row pair per thread group -- the angle runs fastest, so the CTAs
// that read the same rows of the second-difference planes (24 B/px, float64) are co-resident
// and all but the first of them find the rows in L2 (row-fastest order re-read the planes from
// DRAM for every angle: 32 B/px per angle measured, 8.4 after).
// ---------------------------------------------------------------------------
template <int N, typename R>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), ((N / E > 256 || sizeof(R) == 8) ? 1 : 2))
k_curv_rows(Geom g, const double* SB_RESTRICT diffs, const Angle* SB_RESTRICT angles, int angle_base,
            typename Vec<R>::v4* SB_RESTRICT cr, const typename Vec<R>::v2* SB_RESTRICT tw) {
    typedef typename Vec<R>::v2 C2;
    typedef typename Vec<R>::v4 C4;
    constexpr int T = N / E;
    const int grp = sb_tid() / T, t = sb_tid() % T;
    constexpr int GP = (T > 256 ? T : 256) / T;
    C2* sm = (C2*)sb_shared() + grp * sbfft::padded_len(N);
    const int need_rows = g.need_y_hi - g.need_y_lo + 1;
    const int rp = sb_by() * GP + grp;                 // row pair (2 rp, 2 rp + 1)
    const int a_loc = sb_bx();
    const Angle ang = angles[angle_base + a_loc];
    const int KX = N / 2 + 1;
    C4 h0[E / 2 + 1], h1[E / 2 + 1];
#pragma unroll
    for (int f = 0; f < 2; ++f) {
        const int r = 2 * rp + f;
        const bool active = r < need_rows;
        C2 v[E];
        const int gi = wrap(g.oy + g.need_y_lo + (active ? r : 0), g.ny);
#pragma unroll
        for (int q = 0; q < E; ++q) {
            const int qx = t + q * T;
            const int sx = qx < g.split_x ? qx : qx - N;
            C2 val = mk2<R>((R)0, (R)0);
            if (active && sx >= g.need_x_lo && sx <= g.need_x_hi) {
                const int gj = wrap(g.ox + sx, g.nx);
                const long o = (long)slab_row(g, gi) * g.nx + gj, n = (long)g.drows * g.nx;
                const double c = combine_curvature(sb_ldg(diffs + o), sb_ldg(diffs + n + o), sb_ldg(diffs + 2 * n + o), ang);
                val = mk2<R>((R)c, (R)(c * c * g.c2_scale));   // curv, curv**2 (core.py:355)
            }
            if (g.poison && r == 0 && qx == 0) val = mk2<R>((R)NAN, (R)NAN);
            v[q] = val;
        }
        sbfft::forward<N, R>(v, t, sm, tw);
        if (f == 0) hermitian_split_regs<N, R>(v, t, sm, h0);
        else hermitian_split_regs<N, R>(v, t, sm, h1);
    }
    // cr layout: [angle][kx][rpitch rows] C4 (F_row[curv], F_row[curv**2 * c2_scale])
    if (2 * rp < need_rows)
        store_row_pair<N, R>(h0, h1, t, cr + (long)a_loc * KX * g.rpitch + 2 * rp, g.rpitch);
}

// ---------------------------------------------------------------------------
// k_curv_cols<Py>: grid (ceil(KX / GP), n_angles).  Column FFT of both fields.
// fct layout: [angle][field][kx][Py] C2
// ---------------------------------------------------------------------------
template <int N, typename R>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), ((N / E > 256 || sizeof(R) == 8) ? 1 : 2))
k_curv_cols(Geom g, const typename Vec<R>::v4* SB_RESTRICT cr, typename Vec<R>::v2* SB_RESTRICT fct,
            const typename Vec<R>::v2* SB_RESTRICT tw) {
    typedef typename Vec<R>::v2 C2;
    typedef typename Vec<R>::v4 C4;
    constexpr int T = N / E;
    const int grp = sb_tid() / T, t = sb_tid() % T;
    constexpr int GP = (T > 256 ? T : 256) / T;
    C2* sm = (C2*)sb_shared() + grp * sbfft::padded_len(N);
    const int KX = g.Px / 2 + 1;
    const int need_rows = g.need_y_hi - g.need_y_lo + 1;
    const int kx = sb_bx() * GP + grp;
    const bool active = kx < KX;
    const int a_loc = sb_by();
    const C4* src = cr + ((long)a_loc * KX + (active ? kx : 0)) * g.rpitch;     // [angle][kx][row]: coalesced
    if constexpr (sizeof(R) == 4) {
        // both fields from one read of the plane
        C4 w[E];
#pragma unroll
        for (int q = 0; q < E; ++q) {
            const int qy = t + q * T;
            const int sy = qy < g.split_y ? qy : qy - N;
            w[q] = mk4<R>((R)0, (R)0, (R)0, (R)0);
            if (active && sy >= g.need_y_lo && sy <= g.need_y_hi) w[q] = sb_ld_stream(src + (sy - g.need_y_lo));
        }
#pragma unroll
        for (int f = 0; f < 2; ++f) {
            C2 v[E];
#pragma unroll
            for (int q = 0; q < E; ++q) v[q] = f == 0 ? mk2<R>(w[q].x, w[q].y) : mk2<R>(w[q].z, w[q].w);
            sbfft::forward<N, R>(v, t, sm, tw);
            if (active) {
                C2* dst = fct + (((long)a_loc * 2 + f) * KX + kx) * N;
#pragma unroll
                for (int q = 0; q < E; ++q) dst[t + q * T] = v[q];
            }
        }
    } else {
#pragma unroll 1
        for (int f = 0; f < 2; ++f) {
            C2 v[E];
#pragma unroll
            for (int q = 0; q < E; ++q) {
                const int qy = t + q * T;
                const int sy = qy < g.split_y ? qy : qy - N;
                C2 val = mk2<R>((R)0, (R)0);
                if (active && sy >= g.need_y_lo && sy <= g.need_y_hi) {
                    const C4 w = ld4(src + (sy - g.need_y_lo));
                    val = f == 0 ? mk2<R>(w.x, w.y) : mk2<R>(w.z, w.w);
                }
                v[q] = val;
            }
            sbfft::forward<N, R>(v, t, sm, tw);
            if (active) {
                C2* dst = fct + (((long)a_loc * 2 + f) * KX + kx) * N;
#pragma unroll
                for (int q = 0; q < E; ++q) dst[t + q * T] = v[q];
            }
        }
    }
}

// ---------------------------------------------------------------------------
// k_tmpl_rows<Px>: grid (ceil(syp / 2 / GP), n_templates), a row pair per thread group
// trt layout: [template][kx][syp] C4 (F_row[t], F_row[M]), syp even;  part: [template][syp] double2
// ---------------------------------------------------------------------------
// XSPARSE: every template of the batch is narrower than T columns either side of the centre,
// so a thread's only non-zero samples are its first and its last: two template evaluations
// per row instead of sixteen guarded ones (the unrolled float64 exp made this the largest
// kernel of the library, 70 KB of code), and a sparse first FFT stage.
// SQUARED (k_tmpl_rows_sq, the companions of a masked sweep): t**2 * tscale is packed in place of t * tscale
template <int N, typename R, bool XSPARSE, bool SQUARED>
SB_DEVICE void tmpl_rows_body(const Geom& g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, const double* SB_RESTRICT xvec,
                              const double* SB_RESTRICT yvec, typename Vec<R>::v4* SB_RESTRICT trt,
                              double2* SB_RESTRICT part, const typename Vec<R>::v2* SB_RESTRICT tw,
                              const double* SB_RESTRICT box) {
    typedef typename Vec<R>::v2 C2;
    typedef typename Vec<R>::v4 C4;
    constexpr int T = N / E;
    const int grp = sb_tid() / T, t = sb_tid() % T;
    constexpr int GP = (T > 256 ? T : 256) / T;
    C2* sm = (C2*)sb_shared() + grp * sbfft::padded_len(N);
    const int p_loc = sb_by();
    const Tmpl p = tmpls[tmpl_base + p_loc];
    const int rows = p.sy_hi - p.sy_lo + 1;
    const int rp = sb_bx() * GP + grp;                 // row pair (2 rp, 2 rp + 1) of the support box
    const int KX = N / 2 + 1;
    const int a0 = g.ny / 2, b0 = g.nx / 2;
    C4 h0[E / 2 + 1], h1[E / 2 + 1];
#pragma unroll
    for (int f = 0; f < 2; ++f) {
        const int r = 2 * rp + f;
        const bool active = r < rows;
        C2 v[E];
        double cnt = 0.0, ssq = 0.0;
        const double y = active ? sb_ldg(yvec + a0 + p.sy_lo + r) : 0.0;
#pragma unroll
        for (int q = 0; q < E; ++q) {
            const int qx = t + q * T;
            const int b = qx < N / 2 ? qx : qx - N;
            C2 val = mk2<R>((R)0, (R)0);
            if (XSPARSE && q != 0 && q != E - 1) { v[q] = val; continue; }
            if (active && b >= p.sx_lo && b <= p.sx_hi) {
                // kind 2: the plugin's own template() values on the support box (core.py:346)
                const double w = p.kind == 2 ? sb_ldg(box + (long)r * (p.sx_hi - p.sx_lo + 1) + (b - p.sx_lo))
                                             : template_at(p, sb_ldg(xvec + b0 + b), y);
                if (w != 0.0) {                                   // M = template != 0, core.py:348
                    cnt += 1.0;
                    ssq += w * w;
                    val = mk2<R>((R)((SQUARED ? w * w : w) * p.tscale), (R)1);
                }
            }
            v[q] = val;
        }
        // deterministic per-row sums of M and t^2 (two-level, fixed order)
        {
            double2* sd = (double2*)sm;
            sd[t] = make_double2(cnt, ssq);
            sb_sync();
            if ((t & 15) == 0) {
                double a = 0.0, b = 0.0;
                for (int i = 0; i < 16 && t + i < T; ++i) { a += sd[t + i].x; b += sd[t + i].y; }
                sd[t] = make_double2(a, b);
            }
            sb_sync();
            if (t == 0) {
                double a = 0.0, b = 0.0;
                for (int i = 0; i < T; i += 16) { a += sd[i].x; b += sd[i].y; }
                if (active) part[(long)p_loc * g.syp + r] = make_double2(a, b);
            }
            sb_sync();
        }
        if constexpr (XSPARSE) sbfft::forward_sparse2<N, R>(v, t, sm, tw);
        else sbfft::forward<N, R>(v, t, sm, tw);
        if (f == 0) hermitian_split_regs<N, R>(v, t, sm, h0);
        else hermitian_split_regs<N, R>(v, t, sm, h1);
    }
    if (2 * rp < rows)
        store_row_pair<N, R>(h0, h1, t, trt + (long)p_loc * KX * g.syp + 2 * rp, g.syp);
}

template <int N, typename R, bool XSPARSE>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), ((N / E > 256 || sizeof(R) == 8) ? 1 : 2))
k_tmpl_rows(Geom g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, const double* SB_RESTRICT xvec,
            const double* SB_RESTRICT yvec, typename Vec<R>::v4* SB_RESTRICT trt, double2* SB_RESTRICT part,
            const typename Vec<R>::v2* SB_RESTRICT tw, const double* SB_RESTRICT box) {
    tmpl_rows_body<N, R, XSPARSE, false>(g, tmpls, tmpl_base, xvec, yvec, trt, part, tw, box);
}

template <int N, bool XSPARSE>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), (N / E > 256 ? 1 : 2))
k_tmpl_rows_sq(Geom g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, const double* SB_RESTRICT xvec,
               const double* SB_RESTRICT yvec, float4* SB_RESTRICT trt, double2* SB_RESTRICT part,
               const float2* SB_RESTRICT tw) {
    tmpl_rows_body<N, float, XSPARSE, true>(g, tmpls, tmpl_base, xvec, yvec, trt, part, tw, nullptr);
}

// fixed-order sum of the per-row partials of each template
SB_GLOBAL k_tmpl_sums(Geom g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, int count,
                      const double2* SB_RESTRICT part, TSum* SB_RESTRICT sums, FitT* SB_RESTRICT fit) {
    // one 32-thread block per template: lane l adds rows l, l + 32, ..., lane 0 adds the 32
    // partial sums in lane order (fixed order: the result does not depend on the launch)
    const int p_loc = sb_bx();
    if (p_loc >= count) return;
    const Tmpl p = tmpls[tmpl_base + p_loc];
    const int rows = p.sy_hi - p.sy_lo + 1;
    double2* sd = (double2*)sb_shared();
    {
        double a = 0.0, b = 0.0;
        for (int r = sb_tid(); r < rows; r += 32) {
            const double2 v = part[(long)p_loc * g.syp + r];
            a += v.x;
            b += v.y;
        }
        sd[sb_tid()] = make_double2(a, b);
    }
    sb_sync();
    if (sb_tid() != 0) return;
    double n = 0.0, ts = 0.0;
    for (int l = 0; l < 32; ++l) { n += sd[l].x; ts += sd[l].y; }
    TSum s;
    s.n_eps = n + kEps;
    s.ts = ts;
    s.inv_n = 1.0 / s.n_eps;
    s.inv_ts = 1.0 / ts;
    sums[p_loc] = s;
    if (fit) {
        FitT k;
        const double xn = g.norm / p.tscale, tn = g.norm / g.c2_scale;     // powers of two
        const float its_hi = (float)s.inv_ts;
        const float its_lo = (float)(s.inv_ts - (double)its_hi);
        k.amp_k = (float)((double)its_hi * xn);
        k.a_hi = (float)((double)its_hi * (xn * xn / tn));
        k.a_lo = (float)((double)its_lo * (xn * xn / tn));
        k.eps_k = (float)(kEps / tn);
        k.inv_n = (float)s.inv_n;
        k.i_lo = p.i_lo; k.i_hi = p.i_hi; k.j_lo = p.j_lo; k.j_hi = p.j_hi;
        k.idx = p.idx;
        k.errmode = p.errmode;
        k.angle_id = p.angle_id;
        fit[p_loc] = k;
    }
}

// ---------------------------------------------------------------------------
// k_conv_cols<Py>: grid (ceil(KX / GP), n_templates)
// gbuf layout: [template][out_ny][kpitch] C4 = (inverse-column plane of t*curv,
//                                               inverse-column plane of M*curv^2)
// shared memory per group: exchange buffer (padded_len(N)) + park buffer (N): the first
// field's result waits in the park buffer (each thread re-reads only what it wrote, so no
// barrier) until the second is done, and both leave in one 16-byte store.
// ---------------------------------------------------------------------------
// complex64 below 4096 targets three resident CTAs per SM
template <int N, typename R>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), ((N / E > 256 || sizeof(R) == 8) ? 1 : 3))
k_conv_cols(Geom g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, int angle_base,
            const typename Vec<R>::v4* SB_RESTRICT trt, const typename Vec<R>::v2* SB_RESTRICT fct,
            typename Vec<R>::v4* SB_RESTRICT gbuf, const typename Vec<R>::v2* SB_RESTRICT tw) {
    typedef typename Vec<R>::v2 C2;
    typedef typename Vec<R>::v4 C4;
    constexpr int T = N / E;
    const int grp = sb_tid() / T, t = sb_tid() % T;
    constexpr int GP = (T > 256 ? T : 256) / T;
    constexpr int GSM = sbfft::padded_len(N) + N;          // elements of shared memory per group
    C2* sm = (C2*)sb_shared() + grp * GSM;
    C2* park = sm + sbfft::padded_len(N);
    const int KX = g.Px / 2 + 1;
    const int kx = sb_bx() * GP + grp;
    const bool active = kx < KX;
    const int p_loc = sb_by();
    const Tmpl p = tmpls[tmpl_base + p_loc];
    const int a_loc = p.angle_id - angle_base;
    const C4* src = trt + ((long)p_loc * KX + (active ? kx : 0)) * g.syp;
#pragma unroll 1
    for (int f = 0; f < 2; ++f) {
        C2 v[E];
#pragma unroll
        for (int q = 0; q < E; ++q) {
            const int qy = t + q * T;
            const int s = qy < N / 2 ? qy : qy - N;
            C2 val = mk2<R>((R)0, (R)0);
            if (active && s >= p.sy_lo && s <= p.sy_hi) {
                const C4 w = ld4(src + (s - p.sy_lo));
                val = f == 0 ? mk2<R>(w.x, w.y) : mk2<R>(w.z, w.w);
            }
            v[q] = val;
        }
        sbfft::forward<N, R>(v, t, sm, tw);
        {
            const C2* spec = fct + (((long)a_loc * 2 + f) * KX + (active ? kx : 0)) * N;
#pragma unroll
            for (int q = 0; q < E; ++q) {
                const C2 w = ld2(spec + t + q * T);
                const C2 pr = sbfft::cmul(v[q], w);               // core.py:359 / :363
                v[q] = mk2<R>(pr.y, pr.x);                        // swap: inverse via forward
            }
        }
        sbfft::forward<N, R>(v, t, sm, tw);
        if (f == 0) {
#pragma unroll
            for (int q = 0; q < E; ++q) park[t + q * T] = v[q];
        } else if (active) {
            C4* dst = gbuf + (long)p_loc * N * g.kpitch;
#pragma unroll
            for (int q = 0; q < E; ++q) {
                const int m = t + q * T;
                const int io = (m + g.dly) & (N - 1);
                const C2 a = park[m];
                if (io < g.out_ny) dst[gbuf_index(m, kx, g.kpitch)] = gbuf_pack<C2, C4>(a, v[q]);
            }
        }
    }
}

// ---------------------------------------------------------------------------
// k_fit_rows<Px>: grid (ceil(out_ny / GP)); loops over the batch of templates
// ---------------------------------------------------------------------------
struct FitOut {
    float* best_snr;         // [ny][nx]
    float* best_amp;
    int* best_idx;
    double* raw_amp;         // single-template mode (match_template): full planes
    double* raw_snr;
};

// error = (1/n) * (T1 - 2*amp*xcorr + T3) + eps with T1 = ts*amp^2, amp = xcorr/ts
// (core.py:360-366) is algebraically (T3 - xcorr^2/ts)/n + eps: a cancellation.  In the
// complex64 pipeline it is evaluated with error-free float32 products (two-term split of
// xcorr^2 and of 1/ts), which keeps it as accurate as a float64 evaluation of the same
// float32 inputs without touching the FP64 pipe.
struct FitScalars {
    float xn, tn;            // exact powers of two: norm / tscale, norm / c2_scale
    float its_hi, its_lo;    // 1/ts = hi + lo
    float inv_n;
};

SB_DEVICE void fit_pixel(float xraw, float traw, const FitScalars& k, float& amp, float& snr) {
    const float x = xraw * k.xn;                     // xcorr  (exact scaling)
    const float t3 = traw * k.tn;                    // T3     (exact scaling)
    amp = x * k.its_hi;                              // core.py:360
    const float pp = x * x;
    const float pe = fmaf(x, x, -pp);                // x*x = pp + pe exactly
    float num = fmaf(-pp, k.its_hi, t3);             // T3 - x^2/ts
    num = fmaf(-pp, k.its_lo, num);
    num = fmaf(-pe, k.its_hi, num);
    const float t1 = x * amp;                        // core.py:362
    const float err = fmaf(num, k.inv_n, (float)kEps);   // core.py:366
    snr = fabsf(t1 / err);                           // core.py:367
}

template <int N, typename R>
SB_GLOBAL SB_LAUNCH_BOUNDS((N / E > 256 ? N / E : 256), ((N / E > 256 || sizeof(R) == 8) ? 1 : 2))
k_fit_rows(Geom g, const Tmpl* SB_RESTRICT tmpls, int tmpl_base, int count, const int* SB_RESTRICT slots,
           const TSum* SB_RESTRICT sums, const typename Vec<R>::v4* SB_RESTRICT gbuf,
           const double* SB_RESTRICT xvec, const double* SB_RESTRICT yvec, FitOut out,
           const typename Vec<R>::v2* SB_RESTRICT tw) {
    typedef typename Vec<R>::v2 C2;
    typedef typename Vec<R>::v4 C4;
    constexpr int T = N / E;
    const int grp = sb_tid() / T, t = sb_tid() % T;
    constexpr int GP = (T > 256 ? T : 256) / T;
    C2* sm = (C2*)sb_shared() + grp * sbfft::padded_len(N);
    const int io = sb_bx() * GP + grp;
    const bool active = io < g.out_ny;
    const int gi = g.oy + io;
    const int cta_lo = g.oy + sb_bx() * GP;
    const int cta_hi = cta_lo + GP - 1;
    const bool raw = out.raw_amp != nullptr;

    float bs[E], ba[E];
    int bi[E];
    int gj[E];
#pragma unroll
    for (int q = 0; q < E; ++q) {
        const int m = t + q * T;
        const int jo = (m + g.dlx) & (N - 1);
        gj[q] = (active && jo < g.out_nx) ? g.ox + jo : -1;
        bs[q] = 0.f; ba[q] = 0.f; bi[q] = 0x7fffffff;
        if (gj[q] >= 0 && !raw) {
            const long o = (long)gi * g.nx + gj[q];
            bs[q] = out.best_snr[o];
            ba[q] = out.best_amp[o];
            bi[q] = out.best_idx[o];
        }
    }
    const double yv = active ? sb_ldg(yvec + gi) : 0.0;

#pragma unroll 1
    for (int it = 0; it < count; ++it) {
        const int pl = slots ? slots[it] : it;           // batch slot (one best state's templates)
        const Tmpl p = tmpls[tmpl_base + pl];
        if (!raw && (cta_hi < p.i_lo || cta_lo > p.i_hi)) continue;   // whole CTA edge-masked
        const TSum s = sums[pl];
        const C4* grow = gbuf + (long)pl * g.Py * g.kpitch + gbuf_index(((active ? io : 0) - g.dly) & (g.Py - 1), 0, g.kpitch);
        C2 v[E];
#pragma unroll
        for (int q = 0; q < E; ++q) {
            const int k = t + q * T;
            const bool direct = k <= N / 2;
            const int kk = direct ? k : N - k;
            C4 w = mk4<R>((R)0, (R)0, (R)0, (R)0);
            if (active) w = ld4(grow + kGbufRows * kk);
            // X(k) = Gt(k) + i Gm(k);  X(N-k) = conj Gt(k) + i conj Gm(k): both ready in the element (gbuf_pack)
            v[q] = direct ? mk2<R>(w.x, w.y) : mk2<R>(w.z, w.w);
        }
        sbfft::forward<N, R>(v, t, sm, tw);
        const bool row_ok = gi >= p.i_lo && gi <= p.i_hi;
        FitScalars fk;
        fk.xn = (float)(g.norm / p.tscale);
        fk.tn = (float)(g.norm / g.c2_scale);
        fk.its_hi = (float)s.inv_ts;
        fk.its_lo = (float)(s.inv_ts - (double)fk.its_hi);
        fk.inv_n = (float)s.inv_n;
        const double xc_norm = g.norm / p.tscale, t3_norm = g.norm / g.c2_scale;
#pragma unroll
        for (int q = 0; q < E; ++q) {
            if (gj[q] < 0) continue;
            double amp_d = 0.0, snr_d = 0.0;
            float amp_f = 0.f, snr_f = 0.f;
            if (sizeof(R) == 4 && !raw) {
                fit_pixel((float)v[q].y, (float)v[q].x, fk, amp_f, snr_f);
            } else {
                const double xc = (double)v[q].y * xc_norm;          // Re ifft: xcorr   core.py:359
                const double t3 = (double)v[q].x * t3_norm;          // Im ifft: T3      core.py:363
                amp_d = xc * s.inv_ts;                               // core.py:360
                const double t1 = s.ts * amp_d * amp_d;              // core.py:362
                const double err = s.inv_n * (t1 - 2.0 * amp_d * xc + t3) + kEps;   // core.py:366
                snr_d = fabs(t1 / err);                              // core.py:367
                amp_f = (float)amp_d;
                snr_f = (float)snr_d;
            }
            bool kill_snr = false;
            if (p.errmode != 0) {                                // core.py:369-371
                const double xr = sb_add(sb_mul(sb_ldg(xvec + gj[q]), p.ca), sb_mul(yv, p.sa));
                kill_snr = (p.errmode == 1 && xr <= 0.0) || (p.errmode == 2 && xr >= 0.0);
            }
            const bool masked = !row_ok || gj[q] < p.j_lo || gj[q] > p.j_hi;   // core.py:373-375
            if (kill_snr || masked) { snr_f = 0.f; snr_d = 0.0; }
            if (masked) { amp_f = 0.f; amp_d = 0.0; }
            if (raw) {
                const long o = (long)gi * g.nx + gj[q];
                out.raw_amp[o] = amp_d;
                out.raw_snr[o] = snr_d;
            } else {
                // first maximum wins (core.py:230-240); equal positive SNRs resolve to the
                // lower flat index so the result does not depend on batch order
                // a NaN SNR (NaN in the DEM) sticks: 0 * best + 0 * NaN (core.py:230-240)
                if (snr_f != snr_f) {
                    bs[q] = snr_f;
                } else if (snr_f > bs[q] || (snr_f == bs[q] && snr_f > 0.f && p.idx < bi[q])) {
                    bs[q] = snr_f;
                    ba[q] = amp_f;
                    bi[q] = p.idx;
                }
            }
        }
    }
    if (!raw) {
#pragma unroll
        for (int q = 0; q < E; ++q) {
            if (gj[q] < 0) continue;
            const long o = (long)gi * g.nx + gj[q];
            out.best_snr[o] = bs[q];
            out.best_amp[o] = ba[q];
            out.best_idx[o] = bi[q];
        }
    }
}

// ---------------------------------------------------------------------------
// elementwise kernels
// ---------------------------------------------------------------------------
SB_GLOBAL k_best_init(long n, float* snr, float* amp, int* idx) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i < n) { snr[i] = 0.f; amp[i] = 0.f; idx[i] = 0x7fffffff; }
}

// Cross-GPU merge of best states (replaces the parent-side compare over Pool results,
// core.py:185): key = SNR bits (SNR >= 0, so IEEE order == integer order) in the high
// word, inverted flat index in the low word -> integer max picks the highest SNR and,
// on equal SNR, the lowest index.
SB_GLOBAL k_best_pack(long n, const float* SB_RESTRICT snr, const int* SB_RESTRICT idx,
                      unsigned long long* SB_RESTRICT keys) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    unsigned int bits;
    const float s = snr[i];
    memcpy(&bits, &s, 4);
    if (s != s) bits = 0x7FC00000u;        // canonical positive NaN: above every finite SNR as a signed key
    keys[i] = ((unsigned long long)bits << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned int)idx[i]);
}

SB_GLOBAL k_best_select(long n, const float* SB_RESTRICT snr, const float* SB_RESTRICT amp,
                        const int* SB_RESTRICT idx, const unsigned long long* SB_RESTRICT gkeys,
                        float* SB_RESTRICT amp_out) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    unsigned int bits;
    const float s = snr[i];
    memcpy(&bits, &s, 4);
    if (s != s) bits = 0x7FC00000u;
    const unsigned long long own =
        ((unsigned long long)bits << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned int)idx[i]);
    amp_out[i] = (own == gkeys[i] && idx[i] != 0x7fffffff) ? amp[i] : 0.f;
}

SB_GLOBAL k_best_unpack(long n, const unsigned long long* SB_RESTRICT gkeys,
                        const float* SB_RESTRICT amp_in, float* SB_RESTRICT snr, float* SB_RESTRICT amp,
                        int* SB_RESTRICT idx) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    const unsigned long long k = gkeys[i];
    const unsigned int bits = (unsigned int)(k >> 32);
    float s;
    memcpy(&s, &bits, 4);
    snr[i] = s;
    idx[i] = (int)(0xFFFFFFFFu - (unsigned int)(k & 0xFFFFFFFFull));
    amp[i] = amp_in[i];
}

// get_err_mask of the upper-break templates (WindowedTemplate.py:257-267, 294-304): xr <= 0 or
// xr >= 0 with xr = x * cos(alpha) + y * sin(alpha) in float64 (WindowedTemplate.py:57).  Along a
// raster row xr is monotonic in the column (IEEE multiplication and addition are monotonic), so
// the masks are column ranges: per (search angle, raster row) this kernel finds, by bisection
// on the exact float64 expression, the inclusive ranges with xr > 0 (.x .. .y) and xr < 0
// (.z .. .w); empty ranges have lo > hi.  ca / sa: cos / sin of the template's alpha = -angle.
SB_GLOBAL k_err_cross(int ny, int nx, int n_angles, const double* SB_RESTRICT ca_sa, const double* SB_RESTRICT xvec,
                      const double* SB_RESTRICT yvec, int4* SB_RESTRICT cross) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= (long)n_angles * ny) return;
    const int a = (int)(i / ny), row = (int)(i % ny);
    const double ca = ca_sa[2 * a], sa = ca_sa[2 * a + 1];
    const double ys = sb_mul(sb_ldg(yvec + row), sa);
    const bool rising = ca >= 0.0;             // xr does not decrease with the column
    // first column (in the direction of rising xr) with xr >= 0, and with xr > 0
    int lo = 0, hi = nx;                       // count of columns with xr < 0
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int j = rising ? mid : nx - 1 - mid;
        const double xr = sb_add(sb_mul(sb_ldg(xvec + j), ca), ys);
        if (xr < 0.0) lo = mid + 1; else hi = mid;
    }
    const int n_neg = lo;
    lo = n_neg; hi = nx;                       // count of columns with xr <= 0
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int j = rising ? mid : nx - 1 - mid;
        const double xr = sb_add(sb_mul(sb_ldg(xvec + j), ca), ys);
        if (xr <= 0.0) lo = mid + 1; else hi = mid;
    }
    const int n_le = lo;
    int4 r;
    if (rising) { r.x = n_le; r.y = nx - 1; r.z = 0; r.w = n_neg - 1; }
    else { r.x = 0; r.y = nx - 1 - n_le; r.z = nx - n_neg; r.w = nx - 1; }
    cross[i] = r;
}

// Fold `n_cands` candidate best states (e.g. one per rank of an orientation-sharded search)
// for the same `n` pixels into one: highest SNR wins, equal SNRs go to the lower flat index
// (the priority of core.compare's first maximum, core.py:230-240), a NaN SNR sticks
// (0 * best + 0 * NaN).  Candidate c of pixel i is at [c * n + i].
SB_GLOBAL k_best_merge(long n, int n_cands, const float* SB_RESTRICT snr_c, const float* SB_RESTRICT amp_c,
                       const int* SB_RESTRICT idx_c, float* SB_RESTRICT snr, float* SB_RESTRICT amp,
                       int* SB_RESTRICT idx) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    float bs = snr_c[i], ba = amp_c[i];
    int bi = idx_c[i];
    for (int c = 1; c < n_cands; ++c) {
        const float s = snr_c[(long)c * n + i];
        const int k = idx_c[(long)c * n + i];
        if (bs != bs) break;
        if (s != s || s > bs || (s == bs && k < bi)) { bs = s; ba = amp_c[(long)c * n + i]; bi = k; }
    }
    snr[i] = bs; amp[i] = ba; idx[i] = bi;
}

// Fold `n_cands` candidate region planes (e.g. one per rank of an orientation-sharded fit region)
// for the same `n` pixels into the plan's: plane 0 (count) is summed, plane 1 (rank_lo) the minimum,
// plane 2 (rank_hi) the maximum, planes 3 .. n_planes - 1 (orientation words) OR-ed.  Candidate c of
// plane p, pixel i is at [(p * n_cands + c) * n + i]; plane p of the output at [p * plane + i].  The
// output is replaced, not folded into: the candidates include this rank's own planes.  The cleared
// planes of sb_region_sweep (0, 0x7f7f7f7f, -1, no bits) are identities of the four folds.  One
// thread per (plane, pixel).
SB_GLOBAL k_region_merge(long n, int n_planes, int n_cands, long plane, const int* SB_RESTRICT cands,
                         int* SB_RESTRICT planes) {
    const long t = (long)sb_bx() * 256 + sb_tid();
    if (t >= n * n_planes) return;
    const int p = (int)(t / n);
    const long i = t - (long)p * n;
    const int* c = cands + (long)p * n_cands * n + i;
    int v = c[0];
    for (int k = 1; k < n_cands; ++k) {
        const int w = c[(long)k * n];
        v = p == 0 ? v + w : p == 1 ? (w < v ? w : v) : p == 2 ? (w > v ? w : v) : (v | w);
    }
    planes[(long)p * plane + i] = v;
}

// Fold `n_extra` further copies of a best state (copy c of pixel i at [c * stride + i]) into the
// main one in place, with k_best_merge's rule.
SB_GLOBAL k_best_fold(long n, int n_extra, long stride, const float* SB_RESTRICT snr_x, const float* SB_RESTRICT amp_x,
                      const int* SB_RESTRICT idx_x, float* SB_RESTRICT snr, float* SB_RESTRICT amp, int* SB_RESTRICT idx) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    float bs = snr[i], ba = amp[i];
    int bi = idx[i];
    bool changed = false;
    for (int c = 0; c < n_extra; ++c) {
        if (bs != bs) break;
        const float s = snr_x[(long)c * stride + i];
        const int k = idx_x[(long)c * stride + i];
        if (s != s || s > bs || (s == bs && k < bi)) { bs = s; ba = amp_x[(long)c * stride + i]; bi = k; changed = true; }
    }
    if (changed) { snr[i] = bs; amp[i] = ba; idx[i] = bi; }
}

// One pixel of a best state (SNR s, flat index k, amplitude *amp -- read only for a hit) as the
// reference's [amp, age, angle, snr] float64 values (core.py:190-193)
SB_DEVICE void decode_best(float s, int k, const float* SB_RESTRICT amp, const double* SB_RESTRICT age_of,
                           const double* SB_RESTRICT angle_of, int n_idx, double (&o)[4]) {
    const bool hit = s > 0.f && k >= 0 && k < n_idx;
    // NaN in the DEM (dem.py:105): compare's select leaves NaN in amp and snr and 0 in age and
    // angle wherever some template was un-masked (SURVEY 8a-5)
    const bool nan = s != s;
    const double qnan = (double)s;
    o[0] = nan ? qnan : hit ? (double)*amp : 0.0;
    o[1] = hit ? age_of[k] : 0.0;
    o[2] = hit ? angle_of[k] : 0.0;
    o[3] = nan ? qnan : hit ? (double)s : 0.0;
}

// decode the best state into the reference's [amp, age, angle, snr] float64 planes
SB_GLOBAL k_finalize(long n, const float* SB_RESTRICT snr, const float* SB_RESTRICT amp,
                     const int* SB_RESTRICT idx, const double* SB_RESTRICT age_of,
                     const double* SB_RESTRICT angle_of, int n_idx, double* SB_RESTRICT out4) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    double o[4];
    decode_best(snr[i], idx[i], amp + i, age_of, angle_of, n_idx, o);
    out4[i] = o[0];
    out4[n + i] = o[1];
    out4[2 * n + i] = o[2];
    out4[3 * n + i] = o[3];
}

// Age-resolved search (sb_age_range): best state s (pixel i at [s * stride + i]) holds the best fit
// over the orientations at age s.  Folds the n_states states with k_best_merge's rule -- the fold
// the single-state sweep runs in the fit kernel, so planes 0..3 are what k_finalize gives for it --
// and writes [amp, age, angle, snr, age_lo, age_hi]: age_lo / age_hi are the smallest / largest
// decoded age over the states with snr_s > 0 and (double)snr_s >= ratio * (double)snr_best, 0 where
// the fold has no hit (SNR 0 or NaN).  SNRs are read per state (coalesced); idx only to break an SNR tie and
// for the states that count, amp only for the winner.
SB_GLOBAL k_age_range(long n, long stride, int n_states, const float* SB_RESTRICT snr, const float* SB_RESTRICT amp,
                      const int* SB_RESTRICT idx, const double* SB_RESTRICT age_of,
                      const double* SB_RESTRICT angle_of, int n_idx, double ratio, double* SB_RESTRICT out6) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    float bs = snr[i];
    int bst = 0, bi = 0;
    bool have_bi = false;                       // bi = idx of state bst (read on the first tie)
    for (int s = 1; s < n_states; ++s) {
        if (bs != bs) break;
        const float v = snr[(long)s * stride + i];
        bool take = v != v || v > bs;
        if (!take && v == bs) {
            if (!have_bi) { bi = idx[(long)bst * stride + i]; have_bi = true; }
            const int k = idx[(long)s * stride + i];
            take = k < bi;
            if (take) bi = k;
        } else if (take) {
            have_bi = false;
        }
        if (take) { bs = v; bst = s; }
    }
    const long b = (long)bst * stride + i;
    const int kb = bs > 0.f ? (have_bi ? bi : idx[b]) : -1;
    double o[4];
    decode_best(bs, kb, amp + b, age_of, angle_of, n_idx, o);
    double lo = 0.0, hi = 0.0;
    if (bs > 0.f && kb >= 0 && kb < n_idx) {
        const double floor = ratio * (double)bs;
        lo = o[1]; hi = o[1];
        for (int s = 0; s < n_states; ++s) {
            const float v = snr[(long)s * stride + i];
            if (!(v > 0.f && (double)v >= floor)) continue;
            const int k = idx[(long)s * stride + i];
            if (k < 0 || k >= n_idx) continue;
            const double a = age_of[k];
            lo = a < lo ? a : lo;
            hi = a > hi ? a : hi;
        }
    }
    out6[i] = o[0];
    out6[n + i] = o[1];
    out6[2 * n + i] = o[2];
    out6[3 * n + i] = o[3];
    out6[4 * n + i] = lo;
    out6[5 * n + i] = hi;
}

SB_DEVICE int sb_lowest_bit(unsigned m) {
#ifdef SB_EMU
    return __builtin_ctz(m);
#else
    return __ffs(m) - 1;
#endif
}

// Fit confidence region (sb_region_finalize) over the planes the threshold pass wrote (RegionOut,
// sb_fast.cuh; plane stride `plane`, `words` orientation words): [amp, age, angle, snr] of best
// state 0 as k_finalize decodes it, then age_lo / age_hi = rank_age[rank_lo / rank_hi], angle_lo /
// angle_hi = the shortest arc of positions holding every qualifying one, and the count.  Linear
// search: [pos_angle[first], pos_angle[last]].  Periodic: the arc is the complement of the largest
// circular gap between consecutive qualifying positions (equal gaps: the lowest p_lo), and
// angle_hi = pos_angle[p_hi] + pi when it wraps (p_hi < p_lo).  Planes 4..8 are 0 where the pixel
// has no fit (best SNR 0 or NaN).
SB_GLOBAL k_region_finalize(long n, long plane, int words, const float* SB_RESTRICT snr,
                            const float* SB_RESTRICT amp, const int* SB_RESTRICT idx, const int* SB_RESTRICT count,
                            const int* SB_RESTRICT rank_lo, const int* SB_RESTRICT rank_hi,
                            const unsigned* SB_RESTRICT bits, const double* SB_RESTRICT age_of,
                            const double* SB_RESTRICT angle_of, int n_idx, const double* SB_RESTRICT rank_age,
                            const double* SB_RESTRICT pos_angle, int n_pos, int periodic, double* SB_RESTRICT out9) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    const float s = snr[i];
    double o[4];
    decode_best(s, idx[i], amp + i, age_of, angle_of, n_idx, o);
    const int c = count[i];
    double age_lo = 0.0, age_hi = 0.0, ang_lo = 0.0, ang_hi = 0.0;
    if (s > 0.f && c > 0) {
        age_lo = rank_age[rank_lo[i]];
        age_hi = rank_age[rank_hi[i]];
        // qualifying positions in increasing order; the largest gap between two consecutive ones
        int first = -1, prev = -1, gap = 0, gap_lo = 0, gap_hi = 0;
        for (int w = 0; w < words; ++w) {
            unsigned m = bits[(long)w * plane + i];
            while (m != 0u) {
                const int p = 32 * w + sb_lowest_bit(m);
                m &= m - 1u;
                if (first < 0) first = p;
                else if (p - prev > gap) { gap = p - prev; gap_lo = p; gap_hi = prev; }
                prev = p;
            }
        }
        int p_lo = first, p_hi = prev;
        // periodic: the gap across the wrap has the lowest p_lo (first), so it wins a tie
        if (periodic && first + n_pos - prev < gap) { p_lo = gap_lo; p_hi = gap_hi; }
        if (first >= 0) {
            ang_lo = pos_angle[p_lo];
            ang_hi = p_hi < p_lo ? pos_angle[p_hi] + 3.141592653589793 : pos_angle[p_hi];
        }
    }
    out9[i] = o[0];
    out9[n + i] = o[1];
    out9[2 * n + i] = o[2];
    out9[3 * n + i] = o[3];
    out9[4 * n + i] = age_lo;
    out9[5 * n + i] = age_hi;
    out9[6 * n + i] = ang_lo;
    out9[7 * n + i] = ang_hi;
    out9[8 * n + i] = (s > 0.f) ? (double)c : 0.0;
}

// sum over the raster of dxx**2 + dyy**2 (per-block partials, fixed order): gives the
// curvature scale used to balance curv against curv**2 in the packed FFT
// `dem` holds raster rows row0 .. (slab); the sum runs over its rows own_first .. own_first + own_rows - 1
SB_GLOBAL k_curv_sumsq(int ny, int nx, int row0, int drows, int own_first, int own_rows,
                       const double* SB_RESTRICT dem, double dx, double dx2, double dy2, double* SB_RESTRICT partial) {
    double* sd = (double*)sb_shared();
    const long n = (long)own_rows * nx;
    Angle a0, a1;
    a0.ca = 1.0; a0.sa = 0.0; a0.ca2 = 1.0; a0.sa2 = 0.0;
    a1.ca = 0.0; a1.sa = 1.0; a1.ca2 = 0.0; a1.sa2 = 1.0;
    double acc = 0.0;
    for (long i = (long)sb_bx() * 256 + sb_tid(); i < n; i += (long)sb_nbx() * 256) {
        const int r = own_first + (int)(i / nx), c = (int)(i % nx);
        int gr = row0 + r;
        gr -= gr >= ny ? ny : 0;
        const double u = curvature_at(dem, ny, nx, gr, r, drows, c, dx, dx2, dy2, a0);
        const double v = curvature_at(dem, ny, nx, gr, r, drows, c, dx, dx2, dy2, a1);
        acc += u * u + v * v;
    }
    sd[sb_tid()] = acc;
    sb_sync();
    for (int w = 128; w > 0; w >>= 1) {
        if (sb_tid() < w) sd[sb_tid()] += sd[sb_tid() + w];
        sb_sync();
    }
    if (sb_tid() == 0) partial[sb_bx()] = sd[0];
}

// full-raster directional Laplacian in float64 (DEMGrid._calculate_directional_laplacian)
SB_GLOBAL k_laplacian(int ny, int nx, const double* SB_RESTRICT dem, double dx, double dx2,
                      double dy2, Angle a, double* SB_RESTRICT out) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= (long)ny * nx) return;
    const int r = (int)(i / nx);
    out[i] = curvature_at(dem, ny, nx, r, r, ny, (int)(i % nx), dx, dx2, dy2, a);
}

// full-raster template in float64 (WindowedTemplate.template())
SB_GLOBAL k_render_template(int ny, int nx, Tmpl p, const double* SB_RESTRICT xvec,
                            const double* SB_RESTRICT yvec, double* SB_RESTRICT out) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= (long)ny * nx) return;
    const int a = (int)(i / nx) - ny / 2, b = (int)(i % nx) - nx / 2;
    double w = 0.0;
    if (a >= p.sy_lo && a <= p.sy_hi && b >= p.sx_lo && b <= p.sx_hi)
        w = template_at(p, xvec[b + nx / 2], yvec[a + ny / 2]);
    out[i] = w;
}

// ---------------------------------------------------------------------------
// Fit surfaces at chosen pixels (sb_fit_surface, DESIGN.md section 12): the post-mask amp / snr of
// core.py:359-375 of every template at every pixel, by direct float64 sums over the template's
// support box instead of FFTs:
//     xcorr(i, j) = sum_{u,v} t[a0 + u, b0 + v] * curv[(i - u + ny % 2) mod ny, (j - v + nx % 2) mod nx]
//     T3(i, j)    = the same sum of M * curv**2
// A job is up to kFsAges templates of ONE search angle (the ages of an orientation); grid
// (jobs, groups of kFsPix pixels), warp w = template w of the job, lane l = pixel l of the group.
// The union of the job's support boxes is walked in row-major tiles of kFsTile cells: the
// curvature of the group's pixels over a tile is staged in shared memory once for all the
// job's templates, the values of a template once for all pixels.  Each (pixel, template) pair
// is summed by ONE thread, sequentially, in row-major order over the template's own box (cells
// outside it have t = 0 and are skipped), so its bits do not depend on the other pixels or
// templates of the call, on their order or on the batching.  n = sum(M) and ts = sum(t**2) are
// summed the same way by every lane.
// MASKED (SB_NODATA_MASK): the sums run over the cells with V = 1 only (selected, never
// multiplied: the float64 curvature is not finite there); n_valid and ts_m are summed alongside.
// ---------------------------------------------------------------------------
constexpr int kFsAges = 8;                // templates per job = warps per CTA
constexpr int kFsPix = 32;                // pixels per CTA = lanes
constexpr int kFsTile = 128;              // support cells per shared-memory tile
constexpr int kFsPitch = kFsPix + 1;      // curvature tile row pitch (doubles): conflict-free both ways
constexpr size_t kFsSmem = (size_t)(kFsTile * kFsPitch + kFsAges * kFsTile) * sizeof(double);

struct FsJob {
    int first, count;             // templates order[first .. first + count - 1], all of one angle
    int uy_lo, ux_lo, uw, cells;  // union of their support boxes: top-left offset, width, cells
};

template <bool MASKED>
SB_GLOBAL SB_LAUNCH_BOUNDS(kFsAges * kFsPix, 1)
k_fit_surface(int ny, int nx, int row0, int drows, const double* SB_RESTRICT diffs, const double* SB_RESTRICT dem,
              const Angle* SB_RESTRICT angles, const Tmpl* SB_RESTRICT tmpls, const int* SB_RESTRICT order,
              const FsJob* SB_RESTRICT jobs, int n_tmpls, const int* SB_RESTRICT rows, const int* SB_RESTRICT cols, int n_pix,
              const double* SB_RESTRICT xvec, const double* SB_RESTRICT yvec, int poison, double min_coverage,
              double* SB_RESTRICT amp, double* SB_RESTRICT snr) {
    double* cv = (double*)sb_shared();                 // [cell][kFsPitch]: curvature of the group's pixels
    double* tv = cv + kFsTile * kFsPitch;              // [template][cell]: template values
    const FsJob job = jobs[sb_bx()];
    const int w = sb_tid() / kFsPix, lane = sb_tid() % kFsPix;
    const int p0 = sb_by() * kFsPix;
    const bool has_t = w < job.count;
    const int k = has_t ? order[job.first + w] : order[job.first];
    const Tmpl p = tmpls[k];
    const Angle ang = angles[p.angle_id];
    const long plane = (long)drows * nx;
    const int a0 = ny / 2, b0 = nx / 2, oy = ny & 1, ox = nx & 1;

    double xc = 0.0, t3 = 0.0, ts = 0.0, tsm = 0.0;
    int n = 0, nv = 0;
#pragma unroll 1
    for (int f0 = 0; f0 < job.cells; f0 += kFsTile) {
        // curvature at (pixel - offset) for every cell of the tile: consecutive threads take
        // consecutive cells of one pixel (adjacent DEM columns)
#pragma unroll 1
        for (int e = sb_tid(); e < kFsTile * kFsPix; e += kFsAges * kFsPix) {
            const int c = e % kFsTile, q = e / kFsTile, f = f0 + c;
            double val = 0.0;
            if (f < job.cells && p0 + q < n_pix) {
                const int gi = wrap_near(rows[p0 + q] - (job.uy_lo + f / job.uw) + oy, ny);
                const int gj = wrap_near(cols[p0 + q] - (job.ux_lo + f % job.uw) + ox, nx);
                const int li = gi - row0 < 0 ? gi - row0 + ny : gi - row0;
                const long o = (long)li * nx + gj;
                val = combine_curvature(sb_ldg(diffs + o), sb_ldg(diffs + plane + o), sb_ldg(diffs + 2 * plane + o), ang);
                if (MASKED && !stencil_finite(dem, ny, nx, gi, li, drows, gj)) val = NAN;   // V = 0
            }
            cv[c * kFsPitch + q] = val;
        }
        // rows of the tile; a template whose box misses them has nothing here
        const int r_lo = job.uy_lo + f0 / job.uw;
        const int f1 = f0 + kFsTile < job.cells ? f0 + kFsTile : job.cells;       // tile end
        const int r_hi = job.uy_lo + (f1 - 1) / job.uw;
        const bool live = has_t && r_hi >= p.sy_lo && r_lo <= p.sy_hi;
        if (live) {
            for (int c = lane; c < kFsTile; c += kFsPix) {
                const int f = f0 + c;
                const int u = job.uy_lo + f / job.uw, v = job.ux_lo + f % job.uw;
                double t = 0.0;
                if (f < job.cells && u >= p.sy_lo && u <= p.sy_hi && v >= p.sx_lo && v <= p.sx_hi)
                    t = template_at(p, sb_ldg(xvec + b0 + v), sb_ldg(yvec + a0 + u));
                tv[w * kFsTile + c] = t;
            }
        }
        sb_sync();
        if (live) {
#pragma unroll 4
            for (int c = 0; c < f1 - f0; ++c) {
                const double t = tv[w * kFsTile + c];
                if (t == 0.0) continue;                               // M = t != 0 (core.py:348)
                const double cc = cv[c * kFsPitch + lane];
                n += 1;
                ts = fma(t, t, ts);
                if (MASKED && cc != cc) continue;                     // V = 0: not part of the fit
                xc = fma(t, cc, xc);                                  // core.py:359
                t3 = t3 + sb_mul(cc, cc);                             // core.py:355, 363
                if (MASKED) {
                    nv += 1;
                    tsm = fma(t, t, tsm);
                }
            }
        }
        sb_sync();
    }
    const int px = p0 + lane;
    if (!has_t || px >= n_pix) return;
    const int i = rows[px], j = cols[px];
    double nn = sb_add((double)n, kEps), tss = ts;                  // core.py:350, 356
    bool cand = true;
    if (MASKED) {
        const int li = i - row0 < 0 ? i - row0 + ny : i - row0;
        cand = finite_cell(sb_ldg(dem + (long)li * nx + j)) && nv >= (int)ceil(min_coverage * (double)n);
        if (nv != n) { nn = sb_add((double)nv, kEps); tss = tsm; }
    }
    // core.py:360-367, operation for operation
    double a = sb_div(xc, tss);
    const double t1 = sb_mul(tss, sb_mul(a, a));
    const double err = sb_add(sb_mul(sb_div(1.0, nn), sb_add(sb_sub(t1, sb_mul(sb_mul(2.0, a), xc)), t3)), kEps);
    double s = fabs(sb_div(t1, err));
    if (poison) { a = NAN; s = NAN; }                               // a NaN in the DEM reaches every pixel (section 4)
    if (!cand) { a = 0.0; s = 0.0; }
    if (p.errmode != 0) {                                             // core.py:369-371
        const double xr = sb_add(sb_mul(sb_ldg(xvec + j), p.ca), sb_mul(sb_ldg(yvec + i), p.sa));
        if ((p.errmode == 1 && xr <= 0.0) || (p.errmode == 2 && xr >= 0.0)) s = 0.0;
    }
    if (i < p.i_lo || i > p.i_hi || j < p.j_lo || j > p.j_hi) { a = 0.0; s = 0.0; }   // core.py:373-375
    amp[(long)px * n_tmpls + k] = a;
    snr[(long)px * n_tmpls + k] = s;
}

// core.compare (core.py:198-243) on full planes with the reference's exact
// semantics (strict compares; an exact tie zeroes the pixel).  this_age / this_angle
// are scalars when the pointers are null.
SB_GLOBAL k_compare(long n, double* best_amp, double* best_age, double* best_angle, double* best_snr,
                    const double* SB_RESTRICT amp, const double* SB_RESTRICT age_p,
                    const double* SB_RESTRICT angle_p, const double* SB_RESTRICT snr,
                    double age_s, double angle_s) {
    const long i = (long)sb_bx() * 256 + sb_tid();
    if (i >= n) return;
    const double bs = best_snr[i], ts = snr[i];
    const double keep = bs > ts ? 1.0 : 0.0, take = bs < ts ? 1.0 : 0.0;
    const double ta = amp[i];
    const double tg = age_p ? age_p[i] : age_s;
    const double tn = angle_p ? angle_p[i] : angle_s;
    best_amp[i] = sb_add(sb_mul(keep, best_amp[i]), sb_mul(take, ta));
    best_age[i] = sb_add(sb_mul(keep, best_age[i]), sb_mul(take, tg));
    best_angle[i] = sb_add(sb_mul(keep, best_angle[i]), sb_mul(take, tn));
    best_snr[i] = sb_add(sb_mul(keep, bs), sb_mul(take, ts));
}

// debugging / unit-test kernel: batched forward FFT of length N, rows of `in`
template <int N, typename R>
SB_GLOBAL k_fft_rows(int rows, const typename Vec<R>::v2* SB_RESTRICT in, typename Vec<R>::v2* SB_RESTRICT outp, int inverse,
                     const typename Vec<R>::v2* SB_RESTRICT tw) {
    typedef typename Vec<R>::v2 C2;
    constexpr int T = N / E;
    const int grp = sb_tid() / T, t = sb_tid() % T;
    constexpr int GP = (T > 256 ? T : 256) / T;
    C2* sm = (C2*)sb_shared() + grp * sbfft::padded_len(N);
    const int r = sb_bx() * GP + grp;
    const bool active = r < rows;
    C2 v[E];
#pragma unroll
    for (int q = 0; q < E; ++q) {
        C2 a = active ? in[(long)r * N + t + q * T] : mk2<R>((R)0, (R)0);
        v[q] = inverse ? mk2<R>(a.y, a.x) : a;
    }
    sbfft::forward<N, R>(v, t, sm, tw);
    if (active) {
#pragma unroll
        for (int q = 0; q < E; ++q)
            outp[(long)r * N + t + q * T] = inverse ? mk2<R>(v[q].y, v[q].x) : v[q];
    }
}

}  // namespace sb
