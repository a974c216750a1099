// Host side of the C ABI declared in include/scarplet_b200.h: plan, workspace,
// tile / batch scheduling and kernel launches.  No torch types, no CPU compute path.
#include "../../include/scarplet_b200.h"

#include <algorithm>
#include <cstdlib>
#include <map>
#include <string>
#include <type_traits>
#include <vector>

#include "sb_kernels.cuh"
#include "sb_fast.cuh"
#include "sb_aux.cuh"
#include "sb_r64.cuh"

static_assert(sizeof(sb_template) == sizeof(sb::Tmpl), "sb_template / sb::Tmpl layout");
static_assert(sizeof(sb_angle) == sizeof(sb::Angle), "sb_angle / sb::Angle layout");
static_assert(offsetof(sb_template, kind) == offsetof(sb::Tmpl, kind), "layout");
static_assert(offsetof(sb_template, idx) == offsetof(sb::Tmpl, idx), "layout");
static_assert(offsetof(sb_template, state) == offsetof(sb::Tmpl, state), "layout");
static_assert(offsetof(sb_template, i_lo) == offsetof(sb::Tmpl, i_lo), "layout");
static_assert(offsetof(sb_template, tscale) == offsetof(sb::Tmpl, tscale), "layout");

namespace {

thread_local std::string g_err;

int fail(const std::string& msg) {
    g_err = msg;
    return 1;
}

#define SB_TRY(expr)                                                                      \
    do {                                                                                  \
        int _e = (expr);                                                                  \
        if (_e != 0)                                                                      \
            return fail(std::string(#expr) + ": " + sb_rt_error_string(_e) + " (" +       \
                        std::to_string(_e) + ")");                                        \
    } while (0)

#define SB_OK(expr)                     \
    do {                                \
        int _s = (expr);                \
        if (_s != 0) return _s;         \
    } while (0)

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
};

bool is_pow2(int n) { return n > 0 && (n & (n - 1)) == 0; }
constexpr int kMinFft = 128;
constexpr int kMaxFftSupported = 8192;
constexpr int kMaxFftMasked = 4096;      // k_fit_rows_gm's shared memory

// One FFT tile along an axis: domain length P, first output pixel o, out output pixels.
struct TileSpec {
    int P = 0, o = 0, out = 0;
};

struct AxisPlan {
    std::vector<TileSpec> tiles;
    int lo = 0, hi = 0;   // support offsets of the templates along this axis
    bool periodic = false;
    int max_p() const {
        int m = 0;
        for (auto& t : tiles) m = std::max(m, t.P);
        return m;
    }
};

}  // namespace

struct sb_plan {
    int ny = 0, nx = 0;
    double dx = 1, dx2 = 1, dy2 = 1;
    int device = 0;
    sb_stream_t stream = 0;
    bool own_stream = false;
    // Row slab (spatial sharding, SURVEY 8e): this plan computes raster rows slab_lo .. slab_hi - 1
    // and holds DEM rows row0 .. row0 + drows - 1 (mod ny).  Whole raster: 0, ny, 0, ny.
    int slab_lo = 0, slab_hi = 0, row0 = 0, drows = 0;
    double* d_dem = nullptr;
    bool own_dem = false;
    double* d_diffs = nullptr;      // dxx, dxy, dyy planes of the current DEM (dem.py:88-99), complex128 pipeline only
    bool diffs64_valid = false;
    float4* d_diffs32 = nullptr;    // the same, float32, interleaved per pixel (complex64 pipeline)
    double* d_x = nullptr;
    double* d_y = nullptr;
    int n_states = 1;               // best states (one per template scale in a multi-scale search)
    int best_copies = 1;            // copies of the best state (sub-streams of the fit kernel on small rasters)
    float* d_bsnr = nullptr;        // [best_copies][n_states][slab rows][nx]; copy 0 is the state
    float* d_bamp = nullptr;
    int* d_bidx = nullptr;
    std::map<long, void*> tw;      // twiddle tables keyed by 2 * n + (float64 ? 1 : 0); -64: radix-64 core
    int precision = 32;            // 32: complex64 pipeline, 64: complex128 pipeline
    Buf cr, fct, trt, part, gbuf, sums, fit, tmpls, angles, tables, raw, tbox, slots, cross, casa, aux, spec9, coef;
    int fit_substreams = 0;        // 0: automatic (small rasters), else the number of sub-streams of the fit kernel
    int fast = 1;                  // 1: pipelined complex64 kernels (sb_fast.cuh), 0: simple kernels
    // persistent column kernel: 1 always, 0 never, -1 (default) when a search angle carries at least
    // four templates -- with fewer, half of its thread groups idle and the per-angle staging of
    // the spectrum columns is not amortised (C2: 94 ms persistent, 69 ms per-template)
    int conv_persist = -1;
    int conv_r64 = 1;              // Py = 4096: column kernel on the radix-64 core (sb_r64.cuh)
    long launches = 0;
    double c2_scale = 1.0;
    double curv_sumsq = 0.0, curv_count = 0.0;   // over the plan's own rows (slab_lo .. slab_hi)
    bool dem_nonfinite = false;    // the DEM holds a NaN / Inf: every FFT domain is poisoned like the reference's
    // nodata policy (sb_plan_set_nodata): requested, and in force for the current DEM
    int nodata_req = SB_NODATA_PROPAGATE, nodata = SB_NODATA_PROPAGATE;
    double min_cov_req = 1.0, min_cov = 1.0;
    Buf fitm;
    Buf fs_idx, fs_out;            // sb_fit_surface: jobs, template order and pixels; output chunk
    // fit confidence region (sb_region_sweep): planes [count][rank_lo][rank_hi][words] over the plan's
    // rows (allocated on first use), and the per-flat-index age rank / orientation position tables
    Buf region, rtab;
    int region_words = 0, region_npos = 0, region_nranks = 0;
    // secondary fit (sb_secondary_sweep): the winner's orientation position per pixel of the plan's
    // rows (uint16; its per-flat-index position table goes in rtab)
    Buf spos;
    // fit peak (sb_peak_sweep): four neighbour SNR planes and the winner code plane of the plan's rows
    // (allocated on first use), and the ranks / positions of the sweep that wrote them (0: none)
    Buf peak;
    int peak_nranks = 0, peak_npos = 0;
    int profile = 0;
    std::vector<sb_event_t> ev_pool;
    struct EvPair { int kind; sb_event_t a, b; };
    std::vector<EvPair> ev_live;
    size_t ev_used = 0;
    double prof_ms[6] = {0, 0, 0, 0, 0, 0};
    long prof_n[6] = {0, 0, 0, 0, 0, 0};
    long workspace_mb = 0;         // 0: half of the free device memory, at most 48 GB
    int max_fft = kMaxFftSupported;
    int force_pad = 0;
    int mixed_tiles = 1;           // tiles of different FFT lengths along an axis (least wasted area)
    int last_geom[6] = {0, 0, 0, 0, 0, 0};
    double last_fft_area = 0.0;    // sum over tiles of Py * Px of the last sweep

    long brows() const { return slab_hi - slab_lo; }
    long bn() const { return brows() * (long)nx; }          // pixels of one best state
    bool whole() const { return slab_lo == 0 && slab_hi == ny; }
};

namespace {

int ensure(Buf& b, size_t bytes) {
    if (bytes <= b.cap) return 0;
    if (b.p) sb_rt_free(b.p);
    b.p = nullptr;
    b.cap = 0;
    SB_TRY(sb_rt_malloc(&b.p, bytes));
    b.cap = bytes;
    return 0;
}

void release(Buf& b) {
    if (b.p) sb_rt_free(b.p);
    b.p = nullptr;
    b.cap = 0;
}

// a table of `count` elements in pl->tw under `key`: filled on the host and uploaded on first use
template <typename C, typename Fill>
int cached_table(sb_plan* pl, long key, size_t count, Fill fill, const C** out) {
    auto it = pl->tw.find(key);
    if (it == pl->tw.end()) {
        std::vector<C> host(count);
        fill(host.data());
        void* d = nullptr;
        SB_TRY(sb_rt_malloc(&d, count * sizeof(C)));
        SB_TRY(sb_rt_h2d(d, host.data(), count * sizeof(C), pl->stream));
        SB_TRY(sb_rt_sync(pl->stream));
        it = pl->tw.emplace(key, d).first;
    }
    *out = (const C*)it->second;
    return 0;
}

template <typename R>
int twiddles(sb_plan* pl, int n, const typename Vec<R>::v2** out) {
    int count = 0;
    {   // same stage walk as sbfft::fill_twiddles
        int ns = 1;
        for (int s = 0; n > ns; ++s) {
            int rest = n / ns, r = rest >= 16 ? 16 : rest;
            if (s > 0) count += (r - 1) * ns;
            ns *= r;
        }
    }
    return cached_table(pl, 2L * n + (sizeof(R) == 8 ? 1 : 0), std::max(count, 1),
                        [n](typename Vec<R>::v2* h) { sbfft::fill_twiddles<R>(n, h); }, out);
}

// table of the radix-64 core (sb_r64.cuh)
int twiddles64(sb_plan* pl, const float2** out) {
    return cached_table(pl, -64, (size_t)sb64::kTwRows * sb64::R, sb64::fill_twiddles64, out);
}

template <typename F>
int dispatch_n(int n, F&& f) {
#ifdef SB_DEV_N   // developer builds (scratch/devbuild.sh): one FFT length, a tenth of the compile time
    if (n == SB_DEV_N) return f(std::integral_constant<int, SB_DEV_N>{});
    return fail("developer build: only FFT length " + std::to_string(SB_DEV_N));
#else
    switch (n) {
        case 128: return f(std::integral_constant<int, 128>{});
        case 256: return f(std::integral_constant<int, 256>{});
        case 512: return f(std::integral_constant<int, 512>{});
        case 1024: return f(std::integral_constant<int, 1024>{});
        case 2048: return f(std::integral_constant<int, 2048>{});
        case 4096: return f(std::integral_constant<int, 4096>{});
        case 8192: return f(std::integral_constant<int, 8192>{});
        default: return fail("unsupported FFT length " + std::to_string(n));
    }
#endif
}

template <int N, typename R>
struct Shape {
    static constexpr int T = N / sbfft::E;
    static constexpr int threads = T > 256 ? T : 256;
    static constexpr int GP = threads / T;
    static constexpr size_t smem = (size_t)GP * sbfft::padded_len(N) * sizeof(typename Vec<R>::v2);
    // k_conv_cols adds a park buffer of N elements per group
    static constexpr size_t smem_conv = (size_t)GP * (sbfft::padded_len(N) + N) * sizeof(typename Vec<R>::v2);
    // pipelined kernels (sb_fast.cuh): two exchange buffers per group; k_fit_rows_g adds the
    // batch's scalars, the active-template list (+ its length), the flags, the gbuf slots and the
    // compact twiddle table
    static constexpr size_t smem_conv_f = (size_t)GP * 2 * sbfft::padded_len(N) * sizeof(float2);
    static constexpr size_t smem_fit_f = smem_conv_f + sb::kFitMaxBatch * sizeof(sb::FitT) +
                                         (3 * sb::kFitMaxBatch + 2) * sizeof(int) +
                                         (size_t)sbfft::ctw_count<float>(N) * sizeof(float2);
};

// Every kernel launch of the library: a kernel that asks for more than the default 48 KB of
// dynamic shared memory is allowed it first, then it runs on the plan's stream; the launch is
// counted (sb_plan_launch_count) and checked.
template <typename... P, typename... A>
int launch(sb_plan* pl, const char* what, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, A... args) {
#ifndef SB_EMU
    if (smem > 48 * 1024)
        SB_TRY((int)cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
#endif
    SB_LAUNCH(kern, grid, block, smem, pl->stream, args...);
    pl->launches++;
    const int e = sb_rt_last_error();
    if (e != 0) return fail(std::string(what) + ": " + sb_rt_error_string(e));
    return 0;
}

int div_up(long a, long b) { return (int)((a + b - 1) / b); }

enum { K_CURV_ROWS = 0, K_CURV_COLS, K_TMPL_ROWS, K_TMPL_SUMS, K_CONV_COLS, K_FIT_ROWS };

sb_event_t take_event(sb_plan* pl) {
    if (pl->ev_used == pl->ev_pool.size()) {
        sb_event_t e;
        sb_rt_event_create(&e);
        pl->ev_pool.push_back(e);
    }
    return pl->ev_pool[pl->ev_used++];
}

struct ProfScope {   // brackets one launch with events when profiling is on
    sb_plan* pl;
    int kind;
    sb_event_t a{}, b{};
    ProfScope(sb_plan* p, int k) : pl(p), kind(k) {
        if (pl->profile) { a = take_event(pl); sb_rt_event_record(a, pl->stream); }
    }
    ~ProfScope() {
        if (pl->profile) {
            b = take_event(pl);
            sb_rt_event_record(b, pl->stream);
            pl->ev_live.push_back({kind, a, b});
        }
    }
};

void drain_profile(sb_plan* pl) {
    if (pl->ev_live.empty()) return;
    sb_rt_sync(pl->stream);
    for (auto& e : pl->ev_live) {
        pl->prof_ms[e.kind] += sb_rt_event_ms(e.a, e.b);
        pl->prof_n[e.kind]++;
    }
    pl->ev_live.clear();
    pl->ev_used = 0;
}

// curvature RMS -> power-of-two factor that brings curv**2 to the magnitude of curv; a
// non-finite sum means a NaN / Inf somewhere in the DEM: it reaches every output pixel through
// the reference's full-raster fft2 (dem.py:105, core.py:353-363), and tiles or slabs that do
// not hold the cell have to be told
void apply_curv_stats(sb_plan* pl, double sumsq, double count) {
    const double sigma = std::sqrt(sumsq / (2.0 * std::max(count, 1.0)));
    pl->c2_scale = 1.0;
    if (std::isfinite(sigma) && sigma > 1e-150 && sigma < 1e150)
        pl->c2_scale = std::exp2(std::round(-std::log2(sigma)));
    pl->dem_nonfinite = pl->nodata != SB_NODATA_MASK && !std::isfinite(sumsq);
}

long bn_all(const sb_plan* pl) { return pl->bn() * pl->n_states; }

int alloc_best(sb_plan* pl) {
    for (void* p : {(void*)pl->d_bsnr, (void*)pl->d_bamp, (void*)pl->d_bidx})
        if (p) sb_rt_free(p);
    pl->d_bsnr = nullptr; pl->d_bamp = nullptr; pl->d_bidx = nullptr;
    pl->best_copies = 1;
    pl->region_npos = 0;           // region planes of the old rows / states are void
    pl->peak_npos = 0;             // and so are the fit peak's
    const size_t n = (size_t)pl->bn() * pl->n_states;
    int e = 0;
    e |= sb_rt_malloc((void**)&pl->d_bsnr, n * sizeof(float));
    e |= sb_rt_malloc((void**)&pl->d_bamp, n * sizeof(float));
    e |= sb_rt_malloc((void**)&pl->d_bidx, n * sizeof(int));
    if (e) return fail("out of device memory (best state)");
    return sb_best_reset(pl);
}

// angle-independent second differences of the current DEM (once per DEM) and its curvature scale
int after_dem(sb_plan* pl) {
    const long n = (long)pl->drows * pl->nx;
    if (!pl->d_diffs32) SB_TRY(sb_rt_malloc((void**)&pl->d_diffs32, (size_t)n * sizeof(float4)));
    pl->diffs64_valid = false;
    pl->nodata = pl->nodata_req;
    pl->min_cov = pl->min_cov_req;
    const bool masked = pl->nodata == SB_NODATA_MASK;
    if (masked) {
        SB_OK(launch(pl, "k_second_differences_m", sb::k_second_differences_m, dim3(div_up(n, 256)), dim3(256), 0,
                     pl->ny, pl->nx, pl->row0, pl->drows, (const double*)pl->d_dem, pl->dx, pl->dx2, pl->dy2,
                     pl->d_diffs32));
    } else {
        SB_OK(launch(pl, "k_second_differences", sb::k_second_differences, dim3(div_up(n, 256)), dim3(256), 0, pl->ny,
                     pl->nx, pl->row0, pl->drows, (const double*)pl->d_dem, pl->dx, pl->dx2, pl->dy2, (double*)nullptr,
                     pl->d_diffs32));
    }
    // statistics over the plan's own rows only, so that the slabs of a sharded raster add up
    const int own_first = pl->slab_lo - pl->row0 + (pl->slab_lo < pl->row0 ? pl->ny : 0);
    const long own = pl->brows() * (long)pl->nx;
    const int blocks = std::max(1, std::min(1024, div_up(own, 256)));
    SB_OK(ensure(pl->raw, (size_t)blocks * sizeof(double)));
    auto sumsq_kern = masked ? sb::k_curv_sumsq_m : sb::k_curv_sumsq;
    SB_OK(launch(pl, "k_curv_sumsq", sumsq_kern, dim3(blocks), dim3(256), 256 * sizeof(double), pl->ny, pl->nx,
                 pl->row0, pl->drows, own_first, (int)pl->brows(), (const double*)pl->d_dem, pl->dx, pl->dx2, pl->dy2,
                 (double*)pl->raw.p));
    std::vector<double> part(blocks);
    SB_TRY(sb_rt_d2h(part.data(), pl->raw.p, (size_t)blocks * sizeof(double), pl->stream));
    SB_TRY(sb_rt_sync(pl->stream));
    double sum = 0.0;
    for (double v : part) sum += v;
    pl->curv_sumsq = sum;
    pl->curv_count = (double)own;
    apply_curv_stats(pl, sum, (double)own);
    return 0;
}

int ensure_diffs64(sb_plan* pl) {
    if (pl->diffs64_valid) return 0;
    const long n = (long)pl->drows * pl->nx;
    if (!pl->d_diffs) SB_TRY(sb_rt_malloc((void**)&pl->d_diffs, (size_t)n * 3 * sizeof(double)));
    SB_OK(launch(pl, "k_second_differences", sb::k_second_differences, dim3(div_up(n, 256)), dim3(256), 0, pl->ny,
                 pl->nx, pl->row0, pl->drows, (const double*)pl->d_dem, pl->dx, pl->dx2, pl->dy2, pl->d_diffs,
                 (float4*)nullptr));
    pl->diffs64_valid = true;
    return 0;
}

// relative cost per point and AXIS of the per-template kernels at FFT length P (the cost of a tile
// is the product over its two axes), measured (bench.py, one B200): 4096 has the radix-64 column
// kernel; 8192 needs a fourth exchange stage and has no persistent column kernel -- C4 on its
// periodic 8192^2 domain takes 1.36 x the time per pixel of C3 on 4096^2 (1.17 per axis), and
// 9 % less than on 3 x 3 padded tiles of 4096 / 2048
double length_weight(int P) {
    switch (P) {
        case 8192: return 1.2;
        case 4096: return 1.0;
        case 2048: return 1.1;
        case 1024: return 1.15;
        default: return 1.3;
    }
}

// Cover output pixels [r0, r1) of an axis of n pixels with FFT tiles.  A tile of length P
// yields P - ext output pixels (ext = support extent of the templates along the axis); tiles
// of different lengths are mixed so that the summed (weighted) FFT length is least -- e.g.
// 16384 px with a 313 px support: 4 x 4096 + 1 x 2048 = 18432 instead of 5 x 4096 = 20480.
int plan_axis(const sb_plan* pl, int n, int r0, int r1, int lo, int hi, bool allow_periodic, AxisPlan* ax) {
    lo = std::min(lo, 0);
    hi = std::max(hi, 0);
    ax->lo = lo;
    ax->hi = hi;
    ax->tiles.clear();
    const int ext = hi - lo + 1;
    const int len = r1 - r0;
    // complex128 at 8192 would need 270 KB of shared memory per column in k_conv_cols, the masked
    // fit kernel 264 KB per CTA
    const int max_fft = std::min(pl->max_fft, pl->precision == 64 ? 4096
                                              : pl->nodata == SB_NODATA_MASK ? kMaxFftMasked : kMaxFftSupported);
    const bool can_periodic = allow_periodic && r0 == 0 && r1 == n && is_pow2(n) && n >= kMinFft && n <= max_fft &&
                              !pl->force_pad;
    auto take_periodic = [&]() {
        ax->periodic = true;
        ax->tiles.clear();
        TileSpec t;
        t.P = n; t.o = 0; t.out = n;
        ax->tiles.push_back(t);
        return 0;
    };
    if (can_periodic && (!pl->mixed_tiles || n <= 4096)) return take_periodic();
    ax->periodic = false;
    std::vector<int> Ps;
    for (int P = kMinFft; P <= max_fft; P <<= 1) {
        if (P < ext + 1 || hi >= P / 2 || -lo > P / 2 || P - ext < 1) continue;
        Ps.push_back(P);
    }
    if (Ps.empty()) {
        if (can_periodic) return take_periodic();
        return fail("template support (" + std::to_string(ext) + " px) does not fit max_fft=" +
                    std::to_string(max_fft));
    }
    std::vector<int> chosen;
    if (pl->mixed_tiles) {
        // covering knapsack: best[r] = least cost to cover r more pixels
        std::vector<double> best(len + 1, 0.0);
        std::vector<int> pick(len + 1, 0);
        for (int r = 1; r <= len; ++r) {
            best[r] = -1.0;
            for (int P : Ps) {
                const int cap = P - ext;
                // a small per-tile charge keeps the count of tiles (launches, halo re-reads) down
                const double c = P * length_weight(P) + 48.0 + best[std::max(0, r - cap)];
                if (best[r] < 0 || c < best[r] - 1e-9) { best[r] = c; pick[r] = P; }
            }
        }
        // the exact circular domain of a power-of-two axis, when it is cheaper than padded tiles
        if (can_periodic && n * length_weight(n) <= best[len]) return take_periodic();
        for (int r = len; r > 0; r = std::max(0, r - (pick[r] - ext))) chosen.push_back(pick[r]);
        std::sort(chosen.begin(), chosen.end(), [](int a, int b) { return a > b; });
    } else {
        long best_cost = -1;
        int bestP = 0, tiles = 0;
        for (int P : Ps) {
            const int t = div_up(len, P - ext);
            const long cost = (long)t * P;
            // equal cost: 4096, the length the pipelined kernels are tuned for, beats 2048
            if (best_cost < 0 || cost < best_cost || (cost == best_cost && P == 4096)) { best_cost = cost; bestP = P; tiles = t; }
        }
        chosen.assign(tiles, bestP);
    }
    // spread the slack over the tiles in proportion to their capacity (equal lengths -> equal tiles)
    long cap_total = 0;
    for (int P : chosen) cap_total += P - ext;
    int o = r0, left = len;
    long cap_left = cap_total;
    for (size_t i = 0; i < chosen.size(); ++i) {
        const int cap = chosen[i] - ext;
        int out = i + 1 == chosen.size() ? left : (int)std::min<long>(cap, div_up((long)left * cap, cap_left));
        out = std::min(out, cap);
        TileSpec t;
        t.P = chosen[i]; t.o = o; t.out = out;
        ax->tiles.push_back(t);
        o += out;
        left -= out;
        cap_left -= cap;
    }
    if (left != 0) return fail("internal: tile plan does not cover the axis");
    return 0;
}

void fill_axis(const AxisPlan& ax, int n, const TileSpec& t, int* o, int* out_n, int* split, int* dl, int* need_lo,
               int* need_hi) {
    *dl = -(n & 1);
    *o = t.o;
    *out_n = t.out;
    if (ax.periodic) {
        *split = t.P;
        *need_lo = 0;
        *need_hi = t.P - 1;
    } else {
        *split = *out_n - *dl - ax.lo + 1;
        *need_lo = -*dl - ax.hi;
        *need_hi = *out_n - 1 - *dl - ax.lo;
    }
}

struct SweepOut {
    double* raw_amp = nullptr;
    double* raw_snr = nullptr;
    // the threshold pass of a fit confidence region (sb_region_sweep): the fit kernel records the
    // templates that reach each pixel's threshold in these planes; no best state changes
    const sb::RegionOut* region = nullptr;
    // the sweep of a secondary fit (sb_secondary_sweep): every record folds into best state 1, through
    // the fit kernel's separation test
    const sb::SecondOut* second = nullptr;
    // the neighbour pass of a fit peak (sb_peak_sweep): the fit kernel records the axis neighbours of
    // each pixel's winner in these planes; no best state changes
    const sb::PeakOut* peak = nullptr;
};

// the templates of one best state inside a chunk (one launch of the column kernel)
struct SlotGroup {
    int state = 0;
    int off = 0;       // offset into the plan's slot table; -1: the whole chunk, in order
    int count = 0;
    bool err = false;  // some template of the group has a get_err_mask
};
struct Chunk {
    int pb = 0, cnt = 0;
    std::vector<SlotGroup> groups;
};
struct AngleBatch {
    int a0 = 0, a1 = 0;
    std::vector<Chunk> chunks;
};

template <typename R>
int run_sweep_t(sb_plan* pl, const sb_angle* angles, int n_angles, const sb_template* tmpls_in, int n_tmpls,
                SweepOut so, const int32_t* hint) {
    typedef typename Vec<R>::v2 C2;
    typedef typename Vec<R>::v4 C4;
    if (!pl->d_dem) return fail("no DEM set (sb_set_dem_host / sb_set_dem_dev)");
    if (pl->ny < 3 || pl->nx < 3) return fail("raster too small for a template search");
    if (!pl->d_x || !pl->d_y) return fail("no axis vectors set (sb_set_axes_host)");
    if (n_tmpls <= 0 || n_angles <= 0) return 0;
    if (so.raw_amp && !pl->whole()) return fail("match_template planes need a plan over the whole raster");
    constexpr bool kF32 = std::is_same<R, float>::value;
    const bool fast = kF32 && pl->fast;
    // nodata-masked search: complex64 pipelined kernels only
    const bool masked = pl->nodata == SB_NODATA_MASK;
    if (masked && so.raw_amp) return fail("nodata mask: sb_match_template keeps the reference's NaN semantics");
    if (masked && !fast) return fail("nodata mask needs precision 32 and the option fast");
    if (so.region && !fast) return fail("fit region needs precision 32 and the option fast");
    if (so.peak && !fast) return fail("fit peak needs precision 32 and the option fast");
    // a region or peak pass reads best state 0 and writes planes of its own
    const bool reads_best = so.region || so.peak;
    if (!fast) SB_OK(ensure_diffs64(pl));

    // order templates by search angle (then best state) so that each curvature spectrum is built once
    std::vector<sb_template> tm(tmpls_in, tmpls_in + n_tmpls);
    std::stable_sort(tm.begin(), tm.end(), [](const sb_template& a, const sb_template& b) {
        return a.angle_id != b.angle_id ? a.angle_id < b.angle_id : a.state < b.state;
    });
    int lo_y = 0, hi_y = 0, lo_x = 0, hi_x = 0, syp = 1;
    bool any_err = false, multi_state = false;
    for (auto& t : tm) {
        if (t.kind == SB_KIND_RASTER && (n_tmpls != 1 || !pl->tbox.p))
            return fail("raster templates go through sb_match_template_raster, one at a time");
        if (t.angle_id < 0 || t.angle_id >= n_angles) return fail("template angle_id out of range");
        if (t.state < 0 || t.state >= pl->n_states) return fail("template state out of range (option \"states\")");
        if (so.region && t.state != 0) return fail("fit region: every record must be in best state 0 (state != 0)");
        if (so.peak && t.state != 0) return fail("fit peak: every record must be in best state 0 (state != 0)");
        if (t.sy_hi < t.sy_lo || t.sx_hi < t.sx_lo) return fail("empty template support box");
        if (t.sy_lo < -(pl->ny / 2) || t.sy_hi > pl->ny - 1 - pl->ny / 2 || t.sx_lo < -(pl->nx / 2) ||
            t.sx_hi > pl->nx - 1 - pl->nx / 2)
            return fail("template support box exceeds the raster");
        lo_y = std::min(lo_y, t.sy_lo);
        hi_y = std::max(hi_y, t.sy_hi);
        lo_x = std::min(lo_x, t.sx_lo);
        hi_x = std::max(hi_x, t.sx_hi);
        syp = std::max(syp, t.sy_hi - t.sy_lo + 1);
        any_err |= t.errmode != 0;
        multi_state |= t.state != tm[0].state;
    }
    if (hint) {
        // the extents of the WHOLE search this sweep is a share of: FFT domains, tiles and kernel
        // variants are then chosen exactly as the undivided search chooses them
        lo_y = std::min(lo_y, hint[0]); hi_y = std::max(hi_y, hint[1]);
        lo_x = std::min(lo_x, hint[2]); hi_x = std::max(hi_x, hint[3]);
        syp = std::max(syp, hint[1] - hint[0] + 1);
    }
    syp += syp & 1;      // the row kernels store row pairs
    AxisPlan ay, ax;
    SB_OK(plan_axis(pl, pl->ny, pl->slab_lo, pl->slab_hi, lo_y, hi_y, pl->whole(), &ay));
    SB_OK(plan_axis(pl, pl->nx, 0, pl->nx, lo_x, hi_x, true, &ax));
    const int Pym = ay.max_p(), Pxm = ax.max_p();
    if (!pl->whole()) {
        // the curvature rows (+ 1 for the stencil) every tile needs must lie inside the slab's halo
        for (auto& t : ay.tiles) {
            int o, out_n, split, dl, nlo, nhi;
            fill_axis(ay, pl->ny, t, &o, &out_n, &split, &dl, &nlo, &nhi);
            const long first = (long)o + nlo - 1, last = (long)o + nhi + 1;
            const long have_lo = (long)pl->slab_lo - (pl->slab_lo - pl->row0 + (pl->slab_lo < pl->row0 ? pl->ny : 0));
            if (pl->drows < pl->ny && (first < have_lo || last >= have_lo + pl->drows))
                return fail("row slab: halo too small for the template support (need rows " + std::to_string(first) +
                            ".." + std::to_string(last) + ", have " + std::to_string(have_lo) + ".." +
                            std::to_string(have_lo + pl->drows - 1) + ")");
        }
    }

    // batch sizes from the workspace budget (sized for the largest tile)
    const int KXm = Pxm / 2 + 1;
    const int kpitch_m = Pxm / 2 + 8;
    int need_rows_max = 0;
    for (auto& t : ay.tiles) need_rows_max = std::max(need_rows_max, ay.periodic ? t.P : std::min(t.P, t.out + (hi_y - lo_y) + 2));
    const size_t per_angle = (size_t)(need_rows_max + 2) * KXm * sizeof(C4) + (size_t)2 * KXm * Pym * sizeof(C2);
    const size_t per_tmpl = (size_t)KXm * syp * sizeof(C4) + (size_t)Pym * kpitch_m * sizeof(C4) +
                            (size_t)syp * sizeof(double2) + sizeof(sb::TSum);
    size_t budget = (size_t)pl->workspace_mb << 20;
    if (pl->workspace_mb <= 0) {
        // auto: the workspace already held counts as free
        size_t free_b = 0, total_b = 0, held = 0;
        for (const Buf* b : {&pl->cr, &pl->fct, &pl->trt, &pl->part, &pl->gbuf}) held += b->cap;
        if (sb_rt_mem_info(&free_b, &total_b) != 0) free_b = (size_t)16 << 30;
        budget = std::min<size_t>((size_t)48 << 30, std::max<size_t>((size_t)1 << 30, (free_b + held) / 2));
    }
    // templates per angle (max) decides the split of the budget
    std::vector<int> first(n_angles + 1, 0);
    for (auto& t : tm) first[t.angle_id + 1]++;
    int max_per_angle = 1;
    for (int a = 0; a < n_angles; ++a) {
        max_per_angle = std::max(max_per_angle, first[a + 1]);
        first[a + 1] += first[a];
    }
    if (hint) max_per_angle = std::max(max_per_angle, hint[4]);
    // a masked sweep carries a companion per template through the per-template kernels, in the same
    // launches (at most 64 records)
    const int rec_per_tmpl = masked ? 2 : 1;
    int Bt = (int)std::max<size_t>(1, std::min<size_t>(64 / rec_per_tmpl, (budget * 6 / 10) / (per_tmpl * rec_per_tmpl)));
    int Ba = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_angles, (budget * 4 / 10) / per_angle));
    Ba = std::min(Ba, 64);
    if (max_per_angle == 1) Bt = std::min(Bt, Ba), Ba = std::min(Ba, Bt);
    Bt = std::min(Bt, n_tmpls);
    // whole angles per batch when they fit: templates of one angle share the curvature spectra
    if (max_per_angle > 1 && Bt >= max_per_angle) {
        Bt = (Bt / max_per_angle) * max_per_angle;
    }

    const int rpitch_max = need_rows_max + (need_rows_max & 1);
    SB_OK(ensure(pl->cr, (size_t)std::max(Ba, fast ? sb::kDiffPairs : 0) * KXm * rpitch_max * sizeof(C4)));
    if (fast) {
        SB_OK(ensure(pl->spec9, (size_t)2 * sb::kDiffPairs * KXm * Pym * sizeof(float2)));
        SB_OK(ensure(pl->coef, (size_t)n_angles * sizeof(sb::SpecCoef)));
        std::vector<sb::SpecCoef> coef(n_angles);
        for (int a = 0; a < n_angles; ++a) {
            // cos^2, 2 sin cos, sin^2 of the search angle, each rounded to float32, and their products
            const double c2 = (double)(float)angles[a].cos2_a, sc = (double)(float)(2.0 * angles[a].sin_a * angles[a].cos_a),
                         s2 = (double)(float)angles[a].sin2_a;
            const double v[sb::kDiffPlanes] = {c2, -sc, s2, c2 * c2, sc * sc, s2 * s2, -2.0 * c2 * sc, 2.0 * c2 * s2, -2.0 * sc * s2};
            for (int k = 0; k < sb::kDiffPlanes; ++k) coef[a].c[k] = (float)v[k];
            for (int k = sb::kDiffPlanes; k < sb::kDiffPlanes + 3; ++k) coef[a].c[k] = 0.f;
        }
        SB_TRY(sb_rt_h2d(pl->coef.p, coef.data(), coef.size() * sizeof(sb::SpecCoef), pl->stream));
        SB_TRY(sb_rt_sync(pl->stream));
    }
    // masked: orientation slot Ba of fct holds (F[U], F[U]), the spectra the companions multiply by
    SB_OK(ensure(pl->fct, (size_t)(Ba + (masked ? 1 : 0)) * 2 * KXm * Pym * sizeof(C2)));
    const int Br = Bt * rec_per_tmpl;
    SB_OK(ensure(pl->trt, (size_t)Br * KXm * syp * sizeof(C4)));
    SB_OK(ensure(pl->part, (size_t)Br * syp * sizeof(double2)));
    SB_OK(ensure(pl->gbuf, (size_t)Br * Pym * kpitch_m * sizeof(C4)));
    SB_OK(ensure(pl->sums, (size_t)Br * sizeof(sb::TSum)));
    SB_OK(ensure(pl->fit, (size_t)Br * sizeof(sb::FitT)));
    if (masked) SB_OK(ensure(pl->fitm, (size_t)Bt * sizeof(sb::FitM)));
    SB_OK(ensure(pl->tmpls, (size_t)n_tmpls * rec_per_tmpl * sizeof(sb::Tmpl)));
    SB_OK(ensure(pl->angles, (size_t)n_angles * sizeof(sb::Angle)));

    // the schedule: angle batches, chunks of templates, and per chunk the slots of each best state
    std::vector<AngleBatch> batches;
    std::vector<int> slot_table;
    for (int a0 = 0; a0 < n_angles; a0 += Ba) {
        AngleBatch ab;
        ab.a0 = a0;
        ab.a1 = std::min(n_angles, a0 + Ba);
        const int p0 = first[ab.a0], p1 = first[ab.a1];
        for (int pb = p0; pb < p1; pb += Bt) {
            Chunk ch;
            ch.pb = pb;
            ch.cnt = std::min(Bt, p1 - pb);
            std::vector<int> states;
            for (int i = 0; i < ch.cnt; ++i)
                if (std::find(states.begin(), states.end(), tm[pb + i].state) == states.end()) states.push_back(tm[pb + i].state);
            std::sort(states.begin(), states.end());
            for (int s : states) {
                // at most kFitMaxBatch slots per launch of the fit kernel
                SlotGroup gp;
                gp.state = s;
                auto flush = [&]() {
                    if (gp.count == 0) return;
                    if (states.size() == 1 && gp.count == ch.cnt) { gp.off = -1; slot_table.resize(slot_table.size() - gp.count); }
                    ch.groups.push_back(gp);
                    gp.count = 0; gp.err = false;
                };
                gp.off = (int)slot_table.size();
                for (int i = 0; i < ch.cnt; ++i) {
                    if (tm[pb + i].state != s) continue;
                    if (gp.count == sb::kFitMaxBatch) { flush(); gp.off = (int)slot_table.size(); }
                    slot_table.push_back(i);
                    gp.count++;
                    gp.err |= tm[pb + i].errmode != 0;
                }
                flush();
            }
            ab.chunks.push_back(ch);
        }
        if (!ab.chunks.empty()) batches.push_back(ab);
    }
    SB_OK(ensure(pl->slots, std::max<size_t>(1, slot_table.size()) * sizeof(int)));
    if (!slot_table.empty())
        SB_TRY(sb_rt_h2d(pl->slots.p, slot_table.data(), slot_table.size() * sizeof(int), pl->stream));
    // device records: a masked sweep lays each chunk out as its templates, then their companions
    // (k_tmpl_rows_sq packs t**2 with the power of two tscale**2; fct orientation slot Ba = F[U]) --
    // one run of the persistent column kernels, which stage their spectrum column per run of equal slots
    std::vector<sb_template> dev;
    if (masked) {
        dev.resize((size_t)2 * n_tmpls);
        for (auto& ab : batches)
            for (auto& ch : ab.chunks)
                for (int i = 0; i < ch.cnt; ++i) {
                    sb_template t = tm[ch.pb + i];
                    dev[2 * ch.pb + i] = t;
                    t.angle_id = ab.a0 + Ba;
                    t.tscale = t.tscale * t.tscale;
                    dev[2 * ch.pb + ch.cnt + i] = t;
                }
    }
    const std::vector<sb_template>& recs = masked ? dev : tm;
    SB_TRY(sb_rt_h2d(pl->tmpls.p, recs.data(), recs.size() * sizeof(sb::Tmpl), pl->stream));
    SB_TRY(sb_rt_h2d(pl->angles.p, angles, (size_t)n_angles * sizeof(sb::Angle), pl->stream));
    std::vector<double> casa;
    if (any_err && fast && !so.raw_amp) {
        // get_err_mask column ranges per (angle, raster row): cos / sin of the templates' alpha
        casa.assign((size_t)2 * n_angles, 0.0);
        for (auto& t : tm) { casa[2 * t.angle_id] = t.cos_t; casa[2 * t.angle_id + 1] = t.sin_t; }
        SB_OK(ensure(pl->casa, casa.size() * sizeof(double)));
        SB_OK(ensure(pl->cross, (size_t)n_angles * pl->ny * sizeof(int4)));
        SB_TRY(sb_rt_h2d(pl->casa.p, casa.data(), casa.size() * sizeof(double), pl->stream));
        SB_OK(launch(pl, "k_err_cross", sb::k_err_cross, dim3(div_up((long)n_angles * pl->ny, 256)), dim3(256), 0,
                     pl->ny, pl->nx, n_angles, (const double*)pl->casa.p, (const double*)pl->d_x,
                     (const double*)pl->d_y, (int4*)pl->cross.p));
    }
    // the host vectors must outlive the async copies
    SB_TRY(sb_rt_sync(pl->stream));

    // Sub-streams of the fit kernel: a small raster has too few row pairs to fill 148 SMs, so the
    // templates of a launch are dealt to nsub sub-streams (grid.y), each with its own copy of the
    // best state; the copies are folded into the plan's state at the end of the sweep.
    int nsub = 1;
    if (fast && !so.raw_amp) {
        nsub = pl->fit_substreams;
        if (nsub == 0) {
            const int T = std::max(Pxm / sbfft::E, 1), gp = std::max(256 / T, 1);
            const int ctas = div_up(Pym / 2, gp);
            nsub = std::max(1, std::min(8, 300 / std::max(ctas, 1)));
        }
        nsub = std::max(1, std::min(nsub, Bt / 2));
    }
    const long sub_stride = bn_all(pl);
    // (a region or peak pass keeps the sub-streams, whose templates all compare with state 0: no copies)
    if (nsub > 1 && !reads_best) {
        if (nsub > pl->best_copies) {
            // grow the best-state arrays to nsub copies, keeping copy 0 (the accumulated state)
            float *s2 = nullptr, *a2 = nullptr;
            int* i2 = nullptr;
            const size_t n1 = (size_t)sub_stride, nn = n1 * nsub;
            if (sb_rt_malloc((void**)&s2, nn * 4) || sb_rt_malloc((void**)&a2, nn * 4) || sb_rt_malloc((void**)&i2, nn * 4))
                return fail("out of device memory (best-state copies)");
            SB_TRY(sb_rt_d2d(s2, pl->d_bsnr, n1 * 4, pl->stream));
            SB_TRY(sb_rt_d2d(a2, pl->d_bamp, n1 * 4, pl->stream));
            SB_TRY(sb_rt_d2d(i2, pl->d_bidx, n1 * 4, pl->stream));
            SB_TRY(sb_rt_sync(pl->stream));
            sb_rt_free(pl->d_bsnr); sb_rt_free(pl->d_bamp); sb_rt_free(pl->d_bidx);
            pl->d_bsnr = s2; pl->d_bamp = a2; pl->d_bidx = i2;
            pl->best_copies = nsub;
        }
        if (so.second) {
            // state 1's copies only: an empty copy folded into state 0 could rewrite its indices
            const long b1 = pl->bn();
            for (int c = 1; c < nsub; ++c)
                SB_OK(launch(pl, "k_best_init", sb::k_best_init, dim3(div_up(b1, 256)), dim3(256), 0, b1,
                             pl->d_bsnr + c * sub_stride + b1, pl->d_bamp + c * sub_stride + b1,
                             pl->d_bidx + c * sub_stride + b1));
        } else {
            const long cnt_x = (long)(nsub - 1) * sub_stride;
            SB_OK(launch(pl, "k_best_init", sb::k_best_init, dim3(div_up(cnt_x, 256)), dim3(256), 0, cnt_x,
                         pl->d_bsnr + sub_stride, pl->d_bamp + sub_stride, pl->d_bidx + sub_stride));
        }
    }

    pl->last_geom[0] = Pym; pl->last_geom[1] = Pxm; pl->last_geom[2] = (int)ay.tiles.size();
    pl->last_geom[3] = (int)ax.tiles.size(); pl->last_geom[4] = Ba; pl->last_geom[5] = Bt;
    pl->last_fft_area = 0.0;

    const sb::Tmpl* d_tm = (const sb::Tmpl*)pl->tmpls.p;
    const sb::Angle* d_an = (const sb::Angle*)pl->angles.p;
    const long bn = pl->bn();
    const long boff = (long)pl->slab_lo * pl->nx;       // best planes are addressed by raster row

    for (auto& tyS : ay.tiles)
        for (auto& txS : ax.tiles) {
            const int Py = tyS.P, Px = txS.P;
            const int KX = Px / 2 + 1;
            const int kpitch = Px / 2 + 8;
            pl->last_fft_area += (double)Py * Px;
            const C2 *twy = nullptr, *twx = nullptr;
            SB_OK(twiddles<R>(pl, Py, &twy));
            SB_OK(twiddles<R>(pl, Px, &twx));
            sb::Geom g;
            g.ny = pl->ny; g.nx = pl->nx; g.Py = Py; g.Px = Px;
            fill_axis(ay, pl->ny, tyS, &g.oy, &g.out_ny, &g.split_y, &g.dly, &g.need_y_lo, &g.need_y_hi);
            fill_axis(ax, pl->nx, txS, &g.ox, &g.out_nx, &g.split_x, &g.dlx, &g.need_x_lo, &g.need_x_hi);
            g.kpitch = kpitch; g.syp = syp;
            g.dx = pl->dx; g.dx2 = pl->dx2; g.dy2 = pl->dy2;
            g.norm = 1.0 / ((double)Px * (double)Py);
            g.c2_scale = pl->c2_scale;
            g.poison = pl->dem_nonfinite ? 1 : 0;
            g.row0 = pl->row0; g.drows = pl->drows; g.brow0 = pl->slab_lo;
            const int need_rows = g.need_y_hi - g.need_y_lo + 1;
            g.rpitch = need_rows + (need_rows & 1);

            if (fast) {
                // the nine plane spectra of this tile, once: five packed row transforms, column transforms
                SB_OK(dispatch_n(Px, [&](auto nn) {
                    constexpr int N = decltype(nn)::value;
                    using S = Shape<N, float>;
                    auto kern = masked ? sb::k_diff_rows_fm<N> : sb::k_diff_rows_f<N>;
                    ProfScope prof(pl, K_CURV_ROWS);
                    return launch(pl, "k_diff_rows_f", kern, dim3(sb::kDiffPairs, div_up(div_up(need_rows, 2), S::GP)),
                                  dim3(S::threads), S::smem_conv_f, g, (const float4*)pl->d_diffs32, (float4*)pl->cr.p,
                                  (const float2*)twx);
                }));
                SB_OK(dispatch_n(Py, [&](auto nn) {
                    constexpr int N = decltype(nn)::value;
                    using S = Shape<N, float>;
                    ProfScope prof(pl, K_CURV_ROWS);
                    return launch(pl, "k_curv_cols", sb::k_curv_cols<N, float>, dim3(div_up(KX, S::GP), sb::kDiffPairs),
                                  dim3(S::threads), S::smem, g, (const float4*)pl->cr.p, (float2*)pl->spec9.p,
                                  (const float2*)twy);
                }));
                if (masked) {
                    const size_t plane = (size_t)KX * Py;       // float2 elements of one spectrum plane
                    const float2* fu = (const float2*)pl->spec9.p + (size_t)sb::kDiffPlanes * plane;
                    for (int f = 0; f < 2; ++f)
                        SB_TRY(sb_rt_d2d((float2*)pl->fct.p + (size_t)(2 * Ba + f) * plane, fu, plane * sizeof(float2),
                                         pl->stream));
                }
            }
            for (auto& ab : batches) {
                const int a0 = ab.a0, a1 = ab.a1;
                if (fast) {
                    const long n2 = (long)KX * Py / 2;
                    ProfScope prof(pl, K_CURV_COLS);
                    SB_OK(launch(pl, "k_combine_spectra", sb::k_combine_spectra, dim3(div_up(n2, 256)), dim3(256),
                                 (a1 - a0) * sizeof(sb::SpecCoef), n2, a1 - a0, a0, (const sb::SpecCoef*)pl->coef.p,
                                 (const float4*)pl->spec9.p, (float4*)pl->fct.p));
                } else {
                    SB_OK(dispatch_n(Px, [&](auto nn) {
                        constexpr int N = decltype(nn)::value;
                        using S = Shape<N, R>;
                        ProfScope prof(pl, K_CURV_ROWS);
                        return launch(pl, "k_curv_rows", sb::k_curv_rows<N, R>,
                                      dim3(a1 - a0, div_up(div_up(need_rows, 2), S::GP)), dim3(S::threads), S::smem, g,
                                      (const double*)pl->d_diffs, d_an, a0, (C4*)pl->cr.p, twx);
                    }));
                    SB_OK(dispatch_n(Py, [&](auto nn) {
                        constexpr int N = decltype(nn)::value;
                        using S = Shape<N, R>;
                        ProfScope prof(pl, K_CURV_COLS);
                        return launch(pl, "k_curv_cols", sb::k_curv_cols<N, R>, dim3(div_up(KX, S::GP), a1 - a0),
                                      dim3(S::threads), S::smem, g, (const C4*)pl->cr.p, (C2*)pl->fct.p, twy);
                    }));
                }
                for (auto& ch : ab.chunks) {
                    // the chunk's device records (a masked sweep: templates, then companions)
                    const int pb = ch.pb * rec_per_tmpl, cnt = ch.cnt * rec_per_tmpl;
                    SB_OK(dispatch_n(Px, [&](auto nn) {
                        constexpr int N = decltype(nn)::value;
                        using S = Shape<N, R>;
                        ProfScope prof(pl, K_TMPL_ROWS);
                        // narrow templates: two samples per thread (needs a radix-16 first stage)
                        const bool xsparse = N >= 256 && hi_x <= S::T - 1 && lo_x >= -S::T;
                        const int nt = ch.cnt;            // the templates; a masked sweep's companions follow
                        const dim3 grid(div_up(syp / 2, S::GP), nt);
                        auto kern = sb::k_tmpl_rows<N, R, false>;
                        if constexpr (N >= 256) {
                            if (xsparse) kern = sb::k_tmpl_rows<N, R, true>;
                        }
                        SB_OK(launch(pl, "k_tmpl_rows", kern, grid, dim3(S::threads), S::smem, g, d_tm, pb,
                                     (const double*)pl->d_x, (const double*)pl->d_y, (C4*)pl->trt.p,
                                     (double2*)pl->part.p, twx, (const double*)pl->tbox.p));
                        if constexpr (kF32) {
                            if (masked) {
                                // the companions: t**2, records pb + nt ..; trt / part slots nt ..
                                auto kern_sq = sb::k_tmpl_rows_sq<N, false>;
                                if constexpr (N >= 256) {
                                    if (xsparse) kern_sq = sb::k_tmpl_rows_sq<N, true>;
                                }
                                SB_OK(launch(pl, "k_tmpl_rows_sq", kern_sq, grid, dim3(S::threads), S::smem, g, d_tm,
                                             pb + nt, (const double*)pl->d_x, (const double*)pl->d_y,
                                             (float4*)pl->trt.p + (size_t)nt * (N / 2 + 1) * syp,
                                             (double2*)pl->part.p + (size_t)nt * syp, (const float2*)twx));
                            }
                        }
                        return 0;
                    }));
                    {
                        ProfScope prof(pl, K_TMPL_SUMS);
                        SB_OK(launch(pl, "k_tmpl_sums", sb::k_tmpl_sums, dim3(cnt), dim3(32), 32 * sizeof(double2), g,
                                     d_tm, pb, cnt, (const double2*)pl->part.p, (sb::TSum*)pl->sums.p,
                                     (sb::FitT*)pl->fit.p));
                        if (masked)
                            SB_OK(launch(pl, "k_mask_consts", sb::k_mask_consts, dim3(div_up(ch.cnt, 32)), dim3(32), 0,
                                         g, d_tm, pb, ch.cnt, pl->min_cov, (const sb::TSum*)pl->sums.p,
                                         (sb::FitM*)pl->fitm.p));
                    }
                    const bool fast_fit = fast && !so.raw_amp;
                    if constexpr (kF32) {
                        if (fast) {
                            SB_OK(dispatch_n(Py, [&](auto nn) {
                                constexpr int N = decltype(nn)::value;
                                using S = Shape<N, float>;
                                // every template column has at most two non-zero inputs per thread
                                const bool sparse = hi_y <= S::T - 1 && lo_y >= -S::T;
                                ProfScope prof(pl, K_CONV_COLS);
                                const bool persist = pl->conv_persist > 0 || (pl->conv_persist < 0 && max_per_angle >= 4);
                                if constexpr (N == sb64::N) {
                                    if (pl->conv_r64 && persist && cnt <= sb64::kConvRMaxBatch) {
                                        const float2* tw64 = nullptr;
                                        SB_OK(twiddles64(pl, &tw64));
                                        const bool sparse64 = hi_y <= 3 * sb64::R - 1 && lo_y >= -3 * sb64::R;
                                        auto kern = sparse64 ? sb64::k_conv_cols_r<true> : sb64::k_conv_cols_r<false>;
                                        return launch(pl, "k_conv_cols_r", kern, dim3(KX), dim3(sb64::kConvRThreads),
                                                      sb64::kConvRSmem, g, d_tm, pb, cnt, a0, (const float4*)pl->trt.p,
                                                      (const float2*)pl->fct.p, (float4*)pl->gbuf.p, tw64);
                                    }
                                }
                                if constexpr (N >= 1024 && N <= 4096) {
                                    if (persist && cnt <= sb::kConvPMaxBatch) {
                                        constexpr size_t smem_p =
                                            (size_t)(sb::kConvPThreads / S::T) * 2 * sbfft::padded_len(N) * sizeof(float2) +
                                            (size_t)2 * N * sizeof(float2) + sb::kConvPMaxBatch * 4 * sizeof(int) +
                                            (size_t)sbfft::ctw_count<float>(N) * sizeof(float2);
                                        auto kern = sparse ? sb::k_conv_cols_p<N, true> : sb::k_conv_cols_p<N, false>;
                                        return launch(pl, "k_conv_cols_p", kern, dim3(KX), dim3(sb::kConvPThreads),
                                                      smem_p, g, d_tm, pb, cnt, a0, (const float4*)pl->trt.p,
                                                      (const float2*)pl->fct.p, (float4*)pl->gbuf.p,
                                                      (const float2*)twy);
                                    }
                                }
                                auto kern = sparse ? sb::k_conv_cols_f<N, true> : sb::k_conv_cols_f<N, false>;
                                return launch(pl, "k_conv_cols_f", kern, dim3(cnt, div_up(KX, S::GP)), dim3(S::threads),
                                              S::smem_conv_f, g, d_tm, pb, a0, (const float4*)pl->trt.p,
                                              (const float2*)pl->fct.p, (float4*)pl->gbuf.p,
                                              (const float2*)twy);
                            }));
                        }
                    }
                    if (!fast) {
                        SB_OK(dispatch_n(Py, [&](auto nn) {
                            constexpr int N = decltype(nn)::value;
                            using S = Shape<N, R>;
                            ProfScope prof(pl, K_CONV_COLS);
                            return launch(pl, "k_conv_cols", sb::k_conv_cols<N, R>, dim3(div_up(KX, S::GP), cnt),
                                          dim3(S::threads), S::smem_conv, g, d_tm, pb, a0, (const C4*)pl->trt.p,
                                          (const C2*)pl->fct.p, (C4*)pl->gbuf.p, twy);
                        }));
                    }
                    // fold: one launch per best state present in the chunk
                    for (auto& gp : ch.groups) {
                        const int* d_slots = gp.off < 0 ? nullptr : (const int*)pl->slots.p + gp.off;
                        const int state = so.second ? 1 : gp.state;
                        float* bsnr = pl->d_bsnr + (long)state * bn - boff;
                        float* bamp = pl->d_bamp + (long)state * bn - boff;
                        int* bidx = pl->d_bidx + (long)state * bn - boff;
                        if constexpr (kF32) {
                            if (fast_fit) {
                                const int4* cross = gp.err ? (const int4*)pl->cross.p : (const int4*)nullptr;
                                SB_OK(dispatch_n(Px, [&](auto nn) {
                                    constexpr int N = decltype(nn)::value;
                                    using S = Shape<N, float>;
                                    ProfScope prof(pl, K_FIT_ROWS);
                                    const dim3 grid(div_up(Py / 2, S::GP), nsub);
                                    if (so.region) {
                                        if (masked) {
                                            if constexpr (N <= kMaxFftMasked) {
                                                return launch(pl, "k_fit_rows_gmr", sb::k_fit_rows_gmr<N>, grid,
                                                              dim3(S::threads),
                                                              S::smem_fit_f + sb::fit_masked_extra_smem<N>(), g,
                                                              gp.count, d_slots, (const sb::FitT*)pl->fit.p,
                                                              (const sb::FitM*)pl->fitm.p, ch.cnt,
                                                              (const float4*)pl->gbuf.p, (const float2*)twx, cross,
                                                              *so.region);
                                            }
                                            return fail("internal: masked fit at FFT length " + std::to_string(N));
                                        }
                                        return launch(pl, "k_fit_rows_gr", sb::k_fit_rows_gr<N>, grid, dim3(S::threads),
                                                      S::smem_fit_f, g, gp.count, d_slots, (const sb::FitT*)pl->fit.p,
                                                      (const float4*)pl->gbuf.p, (const float2*)twx, cross,
                                                      *so.region);
                                    }
                                    if (so.peak) {
                                        if (masked) {
                                            if constexpr (N <= kMaxFftMasked) {
                                                return launch(pl, "k_fit_rows_gmp", sb::k_fit_rows_gmp<N>, grid,
                                                              dim3(S::threads),
                                                              S::smem_fit_f + sb::fit_masked_extra_smem<N>(), g,
                                                              gp.count, d_slots, (const sb::FitT*)pl->fit.p,
                                                              (const sb::FitM*)pl->fitm.p, ch.cnt,
                                                              (const float4*)pl->gbuf.p, (const float2*)twx, cross,
                                                              *so.peak);
                                            }
                                            return fail("internal: masked fit at FFT length " + std::to_string(N));
                                        }
                                        return launch(pl, "k_fit_rows_gp", sb::k_fit_rows_gp<N>, grid, dim3(S::threads),
                                                      S::smem_fit_f, g, gp.count, d_slots, (const sb::FitT*)pl->fit.p,
                                                      (const float4*)pl->gbuf.p, (const float2*)twx, cross, *so.peak);
                                    }
                                    if (so.second) {
                                        if (masked) {
                                            if constexpr (N <= kMaxFftMasked) {
                                                return launch(pl, "k_fit_rows_gms", sb::k_fit_rows_gms<N>, grid,
                                                              dim3(S::threads),
                                                              S::smem_fit_f + sb::fit_masked_extra_smem<N>(), g,
                                                              gp.count, d_slots, (const sb::FitT*)pl->fit.p,
                                                              (const sb::FitM*)pl->fitm.p, ch.cnt,
                                                              (const float4*)pl->gbuf.p, bsnr, bamp, bidx,
                                                              (const float2*)twx, cross, sub_stride, *so.second);
                                            }
                                            return fail("internal: masked fit at FFT length " + std::to_string(N));
                                        }
                                        return launch(pl, "k_fit_rows_gs", sb::k_fit_rows_gs<N>, grid, dim3(S::threads),
                                                      S::smem_fit_f, g, gp.count, d_slots, (const sb::FitT*)pl->fit.p,
                                                      (const float4*)pl->gbuf.p, bsnr, bamp, bidx, (const float2*)twx,
                                                      cross, sub_stride, *so.second);
                                    }
                                    if (masked) {
                                        // FFT lengths <= 4096 only: the park buffers need 2 N float2 per group
                                        if constexpr (N <= kMaxFftMasked) {
                                            return launch(pl, "k_fit_rows_gm", sb::k_fit_rows_gm<N>, grid,
                                                          dim3(S::threads),
                                                          S::smem_fit_f + sb::fit_masked_extra_smem<N>(), g,
                                                          gp.count, d_slots, (const sb::FitT*)pl->fit.p,
                                                          (const sb::FitM*)pl->fitm.p, ch.cnt,
                                                          (const float4*)pl->gbuf.p, bsnr, bamp, bidx,
                                                          (const float2*)twx, cross, sub_stride);
                                        }
                                        return fail("internal: masked fit at FFT length " + std::to_string(N));
                                    }
                                    // (a variant without the get_err_mask members spills MORE: 564 bytes against 312)
                                    return launch(pl, "k_fit_rows_g", sb::k_fit_rows_g<N>, grid, dim3(S::threads),
                                                  S::smem_fit_f, g, gp.count, d_slots, (const sb::FitT*)pl->fit.p,
                                                  (const float4*)pl->gbuf.p, bsnr, bamp, bidx, (const float2*)twx,
                                                  cross, sub_stride);
                                }));
                                if (g.poison && !reads_best)
                                    SB_OK(launch(pl, "k_poison_windows", sb::k_poison_windows,
                                                 dim3(div_up((long)g.out_ny * g.out_nx, 256)), dim3(256), 0, g,
                                                 gp.count, d_slots, (const sb::FitT*)pl->fit.p, bsnr));
                                continue;
                            }
                        }
                        sb::FitOut fo;
                        fo.best_snr = bsnr; fo.best_amp = bamp; fo.best_idx = bidx;
                        fo.raw_amp = so.raw_amp; fo.raw_snr = so.raw_snr;
                        SB_OK(dispatch_n(Px, [&](auto nn) {
                            constexpr int N = decltype(nn)::value;
                            using S = Shape<N, R>;
                            ProfScope prof(pl, K_FIT_ROWS);
                            return launch(pl, "k_fit_rows", sb::k_fit_rows<N, R>, dim3(div_up(g.out_ny, S::GP)),
                                          dim3(S::threads), S::smem, g, d_tm, pb, gp.count, d_slots,
                                          (const sb::TSum*)pl->sums.p, (const C4*)pl->gbuf.p, (const double*)pl->d_x,
                                          (const double*)pl->d_y, fo, twx);
                        }));
                    }
                }
            }
        }
    // a secondary sweep folds and clears best state 1 alone
    const long st_off = so.second ? bn : 0, st_len = so.second ? bn : sub_stride;
    if (nsub > 1 && !reads_best) {
        SB_OK(launch(pl, "k_best_fold", sb::k_best_fold, dim3(div_up(st_len, 256)), dim3(256), 0, st_len,
                     nsub - 1, sub_stride, (const float*)pl->d_bsnr + sub_stride + st_off,
                     (const float*)pl->d_bamp + sub_stride + st_off, (const int*)pl->d_bidx + sub_stride + st_off,
                     pl->d_bsnr + st_off, pl->d_bamp + st_off, pl->d_bidx + st_off));
    }
    if (masked && !reads_best) {
        SB_OK(launch(pl, "k_best_clear_nodata", sb::k_best_clear_nodata, dim3(div_up(bn, 256)), dim3(256), 0, pl->ny,
                     pl->nx, pl->row0, pl->slab_lo, (int)pl->brows(), so.second ? 1 : pl->n_states, bn,
                     (const double*)pl->d_dem, pl->d_bsnr + st_off, pl->d_bamp + st_off, pl->d_bidx + st_off));
    }
    drain_profile(pl);
    return 0;
}

int run_sweep(sb_plan* pl, const sb_angle* angles, int n_angles, const sb_template* tmpls_in, int n_tmpls,
              SweepOut so, const int32_t* hint = nullptr) {
    if (pl->precision == 64) return run_sweep_t<double>(pl, angles, n_angles, tmpls_in, n_tmpls, so, hint);
    return run_sweep_t<float>(pl, angles, n_angles, tmpls_in, n_tmpls, so, hint);
}

int copy_out(sb_plan* pl, double* dst, const double* src_dev, size_t count, int out_is_device) {
    if (out_is_device)
        SB_TRY(sb_rt_d2d(dst, src_dev, count * sizeof(double), pl->stream));
    else
        SB_TRY(sb_rt_d2h(dst, src_dev, count * sizeof(double), pl->stream));
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

}  // namespace

extern "C" {

const char* sb_last_error(void) { return g_err.c_str(); }

#ifndef SB_SOURCE_HASH
#define SB_SOURCE_HASH "unhashed"
#endif

const char* sb_build_info(void) {
#ifdef SB_EMU
    return "cpu-emulator (test infrastructure)";
#else
    return "cuda sm_100a " SB_SOURCE_HASH;
#endif
}

int sb_plan_create(sb_plan** plan, int ny, int nx, double dx, double dx2, double dy2, int device,
                   void* stream, unsigned flags) {
    (void)flags;
    if (!plan || ny < 1 || nx < 1) return fail("sb_plan_create: bad arguments");
    sb_plan* pl = new sb_plan();
    pl->ny = ny; pl->nx = nx; pl->dx = dx; pl->dx2 = dx2; pl->dy2 = dy2;
    pl->slab_lo = 0; pl->slab_hi = ny; pl->row0 = 0; pl->drows = ny;
#ifndef SB_EMU
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        delete pl;
        return fail("no CUDA device available: scarplet_b200 has no CPU path");
    }
    if (device >= 0) {
        if (cudaSetDevice(device) != cudaSuccess) { delete pl; return fail("cudaSetDevice failed"); }
    }
    cudaGetDevice(&pl->device);
    if (stream) {
        pl->stream = (cudaStream_t)stream;
    } else {
        if (cudaStreamCreateWithFlags(&pl->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete pl;
            return fail("cudaStreamCreate failed");
        }
        pl->own_stream = true;
    }
#else
    (void)device; (void)stream;
#endif
    if (alloc_best(pl) != 0) { sb_plan_destroy(pl); return fail("sb_plan_create: out of device memory"); }
    *plan = pl;
    return 0;
}

int sb_plan_destroy(sb_plan* pl) {
    if (!pl) return 0;
#ifndef SB_EMU
    cudaSetDevice(pl->device);
#endif
    sb_rt_sync(pl->stream);
    if (pl->own_dem && pl->d_dem) sb_rt_free(pl->d_dem);
    if (pl->d_diffs) sb_rt_free(pl->d_diffs);
    if (pl->d_diffs32) sb_rt_free(pl->d_diffs32);
    if (pl->d_x) sb_rt_free(pl->d_x);
    if (pl->d_y) sb_rt_free(pl->d_y);
    if (pl->d_bsnr) sb_rt_free(pl->d_bsnr);
    if (pl->d_bamp) sb_rt_free(pl->d_bamp);
    if (pl->d_bidx) sb_rt_free(pl->d_bidx);
    for (auto& kv : pl->tw) sb_rt_free(kv.second);
    for (auto e : pl->ev_pool) sb_rt_event_destroy(e);
    for (Buf* b : {&pl->cr, &pl->fct, &pl->trt, &pl->part, &pl->gbuf, &pl->sums, &pl->fit, &pl->tmpls, &pl->angles,
                   &pl->tables, &pl->raw, &pl->tbox, &pl->slots, &pl->cross, &pl->casa, &pl->aux, &pl->spec9, &pl->coef,
                   &pl->fitm, &pl->fs_idx, &pl->fs_out, &pl->region, &pl->rtab, &pl->spos, &pl->peak})
        release(*b);
#ifndef SB_EMU
    if (pl->own_stream) cudaStreamDestroy(pl->stream);
#endif
    delete pl;
    return 0;
}

int sb_plan_set_option(sb_plan* pl, const char* key, long value) {
    if (!pl || !key) return fail("sb_plan_set_option: null");
    std::string k(key);
    if (k == "workspace_mb") { pl->workspace_mb = value <= 0 ? 0 : std::max(64L, value); return 0; }
    if (k == "max_fft") {
        if (!is_pow2((int)value) || value < kMinFft || value > kMaxFftSupported)
            return fail("max_fft must be a power of two in [128, 8192]");
        pl->max_fft = (int)value;
        return 0;
    }
    if (k == "force_pad") { pl->force_pad = value != 0; return 0; }
    if (k == "mixed_tiles") { pl->mixed_tiles = value != 0; return 0; }
    if (k == "profile") { pl->profile = value != 0; return 0; }
    if (k == "fast") { pl->fast = value != 0; return 0; }
    if (k == "conv_persist") { pl->conv_persist = (int)value; return 0; }
    if (k == "conv_r64") { pl->conv_r64 = value != 0; return 0; }
    if (k == "fit_substreams") { pl->fit_substreams = (int)std::max(0L, std::min(8L, value)); return 0; }
    if (k == "precision") {
        if (value != 32 && value != 64) return fail("precision must be 32 or 64");
        pl->precision = (int)value;
        return 0;
    }
    if (k == "states") {
        if (value < 1 || value > 64) return fail("states must be in [1, 64]");
        if ((int)value != pl->n_states) {
            pl->n_states = (int)value;
            return alloc_best(pl);
        }
        return 0;
    }
    return fail("unknown option " + k);
}

int sb_plan_set_nodata(sb_plan* pl, int mode, double min_coverage) {
    if (!pl) return fail("null plan");
    if (mode != SB_NODATA_PROPAGATE && mode != SB_NODATA_MASK)
        return fail("sb_plan_set_nodata: mode must be SB_NODATA_PROPAGATE or SB_NODATA_MASK");
    if (!(min_coverage > 0.0 && min_coverage <= 1.0)) return fail("sb_plan_set_nodata: min_coverage must be in (0, 1]");
    if (mode == SB_NODATA_MASK && pl->precision != 32)
        return fail("sb_plan_set_nodata: the nodata mask needs precision 32 (the complex64 pipeline)");
    if (mode == SB_NODATA_MASK && !pl->fast)
        return fail("sb_plan_set_nodata: the nodata mask needs the pipelined kernels (option fast = 1)");
    pl->nodata_req = mode;
    pl->min_cov_req = min_coverage;
    return 0;
}

int sb_plan_set_slab(sb_plan* pl, int row_lo, int row_hi, int halo) {
    if (!pl) return fail("null plan");
    if (row_lo < 0 || row_hi > pl->ny || row_lo >= row_hi || halo < 0) return fail("sb_plan_set_slab: bad rows");
    if (pl->d_dem && pl->own_dem) { sb_rt_free(pl->d_dem); }
    pl->d_dem = nullptr; pl->own_dem = false;
    if (pl->d_diffs) { sb_rt_free(pl->d_diffs); pl->d_diffs = nullptr; }
    if (pl->d_diffs32) { sb_rt_free(pl->d_diffs32); pl->d_diffs32 = nullptr; }
    pl->diffs64_valid = false;
    pl->slab_lo = row_lo; pl->slab_hi = row_hi;
    const long rows = (long)(row_hi - row_lo) + 2L * halo;
    if (rows >= pl->ny) { pl->row0 = 0; pl->drows = pl->ny; }
    else { pl->row0 = ((row_lo - halo) % pl->ny + pl->ny) % pl->ny; pl->drows = (int)rows; }
    return alloc_best(pl);
}

int sb_plan_dem_rows(const sb_plan* pl, int* row0, int* drows) {
    if (!pl) return fail("null plan");
    if (row0) *row0 = pl->row0;
    if (drows) *drows = pl->drows;
    return 0;
}

int sb_plan_curv_stats(const sb_plan* pl, double* sumsq, double* count) {
    if (!pl) return fail("null plan");
    if (sumsq) *sumsq = pl->curv_sumsq;
    if (count) *count = pl->curv_count;
    return 0;
}

int sb_plan_set_curv_stats(sb_plan* pl, double sumsq, double count) {
    if (!pl) return fail("null plan");
    apply_curv_stats(pl, sumsq, count);
    return 0;
}

void* sb_plan_stream(const sb_plan* pl) { return pl ? (void*)pl->stream : nullptr; }

long sb_plan_launch_count(const sb_plan* pl) { return pl ? pl->launches : 0; }

long sb_plan_device_bytes(const sb_plan* pl) {
    if (!pl) return 0;
    size_t b = 0;
    const size_t n = (size_t)pl->drows * pl->nx;
    if (pl->d_dem && pl->own_dem) b += n * sizeof(double);
    if (pl->d_diffs) b += n * 3 * sizeof(double);
    if (pl->d_diffs32) b += n * sizeof(float4);
    b += (size_t)pl->bn() * pl->n_states * pl->best_copies * 12;
    for (const Buf* q : {&pl->cr, &pl->fct, &pl->trt, &pl->part, &pl->gbuf, &pl->sums, &pl->fit, &pl->tmpls, &pl->angles,
                         &pl->tables, &pl->raw, &pl->tbox, &pl->slots, &pl->cross, &pl->casa, &pl->aux, &pl->spec9, &pl->coef,
                         &pl->fitm, &pl->fs_idx, &pl->fs_out, &pl->region, &pl->rtab, &pl->spos, &pl->peak})
        b += q->cap;
    return (long)b;
}

int sb_plan_profile(sb_plan* pl, double* ms6, long* launches6, int reset) {
    if (!pl) return fail("null plan");
    drain_profile(pl);
    for (int i = 0; i < 6; ++i) {
        if (ms6) ms6[i] = pl->prof_ms[i];
        if (launches6) launches6[i] = pl->prof_n[i];
        if (reset) { pl->prof_ms[i] = 0; pl->prof_n[i] = 0; }
    }
    return 0;
}

int sb_plan_last_geometry(const sb_plan* pl, int* out6) {
    if (!pl || !out6) return fail("null");
    for (int i = 0; i < 6; ++i) out6[i] = pl->last_geom[i];
    return 0;
}

double sb_plan_last_fft_area(const sb_plan* pl) { return pl ? pl->last_fft_area : 0.0; }

int sb_set_dem_host(sb_plan* pl, const double* dem_host) {
    if (!pl || !dem_host) return fail("sb_set_dem_host: null");
    const size_t bytes = (size_t)pl->drows * pl->nx * sizeof(double);
    if (!pl->own_dem || !pl->d_dem) {
        pl->d_dem = nullptr;
        SB_TRY(sb_rt_malloc((void**)&pl->d_dem, bytes));
        pl->own_dem = true;
    }
    SB_TRY(sb_rt_h2d(pl->d_dem, dem_host, bytes, pl->stream));
    SB_TRY(sb_rt_sync(pl->stream));
    return after_dem(pl);
}

int sb_set_dem_dev(sb_plan* pl, const double* dem_dev) {
    if (!pl || !dem_dev) return fail("sb_set_dem_dev: null");
    if (pl->own_dem && pl->d_dem) sb_rt_free(pl->d_dem);
    pl->own_dem = false;
    pl->d_dem = const_cast<double*>(dem_dev);
    return after_dem(pl);
}

int sb_set_axes_host(sb_plan* pl, const double* x_host, const double* y_host) {
    if (!pl || !x_host || !y_host) return fail("sb_set_axes_host: null");
    if (!pl->d_x) SB_TRY(sb_rt_malloc((void**)&pl->d_x, (size_t)pl->nx * sizeof(double)));
    if (!pl->d_y) SB_TRY(sb_rt_malloc((void**)&pl->d_y, (size_t)pl->ny * sizeof(double)));
    SB_TRY(sb_rt_h2d(pl->d_x, x_host, (size_t)pl->nx * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(pl->d_y, y_host, (size_t)pl->ny * sizeof(double), pl->stream));
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_directional_laplacian(sb_plan* pl, const sb_angle* angle, double* out, int out_is_device) {
    if (!pl || !angle || !out) return fail("sb_directional_laplacian: null");
    if (!pl->d_dem) return fail("no DEM set");
    if (!pl->whole()) return fail("sb_directional_laplacian needs a plan over the whole raster");
    const long n = (long)pl->ny * pl->nx;
    double* dst = out;
    if (!out_is_device) {
        SB_OK(ensure(pl->raw, (size_t)n * 2 * sizeof(double)));
        dst = (double*)pl->raw.p;
    }
    sb::Angle a;
    a.ca = angle->cos_a; a.sa = angle->sin_a; a.ca2 = angle->cos2_a; a.sa2 = angle->sin2_a;
    SB_OK(launch(pl, "k_laplacian", sb::k_laplacian, dim3(div_up(n, 256)), dim3(256), 0, pl->ny, pl->nx,
                 (const double*)pl->d_dem, pl->dx, pl->dx2, pl->dy2, a, dst));
    if (!out_is_device) return copy_out(pl, out, dst, (size_t)n, 0);
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_render_template(sb_plan* pl, const sb_template* tmpl, double* out, int out_is_device) {
    if (!pl || !tmpl || !out) return fail("sb_render_template: null");
    if (!pl->d_x || !pl->d_y) return fail("no axis vectors set");
    const long n = (long)pl->ny * pl->nx;
    double* dst = out;
    if (!out_is_device) {
        SB_OK(ensure(pl->raw, (size_t)n * 2 * sizeof(double)));
        dst = (double*)pl->raw.p;
    }
    sb::Tmpl t;
    std::memcpy(&t, tmpl, sizeof(t));
    SB_OK(launch(pl, "k_render_template", sb::k_render_template, dim3(div_up(n, 256)), dim3(256), 0, pl->ny, pl->nx, t,
                 (const double*)pl->d_x, (const double*)pl->d_y, dst));
    if (!out_is_device) return copy_out(pl, out, dst, (size_t)n, 0);
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_match_template(sb_plan* pl, const sb_angle* angle, const sb_template* tmpl, double* amp, double* snr,
                      int out_is_device) {
    if (!pl || !angle || !tmpl || !amp || !snr) return fail("sb_match_template: null");
    if (pl->nodata == SB_NODATA_MASK || pl->nodata_req == SB_NODATA_MASK)
        return fail("nodata mask: sb_match_template keeps the reference's NaN semantics");
    const size_t n = (size_t)pl->ny * pl->nx;
    SweepOut so;
    if (out_is_device) {
        so.raw_amp = amp;
        so.raw_snr = snr;
    } else {
        SB_OK(ensure(pl->raw, n * 2 * sizeof(double)));
        so.raw_amp = (double*)pl->raw.p;
        so.raw_snr = so.raw_amp + n;
    }
    sb_template t = *tmpl;
    t.angle_id = 0;
    t.state = 0;
    SB_OK(run_sweep(pl, angle, 1, &t, 1, so));
    if (!out_is_device) {
        SB_TRY(sb_rt_d2h(amp, so.raw_amp, n * sizeof(double), pl->stream));
        SB_TRY(sb_rt_d2h(snr, so.raw_snr, n * sizeof(double), pl->stream));
    }
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_match_template_raster(sb_plan* pl, const sb_angle* angle, const double* box_host, int sy_lo, int sy_hi,
                             int sx_lo, int sx_hi, double tscale, double* amp, double* snr, int out_is_device) {
    if (!pl || !angle || !box_host || !amp || !snr) return fail("sb_match_template_raster: null");
    if (sy_hi < sy_lo || sx_hi < sx_lo) return fail("sb_match_template_raster: empty box");
    const size_t cells = (size_t)(sy_hi - sy_lo + 1) * (size_t)(sx_hi - sx_lo + 1);
    SB_OK(ensure(pl->tbox, cells * sizeof(double)));
    SB_TRY(sb_rt_h2d(pl->tbox.p, box_host, cells * sizeof(double), pl->stream));
    sb_template t;
    std::memset(&t, 0, sizeof(t));
    t.cos_t = 1.0;
    t.sign = 1.0;
    t.tscale = tscale > 0.0 ? tscale : 1.0;
    t.kind = SB_KIND_RASTER;
    t.errmode = SB_ERRMASK_NONE;
    t.sy_lo = sy_lo; t.sy_hi = sy_hi; t.sx_lo = sx_lo; t.sx_hi = sx_hi;
    t.i_lo = 0; t.i_hi = pl->ny - 1; t.j_lo = 0; t.j_hi = pl->nx - 1;     // masks are the caller's
    return sb_match_template(pl, angle, &t, amp, snr, out_is_device);
}

int sb_fit_surface(sb_plan* pl, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                   const int32_t* rows_host, const int32_t* cols_host, int n_pix, double* amp, double* snr,
                   int out_is_device) {
    if (!pl || !angles || !tmpls || (n_pix > 0 && (!rows_host || !cols_host || !amp || !snr)))
        return fail("sb_fit_surface: null");
    if (!pl->d_dem) return fail("sb_fit_surface: no DEM set (sb_set_dem_host / sb_set_dem_dev)");
    if (!pl->d_x || !pl->d_y) return fail("sb_fit_surface: no axis vectors set (sb_set_axes_host)");
    if (n_angles <= 0 || n_tmpls <= 0 || n_pix < 0) return fail("sb_fit_surface: bad counts");
    int lo_y = 0, hi_y = 0;
    for (int k = 0; k < n_tmpls; ++k) {
        const sb_template& t = tmpls[k];
        if (t.kind != SB_KIND_SCARP && t.kind != SB_KIND_RICKER)
            return fail("sb_fit_surface: template " + std::to_string(k) +
                        " has no on-device generator (raster / plugin templates are not supported)");
        if (t.angle_id < 0 || t.angle_id >= n_angles) return fail("sb_fit_surface: template angle_id out of range");
        if (t.sy_hi < t.sy_lo || t.sx_hi < t.sx_lo) return fail("sb_fit_surface: empty template support box");
        if (t.sy_lo < -(pl->ny / 2) || t.sy_hi > pl->ny - 1 - pl->ny / 2 || t.sx_lo < -(pl->nx / 2) ||
            t.sx_hi > pl->nx - 1 - pl->nx / 2)
            return fail("sb_fit_surface: template support box exceeds the raster");
        lo_y = std::min(lo_y, t.sy_lo);
        hi_y = std::max(hi_y, t.sy_hi);
    }
    // pixels: the plan's own rows; on a row slab the curvature rows (+ 1 for the stencil) of every
    // template must lie inside the DEM rows the plan holds (as run_sweep_t requires of its tiles)
    const long have_lo = (long)pl->slab_lo - (pl->slab_lo - pl->row0 + (pl->slab_lo < pl->row0 ? pl->ny : 0));
    for (int q = 0; q < n_pix; ++q) {
        const int r = rows_host[q], c = cols_host[q];
        if (c < 0 || c >= pl->nx || r < pl->slab_lo || r >= pl->slab_hi)
            return fail("sb_fit_surface: pixel " + std::to_string(q) + " (" + std::to_string(r) + ", " +
                        std::to_string(c) + ") outside rows " + std::to_string(pl->slab_lo) + ".." +
                        std::to_string(pl->slab_hi - 1) + " / columns 0.." + std::to_string(pl->nx - 1) + " of the plan");
        const long first = (long)r + (pl->ny & 1) - hi_y - 1, last = (long)r + (pl->ny & 1) - lo_y + 1;
        if (pl->drows < pl->ny && (first < have_lo || last >= have_lo + pl->drows))
            return fail("row slab: halo too small for the template support (pixel row " + std::to_string(r) +
                        " needs rows " + std::to_string(first) + ".." + std::to_string(last) + ", have " +
                        std::to_string(have_lo) + ".." + std::to_string(have_lo + pl->drows - 1) + ")");
    }
    if (n_pix == 0) return 0;

    // jobs: up to kFsAges templates of one angle (caller order within the angle), with the union of their boxes
    std::vector<int> order(n_tmpls);
    for (int k = 0; k < n_tmpls; ++k) order[k] = k;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return tmpls[a].angle_id < tmpls[b].angle_id; });
    std::vector<sb::FsJob> jobs;
    for (int s = 0; s < n_tmpls;) {
        int e = s + 1;
        while (e < n_tmpls && e - s < sb::kFsAges && tmpls[order[e]].angle_id == tmpls[order[s]].angle_id) ++e;
        int y0 = tmpls[order[s]].sy_lo, y1 = tmpls[order[s]].sy_hi, x0 = tmpls[order[s]].sx_lo, x1 = tmpls[order[s]].sx_hi;
        for (int k = s + 1; k < e; ++k) {
            const sb_template& t = tmpls[order[k]];
            y0 = std::min(y0, t.sy_lo); y1 = std::max(y1, t.sy_hi);
            x0 = std::min(x0, t.sx_lo); x1 = std::max(x1, t.sx_hi);
        }
        const long cells = (long)(y1 - y0 + 1) * (x1 - x0 + 1);
        if (cells > 0x7fffffffL) return fail("sb_fit_surface: template support box too large");
        jobs.push_back({s, e - s, y0, x0, x1 - x0 + 1, (int)cells});
        s = e;
    }
    const int n_jobs = (int)jobs.size();
    const size_t jobs_b = jobs.size() * sizeof(sb::FsJob), ints_b = sizeof(int32_t) * ((size_t)n_tmpls + 2 * (size_t)n_pix);
    SB_OK(ensure(pl->fs_idx, jobs_b + ints_b));
    SB_OK(ensure(pl->tmpls, (size_t)n_tmpls * sizeof(sb::Tmpl)));
    SB_OK(ensure(pl->angles, (size_t)n_angles * sizeof(sb::Angle)));
    char* base = (char*)pl->fs_idx.p;
    const sb::FsJob* d_jobs = (const sb::FsJob*)base;
    const int* d_order = (const int*)(base + jobs_b);
    const int* d_rows = d_order + n_tmpls;
    const int* d_cols = d_rows + n_pix;
    SB_TRY(sb_rt_h2d(base, jobs.data(), jobs_b, pl->stream));
    SB_TRY(sb_rt_h2d((void*)d_order, order.data(), (size_t)n_tmpls * sizeof(int), pl->stream));
    SB_TRY(sb_rt_h2d((void*)d_rows, rows_host, (size_t)n_pix * sizeof(int32_t), pl->stream));
    SB_TRY(sb_rt_h2d((void*)d_cols, cols_host, (size_t)n_pix * sizeof(int32_t), pl->stream));
    SB_TRY(sb_rt_h2d(pl->tmpls.p, tmpls, (size_t)n_tmpls * sizeof(sb::Tmpl), pl->stream));
    SB_TRY(sb_rt_h2d(pl->angles.p, angles, (size_t)n_angles * sizeof(sb::Angle), pl->stream));
    SB_OK(ensure_diffs64(pl));

    // pixel chunks: at most 256 MB of output per launch (2 doubles per pixel and template)
    long chunk = ((256L << 20) / (16L * n_tmpls)) / sb::kFsPix * sb::kFsPix;
    chunk = std::max<long>(sb::kFsPix, std::min<long>(chunk, 1L << 20));
    if (!out_is_device) SB_OK(ensure(pl->fs_out, (size_t)std::min<long>(chunk, n_pix) * n_tmpls * 2 * sizeof(double)));
    const bool masked = pl->nodata == SB_NODATA_MASK;
    auto kern = masked ? sb::k_fit_surface<true> : sb::k_fit_surface<false>;
    for (long p0 = 0; p0 < n_pix; p0 += chunk) {
        const int cnt = (int)std::min<long>(chunk, n_pix - p0);
        const size_t off = (size_t)p0 * n_tmpls, vals = (size_t)cnt * n_tmpls;
        double* d_amp = out_is_device ? amp + off : (double*)pl->fs_out.p;
        double* d_snr = out_is_device ? snr + off : d_amp + vals;
        SB_OK(launch(pl, "k_fit_surface", kern, dim3(n_jobs, div_up(cnt, sb::kFsPix)), dim3(sb::kFsAges * sb::kFsPix),
                     sb::kFsSmem, pl->ny, pl->nx, pl->row0, pl->drows, (const double*)pl->d_diffs,
                     (const double*)pl->d_dem, (const sb::Angle*)pl->angles.p, (const sb::Tmpl*)pl->tmpls.p, d_order,
                     d_jobs, n_tmpls, d_rows + p0, d_cols + p0, cnt, (const double*)pl->d_x, (const double*)pl->d_y,
                     pl->dem_nonfinite ? 1 : 0, pl->min_cov, d_amp, d_snr));
        if (!out_is_device) {
            SB_TRY(sb_rt_d2h(amp + off, d_amp, vals * sizeof(double), pl->stream));
            SB_TRY(sb_rt_d2h(snr + off, d_snr, vals * sizeof(double), pl->stream));
        }
    }
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_best_reset(sb_plan* pl) {
    if (!pl) return fail("null plan");
    const long n = pl->bn() * pl->n_states;
    return launch(pl, "k_best_init", sb::k_best_init, dim3(div_up(n, 256)), dim3(256), 0, n, pl->d_bsnr, pl->d_bamp,
                  pl->d_bidx);
}

int sb_sweep(sb_plan* pl, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls) {
    if (!pl || !angles || !tmpls) return fail("sb_sweep: null");
    return run_sweep(pl, angles, n_angles, tmpls, n_tmpls, SweepOut());
}

int sb_sweep_ex(sb_plan* pl, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                const int32_t* whole_search5) {
    if (!pl || !angles || !tmpls) return fail("sb_sweep_ex: null");
    return run_sweep(pl, angles, n_angles, tmpls, n_tmpls, SweepOut(), whole_search5);
}

int sb_finalize_ex(sb_plan* pl, int state, int row_lo, int row_hi, const double* age_of_host,
                   const double* angle_of_host, int n_idx, double* out4, int out_is_device) {
    if (!pl || !age_of_host || !angle_of_host || !out4 || n_idx <= 0) return fail("sb_finalize: bad arguments");
    if (state < 0 || state >= pl->n_states) return fail("sb_finalize: state out of range");
    if (row_lo < pl->slab_lo || row_hi > pl->slab_hi || row_lo >= row_hi) return fail("sb_finalize: rows outside the plan");
    const long n = (long)(row_hi - row_lo) * pl->nx;
    const long off = (long)state * pl->bn() + (long)(row_lo - pl->slab_lo) * pl->nx;
    SB_OK(ensure(pl->tables, (size_t)2 * n_idx * sizeof(double)));
    double* d_age = (double*)pl->tables.p;
    double* d_ang = d_age + n_idx;
    SB_TRY(sb_rt_h2d(d_age, age_of_host, (size_t)n_idx * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d_ang, angle_of_host, (size_t)n_idx * sizeof(double), pl->stream));
    double* dst = out4;
    if (!out_is_device) {
        SB_OK(ensure(pl->raw, (size_t)n * 4 * sizeof(double)));
        dst = (double*)pl->raw.p;
    }
    SB_OK(launch(pl, "k_finalize", sb::k_finalize, dim3(div_up(n, 256)), dim3(256), 0, n,
                 (const float*)pl->d_bsnr + off, (const float*)pl->d_bamp + off, (const int*)pl->d_bidx + off,
                 (const double*)d_age, (const double*)d_ang, n_idx, dst));
    if (!out_is_device) return copy_out(pl, out4, dst, (size_t)n * 4, 0);
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_age_range(sb_plan* pl, int n_states, int row_lo, int row_hi, double snr_ratio, const double* age_of_host,
                 const double* angle_of_host, int n_idx, double* out6, int out_is_device) {
    if (!pl || !age_of_host || !angle_of_host || !out6 || n_idx <= 0) return fail("sb_age_range: bad arguments");
    if (!(snr_ratio > 0.0 && snr_ratio <= 1.0)) return fail("sb_age_range: snr_ratio must be in (0, 1]");
    if (n_states < 1 || n_states > pl->n_states) return fail("sb_age_range: n_states outside 1 .. option \"states\"");
    if (row_lo < pl->slab_lo || row_hi > pl->slab_hi || row_lo >= row_hi) return fail("sb_age_range: rows outside the plan");
    const long n = (long)(row_hi - row_lo) * pl->nx;
    const long off = (long)(row_lo - pl->slab_lo) * pl->nx;
    SB_OK(ensure(pl->tables, (size_t)2 * n_idx * sizeof(double)));
    double* d_age = (double*)pl->tables.p;
    double* d_ang = d_age + n_idx;
    SB_TRY(sb_rt_h2d(d_age, age_of_host, (size_t)n_idx * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d_ang, angle_of_host, (size_t)n_idx * sizeof(double), pl->stream));
    double* dst = out6;
    if (!out_is_device) {
        SB_OK(ensure(pl->raw, (size_t)n * 6 * sizeof(double)));
        dst = (double*)pl->raw.p;
    }
    SB_OK(launch(pl, "k_age_range", sb::k_age_range, dim3(div_up(n, 256)), dim3(256), 0, n, pl->bn(), n_states,
                 (const float*)pl->d_bsnr + off, (const float*)pl->d_bamp + off, (const int*)pl->d_bidx + off,
                 (const double*)d_age, (const double*)d_ang, n_idx, snr_ratio, dst));
    if (!out_is_device) return copy_out(pl, out6, dst, (size_t)n * 6, 0);
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_region_sweep(sb_plan* pl, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                    const int32_t* whole_search5, double snr_ratio, const int32_t* age_rank_host,
                    const int32_t* angle_pos_host, int n_idx, int n_pos) {
    if (!pl || !angles || !tmpls || !age_rank_host || !angle_pos_host || n_idx <= 0)
        return fail("sb_region_sweep: bad arguments");
    if (!(snr_ratio > 0.0 && snr_ratio <= 1.0)) return fail("sb_region_sweep: snr_ratio must be in (0, 1]");
    if (n_pos < 1 || n_pos > 256) return fail("sb_region_sweep: n_pos must be in 1 .. 256");
    if (pl->precision != 32 || !pl->fast) return fail("sb_region_sweep: fit region needs precision 32 and the option fast");
    int n_ranks = 0;
    for (int k = 0; k < n_idx; ++k) {
        if (age_rank_host[k] < 0 || angle_pos_host[k] < 0 || angle_pos_host[k] >= n_pos)
            return fail("sb_region_sweep: age rank or orientation position out of range at flat index " + std::to_string(k));
        n_ranks = std::max(n_ranks, age_rank_host[k] + 1);
    }
    for (int k = 0; k < n_tmpls; ++k)
        if (tmpls[k].idx < 0 || tmpls[k].idx >= n_idx)
            return fail("sb_region_sweep: template flat index outside 0 .. n_idx - 1");
    const int words = (n_pos + 31) / 32;
    const long bn = pl->bn(), boff = (long)pl->slab_lo * pl->nx;
    SB_OK(ensure(pl->region, (size_t)(3 + words) * bn * sizeof(int)));
    SB_OK(ensure(pl->rtab, (size_t)2 * n_idx * sizeof(int32_t)));
    int* planes = (int*)pl->region.p;
    int* tab = (int*)pl->rtab.p;
    SB_TRY(sb_rt_h2d(tab, age_rank_host, (size_t)n_idx * sizeof(int32_t), pl->stream));
    SB_TRY(sb_rt_h2d(tab + n_idx, angle_pos_host, (size_t)n_idx * sizeof(int32_t), pl->stream));
    // count 0, rank_lo 0x7f7f7f7f (above every rank), rank_hi -1, no orientation bits
    SB_TRY(sb_rt_memset(planes, 0, (size_t)bn * sizeof(int), pl->stream));
    SB_TRY(sb_rt_memset(planes + bn, 0x7f, (size_t)bn * sizeof(int), pl->stream));
    SB_TRY(sb_rt_memset(planes + 2 * bn, 0xff, (size_t)bn * sizeof(int), pl->stream));
    SB_TRY(sb_rt_memset(planes + 3 * bn, 0, (size_t)words * bn * sizeof(int), pl->stream));
    sb::RegionOut rg;
    rg.best = pl->d_bsnr - boff;
    rg.count = planes - boff;
    rg.rank_lo = planes + bn - boff;
    rg.rank_hi = planes + 2 * bn - boff;
    rg.bits = (unsigned*)(planes + 3 * bn) - boff;
    rg.age_rank = tab;
    rg.angle_pos = tab + n_idx;
    rg.plane = bn;
    rg.ratio = snr_ratio;
    pl->region_npos = 0;
    SweepOut so;
    so.region = &rg;
    SB_OK(run_sweep(pl, angles, n_angles, tmpls, n_tmpls, so, whole_search5));
    SB_TRY(sb_rt_sync(pl->stream));
    pl->region_words = words;
    pl->region_npos = n_pos;
    pl->region_nranks = n_ranks;
    return 0;
}

int sb_secondary_sweep(sb_plan* pl, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                       const int32_t* whole_search5, const int32_t* angle_pos_host, int n_idx, int n_pos, int periodic,
                       int min_sep_pos) {
    if (!pl || !angles || !tmpls || !angle_pos_host || n_idx <= 0) return fail("sb_secondary_sweep: bad arguments");
    if (pl->n_states < 2) return fail("sb_secondary_sweep: needs 2 best states (option \"states\"), the plan has " +
                                      std::to_string(pl->n_states));
    if (pl->precision != 32 || !pl->fast)
        return fail("sb_secondary_sweep: secondary fit needs precision 32 and the option fast");
    if (n_pos < 1 || n_pos > 256) return fail("sb_secondary_sweep: n_pos must be in 1 .. 256");
    const int max_dist = periodic ? n_pos / 2 : n_pos - 1;
    if (min_sep_pos < 1 || min_sep_pos > max_dist)
        return fail("sb_secondary_sweep: min_sep_pos must be in 1 .. " + std::to_string(max_dist) +
                    " (the largest distance between two orientation positions)");
    for (int k = 0; k < n_idx; ++k)
        if (angle_pos_host[k] < 0 || angle_pos_host[k] >= n_pos)
            return fail("sb_secondary_sweep: orientation position out of range at flat index " + std::to_string(k));
    for (int k = 0; k < n_tmpls; ++k) {
        if (tmpls[k].idx < 0 || tmpls[k].idx >= n_idx)
            return fail("sb_secondary_sweep: template flat index outside 0 .. n_idx - 1");
        if (tmpls[k].state != 0)
            return fail("sb_secondary_sweep: every record must be in best state 0 (state != 0)");
    }
    const long bn = pl->bn(), boff = (long)pl->slab_lo * pl->nx;
    SB_OK(ensure(pl->rtab, (size_t)n_idx * sizeof(int32_t)));
    SB_OK(ensure(pl->spos, (size_t)bn * sizeof(unsigned short)));
    int* tab = (int*)pl->rtab.p;
    unsigned short* pos = (unsigned short*)pl->spos.p;
    SB_TRY(sb_rt_h2d(tab, angle_pos_host, (size_t)n_idx * sizeof(int32_t), pl->stream));
    SB_OK(launch(pl, "k_secondary_pos", sb::k_secondary_pos, dim3(div_up(bn, 256)), dim3(256), 0, bn,
                 (const float*)pl->d_bsnr, (const int*)pl->d_bidx, (const int*)tab, n_idx, pos));
    SB_OK(launch(pl, "k_best_init", sb::k_best_init, dim3(div_up(bn, 256)), dim3(256), 0, bn, pl->d_bsnr + bn,
                 pl->d_bamp + bn, pl->d_bidx + bn));
    sb::SecondOut sec;
    sec.pos = pos - boff;
    sec.angle_pos = tab;
    sec.n_pos = n_pos;
    sec.min_sep = min_sep_pos;
    sec.periodic = periodic ? 1 : 0;
    SweepOut so;
    so.second = &sec;
    SB_OK(run_sweep(pl, angles, n_angles, tmpls, n_tmpls, so, whole_search5));
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_peak_sweep(sb_plan* pl, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                  const int32_t* whole_search5, const int32_t* age_rank_host, const int32_t* angle_pos_host, int n_idx,
                  int n_ranks, int n_pos, int periodic) {
    if (!pl || !angles || !tmpls || !age_rank_host || !angle_pos_host || n_idx <= 0)
        return fail("sb_peak_sweep: bad arguments");
    if (pl->precision != 32 || !pl->fast) return fail("sb_peak_sweep: fit peak needs precision 32 and the option fast");
    // 16-bit fields of the winner code; rank 0xffff is left free for the codes that match nothing
    if (n_ranks < 1 || n_ranks > 0xffff) return fail("sb_peak_sweep: n_ranks must be in 1 .. 65535");
    if (n_pos < 1 || n_pos > 0xffff) return fail("sb_peak_sweep: n_pos must be in 1 .. 65535");
    if (periodic && n_pos < 3) return fail("sb_peak_sweep: a periodic search needs n_pos >= 3");
    for (int k = 0; k < n_idx; ++k)
        if (age_rank_host[k] < 0 || age_rank_host[k] >= n_ranks || angle_pos_host[k] < 0 || angle_pos_host[k] >= n_pos)
            return fail("sb_peak_sweep: age rank or orientation position out of range at flat index " + std::to_string(k));
    for (int k = 0; k < n_tmpls; ++k) {
        if (tmpls[k].idx < 0 || tmpls[k].idx >= n_idx)
            return fail("sb_peak_sweep: template flat index outside 0 .. n_idx - 1");
        if (tmpls[k].state != 0) return fail("sb_peak_sweep: every record must be in best state 0 (state != 0)");
    }
    // per flat index, the winner codes it neighbours: winner rank + 1 (it is age-), rank - 1 (age+),
    // position + 1 (ang-) and position - 1 (ang+), the positions wrapping round in a periodic search
    const int none = (int)0xfffffffeu;
    std::vector<int4> codes(n_idx);
    for (int k = 0; k < n_idx; ++k) {
        const int r = age_rank_host[k], p = angle_pos_host[k];
        const int up = p + 1 < n_pos ? p + 1 : periodic ? 0 : -1, down = p > 0 ? p - 1 : periodic ? n_pos - 1 : -1;
        codes[k].x = r + 1 < n_ranks ? (r + 1) << 16 | p : none;
        codes[k].y = r > 0 ? (r - 1) << 16 | p : none;
        codes[k].z = up >= 0 ? r << 16 | up : none;
        codes[k].w = down >= 0 ? r << 16 | down : none;
    }
    const long bn = pl->bn(), boff = (long)pl->slab_lo * pl->nx;
    SB_OK(ensure(pl->rtab, (size_t)n_idx * (sizeof(int4) + 2 * sizeof(int32_t))));
    SB_OK(ensure(pl->peak, (size_t)5 * bn * sizeof(int)));
    int4* d_codes = (int4*)pl->rtab.p;
    int* d_rank = (int*)(d_codes + n_idx);
    int* d_pos = d_rank + n_idx;
    int* planes = (int*)pl->peak.p;
    unsigned* code = (unsigned*)(planes + 4 * bn);
    SB_TRY(sb_rt_h2d(d_codes, codes.data(), (size_t)n_idx * sizeof(int4), pl->stream));
    SB_TRY(sb_rt_h2d(d_rank, age_rank_host, (size_t)n_idx * sizeof(int32_t), pl->stream));
    SB_TRY(sb_rt_h2d(d_pos, angle_pos_host, (size_t)n_idx * sizeof(int32_t), pl->stream));
    SB_TRY(sb_rt_memset(planes, 0, (size_t)4 * bn * sizeof(int), pl->stream));
    SB_OK(launch(pl, "k_peak_code", sb::k_peak_code, dim3(div_up(bn, 256)), dim3(256), 0, bn, (const float*)pl->d_bsnr,
                 (const int*)pl->d_bidx, (const int*)d_rank, (const int*)d_pos, n_idx, code));
    SB_TRY(sb_rt_sync(pl->stream));                     // `codes` must outlive its copy
    sb::PeakOut pk;
    pk.code = code - boff;
    pk.planes = planes - boff;
    pk.codes = d_codes;
    pk.plane = bn;
    pl->peak_npos = 0;
    SweepOut so;
    so.peak = &pk;
    SB_OK(run_sweep(pl, angles, n_angles, tmpls, n_tmpls, so, whole_search5));
    SB_TRY(sb_rt_sync(pl->stream));
    pl->peak_nranks = n_ranks;
    pl->peak_npos = n_pos;
    return 0;
}

int sb_peak_finalize(sb_plan* pl, int row_lo, int row_hi, const double* age_of_host, const double* angle_of_host,
                     int n_idx, const double* log10_rank_age_host, int n_ranks, int n_pos, int periodic, double step,
                     double* out8) {
    if (!pl || !age_of_host || !angle_of_host || !log10_rank_age_host || !out8 || n_idx <= 0)
        return fail("sb_peak_finalize: bad arguments");
    if (pl->peak_npos == 0) return fail("sb_peak_finalize: no peak sweep since the best state was last allocated");
    if (n_ranks != pl->peak_nranks || n_pos != pl->peak_npos)
        return fail("sb_peak_finalize: n_ranks / n_pos differ from the peak sweep's");
    if (!std::isfinite(step)) return fail("sb_peak_finalize: step must be finite");
    if (row_lo < pl->slab_lo || row_hi > pl->slab_hi || row_lo >= row_hi) return fail("sb_peak_finalize: rows outside the plan");
    const long n = (long)(row_hi - row_lo) * pl->nx;
    const long off = (long)(row_lo - pl->slab_lo) * pl->nx;
    const long bn = pl->bn();
    SB_OK(ensure(pl->tables, (size_t)(2 * n_idx + n_ranks) * sizeof(double)));
    double* d_age = (double*)pl->tables.p;
    double* d_ang = d_age + n_idx;
    double* d_lx = d_ang + n_idx;
    SB_TRY(sb_rt_h2d(d_age, age_of_host, (size_t)n_idx * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d_ang, angle_of_host, (size_t)n_idx * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d_lx, log10_rank_age_host, (size_t)n_ranks * sizeof(double), pl->stream));
    SB_OK(ensure(pl->raw, (size_t)n * 8 * sizeof(double)));
    double* dst = (double*)pl->raw.p;
    const int* planes = (const int*)pl->peak.p + off;
    SB_OK(launch(pl, "k_peak_finalize", sb::k_peak_finalize, dim3(div_up(n, 256)), dim3(256), 0, n, bn,
                 (const float*)pl->d_bsnr + off, (const float*)pl->d_bamp + off, (const int*)pl->d_bidx + off,
                 (const unsigned*)(planes + 4 * bn), (const float*)planes, (const double*)d_age, (const double*)d_ang,
                 n_idx, (const double*)d_lx, n_ranks, n_pos, periodic ? 1 : 0, step, dst));
    return copy_out(pl, out8, dst, (size_t)n * 8, 0);
}

int sb_peak_planes(sb_plan* pl, int32_t** planes_dev) {
    if (!pl || !planes_dev) return fail("sb_peak_planes: bad arguments");
    if (pl->peak_npos == 0) return fail("sb_peak_planes: no peak sweep since the best state was last allocated");
    *planes_dev = (int32_t*)pl->peak.p;
    return 0;
}

int sb_region_finalize(sb_plan* pl, int row_lo, int row_hi, const double* age_of_host, const double* angle_of_host,
                       int n_idx, const double* rank_age_host, int n_ranks, const double* pos_angle_host, int n_pos,
                       int periodic, double* out9, int out_is_device) {
    if (!pl || !age_of_host || !angle_of_host || !rank_age_host || !pos_angle_host || !out9 || n_idx <= 0)
        return fail("sb_region_finalize: bad arguments");
    if (pl->region_npos == 0) return fail("sb_region_finalize: no region sweep since the best state was last allocated");
    if (n_pos != pl->region_npos) return fail("sb_region_finalize: n_pos differs from the region sweep's");
    if (n_ranks < pl->region_nranks) return fail("sb_region_finalize: fewer ages than the region sweep's ranks");
    if (row_lo < pl->slab_lo || row_hi > pl->slab_hi || row_lo >= row_hi) return fail("sb_region_finalize: rows outside the plan");
    const long n = (long)(row_hi - row_lo) * pl->nx;
    const long off = (long)(row_lo - pl->slab_lo) * pl->nx;
    const long bn = pl->bn();
    SB_OK(ensure(pl->tables, (size_t)(2 * n_idx + n_ranks + n_pos) * sizeof(double)));
    double* d_age = (double*)pl->tables.p;
    double* d_ang = d_age + n_idx;
    double* d_rank_age = d_ang + n_idx;
    double* d_pos_angle = d_rank_age + n_ranks;
    SB_TRY(sb_rt_h2d(d_age, age_of_host, (size_t)n_idx * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d_ang, angle_of_host, (size_t)n_idx * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d_rank_age, rank_age_host, (size_t)n_ranks * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d_pos_angle, pos_angle_host, (size_t)n_pos * sizeof(double), pl->stream));
    double* dst = out9;
    if (!out_is_device) {
        SB_OK(ensure(pl->raw, (size_t)n * 9 * sizeof(double)));
        dst = (double*)pl->raw.p;
    }
    const int* planes = (const int*)pl->region.p + off;
    SB_OK(launch(pl, "k_region_finalize", sb::k_region_finalize, dim3(div_up(n, 256)), dim3(256), 0, n, bn,
                 pl->region_words, (const float*)pl->d_bsnr + off, (const float*)pl->d_bamp + off,
                 (const int*)pl->d_bidx + off, planes, planes + bn, planes + 2 * bn, (const unsigned*)(planes + 3 * bn),
                 (const double*)d_age, (const double*)d_ang, n_idx, (const double*)d_rank_age,
                 (const double*)d_pos_angle, n_pos, periodic ? 1 : 0, dst));
    if (!out_is_device) return copy_out(pl, out9, dst, (size_t)n * 9, 0);
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_finalize(sb_plan* pl, const double* age_of_host, const double* angle_of_host, int n_idx, double* out4,
                int out_is_device) {
    if (!pl) return fail("null plan");
    return sb_finalize_ex(pl, 0, pl->slab_lo, pl->slab_hi, age_of_host, angle_of_host, n_idx, out4, out_is_device);
}

int sb_best_state_ex(sb_plan* pl, int state, float** snr_dev, float** amp_dev, int32_t** idx_dev) {
    if (!pl) return fail("null plan");
    if (state < 0 || state >= pl->n_states) return fail("state out of range");
    const long off = (long)state * pl->bn();
    if (snr_dev) *snr_dev = pl->d_bsnr + off;
    if (amp_dev) *amp_dev = pl->d_bamp + off;
    if (idx_dev) *idx_dev = pl->d_bidx + off;
    return 0;
}

int sb_best_state(sb_plan* pl, float** snr_dev, float** amp_dev, int32_t** idx_dev) {
    return sb_best_state_ex(pl, 0, snr_dev, amp_dev, idx_dev);
}

int sb_best_merge(sb_plan* pl, int state, int row_lo, int row_hi, int n_cands, const float* snr_c, const float* amp_c,
                  const int32_t* idx_c) {
    if (!pl || !snr_c || !amp_c || !idx_c || n_cands < 1) return fail("sb_best_merge: bad arguments");
    if (state < 0 || state >= pl->n_states) return fail("sb_best_merge: state out of range");
    if (row_lo < pl->slab_lo || row_hi > pl->slab_hi || row_lo >= row_hi) return fail("sb_best_merge: rows outside the plan");
    const long n = (long)(row_hi - row_lo) * pl->nx;
    const long off = (long)state * pl->bn() + (long)(row_lo - pl->slab_lo) * pl->nx;
    return launch(pl, "k_best_merge", sb::k_best_merge, dim3(div_up(n, 256)), dim3(256), 0, n, n_cands, snr_c, amp_c,
                  (const int*)idx_c, pl->d_bsnr + off, pl->d_bamp + off, pl->d_bidx + off);
}

int sb_region_planes(sb_plan* pl, int32_t** planes_dev, int* n_planes) {
    if (!pl || !planes_dev || !n_planes) return fail("sb_region_planes: bad arguments");
    if (pl->region_npos == 0) return fail("sb_region_planes: no region sweep since the best state was last allocated");
    *planes_dev = (int32_t*)pl->region.p;
    *n_planes = 3 + pl->region_words;
    return 0;
}

int sb_region_merge(sb_plan* pl, int row_lo, int row_hi, int n_cands, const int32_t* cands_dev) {
    if (!pl || !cands_dev || n_cands < 1) return fail("sb_region_merge: bad arguments");
    if (pl->region_npos == 0) return fail("sb_region_merge: no region sweep since the best state was last allocated");
    if (row_lo < pl->slab_lo || row_hi > pl->slab_hi || row_lo >= row_hi) return fail("sb_region_merge: rows outside the plan");
    const long n = (long)(row_hi - row_lo) * pl->nx;
    const long off = (long)(row_lo - pl->slab_lo) * pl->nx;
    const int n_planes = 3 + pl->region_words;
    return launch(pl, "k_region_merge", sb::k_region_merge, dim3(div_up(n * n_planes, 256)), dim3(256), 0, n, n_planes,
                  n_cands, pl->bn(), (const int*)cands_dev, (int*)pl->region.p + off);
}

int sb_best_pack(sb_plan* pl, unsigned long long* keys_dev) {
    if (!pl || !keys_dev) return fail("sb_best_pack: null");
    const long n = pl->bn();
    return launch(pl, "k_best_pack", sb::k_best_pack, dim3(div_up(n, 256)), dim3(256), 0, n, (const float*)pl->d_bsnr,
                  (const int*)pl->d_bidx, keys_dev);
}

int sb_best_select(sb_plan* pl, const unsigned long long* gkeys_dev, float* amp_out_dev) {
    if (!pl || !gkeys_dev || !amp_out_dev) return fail("sb_best_select: null");
    const long n = pl->bn();
    return launch(pl, "k_best_select", sb::k_best_select, dim3(div_up(n, 256)), dim3(256), 0, n,
                  (const float*)pl->d_bsnr, (const float*)pl->d_bamp, (const int*)pl->d_bidx, gkeys_dev, amp_out_dev);
}

int sb_best_unpack(sb_plan* pl, const unsigned long long* gkeys_dev, const float* amp_dev) {
    if (!pl || !gkeys_dev || !amp_dev) return fail("sb_best_unpack: null");
    const long n = pl->bn();
    return launch(pl, "k_best_unpack", sb::k_best_unpack, dim3(div_up(n, 256)), dim3(256), 0, n, gkeys_dev, amp_dev,
                  pl->d_bsnr, pl->d_bamp, pl->d_bidx);
}

int sb_compare_host(sb_plan* pl, double* best4_host, const double* amp, const double* age, const double* angle,
                    const double* snr, double age_s, double angle_s) {
    if (!pl || !best4_host || !amp || !snr) return fail("sb_compare_host: null");
    const long n = (long)pl->ny * pl->nx;
    SB_OK(ensure(pl->raw, (size_t)n * 8 * sizeof(double)));
    double* d = (double*)pl->raw.p;
    SB_TRY(sb_rt_h2d(d, best4_host, (size_t)n * 4 * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d + 4 * n, amp, (size_t)n * sizeof(double), pl->stream));
    SB_TRY(sb_rt_h2d(d + 5 * n, snr, (size_t)n * sizeof(double), pl->stream));
    const double* d_age = nullptr;
    const double* d_ang = nullptr;
    if (age) { SB_TRY(sb_rt_h2d(d + 6 * n, age, (size_t)n * sizeof(double), pl->stream)); d_age = d + 6 * n; }
    if (angle) { SB_TRY(sb_rt_h2d(d + 7 * n, angle, (size_t)n * sizeof(double), pl->stream)); d_ang = d + 7 * n; }
    SB_OK(launch(pl, "k_compare", sb::k_compare, dim3(div_up(n, 256)), dim3(256), 0, n, d, d + n, d + 2 * n, d + 3 * n,
                 (const double*)(d + 4 * n), d_age, d_ang, (const double*)(d + 5 * n), age_s, angle_s));
    return copy_out(pl, best4_host, d, (size_t)n * 4, 0);
}

int sb_curvature_noise_moments(sb_plan* pl, double sigma, double truncate, double* out10_host) {
    if (!pl || !out10_host || !(sigma > 0.0) || !(truncate > 0.0)) return fail("sb_curvature_noise_moments: bad arguments");
    if (!pl->d_dem) return fail("no DEM set");
    if (!pl->whole()) return fail("sb_curvature_noise_moments needs a plan over the whole raster");
    const int ny = pl->ny, nx = pl->nx;
    const long n = (long)ny * nx;
    const int radius = (int)(truncate * sigma + 0.5);          // scipy.ndimage.gaussian_filter1d
    std::vector<double> w(2 * radius + 1);
    {
        double s = 0.0;
        for (int k = -radius; k <= radius; ++k) { w[k + radius] = std::exp(-0.5 / (sigma * sigma) * (double)k * (double)k); s += w[k + radius]; }
        for (auto& v : w) v /= s;
    }
    SB_OK(ensure_diffs64(pl));
    // aux: weights | 4 planes in (dxx, dxy, dyy, nan flag) column-filtered | 4 planes fully filtered | partial sums
    const int blocks = std::max(1, std::min(2048, div_up(n, 256)));
    const size_t wbytes = (w.size() * sizeof(double) + 255) / 256 * 256;
    SB_OK(ensure(pl->aux, wbytes + (size_t)n * 8 * sizeof(double) + (size_t)blocks * 10 * sizeof(double)));
    double* d_w = (double*)pl->aux.p;
    double* d_tmp = (double*)((char*)pl->aux.p + wbytes);
    double* d_low = d_tmp + 4 * n;
    double* d_part = d_low + 4 * n;
    SB_TRY(sb_rt_h2d(d_w, w.data(), w.size() * sizeof(double), pl->stream));
    SB_OK(launch(pl, "k_gauss_axis0", sb::k_gauss_axis0, dim3(div_up(n, 256), 4), dim3(256), 0, ny, nx, radius,
                 (const double*)d_w, (const double*)pl->d_diffs, (const double*)pl->d_dem, d_tmp));
    SB_OK(launch(pl, "k_gauss_axis1", sb::k_gauss_axis1, dim3(div_up(n, 256), 4), dim3(256), 0, ny, nx, radius,
                 (const double*)d_w, (const double*)d_tmp, d_low));
    SB_OK(launch(pl, "k_noise_moments", sb::k_noise_moments, dim3(blocks), dim3(256), 256 * 10 * sizeof(double), n,
                 (const double*)pl->d_diffs, (const double*)pl->d_dem, (const double*)d_low, d_part));
    std::vector<double> part((size_t)blocks * 10);
    SB_TRY(sb_rt_d2h(part.data(), d_part, part.size() * sizeof(double), pl->stream));
    SB_TRY(sb_rt_sync(pl->stream));
    for (int k = 0; k < 10; ++k) {
        double s = 0.0;
        for (int b = 0; b < blocks; ++b) s += part[(size_t)b * 10 + k];
        out10_host[k] = s;
    }
    return 0;
}

int sb_fill_nodata(sb_plan* pl, double* dem_host_inout, double max_search_distance, long* remaining) {
    if (!pl || !dem_host_inout) return fail("sb_fill_nodata: null");
    if (!pl->whole()) return fail("sb_fill_nodata needs a plan over the whole raster");
    const long n = (long)pl->ny * pl->nx;
    SB_OK(ensure(pl->aux, (size_t)n * 2 * sizeof(double) + 1024 * sizeof(long)));
    double* d_in = (double*)pl->aux.p;
    double* d_out = d_in + n;
    long* d_cnt = (long*)(d_out + n);
    SB_TRY(sb_rt_h2d(d_in, dem_host_inout, (size_t)n * sizeof(double), pl->stream));
    SB_TRY(sb_rt_memset(d_cnt, 0, sizeof(long) * 1024, pl->stream));
    const int blocks = div_up(n, 256);
    SB_OK(launch(pl, "k_fill_nodata", sb::k_fill_nodata, dim3(blocks), dim3(256), 0, pl->ny, pl->nx,
                 (const double*)d_in, d_out, max_search_distance, d_cnt));
    std::vector<long> cnt(1024);
    SB_TRY(sb_rt_d2h(cnt.data(), d_cnt, sizeof(long) * 1024, pl->stream));
    SB_OK(copy_out(pl, dem_host_inout, d_out, (size_t)n, 0));
    long left = 0;
    for (long v : cnt) left += v;
    if (remaining) *remaining = left;
    return 0;
}

int sb_debug_fft(sb_plan* pl, int n, int rows, const float* in_host, float* out_host, int inverse) {
    if (!pl || !in_host || !out_host || rows <= 0) return fail("sb_debug_fft: bad arguments");
    const float2* tw = nullptr;
    if (!is_pow2(n) || n < kMinFft || n > kMaxFftSupported) return fail("sb_debug_fft: unsupported length");
    SB_OK(twiddles<float>(pl, n, &tw));
    const size_t bytes = (size_t)rows * n * sizeof(float2);
    SB_OK(ensure(pl->raw, 2 * bytes));
    float2* d_in = (float2*)pl->raw.p;
    float2* d_out = d_in + (size_t)rows * n;
    SB_TRY(sb_rt_h2d(d_in, in_host, bytes, pl->stream));
    if (inverse & 2) {          // the radix-64 core (length 4096 only)
        if (n != sb64::N) return fail("sb_debug_fft: the radix-64 core is length 4096");
        const float2* tw64 = nullptr;
        SB_OK(twiddles64(pl, &tw64));
        constexpr size_t smem = (size_t)(4 * sb64::kXchg + sb64::kTwRows * sb64::R) * sizeof(float2);
        SB_OK(launch(pl, "k_fft4096_r64", sb64::k_fft4096_r64, dim3(div_up(rows, 4)), dim3(256), smem, rows,
                     (const float2*)d_in, d_out, inverse & 1, tw64));
        SB_TRY(sb_rt_d2h(out_host, d_out, bytes, pl->stream));
        SB_TRY(sb_rt_sync(pl->stream));
        return 0;
    }
    SB_OK(dispatch_n(n, [&](auto nn) {
        constexpr int N = decltype(nn)::value;
        using S = Shape<N, float>;
        auto kern = sb::k_fft_rows<N, float>;
        return launch(pl, "k_fft_rows", kern, dim3(div_up(rows, S::GP)), dim3(S::threads), S::smem, rows,
                      (const float2*)d_in, d_out, inverse, tw);
    }));
    SB_TRY(sb_rt_d2h(out_host, d_out, bytes, pl->stream));
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

int sb_debug_fft_bench(sb_plan* pl, int n, int rows, int reps, int radix64, float* ms_per_launch) {
    if (!pl || rows <= 0 || reps <= 0 || !ms_per_launch) return fail("sb_debug_fft_bench: bad arguments");
    if (!is_pow2(n) || n < kMinFft || n > kMaxFftSupported) return fail("sb_debug_fft_bench: unsupported length");
    const size_t bytes = (size_t)rows * n * sizeof(float2);
    SB_OK(ensure(pl->raw, 2 * bytes));
    float2* d_in = (float2*)pl->raw.p;
    float2* d_out = d_in + (size_t)rows * n;
    SB_TRY(sb_rt_memset(d_in, 0, bytes, pl->stream));
    sb_event_t e0, e1;
    sb_rt_event_create(&e0);
    sb_rt_event_create(&e1);
    int rc = 0;
    for (int it = 0; it < reps + 1 && rc == 0; ++it) {
        if (it == 1) sb_rt_event_record(e0, pl->stream);      // the first launch is the warm-up
        if (radix64) {
            if (n != sb64::N) { rc = fail("the radix-64 core is length 4096"); break; }
            const float2* tw64 = nullptr;
            rc = twiddles64(pl, &tw64);
            if (rc) break;
            constexpr size_t smem = (size_t)(4 * sb64::kXchg + sb64::kTwRows * sb64::R) * sizeof(float2);
            rc = launch(pl, "k_fft4096_r64", sb64::k_fft4096_r64, dim3(div_up(rows, 4)), dim3(256), smem, rows,
                        (const float2*)d_in, d_out, 0, tw64);
        } else {
            const float2* tw = nullptr;
            rc = twiddles<float>(pl, n, &tw);
            if (rc) break;
            rc = dispatch_n(n, [&](auto nn) {
                constexpr int N = decltype(nn)::value;
                using S = Shape<N, float>;
                auto kern = sb::k_fft_rows<N, float>;
                return launch(pl, "k_fft_rows", kern, dim3(div_up(rows, S::GP)), dim3(S::threads), S::smem, rows,
                              (const float2*)d_in, d_out, 0, tw);
            });
        }
    }
    sb_rt_event_record(e1, pl->stream);
    sb_rt_sync(pl->stream);
    *ms_per_launch = sb_rt_event_ms(e0, e1) / (float)reps;
    sb_rt_event_destroy(e0);
    sb_rt_event_destroy(e1);
    return rc;
}

int sb_sync(sb_plan* pl) {
    if (!pl) return fail("null plan");
    SB_TRY(sb_rt_sync(pl->stream));
    return 0;
}

}  // extern "C"
