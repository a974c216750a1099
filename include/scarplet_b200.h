/* scarplet_b200 — C ABI of the B200-native template-matching hot path.
 *
 * The reference (stgl/scarplet 0.1.4) is pure Python and has no FFI; its boundary for
 * this path is the Python API of scarplet/core.py and the WindowedTemplate plugin
 * duck type.  Each entry point below replaces the reference interface cited beside
 * it; scarplet_b200/core.py (the host-side mirror) binds them with ctypes and
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions: every function returns 0 on success or a non-zero status and leaves a
 * message retrievable with sb_last_error().  A plan is bound to one CUDA device and
 * is used from one host thread at a time; work is stream-ordered on the plan's
 * stream.  `*_host` pointers are host memory (copied inside the call), `*_dev`
 * pointers are device memory on the plan's device.  Inputs are borrowed and never
 * modified; outputs are caller-allocated.
 */
#ifndef SCARPLET_B200_H
#define SCARPLET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sb_plan sb_plan;

/* One search orientation: the direction of the curvature
 * (dem.py:68-107 `_calculate_directional_laplacian(alpha)`).  The host passes the
 * float64 values NumPy computes so the device reproduces them bit for bit. */
typedef struct sb_angle {
    double cos_a;   /* np.cos(angle)        */
    double sin_a;   /* np.sin(angle)        */
    double cos2_a;  /* np.cos(angle) ** 2   */
    double sin2_a;  /* np.sin(angle) ** 2   */
} sb_angle;

enum { SB_KIND_SCARP = 0, SB_KIND_RICKER = 1,
       SB_KIND_RASTER = 2 /* values supplied by the caller: sb_match_template_raster */ };
enum { SB_ERRMASK_NONE = 0, SB_ERRMASK_XR_LE0 = 1, SB_ERRMASK_XR_GE0 = 2 };

/* One (scale, age, angle) template: what `Template(scale, age, angle, nx, ny, de)`
 * (core.py:345) plus `.template()`, `.get_window_limits()`, `.get_err_mask()`
 * (core.py:346, 369-375) determine.  Everything that must be float64-exact is
 * precomputed by the host. */
typedef struct sb_template {
    double cos_t, sin_t;  /* cos/sin of the template's alpha = -angle (WindowedTemplate.py:151) */
    double c, d;          /* window half-widths (WindowedTemplate.py:63)                     */
    double k0, k1;        /* scarp: 2*kt**1.5*sqrt(pi), 4*kt;  ricker: pi*f, 0               */
    double sign;          /* -1 for RightFacingUpperBreakScarp (WindowedTemplate.py:254)    */
    double tscale;        /* power of two ~ 1/rms(t): balances t against M in the packed FFT  */
    int32_t kind;         /* SB_KIND_*                                                       */
    int32_t errmode;      /* SB_ERRMASK_* (WindowedTemplate.py:257-267, 294-304)             */
    int32_t sy_lo, sy_hi, sx_lo, sx_hi; /* conservative support box, offsets from (ny//2, nx//2) */
    int32_t i_lo, i_hi, j_lo, j_hi;     /* rows/cols NOT masked by get_window_limits (inclusive) */
    int32_t angle_id;     /* index into the sb_angle array                                  */
    int32_t idx;          /* flat result index: tie priority and key into age_of/angle_of   */
    int32_t state;        /* best state the template folds into (0 .. option "states" - 1): one per
                             template scale in a multi-scale search (CHANGELOG.md:20-24)    */
    int32_t reserved;     /* 0 */
} sb_template;

/* flags for sb_plan_create */
#define SB_PLAN_DEFAULT 0u

const char* sb_last_error(void);
/* library / build information: "cuda sm_100a <hash of the sources it was compiled from>" for the product build */
const char* sb_build_info(void);

/* Plan = raster geometry + device workspace.  dx2/dy2 are `dx ** 2`, `dy ** 2` as the
 * host evaluates them (dem.py:95,99).  device < 0 keeps the current device.
 * stream is a cudaStream_t (0 = the plan creates its own). */
int sb_plan_create(sb_plan** plan, int ny, int nx, double dx, double dx2, double dy2,
                   int device, void* stream, unsigned flags);
int sb_plan_destroy(sb_plan* plan);

/* knobs: key in {"workspace_mb", "max_fft", "force_pad", "mixed_tiles", "profile",
 * "precision" (32 = complex64 pipeline, default; 64 = complex128 pipeline),
 * "states" (number of independent best states, default 1; resets them),
 * and the kernel-selection switches, all on by default (off = the slower variant, same results
 * to rounding): "fast" (pipelined complex64 kernels; the curvature spectra of every orientation
 * are combinations of nine plane spectra computed once per FFT tile), "conv_persist" (persistent
 * column kernel: minimum templates per orientation run, 0 = never), "conv_r64" (radix-64 column
 * kernel at Py = 4096), "fit_substreams" (0 = automatic, 1..8 = sub-streams of the row kernel on
 * small rasters)};
 * returns 0 if known */
int sb_plan_set_option(sb_plan* plan, const char* key, long value);

/* Nodata policy of the searches (sb_sweep / sb_sweep_ex); takes effect at the next sb_set_dem_*.
 *   SB_NODATA_PROPAGATE (default): the reference's semantics -- a NaN anywhere in the DEM reaches
 *     every un-masked pixel through the full-raster fft2 (dem.py:105, core.py:353-363).
 *   SB_NODATA_MASK: a masked fit.  V(p) = 1 where the second differences at p (dem.py:88-99) read
 *     only finite DEM cells; the curvature is zeroed where V = 0 and every fit uses the template
 *     cells over V = 1 only: n_valid = n - rint(M (*) (1 - V)), ts_m = ts - t**2 (*) (1 - V),
 *     amp = xcorr / ts_m, error = (T3 - xcorr**2 / ts_m) / (n_valid + eps) + eps.  A template is a
 *     candidate at a pixel only if n_valid >= ceil(min_coverage * n); a pixel whose own DEM cell is
 *     not finite gets no result (0 in all four planes).  With min_coverage = 1 every value equals
 *     the reference's on the same DEM with its holes filled by any values.
 * Fails for min_coverage outside (0, 1] and, for SB_NODATA_MASK, unless the plan runs the complex64
 * pipelined kernels (precision 32, fast = 1); sb_match_template and
 * sb_match_template_raster fail on a masked plan.  FFT tiles of a masked sweep are at most 4096. */
enum { SB_NODATA_PROPAGATE = 0, SB_NODATA_MASK = 1 };
int sb_plan_set_nodata(sb_plan* plan, int mode, double min_coverage);

/* Spatial sharding of one raster over several GPUs (BASELINE config 5, SURVEY 8e; the reference's
 * analogue is file-level tiling, dem.py:249-278).  The plan keeps the geometry of the WHOLE raster
 * (template centring, edge masks and the circular wrap-around of core.py:359 are evaluated in
 * full-raster coordinates) but computes only raster rows row_lo .. row_hi - 1 and holds only the
 * DEM rows row_lo - halo .. row_hi + halo - 1 (periodic in ny).  Call before sb_set_dem_*; the DEM
 * handed to sb_set_dem_* is then that slab (sb_plan_dem_rows: first raster row, row count).
 * halo >= template support along y + 2.  The best state covers the plan's rows only. */
int sb_plan_set_slab(sb_plan* plan, int row_lo, int row_hi, int halo);
int sb_plan_dem_rows(const sb_plan* plan, int* row0, int* drows);
/* curvature statistics of the plan's own rows (sum of dxx^2 + dyy^2, pixel count): a non-finite
 * sum marks a NaN in the DEM.  Slabs of one raster add theirs up and hand the totals back, so that
 * every rank packs with the same scale and knows about a NaN held by another (dem.py:105). */
int sb_plan_curv_stats(const sb_plan* plan, double* sumsq, double* count);
int sb_plan_set_curv_stats(sb_plan* plan, double sumsq, double count);
/* the cudaStream_t the plan's work is ordered on */
void* sb_plan_stream(const sb_plan* plan);
/* device memory held by the plan (bytes) */
long sb_plan_device_bytes(const sb_plan* plan);
/* sum over the FFT tiles of the last sweep of Py * Px (tiling overhead = this / (rows * nx)) */
double sb_plan_last_fft_area(const sb_plan* plan);
/* per-kernel device time (CUDA events on the plan's stream) accumulated while the option
 * "profile" is 1: ms[6], launches[6] in the order k_curv_rows, k_curv_cols, k_tmpl_rows,
 * k_tmpl_sums, k_conv_cols, k_fit_rows.  reset != 0 clears the counters afterwards. */
int sb_plan_profile(sb_plan* plan, double* ms6, long* launches6, int reset);
/* number of kernels launched by this plan so far */
long sb_plan_launch_count(const sb_plan* plan);
/* FFT domain and tile grid chosen by the last sweep: out[0..5] = largest Py, largest Px, tiles_y, tiles_x,
 * angle batch, template batch (tiles of different lengths are mixed along an axis when that wastes less) */
int sb_plan_last_geometry(const sb_plan* plan, int* out6);

/* DEM upload (DEMGrid._griddata, float64 row-major ny x nx) and the centred axis
 * vectors x[nx], y[ny] of WindowedTemplate.py:50-53. */
int sb_set_dem_host(sb_plan* plan, const double* dem_host);
int sb_set_dem_dev(sb_plan* plan, const double* dem_dev);
int sb_set_axes_host(sb_plan* plan, const double* x_host, const double* y_host);

/* DEMGrid._calculate_directional_laplacian (dem.py:68-107): float64 out[ny*nx]. */
int sb_directional_laplacian(sb_plan* plan, const sb_angle* angle, double* out, int out_is_device);

/* WindowedTemplate.template() (WindowedTemplate.py:159-183, 497-520): float64 out[ny*nx]. */
int sb_render_template(sb_plan* plan, const sb_template* tmpl, double* out, int out_is_device);

/* core.match_template (core.py:297-377): amp[ny*nx], snr[ny*nx] float64 for one template. */
int sb_match_template(sb_plan* plan, const sb_angle* angle, const sb_template* tmpl,
                      double* amp, double* snr, int out_is_device);

/* core.match_template for a template the library has no generator for -- the plugin surface
 * of core.py:345-348: any class with `.template()`.  The caller renders the template on the
 * host and passes its values on the box of rows sy_lo..sy_hi x columns sx_lo..sx_hi (offsets
 * from (ny//2, nx//2), row-major float64) that holds every non-zero; outside the box the
 * template is zero.  amp / snr are the raw planes of core.py:360-367: `get_err_mask` /
 * `get_window_limits` (core.py:369-375) are the caller's to apply.  tscale: a power of two
 * near 1 / rms(template) (0 = 1). */
int sb_match_template_raster(sb_plan* plan, const sb_angle* angle, const double* box_host,
                             int sy_lo, int sy_hi, int sx_lo, int sx_hi, double tscale,
                             double* amp, double* snr, int out_is_device);

/* Fit surfaces at chosen pixels: post-mask amp / snr of every template at every pixel by direct
 * float64 correlation (DESIGN §12).  out[p * n_tmpls + k] for pixel p, record k.
 * For pixel p = (rows_host[p], cols_host[p]) and record k the values core.match_template returns
 * there (core.py:359-375, get_err_mask and get_window_limits applied), with the FFTs replaced by
 * sums over the template's support box in float64:
 *   xcorr = sum t[a0 + u, b0 + v] * curv[(i - u + ny % 2) mod ny, (j - v + nx % 2) mod nx],
 *   T3 = the same sum of M * curv**2, (a0, b0) = (ny / 2, nx / 2);
 * t, M, curv are the library's float64 values; n and ts are fixed-order sums over the box.  A
 * pixel's result does not depend on the other pixels of the call, their order or count, nor on
 * the options "precision", "fast" or the FFT tiling: every sum runs in one fixed order.
 * Nodata: SB_NODATA_PROPAGATE with a non-finite DEM cell anywhere -> NaN wherever the masks leave
 * an entry (the reference's full-raster fft2); SB_NODATA_MASK -> the masked fit of
 * sb_plan_set_nodata with the sums taken over the cells with V = 1.
 * Fails without a DEM, for a pixel outside the plan's rows (row slabs) or columns, on a row slab
 * whose halo does not hold a template's support, and for SB_KIND_RASTER records.  Output buffers
 * are the caller's; device scratch is bounded by working through the pixels in chunks. */
int sb_fit_surface(sb_plan* plan, const sb_angle* angles, int n_angles,
                   const sb_template* tmpls, int n_tmpls,
                   const int32_t* rows_host, const int32_t* cols_host, int n_pix,
                   double* amp, double* snr, int out_is_device);

/* Best-fit state (running result of core.compare over a sweep). */
int sb_best_reset(sb_plan* plan);

/* The fan-out of core.calculate_best_fit_parameters / match (core.py:139-195, 266-294)
 * and the fold of core.compare (core.py:198-243) for a list of templates; accumulates
 * into the plan's best state (call sb_best_reset first for a fresh search). */
int sb_sweep(sb_plan* plan, const sb_angle* angles, int n_angles,
             const sb_template* tmpls, int n_tmpls);

/* The same for a SHARE of a larger search (one rank's orientations): whole_search5 =
 * {sy_lo, sy_hi, sx_lo, sx_hi of the union of all support boxes, templates per orientation} of
 * the undivided search.  FFT domains, tiles and kernel variants are then chosen exactly as the
 * undivided search chooses them, which makes the shares' results bit-identical to its. */
int sb_sweep_ex(sb_plan* plan, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                const int32_t* whole_search5);

/* Decode the best state to the reference's stack order [amp, age, angle, snr]
 * (core.py:190-193): out4 is float64[4*ny*nx]; age_of/angle_of are host float64
 * tables indexed by sb_template.idx (n_idx entries). */
int sb_finalize(sb_plan* plan, const double* age_of_host, const double* angle_of_host, int n_idx,
                double* out4, int out_is_device);

/* The same for best state `state` and raster rows row_lo .. row_hi - 1 only:
 * out4 is float64[4 * (row_hi - row_lo) * nx]. */
int sb_finalize_ex(sb_plan* plan, int state, int row_lo, int row_hi, const double* age_of_host,
                   const double* angle_of_host, int n_idx, double* out4, int out_is_device);

/* Age-resolved search (DESIGN §13): best states 0 .. n_states-1 hold one age each (state s = the
 * templates of ages[s]).  For raster rows row_lo .. row_hi-1 writes out6 = float64[6][rows][nx]:
 *   [0..3] amp, age, angle, snr of the fold over the states (highest SNR, then lowest flat index,
 *          a NaN SNR sticks), decoded as sb_finalize_ex decodes a state;
 *   [4], [5] age_lo, age_hi: the smallest / largest age_of[idx_s] over the states s with
 *          snr_s > 0 and (double)snr_s >= snr_ratio * (double)snr_best; 0 where the fold's snr is
 *          0 or NaN (like its age plane).
 * The fold is the one the single-state sweep runs over the same templates, so planes 0..3 equal
 * sb_finalize_ex after a sweep with every record in state 0.  The states are read, not modified.
 * Fails for snr_ratio outside (0, 1], n_states outside 1 .. option "states", and rows outside the
 * plan's rows. */
int sb_age_range(sb_plan* plan, int n_states, int row_lo, int row_hi, double snr_ratio,
                 const double* age_of_host, const double* angle_of_host, int n_idx,
                 double* out6, int out_is_device);

/* Fit confidence region (DESIGN §14), pass 2 of 2: best state 0 must hold the result of a sweep
 * (sb_sweep / sb_sweep_ex) over the same records.  Runs that sweep again with the region variant
 * of the fit kernel, which writes no best state: a record with flat index k qualifies at a pixel
 * when the masks (window, get_err_mask, min_coverage) leave it a candidate there and its float32
 * SNR s satisfies s > 0 and (double)s >= snr_ratio * (double)best, best = state 0's SNR.  The
 * plan's region planes (cleared first; 4 * (3 + ceil(n_pos / 32)) bytes per pixel of the plan's
 * rows, allocated on first use) receive per pixel the count of qualifying records, the lowest and
 * highest age_rank_host[k] and the bits angle_pos_host[k] (in 0 .. n_pos - 1) of them.  Integer
 * atomics: the result does not depend on batches, sub-streams or launch order.
 * Fails for snr_ratio outside (0, 1], n_pos outside 1 .. 256, ranks / positions out of range, a
 * record whose idx is outside 0 .. n_idx - 1 or whose state is not 0, and precision 64 or fast = 0. */
int sb_region_sweep(sb_plan* plan, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                    const int32_t* whole_search5, double snr_ratio, const int32_t* age_rank_host,
                    const int32_t* angle_pos_host, int n_idx, int n_pos);

/* Decode the region planes for raster rows row_lo .. row_hi-1: out9 = float64[9][rows][nx]
 *   [0..3] amp, age, angle, snr of best state 0 (as sb_finalize_ex);
 *   [4], [5] age_lo, age_hi = rank_age_host[lowest / highest rank];
 *   [6], [7] angle_lo, angle_hi: the shortest arc of orientation positions holding every
 *            qualifying one.  periodic = 0: pos_angle_host[first], pos_angle_host[last].
 *            periodic = 1 (positions 0 .. n_pos - 1 close into a circle of pi): the complement of
 *            the largest circular gap between consecutive qualifying positions (equal gaps: the
 *            lowest p_lo), angle_hi = pos_angle_host[p_hi] + pi when the arc wraps (p_hi < p_lo);
 *   [8] the number of qualifying records.
 * Planes 4..8 are 0 where state 0's SNR is 0 or NaN.  Fails without a region sweep since the best
 * state was last allocated (option "states", sb_plan_set_slab), for n_pos other than the sweep's,
 * fewer ranks than the sweep used, and rows outside the plan. */
int sb_region_finalize(sb_plan* plan, int row_lo, int row_hi, const double* age_of_host,
                       const double* angle_of_host, int n_idx, const double* rank_age_host, int n_ranks,
                       const double* pos_angle_host, int n_pos, int periodic, double* out9, int out_is_device);

/* Secondary fit (DESIGN §16): best state 0 must hold the result of a sweep (sb_sweep / sb_sweep_ex)
 * over the same records, on a plan with at least 2 best states.  Resets best state 1 and sweeps the
 * records again into it, folding at each pixel only the records whose orientation position
 * angle_pos_host[idx] (in 0 .. n_pos - 1) is at least min_sep_pos from the position of state 0's
 * winner there: distance |p - q|, or min(|p - q|, n_pos - |p - q|) when periodic.  A pixel whose state
 * 0 SNR is 0 or NaN admits nothing.  Otherwise the fold is the search's (masks, min_coverage, highest
 * SNR then lowest flat index, NaN windows of a NaN DEM, nodata cleared), so state 1 does not depend on
 * batches, sub-streams or launch order; sb_finalize_ex(state 1) decodes it.  State 0 is not modified.
 * Device memory: best state 1 (12 B per pixel) and a 2 B per pixel position plane.
 * Fails for a plan with fewer than 2 states, precision 64 or fast = 0, n_pos outside 1 .. 256,
 * min_sep_pos outside 1 .. (periodic ? n_pos / 2 : n_pos - 1), positions out of range, a record whose
 * idx is outside 0 .. n_idx - 1 or whose state is not 0. */
int sb_secondary_sweep(sb_plan* plan, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                       const int32_t* whole_search5, const int32_t* angle_pos_host, int n_idx, int n_pos,
                       int periodic, int min_sep_pos);

/* Sub-grid fit peak (DESIGN §17), pass 2 of 2: best state 0 must hold the result of a sweep
 * (sb_sweep / sb_sweep_ex) over the same records.  Runs that sweep again with the peak variant of
 * the fit kernel, which writes no best state.  The winner of state 0 at a pixel (where its SNR is
 * > 0) has age rank r = age_rank_host[idx] (0 .. n_ranks - 1) and orientation position
 * p = angle_pos_host[idx] (0 .. n_pos - 1).  The plan's four neighbour planes (float32, cleared
 * first) receive per pixel the largest SNR s > 0 of the records at (r - 1, p), (r + 1, p), (r, p - 1)
 * and (r, p + 1) -- positions wrap round when periodic -- that the masks (window, get_err_mask,
 * min_coverage) leave a candidate there; 0 where there is none.  The winner and its periodic twin
 * are not recorded.  Integer atomics: the result does not depend on batches, sub-streams or launch
 * order.  Device memory: 20 B per pixel of the plan's rows (the four planes and a winner code
 * plane), allocated on first use.
 * Fails for precision 64 or fast = 0, n_ranks or n_pos outside 1 .. 65535 (16-bit fields of the
 * winner code), a periodic search with n_pos < 3, ranks / positions out of range, and a record whose
 * idx is outside 0 .. n_idx - 1 or whose state is not 0. */
int sb_peak_sweep(sb_plan* plan, const sb_angle* angles, int n_angles, const sb_template* tmpls, int n_tmpls,
                  const int32_t* whole_search5, const int32_t* age_rank_host, const int32_t* angle_pos_host,
                  int n_idx, int n_ranks, int n_pos, int periodic);

/* Decode the fit peak for raster rows row_lo .. row_hi-1: out8 = host float64[8][rows][nx]
 *   [0..3] amp, age, angle, snr of best state 0 (as sb_finalize_ex);
 *   [4] age_peak: 10^(x[r] + u), u the vertex of the parabola through (x[r -+ 1], s_age-+) and
 *       (x[r], snr), x = log10_rank_age_host (log10 of the sorted ages), where 0 < r < n_ranks - 1,
 *       both neighbours are > 0 and d- + d+ > 0 (d-+ = snr - s_age-+); the grid age elsewhere;
 *   [5] angle_peak = angle + step * (d- - d+) / (2 (d- + d+)) from the orientation neighbours, where
 *       the winner has both (periodic with n_pos >= 3, or 0 < p < n_pos - 1), they are > 0 and
 *       d- + d+ > 0; the grid angle elsewhere;
 *   [6] snr_peak = snr + the gain of the refined axes;  [7] refined = 1 (age) + 2 (orientation).
 * Float64 without contraction.  Planes 4..7 are 0 where state 0's SNR is 0, [0, 0, NaN, 0] where it
 * is NaN.  Fails without a peak sweep since the best state was last allocated (option "states",
 * sb_plan_set_slab), for n_ranks / n_pos other than the sweep's, and rows outside the plan. */
int sb_peak_finalize(sb_plan* plan, int row_lo, int row_hi, const double* age_of_host, const double* angle_of_host,
                     int n_idx, const double* log10_rank_age_host, int n_ranks, int n_pos, int periodic, double step,
                     double* out8);

/* The neighbour planes of the last peak sweep: int32 device memory, the bits of float32 SNRs >= 0
 * (they order as integers), plane j (0 age-, 1 age+, 2 orientation-, 3 orientation+) of pixel i of
 * the plan's rows at [j * rows * nx + i]. */
int sb_peak_planes(sb_plan* plan, int32_t** planes_dev);

/* Raw best state for a cross-GPU merge: device pointers into the plan, one value per pixel of
 * the plan's rows. */
int sb_best_state(sb_plan* plan, float** snr_dev, float** amp_dev, int32_t** idx_dev);
int sb_best_state_ex(sb_plan* plan, int state, float** snr_dev, float** amp_dev, int32_t** idx_dev);

/* Fold n_cands candidate best states for raster rows row_lo .. row_hi - 1 (device buffers laid out
 * [candidate][row][nx], e.g. what an all-to-all of the ranks' best states delivers) into best
 * state `state`: highest SNR, then lowest flat index; a NaN SNR sticks (core.py:230-240). */
int sb_best_merge(sb_plan* plan, int state, int row_lo, int row_hi, int n_cands, const float* snr_c,
                  const float* amp_c, const int32_t* idx_c);

/* Raw region planes for a cross-GPU merge of a fit confidence region (DESIGN §15): *planes_dev points
 * at plane 0 of the plan's region planes, plane p of pixel i (counted over the plan's rows) at
 * [p * rows * nx + i]; *n_planes = 3 + ceil(n_pos / 32) (count, rank_lo, rank_hi, orientation words).
 * Fails without a region sweep since the best state was last allocated. */
int sb_region_planes(sb_plan* plan, int32_t** planes_dev, int* n_planes);

/* Replace the region planes on raster rows row_lo .. row_hi - 1 by the fold of n_cands candidates
 * (device int32 laid out [plane][candidate][row][nx], e.g. what one all-to-all per plane of the
 * ranks' region planes delivers): count summed, rank_lo minimum, rank_hi maximum, orientation words
 * OR-ed.  Replaced, not folded in: the candidates are expected to include this plan's own planes.
 * Rows outside the band are untouched.  Fails for null pointers, n_cands < 1, rows outside the plan
 * and without a region sweep since the best state was last allocated. */
int sb_region_merge(sb_plan* plan, int row_lo, int row_hi, int n_cands, const int32_t* cands_dev);

/* Cross-GPU merge of best states (the parent-side reduce over Pool results,
 * core.py:185, when the search is sharded over ranks).  All buffers are device memory
 * of ny*nx elements owned by the caller (e.g. torch tensors handed to NCCL):
 *   1. sb_best_pack    keys = (SNR bits << 32) | (0xFFFFFFFF - idx)  -> all-reduce MAX (int64)
 *   2. sb_best_select  amp_out = amp where this rank owns the winning key, else 0 -> all-reduce SUM
 *   3. sb_best_unpack  overwrite the plan's best state with the merged result */
int sb_best_pack(sb_plan* plan, unsigned long long* keys_dev);
int sb_best_select(sb_plan* plan, const unsigned long long* gkeys_dev, float* amp_out_dev);
int sb_best_unpack(sb_plan* plan, const unsigned long long* gkeys_dev, const float* amp_dev);

/* core.compare (core.py:198-243) with the reference's exact strict-compare semantics on
 * float64 host planes: folds (amp, age, angle, snr) into best[4][n].  age/angle may be
 * NULL, in which case the scalars age_s / angle_s are used. */
int sb_compare_host(sb_plan* plan, double* best4_host, const double* amp, const double* age,
                    const double* angle, const double* snr, double age_s, double angle_s);

/* DEMGrid._estimate_curvature_noiselevel (dem.py:152-179): sums, over the pixels whose Gaussian
 * window (sigma, truncate as scipy.ndimage.gaussian_filter) holds no NaN, of the high-passed second
 * differences h = d - lowpass(d) and their products -- out10 = [count, hxx, hxy, hyy, hxx^2, hxy^2,
 * hyy^2, hxx hxy, hxx hyy, hxy hyy].  The directional curvature is linear in (dxx, dxy, dyy)
 * (dem.py:103-104), so mean and standard deviation for every direction follow from these. */
int sb_curvature_noise_moments(sb_plan* plan, double sigma, double truncate, double* out10_host);

/* One pass of nodata filling in place of rasterio.fill.fillnodata (dem.py:406-408): NaN cells of
 * the host raster (ny x nx float64) become the inverse-distance-weighted mean of the nearest valid
 * cell along the eight row / column / diagonal rays within max_search_distance cells;
 * *remaining = cells still NaN. */
int sb_fill_nodata(sb_plan* plan, double* dem_host_inout, double max_search_distance, long* remaining);

/* unit-test hook: batched complex64 FFT of length n (power of two, 128..8192) over rows;
 * inverse: bit 0 = inverse transform, bit 1 = use the radix-64 core (n = 4096 only) */
int sb_debug_fft(sb_plan* plan, int n, int rows, const float* in_host, float* out_host, int inverse);

/* developer hook: device time (ms per launch, CUDA events) of the batched FFT kernel alone on
 * resident data; radix64 != 0 selects the 64 x 64 core (n = 4096) */
int sb_debug_fft_bench(sb_plan* plan, int n, int rows, int reps, int radix64, float* ms_per_launch);

/* synchronise the plan's stream */
int sb_sync(sb_plan* plan);

#ifdef __cplusplus
}
#endif
#endif /* SCARPLET_B200_H */
