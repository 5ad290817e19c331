/*
 * blmx.h -- C ABI of the B200-native BalLeRMix+ composite-likelihood-ratio scan.
 *
 * The reference (bioXiaoheng/BallerMixPlus, BalLeRMix+_v1.py, "v1") has no FFI or
 * plugin interface; its only internal seam is the Python function
 *
 *     calcBaller(window_indice, testSite, InputData, NeutralSFS,
 *                NormalizedBetaBinom, Grids) -> [T, x, a, A, nSites]     (v1:436-507)
 *
 * called once per test centre by the four Scan drivers (v1:539,573,590,606).
 * This library is the batch form of that seam: all per-run state the function
 * reads (InputData.genPos, NeutralSFS.probs/propSizes, NormalizedBetaBinom.normProbs,
 * Grids.A/x/abeta) is loaded once as a "problem"; a scan call takes a batch of
 * (testSite, window) pairs and returns, per centre, the reference's Tmax row.
 *
 * Conventions
 *   - plain C types, caller owns every host buffer, the library keeps no host
 *     pointer after a call returns;
 *   - every function returns 0 on success or a negative blmx_status; the message
 *     is available from blmx_last_error() (thread-local); nothing throws or exits;
 *   - one scan may be in flight per handle; handles are independent;
 *   - there is NO CPU fallback: without a CUDA device every entry point that
 *     computes returns BLMX_ERR_CUDA.
 */
#ifndef BLMX_H
#define BLMX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BLMX_ABI_VERSION 2

typedef enum {
    BLMX_OK = 0,
    BLMX_ERR_ARG = -1,      /* null pointer, negative size, class index out of range ... */
    BLMX_ERR_CUDA = -2,     /* CUDA runtime error (message has the cudaError string)       */
    BLMX_ERR_STATE = -3,    /* scan before load, etc.                                       */
    BLMX_ERR_NOMEM = -4
} blmx_status;

/*
 * One sequence (chromosome) and one statistic's tables.
 *
 *   genpos[i]   InputData.genPos (v1:103,124), the order of the input file.
 *   cls[i]      index of site i's (k, n) class, 0 <= cls[i] < n_classes.
 *   G[c]        NeutralSFS.probs for class c = g(k, n)            (v1:292)
 *   SP[xa][c]   NormalizedBetaBinom.get(x, a) * NeutralSFS.propSizes for class c
 *               (v1:479,492), xa = ix * n_a + ia, with x and a in the ORDER THE
 *               REFERENCE VISITS THEM (iteration order of set(Grids.x), set(Grids.abeta),
 *               v1:473-474).
 *   A[iA]       set(Grids.A) in visiting order                    (v1:453)
 *
 * Exact ties are resolved as the reference resolves them: the first grid point
 * in visiting order (A outer, x, a inner) with the maximal T wins (strict '>',
 * v1:501).
 */
typedef struct {
    int64_t        n_sites;
    const double  *genpos;     /* [n_sites]            */
    const int32_t *cls;        /* [n_sites]            */
    int32_t        n_classes;
    const double  *G;          /* [n_classes]          */
    const double  *SP;         /* [n_x*n_a][n_classes] */
    int32_t        n_x;
    int32_t        n_a;
    int32_t        n_A;
    const double  *A;          /* [n_A]                */
} blmx_problem;

/*
 * Per-centre results, the reference's Tmax = [T, x, a, A, nSites] (v1:451,502)
 * with grid values replaced by their visiting-order indices.
 * No grid point with T > 0  =>  T = 0, iA = ix = ia = -1, nsites = 0
 * (the reference's all-zero row, v1:451).
 */
typedef struct {
    double  *T;        /* [n_centres] CLR = 2*(sum log mix - sum log g)   (v1:499) */
    int32_t *iA;       /* [n_centres] index into problem.A                         */
    int32_t *ix;       /* [n_centres] index into the x visiting order              */
    int32_t *ia;       /* [n_centres] index into the a visiting order              */
    int32_t *nsites;   /* [n_centres] len(subwindow_indice) of the winning A (v1:502) */
} blmx_result;

typedef struct blmx_handle blmx_handle;

int         blmx_abi_version(void);
const char *blmx_last_error(void);
int         blmx_device_count(int *count);

/* Create / destroy a handle bound to one CUDA device. */
int blmx_create(int device, blmx_handle **out);
int blmx_destroy(blmx_handle *h);

/* Copy a problem to the device (H2D) and build the class-sorted site layout.
 * Replaces any problem previously loaded on this handle. */
int blmx_load(blmx_handle *h, const blmx_problem *p);

/*
 * blmx_load for a problem made of several sequences laid end to end (for example the neutral replicates of
 * an empirical null).  Segment s is the site range [seg_start[s], seg_start[s+1]) (the last one ends at
 * n_sites); seg_start[0] == 0, the starts strictly increase and each is < n_sites, n_segments >= 1, else
 * BLMX_ERR_ARG.  Segments only say where genpos is non-decreasing: the sites a centre uses are exactly those
 * of blmx_scan's definition.  A window [lo, hi] inside one segment gets the fast paths of a sorted sequence
 * (distance cut, far field, pruning); a window that crosses a segment boundary is legal and exact, and is
 * evaluated like a window of unsorted input.  If any segment is not non-decreasing (or holds NaN), the whole
 * problem is treated as unsorted, as blmx_load treats such input.  n_segments == 1 is blmx_load.
 */
int blmx_load_segmented(blmx_handle *h, const blmx_problem *p, int64_t n_segments, const int64_t *seg_start);

/*
 * Scan a batch of centres; HOST buffers in and out (H2D of the centre arrays,
 * kernels, D2H of the results, synchronous).  For centre j the sites used are
 * those with lo[j] <= i <= hi[j] (window_indice, inclusive), exp(-A*|genpos[i]-t[j]|)
 * >= 1e-8 and genpos[i] != t[j]                                   (v1:454-457).
 */
int blmx_scan(blmx_handle *h, int64_t n_centres, const double *t, const int64_t *lo,
              const int64_t *hi, const blmx_result *out);

/*
 * Same, DEVICE buffers in and out, asynchronous on `cuda_stream` (a cudaStream_t,
 * NULL = the legacy default stream).  No host synchronisation is performed.
 */
int blmx_scan_device(blmx_handle *h, int64_t n_centres, const double *d_t, const int64_t *d_lo,
                     const int64_t *d_hi, const blmx_result *d_out, void *cuda_stream);

/*
 * The likelihood surface and its profiles.
 *
 * The surface of centre j is T(A, x, a) = 2*(sum log mix - sum log g) (v1:499) at every grid point, the value
 * the maximum of the rows is taken over.  An A with no site in the window (nsites = 0, which the reference
 * skips, v1:458) has T = -inf at every grid point.  T may be NaN or -inf where the tables make it so.
 *
 * The profiles of centre j are maxima of its surface over all but one grid axis, over the A with sites only:
 *   TA[j][iA] = max over (x, a),   Tx[j][ix] = max over (A, a),   Ta[j][ia] = max over (A, x),
 * and nsA[j][iA] = sites used at A.  NaN never wins a maximum (the strict '>' of v1:501); an entry with
 * nothing to take is -inf.  Profiles do not depend on option "report_all": they are never clamped at 0.
 * Indices are visiting-order indices, as in blmx_result; every array is row-major per centre, centres in the
 * order of the call.
 *
 * Both calls take HOST buffers and are synchronous, like blmx_scan.  The library stages the surface through
 * device scratch of at most 1 GiB per launch (fewer centres per launch than option "batch" when n_A*n_x*n_a
 * is large).
 */
typedef struct {
    double  *TA;       /* [n_centres][n_A] */
    double  *Tx;       /* [n_centres][n_x] */
    double  *Ta;       /* [n_centres][n_a] */
    int32_t *nsA;      /* [n_centres][n_A] */
} blmx_profile;

/* blmx_scan plus the profiles: `out` gets exactly what blmx_scan writes (report_all included). */
int blmx_scan_profile(blmx_handle *h, int64_t n_centres, const double *t, const int64_t *lo,
                      const int64_t *hi, const blmx_result *out, const blmx_profile *prof);

/* The full surface of a few centres (for plots and tests): S[j][iA][ix*n_a + ia], nsA[j][iA]. */
int blmx_scan_surface(blmx_handle *h, int64_t n_centres, const double *t, const int64_t *lo,
                      const int64_t *hi, double *S, int32_t *nsA);

/*
 * Local grid refinement (DESIGN.md §3.10): the best point of a finer grid inside a box around each centre's
 * coarse maximum.  The fine grid is given by axes, not by the problem's grid: n_fA fine A values, and n_fx x
 * n_fa fine (x, a) points of which only those that some box needs have a class row.
 *
 * blmx_load_refine loads the fine tables for the problem already on the handle (else BLMX_ERR_STATE):
 *   fA[i]                 fine A values
 *   row_of[ix*n_fa + ia]  row of SP for fine point (ix, ia), or -1 where no box may go
 *   SP[row][c]            NormalizedBetaBinom probabilities * propSizes at that point (as blmx_problem.SP)
 * R = SP/G is formed with the G of the loaded problem, as blmx_load forms it.  The next blmx_load or
 * blmx_load_segmented drops the fine tables.
 *
 * blmx_refine takes, per centre, the window of blmx_scan and box[j][6] = fA0, fA1, fx0, fx1, fa0, fa1, inclusive
 * ranges of fine indices.  Every point of every box must have a row, a box may hold at most 17 x 17 (x, a)
 * points, and no range may be empty or leave its axis (else BLMX_ERR_ARG).  The result, in fine indices, is the
 * box maximum: visiting order fine A, then fine x, then fine a, strict '>' starting from -inf (NaN never wins),
 * an A without sites skipped; T = -inf and -1 indices where nothing qualifies.  There is no far field and no
 * pruning: every site of the window is multiplied in at every point.  HOST buffers, synchronous.
 */
int blmx_load_refine(blmx_handle *h, int64_t n_fA, const double *fA, int64_t n_fx, int64_t n_fa, int64_t n_rows,
                     const int32_t *row_of, const double *SP);
int blmx_refine(blmx_handle *h, int64_t n_centres, const double *t, const int64_t *lo, const int64_t *hi,
                const int32_t *box, const blmx_result *out);

/* One-shot form of the seam: create + load + scan + destroy on `device`. */
int blmx_scan_oneshot(int device, const blmx_problem *p, int64_t n_centres, const double *t,
                      const int64_t *lo, const int64_t *hi, const blmx_result *out);

/*
 * Options (before or after load):
 *   "group"      1 = one FMA+MUL per site-evaluation; 4 = sites are folded four at a time into a
 *                quartic in R = SP/G with non-negative coefficients (default, see DESIGN.md)
 *   "farfield"   1 (default) = sites of a class with alpha*max|D| <= 1/4 (D = SP/G - 1) contribute
 *                through power sums of alpha (series of log(1 + alpha D), truncation < 2^-70 per
 *                site), taken from per-block moments that blmx_load precomputes (the value at the
 *                time of blmx_load decides whether they are built); 0 = every site is evaluated
 *                per grid point
 *   "report_all" 0 (default) = the reference's rule, only a grid point with T > 0 is reported (v1:451,501);
 *                1 = diagnostic: the best grid point is reported whatever the sign of T (the maximum
 *                starts from -inf instead of 0), so that parity checks on neutral data compare a real
 *                T and argmax on every centre instead of the all-zero row
 *   "batch"      centres per kernel launch (scratch = batch * n_A * 16 bytes)
 *   "timing"     1 = record CUDA events around every scan kernel (see blmx_last_kernel_ms)
 *   "prune"      1 (default) = before the scan kernel, prove from an upper bound on T which (centre, A) items
 *                have T <= 0 at every grid point and skip their exact evaluation (their candidate is the
 *                all-zero one whatever their exact T, so the rows do not change); 0 = evaluate every item.
 *                Only the default scan prunes: not with report_all, surfaces or profiles, group 1,
 *                farfield 0, unsorted positions or class rows with inf/nan (nor items whose window crosses
 *                a segment boundary of blmx_load_segmented)
 */
int blmx_set_option(blmx_handle *h, const char *name, int64_t value);

/*
 * Counters of the most recent blmx_scan / blmx_scan_device on this handle
 * (valid after the stream has been synchronised):
 *   site_pairs    sum over (centre, A) of the number of sites used (the realised sum of W)
 *   single_pairs  how many of those were evaluated one site at a time (the rest four at a time)
 *   launches      kernel launches issued
 */
int blmx_last_counters(blmx_handle *h, uint64_t *site_pairs, uint64_t *single_pairs,
                       uint64_t *launches);
/* All work counters (blmx_refine resets them and counts [5] only): [0] site_pairs, [1] single_pairs, [2] far-field block visits (one exp and
 * one DFMA on each of 32 lanes), [3] far-field polynomial terms summed over class visits (one DFMA
 * per term and grid point), [4] site pairs that entered through the far field, [5] index-range
 * violations (always 0; counted only by the -DBLMX_CHECKED build the tests run), [6] of [4], the
 * sites of block remainders summed one by one, [7] quartics evaluated (each covers up to four
 * sites on every grid point). */
int blmx_last_counters6(blmx_handle *h, uint64_t *six, uint64_t *launches);
int blmx_last_counters8(blmx_handle *h, uint64_t *eight, uint64_t *launches);
/* [0..7] as blmx_last_counters8, [8] items proved T <= 0 everywhere and skipped (option "prune"); their sites
 * are counted in [0] and, as they are not multiplied in per grid point, also in [4]. */
int blmx_last_counters9(blmx_handle *h, uint64_t *nine, uint64_t *launches);

/* Far-field layout of the loaded problem: whole blocks, sites per block, bytes of block moments
 * resident on the device (0 blocks: every site is evaluated directly). */
int blmx_problem_info(blmx_handle *h, int64_t *far_blocks, int64_t *far_block_sites, int64_t *moment_bytes);

/*
 * With option "timing" = 1 the library records a CUDA event pair around every scan-kernel
 * launch on the launching stream; this returns their summed duration for the most recent
 * scan (synchronises on the last event).
 */
int blmx_last_kernel_ms(blmx_handle *h, double *total_ms, int64_t *n_launches);

/* Sustained FP64 FMA rate of `device`, measured with a register-resident DFMA
 * loop for about `seconds`; result in TFLOP/s (FMA = 2 flop). */
int blmx_measure_fp64_peak(int device, double seconds, double *tflops, double *sm_mhz_est);

#ifdef __cplusplus
}
#endif
#endif /* BLMX_H */
