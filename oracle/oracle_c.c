/*
 * CPU ORACLE (test infrastructure, not product code) -- plain C restatement of
 * calcBaller, /root/reference/BalLeRMix+_v1.py:436-507 ("v1").
 *
 * Only tests/, __graft_entry__.smoke() and bench.py (cpu_baseline / --impl reference)
 * may load this library.  The product (ballermixplus_b200/) never does.
 * PARITY PINNED: tests/test_oracle_golden.py checks it against the numpy oracle and,
 * through it, against the reference's golden scans.
 *
 * The arithmetic is the reference's, term for term, in the literal form:
 *   alpha_i = exp(-A*|g_i - t|)                                       v1:446,454
 *   used: lo <= i <= hi, alpha_i >= 1e-8, g_i != t                    v1:455-457
 *   mix_i = alpha_i*SP[xa][c_i] + (1 - alpha_i)*G[c_i]                v1:492-494
 *   T = 2*(sum log mix_i - sum logG[c_i])                             v1:496-499
 *   first strict maximum over A (outer), xa (inner) from T = 0        v1:451,501
 * Per-site table reads go through the site's (k, n) class, which is what the
 * per-site arrays of the reference hold.  When genpos is sorted the scan over
 * sites starts from a binary search instead of touching all N sites per A
 * (v1:446-455 masks all N; the selected set is the same).  The two sums are
 * compensated (Neumaier): the reference's np.sum is pairwise (error ~1e-12 on
 * a 20 000-site window) whereas a plain sequential loop drifts by ~3e-9 there,
 * more than the parity bar; the compensated sum is exact to an ulp of the result.
 *
 * Threads: OpenMP over (centre, A) tasks (n_threads <= 0: all available).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct { double s, c; } ksum;               /* Neumaier compensated accumulator */
static inline void ksum_add(ksum *k, double v) {
    double t = k->s + v;
    if (isfinite(t)) {                              /* an inf or nan sum is the sum: log(0) = -inf stays -inf */
        if (fabs(k->s) >= fabs(v)) k->c += (k->s - t) + v; else k->c += (v - t) + k->s;
    }
    k->s = t;
}

static int64_t lower_bound(const double *a, int64_t n, double key) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

/* t_floor: the value a grid point must beat to be reported -- 0 in the reference (v1:451); -inf reports the
 * best grid point of every centre whatever its sign (parity checks on neutral data, where most maxima are <= 0). */
int oracle_scan_floor(int64_t n_sites, const double *genpos, const int32_t *cls, int32_t n_classes,
                      const double *G, const double *SP, int32_t n_xa, int32_t n_A, const double *A,
                      int64_t n_centres, const double *t, const int64_t *lo, const int64_t *hi,
                      double *oT, int32_t *oiA, int32_t *oixa, int32_t *ons, int32_t n_threads,
                      uint64_t *site_pairs, double t_floor) {
    int sorted = 1;
    for (int64_t i = 1; i < n_sites; ++i)
        if (!(genpos[i] >= genpos[i - 1])) { sorted = 0; break; }
    double *logG = (double *)malloc(sizeof(double) * (n_classes > 0 ? n_classes : 1));
    if (!logG) return -1;
    for (int c = 0; c < n_classes; ++c) logG[c] = log(G[c]);          /* v1:299 */
    uint64_t pairs_total = 0;
    int err = 0;
    const int64_t n_tasks = n_centres * (int64_t)n_A;          /* one task per (centre, A) */
    double *cT = (double *)malloc(sizeof(double) * (n_tasks > 0 ? n_tasks : 1));
    int32_t *cxa = (int32_t *)malloc(sizeof(int32_t) * (n_tasks > 0 ? n_tasks : 1));
    int32_t *cns = (int32_t *)malloc(sizeof(int32_t) * (n_tasks > 0 ? n_tasks : 1));
    if (!cT || !cxa || !cns) { free(cT); free(cxa); free(cns); free(logG); return -1; }
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel reduction(+ : pairs_total)
    {
        int64_t cap = 1 << 16;                       /* per-thread scratch, grown on demand */
        double *al = (double *)malloc(sizeof(double) * cap);
        int32_t *cc = (int32_t *)malloc(sizeof(int32_t) * cap);
        if (!al || !cc) {
#pragma omp atomic write
            err = 1;
        } else {
#pragma omp for schedule(dynamic, 1)
            for (int64_t task = 0; task < n_tasks; ++task) {
                const int64_t j = task / n_A;
                const int iA = (int)(task % n_A);
                const double tj = t[j];
                const double a = A[iA];
                int64_t s0 = lo[j] < 0 ? 0 : lo[j];
                int64_t s1 = hi[j] > n_sites - 1 ? n_sites - 1 : hi[j];
                if (sorted && a > 0) {
                    double r = 18.420680743952367 / a * (1.0 + 1e-9);
                    int64_t q0 = lower_bound(genpos, n_sites, tj - r);
                    int64_t q1 = lower_bound(genpos, n_sites, tj + r * (1.0 + 1e-9) + 1e-300);
                    if (q0 > s0) s0 = q0;
                    if (q1 < s1) s1 = q1;
                }
                int64_t m = 0;
                ksum neut = {0.0, 0.0};
                for (int64_t i = s0; i <= s1 && i < n_sites; ++i) {
                    double v = exp(-a * fabs(genpos[i] - tj));           /* v1:446,454 */
                    if (v >= 1e-8 && genpos[i] != tj) {                  /* v1:455 */
                        if (m == cap) {
                            double *al2 = (double *)realloc(al, sizeof(double) * cap * 2);
                            if (al2) al = al2;
                            int32_t *cc2 = (int32_t *)realloc(cc, sizeof(int32_t) * cap * 2);
                            if (cc2) cc = cc2;
                            if (!al2 || !cc2) {
#pragma omp atomic write
                                err = 1;
                                break;
                            }
                            cap *= 2;
                        }
                        al[m] = v; cc[m] = cls[i]; ksum_add(&neut, logG[cls[i]]); ++m;   /* v1:497 */
                    }
                }
                pairs_total += (uint64_t)m;
                const double cl_neut = neut.s + neut.c;
                double bT = t_floor;
                int bxa = -1;
                if (m > 0) {                                             /* v1:458 */
                    for (int xa = 0; xa < n_xa; ++xa) {
                        const double *sp = SP + (size_t)xa * n_classes;
                        ksum sel = {0.0, 0.0};
                        for (int64_t k = 0; k < m; ++k)                  /* v1:494-496 */
                            ksum_add(&sel, log(al[k] * sp[cc[k]] + (1. - al[k]) * G[cc[k]]));
                        double T = 2 * ((sel.s + sel.c) - cl_neut);      /* v1:499 */
                        if (T > bT) { bT = T; bxa = xa; }                /* v1:501 within this A */
                    }
                }
                cT[task] = bT; cxa[task] = bxa; cns[task] = (int32_t)m;
            }
        }
        free(al); free(cc);
    }
    /* v1:453,501: A in visiting order, strict '>' from Tmax = 0 */
    for (int64_t j = 0; j < n_centres; ++j) {
        double bT = t_floor;
        int bA = -1, bxa = -1, bns = 0;
        for (int iA = 0; iA < n_A; ++iA) {
            const int64_t task = j * n_A + iA;
            if (cxa[task] >= 0 && cT[task] > bT) { bT = cT[task]; bA = iA; bxa = cxa[task]; bns = cns[task]; }
        }
        oT[j] = bA >= 0 ? bT : 0.0; oiA[j] = bA; oixa[j] = bxa; ons[j] = bns;
    }
    free(cT); free(cxa); free(cns);
    free(logG);
    if (site_pairs) *site_pairs = pairs_total;
    return err ? -1 : 0;
}

int oracle_scan(int64_t n_sites, const double *genpos, const int32_t *cls, int32_t n_classes,
                const double *G, const double *SP, int32_t n_xa, int32_t n_A, const double *A,
                int64_t n_centres, const double *t, const int64_t *lo, const int64_t *hi,
                double *oT, int32_t *oiA, int32_t *oixa, int32_t *ons, int32_t n_threads,
                uint64_t *site_pairs) {
    return oracle_scan_floor(n_sites, genpos, cls, n_classes, G, SP, n_xa, n_A, A, n_centres, t, lo, hi,
                             oT, oiA, oixa, ons, n_threads, site_pairs, 0.0);
}

int oracle_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
