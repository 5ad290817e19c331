/*
 * CPU ORACLE of the likelihood surface (test infrastructure, not product code): for every (centre, A, xa)
 * the literal T of calcBaller, /root/reference/BalLeRMix+_v1.py:436-507 ("v1"), before any maximum is taken,
 *   alpha_i = exp(-A*|g_i - t|)                                       v1:446,454
 *   used: lo <= i <= hi, alpha_i >= 1e-8, g_i != t                    v1:455-457
 *   T = 2*(sum log(alpha_i*SP[xa][c_i] + (1 - alpha_i)*G[c_i]) - sum log G[c_i])     v1:492-499
 * with the site selection of oracle/oracle_c.c (the same binary-search cut on sorted input) and the same
 * compensated (Neumaier) sums.  An A without sites (v1:458) gets T = -inf at every grid point.
 *
 *   S[j][iA][xa], ns[j][iA]; OpenMP over (centre, A), n_threads <= 0: all available.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct { double s, c; } ksum;
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

int oracle_surface(int64_t n_sites, const double *genpos, const int32_t *cls, int32_t n_classes,
                   const double *G, const double *SP, int32_t n_xa, int32_t n_A, const double *A,
                   int64_t n_centres, const double *t, const int64_t *lo, const int64_t *hi,
                   double *S, int32_t *ns, int32_t n_threads) {
    int sorted = 1;
    for (int64_t i = 1; i < n_sites; ++i)
        if (!(genpos[i] >= genpos[i - 1])) { sorted = 0; break; }
    double *logG = (double *)malloc(sizeof(double) * (n_classes > 0 ? n_classes : 1));
    if (!logG) return -1;
    for (int c = 0; c < n_classes; ++c) logG[c] = log(G[c]);
    int err = 0;
    const int64_t n_tasks = n_centres * (int64_t)n_A;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel
    {
        int64_t cap = n_sites > 0 ? n_sites : 1;
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
                    double v = exp(-a * fabs(genpos[i] - tj));
                    if (v >= 1e-8 && genpos[i] != tj) {
                        al[m] = v; cc[m] = cls[i]; ksum_add(&neut, logG[cls[i]]); ++m;
                    }
                }
                const double cl_neut = neut.s + neut.c;
                double *row = S + (size_t)task * n_xa;
                for (int xa = 0; xa < n_xa; ++xa) {
                    if (m == 0) { row[xa] = -INFINITY; continue; }
                    const double *sp = SP + (size_t)xa * n_classes;
                    ksum sel = {0.0, 0.0};
                    for (int64_t k = 0; k < m; ++k)
                        ksum_add(&sel, log(al[k] * sp[cc[k]] + (1. - al[k]) * G[cc[k]]));
                    row[xa] = 2 * ((sel.s + sel.c) - cl_neut);
                }
                ns[task] = (int32_t)m;
            }
        }
        free(al); free(cc);
    }
    free(logG);
    return err ? -1 : 0;
}
