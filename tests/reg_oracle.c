/* CPU oracle (plain C) for the regularised window DP -- TEST INFRASTRUCTURE ONLY.
 *
 * The flat sliding-window round of oracle/dp_oracle.c (round_oracle) with SquareSplitter.split_with_normalizations
 * (/root/reference/src/pasio/splitters/square_splitter.py:29-65) as the window's DP, in the reference's operation
 * order per cell:
 *     t = (G[s] - s * Lg[len]) + P_i
 *     t = t - nr[ns_i]          (nr != NULL);  i == 0: t = t + refund          :46-49
 *     t = t - lr[len]           (lr != NULL)                                    :51-54
 *     first arg-max, ns_j = prev_j ? ns[prev_j] + 1 : 0, P_j = t[prev_j] + pen  :56-62
 * nr[k] = lambda_n * f(k + 1), lr[len] = lambda_L * g(len) and refund = lambda_n * f(1) are built by numpy with the
 * reference's expressions.  Checked against tests/reg_oracle.py (numpy, object-faithful) in
 * tests/test_regularized_plans.py.  Build: -ffp-contract=off keeps mul and add un-fused like numpy's ufunc loops.
 */
#include <stdint.h>
#include <stdlib.h>

/* Returns 0, or -1 when a table is too short. */
int dp_oracle_reg(const int64_t *C, const int64_t *L, int64_t N,
                  const double *gtab, int64_t n_gtab, const double *ltab, int64_t n_ltab,
                  int alpha_is_int, double alpha, double pen,
                  const double *nr, int64_t n_nr, double refund, const double *lr, int64_t n_lr,
                  double *P, int64_t *prev, int64_t *ns)
{
    int64_t alpha_i = alpha_is_int ? (int64_t)alpha : 0;
    P[0] = 0.0;
    prev[0] = 0;
    ns[0] = 0;
    for (int64_t j = 1; j < N; ++j) {
        double best = 0.0;
        int64_t arg = -1;
        double shifted_j_real = alpha + (double)C[j];
        int64_t shifted_j_int = alpha_i + C[j];
        for (int64_t i = 0; i < j; ++i) {
            int64_t len = L[j] - L[i];
            int64_t idx;
            double s;
            if (alpha_is_int) {
                idx = shifted_j_int - C[i];
                s = (double)idx;
            } else {
                idx = C[j] - C[i];
                s = shifted_j_real - (double)C[i];
            }
            if (idx < 0 || idx >= n_gtab || len < 0 || len >= n_ltab) return -1;
            double sub = s * ltab[len];
            double self = gtab[idx] - sub;
            double t = self + P[i];
            if (nr) {
                if (ns[i] >= n_nr) return -1;
                t = t - nr[ns[i]];
                if (i == 0) t = t + refund;
            }
            if (lr) {
                if (len >= n_lr) return -1;
                t = t - lr[len];
            }
            /* np.argmax: first maximum; a NaN beats everything and the first NaN wins */
            if (arg < 0 || t > best || (t != t && best == best)) { best = t; arg = i; }
        }
        prev[j] = arg;
        ns[j] = arg != 0 ? ns[arg] + 1 : 0;
        P[j] = best + pen;
    }
    return 0;
}

/* One window of the flat round (as in round_oracle): filter, re-base, DP, mark the path in keep[]. */
static int reg_window(const int64_t *Cg, const uint8_t *cp, const int64_t *cand, int64_t st, int64_t en, int constraint,
                      const double *gtab, int64_t n_gtab, const double *ltab, int64_t n_ltab,
                      int alpha_is_int, double alpha, double pen,
                      const double *nr, int64_t n_nr, double refund, const double *lr, int64_t n_lr,
                      int64_t *C, int64_t *L, int64_t *prev, int64_t *ns, double *P, uint8_t *keep, int64_t *cells)
{
    int64_t first = cand[st], last = cand[en - 1];
    int64_t k = 0;
    int all_zero = (Cg[last] - Cg[first]) == 0;
    for (int64_t q = st; q < en; ++q) {
        int64_t p = cand[q];
        int take;
        if (q == st || q == en - 1) take = 1;
        else if (constraint == 2) take = cp[p] != 0;
        else if (constraint == 1) take = !all_zero;
        else take = 1;
        if (take) {
            L[k] = p - first;
            C[k] = Cg[p] - Cg[first];
            ++k;
        }
    }
    int rc = dp_oracle_reg(C, L, k, gtab, n_gtab, ltab, n_ltab, alpha_is_int, alpha, pen, nr, n_nr, refund, lr, n_lr,
                           P, prev, ns);
    if (rc) return rc;
    *cells += k * (k - 1) / 2;
    int64_t q = k - 1;
    keep[first + L[q]] = 1;
    while (q != 0) { q = prev[q]; keep[first + L[q]] = 1; }
    return 0;
}

/* Arguments as round_oracle (oracle/dp_oracle.c) plus the penalty tables; the windows of the round are spread over
 * n_threads OpenMP threads (each only ORs its survivors into keep[]).  Returns 0, -1 table too short, -2 alloc failure. */
int round_oracle_reg(const int64_t *Cg, const uint8_t *cp, int64_t n,
                     const int64_t *cand, int64_t m,
                     int64_t window_size, int64_t window_shift, int constraint,
                     const double *gtab, int64_t n_gtab, const double *ltab, int64_t n_ltab,
                     int alpha_is_int, double alpha, double pen,
                     const double *nr, int64_t n_nr, double refund, const double *lr, int64_t n_lr,
                     uint8_t *keep, int64_t *cells_out, int n_threads)
{
    int64_t cap = window_size + 1;
    int64_t nwin = (m - 1 + window_shift - 1) / window_shift;
    int64_t cells = 0;
    int rc = 0;
    if (n_threads < 1) n_threads = 1;
    keep[0] = 1;
    keep[n] = 1;
#pragma omp parallel num_threads(n_threads) reduction(+ : cells)
    {
        int64_t *C = (int64_t *)malloc(sizeof(int64_t) * cap);
        int64_t *L = (int64_t *)malloc(sizeof(int64_t) * cap);
        int64_t *prev = (int64_t *)malloc(sizeof(int64_t) * cap);
        int64_t *ns = (int64_t *)malloc(sizeof(int64_t) * cap);
        double *P = (double *)malloc(sizeof(double) * cap);
#pragma omp for schedule(dynamic, 4)
        for (int64_t w = 0; w < nwin; ++w) {
            if (!C || !L || !prev || !ns || !P) { rc = -2; continue; }
            int64_t st = w * window_shift;
            int64_t en = st + window_size + 1;
            if (en > m) en = m;
            int r = reg_window(Cg, cp, cand, st, en, constraint, gtab, n_gtab, ltab, n_ltab, alpha_is_int, alpha, pen,
                               nr, n_nr, refund, lr, n_lr, C, L, prev, ns, P, keep, &cells);
            if (r) rc = r;
        }
        free(C); free(L); free(prev); free(ns); free(P);
    }
    if (cells_out) *cells_out = cells;
    return rc;
}
