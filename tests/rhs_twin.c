/*
 * rhs_twin.c — CPU twin of the per-basis arithmetic of libenumgpu's right-hand-side ranging kernel (k_rhs_ranging),
 * for tests/test_rhs_ranges.py only.
 *
 * Compiled with gcc -O2 -ffp-contract=off -march=x86-64-v3, the flags of the CPU oracle (oracle/Makefile): every
 * fma() below is one IEEE-754 fused multiply-add, every other operation a single correctly rounded double operation.
 * tol: eps_piv * max|A_ij| under ENUMGPU_PIVOT_ABSOLUTE, the relative threshold under ENUMGPU_PIVOT_RELATIVE.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#include "enumgpu.h"

static uint64_t binom(int n, int k)
{
    if (k < 0 || n < 0 || k > n) return 0;
    uint64_t r = 1;
    for (int i = 1; i <= k; ++i) r = r * (uint64_t)(n - k + i) / (uint64_t)i;
    return r;
}

/* One basis S (m ascending columns) per DESIGN.md §3.4: W = [A_S | b | e_0 .. e_{m-1}] eliminated as
 * oracle/enumcpu.c eliminates [B | b], every column swept like x; then per row i over k, s = x[k] + eps_feas and
 * v = w_i[k].  Returns 1 if S is singular; else fills lo[i], hi[i], ok[i] (the row counts) and returns 0. */
static int rhs_basis(const enumgpu_problem* p, double eps_feas, int rule, double tol, double eps_opt, const int32_t* S,
                     double* lo, double* hi, int32_t* ok)
{
    const double thr = (rule == ENUMGPU_PIVOT_RELATIVE) ? 0.0 : tol;
    const int m = p->m, lda = p->lda, w = 2 * m + 1;
    double M[ENUMGPU_MAX_M][2 * ENUMGPU_MAX_M + 1], rinv[ENUMGPU_MAX_M], t[ENUMGPU_MAX_M];
    double pmax = 0.0, pmin = INFINITY;
    for (int r = 0; r < m; ++r) {
        for (int j = 0; j < m; ++j) M[r][j] = p->A_colmajor[r + (size_t)S[j] * lda];
        M[r][m] = p->b[r];
        for (int i = 0; i < m; ++i) M[r][m + 1 + i] = (r == i) ? 1.0 : 0.0;
    }
    for (int k = 0; k < m; ++k) {
        int piv = k;
        double best = fabs(M[k][k]);
        for (int r = k + 1; r < m; ++r) {
            double v = fabs(M[r][k]);
            if (v > best) { best = v; piv = r; }
        }
        if (!(best > thr)) return 1;
        if (best > pmax) pmax = best;
        if (best < pmin) pmin = best;
        if (piv != k)
            for (int j = k; j < w; ++j) { double s = M[k][j]; M[k][j] = M[piv][j]; M[piv][j] = s; }
        rinv[k] = 1.0 / M[k][k];
        for (int r = k + 1; r < m; ++r) {
            double l = M[r][k] * rinv[k];
            for (int j = k + 1; j < w; ++j) M[r][j] = fma(-l, M[k][j], M[r][j]);
        }
    }
    if (rule == ENUMGPU_PIVOT_RELATIVE && !(pmin > tol * pmax)) return 1;
    for (int col = m; col < w; ++col) {
        for (int i = 0; i < m; ++i) t[i] = M[i][col];
        for (int k = m - 1; k >= 0; --k) {
            M[k][col] = t[k] * rinv[k];
            for (int i = 0; i < k; ++i) t[i] = fma(-M[i][k], M[k][col], t[i]);
        }
    }
    for (int i = 0; i < m; ++i) {
        double l = -INFINITY, h = INFINITY;
        int good = 1;
        for (int k = 0; k < m; ++k) {
            const double s = M[k][m] + eps_feas, v = M[k][m + 1 + i];
            if (v > eps_opt) {
                const double q = (-s) / v;
                good &= !isnan(q);
                if (q > l) l = q;
            } else if (v < -eps_opt) {
                const double q = s / (-v);
                good &= !isnan(q);
                if (q < h) h = q;
            } else {
                good &= !isnan(v) && s >= 0.0;
            }
        }
        lo[i] = l; hi[i] = h; ok[i] = good && l <= h;
    }
    return 0;
}

/* The m-subsets of J (nJ ascending columns) with ranks r0 .. r0+count-1 in the lexicographic order of C(nJ, m):
 * for subset q, rank[q] its rank among the C(n, m) bases, singular[q], and (if not singular) lo/hi/ok[q*m + i]. */
void rhs_twin_many(const enumgpu_problem* p, double eps_feas, int rule, double tol, double eps_opt, const int32_t* J,
                   int nJ, uint64_t r0, uint64_t count, uint64_t* rank, int32_t* singular, double* lo, double* hi,
                   int32_t* ok)
{
    const int m = p->m, n = p->n;
    int idx[ENUMGPU_MAX_M];
    int32_t S[ENUMGPU_MAX_M];
    uint64_t r = r0;
    for (int i = 0, v = 0; i < m; ++i) {
        for (;;) {
            const uint64_t cnt = binom(nJ - 1 - v, m - 1 - i);
            if (cnt <= r) { r -= cnt; ++v; } else break;
        }
        idx[i] = v++;
    }
    const uint64_t total = binom(n, m);
    for (uint64_t q = 0; q < count; ++q) {
        if (q) {
            int piv = m - 1;
            while (idx[piv] >= nJ - m + piv) --piv;
            ++idx[piv];
            for (int i = piv + 1; i < m; ++i) idx[i] = idx[i - 1] + 1;
        }
        uint64_t acc = 0;
        for (int i = 0; i < m; ++i) {
            S[i] = J[idx[i]];
            acc += binom(n - 1 - S[i], m - i);
        }
        rank[q] = total - 1 - acc;
        singular[q] = rhs_basis(p, eps_feas, rule, tol, eps_opt, S, lo + q * m, hi + q * m, ok + q * m);
    }
}
