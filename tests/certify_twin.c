/*
 * certify_twin.c — CPU twin of libenumgpu's certificate kernel (k_certify), for tests/test_certificate.py only.
 *
 * The test module compiles it with gcc -O2 -ffp-contract=off -march=x86-64-v3, the flags of the CPU oracle
 * (oracle/Makefile): every fma() below is one IEEE-754 fused multiply-add, every other operation a single correctly
 * rounded double operation, so the GPU's certificate can be compared with it bit for bit.
 * tol: eps_piv * max|A_ij| under ENUMGPU_PIVOT_ABSOLUTE, the relative threshold under ENUMGPU_PIVOT_RELATIVE.
 * eps_opt is used as given (no default resolution).
 */
#include <math.h>
#include <string.h>

#include "enumgpu.h"

/* The certificate at one basis (DESIGN.md §3.1), without the fallback to the ray enumeration:
 * W = [B | b | A_0..A_{n-1} | e_0..e_{m-1}] eliminated exactly as oracle/enumcpu.c eliminates [B | b] (same
 * pivot search, threshold, rinv and multipliers l; every extra column receives
 * fma(-l, M[k][j], M[r][j]) in step order), each extra column swept like x, then
 *   r_j = c_j;  r_j = fma(-c[S[k]], u_j[k], r_j)   k = m-1..0
 *   y_i = 0;    y_i = fma(c[S[k]], w_i[k], y_i)    k = m-1..0      (w_i = B^-1 e_i)
 * and the verdict over the nonbasic j in index order (rk_j = maximize ? -r_j : r_j):
 *   UNBOUNDED at the lowest j with rk_j < -eps_opt and every u_j[k] <= eps_opt,
 *   else OPTIMAL if no rk_j < -eps_opt and no rk_j is NaN, else UNDECIDED.
 * Fills out (status, basis_class, entering, m, n, objective, y, reduced_cost, x_B, ray); returns
 * ENUMGPU_OK or ENUMGPU_ERR_ARG for a singular or infeasible basis. */
int certify_twin(const enumgpu_problem* p, double eps_feas, int rule, double tol, double eps_opt,
                 const int32_t* S, enumgpu_certificate* out)
{
    const double thr = (rule == ENUMGPU_PIVOT_RELATIVE) ? 0.0 : tol;
    const int m = p->m, n = p->n, lda = p->lda, w = 2 * m + n + 1;
    double pmax = 0.0, pmin = INFINITY;
    double M[ENUMGPU_MAX_M][2 * ENUMGPU_MAX_M + ENUMGPU_MAX_N + 1];
    double rinv[ENUMGPU_MAX_M], t[ENUMGPU_MAX_M];
    memset(out, 0, sizeof *out);
    out->m = m; out->n = n; out->entering = -1;
    for (int r = 0; r < m; ++r) {
        for (int j = 0; j < m; ++j) M[r][j] = p->A_colmajor[r + (size_t)S[j] * lda];
        M[r][m] = p->b[r];
        for (int j = 0; j < n; ++j) M[r][m + 1 + j] = p->A_colmajor[r + (size_t)j * lda];
        for (int i = 0; i < m; ++i) M[r][m + 1 + n + i] = (r == i) ? 1.0 : 0.0;
    }
    for (int k = 0; k < m; ++k) {
        int piv = k;
        double best = fabs(M[k][k]);
        for (int r = k + 1; r < m; ++r) {
            double v = fabs(M[r][k]);
            if (v > best) { best = v; piv = r; }
        }
        if (!(best > thr)) { out->basis_class = ENUMGPU_BASIS_SINGULAR; out->status = ENUMGPU_CERT_UNDECIDED; return ENUMGPU_ERR_ARG; }
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
    if (rule == ENUMGPU_PIVOT_RELATIVE && !(pmin > tol * pmax)) {
        out->basis_class = ENUMGPU_BASIS_SINGULAR; out->status = ENUMGPU_CERT_UNDECIDED; return ENUMGPU_ERR_ARG;
    }
    /* every column right of B, x included: u = column sweep */
    for (int col = m; col < w; ++col) {
        for (int i = 0; i < m; ++i) t[i] = M[i][col];
        for (int k = m - 1; k >= 0; --k) {
            M[k][col] = t[k] * rinv[k];
            for (int i = 0; i < k; ++i) t[i] = fma(-M[i][k], M[k][col], t[i]);
        }
    }
    int feasible = 1;
    double z = 0.0;
    for (int k = 0; k < m; ++k) {
        out->x_B[k] = M[k][m];
        if (!(M[k][m] >= -eps_feas)) feasible = 0;
    }
    for (int k = m - 1; k >= 0; --k) z = fma(p->c[S[k]], M[k][m], z);
    out->objective = z;
    out->basis_class = feasible ? ENUMGPU_BASIS_FEASIBLE : ENUMGPU_BASIS_INFEASIBLE;
    for (int j = 0; j < n; ++j) {
        double r = p->c[j];
        for (int k = m - 1; k >= 0; --k) r = fma(-p->c[S[k]], M[k][m + 1 + j], r);
        out->reduced_cost[j] = r;
    }
    for (int i = 0; i < m; ++i) {
        double y = 0.0;
        for (int k = m - 1; k >= 0; --k) y = fma(p->c[S[k]], M[k][m + 1 + n + i], y);
        out->y[i] = y;
    }
    if (!feasible) { out->status = ENUMGPU_CERT_UNDECIDED; return ENUMGPU_ERR_ARG; }
    int improving = 0, nan = 0;
    for (int j = 0; j < n; ++j) {
        int basic = 0;
        for (int k = 0; k < m; ++k) basic |= (S[k] == j);
        if (basic) continue;
        const double rk = p->maximize ? -out->reduced_cost[j] : out->reduced_cost[j];
        if (isnan(rk)) { nan = 1; continue; }
        if (!(rk < -eps_opt)) continue;
        improving = 1;
        if (out->entering >= 0) continue;
        int ray = 1;
        for (int k = 0; k < m; ++k) ray &= (M[k][m + 1 + j] <= eps_opt);
        if (ray) out->entering = j;
    }
    if (out->entering >= 0) {
        for (int k = 0; k < m; ++k) out->ray[S[k]] = -M[k][m + 1 + out->entering];
        out->ray[out->entering] = 1.0;
        out->status = ENUMGPU_CERT_UNBOUNDED;
    } else {
        out->status = (!improving && !nan) ? ENUMGPU_CERT_OPTIMAL : ENUMGPU_CERT_UNDECIDED;
    }
    return ENUMGPU_OK;
}
