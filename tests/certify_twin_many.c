/*
 * certify_twin_many.c — the CPU twin of k_certify (tests/certify_twin.c) over many bases, for
 * tests/test_optimal_duals.py only: it is linked with certify_twin.c and built with the same flags.
 * bases[i*m .. i*m+m) is basis i; out[i] receives its certificate (without the ray fallback) and rc[i] the twin's
 * return value.  Returns the number of OPTIMAL certificates among the feasible bases.
 */
#include <stdint.h>

#include "enumgpu.h"

int certify_twin(const enumgpu_problem* p, double eps_feas, int rule, double tol, double eps_opt,
                 const int32_t* S, enumgpu_certificate* out);

uint64_t certify_twin_many(const enumgpu_problem* p, double eps_feas, int rule, double tol, double eps_opt,
                           const int32_t* bases, uint64_t count, int32_t* rc, enumgpu_certificate* out)
{
    uint64_t n_optimal = 0;
    for (uint64_t i = 0; i < count; ++i) {
        rc[i] = certify_twin(p, eps_feas, rule, tol, eps_opt, bases + i * (uint64_t)p->m, out + i);
        n_optimal += (rc[i] == ENUMGPU_OK && out[i].status == ENUMGPU_CERT_OPTIMAL);
    }
    return n_optimal;
}
