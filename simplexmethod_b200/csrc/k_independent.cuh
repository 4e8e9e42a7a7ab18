// k_independent.cuh — ENUMGPU_ALGO_INDEPENDENT: one thread = one basis at a
// time, one complete partial-pivot GE per basis, everything in registers.
//
// This is the literal form of the hot loop of SURVEY §3.3 (gather as
// Canonical.cpp:183-187, solve, feasibility Canonical.cpp:165-177, objective
// Canonical.cpp:79-87).  It exists as (a) the first-principles kernel the
// shared-prefix kernel is checked against on the device, and (b) the kernel
// whose FP64-pipe utilisation is the "one LU per basis" roofline figure.
//
// A, b, c and the binomial table are staged once per CTA in shared memory.
// A thread owns a contiguous chunk of ranks: it unranks the first subset with
// the combinatorial number system and then steps with next-combination, so
// 64-bit integer work is O(1) per basis.  All register arrays are indexed
// with compile-time constants only (full unrolling); the dynamic pivot row is
// handled with predicated selects.
#pragma once

#include "enum_common.cuh"

namespace enumgpu {

constexpr int kIndepThreads = 128;

// x[] and key of one basis; returns 0 feasible, 1 infeasible, 2 singular.
template <int M>
__device__ __forceinline__ int eval_basis_regs(const double* __restrict__ sA,   // [n][M] packed columns
                                               const double* __restrict__ sb,
                                               const double* __restrict__ sc,
                                               const int (&S)[M], double thr, double eps_feas,
                                               double& z_out, double (&x)[M])
{
    double Mx[M][M + 1];
    double rinv[M];
    bool singular = false;   // no early exit inside the elimination (keeps it branch-free)
    static_for<0, M>([&](auto j_) {
        constexpr int j = decltype(j_)::value;
        const double* col = sA + S[j] * M;
        static_for<0, M>([&](auto r_) { constexpr int r = decltype(r_)::value; Mx[r][j] = col[r]; });
    });
    static_for<0, M>([&](auto r_) { constexpr int r = decltype(r_)::value; Mx[r][M] = sb[r]; });

    static_for<0, M>([&](auto k_) {
        constexpr int k = decltype(k_)::value;
        // first maximum of |column k| over rows k..M-1
        int p = k;
        double best = fabs(Mx[k][k]);
        static_for<k + 1, M>([&](auto r_) {
            constexpr int r = decltype(r_)::value;
            const double v = fabs(Mx[r][k]);
            const bool g = v > best;
            best = g ? v : best;
            p = g ? r : p;
        });
        singular |= !(best > thr);
        // swap rows k and p (columns k..M); p is data dependent -> selects
        static_for<k + 1, M>([&](auto r_) {
            constexpr int r = decltype(r_)::value;
            const bool sw = (p == r);
            static_for<k, M + 1>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                const double a = Mx[k][j], bb = Mx[r][j];
                Mx[k][j] = sw ? bb : a;
                Mx[r][j] = sw ? a : bb;
            });
        });
        rinv[k] = __drcp_rn(Mx[k][k]);
        static_for<k + 1, M>([&](auto r_) {
            constexpr int r = decltype(r_)::value;
            const double l = __dmul_rn(Mx[r][k], rinv[k]);
            static_for<k + 1, M + 1>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                Mx[r][j] = fnma(l, Mx[k][j], Mx[r][j]);
            });
        });
    });
    if (singular) return 2;
    // column-sweep back substitution on t = last column
    bool infeasible = false;
    double z = 0.0;
    static_rfor<0, M>([&](auto j_) {
        constexpr int j = decltype(j_)::value;
        x[j] = __dmul_rn(Mx[j][M], rinv[j]);
        infeasible |= !(x[j] >= -eps_feas);
        static_for<0, j>([&](auto i_) {
            constexpr int i = decltype(i_)::value;
            Mx[i][M] = fnma(Mx[i][j], x[j], Mx[i][M]);
        });
        z = __fma_rn(sc[S[j]], x[j], z);
    });
    z_out = z;
    return infeasible ? 1 : 0;
}

// lexicographic successor with static indexing; n - M + i is the max of S[i]
template <int M>
__device__ __forceinline__ void next_subset_regs(int (&S)[M], int n)
{
    int pos = -1, base = 0;
#pragma unroll
    for (int i = 0; i < M; ++i) {
        const bool can = S[i] < n - M + i;
        pos = can ? i : pos;
        base = can ? S[i] + 1 : base;
    }
#pragma unroll
    for (int j = 0; j < M; ++j) S[j] = (j < pos) ? S[j] : base + (j - pos);
}

template <int M>
__global__ void __launch_bounds__(kIndepThreads)
k_independent(const LaunchParams prm, BlockPartial* __restrict__ partials)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = prm.n;
    double*   sA = reinterpret_cast<double*>(smem_raw);          // n*M
    double*   sb = sA + n * M;                                    // M
    double*   sc = sb + M;                                        // n
    uint64_t* sbin = reinterpret_cast<uint64_t*>(sc + n);         // kBinomRows*kBinomCols

    for (int idx = threadIdx.x; idx < n * M; idx += kIndepThreads) {
        const int j = idx / M, r = idx - j * M;
        sA[idx] = prm.A[r + (size_t)j * prm.lda];
    }
    for (int idx = threadIdx.x; idx < M; idx += kIndepThreads) sb[idx] = prm.b[idx];
    for (int idx = threadIdx.x; idx < n; idx += kIndepThreads) sc[idx] = prm.c[idx];
    for (int idx = threadIdx.x; idx < kBinomRows * kBinomCols; idx += kIndepThreads) sbin[idx] = prm.binom[idx];
    __syncthreads();

    double   best_key = __longlong_as_double(0x7ff0000000000000LL);   // +inf
    uint64_t best_rank = ~0ull;
    uint32_t ns = 0, ni = 0, nf = 0;

    // block-granular windows dealt round-robin to the shards
    const uint64_t gtid = ((uint64_t)blockIdx.x * prm.shard_count + prm.shard_index) * kIndepThreads + threadIdx.x;
    uint64_t r0 = prm.rank_begin + gtid * prm.chunk;
    if (r0 < prm.rank_end) {
        uint64_t r1 = r0 + prm.chunk;
        if (r1 > prm.rank_end) r1 = prm.rank_end;
        int S[M];
        {
            int St[kMaxM];
            unrank_lex(sbin, n, M, r0, St);
#pragma unroll
            for (int i = 0; i < M; ++i) S[i] = St[i];
        }
        for (uint64_t r = r0; r < r1; ++r) {
            double z, x[M];
            const int st = eval_basis_regs<M>(sA, sb, sc, S, prm.thr, prm.eps_feas, z, x);
            if (st == 2) ++ns;
            else if (st == 1) ++ni;
            else {
                ++nf;
                const double key = prm.maximize ? -z : z;
                if (prm.list_count && in_window(key, prm.list_key_max)) list_append(prm.list_count, prm.list_ranks, prm.list_cap, r);
                if (better(key, r, best_key, best_rank)) { best_key = key; best_rank = r; }
            }
            next_subset_regs<M>(S, n);
        }
    }
    block_reduce<kIndepThreads>(best_key, best_rank, ns, ni, nf, partials + blockIdx.x);
    finalize_if_last(prm, reinterpret_cast<unsigned char*>(sbin + kBinomRows * kBinomCols), sbin);
}

// Run-time m (local-memory arrays): m above the register-resident range, and every m under the
// relative (Eigen-like) singularity rule.
__global__ void __launch_bounds__(kIndepThreads)
k_independent_generic(const LaunchParams prm, BlockPartial* __restrict__ partials)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = prm.n, m = prm.m;
    double*   sA = reinterpret_cast<double*>(smem_raw);
    double*   sb = sA + n * m;
    double*   sc = sb + m;
    uint64_t* sbin = reinterpret_cast<uint64_t*>(sc + n);
    for (int idx = threadIdx.x; idx < n * m; idx += kIndepThreads) {
        const int j = idx / m, r = idx - j * m;
        sA[idx] = prm.A[r + (size_t)j * prm.lda];
    }
    for (int idx = threadIdx.x; idx < m; idx += kIndepThreads) sb[idx] = prm.b[idx];
    for (int idx = threadIdx.x; idx < n; idx += kIndepThreads) sc[idx] = prm.c[idx];
    for (int idx = threadIdx.x; idx < kBinomRows * kBinomCols; idx += kIndepThreads) sbin[idx] = prm.binom[idx];
    __syncthreads();

    double   best_key = __longlong_as_double(0x7ff0000000000000LL);
    uint64_t best_rank = ~0ull;
    uint32_t ns = 0, ni = 0, nf = 0;
    const uint64_t gtid = ((uint64_t)blockIdx.x * prm.shard_count + prm.shard_index) * kIndepThreads + threadIdx.x;
    const uint64_t r0 = prm.rank_begin + gtid * prm.chunk;
    if (r0 < prm.rank_end) {
        uint64_t r1 = r0 + prm.chunk;
        if (r1 > prm.rank_end) r1 = prm.rank_end;
        int S[kMaxM];
        unrank_lex(sbin, n, m, r0, S);
        for (uint64_t r = r0; r < r1; ++r) {
            double z, x[kMaxM];
            const int st = eval_basis_generic(sA, m, sb, sc, m, S, prm.thr, prm.eps_feas, x, &z, prm.pivot_rule, prm.rel_eps);
            if (st == 2) ++ns;
            else if (st == 1) ++ni;
            else {
                ++nf;
                const double key = prm.maximize ? -z : z;
                if (prm.list_count && in_window(key, prm.list_key_max)) list_append(prm.list_count, prm.list_ranks, prm.list_cap, r);
                if (better(key, r, best_key, best_rank)) { best_key = key; best_rank = r; }
            }
            int i = m - 1;
            while (i >= 0 && S[i] == n - m + i) --i;
            if (i >= 0) { ++S[i]; for (int j = i + 1; j < m; ++j) S[j] = S[j - 1] + 1; }
        }
    }
    block_reduce<kIndepThreads>(best_key, best_rank, ns, ni, nf, partials + blockIdx.x);
    finalize_if_last(prm, reinterpret_cast<unsigned char*>(sbin + kBinomRows * kBinomCols), sbin);
}

}  // namespace enumgpu
