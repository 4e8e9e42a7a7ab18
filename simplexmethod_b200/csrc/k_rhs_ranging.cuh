// k_rhs_ranging.cuh — right-hand-side ranging by enumeration (enumgpu_rhs_ranges, DESIGN.md §3.4).
//
// The duals y* stay optimal for b + delta * e_i iff some basis T of the tight columns J is feasible there, so the
// range of row i is the union of the feasibility intervals of the nonsingular m-subsets T of J, feasible at b or not.
// Nothing bounds C(|J|, m) (c = 0 makes J every column), so the kernel runs one warp per basis:
//   k_rhs_ranging<M>       warps grid-stride over runs of kRhsRun consecutive ranks of C(|J|, M): unrank once per
//                          run, then step to the next subset; lane j owns column j of W = [A_T | b | e_0 .. e_{M-1}]
//                          in registers (at M = 16 lane 0 also owns column 32, e_15, once its own column 0 has served
//                          as the first pivot column).  The pivot column's multipliers go out by __shfl_sync, so
//                          every element receives fnma(l, W[k][j], W[r][j]) in step order, as in block_eliminate;
//                          U goes to the warp's shared memory for the column sweeps.  The lane of e_i then holds w_i
//                          and forms row i's interval; it keeps the best (limit, rank) of its row in registers over
//                          all its bases, and the block merges its warps' into its slot of `best`.
//   k_rhs_ranging_finish   one thread per row: the maximum over the blocks' slots, and the output row.
// Each limit is one addition and one IEEE division of frozen bits, and the maximum of (limit, lowest rank) does not
// depend on the order of evaluation: any grid, any run length gives the same bits.
#pragma once

#include "enum_common.cuh"

namespace enumgpu {

constexpr int kRhsThreads = 256;
constexpr int kRhsWarps = kRhsThreads / 32;
constexpr uint32_t kRhsRun = 64;      // consecutive ranks per warp between two unranks

// Row i's interval at one basis (w = w_i, x = x_B): *lo, *hi; false if the row does not count.
template <int M>
__device__ __forceinline__ bool rhs_row(const double (&w)[M], const double* __restrict__ x, double eps_feas,
                                       double eps_opt, double* lo_out, double* hi_out)
{
    double lo = __longlong_as_double((long long)0xfff0000000000000ull), hi = __longlong_as_double(0x7ff0000000000000LL);
    bool ok = true;
    static_for<0, M>([&](auto K) {
        constexpr int k = decltype(K)::value;
        const double s = __dadd_rn(x[k], eps_feas), v = w[k];
        if (v > eps_opt) {
            const double q = __ddiv_rn(-s, v);
            ok &= (q == q);
            if (q > lo) lo = q;
        } else if (v < -eps_opt) {
            const double q = __ddiv_rn(s, -v);
            ok &= (q == q);
            if (q < hi) hi = q;
        } else {
            ok &= (v == v) && (s >= 0.0);
        }
    });
    *lo_out = lo; *hi_out = hi;
    return ok && lo <= hi;
}

// (value, rank) max with ties to the lowest rank; value < 0 is "no candidate"
__device__ __forceinline__ void rhs_offer(double v, uint64_t rank, double& best, uint64_t& best_rank)
{
    if (v >= 0.0 && (v > best || (v == best && rank < best_rank))) { best = v; best_rank = rank; }
}

// A: packed (lda = M) | b, on the device.  J: the n_tight tight columns, ascending.  total: C(n_tight, M);
// total_full: C(n, M).  best: gridDim.x slots of 2M Best (increase of row i at i, decrease at M + i).
// counters[0] += singular bases; counters[1] <- 1 if S* (rank_star) is singular or one of its rows does not contain 0.
template <int M>
__global__ void __launch_bounds__(kRhsThreads)
k_rhs_ranging(const double* __restrict__ A, const double* __restrict__ b, const int32_t* __restrict__ J, int n_tight,
              int n, const uint64_t* __restrict__ binom, uint64_t total, uint64_t total_full, uint64_t rank_star,
              double thr, int pivot_rule, double rel_eps, double eps_feas, double eps_opt, Best* __restrict__ best,
              unsigned long long* __restrict__ counters)
{
    constexpr bool kTwo = 2 * M + 1 > 32;                 // M = 16: lane 0 also owns column 2M = e_{M-1}
    __shared__ double s_A[M * kMaxN + M];
    __shared__ uint64_t s_binom[kBinomRows * kBinomCols];
    __shared__ int s_J[kMaxN];
    __shared__ double s_U[kRhsWarps][M * M];               // column j at [j * M], rows 0..M-1
    __shared__ double s_x[kRhsWarps][M];
    __shared__ double s_bv[kRhsWarps][2 * M];
    __shared__ uint64_t s_br[kRhsWarps][2 * M];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < M * n; e += kRhsThreads) s_A[e] = A[e];
    for (int e = tid; e < M; e += kRhsThreads) s_A[M * n + e] = b[e];
    for (int e = tid; e < kBinomRows * kBinomCols; e += kRhsThreads) s_binom[e] = binom[e];
    for (int e = tid; e < n_tight; e += kRhsThreads) s_J[e] = J[e];
    __syncthreads();
    const double* sb = s_A + M * n;
    double* U = s_U[warp];
    double* xs = s_x[warp];
    const unsigned full = 0xffffffffu;
    // this lane's row: lanes M+1 .. 2M own e_0 .. e_{M-1}; at M = 16 lane 0 owns row 15 through its second column
    const int row = (lane > M && lane <= 2 * M) ? lane - M - 1 : -1;
    double inc = -1.0, dec = -1.0, inc2 = -1.0, dec2 = -1.0;
    uint64_t inc_r = ~0ull, dec_r = ~0ull, inc2_r = ~0ull, dec2_r = ~0ull;
    unsigned long long n_sing = 0;

    const uint64_t n_runs = (total + kRhsRun - 1) / kRhsRun;
    const uint64_t n_warps = (uint64_t)gridDim.x * kRhsWarps;
    for (uint64_t run = (uint64_t)blockIdx.x * kRhsWarps + warp; run < n_runs; run += n_warps) {
        const uint64_t r0 = run * kRhsRun, r1 = min(r0 + kRhsRun, total);
        int idx[M];
        {
            uint64_t r = r0;
            int v = 0;
            static_for<0, M>([&](auto I) {
                constexpr int i = decltype(I)::value;
                for (;;) {
                    const uint64_t cnt = s_binom[(n_tight - 1 - v) * kBinomCols + (M - 1 - i)];
                    if (cnt <= r) { r -= cnt; ++v; } else break;
                }
                idx[i] = v++;
            });
        }
        for (uint64_t r = r0; r < r1; ++r) {
            if (r != r0) {                                 // the next subset in lexicographic order
                int piv = 0;
                static_for<0, M>([&](auto I) {
                    constexpr int i = decltype(I)::value;
                    if (idx[i] < n_tight - M + i) piv = i;
                });
                static_for<0, M>([&](auto I) {
                    constexpr int i = decltype(I)::value;
                    if (i == piv) ++idx[i];
                    if constexpr (i > 0) { if (i > piv) idx[i] = idx[i - 1] + 1; }
                });
            }
            // the basis's columns, its rank among the C(n, M) bases, and this lane's column of W
            uint64_t acc = 0;
            int col = 0;
            static_for<0, M>([&](auto I) {
                constexpr int i = decltype(I)::value;
                const int cj = s_J[idx[i]];
                acc += s_binom[(n - 1 - cj) * kBinomCols + (M - i)];
                if (lane == i) col = cj;
            });
            const uint64_t rank = total_full - 1 - acc;
            double w[M], w2[kTwo ? M : 1];
            static_for<0, M>([&](auto R) {
                constexpr int r_ = decltype(R)::value;
                w[r_] = lane < M ? s_A[col * M + r_] : lane == M ? sb[r_] : (lane - M - 1 == r_ ? 1.0 : 0.0);
                if constexpr (kTwo) w2[r_] = r_ == M - 1 ? 1.0 : 0.0;
            });
            // elimination: the pivot rule, threshold and operations of block_eliminate
            bool singular = false;
            double pmax = 0.0, pmin = __longlong_as_double(0x7ff0000000000000LL), rinv[M];
            static_for<0, M>([&](auto K) {
                constexpr int k = decltype(K)::value;
                if (singular) return;
                double bestv = fabs(w[k]);
                int p = k;
                static_for<k + 1, M>([&](auto R) {
                    constexpr int r_ = decltype(R)::value;
                    const double v = fabs(w[r_]);
                    if (v > bestv) { bestv = v; p = r_; }
                });
                bestv = __shfl_sync(full, bestv, k);
                p = __shfl_sync(full, p, k);
                if (!(bestv > thr)) { singular = true; return; }
                if (bestv > pmax) pmax = bestv;
                if (bestv < pmin) pmin = bestv;
                static_for<k + 1, M>([&](auto R) {
                    constexpr int r_ = decltype(R)::value;
                    if (r_ == p) {
                        const double t = w[k]; w[k] = w[r_]; w[r_] = t;
                        if constexpr (kTwo) { const double t2 = w2[k]; w2[k] = w2[r_]; w2[r_] = t2; }
                    }
                });
                const double ri = __shfl_sync(full, __drcp_rn(w[k]), k);
                rinv[k] = ri;
                static_for<k + 1, M>([&](auto R) {
                    constexpr int r_ = decltype(R)::value;
                    const double l = __shfl_sync(full, __dmul_rn(w[r_], ri), k);
                    w[r_] = fnma(l, w[k], w[r_]);
                    if constexpr (kTwo) w2[r_] = fnma(l, w2[k], w2[r_]);
                });
            });
            if (!singular && pivot_rule == ENUMGPU_PIVOT_RELATIVE) singular = !(pmin > __dmul_rn(rel_eps, pmax));
            if (singular) {
                if (lane == 0) ++n_sing;
                if (rank == rank_star && lane == 0) counters[1] = 1ull;
                continue;
            }
            // U to shared memory, then the column sweeps of b and the e_i (and of every other column: idle lanes)
            if (lane < M) static_for<0, M>([&](auto R) { constexpr int r_ = decltype(R)::value; U[lane * M + r_] = w[r_]; });
            __syncwarp();
            static_rfor<0, M>([&](auto Jc) {
                constexpr int j = decltype(Jc)::value;
                const double xj = __dmul_rn(w[j], rinv[j]);
                w[j] = xj;
                [[maybe_unused]] double xj2 = 0.0;
                if constexpr (kTwo) { xj2 = __dmul_rn(w2[j], rinv[j]); w2[j] = xj2; }
                static_for<0, j>([&](auto I) {
                    constexpr int i = decltype(I)::value;
                    const double u = U[j * M + i];
                    w[i] = fnma(u, xj, w[i]);
                    if constexpr (kTwo) w2[i] = fnma(u, xj2, w2[i]);
                });
            });
            if (lane == M) static_for<0, M>([&](auto R) { constexpr int r_ = decltype(R)::value; xs[r_] = w[r_]; });
            __syncwarp();
            bool foreign = false;
            if (row >= 0) {
                double lo, hi;
                if (rhs_row<M>(w, xs, eps_feas, eps_opt, &lo, &hi)) {
                    rhs_offer(hi, rank, inc, inc_r);
                    rhs_offer(-lo, rank, dec, dec_r);
                    foreign = !(lo <= 0.0 && hi >= 0.0);
                } else {
                    foreign = true;
                }
            }
            if constexpr (kTwo) {
                if (lane == 0) {
                    double lo, hi;
                    if (rhs_row<M>(w2, xs, eps_feas, eps_opt, &lo, &hi)) {
                        rhs_offer(hi, rank, inc2, inc2_r);
                        rhs_offer(-lo, rank, dec2, dec2_r);
                        foreign = !(lo <= 0.0 && hi >= 0.0);
                    } else {
                        foreign = true;
                    }
                }
            }
            if (rank == rank_star && foreign) counters[1] = 1ull;
            __syncwarp();                                  // U and x are rewritten by the next basis
        }
    }
    if (lane == 0 && n_sing) atomicAdd(&counters[0], n_sing);
    // the block's best per slot: warps in index order
    if (row >= 0) {
        s_bv[warp][row] = inc; s_br[warp][row] = inc_r;
        s_bv[warp][M + row] = dec; s_br[warp][M + row] = dec_r;
    }
    if constexpr (kTwo) {
        if (lane == 0) {
            s_bv[warp][M - 1] = inc2; s_br[warp][M - 1] = inc2_r;
            s_bv[warp][2 * M - 1] = dec2; s_br[warp][2 * M - 1] = dec2_r;
        }
    }
    __syncthreads();
    if (tid < 2 * M) {
        double v = -1.0;
        uint64_t k = ~0ull;
        for (int wp = 0; wp < kRhsWarps; ++wp) rhs_offer(s_bv[wp][tid], s_br[wp][tid], v, k);
        best[(size_t)blockIdx.x * 2 * M + tid] = Best{v, k};
    }
}

// Row i (one thread each): the maximum over the n_blocks slots; +inf gets rank UINT64_MAX, and a row without any
// candidate (only with a foreign dual, which the host refuses) gets NaN.
__global__ void __launch_bounds__(32)
k_rhs_ranging_finish(const Best* __restrict__ best, int n_blocks, int m, const double* __restrict__ y,
                     enumgpu_rhs_range* __restrict__ out)
{
    const int i = threadIdx.x;
    if (i >= m) return;
    double lim[2];
    uint64_t rk[2];
    for (int t = 0; t < 2; ++t) {
        lim[t] = -1.0; rk[t] = ~0ull;
        for (int s = 0; s < n_blocks; ++s) {
            const Best v = best[(size_t)s * 2 * m + t * m + i];
            rhs_offer(v.key, v.rank, lim[t], rk[t]);
        }
        if (lim[t] < 0.0) lim[t] = __longlong_as_double(0x7ff8000000000000LL);
        if (!(lim[t] < __longlong_as_double(0x7ff0000000000000LL))) rk[t] = ~0ull;
    }
    enumgpu_rhs_range r;
    r.shadow_price = y[i];
    r.increase = lim[0]; r.increase_rank = rk[0];
    r.decrease = lim[1]; r.decrease_rank = rk[1];
    out[i] = r;
}

}  // namespace enumgpu
