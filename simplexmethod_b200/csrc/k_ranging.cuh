// k_ranging.cuh — cost ranging by enumeration (enumgpu_cost_ranges, DESIGN.md §3.3).
//
// The vertex x* stays optimal for the key-sense cost ck + delta * e_j iff no feasible basis and no extreme ray does
// better at that cost.  The host lists the feasible bases of the LP and, where m + 1 rows fit, those of the auxiliary
// LP [A; s*1'] d = (0, ..., 0, s) (its feasible bases are the extreme rays, normalised to 1'd = 1); k_obj_values
// gives S and x_B (or d) of every listed rank, and these kernels finish the job:
//   k_ranging          one thread per listed basis: its key (or ck.d) in the frozen order, then its <= 2m touched
//                      columns; each candidate (ratio, rank) of a column's up or down limit is folded into per-block
//                      minima in shared memory.  A nonnegative double orders like its bits, so the fold is a 64-bit
//                      atomicMin on the ratio, then, after a barrier, a second walk that takes the lowest rank among
//                      the candidates at that ratio.  The block's minima merge into its slice of the previous
//                      chunks' (fixed grid: slice b is always block b).
//   k_ranging_finish   one thread per column: the minimum over the slices, a ray where its ratio is strictly
//                      smaller than the vertex limit, and key-sense up / down mapped to the true sense.
// Every ratio is one subtraction and one IEEE division of frozen bits, and the minimum of (ratio, rank) does not
// depend on the order of evaluation: both kernel families, any chunking and any split of the listing give the same bits.
#pragma once

#include "enum_common.cuh"

namespace enumgpu {

constexpr int kRangeThreads = 256;

// Slots of a column j in a slice's row of 3n Best entries: up (vertices) j, down (vertices) n + j, down (rays) 2n + j.
// Inputs of one launch over a chunk of `count` listed bases, S_in / x_in as k_obj_values leaves them ([rows][count]):
//   rays = 0: rows = m, c = the LP's costs, the key is maximize ? -z : z; Delta k = key - key_star.
//   rays = 1: rows = m + 1, c = ck, the key is ck.d itself.
// xs: x* dense (0 outside S*), tol: eps_opt * max(1, |x*_j|), Sstar: the m columns of S*.
// flags[0] <- 1 if a basis has key < key_star (opt came from other options); flags[1] <- 1 if a ray has ck.d < -eps_opt.
__global__ void __launch_bounds__(kRangeThreads)
k_ranging(const uint8_t* __restrict__ S_in, const double* __restrict__ x_in, const uint64_t* __restrict__ ranks,
          uint32_t count, int rows, int n, int rays, int maximize, const double* __restrict__ c,
          const double* __restrict__ xs, const double* __restrict__ tol, const int32_t* __restrict__ Sstar, int m,
          double key_star, double tau_k, double eps_opt, int first, Best* __restrict__ best, int* __restrict__ flags)
{
    __shared__ unsigned long long s_ratio[2 * kMaxN], s_rank[2 * kMaxN];
    __shared__ double s_c[kMaxN], s_xs[kMaxN], s_tol[kMaxN];
    __shared__ int s_S[kMaxM];
    const int tid = threadIdx.x, n_slots = rays ? n : 2 * n;
    for (int j = tid; j < n; j += kRangeThreads) { s_c[j] = c[j]; s_xs[j] = xs[j]; s_tol[j] = tol[j]; }
    for (int j = tid; j < m; j += kRangeThreads) s_S[j] = Sstar[j];
    for (int s = tid; s < n_slots; s += kRangeThreads) { s_ratio[s] = 0x7ff0000000000000ull; s_rank[s] = ~0ull; }
    __syncthreads();

    // pass 0: the least ratio bits of every slot; pass 1: the least rank among the candidates at that ratio
    for (int pass = 0; pass < 2; ++pass) {
        for (uint32_t i = blockIdx.x * kRangeThreads + tid; i < count; i += gridDim.x * kRangeThreads) {
            const uint64_t rank = ranks[i];
            auto offer = [&](int slot, double ratio) {
                const unsigned long long bits = (unsigned long long)__double_as_longlong(ratio);
                if (pass == 0) { if (bits < s_ratio[slot]) atomicMin(&s_ratio[slot], bits); }
                else if (bits == s_ratio[slot]) atomicMin(&s_rank[slot], (unsigned long long)rank);
            };
            double z = 0.0;
            for (int j = rows - 1; j >= 0; --j) z = __fma_rn(s_c[S_in[(size_t)j * count + i]], x_in[(size_t)j * count + i], z);
            if (rays) {
                if (z != z) continue;
                if (z < -eps_opt) { if (pass == 0) flags[1] = 1; continue; }
                for (int j = 0; j < rows; ++j) {
                    const double d = x_in[(size_t)j * count + i];
                    if (d > eps_opt) offer(S_in[(size_t)j * count + i], z <= eps_opt ? 0.0 : __ddiv_rn(z, d));
                }
                continue;
            }
            const double dk = (maximize ? -z : z) - key_star;
            if (dk != dk) continue;
            if (dk < 0.0) { if (pass == 0) flags[0] = 1; continue; }
            auto column = [&](int col, double dx) {
                if (dx != dx || fabs(dx) <= s_tol[col]) return;
                const double ratio = dk <= tau_k ? 0.0 : __ddiv_rn(dk, fabs(dx));
                if (ratio != ratio) return;                       // inf / inf: never a limit, as better() has it
                offer(dx < 0.0 ? col : n + col, ratio);
            };
            uint64_t in_B = 0;
            for (int j = 0; j < rows; ++j) {
                const int col = S_in[(size_t)j * count + i];
                in_B |= 1ull << col;
                column(col, x_in[(size_t)j * count + i] - s_xs[col]);
            }
            for (int k = 0; k < m; ++k)
                if (!((in_B >> s_S[k]) & 1)) column(s_S[k], 0.0 - s_xs[s_S[k]]);
        }
        __syncthreads();
    }
    // merge with the slice's minima of the earlier chunks
    Best* row = best + (size_t)blockIdx.x * 3 * n + (rays ? 2 * n : 0);
    for (int s = tid; s < n_slots; s += kRangeThreads) {
        double r = __longlong_as_double((long long)s_ratio[s]);
        uint64_t k = s_rank[s];
        if (!first && better(row[s].key, row[s].rank, r, k)) { r = row[s].key; k = row[s].rank; }
        row[s].key = r; row[s].rank = k;
    }
}

// Per column: the minima over the slices of the vertex launches (n_vslices, 0 if none ran) and of the ray launches
// (n_rslices), then the true-sense range.
__global__ void __launch_bounds__(kRangeThreads)
k_ranging_finish(const Best* __restrict__ best, int n_vslices, int n_rslices, int n, int maximize,
                 enumgpu_cost_range* __restrict__ out)
{
    const int j = blockIdx.x * kRangeThreads + threadIdx.x;
    if (j >= n) return;
    Best lim[3];
    for (int t = 0; t < 3; ++t) {
        lim[t].key = __longlong_as_double(0x7ff0000000000000LL);
        lim[t].rank = ~0ull;
        const int slices = t < 2 ? n_vslices : n_rslices;
        for (int s = 0; s < slices; ++s) {
            const Best v = best[(size_t)s * 3 * n + t * n + j];
            if (better(v.key, v.rank, lim[t].key, lim[t].rank)) lim[t] = v;
        }
    }
    const bool ray = lim[2].key < lim[1].key;              // a ray takes over only when strictly smaller
    const Best up = lim[0], down = ray ? lim[2] : lim[1];
    enumgpu_cost_range r;
    if (maximize) {                                        // a rise of c_j is a fall of ck_j
        r.increase = down.key; r.increase_rank = down.rank; r.increase_ray = ray ? 1 : 0;
        r.decrease = up.key; r.decrease_rank = up.rank; r.decrease_ray = 0;
    } else {
        r.increase = up.key; r.increase_rank = up.rank; r.increase_ray = 0;
        r.decrease = down.key; r.decrease_rank = down.rank; r.decrease_ray = ray ? 1 : 0;
    }
    out[j] = r;
}

}  // namespace enumgpu
