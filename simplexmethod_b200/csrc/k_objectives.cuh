// k_objectives.cuh — many cost vectors over one feasible set (enumgpu_solve_objectives, DESIGN.md §3.2).
//
// Which bases are singular, infeasible or feasible, and the x_B of every feasible one, depend on A, b and the
// tolerances only; the cost vector enters in the last m FMAs of a feasible basis, z = fma(c[S[j]], x[j], z) for
// j = m-1 .. 0.  So the feasible bases are listed once (the enumeration kernels' listing, key bound +inf), and these
// kernels finish the job for K cost vectors:
//   k_obj_values<M>   one thread per listed rank: unrank, the frozen GE in registers (eval_basis_regs<M>, the
//                     per-basis arithmetic of k_independent), S and x_B to a chunk buffer.  Runs once per listed
//                     basis, whatever K is.
//   k_objectives<M>   the hot loop: a 2-D grid of slices of the chunk x tiles of W objectives.  A block stages its C
//                     tile [column][objective] in shared memory once, then a tile of (S, x_B) at a time; thread t owns
//                     objective t % W and the bases t / W, t / W + 256 / W, ... of each tile, and keeps its best
//                     (key, rank) in registers.  One block reduction per objective at the end folds the 256 / W lanes
//                     of an objective and merges them into that slice's best of the previous chunks.
//   k_obj_finish      one thread per objective: the minimum over the slices, then the winner re-evaluated with
//                     eval_basis_generic and the objective's own costs — the operations, and so the bits, of the
//                     enumeration record's finalize.
// The key of a basis is maximize ? -z : z with z in the frozen order, and bases are compared with better(): the
// lexicographic minimum of (key, rank) over the listed bases is what enumgpu_solve's reduction finds, in any order of
// evaluation.  NaN keys never win, exactly as there.
#pragma once

#include "enum_common.cuh"
#include "k_independent.cuh"

namespace enumgpu {

constexpr int kObjThreads = 256;      // threads per block of all three kernels
constexpr int kObjTile = 256;         // bases staged in shared memory at a time by k_objectives

// S[j] (a byte: n <= 64) and x_B[j] of listed basis i of a chunk: row j of the chunk buffers, S_out[j * count + i]
template <int M>
__global__ void __launch_bounds__(kObjThreads)
k_obj_values(const double* __restrict__ A, const double* __restrict__ b, const uint64_t* __restrict__ binom, int n,
             const uint64_t* __restrict__ ranks, uint32_t count, uint8_t* __restrict__ S_out, double* __restrict__ x_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double*   sA = reinterpret_cast<double*>(smem_raw);          // n*M, packed columns (the problem's device copy is)
    double*   sb = sA + n * M;                                    // M
    double*   sz = sb + M;                                        // n zeros: the z eval_basis_regs forms is not used
    uint64_t* sbin = reinterpret_cast<uint64_t*>(sz + n);
    for (int i = threadIdx.x; i < n * M; i += kObjThreads) sA[i] = A[i];
    for (int i = threadIdx.x; i < M; i += kObjThreads) sb[i] = b[i];
    for (int i = threadIdx.x; i < n; i += kObjThreads) sz[i] = 0.0;
    for (int i = threadIdx.x; i < kBinomRows * kBinomCols; i += kObjThreads) sbin[i] = binom[i];
    __syncthreads();
    const uint32_t i = blockIdx.x * kObjThreads + threadIdx.x;
    if (i >= count) return;
    int S[M];
    {
        int St[kMaxM];
        unrank_lex(sbin, n, M, ranks[i], St);
#pragma unroll
        for (int j = 0; j < M; ++j) S[j] = St[j];
    }
    double z, x[M];
    // thr = 0: a listed basis passed the enumeration's singularity rule, so every pivot is > 0 (both rules); the
    // class is known (feasible) and the rule never changes the bits of x_B
    eval_basis_regs<M>(sA, sb, sz, S, 0.0, 0.0, z, x);
#pragma unroll
    for (int j = 0; j < M; ++j) {
        S_out[(size_t)j * count + i] = (uint8_t)S[j];
        x_out[(size_t)j * count + i] = x[j];
    }
}

// run-time m (m = 13..16): local-memory arrays, the same arithmetic
__global__ void __launch_bounds__(kObjThreads)
k_obj_values_generic(const double* __restrict__ A, const double* __restrict__ b, const uint64_t* __restrict__ binom, int m,
                     int n, const uint64_t* __restrict__ ranks, uint32_t count, uint8_t* __restrict__ S_out,
                     double* __restrict__ x_out)
{
    const uint32_t i = blockIdx.x * kObjThreads + threadIdx.x;
    if (i >= count) return;
    int S[kMaxM];
    unrank_lex(binom, n, m, ranks[i], S);
    double z, x[kMaxM];
    eval_basis_generic(A, m, b, A, m, S, 0.0, 0.0, x, &z);     // c = A: any n readable doubles, z is not used
    for (int j = 0; j < m; ++j) {
        S_out[(size_t)j * count + i] = (uint8_t)S[j];
        x_out[(size_t)j * count + i] = x[j];
    }
}

// best (key, rank) per (slice, objective): Best best[slice * k + objective]
// C: the K cost vectors, cost vector o at C[o * n .. o * n + n).  W: objectives per block, a power of two <= 256.
// first: this is the first chunk, so the slice's previous best is (+inf, none).
template <int M>
__global__ void __launch_bounds__(kObjThreads)
k_objectives(const uint8_t* __restrict__ S_in, const double* __restrict__ x_in, const uint64_t* __restrict__ ranks,
             uint32_t count, int n, int maximize, const double* __restrict__ C, int32_t k, int W, int first,
             Best* __restrict__ best)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double*   sx = reinterpret_cast<double*>(smem_raw);           // [M][kObjTile]
    uint64_t* sr = reinterpret_cast<uint64_t*>(sx + M * kObjTile); // [kObjTile]
    double*   sC = reinterpret_cast<double*>(sr + kObjTile);      // [n][W]
    uint8_t*  sS = reinterpret_cast<uint8_t*>(sC + n * W);        // [M][kObjTile]
    __shared__ double   s_key[kObjThreads];
    __shared__ uint64_t s_rank[kObjThreads];

    const int tid = threadIdx.x, ol = tid & (W - 1), bl = tid / W, L = kObjThreads / W;
    const int32_t o0 = (int32_t)blockIdx.y * W, o = o0 + ol;
    for (int e = tid; e < n * W; e += kObjThreads) {
        const int j = e % n, t = e / n;
        sC[j * W + t] = (o0 + t < k) ? C[(size_t)(o0 + t) * n + j] : 0.0;
    }
    // the block's slice of the chunk
    const uint32_t per = (count + gridDim.x - 1) / gridDim.x;
    const uint32_t lo = min(count, blockIdx.x * per), hi = min(count, lo + per);

    double   bkey = __longlong_as_double(0x7ff0000000000000LL);   // +inf
    uint64_t brank = ~0ull;
    for (uint32_t t0 = lo; t0 < hi; t0 += kObjTile) {
        const int tn = (int)min((uint32_t)kObjTile, hi - t0);
        __syncthreads();                                              // the previous tile is consumed (and sC written)
        for (int e = tid; e < M * tn; e += kObjThreads) {
            const int j = e / tn, i = e - j * tn;
            sx[j * kObjTile + i] = x_in[(size_t)j * count + t0 + i];
            sS[j * kObjTile + i] = S_in[(size_t)j * count + t0 + i];
        }
        for (int i = tid; i < tn; i += kObjThreads) sr[i] = ranks[t0 + i];
        __syncthreads();
        for (int i = bl; i < tn; i += L) {
            double z = 0.0;
            static_rfor<0, M>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                z = __fma_rn(sC[sS[j * kObjTile + i] * W + ol], sx[j * kObjTile + i], z);
            });
            const double key = maximize ? -z : z;
            const uint64_t r = sr[i];
            if (better(key, r, bkey, brank)) { bkey = key; brank = r; }
        }
    }
    // fold the L lanes of each objective, then merge with the slice's best of the earlier chunks
    s_key[tid] = bkey; s_rank[tid] = brank;
    __syncthreads();
    if (bl == 0 && o < k) {
        for (int l = 1; l < L; ++l) {
            const double k2 = s_key[l * W + ol];
            const uint64_t r2 = s_rank[l * W + ol];
            if (better(k2, r2, bkey, brank)) { bkey = k2; brank = r2; }
        }
        Best* slot = best + (size_t)blockIdx.x * k + o;
        if (!first && better(slot->key, slot->rank, bkey, brank)) { bkey = slot->key; brank = slot->rank; }
        slot->key = bkey; slot->rank = brank;
    }
}

// Per objective: the minimum over n_slices slices (none if n_slices = 0: nothing was listed), then the record of the
// winner as the enumeration's finalize writes it (basis, x_B, objective; zeros and NaN without a winner).  The
// counters and algo_used are the listing's, filled in by the host.  A: packed, lda = m.
__global__ void __launch_bounds__(kObjThreads)
k_obj_finish(const Best* __restrict__ best, int n_slices, const double* __restrict__ A, const double* __restrict__ b,
             const double* __restrict__ C, const uint64_t* __restrict__ binom, int m, int n, int32_t k,
             enumgpu_partial* __restrict__ out)
{
    const int32_t o = (int32_t)(blockIdx.x * kObjThreads + threadIdx.x);
    if (o >= k) return;
    double   key = __longlong_as_double(0x7ff0000000000000LL);
    uint64_t rank = ~0ull;
    for (int s = 0; s < n_slices; ++s) {
        const Best v = best[(size_t)s * k + o];
        if (better(v.key, v.rank, key, rank)) { key = v.key; rank = v.rank; }
    }
    enumgpu_partial* r = out + o;
    r->key = key; r->best_rank = rank;
    r->n_bases = r->n_singular = r->n_infeasible = r->n_feasible = 0;
    r->m = m; r->algo_used = 0;
    for (int i = 0; i < kMaxM; ++i) { r->x_B[i] = 0.0; r->basis[i] = 0; }
    r->objective = __longlong_as_double(0x7ff8000000000000LL);
    if (rank == ~0ull) return;
    int S[kMaxM];
    unrank_lex(binom, n, m, rank, S);
    double x[kMaxM], z = 0.0;
    eval_basis_generic(A, m, b, C + (size_t)o * n, m, S, 0.0, 0.0, x, &z);
    for (int i = 0; i < m; ++i) { r->x_B[i] = x[i]; r->basis[i] = S[i]; }
    r->objective = z;
}

}  // namespace enumgpu
