// enum_common.cuh — shared device-side definitions of libenumgpu (sm_100a).
//
// The per-basis arithmetic implemented by every kernel here is the frozen
// definition of DESIGN.md §3 (restated in oracle/enumcpu.c for the checker):
// partial-pivot GE with one reciprocal per pivot, explicit FMAs, column-sweep
// back substitution, feasibility x >= -eps, objective accumulated from the
// last basic variable to the first.  Reference semantics: gather
// Canonical.cpp:183-187, singular rejected SimplexSolover.h:124-126, feasible
// Canonical.cpp:165-177, objective Canonical.cpp:79-87.
#pragma once

#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

#include "../../include/enumgpu.h"

namespace enumgpu {

constexpr int kMaxM = ENUMGPU_MAX_M;
constexpr int kMaxN = ENUMGPU_MAX_N;
constexpr int kBinomRows = kMaxN + 1;   // top index 0..64
constexpr int kBinomCols = kMaxM + 1;   // k index 0..16

struct BlockPartial;

// Per-enqueue control block in device memory, zero before the first launch of an enqueue and zero again
// after its last block has finished (that block resets it): the work counter of k_shared and the ticket
// that tells a finishing block whether it is the last one of the whole enqueue.
struct Ctrl {
    unsigned long long unit_counter;
    unsigned int ticket;
    unsigned int pad_;
};

// Everything a kernel needs besides the matrix data.  Passed by value.
struct LaunchParams {
    const double* A;        // device, column-major
    const double* b;
    const double* c;
    const uint64_t* binom;  // device, [kBinomRows][kBinomCols], C(top,k)
    int32_t  m, n, lda, maximize;
    double   eps_feas;
    double   thr;           // eps_piv * max|A_ij|
    uint64_t rank_begin, rank_end;
    uint32_t chunk;         // ranks per thread (independent kernel)
    uint32_t shard_index;   // interleaved sharding: this launch owns the work
    uint32_t shard_count;   // windows whose index is shard_index mod shard_count
    // optional listing of the feasible bases (enumgpu_list_window): ranks are appended in
    // arbitrary order; *list_count counts all of them, only the first list_cap are stored.
    // A feasible basis is listed iff in_window(key, list_key_max) (+inf lists all of them).
    unsigned long long* list_count;
    uint64_t* list_ranks;
    uint64_t  list_cap;
    double    list_key_max;
    // singularity rule: ENUMGPU_PIVOT_ABSOLUTE (thr above) or ENUMGPU_PIVOT_RELATIVE (thr = 0, rel_eps below;
    // the run-time-m kernels only)
    int32_t  pivot_rule;
    int32_t  algo_used;     // written to the record
    double   rel_eps;
    // fused finalize: the last block of the enqueue (ticket == total_blocks - 1) reduces all_parts[0..total_blocks)
    // into *record and resets *ctrl
    Ctrl*            ctrl;
    BlockPartial*    all_parts;
    uint32_t         total_blocks;
    enumgpu_partial* record;
};

// +inf lists every feasible basis, NaN keys included; a finite bound never lists a NaN key
__device__ __forceinline__ bool in_window(double key, double key_max)
{
    return key <= key_max || key_max == __longlong_as_double(0x7ff0000000000000LL);
}

__device__ __forceinline__ void list_append(unsigned long long* count, uint64_t* ranks, uint64_t cap, uint64_t rank)
{
    const unsigned long long pos = atomicAdd(count, 1ull);
    if (pos < cap) ranks[pos] = rank;
}

// (key, rank) pair + counters: what every thread / warp / block / GPU reduces.
struct Best {
    double   key;
    uint64_t rank;
};

__device__ __forceinline__ bool better(double k1, uint64_t r1, double k2, uint64_t r2)
{
    return (k1 < k2) || (k1 == k2 && r1 < r2);
}

struct BlockPartial {          // one per block, reduced by the finalize kernel
    double   key;
    uint64_t rank;
    uint64_t n_sing, n_infeas, n_feas;
};

// Compile-time loop: f(integral_constant<int,I>) for I in [B, E).  '#pragma
// unroll' is only a request — nvcc leaves inner loops of large unrolled nests
// rolled, which turns register arrays into local memory.  This cannot.
template <int B, int E, class F>
__device__ __forceinline__ void static_for(F&& f)
{
    if constexpr (B < E) {
        f(std::integral_constant<int, B>{});
        static_for<B + 1, E>(f);
    }
}
// same, descending: I = E-1 ... B
template <int B, int E, class F>
__device__ __forceinline__ void static_rfor(F&& f)
{
    if constexpr (B < E) {
        f(std::integral_constant<int, E - 1>{});
        static_rfor<B, E - 1>(f);
    }
}

// IEEE double ops that must not be contracted or reassociated.
__device__ __forceinline__ double fnma(double a, double b, double c) { return __fma_rn(-a, b, c); }

// ---------------------------------------------------------------------------
// Warp + block reduction of (key, rank) by lexicographic min and of counters
// by sum.  Result valid in thread 0 of the block.
template <int kThreads, class Count>     // Count: uint32_t or uint64_t per-thread counters
__device__ __forceinline__ void block_reduce(double& key, uint64_t& rank,
                                             Count& ns, Count& ni, Count& nf,
                                             BlockPartial* out_slot, int n_warps = kThreads / 32)
{
    constexpr int kWarps = kThreads / 32;   // capacity; n_warps <= kWarps are live
    __shared__ double   s_key[kWarps];
    __shared__ uint64_t s_rank[kWarps];
    __shared__ uint64_t s_cnt[kWarps][3];
    const unsigned full = 0xffffffffu;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        double   k2 = __shfl_down_sync(full, key, off);
        uint64_t r2 = __shfl_down_sync(full, rank, off);
        if (better(k2, r2, key, rank)) { key = k2; rank = r2; }
        ns += __shfl_down_sync(full, ns, off);
        ni += __shfl_down_sync(full, ni, off);
        nf += __shfl_down_sync(full, nf, off);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_key[warp] = key; s_rank[warp] = rank; s_cnt[warp][0] = ns; s_cnt[warp][1] = ni; s_cnt[warp][2] = nf; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double bk = s_key[0]; uint64_t br = s_rank[0];
        uint64_t cs = s_cnt[0][0], ci = s_cnt[0][1], cf = s_cnt[0][2];
        for (int w = 1; w < n_warps; ++w) {
            if (better(s_key[w], s_rank[w], bk, br)) { bk = s_key[w]; br = s_rank[w]; }
            cs += s_cnt[w][0]; ci += s_cnt[w][1]; cf += s_cnt[w][2];
        }
        out_slot->key = bk; out_slot->rank = br;
        out_slot->n_sing = cs; out_slot->n_infeas = ci; out_slot->n_feas = cf;
    }
}

// Unrank r into S[0..m) using a binomial table in (shared) memory.
__device__ __forceinline__ void unrank_lex(const uint64_t* __restrict__ binom, int n, int m,
                                           uint64_t r, int* S)
{
    int v = 0;
    for (int i = 0; i < m; ++i) {
        for (;;) {
            uint64_t cnt = binom[(n - 1 - v) * kBinomCols + (m - 1 - i)];
            if (cnt <= r) { r -= cnt; ++v; } else break;
        }
        S[i] = v++;
    }
}

// One basis with run-time m (local-memory arrays): used once per enqueue, by
// one thread, to materialise x_B / objective of the winning basis on the device.
__device__ inline int eval_basis_generic(const double* A, int lda, const double* b, const double* c, int m,
                                  const int* S, double thr, double eps_feas, double* x, double* z_out,
                                  int pivot_rule = ENUMGPU_PIVOT_ABSOLUTE, double rel_eps = 0.0)
{
    double Mx[kMaxM][kMaxM + 1];
    double rinv[kMaxM];
    double pmax = 0.0, pmin = __longlong_as_double(0x7ff0000000000000LL);
    for (int j = 0; j < m; ++j)
        for (int r = 0; r < m; ++r) Mx[r][j] = A[r + (size_t)S[j] * lda];
    for (int r = 0; r < m; ++r) Mx[r][m] = b[r];
    for (int k = 0; k < m; ++k) {
        int p = k;
        double best = fabs(Mx[k][k]);
        for (int r = k + 1; r < m; ++r) {
            const double v = fabs(Mx[r][k]);
            if (v > best) { best = v; p = r; }
        }
        if (!(best > thr)) return 2;
        if (best > pmax) pmax = best;
        if (best < pmin) pmin = best;
        if (p != k)
            for (int j = k; j <= m; ++j) { const double t = Mx[k][j]; Mx[k][j] = Mx[p][j]; Mx[p][j] = t; }
        rinv[k] = __drcp_rn(Mx[k][k]);
        for (int r = k + 1; r < m; ++r) {
            const double l = __dmul_rn(Mx[r][k], rinv[k]);
            for (int j = k + 1; j <= m; ++j) Mx[r][j] = fnma(l, Mx[k][j], Mx[r][j]);
        }
    }
    if (pivot_rule == ENUMGPU_PIVOT_RELATIVE && !(pmin > __dmul_rn(rel_eps, pmax))) return 2;
    bool infeasible = false;
    double z = 0.0;
    for (int j = m - 1; j >= 0; --j) {
        x[j] = __dmul_rn(Mx[j][m], rinv[j]);
        infeasible |= !(x[j] >= -eps_feas);
        for (int i = 0; i < j; ++i) Mx[i][m] = fnma(Mx[i][j], x[j], Mx[i][m]);
        z = __fma_rn(c[S[j]], x[j], z);
    }
    *z_out = z;
    return infeasible ? 1 : 0;
}

// ---------------------------------------------------------------------------
// Fused finalize.  Every block of an enqueue (which may consist of up to three launches on one stream: the
// shared kernel and the independent kernel on the ragged head and tail of the range) calls this after it has
// written its BlockPartial.  The block that draws the last ticket reduces all partials, writes the 256-byte
// record — x_B and the objective of the winning basis re-evaluated on the device by warp 0, lane j owning
// column j of [B | b]: every element receives the same operations in the same order as in
// eval_basis_generic — and resets the control block for the next enqueue.  `scratch`: >= kFinalizeScratch bytes
// of shared memory that the block no longer needs (8-byte aligned).  blockDim.x: a multiple of 32, <= 1024.
constexpr int kFinalizeScratch = 8 * (kMaxM * (kMaxM + 1) + kMaxM) + 4 * kMaxM + 32 * 40 + 16;

// `sbinom`: the block's shared-memory copy of the binomial table (row stride kBinomCols), still intact — unranking the
// winner from global memory is a chain of ~n+m dependent L2 reads, 8 us of the 20 the finalize took.
__device__ __forceinline__ void finalize_if_last(const LaunchParams& prm, unsigned char* scratch, const uint64_t* sbinom)
{
    __shared__ int s_is_last;
    if (threadIdx.x == 0) {
        __threadfence();                                   // this block's partial is visible before its ticket
        const unsigned t = atomicAdd(&prm.ctrl->ticket, 1u);
        s_is_last = (t + 1u == prm.total_blocks);
    }
    __syncthreads();
    if (!s_is_last) return;
    __threadfence();

    double*   s_M    = reinterpret_cast<double*>(scratch);                 // [kMaxM][kMaxM+1]
    double*   s_rinv = s_M + kMaxM * (kMaxM + 1);                          // [kMaxM]
    int*      s_S    = reinterpret_cast<int*>(s_rinv + kMaxM);             // [kMaxM]
    double*   s_wkey = reinterpret_cast<double*>(s_S + kMaxM);             // [32]
    uint64_t* s_wrank = reinterpret_cast<uint64_t*>(s_wkey + 32);          // [32]
    uint64_t* s_wcnt = s_wrank + 32;                                       // [3][32]
    uint64_t* s_best = s_wcnt + 96;                                        // [1] winning rank
    constexpr int kLd = kMaxM + 1;

    double   key = __longlong_as_double(0x7ff0000000000000LL);
    uint64_t rank = ~0ull, cs = 0, ci = 0, cf = 0;
    for (uint32_t i = threadIdx.x; i < prm.total_blocks; i += blockDim.x) {
        const BlockPartial* bp = prm.all_parts + i;
        const double k2 = __ldcg(&bp->key);
        const uint64_t r2 = __ldcg(&bp->rank);
        if (better(k2, r2, key, rank)) { key = k2; rank = r2; }
        cs += __ldcg(&bp->n_sing); ci += __ldcg(&bp->n_infeas); cf += __ldcg(&bp->n_feas);
    }
    const unsigned full = 0xffffffffu;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double   k2 = __shfl_down_sync(full, key, off);
        const uint64_t r2 = __shfl_down_sync(full, rank, off);
        if (better(k2, r2, key, rank)) { key = k2; rank = r2; }
        cs += __shfl_down_sync(full, cs, off);
        ci += __shfl_down_sync(full, ci, off);
        cf += __shfl_down_sync(full, cf, off);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = (int)(blockDim.x >> 5);
    if (lane == 0) { s_wkey[warp] = key; s_wrank[warp] = rank; s_wcnt[warp] = cs; s_wcnt[32 + warp] = ci; s_wcnt[64 + warp] = cf; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < n_warps; ++w) {
            if (better(s_wkey[w], s_wrank[w], key, rank)) { key = s_wkey[w]; rank = s_wrank[w]; }
            cs += s_wcnt[w]; ci += s_wcnt[32 + w]; cf += s_wcnt[64 + w];
        }
        enumgpu_partial* r = prm.record;
        r->key = key; r->best_rank = rank;
        r->n_bases = cs + ci + cf;                         // every visited rank is in exactly one class
        r->n_singular = cs; r->n_infeasible = ci; r->n_feasible = cf;
        r->m = prm.m; r->algo_used = prm.algo_used;
        for (int i = 0; i < kMaxM; ++i) { r->x_B[i] = 0.0; r->basis[i] = 0; }
        r->objective = __longlong_as_double(0x7ff8000000000000LL);
        s_best[0] = rank;
        if (rank != ~0ull) unrank_lex(sbinom, prm.n, prm.m, rank, s_S);
        prm.ctrl->unit_counter = 0ull;                     // ready for the next enqueue on this control block
        prm.ctrl->ticket = 0u;
    }
    __syncthreads();
    if (threadIdx.x < 32 && s_best[0] != ~0ull) {
        const int m = prm.m;
        if (lane <= m)
            for (int r = 0; r < m; ++r) s_M[r * kLd + lane] = lane < m ? prm.A[r + (size_t)s_S[lane] * prm.lda] : prm.b[r];
        __syncwarp();
        // (the warp spreads the independent elements of each step over its lanes; every element still receives
        // the operations of eval_basis_generic in the same order — the serial version took 8 us of a launch)
        for (int k = 0; k < m; ++k) {
            // first maximum of |M[r][k]| over r >= k: lane r holds row r's candidate, a shuffle arg-max picks the
            // largest value and, among equal ones, the lowest row (what the serial scan with '>' keeps)
            double best = (lane >= k && lane < m) ? fabs(s_M[lane * kLd + k]) : -1.0;
            int p = lane;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double v2 = __shfl_xor_sync(full, best, off);
                const int p2 = __shfl_xor_sync(full, p, off);
                if (v2 > best || (v2 == best && p2 < p)) { best = v2; p = p2; }
            }
            if (p != k && lane >= k && lane <= m) { const double t = s_M[k * kLd + lane]; s_M[k * kLd + lane] = s_M[p * kLd + lane]; s_M[p * kLd + lane] = t; }
            __syncwarp();
            const double rinv = __drcp_rn(s_M[k * kLd + k]);
            if (lane == 0) s_rinv[k] = rinv;
            const int cols = m - k, n_el = (m - 1 - k) * cols;          // rows k+1..m-1, columns k+1..m
            for (int e = lane; e < n_el; e += 32) {
                const int r = k + 1 + e / cols, j = k + 1 + e % cols;
                s_M[r * kLd + j] = fnma(__dmul_rn(s_M[r * kLd + k], rinv), s_M[k * kLd + j], s_M[r * kLd + j]);
            }
            __syncwarp();
        }
        enumgpu_partial* r = prm.record;
        double z = 0.0;                                             // lane 0's
        for (int j = m - 1; j >= 0; --j) {
            const double xj = __dmul_rn(s_M[j * kLd + m], s_rinv[j]);      // the same value in every lane
            __syncwarp();
            if (lane < j) s_M[lane * kLd + m] = fnma(s_M[lane * kLd + j], xj, s_M[lane * kLd + m]);
            if (lane == 0) {
                z = __fma_rn(prm.c[s_S[j]], xj, z);
                r->x_B[j] = xj; r->basis[j] = s_S[j];
            }
            __syncwarp();
        }
        if (lane == 0) r->objective = z;
    }
}

}  // namespace enumgpu
