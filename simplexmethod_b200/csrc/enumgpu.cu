// enumgpu.cu — host side of libenumgpu (C ABI of include/enumgpu.h) and the
// small service kernels (finalize, scale, FP64 peak probe).  The enumeration
// kernels live in k_independent.cuh and k_shared.cuh.
//
// No CPU fallback: every solve entry point needs a CUDA device and returns
// ENUMGPU_ERR_CUDA without one.  The only host arithmetic is argument checking,
// binomials and the merge of per-device partial records.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "enum_common.cuh"
#include "k_independent.cuh"
#include "k_shared.cuh"

using namespace enumgpu;

// ------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                        \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess)                                                          \
            return fail(ENUMGPU_ERR_CUDA, "%s failed: %s (%s:%d)", #call,               \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                    \
    } while (0)

// --------------------------------------------------------------- binomials
namespace {

struct BinomTable {
    uint64_t v[kBinomRows][kBinomCols];
    BinomTable()
    {
        // Pascal's triangle; 0 marks "would pass 2^63" (never hit for n<=64,k<=16)
        for (int n = 0; n < kBinomRows; ++n) {
            for (int k = 0; k < kBinomCols; ++k) v[n][k] = 0;
            v[n][0] = 1;
            for (int k = 1; k < kBinomCols && k <= n; ++k) {
                const uint64_t a = v[n - 1][k - 1], b = (k <= n - 1) ? v[n - 1][k] : 0;
                const bool bad = (a == 0) || ((k <= n - 1) && b == 0) || ((a + b) >> 63);
                v[n][k] = bad ? 0 : a + b;
            }
        }
    }
};
const BinomTable& binom_table()
{
    static const BinomTable t;   // immutable after construction (thread-safe init)
    return t;
}

}  // namespace

extern "C" uint64_t enumgpu_binomial(int32_t n, int32_t k)
{
    if (n < 0 || k < 0 || k > n || n > kMaxN) return 0;
    if (k > n - k) k = n - k;
    if (k > kMaxM) {
        // outside the table: multiplicative formula with overflow check
        unsigned __int128 r = 1;
        for (int i = 1; i <= k; ++i) {
            r = r * (unsigned)(n - k + i) / (unsigned)i;
            if (r >> 63) return 0;
        }
        return (uint64_t)r;
    }
    return binom_table().v[n][k];
}

static uint64_t binom_mk(int top, int k)   // C(top,k) for the (n<=64, k<=16) domain
{
    if (top < 0 || k < 0 || k > top) return 0;
    return binom_table().v[top][k];
}

extern "C" uint64_t enumgpu_rank(int32_t n, int32_t m, const int32_t* S)
{
    if (!S || m < 1 || m > kMaxM || n < m || n > kMaxN) return UINT64_MAX;
    uint64_t acc = 0;
    for (int i = 0; i < m; ++i) {
        if (S[i] < 0 || S[i] >= n || (i && S[i] <= S[i - 1])) return UINT64_MAX;
        acc += binom_mk(n - 1 - S[i], m - i);
    }
    return binom_mk(n, m) - 1 - acc;
}

extern "C" int enumgpu_unrank(int32_t n, int32_t m, uint64_t r, int32_t* S)
{
    if (!S || m < 1 || m > kMaxM || n < m || n > kMaxN) return fail(ENUMGPU_ERR_ARG, "unrank: bad (n,m)");
    if (r >= binom_mk(n, m)) return fail(ENUMGPU_ERR_RANGE, "unrank: rank out of range");
    int v = 0;
    for (int i = 0; i < m; ++i) {
        for (;;) {
            const uint64_t cnt = binom_mk(n - 1 - v, m - 1 - i);
            if (cnt <= r) { r -= cnt; ++v; } else break;
        }
        S[i] = v++;
    }
    return 0;
}

extern "C" uint64_t enumgpu_shard_begin(int32_t m, int32_t n, uint64_t rank_begin, uint64_t rank_end, int32_t i, int32_t n_shards)
{
    if (rank_end < rank_begin || n_shards < 1) return rank_end;
    if (i <= 0) return rank_begin;
    if (i >= n_shards) return rank_end;
    return rank_begin + shard_boundary(m, n, rank_end - rank_begin, i, n_shards);
}

extern "C" int enumgpu_version(void) { return ENUMGPU_VERSION; }
extern "C" const char* enumgpu_last_error(void) { return g_err; }

extern "C" int enumgpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ---------------------------------------------------------- service kernels

// max |A_ij| -> *out   (one block)
__global__ void k_scale(const double* __restrict__ A, int m, int n, int lda, double* out)
{
    __shared__ double s[256];
    double v = 0.0;
    for (int idx = threadIdx.x; idx < m * n; idx += blockDim.x) {
        const int j = idx / m, i = idx - j * m;
        v = fmax(v, fabs(A[i + (size_t)j * lda]));
    }
    s[threadIdx.x] = v;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) s[threadIdx.x] = fmax(s[threadIdx.x], s[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = s[0];
}

// An enqueue over an empty rank range launches no enumeration block: this writes its neutral record.
__global__ void k_empty_record(int m, int algo_used, enumgpu_partial* __restrict__ out)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    enumgpu_partial r;
    r.key = __longlong_as_double(0x7ff0000000000000LL); r.best_rank = ~0ull;
    r.n_bases = r.n_singular = r.n_infeasible = r.n_feasible = 0;
    r.m = m; r.algo_used = algo_used;
    for (int i = 0; i < kMaxM; ++i) { r.x_B[i] = 0.0; r.basis[i] = 0; }
    r.objective = __longlong_as_double(0x7ff8000000000000LL);
    *out = r;
}

// Block-wide partial-pivot elimination of W = [B | further columns] (column-major, m rows, `width` >= m+1 columns,
// in global memory, overwritten), the frozen arithmetic of DESIGN.md §3: every column right of B receives the same
// operations in the same order as column m (= b) does in eval_basis_generic, so adding columns changes no bit of
// the others.  The block only spreads independent elements of one step over its threads; the data-dependent
// decisions (pivot search, thresholds) are made by thread 0 in index order.  Returns true (on every thread) if the
// basis is singular under pivot_rule.
__device__ bool block_eliminate(double* __restrict__ W, int m, int width, double thr, int pivot_rule, double rel_eps,
                                double* __restrict__ rinv)
{
    __shared__ int s_p, s_stop;
    const int tid = threadIdx.x, nt = blockDim.x;
    const size_t ld = (size_t)m;
    double pmax = 0.0, pmin = __longlong_as_double(0x7ff0000000000000LL);   // thread 0 only
    for (int k = 0; k < m; ++k) {
        if (tid == 0) {
            int p = k;
            double best = fabs(W[k + k * ld]);
            for (int r = k + 1; r < m; ++r) {
                const double v = fabs(W[r + k * ld]);
                if (v > best) { best = v; p = r; }
            }
            s_p = p;
            s_stop = !(best > thr);
            if (best > pmax) pmax = best;
            if (best < pmin) pmin = best;
        }
        __syncthreads();
        if (s_stop) return true;
        const int p = s_p;
        if (p != k)
            for (int j = k + tid; j < width; j += nt) { const double t = W[k + j * ld]; W[k + j * ld] = W[p + j * ld]; W[p + j * ld] = t; }
        __syncthreads();
        const double ri = __drcp_rn(W[k + k * ld]);
        if (tid == 0) rinv[k] = ri;
        const int rows = m - 1 - k, cols = width - 1 - k;         // rows k+1..m-1, columns k+1..width-1
        for (long long e = tid; e < (long long)rows * cols; e += nt) {
            const int r = k + 1 + (int)(e % rows), j = k + 1 + (int)(e / rows);
            W[r + j * ld] = fnma(__dmul_rn(W[r + k * ld], ri), W[k + j * ld], W[r + j * ld]);
        }
        __syncthreads();
    }
    if (tid == 0) s_stop = (pivot_rule == ENUMGPU_PIVOT_RELATIVE) && !(pmin > __dmul_rn(rel_eps, pmax));
    __syncthreads();
    return s_stop;
}

// Column sweep of column m of an eliminated W: x[0..m) and, on thread 0, z and the class (0 feasible, 1 infeasible).
__device__ void block_solve_x(double* __restrict__ W, const double* __restrict__ cB, int m, double eps_feas,
                              const double* __restrict__ rinv, double* __restrict__ x, double* z_out, int* cls_out)
{
    __shared__ double s_x;
    const int tid = threadIdx.x, nt = blockDim.x;
    const size_t ld = (size_t)m;
    bool infeasible = false;       // thread 0 only
    double z = 0.0;
    for (int j = m - 1; j >= 0; --j) {
        if (tid == 0) {
            const double xj = __dmul_rn(W[j + m * ld], rinv[j]);
            s_x = xj;
            x[j] = xj;
            infeasible |= !(xj >= -eps_feas);
            z = __fma_rn(cB[j], xj, z);
        }
        __syncthreads();
        const double xj = s_x;
        for (int i = tid; i < j; i += nt) W[i + m * ld] = fnma(W[i + j * ld], xj, W[i + m * ld]);
        __syncthreads();
    }
    if (tid == 0) { *z_out = z; *cls_out = infeasible ? 1 : 0; }
}

// One basis of ANY size (the device side of enumgpu_eval_basis, which stands in for Canonical::GetBasicSolution /
// IsFeasibleBasis of a Canonical of any dimensions): one block on W = [B | b] (m x (m+1)).
// out: x[0..m), then z, then the class as a double.
__global__ void __launch_bounds__(256)
k_eval_any(double* __restrict__ W, const double* __restrict__ cB, int m, double thr, double eps_feas,
           int pivot_rule, double rel_eps, double* __restrict__ rinv, double* __restrict__ out)
{
    if (block_eliminate(W, m, m + 1, thr, pivot_rule, rel_eps, rinv)) { if (threadIdx.x == 0) out[m + 1] = 2.0; return; }
    double z;
    int cls;
    block_solve_x(W, cB, m, eps_feas, rinv, out, &z, &cls);
    if (threadIdx.x == 0) { out[m] = z; out[m + 1] = (double)cls; }
}

// The certificate of a basis (enumgpu_certify, DESIGN.md §3): block i certifies basis S_all[i*m .. i*m+m) in its own
// slab of scratch (certify_slab doubles): W = [B | b | A_0 .. A_{n-1} | e_0 .. e_{m-1}] (m x (2m+n+1)), then c_B and
// room for 1/pivot; it writes out_all[i].  After the shared elimination and x, thread t sweeps extra column t:
// u_j = B^-1 a_j and r_j for t = j < n, w_i = B^-1 e_i and y_i for t = n+i.  Thread 0 then decides the verdict in
// column order.  A: packed (lda = m); c: all n costs.
constexpr int kCertifyThreads = 128;
static_assert(kCertifyThreads >= kMaxN + kMaxM, "one thread per extra column");
__host__ __device__ inline size_t certify_slab(int m, int n) { return (size_t)m * (2 * m + n + 1) + 2 * (size_t)m; }
__global__ void __launch_bounds__(kCertifyThreads)
k_certify(const double* __restrict__ A, const double* __restrict__ b, const double* __restrict__ c,
          const int* __restrict__ S_all, int m, int n, int maximize, double thr, double eps_feas, int pivot_rule,
          double rel_eps, double eps_opt, double* __restrict__ scratch, enumgpu_certificate* __restrict__ out_all)
{
    const int* __restrict__ S = S_all + (size_t)blockIdx.x * m;
    double* __restrict__ W = scratch + (size_t)blockIdx.x * certify_slab(m, n);
    double* __restrict__ cB = W + (size_t)m * (2 * m + n + 1);
    double* __restrict__ rinv = cB + m;
    enumgpu_certificate* __restrict__ out = out_all + blockIdx.x;
    for (int e = threadIdx.x; e < m * (2 * m + n + 1); e += blockDim.x) {
        const int j = e / m, r = e - j * m;
        W[e] = j < m ? A[r + (size_t)S[j] * m] : j == m ? b[r] : j <= m + n ? A[r + (size_t)(j - m - 1) * m]
             : (r == j - m - 1 - n ? 1.0 : 0.0);
    }
    for (int j = threadIdx.x; j < m; j += blockDim.x) cB[j] = c[S[j]];
    __syncthreads();
    const int tid = threadIdx.x;
    const size_t ld = (size_t)m;
    if (tid == 0) { out->m = m; out->n = n; out->entering = -1; }
    if (block_eliminate(W, m, 2 * m + n + 1, thr, pivot_rule, rel_eps, rinv)) {
        if (tid == 0) { out->basis_class = ENUMGPU_BASIS_SINGULAR; out->status = ENUMGPU_CERT_UNDECIDED; }
        return;
    }
    int cls = 0;
    block_solve_x(W, cB, m, eps_feas, rinv, out->x_B, &out->objective, &cls);
    if (tid < n + m) {                      // the same column sweep as for x, on column m+1+tid
        double* col = W + (size_t)(m + 1 + tid) * ld;
        double t[kMaxM];
        for (int i = 0; i < m; ++i) t[i] = col[i];
        double acc = tid < n ? c[tid] : 0.0;
        for (int k = m - 1; k >= 0; --k) {
            const double uk = __dmul_rn(t[k], rinv[k]);
            col[k] = uk;
            for (int i = 0; i < k; ++i) t[i] = fnma(W[i + k * ld], uk, t[i]);
        }
        for (int k = m - 1; k >= 0; --k)
            acc = tid < n ? fnma(cB[k], col[k], acc) : __fma_rn(cB[k], col[k], acc);
        if (tid < n) out->reduced_cost[tid] = acc;
        else out->y[tid - n] = acc;
    }
    __syncthreads();
    if (tid != 0) return;
    out->basis_class = cls;
    int entering = -1;
    bool improving = false, nan = false;
    for (int j = 0; j < n; ++j) {
        bool basic = false;
        for (int k = 0; k < m; ++k) basic |= (S[k] == j);
        if (basic) continue;
        const double r = out->reduced_cost[j], rk = maximize ? -r : r;
        if (rk != rk) { nan = true; continue; }
        if (!(rk < -eps_opt)) continue;
        improving = true;
        if (entering >= 0) continue;
        const double* u = W + (size_t)(m + 1 + j) * ld;
        bool ray = true;
        for (int k = 0; k < m; ++k) ray &= (u[k] <= eps_opt);
        if (ray) entering = j;
    }
    for (int j = 0; j < n; ++j) out->ray[j] = 0.0;
    if (entering >= 0) {
        const double* u = W + (size_t)(m + 1 + entering) * ld;
        for (int k = 0; k < m; ++k) out->ray[S[k]] = -u[k];
        out->ray[entering] = 1.0;
    }
    out->entering = entering;
    out->status = entering >= 0 ? ENUMGPU_CERT_UNBOUNDED : (!improving && !nan) ? ENUMGPU_CERT_OPTIMAL : ENUMGPU_CERT_UNDECIDED;
}

// Register-resident DFMA chains: the measured FP64 roofline denominator.  kChains independent chains per thread;
// the per-SM microbenchmark (scripts/micro/fp64_lat.cu) reaches 1.98 of the 2 DFMA warp-instructions per cycle an
// SM can issue with 4 chains x 16 warps, and so does this kernel with one 512-thread block per SM.
template <int kChains>
__global__ void __launch_bounds__(512) k_dfma_peak(double* out, int iters, double a, double b, unsigned long long* clk)
{
    double v[kChains];
#pragma unroll
    for (int c = 0; c < kChains; ++c) v[c] = threadIdx.x + c;
    unsigned long long c0 = 0, g0 = 0;
    if (clk && blockIdx.x == 0 && threadIdx.x == 0) { c0 = clock64(); asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g0)); }
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
#pragma unroll
            for (int c = 0; c < kChains; ++c) v[c] = __fma_rn(v[c], a, b);
        }
    }
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < kChains; ++c) s += v[c];
    if (s == 12345.678) out[0] = s;   // never true; keeps the chains alive
    if (clk && blockIdx.x == 0 && threadIdx.x == 0) {       // SM cycles and nanoseconds this block's thread 0 spent in the loop
        unsigned long long g1;
        const unsigned long long c1 = clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
        clk[0] = c1 - c0; clk[1] = g1 - g0;
    }
}

// Best of a few occupancies (the FP64 pipe saturates from 16 warps x 4 chains per SM on; more resident warps only
// add scheduling noise) and of `repeats` launches each; ~30 ms per launch so that clocks settle under load.
// detail[1] = SM clock in MHz during the best launch (clock64 against globaltimer, one thread of block 0); detail[0] =
// that block's own DFMA warp-instructions per SM cycle (a per-block figure: meaningful for the one-block-per-SM
// configurations only).  Tells a probe below nominal apart: issue rate or clock.
extern "C" double enumgpu_fp64_peak_detail(int32_t repeats, double* detail)
{
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
        fail(ENUMGPU_ERR_CUDA, "fp64 peak probe: no CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
        return -1.0;
    }
    if (repeats < 1) repeats = 3;
    double* d = nullptr;
    cudaEvent_t e0, e1;
    if (cudaMalloc(&d, 32) != cudaSuccess || cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) {
        fail(ENUMGPU_ERR_CUDA, "fp64 peak probe: %s", cudaGetErrorString(cudaGetLastError()));
        return -1.0;
    }
    double best = 0.0;
    const struct { int chains, threads, blocks_per_sm; } cfg[] = {{4, 512, 1}, {8, 512, 1}, {8, 256, 4}, {4, 512, 2}};
    for (const auto& c : cfg) {
        const int blocks = sms * c.blocks_per_sm;
        // ~6e7 cycles of FP64 pipe per launch: iters * 16 * chains DFMA per thread, 2 cycles per warp-DFMA per sub-core
        const int iters = (int)(6.0e7 / (16.0 * c.chains * 2.0 * (c.threads / 128) * c.blocks_per_sm));
        for (int r = 0; r < repeats + 1; ++r) {
            cudaEventRecord(e0);
            unsigned long long* clk = reinterpret_cast<unsigned long long*>(d + 1);
            if (c.chains == 4) k_dfma_peak<4><<<blocks, c.threads>>>(d, iters, 1.0000001, 1e-9, clk);
            else k_dfma_peak<8><<<blocks, c.threads>>>(d, iters, 1.0000001, 1e-9, clk);
            cudaEventRecord(e1);
            if (cudaEventSynchronize(e1) != cudaSuccess) { fail(ENUMGPU_ERR_CUDA, "fp64 peak probe: %s", cudaGetErrorString(cudaGetLastError())); best = -1.0; break; }
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            const double flops = 2.0 * 16.0 * c.chains * (double)iters * (double)blocks * c.threads;
            const double tf = flops / (ms * 1e-3) * 1e-12;
            if (r > 0 && tf > best) {
                best = tf;
                unsigned long long h[2] = {0, 0};
                if (detail && cudaMemcpy(h, clk, 16, cudaMemcpyDeviceToHost) == cudaSuccess && h[0] && h[1]) {
                    // warp-DFMAs of one SM = iters * 16 * chains * warps per SM
                    detail[0] = (double)iters * 16.0 * c.chains * (c.threads / 32) * c.blocks_per_sm / (double)h[0];
                    detail[1] = (double)h[0] / (double)h[1] * 1e3;
                }
            }
        }
        if (best < 0) break;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    return best;
}

extern "C" double enumgpu_fp64_peak_tflops(int32_t repeats) { return enumgpu_fp64_peak_detail(repeats, nullptr); }

// ------------------------------------------------------------ launch logic

// Stream-ordered device buffer that returns itself to the pool when it goes out of scope — on the
// error paths too (the free is enqueued behind the kernels that use the buffer).
struct StreamBuf {
    void* p = nullptr;
    cudaStream_t st = nullptr;
    StreamBuf() = default;
    StreamBuf(const StreamBuf&) = delete;
    StreamBuf& operator=(const StreamBuf&) = delete;
    ~StreamBuf() { if (p) cudaFreeAsync(p, st); }
    cudaError_t alloc(size_t bytes, cudaStream_t s) { st = s; return cudaMallocAsync(&p, bytes, s); }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

// Stream-ordered allocations come from the device's default memory pool.  Its
// default release threshold (0) hands memory back to the OS at every
// synchronisation, which makes each solve pay a fresh OS allocation; keep it.
static void keep_pool_memory(int dev)
{
    static const bool enabled = [] { const char* e = getenv("ENUMGPU_KEEP_POOL"); return !(e && e[0] == '0'); }();
    if (!enabled) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    } else cudaGetLastError();
}

template <int M>
static cudaError_t launch_independent(const LaunchParams& prm, BlockPartial* parts, uint32_t blocks, cudaStream_t st)
{
    const size_t smem = (size_t)(prm.n * M + M + prm.n) * sizeof(double) + sizeof(uint64_t) * kBinomRows * kBinomCols + kFinalizeScratch;
    cudaError_t e = cudaFuncSetAttribute(k_independent<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_independent<M><<<blocks, kIndepThreads, smem, st>>>(prm, parts);
    return cudaGetLastError();
}

static cudaError_t dispatch_independent(const LaunchParams& prm, BlockPartial* parts, uint32_t blocks, cudaStream_t st)
{
    if (prm.pivot_rule == ENUMGPU_PIVOT_ABSOLUTE) switch (prm.m) {
#define ENUMGPU_CASE(M_) case M_: return launch_independent<M_>(prm, parts, blocks, st);
#ifdef ENUMGPU_DEV_BUILD      // kernel experiments: fewer instantiations (the others fall to the run-time-m kernel)
        ENUMGPU_CASE(7) ENUMGPU_CASE(8) ENUMGPU_CASE(10)
#else
        ENUMGPU_CASE(1) ENUMGPU_CASE(2) ENUMGPU_CASE(3) ENUMGPU_CASE(4)
        ENUMGPU_CASE(5) ENUMGPU_CASE(6) ENUMGPU_CASE(7) ENUMGPU_CASE(8)
        ENUMGPU_CASE(9) ENUMGPU_CASE(10) ENUMGPU_CASE(11) ENUMGPU_CASE(12)
#endif
#undef ENUMGPU_CASE
    }
    // m = 13..16, and every m under the relative singularity rule: run-time-m kernel (arrays in local memory)
    const size_t smem = (size_t)(prm.n * prm.m + prm.m + prm.n) * sizeof(double) + sizeof(uint64_t) * kBinomRows * kBinomCols + kFinalizeScratch;
    cudaError_t e = cudaFuncSetAttribute(k_independent_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_independent_generic<<<blocks, kIndepThreads, smem, st>>>(prm, parts);
    return cudaGetLastError();
}

// Per-device copies of the constant lookup tables (binomials; the item tables of k_shared for one value of
// g_max = n - (m-4)), made once per process and device with a synchronous copy and never freed or changed, so
// any stream may read them.  Uploading them on every call cost two pageable H2D copies (~25 us) per launch.
struct DeviceTables {
    int rcp_state = 0;                       // 0 not checked, 1 k_shared's reciprocal == __drcp_rn here, 2 it is not
    const uint64_t* binom = nullptr;
    std::map<int, std::pair<const uint32_t*, size_t>> items;   // g_max -> (triples then 4-tuples, number of triples)
    std::map<int, const uint64_t*> wprefix;                    // n << 8 | m -> weight prefix sums (k_shared.cuh)
};
static std::mutex g_tables_mu;
static std::map<int, DeviceTables> g_tables;

// a cached pointer stops being device memory if the application resets the device between calls
static bool still_device_memory(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice;
}

static int device_binom(int dev, const uint64_t** out)
{
    std::lock_guard<std::mutex> lock(g_tables_mu);
    DeviceTables& t = g_tables[dev];
    if (t.binom && !still_device_memory(t.binom)) t = DeviceTables();
    if (!t.binom) {
        void* p = nullptr;
        CU(cudaMalloc(&p, sizeof(BinomTable)));
        CU(cudaMemcpy(p, &binom_table().v[0][0], sizeof(BinomTable), cudaMemcpyHostToDevice));
        t.binom = static_cast<const uint64_t*>(p);
    }
    *out = t.binom;
    return 0;
}

static int device_items(int dev, int g_max, const uint32_t** tri, const uint32_t** quad, uint32_t* n_tri = nullptr, uint32_t* n_quad = nullptr)
{
    std::lock_guard<std::mutex> lock(g_tables_mu);
    DeviceTables& t = g_tables[dev];
    auto it = t.items.find(g_max);
    if (it != t.items.end() && !still_device_memory(it->second.first)) { t.items.erase(it); it = t.items.end(); }
    if (it == t.items.end()) {
        std::vector<uint32_t> h = make_triples(g_max);          // item tables: triples, then 4-tuples, each padded
        const size_t n_tri = h.size();
        h.insert(h.end(), (size_t)kItemTabPad, 0u);
        const std::vector<uint32_t> q = make_quads(kTailR - 1);
        h.insert(h.end(), q.begin(), q.end());
        h.insert(h.end(), (size_t)kItemTabPad, 0u);
        void* p = nullptr;
        CU(cudaMalloc(&p, sizeof(uint32_t) * (h.size() + 1)));
        CU(cudaMemcpy(p, h.data(), sizeof(uint32_t) * h.size(), cudaMemcpyHostToDevice));
        it = t.items.emplace(g_max, std::make_pair(static_cast<const uint32_t*>(p), n_tri)).first;
    }
    *tri = it->second.first;
    *quad = it->second.first + it->second.second + kItemTabPad;
    if (n_tri) *n_tri = (uint32_t)it->second.second;
    if (n_quad) *n_quad = (uint32_t)binom_mk(kTailR - 1, 4);
    return 0;
}

static int device_wprefix(int dev, int n, int m, const uint64_t** out)
{
    std::lock_guard<std::mutex> lock(g_tables_mu);
    DeviceTables& t = g_tables[dev];
    const int key = (n << 8) | m;
    auto it = t.wprefix.find(key);
    if (it != t.wprefix.end() && !still_device_memory(it->second)) { t.wprefix.erase(it); it = t.wprefix.end(); }
    if (it == t.wprefix.end()) {
        auto C = [](int top, int k) -> uint64_t { return binom_mk(top, k); };
        const std::vector<uint64_t> h = make_weight_prefix(C, n, m);
        void* p = nullptr;
        CU(cudaMalloc(&p, sizeof(uint64_t) * h.size()));
        CU(cudaMemcpy(p, h.data(), sizeof(uint64_t) * h.size(), cudaMemcpyHostToDevice));
        it = t.wprefix.emplace(key, static_cast<const uint64_t*>(p)).first;
    }
    *out = it->second;
    return 0;
}

struct Resolved {       // options with defaults applied and the range checked
    double eps_feas, eps_piv;
    uint64_t begin, end, total;
    int algo, rule;
    uint32_t shard_index, shard_count;
};

static int resolve(const enumgpu_problem* p, const enumgpu_options* o, Resolved* r, bool host_ptrs)
{
    if (!p) return fail(ENUMGPU_ERR_ARG, "problem is NULL");
    if (!p->A_colmajor || !p->b || !p->c) return fail(ENUMGPU_ERR_ARG, "A, b or c is NULL");
    if (p->m < 1 || p->m > kMaxM) return fail(ENUMGPU_ERR_ARG, "m=%d outside 1..%d", p->m, kMaxM);
    if (p->n < p->m) return fail(ENUMGPU_ERR_ARG, "n=%d < m=%d: no basis exists", p->n, p->m);
    if (p->n > kMaxN) return fail(ENUMGPU_ERR_ARG, "n=%d above ENUMGPU_MAX_N=%d", p->n, kMaxN);
    if (p->lda < p->m) return fail(ENUMGPU_ERR_ARG, "lda=%d < m=%d", p->lda, p->m);
    r->total = binom_mk(p->n, p->m);
    if (r->total == 0) return fail(ENUMGPU_ERR_RANGE, "C(%d,%d) does not fit 63 bits", p->n, p->m);
    r->rule = o ? o->pivot_rule : ENUMGPU_PIVOT_ABSOLUTE;
    if (r->rule != ENUMGPU_PIVOT_ABSOLUTE && r->rule != ENUMGPU_PIVOT_RELATIVE) return fail(ENUMGPU_ERR_ARG, "unknown pivot_rule %d", r->rule);
    r->eps_feas = (o && o->eps_feas >= 0) ? o->eps_feas : 1e-9;
    r->eps_piv = (o && o->eps_piv >= 0) ? o->eps_piv : (r->rule == ENUMGPU_PIVOT_RELATIVE ? (double)p->m * 0x1p-52 : 1e-9);
    // -0.0 passes the tests above and means 0.  Store +0.0: k_shared classifies leaf components by the high word of
    // -eps_feas, whose sign bit must be set (with -(-0.0) = +0.0 every positive component would count as negative).
    if (r->eps_feas == 0.0) r->eps_feas = 0.0;
    if (r->eps_piv == 0.0) r->eps_piv = 0.0;
    r->begin = o ? o->rank_begin : 0;
    r->end = o ? o->rank_end : 0;
    if (r->begin == 0 && r->end == 0) r->end = r->total;
    if (r->begin > r->end || r->end > r->total)
        return fail(ENUMGPU_ERR_RANGE, "rank range [%llu,%llu) outside [0,%llu)", (unsigned long long)r->begin,
                    (unsigned long long)r->end, (unsigned long long)r->total);
    r->shard_index = 0; r->shard_count = 1;
    if (o && (o->shard_count != 0 || o->shard_index != 0)) {
        if (o->shard_count < 1 || o->shard_index < 0 || o->shard_index >= o->shard_count)
            return fail(ENUMGPU_ERR_ARG, "shard %d of %d is not valid", o->shard_index, o->shard_count);
        r->shard_index = (uint32_t)o->shard_index; r->shard_count = (uint32_t)o->shard_count;
    }
    r->algo = o ? o->algo : ENUMGPU_ALGO_AUTO;
    if (r->algo < ENUMGPU_ALGO_AUTO || r->algo > ENUMGPU_ALGO_SHARED) return fail(ENUMGPU_ERR_ARG, "unknown algo %d", r->algo);
    if (host_ptrs) {
        for (int j = 0; j < p->n; ++j) {
            if (!std::isfinite(p->c[j])) return fail(ENUMGPU_ERR_NONFINITE, "c[%d] is not finite", j);
            for (int i = 0; i < p->m; ++i)
                if (!std::isfinite(p->A_colmajor[i + (size_t)j * p->lda])) return fail(ENUMGPU_ERR_NONFINITE, "A(%d,%d) is not finite", i, j);
        }
        for (int i = 0; i < p->m; ++i)
            if (!std::isfinite(p->b[i])) return fail(ENUMGPU_ERR_NONFINITE, "b[%d] is not finite", i);
    }
    return 0;
}

// Device scratch of one enqueue: the control block (zero on entry; the last block of the enqueue resets it) and
// room for the per-block partials.  A handle owns one and reuses it call after call — no allocation and no
// memset on the hot path; the handle-free entry points take both from the stream-ordered pool per call.
struct Scratch {
    Ctrl* ctrl = nullptr;
    BlockPartial* parts = nullptr;
    size_t parts_cap = 0;      // elements
    unsigned char* queue = nullptr;   // survivor stacks of the shared kernel's warps (k_shared.cuh: queue_warp_bytes(n) each)
    size_t queue_cap = 0;      // bytes
};

static int scratch_reserve_queue(Scratch* sc, size_t bytes, cudaStream_t st)
{
    if (bytes <= sc->queue_cap) return 0;
    void* p = nullptr;
    CU(cudaMallocAsync(&p, bytes, st));
    if (sc->queue) cudaFreeAsync(sc->queue, st);
    sc->queue = static_cast<unsigned char*>(p);
    sc->queue_cap = bytes;
    return 0;
}

static int scratch_reserve(Scratch* sc, size_t n_parts, cudaStream_t st)
{
    if (n_parts <= sc->parts_cap) return 0;
    size_t cap = sc->parts_cap ? sc->parts_cap : 1024;
    while (cap < n_parts) cap *= 2;
    void* p = nullptr;
    CU(cudaMallocAsync(&p, cap * sizeof(BlockPartial), st));
    if (sc->parts) cudaFreeAsync(sc->parts, st);          // stream-ordered: earlier enqueues on st are done with it
    sc->parts = static_cast<BlockPartial*>(p);
    sc->parts_cap = cap;
    return 0;
}

// Is the branch-free reciprocal of k_shared bit-identical to __drcp_rn on this device with this build?
// Checked once per process and device (a 4 M-operand run of the self-test, ~0.1 ms) before the shared kernel is
// first used; on a mismatch — a toolkit or driver that expands the intrinsic differently — the library falls back
// to the independent kernel (plain __drcp_rn) and says so in enumgpu_last_error().
static int rcp_selftest_device(uint64_t n_operands, uint64_t seed, uint64_t* n_mismatch, double* first_bad, cudaStream_t st);
static bool shared_rcp_trusted(int dev);

// Enqueue everything for one rank range on one stream of the current device.
// scale_host < 0: max|A_ij| is computed on the device first (one synchronisation of st).
static int enqueue_range(const enumgpu_problem* pd, double scale_host, const Resolved& rs, uint64_t begin, uint64_t end,
                         uint32_t shard_index, uint32_t shard_count,
                         cudaStream_t st, enumgpu_partial* partial_dev, int32_t* n_launches, Scratch* scratch = nullptr,
                         unsigned long long* list_count = nullptr, uint64_t* list_ranks = nullptr, uint64_t list_cap = 0,
                         double list_key_max = INFINITY)
{
    int launches = 0;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    keep_pool_memory(dev);
    const uint64_t* d_binom = nullptr;                      // per-device constant table
    {
        const int rc_t = device_binom(dev, &d_binom);
        if (rc_t) return rc_t;
    }

    if (scale_host < 0 && rs.rule == ENUMGPU_PIVOT_ABSOLUTE) {
        StreamBuf b_scale;
        CU(b_scale.alloc(sizeof(double), st));
        double* d_scale = b_scale.as<double>();
        k_scale<<<1, 256, 0, st>>>(pd->A_colmajor, pd->m, pd->n, pd->lda, d_scale);
        CU(cudaGetLastError());
        ++launches;
        // the threshold is a launch parameter: fetch the scale (8 bytes)
        CU(cudaMemcpyAsync(&scale_host, d_scale, sizeof(double), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }

    LaunchParams prm;
    prm.A = pd->A_colmajor; prm.b = pd->b; prm.c = pd->c; prm.binom = d_binom;
    prm.m = pd->m; prm.n = pd->n; prm.lda = pd->lda; prm.maximize = pd->maximize ? 1 : 0;
    prm.eps_feas = rs.eps_feas;
    prm.pivot_rule = rs.rule;
    prm.thr = rs.rule == ENUMGPU_PIVOT_RELATIVE ? 0.0 : rs.eps_piv * scale_host;
    prm.rel_eps = rs.rule == ENUMGPU_PIVOT_RELATIVE ? rs.eps_piv : 0.0;
    prm.rank_begin = begin; prm.rank_end = end; prm.chunk = 1;
    prm.shard_index = 0; prm.shard_count = 1;
    prm.list_count = list_count; prm.list_ranks = list_ranks; prm.list_cap = list_cap; prm.list_key_max = list_key_max;
    const bool first_shard = (shard_index == 0), last_shard = (shard_index + 1 == shard_count);

    int algo = rs.algo;
    if (algo == ENUMGPU_ALGO_AUTO) algo = shared_supported(prm.m, prm.n) ? ENUMGPU_ALGO_SHARED : ENUMGPU_ALGO_INDEPENDENT;
    if (algo == ENUMGPU_ALGO_SHARED && !shared_supported(prm.m, prm.n)) algo = ENUMGPU_ALGO_INDEPENDENT;
    // the relative rule decides after the last pivot: nothing can be pruned at a shared prefix (enumgpu.h)
    if (rs.rule == ENUMGPU_PIVOT_RELATIVE) algo = ENUMGPU_ALGO_INDEPENDENT;
    // k_shared's branch-free reciprocal equals __drcp_rn only for 2^-1000 < |pivot| < 2^1000.  Accepted
    // pivots satisfy thr < |pivot| <= 2^m * max|A|, so the kernel is used only when those bounds sit
    // inside that range (always, unless the caller sets eps_piv = 0 or the data is scaled absurdly);
    // otherwise the independent kernel (plain __drcp_rn) runs — same arithmetic, slower.
    if (algo == ENUMGPU_ALGO_SHARED && !(prm.thr >= 1e-290 && scale_host <= 1e290)) algo = ENUMGPU_ALGO_INDEPENDENT;
    if (algo == ENUMGPU_ALGO_SHARED && !shared_rcp_trusted(dev)) algo = ENUMGPU_ALGO_INDEPENDENT;
    prm.algo_used = algo;

    // independent kernel over [b0, b1): grid geometry
    auto indep_geom = [&](uint64_t b0, uint64_t b1, uint32_t* chunk_out) -> uint64_t {
        const uint64_t span = b1 - b0;
        if (span == 0) { *chunk_out = 1; return 0; }
        const uint64_t want_threads = (uint64_t)sms * 2048 * 8;
        uint64_t chunk = (span + want_threads - 1) / want_threads;
        if (chunk < 1) chunk = 1;
        if (chunk > 1024) chunk = 1024;
        *chunk_out = (uint32_t)chunk;
        const uint64_t threads = (span + chunk - 1) / chunk;
        return (threads + kIndepThreads - 1) / kIndepThreads;
    };
    // blocks of the independent kernel owned by this shard (block windows are dealt round-robin)
    auto shard_blocks = [&](uint64_t blocks) -> uint64_t {
        return blocks > shard_index ? (blocks - shard_index + shard_count - 1) / shard_count : 0;
    };

    // ---- geometry of every launch of this enqueue (the kernels need the total block count: the block that
    // ---- finishes last, whichever launch it belongs to, writes the record) ----
    uint32_t chunk_head = 1, chunk_tail = 1, chunk_all = 1;
    uint64_t head_blocks = 0, tail_blocks = 0, k2_blocks = 0, all_blocks = 0;
    uint64_t lo = begin, hi = end;
    SharedParams sp;
    size_t smem = 0;
    int wpc = 0;
    const uint32_t *d_tri = nullptr, *d_quad = nullptr;          // per-device constant item tables
    if (algo == ENUMGPU_ALGO_SHARED) {
        // The shared kernel works on whole child tasks (all bases with the same
        // first m-4 columns).  [lo, hi) is the child-aligned core of the range;
        // the ragged head [begin, lo) and tail [hi, end) — each shorter than one
        // child — go to the independent kernel.  Same arithmetic, same bits.
        const int m = prm.m, n = prm.n, P = m - kT;
        // the atomic piece of work containing rank r: a child task, or — if its column is one of the
        // last kTailR — the tail group of its parent (all children from column t0 on are processed together)
        auto child_of = [&](uint64_t r, uint64_t* first, uint64_t* count) {
            int32_t S[kMaxM];
            enumgpu_unrank(n, m, r, S);
            const int t0 = std::max(S[P - 2] + 1, n - kTailR);
            if (S[P - 1] >= t0) {
                S[P - 1] = t0;
                for (int i = 0; i < kT; ++i) S[P + i] = t0 + 1 + i;
                *first = enumgpu_rank(n, m, S);
                *count = binom_mk(n - t0, kT + 1);
                return;
            }
            const int rc = n - 1 - S[P - 1];
            uint64_t within = binom_mk(rc, kT) - 1;
            for (int i = 0; i < kT; ++i) within -= binom_mk(n - 1 - S[P + i], kT - i);
            *first = r - within;
            *count = binom_mk(rc, kT);
        };
        if (begin < end) {
            uint64_t f, c;
            child_of(begin, &f, &c);
            lo = (f == begin) ? begin : f + c;
            if (end < rs.total) { child_of(end, &f, &c); hi = f; }
            if (lo > hi) { lo = hi = begin; }
        }
        if (lo >= hi) {                       // no whole child inside: everything is "head"
            lo = hi = end;
        }
        head_blocks = first_shard ? indep_geom(begin, lo, &chunk_head) : 0;
        tail_blocks = last_shard ? indep_geom(hi, end, &chunk_tail) : 0;
        sp.lo = lo; sp.hi = hi;
        if (lo < hi) {
            const size_t cta = shared_cta_bytes(m, n) + 32, per_warp = (shared_warp_bytes(m, n) + 15) & ~size_t(15);
            int max_smem = 0;
            CU(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
#ifdef ENUMGPU_CHECK
            max_smem -= 1024;                 // the checked build's static window table
#endif
            wpc = (int)(((size_t)max_smem - cta) / per_warp);
            if (wpc > kMaxWarps) wpc = kMaxWarps;
            if (wpc < 1) return fail(ENUMGPU_ERR_ARG, "shared kernel: (m,n)=(%d,%d) does not fit shared memory", m, n);
            smem = cta + per_warp * wpc;
            // unit = window of G on the weight axis (k_shared.cuh: subtree_weight); G depends on the range
            // only — never on the device or the shard count — so all shards agree on the windows
            auto C = [](int top, int k) -> uint64_t { return binom_mk(top, k); };
            int32_t Slo[kMaxM], Shi[kMaxM];
            enumgpu_unrank(n, m, lo, Slo);
            sp.plan.w_lo = weight_of_child(C, n, m, Slo);
            if (hi < rs.total) { enumgpu_unrank(n, m, hi, Shi); sp.plan.w_hi = weight_of_child(C, n, m, Shi); }
            else {
                sp.plan.w_hi = 0;
                for (int v = 0; v <= n - m; ++v) sp.plan.w_hi += subtree_weight(C, n, m, 0, v);   // end of the weight axis
            }
            const uint64_t span = sp.plan.w_hi - sp.plan.w_lo;
            // Unit size.  Two costs pull against each other: every unit start is ~11 us of a warp's time (descent on
            // the weight axis, the depth-(q-1) tableau rebuilt from A, three level steps), and the launch ends when the
            // slowest warp finishes its last unit (a quarter of a unit's duration with the last round cut in four).
            // With W = the work per warp (weight x 17.5 ns, spread over 16 warps x 148 SMs x shards) the sum
            // T x 11 us + W / 4T is smallest at T = sqrt(W / 44 us) units per warp; measured optima sit a little above
            // that unit size (sweeps in profiles/r2_unit_sweep.txt: m=12,n=40 48.2 ms at 65536 vs 49.0 at 2^-18 of the
            // range; m=10,n=30 0.38-0.40 ms at 8192-16384 vs 0.575 at the old floor of 1024), hence the 80.
            // G depends on the range and the shard count only, so all shards of a run agree on the windows.
            const double warps_total = 16.0 * 148.0 * (double)shard_count;
            const double work_us = (double)span * 0.0175 / warps_total;
            double unit_k = 80.0;
#ifdef ENUMGPU_DEV_BUILD
            if (const char* e = getenv("ENUMGPU_UNIT_K")) unit_k = atof(e);
#endif
            double units_per_warp = sqrt(work_us / unit_k);
            if (units_per_warp < 1.0) units_per_warp = 1.0;
            uint64_t G = (uint64_t)((double)span / (warps_total * units_per_warp));
            uint64_t g_min = 1024;
#ifdef ENUMGPU_DEV_BUILD            // kernel experiments only: unit size from the environment
            if (const char* e = getenv("ENUMGPU_UNIT_SHIFT")) G = span >> atoi(e);
            if (const char* e = getenv("ENUMGPU_UNIT_MIN")) g_min = (uint64_t)atoll(e);
#endif
            uint64_t g_max = 131072;
#ifdef ENUMGPU_DEV_BUILD
            if (const char* e = getenv("ENUMGPU_UNIT_CAP")) g_max = (uint64_t)atoll(e);
#endif
            if (G < g_min) G = g_min;
            if (G > g_max) G = g_max;
            G -= G % kFineSplit;
            sp.plan.unit_weight = G;
            const uint64_t nu_all = (span + G - 1) / G;
            const uint64_t nu = nu_all > shard_index ? (nu_all - shard_index + shard_count - 1) / shard_count : 0;
            sp.warps_per_cta = wpc;
            k2_blocks = (uint64_t)sms;
            if (k2_blocks * wpc > nu) k2_blocks = (nu + wpc - 1) / wpc;
            // the last round of units (one per warp) is dealt in kFineSplit pieces each (k_shared.cuh: handout_window).
            // measured at m=12, n=40 (1/8 shard; full range): none 7.15; 54.92 ms, 1 round x 4 pieces 7.06; 54.79,
            // 1 x 2 7.08, 1 x 8 7.14, 2 x 4 7.14, 4 x 4 7.30 — pieces are dear (a child cut by a boundary is built twice)
            if (!plan_handouts(nu_all, shard_index, shard_count, k2_blocks * (uint64_t)wpc, &sp.plan))
                return fail(ENUMGPU_ERR_RANGE, "rank range too large for one launch");
            if (k2_blocks) {
                int rc_t = device_items(dev, n - P, &d_tri, &d_quad, &sp.n_tri, &sp.n_quad);
                if (rc_t == 0) rc_t = device_wprefix(dev, n, m, &sp.wprefix);
                if (rc_t) return rc_t;
            }
        }
    } else {
        all_blocks = shard_blocks(indep_geom(begin, end, &chunk_all));
    }
    const uint64_t total_blocks = head_blocks + tail_blocks + k2_blocks + all_blocks;
    if (total_blocks > 0x7fffffffull) return fail(ENUMGPU_ERR_RANGE, "rank range too large for one launch");

    if (total_blocks == 0) {   // empty range: the neutral record
        k_empty_record<<<1, 32, 0, st>>>(prm.m, algo, partial_dev);
        CU(cudaGetLastError());
        if (n_launches) *n_launches = launches + 1;
        return 0;
    }

    // ---- scratch: control block + per-block partials ----
    StreamBuf b_parts, b_ctrl, b_queue;
    const size_t queue_bytes = (size_t)k2_blocks * (size_t)wpc * queue_warp_bytes(pd->n);   // the stacks need no initialisation
    if (scratch) {
        int rc_s = scratch_reserve(scratch, (size_t)total_blocks, st);
        if (rc_s == 0 && queue_bytes) rc_s = scratch_reserve_queue(scratch, queue_bytes, st);
        if (rc_s) return rc_s;
        prm.ctrl = scratch->ctrl;
        prm.all_parts = scratch->parts;
        sp.queue = scratch->queue;
    } else {
        if (queue_bytes) CU(b_queue.alloc(queue_bytes, st));
        sp.queue = b_queue.as<unsigned char>();
        CU(b_parts.alloc(sizeof(BlockPartial) * total_blocks, st));
        CU(b_ctrl.alloc(sizeof(Ctrl), st));
        CU(cudaMemsetAsync(b_ctrl.p, 0, sizeof(Ctrl), st));
        prm.ctrl = b_ctrl.as<Ctrl>();
        prm.all_parts = b_parts.as<BlockPartial>();
    }
    prm.total_blocks = (uint32_t)total_blocks;
    prm.record = partial_dev;

    uint32_t slot = 0;
    if (k2_blocks) {
        sp.base = prm;
        sp.tri = d_tri; sp.quad = d_quad;
        CU(dispatch_shared(sp, prm.all_parts + slot, (int)k2_blocks, 32 * wpc, smem, st));
        ++launches;
        slot += (uint32_t)k2_blocks;
    }
    if (head_blocks) {
        LaunchParams hp = prm; hp.rank_begin = begin; hp.rank_end = lo; hp.chunk = chunk_head;
        CU(dispatch_independent(hp, prm.all_parts + slot, (uint32_t)head_blocks, st));
        ++launches; slot += (uint32_t)head_blocks;
    }
    if (tail_blocks) {
        LaunchParams tp = prm; tp.rank_begin = hi; tp.rank_end = end; tp.chunk = chunk_tail;
        CU(dispatch_independent(tp, prm.all_parts + slot, (uint32_t)tail_blocks, st));
        ++launches; slot += (uint32_t)tail_blocks;
    }
    if (all_blocks) {
        prm.chunk = chunk_all;
        prm.shard_index = shard_index; prm.shard_count = shard_count;
        CU(dispatch_independent(prm, prm.all_parts + slot, (uint32_t)all_blocks, st));
        ++launches; slot += (uint32_t)all_blocks;
    }
    if (n_launches) *n_launches = launches;
    return 0;
}

extern "C" int enumgpu_enqueue_device(const enumgpu_problem* p_dev, double scale_A, const enumgpu_options* o,
                                      enumgpu_partial* partial_dev, int32_t* n_launches)
{
    g_err[0] = 0;
    Resolved rs;
    int rc = resolve(p_dev, o, &rs, false);
    if (rc) return rc;
    if (!partial_dev) return fail(ENUMGPU_ERR_ARG, "partial_dev is NULL");
    if (enumgpu_device_count() < 1) return fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");
    cudaStream_t st = o ? (cudaStream_t)o->stream : nullptr;
    return enqueue_range(p_dev, scale_A, rs, rs.begin, rs.end, rs.shard_index, rs.shard_count, st, partial_dev, n_launches);
}

extern "C" void enumgpu_partial_to_result(const enumgpu_partial* ph, enumgpu_result* out)
{
    memset(out, 0, sizeof *out);
    out->m = ph->m;
    out->key = ph->key;
    out->best_rank = ph->best_rank;
    out->n_bases = ph->n_bases;
    out->n_singular = ph->n_singular;
    out->n_infeasible = ph->n_infeasible;
    out->n_feasible = ph->n_feasible;
    out->objective = ph->objective;
    out->algo_used = ph->algo_used;
    for (int i = 0; i < kMaxM; ++i) { out->basis[i] = ph->basis[i]; out->x_B[i] = ph->x_B[i]; }
    out->status = (ph->best_rank == UINT64_MAX) ? ENUMGPU_NO_FEASIBLE : ENUMGPU_OK;
}

extern "C" void enumgpu_merge_partial(enumgpu_partial* acc, const enumgpu_partial* part)
{
    const bool take = (part->key < acc->key) || (part->key == acc->key && part->best_rank < acc->best_rank);
    const uint64_t nb = acc->n_bases + part->n_bases, ns = acc->n_singular + part->n_singular,
                   ni = acc->n_infeasible + part->n_infeasible, nf = acc->n_feasible + part->n_feasible;
    if (take) *acc = *part;
    acc->n_bases = nb; acc->n_singular = ns; acc->n_infeasible = ni; acc->n_feasible = nf;
}

extern "C" int enumgpu_eval_basis(const enumgpu_problem* p, const enumgpu_options* o, const int32_t* basis,
                                  double* x_B, double* objective, int32_t* basis_class)
{
    g_err[0] = 0;
    // Stands in for Canonical::GetBasicSolution / IsFeasibleBasis (Canonical.cpp:165-197), which work for a
    // Canonical of any size and any index list its constructor accepted: no ENUMGPU_MAX_M / MAX_N limit here,
    // repeated indices are allowed (the basis is then singular).
    if (!p || !p->A_colmajor || !p->b || !p->c) return fail(ENUMGPU_ERR_ARG, "eval_basis: problem, A, b or c is NULL");
    if (!basis || !x_B || !objective || !basis_class) return fail(ENUMGPU_ERR_ARG, "eval_basis: NULL argument");
    const int m = p->m, n = p->n;
    if (m < 1 || n < 1 || p->lda < m) return fail(ENUMGPU_ERR_ARG, "eval_basis: bad dimensions m=%d n=%d lda=%d", m, n, p->lda);
    const int rule = o ? o->pivot_rule : ENUMGPU_PIVOT_ABSOLUTE;
    if (rule != ENUMGPU_PIVOT_ABSOLUTE && rule != ENUMGPU_PIVOT_RELATIVE) return fail(ENUMGPU_ERR_ARG, "unknown pivot_rule %d", rule);
    const double eps_feas = (o && o->eps_feas >= 0) ? o->eps_feas : 1e-9;
    const double eps_piv = (o && o->eps_piv >= 0) ? o->eps_piv : (rule == ENUMGPU_PIVOT_RELATIVE ? (double)m * 0x1p-52 : 1e-9);
    for (int i = 0; i < m; ++i)
        if (basis[i] < 0 || basis[i] >= n) return fail(ENUMGPU_ERR_ARG, "basis index %d out of range", basis[i]);
    double scale = 0.0;
    for (int j = 0; j < n; ++j) {
        if (!std::isfinite(p->c[j])) return fail(ENUMGPU_ERR_NONFINITE, "c[%d] is not finite", j);
        for (int i = 0; i < m; ++i) {
            const double v = p->A_colmajor[i + (size_t)j * p->lda];
            if (!std::isfinite(v)) return fail(ENUMGPU_ERR_NONFINITE, "A(%d,%d) is not finite", i, j);
            scale = fmax(scale, fabs(v));
        }
    }
    for (int i = 0; i < m; ++i)
        if (!std::isfinite(p->b[i])) return fail(ENUMGPU_ERR_NONFINITE, "b[%d] is not finite", i);
    if (enumgpu_device_count() < 1) return fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");
    // gather (Canonical.cpp:183-187): W = [A(:, basis) | b] column-major, then c_B, then room for 1/pivot
    const size_t w_elems = (size_t)m * (m + 1);
    std::vector<double> stage(w_elems + 2 * (size_t)m);
    for (int j = 0; j < m; ++j) memcpy(&stage[(size_t)j * m], p->A_colmajor + (size_t)basis[j] * p->lda, sizeof(double) * m);
    memcpy(&stage[(size_t)m * m], p->b, sizeof(double) * m);
    for (int j = 0; j < m; ++j) stage[w_elems + j] = p->c[basis[j]];
    int dev = 0;
    cudaGetDevice(&dev);
    keep_pool_memory(dev);
    cudaStream_t st = nullptr;
    CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    std::vector<double> h_out((size_t)m + 2, 0.0);
    auto body = [&]() -> int {
        StreamBuf b_in, b_out;
        CU(b_in.alloc(stage.size() * sizeof(double), st));
        CU(b_out.alloc(h_out.size() * sizeof(double), st));
        double* d_in = b_in.as<double>();
        CU(cudaMemcpyAsync(d_in, stage.data(), stage.size() * sizeof(double), cudaMemcpyHostToDevice, st));
        CU(cudaMemsetAsync(b_out.p, 0, h_out.size() * sizeof(double), st));
        k_eval_any<<<1, 256, 0, st>>>(d_in, d_in + w_elems, m, rule == ENUMGPU_PIVOT_RELATIVE ? 0.0 : eps_piv * scale, eps_feas,
                                      rule, eps_piv, d_in + w_elems + m, b_out.as<double>());
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(h_out.data(), b_out.p, h_out.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        return 0;
    };
    const int rc = body();
    cudaStreamDestroy(st);
    if (rc) return rc;
    for (int i = 0; i < m; ++i) x_B[i] = h_out[i];
    *objective = h_out[m];
    *basis_class = (int32_t)h_out[m + 1];
    return ENUMGPU_OK;
}

// many bases by rank, one thread each
__global__ void k_eval_ranks(const LaunchParams prm, const uint64_t* __restrict__ ranks, uint64_t count,
                             double* __restrict__ xB, double* __restrict__ obj, int32_t* __restrict__ cls)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    int S[kMaxM];
    unrank_lex(prm.binom, prm.n, prm.m, ranks[i], S);
    double x[kMaxM], z = 0.0;
    for (int j = 0; j < kMaxM; ++j) x[j] = 0.0;
    cls[i] = eval_basis_generic(prm.A, prm.lda, prm.b, prm.c, prm.m, S, prm.thr, prm.eps_feas, x, &z, prm.pivot_rule, prm.rel_eps);
    for (int j = 0; j < prm.m; ++j) xB[i * prm.m + j] = x[j];
    obj[i] = z;
}

// host copy of the problem on the current device: A (packed, lda = m) | b | c, and max|A_ij|
struct DeviceProblem {
    StreamBuf buf;
    enumgpu_problem dp;
    double scale = 0.0;
};
static int upload_problem(const enumgpu_problem* p, cudaStream_t st, DeviceProblem* out)
{
    const int m = p->m, n = p->n;
    std::vector<double> stage((size_t)m * n + m + n);
    for (int j = 0; j < n; ++j)
        for (int i = 0; i < m; ++i) {
            const double v = p->A_colmajor[i + (size_t)j * p->lda];
            stage[(size_t)j * m + i] = v;
            out->scale = fmax(out->scale, fabs(v));
        }
    memcpy(&stage[(size_t)m * n], p->b, sizeof(double) * m);
    memcpy(&stage[(size_t)m * n + m], p->c, sizeof(double) * n);
    CU(out->buf.alloc(stage.size() * sizeof(double), st));
    CU(cudaMemcpyAsync(out->buf.p, stage.data(), stage.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    out->dp = *p;
    out->dp.lda = m;
    out->dp.A_colmajor = out->buf.as<double>();
    out->dp.b = out->buf.as<double>() + (size_t)m * n;
    out->dp.c = out->dp.b + m;
    return 0;
}

// enumgpu_list_window into `ranks` (capacity entries), or, with `fit`, into *fit resized to the number listed (the
// library's own callers, which ask for a large capacity and usually receive a few entries).
static int list_window(const enumgpu_problem* p, const enumgpu_options* o, double key_max, uint64_t* ranks, uint64_t capacity,
                       std::vector<uint64_t>* fit, uint64_t* n_listed, enumgpu_result* out, uint64_t* n_window = nullptr)
{
    g_err[0] = 0;
    if (!out || !n_listed) return fail(ENUMGPU_ERR_ARG, "list_window: NULL argument");
    memset(out, 0, sizeof *out);
    *n_listed = 0;
    if (capacity && !ranks && !fit) return out->status = fail(ENUMGPU_ERR_ARG, "list_window: ranks is NULL but capacity is %llu", (unsigned long long)capacity);
    Resolved rs;
    int rc = resolve(p, o, &rs, true);
    if (rc) return out->status = rc;
    if (enumgpu_device_count() < 1) return out->status = fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");
    int dev = 0;
    cudaGetDevice(&dev);
    keep_pool_memory(dev);
    cudaStream_t st = nullptr;
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess)
        return out->status = fail(ENUMGPU_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(cudaGetLastError()));
    enumgpu_partial h_part;
    unsigned long long h_count = 0;
    int32_t launches = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto body = [&]() -> int {
        DeviceProblem D;
        int r2 = upload_problem(p, st, &D);
        if (r2) return r2;
        StreamBuf b_part, b_count, b_ranks;
        CU(b_part.alloc(sizeof(enumgpu_partial), st));
        CU(b_count.alloc(sizeof(unsigned long long), st));
        CU(b_ranks.alloc(sizeof(uint64_t) * (capacity ? capacity : 1), st));
        CU(cudaMemsetAsync(b_count.p, 0, sizeof(unsigned long long), st));
        CU(cudaEventCreate(&e0));
        CU(cudaEventCreate(&e1));
        CU(cudaEventRecord(e0, st));
        r2 = enqueue_range(&D.dp, D.scale, rs, rs.begin, rs.end, rs.shard_index, rs.shard_count, st, b_part.as<enumgpu_partial>(),
                           &launches, nullptr, b_count.as<unsigned long long>(), b_ranks.as<uint64_t>(), capacity, key_max);
        if (r2) return r2;
        CU(cudaEventRecord(e1, st));
        CU(cudaMemcpyAsync(&h_part, b_part.p, sizeof h_part, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(&h_count, b_count.p, sizeof h_count, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        const uint64_t k = h_count < capacity ? (uint64_t)h_count : capacity;
        if (fit) { fit->resize(k); ranks = fit->data(); }
        if (n_window) *n_window = h_count;
        if (k) CU(cudaMemcpy(ranks, b_ranks.p, sizeof(uint64_t) * k, cudaMemcpyDeviceToHost));
        *n_listed = k;
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        enumgpu_partial_to_result(&h_part, out);
        out->kernel_ms = ms;
        out->n_launches = launches;
        return 0;
    };
    rc = body();
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaStreamDestroy(st);
    if (rc) return out->status = rc;
    std::sort(ranks, ranks + *n_listed);     // the device appends in arrival order; hand them out ascending
    return out->status;
}

extern "C" int enumgpu_list_window(const enumgpu_problem* p, const enumgpu_options* o, double key_max, uint64_t* ranks,
                                   uint64_t capacity, uint64_t* n_listed, enumgpu_result* out)
{
    return list_window(p, o, key_max, ranks, capacity, nullptr, n_listed, out);
}

extern "C" int enumgpu_list_feasible(const enumgpu_problem* p, const enumgpu_options* o, uint64_t* ranks, uint64_t capacity,
                                     uint64_t* n_listed, enumgpu_result* out)
{
    return list_window(p, o, INFINITY, ranks, capacity, nullptr, n_listed, out);
}

extern "C" int enumgpu_eval_ranks(const enumgpu_problem* p, const enumgpu_options* o, const uint64_t* ranks, uint64_t count,
                                  double* x_B, double* objective, int32_t* basis_class)
{
    g_err[0] = 0;
    Resolved rs;
    int rc = resolve(p, o, &rs, true);
    if (rc) return rc;
    if (count == 0) return ENUMGPU_OK;
    if (!ranks || !x_B || !objective || !basis_class) return fail(ENUMGPU_ERR_ARG, "eval_ranks: NULL argument");
    for (uint64_t i = 0; i < count; ++i)
        if (ranks[i] >= rs.total) return fail(ENUMGPU_ERR_RANGE, "eval_ranks: rank %llu out of range", (unsigned long long)ranks[i]);
    if (count > (1ull << 31)) return fail(ENUMGPU_ERR_RANGE, "eval_ranks: too many bases in one call");
    if (enumgpu_device_count() < 1) return fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");
    int dev = 0;
    cudaGetDevice(&dev);
    keep_pool_memory(dev);
    cudaStream_t st = nullptr;
    CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    auto body = [&]() -> int {
        DeviceProblem D;
        int r2 = upload_problem(p, st, &D);
        if (r2) return r2;
        const int m = p->m;
        StreamBuf b_ranks, b_x, b_z, b_cls;
        const uint64_t* d_binom = nullptr;
        r2 = device_binom(dev, &d_binom);
        if (r2) return r2;
        CU(b_ranks.alloc(sizeof(uint64_t) * count, st));
        CU(b_x.alloc(sizeof(double) * count * m, st));
        CU(b_z.alloc(sizeof(double) * count, st));
        CU(b_cls.alloc(sizeof(int32_t) * count, st));
        CU(cudaMemcpyAsync(b_ranks.p, ranks, sizeof(uint64_t) * count, cudaMemcpyHostToDevice, st));
        LaunchParams prm{};
        prm.A = D.dp.A_colmajor; prm.b = D.dp.b; prm.c = D.dp.c; prm.binom = d_binom;
        prm.m = m; prm.n = p->n; prm.lda = m; prm.maximize = p->maximize ? 1 : 0;
        prm.eps_feas = rs.eps_feas;
        prm.pivot_rule = rs.rule;
        prm.thr = rs.rule == ENUMGPU_PIVOT_RELATIVE ? 0.0 : rs.eps_piv * D.scale;
        prm.rel_eps = rs.rule == ENUMGPU_PIVOT_RELATIVE ? rs.eps_piv : 0.0;
        const unsigned blocks = (unsigned)((count + 127) / 128);
        k_eval_ranks<<<blocks, 128, 0, st>>>(prm, b_ranks.as<uint64_t>(), count, b_x.as<double>(), b_z.as<double>(), b_cls.as<int32_t>());
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(x_B, b_x.p, sizeof(double) * count * m, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(objective, b_z.p, sizeof(double) * count, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(basis_class, b_cls.p, sizeof(int32_t) * count, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        return 0;
    };
    rc = body();
    cudaStreamDestroy(st);
    return rc;
}

// ------------------------------------------------------------------ self-test of the branch-free reciprocal
// operand i of the test: i < kRcpEdge are structured (every power of two 2^e, e in [-1000, 1000], and its two
// neighbours, both signs); the rest are random: sign, exponent uniform in [-1000, 1000], 52 random mantissa bits
constexpr uint64_t kRcpEdge = 2001ull * 3ull * 2ull;
__device__ __forceinline__ double rcp_test_operand(uint64_t i, uint64_t seed)
{
    if (i < kRcpEdge) {
        const int e = (int)(i / 6) - 1000, v = (int)(i % 6);
        uint64_t bits = (uint64_t)(1023 + e) << 52;
        bits += (uint64_t)(int64_t)((v % 3) - 1);            // 2^e - 1 ulp, 2^e, 2^e + 1 ulp
        if (v >= 3) bits |= 1ull << 63;
        return __longlong_as_double((long long)bits);
    }
    uint64_t z = seed + (i + 1) * 0x9E3779B97F4A7C15ull;     // SplitMix64 of the index
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    const uint64_t mant = z & ((1ull << 52) - 1), sign = (z >> 63) << 63;
    const uint64_t e = 23 + ((z >> 52) & 0x7ff) % 2001;      // biased exponent 23 .. 2023  <->  2^-1000 .. 2^1000
    return __longlong_as_double((long long)(sign | (e << 52) | mant));
}
__global__ void __launch_bounds__(256)
k_rcp_selftest(uint64_t n, uint64_t seed, unsigned long long* n_bad, unsigned long long* first_bad_bits)
{
    unsigned long long bad = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const double x = rcp_test_operand(i, seed);
        // 2^1000 + 1 ulp and beyond the range the host guard admits are part of the structured set on purpose only
        // up to |x| = 2^1000 exactly; skip the two operands above it
        if (fabs(x) > 0x1p1000 || fabs(x) < 0x1p-1000) continue;
        const double a = rcp_nobranch(x), b = __drcp_rn(x);
        if (__double_as_longlong(a) != __double_as_longlong(b)) {
            if (bad == 0) atomicCAS(first_bad_bits, 0ull, (unsigned long long)__double_as_longlong(x));
            ++bad;
        }
    }
    if (bad) atomicAdd(n_bad, bad);
}

static int rcp_selftest_device(uint64_t n_operands, uint64_t seed, uint64_t* n_mismatch, double* first_bad, cudaStream_t st)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    unsigned long long* d = nullptr;
    CU(cudaMalloc(&d, 16));
    auto body = [&]() -> int {
        CU(cudaMemsetAsync(d, 0, 16, st));
        k_rcp_selftest<<<sms * 8, 256, 0, st>>>(n_operands, seed, d, d + 1);
        CU(cudaGetLastError());
        unsigned long long h[2] = {0, 0};
        CU(cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        *n_mismatch = h[0];
        if (first_bad) memcpy(first_bad, &h[1], 8);
        return 0;
    };
    const int rc = body();
    cudaFree(d);
    return rc;
}

extern "C" int enumgpu_selftest_rcp(uint64_t n_operands, uint64_t seed, uint64_t* n_mismatch, double* first_bad)
{
    g_err[0] = 0;
    if (!n_mismatch) return fail(ENUMGPU_ERR_ARG, "selftest_rcp: n_mismatch is NULL");
    if (enumgpu_device_count() < 1) return fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");
    return rcp_selftest_device(n_operands, seed, n_mismatch, first_bad, nullptr);
}

static bool shared_rcp_trusted(int dev)
{
    std::lock_guard<std::mutex> lock(g_tables_mu);
    DeviceTables& t = g_tables[dev];
    if (t.rcp_state == 0) {
        uint64_t bad = 1;
        double first = 0.0;
        const int rc = rcp_selftest_device(1ull << 22, 0x5EEDull, &bad, &first, nullptr);
        t.rcp_state = (rc == 0 && bad == 0) ? 1 : 2;
        if (t.rcp_state == 2)
            fail(ENUMGPU_OK, "warning: the shared kernel's reciprocal differs from __drcp_rn on device %d (%llu of 2^22 operands, "
                             "first %a): using the independent kernel", dev, (unsigned long long)bad, first);
    }
    return t.rcp_state == 1;
}

// ------------------------------------------------------------------ handles
// Everything a solve needs that outlives the call: a stream, two events, pinned staging for the inputs and the
// 256-byte record, the device copy of the inputs and the enqueue scratch.  With a handle a solve is: pack into
// pinned memory, one H2D copy, one kernel, one D2H copy, one synchronisation — nothing is created, allocated,
// cleared or destroyed per call.
struct enumgpu_handle {
    int dev = 0;
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    double* h_in = nullptr;              // pinned, kStageDoubles
    enumgpu_partial* h_part = nullptr;   // pinned
    double* d_in = nullptr;              // device, kStageDoubles
    enumgpu_partial* d_part = nullptr;
    Scratch scratch;
};
constexpr size_t kStageDoubles = (size_t)kMaxM * kMaxN + kMaxM + kMaxN;

extern "C" void enumgpu_destroy(enumgpu_handle* h)
{
    if (!h) return;
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(h->dev);
    if (h->st) cudaStreamSynchronize(h->st);
    if (h->scratch.parts) cudaFree(h->scratch.parts);
    if (h->scratch.queue) cudaFree(h->scratch.queue);
    if (h->scratch.ctrl) cudaFree(h->scratch.ctrl);
    if (h->d_part) cudaFree(h->d_part);
    if (h->d_in) cudaFree(h->d_in);
    if (h->h_part) cudaFreeHost(h->h_part);
    if (h->h_in) cudaFreeHost(h->h_in);
    if (h->e0) cudaEventDestroy(h->e0);
    if (h->e1) cudaEventDestroy(h->e1);
    if (h->st) cudaStreamDestroy(h->st);
    cudaGetLastError();
    cudaSetDevice(cur);
    delete h;
}

extern "C" int enumgpu_create(int32_t device, enumgpu_handle** out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "create: out is NULL");
    *out = nullptr;
    const int have = enumgpu_device_count();
    if (have < 1) return fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");
    int cur = 0;
    cudaGetDevice(&cur);
    if (device < 0) device = cur;
    if (device >= have) return fail(ENUMGPU_ERR_ARG, "device ordinal %d not present (%d devices)", device, have);
    enumgpu_handle* h = new enumgpu_handle;
    h->dev = device;
    auto body = [&]() -> int {
        CU(cudaSetDevice(device));
        keep_pool_memory(device);
        CU(cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking));
        CU(cudaEventCreate(&h->e0));
        CU(cudaEventCreate(&h->e1));
        CU(cudaMallocHost(&h->h_in, kStageDoubles * sizeof(double)));
        CU(cudaMallocHost(&h->h_part, sizeof(enumgpu_partial)));
        CU(cudaMalloc(&h->d_in, kStageDoubles * sizeof(double)));
        CU(cudaMalloc(&h->d_part, sizeof(enumgpu_partial)));
        CU(cudaMalloc(&h->scratch.ctrl, sizeof(Ctrl)));
        CU(cudaMemset(h->scratch.ctrl, 0, sizeof(Ctrl)));
        {   // stream-ordered allocations (they are regrown with cudaMallocAsync / cudaFreeAsync on demand)
            const int rc_s = scratch_reserve(&h->scratch, 1024, h->st);
            if (rc_s) return rc_s;
            int sms = 148;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
            const int rc_q = scratch_reserve_queue(&h->scratch, (size_t)sms * kMaxWarps * queue_warp_bytes(40), h->st);   // grown on demand for n > 40
            if (rc_q) return rc_q;
            CU(cudaStreamSynchronize(h->st));
        }
        const uint64_t* binom = nullptr;                 // constant tables and the reciprocal self-check: now, not in the first solve
        const int rc_t = device_binom(device, &binom);
        if (rc_t) return rc_t;
        shared_rcp_trusted(device);
        return 0;
    };
    const int rc = body();
    cudaSetDevice(cur);
    if (rc) { enumgpu_destroy(h); return rc; }
    *out = h;
    return ENUMGPU_OK;
}

// a failed enqueue may leave the control block half-used: clear it (and whatever is in flight) before the next call
static void handle_recover(enumgpu_handle* h)
{
    cudaStreamSynchronize(h->st);
    cudaGetLastError();
    cudaMemset(h->scratch.ctrl, 0, sizeof(Ctrl));
}

// Host-buffer solve on n_handles devices at once (one handle per device): device i takes the interleaved rank
// windows i, i + n, ... of the caller's shard; everything is enqueued on every device before the first
// synchronisation; the records merge on the host (associative, commutative).
extern "C" int enumgpu_solve_hv(enumgpu_handle* const* hs, int32_t n_handles, const enumgpu_problem* p, const enumgpu_options* o,
                                enumgpu_result* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "out is NULL");
    memset(out, 0, sizeof *out);
    if (!hs || n_handles < 1 || n_handles > ENUMGPU_MAX_DEVICES) return out->status = fail(ENUMGPU_ERR_ARG, "bad handle list");
    for (int i = 0; i < n_handles; ++i)
        if (!hs[i]) return out->status = fail(ENUMGPU_ERR_ARG, "handle %d is NULL", i);
    Resolved rs;
    int rc = resolve(p, o, &rs, true);
    if (rc) return out->status = rc;
    const int m = p->m, n = p->n;
    // pack A (lda -> m), b, c into the pinned staging buffer of handle 0; max|A_ij| in the same pass
    enumgpu_handle* h0 = hs[0];
    double scale = 0.0;
    for (int j = 0; j < n; ++j)
        for (int i = 0; i < m; ++i) {
            const double v = p->A_colmajor[i + (size_t)j * p->lda];
            h0->h_in[(size_t)j * m + i] = v;
            scale = fmax(scale, fabs(v));
        }
    memcpy(h0->h_in + (size_t)m * n, p->b, sizeof(double) * m);
    memcpy(h0->h_in + (size_t)m * n + m, p->c, sizeof(double) * n);
    const size_t bytes = ((size_t)m * n + m + n) * sizeof(double);
    int cur = 0;
    cudaGetDevice(&cur);
    int32_t launches[ENUMGPU_MAX_DEVICES] = {0};
    auto body = [&]() -> int {
        for (int i = 0; i < n_handles; ++i) {
            enumgpu_handle* h = hs[i];
            const uint32_t sh_index = rs.shard_index + rs.shard_count * (uint32_t)i, sh_count = rs.shard_count * (uint32_t)n_handles;
            CU(cudaSetDevice(h->dev));
            CU(cudaMemcpyAsync(h->d_in, h0->h_in, bytes, cudaMemcpyHostToDevice, h->st));
            enumgpu_problem dp = *p;
            dp.lda = m;
            dp.A_colmajor = h->d_in;
            dp.b = h->d_in + (size_t)m * n;
            dp.c = dp.b + m;
            CU(cudaEventRecord(h->e0, h->st));
            const int r2 = enqueue_range(&dp, scale, rs, rs.begin, rs.end, sh_index, sh_count, h->st, h->d_part, &launches[i], &h->scratch);
            if (r2) return r2;
            CU(cudaEventRecord(h->e1, h->st));
            CU(cudaMemcpyAsync(h->h_part, h->d_part, sizeof(enumgpu_partial), cudaMemcpyDeviceToHost, h->st));
        }
        double ms_max = 0.0;
        int n_launches = 0;
        enumgpu_partial acc;
        for (int i = 0; i < n_handles; ++i) {
            enumgpu_handle* h = hs[i];
            CU(cudaSetDevice(h->dev));
            CU(cudaStreamSynchronize(h->st));
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, h->e0, h->e1));
            ms_max = fmax(ms_max, (double)ms);
            n_launches += launches[i];
            if (i == 0) acc = *h->h_part;
            else enumgpu_merge_partial(&acc, h->h_part);
        }
        enumgpu_partial_to_result(&acc, out);
        out->kernel_ms = ms_max;
        out->n_launches = n_launches;
        return 0;
    };
    rc = body();
    if (rc) for (int i = 0; i < n_handles; ++i) { cudaSetDevice(hs[i]->dev); handle_recover(hs[i]); }
    cudaSetDevice(cur);
    if (rc) { out->status = rc; return rc; }
    return out->status;
}

extern "C" int enumgpu_solve_h(enumgpu_handle* h, const enumgpu_problem* p, const enumgpu_options* o, enumgpu_result* out)
{
    return enumgpu_solve_hv(&h, 1, p, o, out);
}

extern "C" int enumgpu_enqueue_h(enumgpu_handle* h, const enumgpu_problem* p_dev, double scale_A, const enumgpu_options* o,
                                 enumgpu_partial* partial_dev, int32_t* n_launches)
{
    g_err[0] = 0;
    if (!h) return fail(ENUMGPU_ERR_ARG, "handle is NULL");
    Resolved rs;
    int rc = resolve(p_dev, o, &rs, false);
    if (rc) return rc;
    if (!partial_dev) return fail(ENUMGPU_ERR_ARG, "partial_dev is NULL");
    int cur = 0;
    cudaGetDevice(&cur);
    if (cur != h->dev) return fail(ENUMGPU_ERR_ARG, "enqueue_h: the handle belongs to device %d, the current device is %d", h->dev, cur);
    cudaStream_t st = (o && o->stream) ? (cudaStream_t)o->stream : h->st;
    rc = enqueue_range(p_dev, scale_A, rs, rs.begin, rs.end, rs.shard_index, rs.shard_count, st, partial_dev, n_launches, &h->scratch);
    if (rc) { cudaStreamSynchronize(st); handle_recover(h); }
    return rc;
}

// enumgpu_enqueue_h for HOST inputs: pack A|b|c into the handle's pinned staging buffer, one H2D copy and the
// enumeration, all on one stream, no synchronisation.  The building block of a one-process-per-GPU solve
// (dist.ShardedEnumeration): the caller appends its collective and one D2H copy to the same stream.
extern "C" int enumgpu_enqueue_host_h(enumgpu_handle* h, const enumgpu_problem* p, const enumgpu_options* o,
                                      enumgpu_partial* partial_dev, int32_t* n_launches)
{
    g_err[0] = 0;
    if (!h) return fail(ENUMGPU_ERR_ARG, "handle is NULL");
    Resolved rs;
    int rc = resolve(p, o, &rs, true);
    if (rc) return rc;
    if (!partial_dev) return fail(ENUMGPU_ERR_ARG, "partial_dev is NULL");
    int cur = 0;
    cudaGetDevice(&cur);
    if (cur != h->dev) return fail(ENUMGPU_ERR_ARG, "enqueue_host_h: the handle belongs to device %d, the current device is %d", h->dev, cur);
    const int m = p->m, n = p->n;
    double scale = 0.0;
    for (int j = 0; j < n; ++j)
        for (int i = 0; i < m; ++i) {
            const double v = p->A_colmajor[i + (size_t)j * p->lda];
            h->h_in[(size_t)j * m + i] = v;
            scale = fmax(scale, fabs(v));
        }
    memcpy(h->h_in + (size_t)m * n, p->b, sizeof(double) * m);
    memcpy(h->h_in + (size_t)m * n + m, p->c, sizeof(double) * n);
    cudaStream_t st = (o && o->stream) ? (cudaStream_t)o->stream : h->st;
    auto body = [&]() -> int {
        CU(cudaMemcpyAsync(h->d_in, h->h_in, ((size_t)m * n + m + n) * sizeof(double), cudaMemcpyHostToDevice, st));
        enumgpu_problem dp = *p;
        dp.lda = m;
        dp.A_colmajor = h->d_in;
        dp.b = h->d_in + (size_t)m * n;
        dp.c = dp.b + m;
        return enqueue_range(&dp, scale, rs, rs.begin, rs.end, rs.shard_index, rs.shard_count, st, partial_dev, n_launches, &h->scratch);
    };
    rc = body();
    if (rc) { cudaStreamSynchronize(st); handle_recover(h); }
    return rc;
}

// merge n partial records (host memory, e.g. the result of an all-gather) into one result struct
extern "C" void enumgpu_merge_records(const enumgpu_partial* recs, int32_t n, enumgpu_result* out)
{
    enumgpu_partial acc = recs[0];
    for (int i = 1; i < n; ++i) enumgpu_merge_partial(&acc, &recs[i]);
    enumgpu_partial_to_result(&acc, out);
}

extern "C" void* enumgpu_handle_stream(enumgpu_handle* h) { return h ? (void*)h->st : nullptr; }

extern "C" int enumgpu_solve_device(const enumgpu_problem* p_dev, double scale_A, const enumgpu_options* o, enumgpu_result* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "out is NULL");
    memset(out, 0, sizeof *out);
    Resolved rs;
    int rc = resolve(p_dev, o, &rs, false);
    if (rc) return out->status = rc;
    if (enumgpu_device_count() < 1) return out->status = fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");

    cudaStream_t st = o ? (cudaStream_t)o->stream : nullptr;
    bool own_stream = false;
    if (!st) {
        if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess)
            return out->status = fail(ENUMGPU_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(cudaGetLastError()));
        own_stream = true;
    }
    enumgpu_partial h_part;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int32_t launches = 0;
    auto body = [&]() -> int {
        CU(cudaEventCreate(&e0));
        CU(cudaEventCreate(&e1));
        StreamBuf b_part;
        CU(b_part.alloc(sizeof(enumgpu_partial), st));
        enumgpu_partial* d_part = b_part.as<enumgpu_partial>();
        CU(cudaEventRecord(e0, st));
        int r2 = enqueue_range(p_dev, scale_A, rs, rs.begin, rs.end, rs.shard_index, rs.shard_count, st, d_part, &launches);
        if (r2) return r2;
        CU(cudaEventRecord(e1, st));
        CU(cudaMemcpyAsync(&h_part, d_part, sizeof h_part, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        enumgpu_partial_to_result(&h_part, out);
        out->kernel_ms = ms;
        out->n_launches = launches;
        return 0;
    };
    rc = body();
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (own_stream) cudaStreamDestroy(st);
    if (rc) { out->status = rc; return rc; }
    return out->status;
}

// Handle-free convenience form: temporary handles for the device list, one enumgpu_solve_hv, destroy.  Callers
// that solve repeatedly keep handles (EnumerationSolver does): creating one costs pinned and device allocations.
extern "C" int enumgpu_solve(const enumgpu_problem* p, const enumgpu_options* o, enumgpu_result* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "out is NULL");
    memset(out, 0, sizeof *out);
    Resolved rs;
    int rc = resolve(p, o, &rs, true);
    if (rc) return out->status = rc;
    const int have = enumgpu_device_count();
    if (have < 1) return out->status = fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");

    int nd = (o && o->n_devices > 0) ? o->n_devices : 1;
    if (nd > ENUMGPU_MAX_DEVICES) return out->status = fail(ENUMGPU_ERR_ARG, "n_devices=%d above %d", nd, ENUMGPU_MAX_DEVICES);
    int cur = 0;
    cudaGetDevice(&cur);
    enumgpu_handle* hs[ENUMGPU_MAX_DEVICES] = {nullptr};
    for (int i = 0; i < nd && rc == 0; ++i) {
        const int d = (o && o->n_devices > 0) ? (o->devices ? o->devices[i] : i) : cur;
        if (d < 0 || d >= have) rc = fail(ENUMGPU_ERR_ARG, "device ordinal %d not present (%d devices)", d, have);
        else rc = enumgpu_create(d, &hs[i]);
    }
    if (rc == 0) rc = enumgpu_solve_hv(hs, nd, p, o, out);
    char keep[sizeof g_err];
    memcpy(keep, g_err, sizeof keep);                      // destroying the handles must not lose the message
    for (int i = 0; i < nd; ++i) enumgpu_destroy(hs[i]);
    memcpy(g_err, keep, sizeof keep);
    if (rc < 0) out->status = rc;
    return rc < 0 ? rc : out->status;
}

// ------------------------------------------------------------------ certificate and rays (DESIGN.md §3)

static enumgpu_options whole_space_options(const enumgpu_options* o)
{
    enumgpu_options oc{};
    oc.eps_feas = oc.eps_piv = -1.0;
    if (o) oc = *o;
    oc.rank_begin = oc.rank_end = 0;
    oc.shard_index = oc.shard_count = 0;
    return oc;
}

// The auxiliary LP [A; s*ck'] d = (0, ..., 0, -1), cost 0, minimise: its feasible bases are the extreme rays of
// {d >= 0, A d = 0} with ck.d < 0.  s = 2^e, the largest power of two with s*max|ck_j| <= max|A_ij|, keeps
// max|A'_ij| = max|A_ij| and with it the pivot threshold.
extern "C" int enumgpu_find_ray(const enumgpu_problem* p, const enumgpu_options* o, enumgpu_result* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "out is NULL");
    memset(out, 0, sizeof *out);
    Resolved rs;
    const enumgpu_options oc = whole_space_options(o);   // the caller's rank range is one of the auxiliary space
    int rc = resolve(p, &oc, &rs, true);
    if (rc) return out->status = rc;
    const int m = p->m, n = p->n, ma = m + 1;
    if (ma > kMaxM) return out->status = fail(ENUMGPU_ERR_ARG, "find_ray: the auxiliary LP needs m+1 = %d rows, above %d", ma, kMaxM);
    double amax = 0.0, cmax = 0.0;
    for (int j = 0; j < n; ++j) {
        cmax = fmax(cmax, fabs(p->c[j]));
        for (int i = 0; i < m; ++i) amax = fmax(amax, fabs(p->A_colmajor[i + (size_t)j * p->lda]));
    }
    out->m = ma;
    if (n < ma || cmax == 0.0) {          // no basis of m+1 columns, or no direction can decrease ck.x
        out->key = INFINITY; out->best_rank = UINT64_MAX; out->objective = NAN;
        return out->status = ENUMGPU_NO_FEASIBLE;
    }
    if (amax == 0.0) return out->status = fail(ENUMGPU_ERR_RANGE, "find_ray: A = 0 leaves no scale for the cost row");
    int ea = 0, ec = 0;
    const double fa = frexp(amax, &ea), fc = frexp(cmax, &ec);
    const int e = ea - ec - (fc > fa ? 1 : 0);
    std::vector<double> Aa((size_t)ma * n), ba(ma, 0.0), ca(n, 0.0);
    for (int j = 0; j < n; ++j) {
        for (int i = 0; i < m; ++i) Aa[(size_t)j * ma + i] = p->A_colmajor[i + (size_t)j * p->lda];
        const double ck = p->maximize ? -p->c[j] : p->c[j];
        const double v = ldexp(ck, e);
        if (ldexp(v, -e) != ck) return out->status = fail(ENUMGPU_ERR_RANGE, "find_ray: c[%d] * 2^%d is not exact", j, e);
        Aa[(size_t)j * ma + m] = v;
    }
    ba[m] = -1.0;
    const enumgpu_problem aux{ma, n, ma, 0, Aa.data(), ba.data(), ca.data()};
    return enumgpu_solve(&aux, o, out);
}

// k_certify on a list of bases, kCertifyChunk blocks per launch at most: the device copy of the LP, the scratch
// slabs and the staging of the bases and certificates are sized by the chunk, not by the number of bases.
constexpr uint32_t kCertifyChunk = 4096;
struct Certifier {
    struct OwnedStream {               // declared first: destroyed after the buffers have queued their frees on it
        cudaStream_t s = nullptr;
        ~OwnedStream() { if (s) cudaStreamDestroy(s); }
    } owned;
    cudaStream_t st = nullptr;
    DeviceProblem D;
    StreamBuf b_scratch, b_S, b_out;
    double thr = 0.0;
    int32_t launches = 0;

    int init(const enumgpu_problem* p, const Resolved& rs)
    {
        int dev = 0;
        cudaGetDevice(&dev);
        keep_pool_memory(dev);
        CU(cudaStreamCreateWithFlags(&owned.s, cudaStreamNonBlocking));
        st = owned.s;
        const int rc = upload_problem(p, st, &D);
        if (rc) return rc;
        thr = rs.rule == ENUMGPU_PIVOT_RELATIVE ? 0.0 : rs.eps_piv * D.scale;
        CU(b_scratch.alloc(sizeof(double) * certify_slab(p->m, p->n) * kCertifyChunk, st));
        CU(b_S.alloc(sizeof(int32_t) * p->m * kCertifyChunk, st));
        CU(b_out.alloc(sizeof(enumgpu_certificate) * kCertifyChunk, st));
        return 0;
    }
    // count <= kCertifyChunk bases of m columns each (host); out[i] as the kernel leaves it, n_launches = 1
    int run(const enumgpu_problem* p, const Resolved& rs, const int32_t* bases, uint32_t count, double eps_opt,
            enumgpu_certificate* out)
    {
        const int m = p->m, n = p->n;
        CU(cudaMemcpyAsync(b_S.p, bases, sizeof(int32_t) * m * count, cudaMemcpyHostToDevice, st));
        CU(cudaMemsetAsync(b_out.p, 0, sizeof(enumgpu_certificate) * count, st));
        k_certify<<<count, kCertifyThreads, 0, st>>>(D.dp.A_colmajor, D.dp.b, D.dp.c, b_S.as<int>(), m, n, p->maximize ? 1 : 0,
                                                     thr, rs.eps_feas, rs.rule, rs.eps_piv, eps_opt, b_scratch.as<double>(),
                                                     b_out.as<enumgpu_certificate>());
        CU(cudaGetLastError());
        ++launches;
        CU(cudaMemcpyAsync(out, b_out.p, sizeof(enumgpu_certificate) * count, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        for (uint32_t i = 0; i < count; ++i) out[i].n_launches = 1;
        return 0;
    }
};

static double resolve_eps_opt(double eps_opt)
{
    if (!(eps_opt >= 0)) return 1e-9;                    // negative (or NaN): the default
    return eps_opt == 0.0 ? 0.0 : eps_opt;               // -0.0 means 0
}

static int check_bases(const enumgpu_problem* p, const int32_t* bases, uint64_t count, const char* who)
{
    if (!bases) return fail(ENUMGPU_ERR_ARG, "%s: basis is NULL", who);
    for (uint64_t i = 0; i < count * (uint64_t)p->m; ++i)
        if (bases[i] < 0 || bases[i] >= p->n) return fail(ENUMGPU_ERR_ARG, "%s: basis index %d out of range", who, bases[i]);
    return 0;
}

// The certificate of one basis without the ray fallback; ENUMGPU_ERR_ARG for a singular or infeasible basis.
static int certify_one(const enumgpu_problem* p, const Resolved& rs, const int32_t* basis, double eps_opt,
                       enumgpu_certificate* out)
{
    if (enumgpu_device_count() < 1) return out->status = fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");
    Certifier cf;
    int rc = cf.init(p, rs);
    if (rc == 0) rc = cf.run(p, rs, basis, 1, eps_opt, out);
    if (rc) { out->status = rc; return rc; }
    if (out->basis_class != ENUMGPU_BASIS_FEASIBLE)
        return out->status = fail(ENUMGPU_ERR_ARG, "certify: the basis is %s", out->basis_class == ENUMGPU_BASIS_SINGULAR ? "singular" : "infeasible");
    return ENUMGPU_OK;
}

// An undecided certificate (a degenerate vertex) decided by enumerating the extreme rays, where m+1 rows fit.
static int ray_fallback(const enumgpu_problem* p, const enumgpu_options* oc, enumgpu_certificate* out)
{
    if (out->status != ENUMGPU_CERT_UNDECIDED || p->m + 1 > kMaxM) return ENUMGPU_OK;
    enumgpu_result aux;
    const int rc = enumgpu_find_ray(p, oc, &aux);
    if (rc < 0) return out->status = rc;
    out->n_launches += aux.n_launches;
    out->n_aux_bases = aux.n_bases;
    out->n_rays = aux.n_feasible;
    if (rc == ENUMGPU_OK) {
        out->status = ENUMGPU_CERT_UNBOUNDED;
        for (int i = 0; i < aux.m; ++i) out->ray[aux.basis[i]] = aux.x_B[i];
    } else if (aux.n_feasible == 0) {
        out->status = ENUMGPU_CERT_BOUNDED;
    }                                     // feasible aux bases whose key is NaN (overflow): stays UNDECIDED
    return ENUMGPU_OK;
}

extern "C" int enumgpu_certify(const enumgpu_problem* p, const enumgpu_options* o, const int32_t* basis, double eps_opt,
                               enumgpu_certificate* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "certify: out is NULL");
    memset(out, 0, sizeof *out);
    out->entering = -1;
    const enumgpu_options oc = whole_space_options(o);
    Resolved rs;
    int rc = resolve(p, &oc, &rs, true);
    if (rc || (rc = check_bases(p, basis, 1, "certify"))) return out->status = rc;
    rc = certify_one(p, rs, basis, resolve_eps_opt(eps_opt), out);
    if (rc) return rc;
    return ray_fallback(p, &oc, out);
}

extern "C" int enumgpu_certify_bases(const enumgpu_problem* p, const enumgpu_options* o, const int32_t* bases, uint64_t count,
                                     double eps_opt, enumgpu_certificate* out)
{
    g_err[0] = 0;
    if (count && !out) return fail(ENUMGPU_ERR_ARG, "certify_bases: out is NULL");
    const enumgpu_options oc = whole_space_options(o);
    Resolved rs;
    int rc = resolve(p, &oc, &rs, true);
    if (rc || (rc = check_bases(p, bases, count, "certify_bases"))) return rc;
    if (count == 0) return ENUMGPU_OK;
    if (enumgpu_device_count() < 1) return fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)");
    eps_opt = resolve_eps_opt(eps_opt);
    Certifier cf;
    if ((rc = cf.init(p, rs))) return rc;
    for (uint64_t i = 0; i < count; i += kCertifyChunk) {
        const uint32_t k = (uint32_t)std::min<uint64_t>(kCertifyChunk, count - i);
        if ((rc = cf.run(p, rs, bases + i * p->m, k, eps_opt, out + i))) return rc;
        for (uint32_t j = 0; j < k; ++j)
            if (out[i + j].basis_class != ENUMGPU_BASIS_FEASIBLE) out[i + j].status = ENUMGPU_ERR_ARG;
    }
    return ENUMGPU_OK;
}

extern "C" int enumgpu_certify_optimum(const enumgpu_problem* p, const enumgpu_options* o, const enumgpu_result* opt,
                                       double eps_opt, uint64_t max_window, enumgpu_optimum* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "certify_optimum: out is NULL");
    memset(out, 0, sizeof *out);
    out->cert.entering = -1;
    out->window_index = UINT64_MAX;
    const enumgpu_options oc = whole_space_options(o);
    Resolved rs;
    int rc = resolve(p, &oc, &rs, true);
    if (rc) return out->cert.status = rc;
    if (!opt || opt->status != ENUMGPU_OK || opt->m != p->m)
        return out->cert.status = fail(ENUMGPU_ERR_ARG, "certify_optimum: opt is not an optimum of this LP (status OK, m = %d)", p->m);
    const int m = p->m, n = p->n;
    int32_t S[kMaxM];
    if (opt->best_rank >= rs.total || enumgpu_unrank(n, m, opt->best_rank, S) != 0 || memcmp(S, opt->basis, sizeof(int32_t) * m))
        return out->cert.status = fail(ENUMGPU_ERR_ARG, "certify_optimum: opt->basis is not unrank(opt->best_rank)");
    eps_opt = resolve_eps_opt(eps_opt);
    if (max_window == 0) max_window = 1ull << 24;
    memcpy(out->basis, S, sizeof(int32_t) * m);
    out->rank = opt->best_rank;
    out->key_bound = opt->key + eps_opt * fmax(1.0, fabs(opt->key));
    out->source = ENUMGPU_OPT_WINNER;
    // 1. the winner
    rc = certify_one(p, rs, S, eps_opt, &out->cert);
    out->n_launches = out->cert.n_launches;
    if (rc || out->cert.status != ENUMGPU_CERT_UNDECIDED) return rc;
    // 2. the window: the feasible bases whose key is at most key_bound, among them every optimal basis
    std::vector<uint64_t> window;
    enumgpu_result lr;
    uint64_t n_listed = 0;
    rc = list_window(p, &oc, out->key_bound, nullptr, max_window, &window, &n_listed, &lr, &out->n_window);
    out->n_launches += lr.n_launches;
    if (rc < 0) return out->cert.status = rc;
    // 3. its bases in ascending rank, a chunk at a time, up to the first chunk with an OPTIMAL one
    if (out->n_window <= max_window) {
        Certifier cf;
        if ((rc = cf.init(p, rs))) return out->cert.status = rc;
        std::vector<int32_t> bases((size_t)kCertifyChunk * m);
        std::vector<enumgpu_certificate> certs(kCertifyChunk);
        for (uint64_t i = 0; i < n_listed; i += kCertifyChunk) {
            const uint32_t k = (uint32_t)std::min<uint64_t>(kCertifyChunk, n_listed - i);
            for (uint32_t j = 0; j < k; ++j) enumgpu_unrank(n, m, window[i + j], &bases[(size_t)j * m]);
            rc = cf.run(p, rs, bases.data(), k, eps_opt, certs.data());
            out->n_launches += 1;
            if (rc) return out->cert.status = rc;
            for (uint32_t j = 0; j < k; ++j)
                if (certs[j].basis_class == ENUMGPU_BASIS_FEASIBLE && certs[j].status == ENUMGPU_CERT_OPTIMAL) {
                    out->cert = certs[j];
                    memcpy(out->basis, &bases[(size_t)j * m], sizeof(int32_t) * m);
                    out->rank = window[i + j];
                    out->window_index = i + j;
                    out->source = ENUMGPU_OPT_WINDOW;
                    return ENUMGPU_OK;
                }
        }
    }
    // 4. no optimal basis in the window, or a window above max_window: enumgpu_certify's answer at the winner
    out->source = ENUMGPU_OPT_FALLBACK;
    const int32_t before = out->cert.n_launches;
    rc = ray_fallback(p, &oc, &out->cert);
    out->n_launches += out->cert.n_launches - before;
    return rc;
}

#ifdef ENUMGPU_TRACE
// diagnostic build only: copies out the per-warp start/stop times of the last k_shared launch
extern "C" int enumgpu_trace_read(unsigned long long* out, int n_words)
{
    return (int)cudaMemcpyFromSymbol(out, enumgpu::g_trace, sizeof(unsigned long long) * (size_t)n_words);
}
extern "C" int enumgpu_trace_phase(unsigned long long* out, int n_words)
{
    return (int)cudaMemcpyFromSymbol(out, enumgpu::g_trace_phase, sizeof(unsigned long long) * (size_t)n_words);
}
extern "C" int enumgpu_trace_done(unsigned long long* out2)
{
    int rc = (int)cudaMemcpyFromSymbol(out2, enumgpu::g_trace_done, sizeof(unsigned long long) * 2);
    unsigned long long z[2] = {0, 0};
    cudaMemcpyToSymbol(enumgpu::g_trace_done, z, sizeof z);
    return rc;
}
#endif
