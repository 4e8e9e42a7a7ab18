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
#include "k_objectives.cuh"
#include "k_ranging.cuh"
#include "k_rhs_ranging.cuh"

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

// the solve entries call this after checking their arguments (no CPU fallback); *count = the number of devices
static int require_device(int* count = nullptr)
{
    const int n = enumgpu_device_count();
    if (count) *count = n;
    return n < 1 ? fail(ENUMGPU_ERR_CUDA, "no CUDA device available (libenumgpu has no CPU fallback)") : 0;
}

// ------------------------------------------------------ per-call streams and buffers

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

// The stream of one handle-free call on the current device: a non-blocking stream of its own, or the caller's,
// and with `timed` the two events of kernel_ms.  The destructor destroys what open() created, so declare it
// before the call's StreamBufs: they queue their frees on its stream while that still exists.
struct CallStream {
    int dev = 0;
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool own = false;
    CallStream() = default;
    CallStream(const CallStream&) = delete;
    CallStream& operator=(const CallStream&) = delete;
    ~CallStream()
    {
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        if (own) cudaStreamDestroy(st);
    }
    int open(bool timed, cudaStream_t caller = nullptr)
    {
        cudaGetDevice(&dev);
        keep_pool_memory(dev);
        if (caller) st = caller;
        else { CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)); own = true; }
        if (timed) { CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1)); }
        return 0;
    }
};

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
    CallStream cs;
    StreamBuf b;
    if (cs.open(true)) return -1.0;
    if (b.alloc(32, cs.st) != cudaSuccess) {
        fail(ENUMGPU_ERR_CUDA, "fp64 peak probe: %s", cudaGetErrorString(cudaGetLastError()));
        return -1.0;
    }
    double* d = b.as<double>();
    double best = 0.0;
    const struct { int chains, threads, blocks_per_sm; } cfg[] = {{4, 512, 1}, {8, 512, 1}, {8, 256, 4}, {4, 512, 2}};
    for (const auto& c : cfg) {
        const int blocks = sms * c.blocks_per_sm;
        // ~6e7 cycles of FP64 pipe per launch: iters * 16 * chains DFMA per thread, 2 cycles per warp-DFMA per sub-core
        const int iters = (int)(6.0e7 / (16.0 * c.chains * 2.0 * (c.threads / 128) * c.blocks_per_sm));
        for (int r = 0; r < repeats + 1; ++r) {
            cudaEventRecord(cs.e0, cs.st);
            unsigned long long* clk = reinterpret_cast<unsigned long long*>(d + 1);
            if (c.chains == 4) k_dfma_peak<4><<<blocks, c.threads, 0, cs.st>>>(d, iters, 1.0000001, 1e-9, clk);
            else k_dfma_peak<8><<<blocks, c.threads, 0, cs.st>>>(d, iters, 1.0000001, 1e-9, clk);
            cudaEventRecord(cs.e1, cs.st);
            if (cudaEventSynchronize(cs.e1) != cudaSuccess) { fail(ENUMGPU_ERR_CUDA, "fp64 peak probe: %s", cudaGetErrorString(cudaGetLastError())); best = -1.0; break; }
            float ms = 0.f;
            cudaEventElapsedTime(&ms, cs.e0, cs.e1);
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
    return best;
}

extern "C" double enumgpu_fp64_peak_tflops(int32_t repeats) { return enumgpu_fp64_peak_detail(repeats, nullptr); }

// ------------------------------------------------------------ launch logic

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

// pivot_rule, eps_feas and eps_piv of the options, defaults applied (the default eps_piv depends on the rule and m)
static int resolve_tolerances(const enumgpu_options* o, int m, Resolved* r)
{
    r->rule = o ? o->pivot_rule : ENUMGPU_PIVOT_ABSOLUTE;
    if (r->rule != ENUMGPU_PIVOT_ABSOLUTE && r->rule != ENUMGPU_PIVOT_RELATIVE) return fail(ENUMGPU_ERR_ARG, "unknown pivot_rule %d", r->rule);
    r->eps_feas = (o && o->eps_feas >= 0) ? o->eps_feas : 1e-9;
    r->eps_piv = (o && o->eps_piv >= 0) ? o->eps_piv : (r->rule == ENUMGPU_PIVOT_RELATIVE ? (double)m * 0x1p-52 : 1e-9);
    // -0.0 passes the tests above and means 0.  Store +0.0: k_shared classifies leaf components by the high word of
    // -eps_feas, whose sign bit must be set (with -(-0.0) = +0.0 every positive component would count as negative).
    if (r->eps_feas == 0.0) r->eps_feas = 0.0;
    if (r->eps_piv == 0.0) r->eps_piv = 0.0;
    return 0;
}

static double resolve_eps_opt(double eps_opt)
{
    if (!(eps_opt >= 0)) return 1e-9;                    // negative (or NaN): the default
    return eps_opt == 0.0 ? 0.0 : eps_opt;               // -0.0 means 0
}

// A, b and c of a problem in host memory are finite
static int check_finite(const enumgpu_problem* p)
{
    for (int j = 0; j < p->n; ++j) {
        if (!std::isfinite(p->c[j])) return fail(ENUMGPU_ERR_NONFINITE, "c[%d] is not finite", j);
        for (int i = 0; i < p->m; ++i)
            if (!std::isfinite(p->A_colmajor[i + (size_t)j * p->lda])) return fail(ENUMGPU_ERR_NONFINITE, "A(%d,%d) is not finite", i, j);
    }
    for (int i = 0; i < p->m; ++i)
        if (!std::isfinite(p->b[i])) return fail(ENUMGPU_ERR_NONFINITE, "b[%d] is not finite", i);
    return 0;
}

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
    if (const int rc = resolve_tolerances(o, p->m, r)) return rc;
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
    return host_ptrs ? check_finite(p) : 0;
}

// the absolute rule's singularity threshold eps_piv * max|A_ij|; the relative rule tests each basis (thr = 0)
static double pivot_threshold(const Resolved& rs, double scale)
{
    return rs.rule == ENUMGPU_PIVOT_RELATIVE ? 0.0 : rs.eps_piv * scale;
}

// The fields of the launch parameters that follow from the problem (device pointers) and the tolerances
static LaunchParams problem_params(const enumgpu_problem* pd, const uint64_t* d_binom, const Resolved& rs, double scale)
{
    LaunchParams prm{};
    prm.A = pd->A_colmajor; prm.b = pd->b; prm.c = pd->c; prm.binom = d_binom;
    prm.m = pd->m; prm.n = pd->n; prm.lda = pd->lda; prm.maximize = pd->maximize ? 1 : 0;
    prm.eps_feas = rs.eps_feas;
    prm.pivot_rule = rs.rule;
    prm.thr = pivot_threshold(rs, scale);
    prm.rel_eps = rs.rule == ENUMGPU_PIVOT_RELATIVE ? rs.eps_piv : 0.0;
    return prm;
}

// max|A_ij| of a problem in host memory
static double max_abs_A(const enumgpu_problem* p)
{
    double s = 0.0;
    for (int j = 0; j < p->n; ++j)
        for (int i = 0; i < p->m; ++i) s = fmax(s, fabs(p->A_colmajor[i + (size_t)j * p->lda]));
    return s;
}

// The packed copy of a problem that the device works on: A (lda = m), then b, then c
static size_t packed_doubles(const enumgpu_problem* p) { return (size_t)p->m * p->n + p->m + p->n; }

// packs host problem p into out[packed_doubles(p)]; returns max|A_ij|
static double pack_problem(const enumgpu_problem* p, double* out)
{
    const int m = p->m, n = p->n;
    for (int j = 0; j < n; ++j) memcpy(out + (size_t)j * m, p->A_colmajor + (size_t)j * p->lda, sizeof(double) * m);
    memcpy(out + (size_t)m * n, p->b, sizeof(double) * m);
    memcpy(out + (size_t)m * n + m, p->c, sizeof(double) * n);
    return max_abs_A(p);
}

// p as it reads from its packed copy at d (device memory)
static enumgpu_problem packed_view(const enumgpu_problem* p, const double* d)
{
    enumgpu_problem dp = *p;
    dp.lda = p->m;
    dp.A_colmajor = d;
    dp.b = d + (size_t)p->m * p->n;
    dp.c = dp.b + p->m;
    return dp;
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
static int rcp_selftest_device(uint64_t n_operands, uint64_t seed, uint64_t* n_mismatch, double* first_bad);
static bool shared_rcp_trusted(int dev);

// The listing of an enqueue (enumgpu_list_window): the feasible ranks whose key is at most key_max, appended in
// arrival order; *count (device memory, zero on entry) counts all of them, ranks[0, cap) holds the first cap.
struct Listing {
    unsigned long long* count;
    uint64_t* ranks;
    uint64_t cap;
    double key_max;
};

// Enqueue everything for the rank range and shard of rs on one stream of the current device.
// scale_host < 0: max|A_ij| is computed on the device first (one synchronisation of st).
static int enqueue_range(const enumgpu_problem* pd, double scale_host, const Resolved& rs, cudaStream_t st,
                         enumgpu_partial* partial_dev, int32_t* n_launches, Scratch* scratch = nullptr,
                         const Listing* list = nullptr)
{
    const uint64_t begin = rs.begin, end = rs.end;
    const uint32_t shard_index = rs.shard_index, shard_count = rs.shard_count;
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

    LaunchParams prm = problem_params(pd, d_binom, rs, scale_host);
    prm.rank_begin = begin; prm.rank_end = end; prm.chunk = 1;
    prm.shard_index = 0; prm.shard_count = 1;
    const Listing l = list ? *list : Listing{nullptr, nullptr, 0, INFINITY};
    prm.list_count = l.count; prm.list_ranks = l.ranks; prm.list_cap = l.cap; prm.list_key_max = l.key_max;
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
            // the kernel's static shared memory counts against the same maximum as the dynamic window
            // (without it the window of (m, n) = (10, 64) left too little room and the launch was refused)
            size_t static_smem = 0;
            sp.base = prm;                    // m and n select the instantiation
            CU(dispatch_shared(sp, nullptr, 0, 0, 0, st, &static_smem));
            wpc = (int)(((size_t)max_smem - cta - static_smem) / per_warp);
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
    if ((rc = require_device())) return rc;
    cudaStream_t st = o ? (cudaStream_t)o->stream : nullptr;
    return enqueue_range(p_dev, scale_A, rs, st, partial_dev, n_launches);
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
    Resolved rs{};
    int rc = resolve_tolerances(o, m, &rs);
    if (rc) return rc;
    for (int i = 0; i < m; ++i)
        if (basis[i] < 0 || basis[i] >= n) return fail(ENUMGPU_ERR_ARG, "basis index %d out of range", basis[i]);
    if ((rc = check_finite(p)) || (rc = require_device())) return rc;
    // gather (Canonical.cpp:183-187): W = [A(:, basis) | b] column-major, then c_B, then room for 1/pivot
    const size_t w_elems = (size_t)m * (m + 1);
    std::vector<double> stage(w_elems + 2 * (size_t)m);
    for (int j = 0; j < m; ++j) memcpy(&stage[(size_t)j * m], p->A_colmajor + (size_t)basis[j] * p->lda, sizeof(double) * m);
    memcpy(&stage[(size_t)m * m], p->b, sizeof(double) * m);
    for (int j = 0; j < m; ++j) stage[w_elems + j] = p->c[basis[j]];
    std::vector<double> h_out((size_t)m + 2, 0.0);
    CallStream cs;
    StreamBuf b_in, b_out;
    if ((rc = cs.open(false))) return rc;
    CU(b_in.alloc(stage.size() * sizeof(double), cs.st));
    CU(b_out.alloc(h_out.size() * sizeof(double), cs.st));
    double* d_in = b_in.as<double>();
    CU(cudaMemcpyAsync(d_in, stage.data(), stage.size() * sizeof(double), cudaMemcpyHostToDevice, cs.st));
    CU(cudaMemsetAsync(b_out.p, 0, h_out.size() * sizeof(double), cs.st));
    k_eval_any<<<1, 256, 0, cs.st>>>(d_in, d_in + w_elems, m, pivot_threshold(rs, max_abs_A(p)), rs.eps_feas, rs.rule, rs.eps_piv,
                                     d_in + w_elems + m, b_out.as<double>());
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h_out.data(), b_out.p, h_out.size() * sizeof(double), cudaMemcpyDeviceToHost, cs.st));
    CU(cudaStreamSynchronize(cs.st));
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
    std::vector<double> stage(packed_doubles(p));
    out->scale = pack_problem(p, stage.data());
    CU(out->buf.alloc(stage.size() * sizeof(double), st));
    CU(cudaMemcpyAsync(out->buf.p, stage.data(), stage.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    out->dp = packed_view(p, out->buf.as<double>());
    return 0;
}

// The timed enumeration of a synchronous entry: record e0, enqueue the range of rs, record e1, then the record
// (and the listing's count into *h_count) back to the host with one synchronisation, and the result into *out.
static int enumerate_timed(const enumgpu_problem* pd, double scale, const Resolved& rs, const CallStream& cs,
                           const Listing* list, unsigned long long* h_count, enumgpu_result* out)
{
    StreamBuf b_part;
    CU(b_part.alloc(sizeof(enumgpu_partial), cs.st));
    enumgpu_partial h_part;
    int32_t launches = 0;
    CU(cudaEventRecord(cs.e0, cs.st));
    const int rc = enqueue_range(pd, scale, rs, cs.st, b_part.as<enumgpu_partial>(), &launches, nullptr, list);
    if (rc) return rc;
    CU(cudaEventRecord(cs.e1, cs.st));
    CU(cudaMemcpyAsync(&h_part, b_part.p, sizeof h_part, cudaMemcpyDeviceToHost, cs.st));
    if (list) CU(cudaMemcpyAsync(h_count, list->count, sizeof *h_count, cudaMemcpyDeviceToHost, cs.st));
    CU(cudaStreamSynchronize(cs.st));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, cs.e0, cs.e1));
    enumgpu_partial_to_result(&h_part, out);
    out->kernel_ms = ms;
    out->n_launches = launches;
    return 0;
}

// The device part of list_window: *out, the count of the window, and the first `capacity` ranks, ascending.
static int list_window_device(const enumgpu_problem* p, const Resolved& rs, double key_max, uint64_t* ranks, uint64_t capacity,
                              std::vector<uint64_t>* fit, uint64_t* n_listed, enumgpu_result* out, uint64_t* n_window)
{
    CallStream cs;
    DeviceProblem D;
    StreamBuf b_count, b_ranks;
    int rc;
    if ((rc = cs.open(true)) || (rc = upload_problem(p, cs.st, &D))) return rc;
    CU(b_count.alloc(sizeof(unsigned long long), cs.st));
    CU(b_ranks.alloc(sizeof(uint64_t) * (capacity ? capacity : 1), cs.st));
    CU(cudaMemsetAsync(b_count.p, 0, sizeof(unsigned long long), cs.st));
    const Listing list{b_count.as<unsigned long long>(), b_ranks.as<uint64_t>(), capacity, key_max};
    unsigned long long h_count = 0;
    if ((rc = enumerate_timed(&D.dp, D.scale, rs, cs, &list, &h_count, out))) return rc;
    const uint64_t k = h_count < capacity ? (uint64_t)h_count : capacity;
    if (fit) { fit->resize(k); ranks = fit->data(); }
    if (n_window) *n_window = h_count;
    if (k) CU(cudaMemcpy(ranks, b_ranks.p, sizeof(uint64_t) * k, cudaMemcpyDeviceToHost));
    *n_listed = k;
    std::sort(ranks, ranks + k);             // the device appends in arrival order; hand them out ascending
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
    if (rc == 0) rc = require_device();
    if (rc == 0) rc = list_window_device(p, rs, key_max, ranks, capacity, fit, n_listed, out, n_window);
    if (rc) return out->status = rc;
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
    if ((rc = require_device())) return rc;
    CallStream cs;
    DeviceProblem D;
    StreamBuf b_ranks, b_x, b_z, b_cls;
    const uint64_t* d_binom = nullptr;
    if ((rc = cs.open(false)) || (rc = upload_problem(p, cs.st, &D)) || (rc = device_binom(cs.dev, &d_binom))) return rc;
    const int m = p->m;
    CU(b_ranks.alloc(sizeof(uint64_t) * count, cs.st));
    CU(b_x.alloc(sizeof(double) * count * m, cs.st));
    CU(b_z.alloc(sizeof(double) * count, cs.st));
    CU(b_cls.alloc(sizeof(int32_t) * count, cs.st));
    CU(cudaMemcpyAsync(b_ranks.p, ranks, sizeof(uint64_t) * count, cudaMemcpyHostToDevice, cs.st));
    const LaunchParams prm = problem_params(&D.dp, d_binom, rs, D.scale);
    const unsigned blocks = (unsigned)((count + 127) / 128);
    k_eval_ranks<<<blocks, 128, 0, cs.st>>>(prm, b_ranks.as<uint64_t>(), count, b_x.as<double>(), b_z.as<double>(), b_cls.as<int32_t>());
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(x_B, b_x.p, sizeof(double) * count * m, cudaMemcpyDeviceToHost, cs.st));
    CU(cudaMemcpyAsync(objective, b_z.p, sizeof(double) * count, cudaMemcpyDeviceToHost, cs.st));
    CU(cudaMemcpyAsync(basis_class, b_cls.p, sizeof(int32_t) * count, cudaMemcpyDeviceToHost, cs.st));
    CU(cudaStreamSynchronize(cs.st));
    return 0;
}

// ------------------------------------------------------------------ many objectives over one feasible set (DESIGN.md §3.2)

constexpr int32_t  kMaxObjectives = 1 << 20;
constexpr uint32_t kObjChunk = 1u << 21;      // listed bases per k_obj_values + k_objectives pass (chunk buffers: 9 B/row)

struct ObjPass {
    enumgpu_problem dp;                       // device copy, A packed (lda = m)
    const uint64_t* binom;
    const double* C;                          // device, cost vector i at C[i * n]
    int32_t k;
    int W;                                    // objectives per block (power of two <= kObjThreads)
    dim3 grid;                                // slices x objective tiles
    uint8_t* S;                               // chunk buffers, [m][chunk]
    double* x;
    Best* best;                               // [slices][k]
    cudaStream_t st;
};

// S and x_B of `count` listed ranks of the device problem dp into the chunk buffers S, x ([M][count]): 1 launch
template <int M>
static cudaError_t obj_values(const enumgpu_problem& dp, const uint64_t* binom, const uint64_t* ranks, uint32_t count,
                              uint8_t* S, double* x, cudaStream_t st)
{
    const int n = dp.n;
    const unsigned blocks = (count + kObjThreads - 1) / kObjThreads;
    if constexpr (M <= 12) {
        const size_t smem = (size_t)(n * M + M + n) * sizeof(double) + sizeof(uint64_t) * kBinomRows * kBinomCols;
        k_obj_values<M><<<blocks, kObjThreads, smem, st>>>(dp.A_colmajor, dp.b, binom, n, ranks, count, S, x);
    } else {
        k_obj_values_generic<<<blocks, kObjThreads, 0, st>>>(dp.A_colmajor, dp.b, binom, M, n, ranks, count, S, x);
    }
    return cudaGetLastError();
}

static cudaError_t dispatch_obj_values(const enumgpu_problem& dp, const uint64_t* binom, const uint64_t* ranks,
                                       uint32_t count, uint8_t* S, double* x, cudaStream_t st)
{
    switch (dp.m) {
#define ENUMGPU_CASE(M_) case M_: return obj_values<M_>(dp, binom, ranks, count, S, x, st);
        ENUMGPU_CASE(1) ENUMGPU_CASE(2) ENUMGPU_CASE(3) ENUMGPU_CASE(4)
        ENUMGPU_CASE(5) ENUMGPU_CASE(6) ENUMGPU_CASE(7) ENUMGPU_CASE(8)
        ENUMGPU_CASE(9) ENUMGPU_CASE(10) ENUMGPU_CASE(11) ENUMGPU_CASE(12)
        ENUMGPU_CASE(13) ENUMGPU_CASE(14) ENUMGPU_CASE(15) ENUMGPU_CASE(16)
#undef ENUMGPU_CASE
    }
    return cudaErrorInvalidValue;
}

// x_B of `count` listed ranks, then their keys under every cost vector: 2 launches
template <int M>
static cudaError_t objectives_chunk(const ObjPass& a, const uint64_t* ranks, uint32_t count, int first)
{
    const int n = a.dp.n;
    cudaError_t e = obj_values<M>(a.dp, a.binom, ranks, count, a.S, a.x, a.st);
    if (e != cudaSuccess) return e;
    const size_t smem = (size_t)M * kObjTile * (sizeof(double) + 1) + kObjTile * sizeof(uint64_t) + (size_t)n * a.W * sizeof(double);
    e = cudaFuncSetAttribute(k_objectives<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_objectives<M><<<a.grid, kObjThreads, smem, a.st>>>(a.S, a.x, ranks, count, n, a.dp.maximize ? 1 : 0, a.C, a.k, a.W, first,
                                                          a.best);
    return cudaGetLastError();
}

static cudaError_t dispatch_objectives(const ObjPass& a, const uint64_t* ranks, uint32_t count, int first)
{
    switch (a.dp.m) {
#define ENUMGPU_CASE(M_) case M_: return objectives_chunk<M_>(a, ranks, count, first);
        ENUMGPU_CASE(1) ENUMGPU_CASE(2) ENUMGPU_CASE(3) ENUMGPU_CASE(4)
        ENUMGPU_CASE(5) ENUMGPU_CASE(6) ENUMGPU_CASE(7) ENUMGPU_CASE(8)
        ENUMGPU_CASE(9) ENUMGPU_CASE(10) ENUMGPU_CASE(11) ENUMGPU_CASE(12)
        ENUMGPU_CASE(13) ENUMGPU_CASE(14) ENUMGPU_CASE(15) ENUMGPU_CASE(16)
#undef ENUMGPU_CASE
    }
    return cudaErrorInvalidValue;
}

// The listing of every feasible basis of a rank range for the entries that consume them all (DESIGN.md §3.2, §3.3).
// init() sizes the device list: max_list ranks (0 selects 2^26), never more than the largest range has.  run() lists
// the feasible ranks of rs's range of the device problem D (key bound +inf) and hands each listing to
// consume(record of the listed range, device ranks, count).  With more feasible bases than the list holds, the range
// is cut into contiguous sub-ranges of about cap / 2 expected feasible bases each, and one that still overflows is
// halved; the sub-ranges are consumed in ascending order.  Disjoint ranges merge exactly (enumgpu_merge_partial).
struct FeasibleLists {
    StreamBuf b_list, b_count, b_part;
    uint64_t cap = 0;

    int init(uint64_t max_list, uint64_t max_span, cudaStream_t st)
    {
        if (max_list == 0) max_list = 1ull << 26;
        cap = std::max<uint64_t>(1, std::min(max_list, max_span));
        CU(b_list.alloc(cap * sizeof(uint64_t), st));
        CU(b_count.alloc(sizeof(unsigned long long), st));
        CU(b_part.alloc(sizeof(enumgpu_partial), st));
        return 0;
    }

    template <class Consume>
    int run(const DeviceProblem& D, const Resolved& rs, cudaStream_t st, int32_t* launches, Consume&& consume)
    {
        const uint64_t span = rs.end - rs.begin, cap_r = std::max<uint64_t>(1, std::min(cap, span));
        const Listing listing{b_count.as<unsigned long long>(), b_list.as<uint64_t>(), cap_r, INFINITY};
        // the feasible ranks of [lo, hi) into b_list (all of them if *count <= cap_r) and the range's record
        auto list = [&](uint64_t lo, uint64_t hi, enumgpu_partial* lp, uint64_t* count) -> int {
            CU(cudaMemsetAsync(b_count.p, 0, sizeof(unsigned long long), st));
            Resolved sub = rs;
            sub.begin = lo; sub.end = hi;
            int32_t nl = 0;
            const int r3 = enqueue_range(&D.dp, D.scale, sub, st, b_part.as<enumgpu_partial>(), &nl, nullptr, &listing);
            if (r3) return r3;
            *launches += nl;
            unsigned long long h = 0;
            CU(cudaMemcpyAsync(lp, b_part.p, sizeof *lp, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(&h, b_count.p, sizeof h, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            *count = h;
            return 0;
        };
        const uint64_t* ranks = b_list.as<uint64_t>();
        enumgpu_partial lp;
        uint64_t count = 0;
        int rc;
        if ((rc = list(rs.begin, rs.end, &lp, &count))) return rc;
        if (count <= cap_r) return consume(lp, ranks, count);
        const uint64_t per = std::max<uint64_t>(1, cap_r / 2), parts = std::min(span, (count + per - 1) / per);
        std::vector<std::pair<uint64_t, uint64_t>> todo;            // a stack: ascending ranges from its back
        for (uint64_t i = parts; i-- > 0;)
            todo.emplace_back(rs.begin + (uint64_t)((unsigned __int128)span * i / parts),
                              rs.begin + (uint64_t)((unsigned __int128)span * (i + 1) / parts));
        while (!todo.empty()) {
            const auto [lo, hi] = todo.back();
            todo.pop_back();
            if ((rc = list(lo, hi, &lp, &count))) return rc;
            if (count <= cap_r) {
                if ((rc = consume(lp, ranks, count))) return rc;
                continue;
            }
            const uint64_t mid = lo + (hi - lo) / 2;                 // a single rank never overflows: cap_r >= 1
            todo.emplace_back(mid, hi);
            todo.emplace_back(lo, mid);
        }
        return 0;
    }
};

// The device part of enumgpu_solve_objectives for q (c = column 0 of C) and the resolved options: out[0, k).
static int solve_objectives_device(const enumgpu_problem* q, const Resolved& rs, int32_t k, const double* C, int32_t ldc,
                                   uint64_t max_list, enumgpu_result* out)
{
    const int m = q->m, n = q->n;
    CallStream cs;
    DeviceProblem D;
    FeasibleLists fl;
    StreamBuf b_C, b_S, b_x, b_best, b_rec;
    ObjPass a;
    int rc;
    if ((rc = cs.open(true)) || (rc = upload_problem(q, cs.st, &D)) || (rc = device_binom(cs.dev, &a.binom))) return rc;
    // the list never holds more than the range has ranks
    if ((rc = fl.init(max_list, rs.end - rs.begin, cs.st))) return rc;
    const uint32_t chunk = (uint32_t)std::min<uint64_t>(kObjChunk, fl.cap);
    const cudaStream_t st = cs.st;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cs.dev);
    std::vector<enumgpu_partial> acc((size_t)k), recs((size_t)k);
    int32_t launches = 0;
    a.dp = D.dp;
    std::vector<double> hC((size_t)k * n);
    for (int32_t i = 0; i < k; ++i) memcpy(&hC[(size_t)i * n], C + (size_t)i * ldc, sizeof(double) * n);
    a.k = k;
    a.W = 1;
    while (a.W < k && a.W < kObjThreads) a.W *= 2;
    const uint32_t tiles = (uint32_t)((k + a.W - 1) / a.W);
    const uint32_t slices = std::max<uint32_t>(1, (uint32_t)(4 * sms) / tiles);
    a.grid = dim3(slices, tiles);
    a.st = st;
    CU(b_C.alloc(hC.size() * sizeof(double), st));
    CU(b_S.alloc((size_t)chunk * m, st));
    CU(b_x.alloc((size_t)chunk * m * sizeof(double), st));
    CU(b_best.alloc((size_t)slices * k * sizeof(Best), st));
    CU(b_rec.alloc((size_t)k * sizeof(enumgpu_partial), st));
    CU(cudaMemcpyAsync(b_C.p, hC.data(), hC.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    a.C = b_C.as<double>(); a.S = b_S.as<uint8_t>(); a.x = b_x.as<double>(); a.best = b_best.as<Best>();
    CU(cudaEventRecord(cs.e0, st));

    // every objective's best over the listed ranks, merged into acc with the range's counters
    bool have = false;
    auto absorb = [&](const enumgpu_partial& lp, const uint64_t* ranks, uint64_t count) -> int {
        for (uint64_t c0 = 0; c0 < count; c0 += chunk) {
            CU(dispatch_objectives(a, ranks + c0, (uint32_t)std::min<uint64_t>(chunk, count - c0), c0 == 0));
            launches += 2;
        }
        k_obj_finish<<<(unsigned)((k + kObjThreads - 1) / kObjThreads), kObjThreads, 0, st>>>(
            a.best, count ? (int)slices : 0, D.dp.A_colmajor, D.dp.b, a.C, a.binom, m, n, k, b_rec.as<enumgpu_partial>());
        CU(cudaGetLastError());
        ++launches;
        CU(cudaMemcpyAsync(recs.data(), b_rec.p, (size_t)k * sizeof(enumgpu_partial), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        for (int32_t i = 0; i < k; ++i) {
            enumgpu_partial& r = recs[i];
            r.n_bases = lp.n_bases; r.n_singular = lp.n_singular; r.n_infeasible = lp.n_infeasible; r.n_feasible = lp.n_feasible;
            r.algo_used = lp.algo_used;
            if (have) enumgpu_merge_partial(&acc[i], &r);
            else acc[i] = r;
        }
        have = true;
        return 0;
    };
    if ((rc = fl.run(D, rs, st, &launches, absorb))) return rc;
    CU(cudaEventRecord(cs.e1, st));
    CU(cudaStreamSynchronize(st));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, cs.e0, cs.e1));
    for (int32_t i = 0; i < k; ++i) {
        enumgpu_partial_to_result(&acc[i], &out[i]);
        out[i].kernel_ms = ms;
        out[i].n_launches = launches;
    }
    return ENUMGPU_OK;
}

extern "C" int enumgpu_solve_objectives(const enumgpu_problem* p, const enumgpu_options* o, int32_t k, const double* C,
                                        int32_t ldc, uint64_t max_list, enumgpu_result* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "solve_objectives: out is NULL");
    if (k < 1 || k > kMaxObjectives) return fail(ENUMGPU_ERR_ARG, "solve_objectives: k=%d outside 1..%d", k, kMaxObjectives);
    memset(out, 0, sizeof(enumgpu_result) * (size_t)k);
    auto all = [&](int rc) { for (int32_t i = 0; i < k; ++i) out[i].status = rc; return rc; };
    if (!p) return all(fail(ENUMGPU_ERR_ARG, "problem is NULL"));
    if (!C) return all(fail(ENUMGPU_ERR_ARG, "solve_objectives: C is NULL"));
    if (ldc < p->n) return all(fail(ENUMGPU_ERR_ARG, "solve_objectives: ldc=%d < n=%d", ldc, p->n));
    if (o && (o->shard_index != 0 || o->shard_count != 0))
        return all(fail(ENUMGPU_ERR_ARG, "solve_objectives: shards are not supported (split the range with enumgpu_shard_begin)"));
    enumgpu_problem q = *p;
    q.c = C;                                  // p->c is not read; column 0 stands in where the enumeration wants a c
    Resolved rs;
    int rc = resolve(&q, o, &rs, true);
    if (rc) return all(rc);
    for (int32_t i = 0; i < k; ++i)
        for (int j = 0; j < p->n; ++j)
            if (!std::isfinite(C[j + (size_t)i * ldc])) return all(fail(ENUMGPU_ERR_NONFINITE, "C(%d,%d) is not finite", j, i));
    if ((rc = require_device()) || (rc = solve_objectives_device(&q, rs, k, C, ldc, max_list, out))) return all(rc);
    return ENUMGPU_OK;
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

static int rcp_selftest_device(uint64_t n_operands, uint64_t seed, uint64_t* n_mismatch, double* first_bad)
{
    CallStream cs;
    StreamBuf b;
    if (const int rc = cs.open(false)) return rc;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cs.dev);
    CU(b.alloc(16, cs.st));
    unsigned long long* d = b.as<unsigned long long>();
    CU(cudaMemsetAsync(d, 0, 16, cs.st));
    k_rcp_selftest<<<sms * 8, 256, 0, cs.st>>>(n_operands, seed, d, d + 1);
    CU(cudaGetLastError());
    unsigned long long h[2] = {0, 0};
    CU(cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, cs.st));
    CU(cudaStreamSynchronize(cs.st));
    *n_mismatch = h[0];
    if (first_bad) memcpy(first_bad, &h[1], 8);
    return 0;
}

extern "C" int enumgpu_selftest_rcp(uint64_t n_operands, uint64_t seed, uint64_t* n_mismatch, double* first_bad)
{
    g_err[0] = 0;
    if (!n_mismatch) return fail(ENUMGPU_ERR_ARG, "selftest_rcp: n_mismatch is NULL");
    if (const int rc = require_device()) return rc;
    return rcp_selftest_device(n_operands, seed, n_mismatch, first_bad);
}

static bool shared_rcp_trusted(int dev)
{
    std::lock_guard<std::mutex> lock(g_tables_mu);
    DeviceTables& t = g_tables[dev];
    if (t.rcp_state == 0) {
        uint64_t bad = 1;
        double first = 0.0;
        const int rc = rcp_selftest_device(1ull << 22, 0x5EEDull, &bad, &first);
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
    int have = 0;
    if (const int rc = require_device(&have)) return rc;
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
    // the packed problem in the pinned staging buffer of handle 0
    enumgpu_handle* h0 = hs[0];
    const double scale = pack_problem(p, h0->h_in);
    const size_t bytes = packed_doubles(p) * sizeof(double);
    int cur = 0;
    cudaGetDevice(&cur);
    int32_t launches[ENUMGPU_MAX_DEVICES] = {0};
    auto body = [&]() -> int {
        for (int i = 0; i < n_handles; ++i) {
            enumgpu_handle* h = hs[i];
            Resolved rd = rs;
            rd.shard_index = rs.shard_index + rs.shard_count * (uint32_t)i;
            rd.shard_count = rs.shard_count * (uint32_t)n_handles;
            CU(cudaSetDevice(h->dev));
            CU(cudaMemcpyAsync(h->d_in, h0->h_in, bytes, cudaMemcpyHostToDevice, h->st));
            const enumgpu_problem dp = packed_view(p, h->d_in);
            CU(cudaEventRecord(h->e0, h->st));
            const int r2 = enqueue_range(&dp, scale, rd, h->st, h->d_part, &launches[i], &h->scratch);
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

// enumgpu_enqueue_h (host_ptrs false: p and scale_A as the caller gives them) and enumgpu_enqueue_host_h (host_ptrs
// true: p is packed into the handle's pinned staging buffer and copied to the device first), on o->stream or the
// handle's stream.  A failure leaves the handle ready for the next call.
static int handle_enqueue(const char* who, enumgpu_handle* h, const enumgpu_problem* p, bool host_ptrs, double scale_A,
                          const enumgpu_options* o, enumgpu_partial* partial_dev, int32_t* n_launches)
{
    g_err[0] = 0;
    if (!h) return fail(ENUMGPU_ERR_ARG, "handle is NULL");
    Resolved rs;
    int rc = resolve(p, o, &rs, host_ptrs);
    if (rc) return rc;
    if (!partial_dev) return fail(ENUMGPU_ERR_ARG, "partial_dev is NULL");
    int cur = 0;
    cudaGetDevice(&cur);
    if (cur != h->dev) return fail(ENUMGPU_ERR_ARG, "%s: the handle belongs to device %d, the current device is %d", who, h->dev, cur);
    cudaStream_t st = (o && o->stream) ? (cudaStream_t)o->stream : h->st;
    enumgpu_problem dp = *p;
    if (host_ptrs) {
        scale_A = pack_problem(p, h->h_in);
        dp = packed_view(p, h->d_in);
        const cudaError_t e = cudaMemcpyAsync(h->d_in, h->h_in, packed_doubles(p) * sizeof(double), cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) rc = fail(ENUMGPU_ERR_CUDA, "%s: H2D copy failed: %s", who, cudaGetErrorString(e));
    }
    if (rc == 0) rc = enqueue_range(&dp, scale_A, rs, st, partial_dev, n_launches, &h->scratch);
    if (rc) { cudaStreamSynchronize(st); handle_recover(h); }
    return rc;
}

extern "C" int enumgpu_enqueue_h(enumgpu_handle* h, const enumgpu_problem* p_dev, double scale_A, const enumgpu_options* o,
                                 enumgpu_partial* partial_dev, int32_t* n_launches)
{
    return handle_enqueue("enqueue_h", h, p_dev, false, scale_A, o, partial_dev, n_launches);
}

// enumgpu_enqueue_h for HOST inputs: pack A|b|c into the handle's pinned staging buffer, one H2D copy and the
// enumeration, all on one stream, no synchronisation.  The building block of a one-process-per-GPU solve
// (dist.ShardedEnumeration): the caller appends its collective and one D2H copy to the same stream.
extern "C" int enumgpu_enqueue_host_h(enumgpu_handle* h, const enumgpu_problem* p, const enumgpu_options* o,
                                      enumgpu_partial* partial_dev, int32_t* n_launches)
{
    return handle_enqueue("enqueue_host_h", h, p, true, 0.0, o, partial_dev, n_launches);
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
    if (rc == 0) rc = require_device();
    if (rc) return out->status = rc;
    CallStream cs;
    rc = cs.open(true, o ? (cudaStream_t)o->stream : nullptr);
    if (rc == 0) rc = enumerate_timed(p_dev, scale_A, rs, cs, nullptr, nullptr, out);
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
    int have = 0;
    if (rc == 0) rc = require_device(&have);
    if (rc) return out->status = rc;

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

// The auxiliary LP of the ray enumerations: [A; s*row'] d = (0, ..., 0, rhs), cost 0, minimise; the caller sets rhs
// (b[m]).  s = 2^e, the largest power of two with s*max|row_j| <= max|A_ij|, keeps max|A'_ij| = max|A_ij| and with it
// the pivot threshold.  max|row_j| > 0.  ENUMGPU_ERR_RANGE when max|A_ij| = 0 or scaling by s would lose bits of a row_j.
struct AuxLP {
    std::vector<double> A, b, c;
    enumgpu_problem p;
    double s;
};
static int build_aux_lp(const enumgpu_problem* p, const double* row, const char* who, AuxLP* out)
{
    const int m = p->m, n = p->n, ma = m + 1;
    const double amax = max_abs_A(p);
    double rmax = 0.0;
    for (int j = 0; j < n; ++j) rmax = fmax(rmax, fabs(row[j]));
    if (amax == 0.0) return fail(ENUMGPU_ERR_RANGE, "%s: A = 0 leaves no scale for the auxiliary row", who);
    int ea = 0, er = 0;
    const double fa = frexp(amax, &ea), fr = frexp(rmax, &er);
    const int e = ea - er - (fr > fa ? 1 : 0);
    out->A.assign((size_t)ma * n, 0.0);
    out->b.assign(ma, 0.0);
    out->c.assign(n, 0.0);
    for (int j = 0; j < n; ++j) {
        for (int i = 0; i < m; ++i) out->A[(size_t)j * ma + i] = p->A_colmajor[i + (size_t)j * p->lda];
        const double v = ldexp(row[j], e);
        if (ldexp(v, -e) != row[j]) return fail(ENUMGPU_ERR_RANGE, "%s: row[%d] * 2^%d is not exact", who, j, e);
        out->A[(size_t)j * ma + m] = v;
    }
    out->s = ldexp(1.0, e);
    out->p = enumgpu_problem{ma, n, ma, 0, out->A.data(), out->b.data(), out->c.data()};
    return 0;
}

// The auxiliary LP with row ck and rhs -1: its feasible bases are the extreme rays of {d >= 0, A d = 0} with ck.d < 0.
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
    std::vector<double> ck(n);
    double cmax = 0.0;
    for (int j = 0; j < n; ++j) {
        ck[j] = p->maximize ? -p->c[j] : p->c[j];
        cmax = fmax(cmax, fabs(p->c[j]));
    }
    out->m = ma;
    if (n < ma || cmax == 0.0) {          // no basis of m+1 columns, or no direction can decrease ck.x
        out->key = INFINITY; out->best_rank = UINT64_MAX; out->objective = NAN;
        return out->status = ENUMGPU_NO_FEASIBLE;
    }
    AuxLP aux;
    if ((rc = build_aux_lp(p, ck.data(), "find_ray", &aux))) return out->status = rc;
    aux.b[m] = -1.0;
    return enumgpu_solve(&aux.p, o, out);
}

// k_certify on a list of bases, kCertifyChunk blocks per launch at most: the device copy of the LP, the scratch
// slabs and the staging of the bases and certificates are sized by the chunk, not by the number of bases.
constexpr uint32_t kCertifyChunk = 4096;
struct Certifier {
    CallStream cs;                     // declared first: destroyed after the buffers have queued their frees on it
    DeviceProblem D;
    StreamBuf b_scratch, b_S, b_out;
    double thr = 0.0;

    int init(const enumgpu_problem* p, const Resolved& rs)
    {
        int rc;
        if ((rc = cs.open(false)) || (rc = upload_problem(p, cs.st, &D))) return rc;
        thr = pivot_threshold(rs, D.scale);
        CU(b_scratch.alloc(sizeof(double) * certify_slab(p->m, p->n) * kCertifyChunk, cs.st));
        CU(b_S.alloc(sizeof(int32_t) * p->m * kCertifyChunk, cs.st));
        CU(b_out.alloc(sizeof(enumgpu_certificate) * kCertifyChunk, cs.st));
        return 0;
    }
    // count <= kCertifyChunk bases of m columns each (host); out[i] as the kernel leaves it, n_launches = 1
    int run(const enumgpu_problem* p, const Resolved& rs, const int32_t* bases, uint32_t count, double eps_opt,
            enumgpu_certificate* out)
    {
        const int m = p->m, n = p->n;
        CU(cudaMemcpyAsync(b_S.p, bases, sizeof(int32_t) * m * count, cudaMemcpyHostToDevice, cs.st));
        CU(cudaMemsetAsync(b_out.p, 0, sizeof(enumgpu_certificate) * count, cs.st));
        k_certify<<<count, kCertifyThreads, 0, cs.st>>>(D.dp.A_colmajor, D.dp.b, D.dp.c, b_S.as<int>(), m, n, p->maximize ? 1 : 0,
                                                        thr, rs.eps_feas, rs.rule, rs.eps_piv, eps_opt, b_scratch.as<double>(),
                                                        b_out.as<enumgpu_certificate>());
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(out, b_out.p, sizeof(enumgpu_certificate) * count, cudaMemcpyDeviceToHost, cs.st));
        CU(cudaStreamSynchronize(cs.st));
        for (uint32_t i = 0; i < count; ++i) out[i].n_launches = 1;
        return 0;
    }
};

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
    Certifier cf;
    int rc = require_device();
    if (rc == 0) rc = cf.init(p, rs);
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
    eps_opt = resolve_eps_opt(eps_opt);
    Certifier cf;
    if ((rc = require_device()) || (rc = cf.init(p, rs))) return rc;
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

// ------------------------------------------------------------------ cost ranging (DESIGN.md §3.3)

// The device part of enumgpu_cost_ranges: both listings, the ranging kernels over each listed chunk, the finish.
// aux: the ray LP, or NULL where m + 1 rows do not fit or n = m.
static int cost_ranges_device(const enumgpu_problem* p, const Resolved& rs, const AuxLP* aux, const Resolved& rsa,
                              const enumgpu_result* opt, double eps_opt, uint64_t max_list, enumgpu_ranging* out)
{
    const int m = p->m, n = p->n, rows = aux ? m + 1 : m;
    CallStream cs;
    DeviceProblem D, Da;
    FeasibleLists fl;
    StreamBuf b_S, b_x, b_vec, b_Sstar, b_best, b_flags, b_out;
    const uint64_t* binom = nullptr;
    int rc;
    if ((rc = cs.open(true)) || (rc = upload_problem(p, cs.st, &D)) || (rc = device_binom(cs.dev, &binom))) return rc;
    if (aux && (rc = upload_problem(&aux->p, cs.st, &Da))) return rc;
    const cudaStream_t st = cs.st;
    if ((rc = fl.init(max_list, std::max(rs.total, aux ? rsa.total : 0), st))) return rc;
    const uint32_t chunk = (uint32_t)std::min<uint64_t>(kObjChunk, fl.cap);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cs.dev);
    const unsigned slices = (unsigned)(4 * sms);
    // c | ck | x* | eps_opt * max(1, |x*_j|)
    std::vector<double> vec((size_t)4 * n, 0.0);
    for (int j = 0; j < n; ++j) {
        vec[j] = p->c[j];
        vec[n + j] = p->maximize ? -p->c[j] : p->c[j];
    }
    for (int i = 0; i < m; ++i) vec[2 * n + opt->basis[i]] = opt->x_B[i];
    for (int j = 0; j < n; ++j) vec[3 * n + j] = eps_opt * fmax(1.0, fabs(vec[2 * n + j]));
    const double key_star = opt->key, tau_k = eps_opt * fmax(1.0, fabs(key_star));
    CU(b_S.alloc((size_t)chunk * rows, st));
    CU(b_x.alloc((size_t)chunk * rows * sizeof(double), st));
    CU(b_vec.alloc(vec.size() * sizeof(double), st));
    CU(b_Sstar.alloc(sizeof(int32_t) * m, st));
    CU(b_best.alloc((size_t)slices * 3 * n * sizeof(Best), st));
    CU(b_flags.alloc(2 * sizeof(int), st));
    CU(b_out.alloc((size_t)n * sizeof(enumgpu_cost_range), st));
    CU(cudaMemcpyAsync(b_vec.p, vec.data(), vec.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(b_Sstar.p, opt->basis, sizeof(int32_t) * m, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(b_flags.p, 0, 2 * sizeof(int), st));
    const double* d_vec = b_vec.as<double>();
    int32_t launches = 0;
    CU(cudaEventRecord(cs.e0, st));

    // the candidates of every listed basis of the family `ray` (problem *P) folded into the slices' minima
    bool have[2] = {false, false};
    int ray = 0;
    const DeviceProblem* P = &D;
    uint64_t* n_bases = &out->n_vertex_bases;
    auto absorb = [&](const enumgpu_partial& lp, const uint64_t* ranks, uint64_t count) -> int {
        *n_bases += lp.n_feasible;
        for (uint64_t c0 = 0; c0 < count; c0 += chunk) {
            const uint32_t k = (uint32_t)std::min<uint64_t>(chunk, count - c0);
            CU(dispatch_obj_values(P->dp, binom, ranks + c0, k, b_S.as<uint8_t>(), b_x.as<double>(), st));
            k_ranging<<<slices, kRangeThreads, 0, st>>>(b_S.as<uint8_t>(), b_x.as<double>(), ranks + c0, k, P->dp.m, n, ray,
                                                       p->maximize ? 1 : 0, d_vec + (ray ? n : 0), d_vec + 2 * n, d_vec + 3 * n,
                                                       b_Sstar.as<int32_t>(), m, key_star, tau_k, eps_opt, have[ray] ? 0 : 1,
                                                       b_best.as<Best>(), b_flags.as<int>());
            CU(cudaGetLastError());
            launches += 2;
            have[ray] = true;
        }
        return 0;
    };
    if ((rc = fl.run(D, rs, st, &launches, absorb))) return rc;
    if (aux) {
        ray = 1; P = &Da; n_bases = &out->n_ray_bases;
        if ((rc = fl.run(Da, rsa, st, &launches, absorb))) return rc;
    }
    k_ranging_finish<<<(unsigned)((n + kRangeThreads - 1) / kRangeThreads), kRangeThreads, 0, st>>>(
        b_best.as<Best>(), have[0] ? (int)slices : 0, have[1] ? (int)slices : 0, n, p->maximize ? 1 : 0,
        b_out.as<enumgpu_cost_range>());
    CU(cudaGetLastError());
    ++launches;
    CU(cudaEventRecord(cs.e1, st));
    int flags[2] = {0, 0};
    CU(cudaMemcpyAsync(out->range, b_out.p, (size_t)n * sizeof(enumgpu_cost_range), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(flags, b_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, cs.e0, cs.e1));
    out->kernel_ms = ms;
    out->n_launches = launches;
    if (flags[0]) return fail(ENUMGPU_ERR_ARG, "cost_ranges: a feasible basis has a key below opt->key (opt came from other options)");
    if (flags[1]) {
        out->status = ENUMGPU_CERT_UNBOUNDED;
        for (int j = 0; j < n; ++j)
            out->range[j] = enumgpu_cost_range{NAN, NAN, UINT64_MAX, UINT64_MAX, 0, 0};
    } else {
        out->status = (m + 1 > kMaxM && n > m) ? ENUMGPU_CERT_UNDECIDED : ENUMGPU_CERT_OPTIMAL;
    }
    return ENUMGPU_OK;
}

extern "C" int enumgpu_cost_ranges(const enumgpu_problem* p, const enumgpu_options* o, const enumgpu_result* opt,
                                   double eps_opt, uint64_t max_list, enumgpu_ranging* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "cost_ranges: out is NULL");
    memset(out, 0, sizeof *out);
    if (o && (o->rank_begin != 0 || o->rank_end != 0))
        return out->status = fail(ENUMGPU_ERR_ARG, "cost_ranges: a rank range is not supported (the ranges are a statement about the whole space)");
    if (o && (o->shard_index != 0 || o->shard_count != 0))
        return out->status = fail(ENUMGPU_ERR_ARG, "cost_ranges: shards are not supported");
    const enumgpu_options oc = whole_space_options(o);
    Resolved rs, rsa{};
    int rc = resolve(p, &oc, &rs, true);
    if (rc) return out->status = rc;
    const int m = p->m, n = p->n;
    out->n = n;
    if (!opt || opt->status != ENUMGPU_OK || opt->m != m || opt->n_bases != rs.total)
        return out->status = fail(ENUMGPU_ERR_ARG, "cost_ranges: opt is not the whole-range optimum of this LP (status OK, m = %d, n_bases = C(%d, %d))", m, n, m);
    int32_t S[kMaxM];
    if (opt->best_rank >= rs.total || enumgpu_unrank(n, m, opt->best_rank, S) != 0 || memcmp(S, opt->basis, sizeof(int32_t) * m))
        return out->status = fail(ENUMGPU_ERR_ARG, "cost_ranges: opt->basis is not unrank(opt->best_rank)");
    eps_opt = resolve_eps_opt(eps_opt);
    // the rays: the feasible bases of [A; s*1'] d = (0, ..., 0, s), normalised to 1'd = 1
    AuxLP aux;
    const bool rays = m + 1 <= kMaxM && n > m;
    if (rays) {
        const std::vector<double> ones(n, 1.0);
        if ((rc = build_aux_lp(p, ones.data(), "cost_ranges", &aux))) return out->status = rc;
        aux.b[m] = aux.s;
        if ((rc = resolve(&aux.p, &oc, &rsa, true))) return out->status = rc;
    }
    if ((rc = require_device()) || (rc = cost_ranges_device(p, rs, rays ? &aux : nullptr, rsa, opt, eps_opt, max_list, out)))
        return out->status = rc;
    return ENUMGPU_OK;
}

// ------------------------------------------------------------------ right-hand-side ranging (DESIGN.md §3.4)

struct RhsLaunch {
    const double* A;
    const int32_t* J;
    int n_tight, n;
    const uint64_t* binom;
    uint64_t total, total_full, rank_star;
    double thr, rel_eps, eps_feas, eps_opt;
    int rule;
    Best* best;
    unsigned long long* counters;
};

// The grid is the resident blocks that fill the device, or fewer when the runs of kRhsRun ranks are fewer; the block
// count sizes `best`, so it comes back in *blocks.  a.best == nullptr: only the grid.
template <int M>
static cudaError_t launch_rhs(const RhsLaunch& a, int dev, cudaStream_t st, unsigned* blocks)
{
    if (!a.best) {
        int sms = 148, per_sm = 1;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_rhs_ranging<M>, kRhsThreads, 0);
        if (e != cudaSuccess) return e;
        const uint64_t need = ((a.total + kRhsRun - 1) / kRhsRun + kRhsWarps - 1) / kRhsWarps;
        *blocks = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(need, (uint64_t)sms * std::max(per_sm, 1)));
        return cudaSuccess;
    }
    k_rhs_ranging<M><<<*blocks, kRhsThreads, 0, st>>>(a.A, a.A + (size_t)M * a.n, a.J, a.n_tight, a.n, a.binom, a.total,
                                                      a.total_full, a.rank_star, a.thr, a.rule, a.rel_eps, a.eps_feas,
                                                      a.eps_opt, a.best, a.counters);
    return cudaGetLastError();
}

static cudaError_t dispatch_rhs(int m, const RhsLaunch& a, int dev, cudaStream_t st, unsigned* blocks)
{
    switch (m) {
#define ENUMGPU_CASE(M_) case M_: return launch_rhs<M_>(a, dev, st, blocks);
        ENUMGPU_CASE(1) ENUMGPU_CASE(2) ENUMGPU_CASE(3) ENUMGPU_CASE(4)
        ENUMGPU_CASE(5) ENUMGPU_CASE(6) ENUMGPU_CASE(7) ENUMGPU_CASE(8)
        ENUMGPU_CASE(9) ENUMGPU_CASE(10) ENUMGPU_CASE(11) ENUMGPU_CASE(12)
        ENUMGPU_CASE(13) ENUMGPU_CASE(14) ENUMGPU_CASE(15) ENUMGPU_CASE(16)
#undef ENUMGPU_CASE
    }
    return cudaErrorInvalidValue;
}

// The device part of enumgpu_rhs_ranges: every m-subset of J (out->tight) in one launch, then the finish.
static int rhs_ranges_device(const enumgpu_problem* p, const Resolved& rs, const enumgpu_optimum* dual, double eps_opt,
                             enumgpu_rhs_ranging* out)
{
    const int m = p->m, n = p->n;
    CallStream cs;
    DeviceProblem D;
    StreamBuf b_J, b_y, b_best, b_cnt, b_out;
    const uint64_t* binom = nullptr;
    int rc;
    if ((rc = cs.open(true)) || (rc = upload_problem(p, cs.st, &D)) || (rc = device_binom(cs.dev, &binom))) return rc;
    const cudaStream_t st = cs.st;
    RhsLaunch a{D.dp.A_colmajor, nullptr, out->n_tight, n, binom, out->n_bases, rs.total, dual->rank,
                pivot_threshold(rs, D.scale), rs.rule == ENUMGPU_PIVOT_RELATIVE ? rs.eps_piv : 0.0, rs.eps_feas, eps_opt,
                rs.rule, nullptr, nullptr};
    unsigned blocks = 0;
    CU(dispatch_rhs(m, a, cs.dev, st, &blocks));
    CU(b_J.alloc(sizeof(int32_t) * out->n_tight, st));
    CU(b_y.alloc(sizeof(double) * m, st));
    CU(b_best.alloc(sizeof(Best) * 2 * m * blocks, st));
    CU(b_cnt.alloc(2 * sizeof(unsigned long long), st));
    CU(b_out.alloc(sizeof(enumgpu_rhs_range) * m, st));
    CU(cudaMemcpyAsync(b_J.p, out->tight, sizeof(int32_t) * out->n_tight, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(b_y.p, dual->cert.y, sizeof(double) * m, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(b_cnt.p, 0, 2 * sizeof(unsigned long long), st));
    a.J = b_J.as<int32_t>();
    a.best = b_best.as<Best>();
    a.counters = b_cnt.as<unsigned long long>();
    CU(cudaEventRecord(cs.e0, st));
    CU(dispatch_rhs(m, a, cs.dev, st, &blocks));
    k_rhs_ranging_finish<<<1, 32, 0, st>>>(b_best.as<Best>(), (int)blocks, m, b_y.as<double>(), b_out.as<enumgpu_rhs_range>());
    CU(cudaGetLastError());
    CU(cudaEventRecord(cs.e1, st));
    unsigned long long cnt[2] = {0, 0};
    CU(cudaMemcpyAsync(out->range, b_out.p, sizeof(enumgpu_rhs_range) * m, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(cnt, b_cnt.p, sizeof cnt, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, cs.e0, cs.e1));
    out->kernel_ms = ms;
    out->n_launches = 2;
    out->n_singular = cnt[0];
    if (cnt[1]) return fail(ENUMGPU_ERR_ARG, "rhs_ranges: the basis of dual is singular or infeasible under these options (dual came from other options)");
    out->status = ENUMGPU_CERT_OPTIMAL;
    return ENUMGPU_OK;
}

extern "C" int enumgpu_rhs_ranges(const enumgpu_problem* p, const enumgpu_options* o, const enumgpu_optimum* dual,
                                  double eps_opt, enumgpu_rhs_ranging* out)
{
    g_err[0] = 0;
    if (!out) return fail(ENUMGPU_ERR_ARG, "rhs_ranges: out is NULL");
    memset(out, 0, sizeof *out);
    if (o && (o->rank_begin != 0 || o->rank_end != 0))
        return out->status = fail(ENUMGPU_ERR_ARG, "rhs_ranges: a rank range is not supported (the ranges are a statement about the whole space)");
    if (o && (o->shard_index != 0 || o->shard_count != 0))
        return out->status = fail(ENUMGPU_ERR_ARG, "rhs_ranges: shards are not supported");
    const enumgpu_options oc = whole_space_options(o);
    Resolved rs;
    int rc = resolve(p, &oc, &rs, true);
    if (rc) return out->status = rc;
    const int m = p->m, n = p->n;
    out->m = m;
    int32_t S[kMaxM];
    if (!dual || dual->cert.m != m || dual->cert.n != n || dual->cert.status < 0 || dual->rank >= rs.total ||
        enumgpu_unrank(n, m, dual->rank, S) != 0 || memcmp(S, dual->basis, sizeof(int32_t) * m))
        return out->status = fail(ENUMGPU_ERR_ARG, "rhs_ranges: dual is not an optimum of this LP (enumgpu_certify_optimum, m = %d, n = %d)", m, n);
    if (dual->cert.status != ENUMGPU_CERT_OPTIMAL) {     // no dual-feasible y*: no ranges
        out->status = dual->cert.status;
        for (int i = 0; i < m; ++i) out->range[i] = enumgpu_rhs_range{NAN, NAN, NAN, UINT64_MAX, UINT64_MAX};
        return ENUMGPU_OK;
    }
    eps_opt = resolve_eps_opt(eps_opt);
    // J: the basis and every column whose reduced cost is tight at y*
    for (int j = 0, k = 0; j < n; ++j) {
        const bool basic = k < m && S[k] == j;
        if (basic) ++k;
        const double r = dual->cert.reduced_cost[j], rk = p->maximize ? -r : r;
        if (basic || rk <= eps_opt) out->tight[out->n_tight++] = j;
    }
    out->n_bases = binom_mk(out->n_tight, m);
    if ((rc = require_device()) || (rc = rhs_ranges_device(p, rs, dual, eps_opt, out))) {
        out->status = rc;
        return rc;
    }
    return ENUMGPU_OK;
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
