// pareben.cu -- host side of libpareben.so: problem upload, per-fold layout kernels, the
// persistent batched-fit launch, and the extern "C" entry points declared in include/pareben.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -fmad=false --shared ...
// (-fmad=false keeps the scalar decision formulas un-contracted like the reference's x86 build;
//  the hot loops use explicit fma()).
#include "../../include/pareben.h"
#include "common.cuh"
#include "fit_launch.h"
#include "stream_launch.h"

#include <algorithm>
#include <map>
#include <thread>
#include <chrono>
#include <mutex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace pareben;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) { g_err = msg; return code; }

// 0 = auto, 1 = cached kernel (fit_kernel.cuh), 2 = streaming kernels (stream.cuh)
int g_mode = 0;

// Streaming mode is for candidate sets whose per-fit cache cannot exist (config 5: Kc = 2e8).  Auto: above
// PAREBEN_STREAM_KC candidates (default 4,000,000: at 64 active bases the cache alone would be 2 GB per resident fit).
bool want_streaming(int kc, int prior)
{
    if (prior != PAREBEN_GAUSSIAN) return false;          // the binomial solver has no streaming form yet
    if (g_mode == 1) return false;
    if (g_mode == 2) return true;
    const char *e = getenv("PAREBEN_STREAM_KC");
    const long long lim = e ? atoll(e) : 4000000LL;
    return (long long)kc > lim;
}

// Per-device pool of device allocations.  cudaMalloc/cudaFree synchronise the device and can
// take hundreds of milliseconds for multi-GB buffers, which would dominate a CrossValidate call
// on a small problem; freed buffers are therefore parked here (exact-size reuse, or best fit for
// the big work slab) and only returned to the driver by pareben_release_cache().
struct PoolEntry { void *ptr; size_t bytes; };
struct DevPool { std::vector<PoolEntry> free_list; size_t parked = 0; };
DevPool g_pool[64];
std::mutex g_cache_mu;
constexpr size_t POOL_MAX_ENTRIES = 512;

void *pool_take(int device, size_t bytes, bool best_fit, size_t *got)
{
    std::lock_guard<std::mutex> lk(g_cache_mu);
    DevPool &pl = g_pool[device & 63];
    int pick = -1;
    for (int i = 0; i < (int)pl.free_list.size(); i++) {
        const size_t b = pl.free_list[i].bytes;
        if (b == bytes) { pick = i; break; }
        if (best_fit && b > bytes && b <= bytes + bytes / 2 && (pick < 0 || b < pl.free_list[pick].bytes)) pick = i;
    }
    if (pick < 0) return nullptr;
    PoolEntry e = pl.free_list[pick];
    pl.free_list.erase(pl.free_list.begin() + pick);
    pl.parked -= e.bytes;
    if (got) *got = e.bytes;
    return e.ptr;
}

// Parked bytes per device are capped (PAREBEN_POOL_MAX_MB, default 8 GiB): a buffer that would push the pool past
// the cap goes straight back to the driver, so one huge problem does not starve the next one of a different size.
size_t pool_cap_bytes()
{
    static size_t cap = [] { const char *e = getenv("PAREBEN_POOL_MAX_MB"); return (size_t)(e ? atoll(e) : 8192) << 20; }();
    return cap;
}

void pool_give(int device, void *ptr, size_t bytes)
{
    if (!ptr) return;
    std::lock_guard<std::mutex> lk(g_cache_mu);
    DevPool &pl = g_pool[device & 63];
    if (pl.free_list.size() >= POOL_MAX_ENTRIES || pl.parked + bytes > pool_cap_bytes()) { cudaFree(ptr); return; }
    pl.free_list.push_back(PoolEntry{ptr, bytes});
    pl.parked += bytes;
}

// Return every parked buffer of `device` to the driver (the current device must be `device`).
size_t pool_release_device(int device)
{
    std::lock_guard<std::mutex> lk(g_cache_mu);
    DevPool &pl = g_pool[device & 63];
    const size_t freed = pl.parked;
    for (const PoolEntry &e : pl.free_list) cudaFree(e.ptr);
    pl.free_list.clear(); pl.parked = 0;
    return freed;
}

size_t pool_parked(int device)
{
    std::lock_guard<std::mutex> lk(g_cache_mu);
    return g_pool[device & 63].parked;
}

// cudaMalloc that, on failure, gives the pool's idle buffers back to the driver and tries once more.
cudaError_t malloc_retry(int device, void **p, size_t bytes)
{
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaErrorMemoryAllocation && pool_parked(device) > 0) {
        (void)cudaGetLastError();
        pool_release_device(device);
        e = cudaMalloc(p, bytes);
    }
    return e;
}

#define CU(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            char buf_[512];                                                                       \
            snprintf(buf_, sizeof buf_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            throw std::make_pair((int)(e_ == cudaErrorMemoryAllocation ? PAREBEN_ENOMEM : PAREBEN_ECUDA), std::string(buf_)); \
        }                                                                                         \
    } while (0)

// ---------------------------------------------------------------------------------------------
// layout kernels
// Xout[r][k] = Xcol[k*N + rows[r]]  (column-major in, row-major compacted out), 32x32 tiles
__global__ void gather_rows_kernel(const double *__restrict__ Xcol, int N, int K, const int *__restrict__ rows,
                                   int nrows, double *__restrict__ Xout)
{
    __shared__ double tile[32][33];
    const int r0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
    for (int kk = threadIdx.y; kk < 32; kk += blockDim.y) {
        const int r = r0 + threadIdx.x, k = k0 + kk;
        if (r < nrows && k < K) tile[kk][threadIdx.x] = Xcol[(size_t)k * N + rows[r]];
    }
    __syncthreads();
    for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
        const int r = r0 + rr, k = k0 + threadIdx.x;
        if (r < nrows && k < K) Xout[(size_t)r * K + k] = tile[threadIdx.x][rr];
    }
}

__global__ void gather_vec_kernel(const double *__restrict__ y, const int *__restrict__ rows, int nrows,
                                  double *__restrict__ out)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < nrows) out[r] = y[rows[r]];
}

__global__ void to_int8_kernel(const double *__restrict__ in, size_t n, int8_t *__restrict__ out)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (int8_t)in[i];
}

// Transposed, row-padded copy of a row-major matrix: out[k*ldt + r] = X[r*K + k] (zero for r >= nrows), as int8 or f64.
template <class T>
__global__ void transpose_pad_kernel(const double *__restrict__ X, int nrows, int K, int ldt, T *__restrict__ out)
{
    __shared__ double tile[32][33];
    const int r0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
    for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
        const int r = r0 + rr, k = k0 + threadIdx.x;
        tile[rr][threadIdx.x] = (r < nrows && k < K) ? X[(size_t)r * K + k] : 0.0;
    }
    __syncthreads();
    for (int kk = threadIdx.y; kk < 32; kk += blockDim.y) {
        const int r = r0 + threadIdx.x, k = k0 + kk;
        // rows of every group of 16 are stored permuted: physical position 4a + b holds row 4b + a (see mma_pass)
        const int rp = (r & ~15) | ((r & 3) << 2) | ((r >> 2) & 3);
        if (r < ldt && k < K) out[(size_t)k * ldt + rp] = (T)tile[threadIdx.x][kk];
    }
}

// scale[c] = sqrt(sum_h x_c[h]^2), 1 when the column is all zero (MainEff.c:87-99, NeFull2.c:100-135)
template <bool EPIS>
__global__ void scales_kernel(const double *__restrict__ X, int N, int K, int Kc, double *__restrict__ scale)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Kc) return;
    Cand<EPIS> cd(c, K);
    double z = 0;
    for (int h = 0; h < N; h++) { const double x = cd.at(X + (size_t)h * K); z = fma(x, x, z); }
    if (z == 0) z = 1;
    scale[c] = sqrt(z);
}

// lambda_max pieces (R/BuildGrid.R:5-32): max over candidates of x_c' r / ||x_c||
template <bool EPIS>
__global__ void lambda_max_kernel(const double *__restrict__ X, int N, int K, int c_begin, int c_end,
                                  const double *__restrict__ resp, double *__restrict__ block_max)
{
    __shared__ double red[32];
    const int c = c_begin + blockIdx.x * blockDim.x + threadIdx.x;
    double v = -1e300;
    if (c < c_end) {
        Cand<EPIS> cd(c, K);
        double z = 0, nn = 0;
        for (int h = 0; h < N; h++) { const double x = cd.at(X + (size_t)h * K); z = fma(x, resp[h], z); nn = fma(x, x, nn); }
        if (nn > 0) v = z / sqrt(nn);
    }
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = red[0];
        for (int w = 1; w < (int)(blockDim.x >> 5); w++) m = fmax(m, red[w]);
        block_max[blockIdx.x] = m;
    }
}

// FP64 FMA peak probe: 8 independent chains per thread.
__global__ void dfma_peak_kernel(double *out, int iters)
{
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-7;
    for (int i = 0; i < iters; i++) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// FP64 tensor-core probe: mma.sync.m8n8k4.f64 chains (DMMA), 4 independent accumulator pairs.
__global__ void dmma_peak_kernel(double *out, int iters)
{
    double a = 1.0 + threadIdx.x * 1e-9, b = 1.0000001;
    double c0 = 0, c1 = 0, d0 = 0, d1 = 0, e0 = 0, e1 = 0, f0 = 0, f1 = 0;
    for (int i = 0; i < iters; i++) {
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(e0), "+d"(e1) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(f0), "+d"(f1) : "d"(a), "d"(b));
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = c0 + c1 + d0 + d1 + e0 + e1 + f0 + f1;
}

Variant make_variant(int epis, int prior)
{   // SURVEY.md Appendix A, "variant constant table"
    Variant v;
    v.epis = epis; v.binomial = prior == PAREBEN_BINOMIAL;
    if (!v.binomial) {
        if (!epis) { v.n_add = 0.9;  v.ml_delta = 1e-3; v.reest_tol = 1e-3; v.init_alpha_max = 1e2; v.init_alpha_min = 0; }
        else       { v.n_add = 0.99; v.ml_delta = 1e-2; v.reest_tol = 0.1;  v.init_alpha_max = 1e3; v.init_alpha_min = 0; }
    } else {
        if (!epis) { v.n_add = 0.90; v.ml_delta = 1e-3; v.reest_tol = 1e-3; v.init_alpha_max = 1e3; v.init_alpha_min = 1e-3; }
        else       { v.n_add = 0.99; v.ml_delta = 1e-3; v.reest_tol = 1e-3; v.init_alpha_max = 1e3; v.init_alpha_min = 1e-3; }
    }
    return v;
}

}  // namespace

// single-locus statistic |ys' xs| / n of SL_filter.R:21,37 for candidates [c_begin, c_end): two passes over the rows
// (mean, then centred sums) like R's scale()
template <bool EPIS>
__global__ void sl_stat_kernel(const double *__restrict__ X, int N, int K, int c_begin, int c_end,
                               const double *__restrict__ ys, double *__restrict__ stat)
{
    const int c = c_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= c_end) return;
    Cand<EPIS> cd(c, K);
    double sx = 0;
    for (int h = 0; h < N; h++) sx += cd.at(X + (size_t)h * K);
    const double mean = sx / N;
    double ss = 0, sy = 0;
    for (int h = 0; h < N; h++) { const double d = cd.at(X + (size_t)h * K) - mean; ss = fma(d, d, ss); sy = fma(d, ys[h], sy); }
    const double sd = sqrt(ss / (N - 1));
    stat[c - c_begin] = fabs(sy / sd) / N;          // sd == 0 -> NaN or Inf*0: never passes the host's `> tau` test
}

// ---------------------------------------------------------------------------------------------
struct pareben_problem {
    int device = 0;
    int n = 0, k = 0, kc = 0, n_folds = 0, epis = 0, prior = 0, cap = 0, nmax = 0, min_ntr = 0;
    int sm_count = 0;
    std::vector<PoolEntry> allocs;       // every device buffer of this problem (returned to the pool on destroy)
    FoldData *d_folds = nullptr;
    std::vector<FoldData> h_folds;
    double *d_Xcol = nullptr, *d_y = nullptr;     // full data, column-major (kept for lambda_max)
    char *d_slabs = nullptr; size_t slab_stride = 0, slab_total = 0; int n_slabs = 0;
    double *d_flops = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int threads = 256;                   // threads per block actually launched
    double last_flops = 0, last_ms = 0; int last_launches = 0;
    bool streaming = false;              // fits run through the streaming kernels (no per-candidate arrays anywhere)
    // Gram organisation (Gaussian, cached kernels): FoldData::C per fold, built on first use and kept with the problem
    int gram_state = 0;                  // 0 = undecided, 1 = in use, -1 = refused (memory or too little work)
    double gram_ms = 0; int gram_launches = 0;      // time / launches spent building C in the last run_fits call
    double last_avoided = 0;             // model flops of the last call that the Gram organisation did not execute
    long long grid_fits_hint = 0;        // fits of the WHOLE grid a sharded call belongs to (0 = unknown): the work test must not
                                         // depend on how many ways the grid is split, or 1- and 8-GPU tables could differ in rounding
    double last_scan_ms = 0, last_scan_flops = 0; int last_scan_launches = 0, last_rounds = 0;

    template <class T> T *dalloc(size_t n)
    {
        const size_t bytes = (std::max<size_t>(n, 1) * sizeof(T) + 255) & ~(size_t)255;
        void *p = pool_take(device, bytes, false, nullptr);
        if (!p) CU(malloc_retry(device, &p, bytes));
        allocs.push_back(PoolEntry{p, bytes});
        return static_cast<T *>(p);
    }
    ~pareben_problem()
    {
        cudaSetDevice(device);
        pool_give(device, d_slabs, slab_total);
        for (const PoolEntry &e : allocs) pool_give(device, e.ptr, e.bytes);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
    }
};

static int reference_basis_max(int n_train, int k, int kc, int epis, int prior)
{
    if (prior == PAREBEN_BINOMIAL) return epis ? 2 * k : k;                        // bMax (EBelasticNet.Binomial.R:8,30)
    if (!epis) { int b = (int)(1e7 / kc); return b > kc ? kc : b; }                // MainEff.c:68-69
    return n_train > k ? 2 * k : (n_train < 200 ? 4 * k : k);                      // NeFull2.c:67-80
}

// The per-block work slabs are only needed by the fit kernel: they are sized and allocated at the first
// pareben_run_fits / pareben_fit of a problem (lambda_max and the single-locus prefilter never touch them, and an
// Epis problem's candidate cache can be far larger than those two need).  Throws like the CU() macro.
static void ensure_slabs(pareben_problem *p)
{
    if (p->d_slabs) return;
    // basis cap: the reference's basisMax, bounded so that the per-block slab stays reasonable.
    int cap = reference_basis_max(p->min_ntr, p->k, p->kc, p->epis, p->prior);
    const char *env_cap = getenv("PAREBEN_BASIS_CAP");
    int hard = env_cap ? atoi(env_cap) : 1024;
    if (hard < 2) hard = 2;
    if (p->prior == PAREBEN_BINOMIAL) cap += 1;       // slot 0 is the intercept
    p->cap = std::min(cap, hard);
    if (p->cap < 2) p->cap = 2;

    // persistent grid: blocks per SM limited by memory for slabs
    p->slab_stride = slab_bytes(p->cap, p->nmax, p->kc);
    // resident blocks per SM of the kernel variant this problem will launch (asked once per variant:
    // the occupancy query, like cudaMemGetInfo below, costs up to tens of milliseconds)
    int per_sm = 1;
    {
        // Block size: measured on B200 (config 2 / bundled Gaussian): 256 threads x 2 blocks per SM beats
        // 128 x 4 (-5 % / -43 %) and 64 x 8 (-40 % / -70 %) (measured with an earlier build that had a run-time block size).
        p->threads = FIT_THREADS_HOST;     // gram_tiled() maps 16 x 16 register blocks onto exactly 256 threads
        static int occ_cache[4] = {0, 0, 0, 0};
        int &occ = occ_cache[(p->prior == PAREBEN_BINOMIAL ? 2 : 0) + (p->epis ? 1 : 0)];
        if (!occ) {
            cudaError_t e;
            if (p->prior == PAREBEN_GAUSSIAN) e = p->epis ? occupancy_ge(&occ, p->threads) : occupancy_gm(&occ, p->threads);
            else e = p->epis ? occupancy_be(&occ, p->threads) : occupancy_bm(&occ, p->threads);
            CU(e);
        }
        per_sm = std::max(1, occ);
    }
    const char *env_bps = getenv("PAREBEN_BLOCKS_PER_SM");
    if (env_bps) per_sm = std::max(1, std::min(per_sm, atoi(env_bps)));
    // First try the pool with the full-occupancy slab (the steady state of repeated CrossValidate calls);
    // only a miss pays for cudaMemGetInfo and cudaMalloc.
    p->n_slabs = per_sm * p->sm_count;
    p->slab_total = (size_t)p->n_slabs * p->slab_stride;
    {
        size_t got = 0;
        void *q = pool_take(p->device, p->slab_total, true, &got);
        if (q) { p->d_slabs = (char *)q; p->slab_total = got; }
    }
    if (!p->d_slabs) {
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        // idle pool buffers count as free: when the full-occupancy slab does not fit beside them they are released first
        if ((size_t)per_sm * p->sm_count * p->slab_stride > free_b / 2 && pool_parked(p->device) > 0) {
            pool_release_device(p->device);
            CU(cudaMemGetInfo(&free_b, &total_b));
        }
        while (per_sm > 1 && (size_t)per_sm * p->sm_count * p->slab_stride > free_b / 2) per_sm--;
        p->n_slabs = per_sm * p->sm_count;
        while (p->n_slabs > 1 && (size_t)p->n_slabs * p->slab_stride > free_b - (free_b >> 3)) p->n_slabs /= 2;   // huge problems: fewer blocks
        p->slab_total = (size_t)p->n_slabs * p->slab_stride;
        if (p->slab_total > free_b - (free_b >> 3))
            throw std::make_pair((int)PAREBEN_ENOMEM, std::string("per-block work slabs do not fit in device memory; lower PAREBEN_BASIS_CAP"));
        void *q = nullptr;
        CU(malloc_retry(p->device, &q, p->slab_total));
        p->d_slabs = (char *)q;
    }
}

// Gram organisation of the Gaussian fits (fold_gram_kernel, fit_kernel.cuh).  C costs 8 Kc^2 bytes and 2 N Kc^2 flops per
// fold; a fit then never contracts the training matrix against a basis column again.  Worth it when the call has enough
// work to amortise it (a fit contracts ~ (outer iterations) x (active set) + (adds) columns, hundreds for a grid point)
// and the matrices fit beside the work slabs.  PAREBEN_GRAM=0 / 1 overrides the work test (never the memory test).
// Once built, C stays with the problem handle: BuildGrid -> cv_grid -> LocalSearch share it.  Throws like CU().
static void ensure_gram(pareben_problem *p, int n_fits, const int *fold)
{
    p->gram_ms = 0; p->gram_launches = 0;
    if (p->prior != PAREBEN_GAUSSIAN || p->streaming) return;
    const char *env = getenv("PAREBEN_GRAM");
    const int forced = env ? atoi(env) : -1;
    if (forced == 0) {
        if (p->gram_state == 1) {       // drop the pointers (the buffers stay in p->allocs until the problem is destroyed)
            for (FoldData &F : p->h_folds) F.C = nullptr;
            CU(cudaMemcpyAsync(p->d_folds, p->h_folds.data(), sizeof(FoldData) * p->h_folds.size(), cudaMemcpyHostToDevice, p->stream));
            p->gram_state = 0;
        }
        return;
    }
    if (p->gram_state < 0) return;
    std::vector<int> need;              // folds of this call whose C does not exist yet
    {
        std::vector<char> seen(p->h_folds.size(), 0);
        for (int i = 0; i < n_fits; i++) if (!seen[fold[i]]) { seen[fold[i]] = 1; if (!p->h_folds[fold[i]].C) need.push_back(fold[i]); }
    }
    if (need.empty()) return;
    const size_t bytes_per_fold = ((size_t)p->kc * p->kc * sizeof(double) + 255) & ~(size_t)255;
    if (p->gram_state == 0) {
        int n_distinct = 0;
        { std::vector<char> seen(p->h_folds.size(), 0); for (int i = 0; i < n_fits; i++) if (!seen[fold[i]]) { seen[fold[i]] = 1; n_distinct++; } }
        const double work_fits = (double)std::max<long long>(n_fits, p->grid_fits_hint);
        if (forced != 1 && (double)n_distinct * p->kc > 512.0 * work_fits) return;   // too little work in this call: decide again next time
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        free_b += pool_parked(p->device);
        const size_t all_folds = bytes_per_fold * (size_t)std::max(1, p->n_folds);
        if (all_folds > free_b / 2) { p->gram_state = -1; return; }
        p->gram_state = 1;
    }
    for (int f : need) p->h_folds[f].C = p->dalloc<double>(bytes_per_fold / sizeof(double));
    int *d_list = p->dalloc<int>(need.size() + 1);           // fold list + the work counter (small, kept with the problem)
    std::vector<int> h_list(need);
    h_list.push_back(0);
    CU(cudaMemcpyAsync(d_list, h_list.data(), sizeof(int) * h_list.size(), cudaMemcpyHostToDevice, p->stream));
    CU(cudaMemcpyAsync(p->d_folds, p->h_folds.data(), sizeof(FoldData) * p->h_folds.size(), cudaMemcpyHostToDevice, p->stream));
    Problem P;
    P.N = p->n; P.K = p->k; P.Kc = p->kc; P.n_folds = p->n_folds; P.epis = p->epis; P.prior = p->prior;
    P.cap = p->cap; P.nmax = p->nmax; P.folds = p->d_folds;
    const int chunks = (p->kc + 31) / 32;
    const int grid = (int)std::min<long long>(p->n_slabs, (long long)chunks * (long long)need.size());
    CU(cudaEventRecord(p->ev0, p->stream));
    CU((p->epis ? launch_gram_ge : launch_gram_gm)(grid, p->threads, p->stream, P, d_list, (int)need.size(), p->d_slabs, p->slab_stride,
                                                   d_list + need.size()));
    CU(cudaEventRecord(p->ev1, p->stream));
    CU(cudaStreamSynchronize(p->stream));       // h_list goes out of scope; and the build time is reported
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
    p->gram_ms = ms; p->gram_launches = 1;
}

extern "C" int pareben_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}
extern "C" const char *pareben_last_error(void) { return g_err.c_str(); }
extern "C" int pareben_version(void) { return PAREBEN_VERSION; }

extern "C" int pareben_problem_create(pareben_problem **out, int device, const double *basis, int n, int k,
                                      const double *target, const int *fold_id, int n_folds, int epis, int prior)
{
    if (!out || !basis || !target || n < 2 || k < 1 || n_folds < 0 || (n_folds > 0 && !fold_id))
        return fail(PAREBEN_EINVAL, "pareben_problem_create: bad argument");
    if (prior != PAREBEN_GAUSSIAN && prior != PAREBEN_BINOMIAL) return fail(PAREBEN_EINVAL, "prior must be 0 or 1");
    if (epis && (long long)k * (k + 1) / 2 > 0x7fffffffLL) return fail(PAREBEN_EINVAL, "k(k+1)/2 exceeds int32");
    if (pareben_device_count() <= device || device < 0) return fail(PAREBEN_ENODEVICE, "no usable CUDA device");
    pareben_problem *p = new pareben_problem();
    try {
        p->device = device;
        CU(cudaSetDevice(device));
        {   // cudaGetDeviceProperties costs milliseconds: ask once per device
            static int sm_cache[64] = {0};
            if (!sm_cache[device & 63]) CU(cudaDeviceGetAttribute(&sm_cache[device & 63], cudaDevAttrMultiProcessorCount, device));
            p->sm_count = sm_cache[device & 63];
        }
        const bool timing = getenv("PAREBEN_TIMING") != nullptr;
        auto tc0 = std::chrono::steady_clock::now();
        auto lap = [&](const char *what) {
            if (!timing) return;
            auto t = std::chrono::steady_clock::now();
            fprintf(stderr, "[pareben]   create: %-28s %.2f ms\n", what, std::chrono::duration<double, std::milli>(t - tc0).count());
            tc0 = t;
        };
        p->n = n; p->k = k; p->epis = epis; p->prior = prior; p->n_folds = n_folds;
        p->kc = epis ? (int)((long long)k * (k + 1) / 2) : k;
        p->streaming = want_streaming(p->kc, prior);
        if (p->streaming && n_folds + 1 > STREAM_MAX_FOLDS) throw std::make_pair((int)PAREBEN_EINVAL, std::string("streaming mode supports at most 255 folds"));
        CU(cudaStreamCreate(&p->stream));
        CU(cudaEventCreate(&p->ev0)); CU(cudaEventCreate(&p->ev1));

        p->d_Xcol = p->dalloc<double>((size_t)n * k);
        p->d_y = p->dalloc<double>(n);
        CU(cudaMemcpyAsync(p->d_Xcol, basis, sizeof(double) * n * k, cudaMemcpyHostToDevice, p->stream));
        CU(cudaMemcpyAsync(p->d_y, target, sizeof(double) * n, cudaMemcpyHostToDevice, p->stream));

        // Genotype-coded designs (every entry an integer in [-127, 127], e.g. {-1, 0, 1}) also get an
        // int8 copy of the training matrices: the score contraction reads 1 byte instead of 8 per
        // element and widens in registers (exact).
        bool small_int = true;
        for (size_t i = 0, e = (size_t)n * k; small_int && i < e; i++) {
            const double v = basis[i];
            if (!(v >= -127.0 && v <= 127.0) || v != (double)(int)v) small_int = false;
        }
        lap("stream/events/h2d enqueue/scan");
        // row lists per fold: index 0 = all rows (only materialised when n_folds == 0)
        const int nf = n_folds;
        p->h_folds.assign(nf + 1, FoldData{});
        int min_ntr = n;
        for (int f = (nf == 0 ? 0 : 1); f <= nf; f++) {
            std::vector<int> tr, te;
            for (int r = 0; r < n; r++) {
                if (f == 0) tr.push_back(r);
                else {
                    if (fold_id[r] < 1 || fold_id[r] > nf) throw std::make_pair((int)PAREBEN_EINVAL, std::string("fold_id out of range"));
                    (fold_id[r] != f ? tr : te).push_back(r);
                }
            }
            if (tr.size() < 2) throw std::make_pair((int)PAREBEN_EINVAL, std::string("a fold leaves fewer than 2 training rows"));
            FoldData &F = p->h_folds[f];
            F.ntr = (int)tr.size(); F.nte = (int)te.size();
            p->nmax = std::max(p->nmax, F.ntr);
            min_ntr = std::min(min_ntr, F.ntr);
            int *d_rows = p->dalloc<int>(tr.size() + te.size());
            CU(cudaMemcpyAsync(d_rows, tr.data(), sizeof(int) * tr.size(), cudaMemcpyHostToDevice, p->stream));
            if (!te.empty())
                CU(cudaMemcpyAsync(d_rows + tr.size(), te.data(), sizeof(int) * te.size(), cudaMemcpyHostToDevice, p->stream));
            CU(cudaStreamSynchronize(p->stream));      // tr/te go out of scope
            double *Xtr = p->dalloc<double>((size_t)F.ntr * k), *ytr = p->dalloc<double>(F.ntr);
            double *Xte = p->dalloc<double>((size_t)F.nte * k), *yte = p->dalloc<double>(F.nte);
            double *scale = p->streaming ? nullptr : p->dalloc<double>(p->kc);     // streaming: norms are computed on the fly
            dim3 blk(32, 8);
            gather_rows_kernel<<<dim3((F.ntr + 31) / 32, (k + 31) / 32), blk, 0, p->stream>>>(p->d_Xcol, n, k, d_rows, F.ntr, Xtr);
            gather_vec_kernel<<<(F.ntr + 255) / 256, 256, 0, p->stream>>>(p->d_y, d_rows, F.ntr, ytr);
            if (F.nte > 0) {
                gather_rows_kernel<<<dim3((F.nte + 31) / 32, (k + 31) / 32), blk, 0, p->stream>>>(p->d_Xcol, n, k, d_rows + F.ntr, F.nte, Xte);
                gather_vec_kernel<<<(F.nte + 255) / 256, 256, 0, p->stream>>>(p->d_y, d_rows + F.ntr, F.nte, yte);
            }
            if (scale) {
                if (epis) scales_kernel<true><<<(p->kc + 255) / 256, 256, 0, p->stream>>>(Xtr, F.ntr, k, p->kc, scale);
                else scales_kernel<false><<<(p->kc + 255) / 256, 256, 0, p->stream>>>(Xtr, F.ntr, k, p->kc, scale);
            }
            F.Xtr = Xtr; F.ytr = ytr; F.Xte = Xte; F.yte = yte; F.scale = scale; F.Xtr8 = nullptr;
            F.XT8 = nullptr; F.XTd = nullptr; F.C = nullptr;
            F.ldt = (F.ntr + 63) & ~63;      // whole stages of the contraction (KT = 64 rows)
            {
                const dim3 tg((F.ldt + 31) / 32, (k + 31) / 32);
                if (small_int) {
                    int8_t *t8 = p->dalloc<int8_t>((size_t)F.ldt * k + 16);
                    transpose_pad_kernel<int8_t><<<tg, blk, 0, p->stream>>>(Xtr, F.ntr, k, F.ldt, t8);
                    F.XT8 = t8;
                } else {
                    double *td = p->dalloc<double>((size_t)F.ldt * k + 4);
                    transpose_pad_kernel<double><<<tg, blk, 0, p->stream>>>(Xtr, F.ntr, k, F.ldt, td);
                    F.XTd = td;
                }
            }
            if (small_int) {
                int8_t *x8 = p->dalloc<int8_t>((size_t)F.ntr * k + 16);
                to_int8_kernel<<<std::min<size_t>(1024, ((size_t)F.ntr * k + 255) / 256), 256, 0, p->stream>>>(Xtr, (size_t)F.ntr * k, x8);
                F.Xtr8 = x8;
            }
        }
        CU(cudaGetLastError());
        lap("per-fold layout (enqueue)");
        p->d_folds = p->dalloc<FoldData>(nf + 1);
        CU(cudaMemcpyAsync(p->d_folds, p->h_folds.data(), sizeof(FoldData) * (nf + 1), cudaMemcpyHostToDevice, p->stream));

        p->min_ntr = min_ntr;
        p->d_flops = p->dalloc<double>(2);
        CU(cudaStreamSynchronize(p->stream));
        lap("final sync");
    } catch (std::pair<int, std::string> &e) {
        delete p;
        return fail(e.first, e.second);
    }
    *out = p;
    return PAREBEN_OK;
}

extern "C" void pareben_problem_destroy(pareben_problem *p) { delete p; }

extern "C" void pareben_release_cache(void)
{
    int cur = 0;
    cudaGetDevice(&cur);
    for (int d = 0; d < 64; d++) {
        if (pool_parked(d) == 0) continue;
        cudaSetDevice(d);
        pool_release_device(d);
    }
    cudaSetDevice(cur);
}

namespace {

struct DumpBuffers { int *m = nullptr, *used = nullptr; double *beta = nullptr, *var = nullptr, *scalars = nullptr; };

// Streaming mode (stream.cuh): every fit keeps only its active set; all fits advance in lock-step rounds of
//   stream_advance_kernel (one block per fit)  ->  stream_scan_kernel (one dense contraction per fold for all waiting fits)
// until no fit is waiting for a scan.  One 4-byte-per-fold read-back per round tells the host when to stop.
int run_fits_streaming(pareben_problem *p, int n_fits, const int *fold, const double *alpha, const double *lambda,
                       double *fold_err, int *status, int *n_selected, int *n_iter, DumpBuffers *dump)
{
    std::vector<std::pair<void *, size_t>> scratch;
    cudaEvent_t es0 = nullptr, es1 = nullptr;
    try {
        CU(cudaSetDevice(p->device));
        const int nf1 = p->n_folds + 1;
        auto tmp_alloc = [&](size_t bytes) {
            bytes = (std::max<size_t>(bytes, 8) + 255) & ~(size_t)255;
            void *q = pool_take(p->device, bytes, false, nullptr);
            if (!q) CU(malloc_retry(p->device, &q, bytes));
            scratch.emplace_back(q, bytes); return q; };
        // basis cap: the reference's basisMax, bounded by PAREBEN_BASIS_CAP and by what n_fits active sets may occupy
        int cap = reference_basis_max(p->min_ntr, p->k, p->kc, p->epis, p->prior);
        const char *env_cap = getenv("PAREBEN_BASIS_CAP");
        cap = std::max(2, std::min(cap, env_cap ? atoi(env_cap) : 1024));
        const int list_cap = 4096;
        const int LD = phi_ld(p->nmax);
        auto fit_doubles = [&](int c) { return (size_t)4 * c * c + (size_t)LD * c + (size_t)12 * (c + 1) + (size_t)4 * p->nmax + (size_t)2 * list_cap + 16; };
        auto fit_ints = [&](int c) { return (size_t)2 * c + (size_t)4 * (c + list_cap) + list_cap + 16; };
        auto fit_bytes = [&](int c) { return ((fit_doubles(c) * 8 + fit_ints(c) * 4) + 255) & ~(size_t)255; };
        {
            size_t free_b = 0, total_b = 0;
            CU(cudaMemGetInfo(&free_b, &total_b));
            free_b += pool_parked(p->device);
            while (cap > 16 && fit_bytes(cap) * (size_t)n_fits > free_b / 2) cap = cap * 3 / 4;
        }
        p->cap = cap;
        const size_t stride = fit_bytes(cap);
        char *d_state = (char *)tmp_alloc(stride * (size_t)n_fits);
        StreamFit *d_fits = (StreamFit *)tmp_alloc(sizeof(StreamFit) * (size_t)n_fits);
        std::vector<StreamFit> h_fits(n_fits);
        std::vector<int> per_fold(nf1, 0);
        for (int i = 0; i < n_fits; i++) {
            if (fold[i] < 0 || fold[i] > p->n_folds || (p->n_folds > 0 && fold[i] == 0) || !p->h_folds[fold[i]].Xtr)
                return fail(PAREBEN_EINVAL, "pareben_run_fits: fold label not available in this problem");
            per_fold[fold[i]]++;
            StreamFit f;
            memset(&f, 0, sizeof f);
            f.fold = fold[i]; f.out_index = i; f.lambda = lambda[i]; f.alpha_en = alpha[i]; f.phase = SP_START;
            double *d = reinterpret_cast<double *>(d_state + stride * (size_t)i);
            const size_t cc = (size_t)cap * cap;
            f.sigma = d; d += cc; f.sigma_new = d; d += cc; f.H = d; d += cc; f.ptp = d; d += cc;
            f.phi = d; d += (size_t)LD * cap;
            f.mu = d; d += cap + 1; f.alpha = d; d += cap + 1; f.gamma = d; d += cap + 1; f.tmp = d; d += cap + 1; f.u = d; d += cap + 1;
            f.colk = d; d += 2 * (cap + 1); f.ascale = d; d += cap + 1; f.s_in = d; d += cap + 1; f.q_in = d; d += cap + 1;
            f.dml_in = d; d += cap + 1; f.aroot_in = d; d += cap + 1;
            f.t = d; d += p->nmax; f.e = d; d += p->nmax; f.d = d; d += p->nmax; f.phinew = d; d += p->nmax;
            f.list_dml = d; d += list_cap; f.list_aroot = d; d += list_cap;
            int *ip = reinterpret_cast<int *>(d);
            f.used = ip; ip += cap; f.act_in = ip; ip += cap;
            f.blk_c = ip; ip += 2 * (cap + list_cap); f.blk_src = ip; ip += 2 * (cap + list_cap);
            f.list_c = ip; ip += list_cap;
            h_fits[i] = f;
        }
        CU(cudaMemcpyAsync(d_fits, h_fits.data(), sizeof(StreamFit) * (size_t)n_fits, cudaMemcpyHostToDevice, p->stream));
        // per-(fold, class) round buffers: index STREAM_CLASSES * f + cls (stream.cuh)
        const int nvf = STREAM_CLASSES * nf1;
        std::vector<StreamFold> h_sf(nvf);
        for (int vf = 0; vf < nvf; vf++) {
            StreamFold sf; memset(&sf, 0, sizeof sf);
            const int f = vf / STREAM_CLASSES, cls = vf % STREAM_CLASSES;
            if (per_fold[f] > 0) {
                const int per = class_fits_per_tile(cls);
                const int n_rt = (per_fold[f] + per - 1) / per;
                sf.max_slots = n_rt * SN;
                sf.E = (double *)tmp_alloc(sizeof(double) * e_tile_doubles(p->h_folds[f].ldt) * n_rt);
                CU(cudaMemsetAsync(sf.E, 0, sizeof(double) * e_tile_doubles(p->h_folds[f].ldt) * n_rt, p->stream));
                sf.par = (ScanSlot *)tmp_alloc(sizeof(ScanSlot) * sf.max_slots);
                sf.slot_fit = (int *)tmp_alloc(sizeof(int) * sf.max_slots);
            }
            h_sf[vf] = sf;
        }
        StreamFold *d_sf = (StreamFold *)tmp_alloc(sizeof(StreamFold) * nvf);
        CU(cudaMemcpyAsync(d_sf, h_sf.data(), sizeof(StreamFold) * nvf, cudaMemcpyHostToDevice, p->stream));
        int *d_nslots = (int *)tmp_alloc(sizeof(int) * nvf);
        const int scan_grid = p->sm_count;
        double *d_wscratch = (double *)tmp_alloc(sizeof(double) * (size_t)scan_grid * SCAN_WARPS * cap);
        double *d_err = (double *)tmp_alloc(sizeof(double) * n_fits);
        int *d_ints = (int *)tmp_alloc(sizeof(int) * 3 * n_fits);
        CU(cudaMemsetAsync(p->d_flops, 0, 2 * sizeof(double), p->stream));
        CU(cudaMemsetAsync(d_nslots, 0, sizeof(int) * nvf, p->stream));
        StreamShared sh;
        sh.folds = d_sf; sh.n_slots = d_nslots; sh.list_cap = list_cap; sh.warp_scratch = d_wscratch; sh.flops = p->d_flops;
        FitOutputs out;
        out.fold_err = d_err; out.status = d_ints; out.n_selected = d_ints + n_fits; out.n_iter = d_ints + 2 * n_fits;
        out.m_out = nullptr; out.used_out = nullptr; out.beta_out = nullptr; out.var_out = nullptr; out.scalars_out = nullptr;
        out.flops = p->d_flops;
        if (dump) {
            dump->m = (int *)tmp_alloc(sizeof(int) * (1 + cap));
            dump->used = dump->m + 1;
            dump->beta = (double *)tmp_alloc(sizeof(double) * (2 * cap + 4));
            dump->var = dump->beta + cap; dump->scalars = dump->var + cap;
            out.m_out = dump->m; out.used_out = dump->used; out.beta_out = dump->beta; out.var_out = dump->var; out.scalars_out = dump->scalars;
        }
        Problem P;
        P.N = p->n; P.K = p->k; P.Kc = p->kc; P.n_folds = p->n_folds; P.epis = p->epis; P.prior = p->prior;
        P.cap = cap; P.nmax = p->nmax; P.folds = p->d_folds;
        const Variant v = make_variant(p->epis, p->prior);
        auto advance = [&] { CU((p->epis ? launch_stream_advance_ge : launch_stream_advance_gm)(n_fits, p->stream, P, v, d_fits, sh, out)); };
        auto scan = [&] { CU((p->epis ? launch_stream_scan_ge : launch_stream_scan_gm)(scan_grid, p->stream, P, d_fits, sh)); };
        CU(cudaEventCreate(&es0)); CU(cudaEventCreate(&es1));
        std::vector<int> h_nslots(nvf);
        double scan_ms = 0, scan_flops = 0;
        int rounds = 0, scans = 0;
        const bool timing = getenv("PAREBEN_TIMING") != nullptr;
        CU(cudaEventRecord(p->ev0, p->stream));
        advance();
        for (;;) {
            CU(cudaMemcpyAsync(h_nslots.data(), d_nslots, sizeof(int) * nvf, cudaMemcpyDeviceToHost, p->stream));
            CU(cudaStreamSynchronize(p->stream));
            float last_scan_ms = 0;
            if (scans > 0) { CU(cudaEventElapsedTime(&last_scan_ms, es0, es1)); scan_ms += last_scan_ms; }
            long long waiting = 0;
            double fl = 0;
            long long waiting_b = 0;
            for (int vf = 0; vf < nvf; vf++) { waiting += h_nslots[vf]; if (vf % STREAM_CLASSES == 0) waiting_b += h_nslots[vf]; fl += 2.0 * p->h_folds[vf / STREAM_CLASSES].ntr * (double)p->kc * h_nslots[vf]; }
            if (timing) fprintf(stderr, "[pareben] stream round %d: %lld fits waiting (%lld not on the initial basis), last scan %.1f ms\n", rounds, waiting, waiting_b, last_scan_ms);
            if (waiting == 0) break;
            scan_flops += fl;
            CU(cudaEventRecord(es0, p->stream));
            scan();
            CU(cudaEventRecord(es1, p->stream));
            scans++;
            CU(cudaMemsetAsync(d_nslots, 0, sizeof(int) * nvf, p->stream));
            advance();
            rounds++;
        }
        CU(cudaEventRecord(p->ev1, p->stream));
        std::vector<int> h_ints(3 * (size_t)n_fits);
        std::vector<double> h_err(n_fits);
        CU(cudaMemcpyAsync(h_err.data(), d_err, sizeof(double) * n_fits, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaMemcpyAsync(h_ints.data(), d_ints, sizeof(int) * 3 * n_fits, cudaMemcpyDeviceToHost, p->stream));
        double h_flops = 0;
        CU(cudaMemcpyAsync(&h_flops, p->d_flops, sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
        p->last_ms = ms; p->last_flops = h_flops; p->last_launches = 1 + scans + rounds;
        p->last_scan_ms = scan_ms; p->last_scan_flops = scan_flops; p->last_scan_launches = scans; p->last_rounds = rounds;
        for (int i = 0; i < n_fits; i++) {
            if (fold_err) fold_err[i] = h_err[i];
            if (status) status[i] = h_ints[i];
            if (n_selected) n_selected[i] = h_ints[n_fits + i];
            if (n_iter) n_iter[i] = h_ints[2 * (size_t)n_fits + i];
        }
        if (dump) {
            int *hm = (int *)malloc(sizeof(int) * (1 + cap));
            double *hb = (double *)malloc(sizeof(double) * (2 * cap + 4));
            CU(cudaMemcpy(hm, dump->m, sizeof(int) * (1 + cap), cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(hb, dump->beta, sizeof(double) * (2 * cap + 4), cudaMemcpyDeviceToHost));
            dump->m = hm; dump->used = hm + 1; dump->beta = hb; dump->var = hb + cap; dump->scalars = hb + 2 * cap;
        }
        cudaEventDestroy(es0); cudaEventDestroy(es1);
        for (auto &q : scratch) pool_give(p->device, q.first, q.second);
    } catch (std::pair<int, std::string> &e) {
        if (es0) cudaEventDestroy(es0);
        if (es1) cudaEventDestroy(es1);
        for (auto &q : scratch) pool_give(p->device, q.first, q.second);
        return fail(e.first, e.second);
    }
    return PAREBEN_OK;
}

int run_fits_impl(pareben_problem *p, int n_fits, const int *fold, const double *alpha, const double *lambda,
                  double *fold_err, int *status, int *n_selected, int *n_iter, DumpBuffers *dump)
{
    if (!p || n_fits < 0 || (n_fits > 0 && (!fold || !alpha || !lambda))) return fail(PAREBEN_EINVAL, "pareben_run_fits: bad argument");
    if (n_fits == 0) return PAREBEN_OK;
    if (p->streaming) return run_fits_streaming(p, n_fits, fold, alpha, lambda, fold_err, status, n_selected, n_iter, dump);
    void *scratch[8] = {nullptr};
    size_t scratch_bytes[8] = {0};
    int ns = 0;
    try {
        CU(cudaSetDevice(p->device));
        ensure_slabs(p);
        for (int i = 0; i < n_fits; i++)
            if (fold[i] < 0 || fold[i] > p->n_folds || (p->n_folds > 0 && fold[i] == 0) || !p->h_folds[fold[i]].Xtr)
                return fail(PAREBEN_EINVAL, "pareben_run_fits: fold label not available in this problem");
        ensure_gram(p, n_fits, fold);
        std::vector<FitTask> tasks(n_fits);
        // groups: fits that share (alpha, lambda) -- one row of the reference's ParameterGrid -- differ only in the fold
        // and cost about the same; the device scheduler prices a group by its first finished fit (fit_kernel.cuh)
        std::map<std::pair<double, double>, int> group_of;
        for (int i = 0; i < n_fits; i++) {
            if (fold[i] < 0 || fold[i] > p->n_folds || (p->n_folds > 0 && fold[i] == 0) || !p->h_folds[fold[i]].Xtr)
                return fail(PAREBEN_EINVAL, "pareben_run_fits: fold label not available in this problem");
            const auto key = std::make_pair(alpha[i], lambda[i]);
            auto it = group_of.find(key);
            if (it == group_of.end()) it = group_of.emplace(key, (int)group_of.size()).first;
            tasks[i] = FitTask{fold[i], alpha[i], lambda[i], i, it->second};
        }
        const int n_groups = (int)group_of.size();
        // host order: rising lambda (larger active sets first) is the prior; one pilot per group goes to the front
        std::stable_sort(tasks.begin(), tasks.end(), [](const FitTask &a, const FitTask &b) { return a.lambda < b.lambda; });
        {
            std::vector<char> seen(n_groups, 0);
            std::vector<FitTask> pilots, rest;
            pilots.reserve(n_groups); rest.reserve(n_fits);
            for (const FitTask &t : tasks) { if (!seen[t.group]) { seen[t.group] = 1; pilots.push_back(t); } else rest.push_back(t); }
            tasks = pilots;
            tasks.insert(tasks.end(), rest.begin(), rest.end());
        }
        auto tmp_alloc = [&](size_t bytes) {
            bytes = (std::max<size_t>(bytes, 8) + 255) & ~(size_t)255;
            void *q = pool_take(p->device, bytes, false, nullptr);
            if (!q) CU(malloc_retry(p->device, &q, bytes));
            scratch_bytes[ns] = bytes; scratch[ns++] = q; return q; };
        FitTask *d_tasks = (FitTask *)tmp_alloc(sizeof(FitTask) * n_fits);
        double *d_err = (double *)tmp_alloc(sizeof(double) * n_fits);
        int *d_ints = (int *)tmp_alloc(sizeof(int) * 3 * n_fits);
        const size_t sched_bytes = sizeof(unsigned long long) * 2 * n_groups + sizeof(int) * n_fits;
        unsigned long long *d_sched = (unsigned long long *)tmp_alloc(sched_bytes);
        Sched sched;
        sched.t_start = d_sched; sched.cost = d_sched + n_groups; sched.taken = reinterpret_cast<int *>(d_sched + 2 * (size_t)n_groups);
        CU(cudaMemcpyAsync(d_tasks, tasks.data(), sizeof(FitTask) * n_fits, cudaMemcpyHostToDevice, p->stream));
        CU(cudaMemsetAsync(d_sched, 0, sched_bytes, p->stream));
        CU(cudaMemsetAsync(p->d_flops, 0, 2 * sizeof(double), p->stream));
        FitOutputs out;
        out.fold_err = d_err; out.status = d_ints; out.n_selected = d_ints + n_fits; out.n_iter = d_ints + 2 * n_fits;
        out.m_out = nullptr; out.used_out = nullptr; out.beta_out = nullptr; out.var_out = nullptr; out.scalars_out = nullptr;
        out.flops = p->d_flops;
        if (dump) {
            dump->m = (int *)tmp_alloc(sizeof(int) * (1 + p->cap));
            dump->used = dump->m + 1;
            dump->beta = (double *)tmp_alloc(sizeof(double) * (2 * p->cap + 4));
            dump->var = dump->beta + p->cap; dump->scalars = dump->var + p->cap;
            out.m_out = dump->m; out.used_out = dump->used; out.beta_out = dump->beta; out.var_out = dump->var; out.scalars_out = dump->scalars;
        }
        Problem P;
        P.N = p->n; P.K = p->k; P.Kc = p->kc; P.n_folds = p->n_folds; P.epis = p->epis; P.prior = p->prior;
        P.cap = p->cap; P.nmax = p->nmax; P.folds = p->d_folds;
        const Variant v = make_variant(p->epis, p->prior);
        int grid = std::min(p->n_slabs, n_fits);
        // A launch with few fits per SM (one shard of a grid split over 8 GPUs: 250 fits for 148 SMs): a binomial fit that has
        // an SM to itself -- all four tensor pipes, the whole L1 -- finishes sooner than two sharing it, and the launch is as long
        // as its longest fits.  Measured (scripts/shard_blocks.py, config-2 shards): 200 / 250 / 286 / 334 fits 40.1 / 57.0 / 58.8 /
        // 61.4 ms with two blocks per SM against 36.5 / 52.9 / 53.0 / 55.2 ms with one; from 400 fits on two blocks win (42.9
        // against 49.5 ms), and the Gaussian kernel never gains.  The tables do not depend on the grid size.
        if (p->prior == PAREBEN_BINOMIAL && !getenv("PAREBEN_BLOCKS_PER_SM") && n_fits > p->sm_count && (long long)n_fits * 10 <= (long long)p->sm_count * 23)
            grid = std::min(grid, p->sm_count);
        CU(cudaEventRecord(p->ev0, p->stream));
        if (p->prior == PAREBEN_GAUSSIAN)
            CU((p->epis ? launch_fit_ge : launch_fit_gm)(grid, p->threads, p->stream, P, v, d_tasks, n_fits, sched, p->d_slabs, p->slab_stride, out));
        else
            CU((p->epis ? launch_fit_be : launch_fit_bm)(grid, p->threads, p->stream, P, v, d_tasks, n_fits, sched, p->d_slabs, p->slab_stride, out));
        CU(cudaEventRecord(p->ev1, p->stream));
        std::vector<int> h_ints(3 * (size_t)n_fits);
        std::vector<double> h_err(n_fits);
        CU(cudaMemcpyAsync(h_err.data(), d_err, sizeof(double) * n_fits, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaMemcpyAsync(h_ints.data(), d_ints, sizeof(int) * 3 * n_fits, cudaMemcpyDeviceToHost, p->stream));
        double h_flops2[2] = {0, 0};
        CU(cudaMemcpyAsync(h_flops2, p->d_flops, 2 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        const double h_flops = h_flops2[0];
        p->last_avoided = h_flops2[1];
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
        p->last_ms = ms + p->gram_ms; p->last_flops = h_flops; p->last_launches = 1 + p->gram_launches;      // a call that had to build C pays for it
        for (int i = 0; i < n_fits; i++) {
            if (fold_err) fold_err[i] = h_err[i];
            if (status) status[i] = h_ints[i];
            if (n_selected) n_selected[i] = h_ints[n_fits + i];
            if (n_iter) n_iter[i] = h_ints[2 * (size_t)n_fits + i];
        }
        if (dump) {   // copy the dump to host-side mirrors allocated by the caller (reuse pointers)
            int *hm = (int *)malloc(sizeof(int) * (1 + p->cap));
            double *hb = (double *)malloc(sizeof(double) * (2 * p->cap + 4));
            CU(cudaMemcpy(hm, dump->m, sizeof(int) * (1 + p->cap), cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(hb, dump->beta, sizeof(double) * (2 * p->cap + 4), cudaMemcpyDeviceToHost));
            dump->m = hm; dump->used = hm + 1; dump->beta = hb; dump->var = hb + p->cap; dump->scalars = hb + 2 * p->cap;
        }
        for (int i = 0; i < ns; i++) pool_give(p->device, scratch[i], scratch_bytes[i]);
    } catch (std::pair<int, std::string> &e) {
        for (int i = 0; i < ns; i++) pool_give(p->device, scratch[i], scratch_bytes[i]);
        return fail(e.first, e.second);
    }
    return PAREBEN_OK;
}

}  // namespace

extern "C" int pareben_run_fits(pareben_problem *p, int n_fits, const int *fold, const double *alpha,
                                const double *lambda, double *fold_err, int *status, int *n_selected, int *n_iter)
{
    return run_fits_impl(p, n_fits, fold, alpha, lambda, fold_err, status, n_selected, n_iter, nullptr);
}

// Cost-aware interleaving (SURVEY.md 8e): order fits by falling expected cost (rising lambda,
// ties by fit number) and deal them round-robin, so every shard gets the same cost mix.
// Pure host logic (no device needed).
extern "C" int pareben_shard_plan(const double *lambda, int n_grid, int n_folds, int shard, int n_shards,
                                  int *fit_index, int *n_mine)
{
    if (!lambda || !fit_index || !n_mine || n_grid < 1 || n_folds < 1 || n_shards < 1 || shard < 0 || shard >= n_shards)
        return fail(PAREBEN_EINVAL, "pareben_shard_plan: bad argument");
    const int total = n_grid * n_folds;
    std::vector<int> order(total);
    for (int i = 0; i < total; i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return lambda[a / n_folds] < lambda[b / n_folds]; });
    std::vector<int> mine;
    for (int r = shard; r < total; r += n_shards) mine.push_back(order[r]);
    std::sort(mine.begin(), mine.end());
    for (size_t i = 0; i < mine.size(); i++) fit_index[i] = mine[i];
    *n_mine = (int)mine.size();
    return PAREBEN_OK;
}

namespace {

// One sub-shard of a grid call on one device: upload, lay out, run, scatter into the caller's tables.
int cv_grid_on_device(const double *basis, int n, int k, const double *target, const int *fold_id, int n_folds,
                      const double *alpha, const double *lambda, int n_grid, int epis, int prior, int device,
                      int shard, int n_shards, double *fold_err, int *status, int *n_selected)
{
    const int total = n_grid * n_folds;
    std::vector<int> mine(total);
    int m = 0;
    pareben_shard_plan(lambda, n_grid, n_folds, shard, n_shards, mine.data(), &m);
    if (m == 0) return PAREBEN_OK;
    pareben_problem *p = nullptr;
    const bool timing = getenv("PAREBEN_TIMING") != nullptr;
    auto t0 = std::chrono::steady_clock::now();
    int rc = pareben_problem_create(&p, device, basis, n, k, target, fold_id, n_folds, epis, prior);
    if (rc != PAREBEN_OK) return rc;
    auto t1 = std::chrono::steady_clock::now();
    std::vector<int> fold(m), st(m), ns(m);
    std::vector<double> a(m), l(m), err(m);
    for (int i = 0; i < m; i++) {
        const int fit = mine[i];
        fold[i] = fit % n_folds + 1; a[i] = alpha[fit / n_folds]; l[i] = lambda[fit / n_folds];
    }
    p->grid_fits_hint = total;
    rc = pareben_run_fits(p, m, fold.data(), a.data(), l.data(), err.data(), st.data(), ns.data(), nullptr);
    auto t2 = std::chrono::steady_clock::now();
    const double kernel_ms = p->last_ms;
    pareben_problem_destroy(p);
    if (timing) {
        auto t3 = std::chrono::steady_clock::now();
        auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        fprintf(stderr, "[pareben] cv_grid dev %d: create %.2f ms, run_fits %.2f ms (kernel %.2f ms), destroy %.2f ms\n",
                device, ms(t0, t1), ms(t1, t2), kernel_ms, ms(t2, t3));
    }
    if (rc != PAREBEN_OK) return rc;
    for (int i = 0; i < m; i++) {
        fold_err[mine[i]] = err[i];
        if (status) status[mine[i]] = st[i];
        if (n_selected) n_selected[mine[i]] = ns[i];
    }
    return PAREBEN_OK;
}

}  // namespace

// n_devices GPUs (device, device + 1, ...) share this call's shard: the foreach fan-out of R/CrossValidate.R:66-70
// over the box's GPUs from ONE call on ONE host thread of the caller.  Each device is driven by its own worker thread
// (upload, layout kernels, one fit launch, read-back); the workers write disjoint entries of the caller's tables, so
// the "gather" is the join.  No R API is touched from the workers.
extern "C" int pareben_cv_grid(const double *basis, int n, int k, const double *target, const int *fold_id,
                               int n_folds, const double *alpha, const double *lambda, int n_grid, int epis,
                               int prior, int n_devices, int device, int shard, int n_shards, double *fold_err,
                               int *status, int *n_selected)
{
    if (n_folds < 1 || n_grid < 1 || !alpha || !lambda || !fold_err) return fail(PAREBEN_EINVAL, "pareben_cv_grid: bad argument");
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail(PAREBEN_EINVAL, "pareben_cv_grid: bad shard");
    const int visible = pareben_device_count();
    if (visible < 1) return fail(PAREBEN_ENODEVICE, "no usable CUDA device");
    if (n_devices == 0) n_devices = visible - device;                 // 0 = every device from `device` on
    if (device < 0 || n_devices < 1 || device + n_devices > visible) return fail(PAREBEN_ENODEVICE, "pareben_cv_grid: device range not available");
    if (n_devices == 1)
        return cv_grid_on_device(basis, n, k, target, fold_id, n_folds, alpha, lambda, n_grid, epis, prior, device,
                                 shard, n_shards, fold_err, status, n_selected);
    std::vector<int> rcs(n_devices, PAREBEN_OK);
    std::vector<std::string> msgs(n_devices);
    std::vector<std::thread> workers;
    for (int d = 0; d < n_devices; d++)
        workers.emplace_back([&, d] {
            rcs[d] = cv_grid_on_device(basis, n, k, target, fold_id, n_folds, alpha, lambda, n_grid, epis, prior, device + d,
                                       shard * n_devices + d, n_shards * n_devices, fold_err, status, n_selected);
            if (rcs[d] != PAREBEN_OK) msgs[d] = g_err;                // g_err is thread-local: carry the text back
        });
    for (std::thread &w : workers) w.join();
    for (int d = 0; d < n_devices; d++)
        if (rcs[d] != PAREBEN_OK) return fail(rcs[d], "device " + std::to_string(device + d) + ": " + msgs[d]);
    return PAREBEN_OK;
}

extern "C" int pareben_fit(pareben_problem *p, double alpha, double lambda, double *beta_table, double *wald,
                           double *intercept, double *extra, int *status)
{
    if (!p || !beta_table) return fail(PAREBEN_EINVAL, "pareben_fit: bad argument");
    if (p->n_folds != 0) return fail(PAREBEN_EINVAL, "pareben_fit needs a problem created with n_folds == 0");
    DumpBuffers dump;
    int fold = 0, st = 0;
    double err = 0;
    int rc = run_fits_impl(p, 1, &fold, &alpha, &lambda, &err, &st, nullptr, nullptr, &dump);
    if (rc != PAREBEN_OK) return rc;
    const int k = p->k, kc = p->kc;
    const int M = dump.m[0];
    if (p->prior == PAREBEN_GAUSSIAN) {
        const int ncol = p->epis ? 5 : 4;
        // loci columns (MainEff.c:87-91, NeFull2.c:100-134)
        for (int c = 0; c < k; c++) { beta_table[c] = c + 1; beta_table[(size_t)kc + c] = c + 1; }
        if (p->epis) { size_t kk = k; for (int i = 0; i < k - 1; i++) for (int j = i + 1; j < k; j++, kk++) { beta_table[kk] = i + 1; beta_table[(size_t)kc + kk] = j + 1; } }
        for (size_t z = (size_t)2 * kc; z < (size_t)ncol * kc; z++) beta_table[z] = 0;
        for (int i = 0; i < M; i++) {
            const int c = dump.used[i] - 1;
            beta_table[(size_t)2 * kc + c] = dump.beta[i];
            beta_table[(size_t)3 * kc + c] = dump.var[i];
            if (p->epis) beta_table[(size_t)4 * kc + c] = dump.used[i];
        }
        if (intercept) intercept[0] = dump.scalars[1];
    } else {
        if (!p->epis) {      // k x 4 indexed by column id (NEmainEff.c:270-291, 364-371)
            for (int c = 0; c < k; c++) { beta_table[c] = c + 1; beta_table[(size_t)k + c] = c + 1; beta_table[(size_t)2 * k + c] = 0; beta_table[(size_t)3 * k + c] = 0; }
            for (int i = 0; i < M; i++) { const int c = dump.used[i] - 1; beta_table[(size_t)2 * k + c] = dump.beta[i]; beta_table[(size_t)3 * k + c] = dump.var[i]; }
        } else {             // compact 2k x 4 in Used order with decoded loci (NeFull.c:168-208)
            const int rows = 2 * k;
            for (size_t z = 0; z < (size_t)4 * rows; z++) beta_table[z] = 0;
            for (int i = 0; i < M && i < rows; i++) {
                const int c = dump.used[i] - 1;
                int li = c, lj = c;
                if (c >= k) { long long pp = (long long)c - k; int ii = 0; while ((long long)(ii + 1) * (2LL * k - (ii + 1) - 1) / 2 <= pp) ii++; li = ii; lj = (int)(pp - (long long)ii * (2LL * k - ii - 1) / 2) + ii + 1; }
                beta_table[i] = li + 1; beta_table[(size_t)rows + i] = lj + 1;
                beta_table[(size_t)2 * rows + i] = dump.beta[i]; beta_table[(size_t)3 * rows + i] = dump.var[i];
            }
        }
        if (intercept) { intercept[0] = dump.scalars[1]; intercept[1] = dump.scalars[2]; }
    }
    if (wald) wald[0] = dump.scalars[0];
    if (extra) extra[0] = dump.scalars[3];
    if (status) status[0] = st;
    free(dump.m); free(dump.beta);
    return PAREBEN_OK;
}

// The grid call on a problem that is already resident (one upload serves BuildGrid's lambda_max, the grid and any
// LocalSearch refinement): same table layout and shard assignment as pareben_cv_grid.
extern "C" int pareben_problem_cv_grid(pareben_problem *p, const double *alpha, const double *lambda, int n_grid, int shard,
                                       int n_shards, double *fold_err, int *status, int *n_selected)
{
    if (!p || !alpha || !lambda || !fold_err || n_grid < 1) return fail(PAREBEN_EINVAL, "pareben_problem_cv_grid: bad argument");
    if (p->n_folds < 1) return fail(PAREBEN_EINVAL, "pareben_problem_cv_grid needs a problem created with folds");
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail(PAREBEN_EINVAL, "pareben_problem_cv_grid: bad shard");
    const int nf = p->n_folds, total = n_grid * nf;
    std::vector<int> mine(total);
    int m = 0;
    int rc = pareben_shard_plan(lambda, n_grid, nf, shard, n_shards, mine.data(), &m);
    if (rc != PAREBEN_OK || m == 0) return rc;
    std::vector<int> fold(m), st(m), ns(m);
    std::vector<double> a(m), l(m), err(m);
    for (int i = 0; i < m; i++) { fold[i] = mine[i] % nf + 1; a[i] = alpha[mine[i] / nf]; l[i] = lambda[mine[i] / nf]; }
    p->grid_fits_hint = total;
    rc = pareben_run_fits(p, m, fold.data(), a.data(), l.data(), err.data(), st.data(), ns.data(), nullptr);
    p->grid_fits_hint = 0;
    if (rc != PAREBEN_OK) return rc;
    for (int i = 0; i < m; i++) {
        fold_err[mine[i]] = err[i];
        if (status) status[mine[i]] = st[i];
        if (n_selected) n_selected[mine[i]] = ns[i];
    }
    return PAREBEN_OK;
}

// ---------------------------------------------------------------------------------------------
// The four `.C` entry points of EBEN, same names and argument lists (MainEff.c:55-57, NeFull2.c:57-58,
// NEmainEff.c:236-238, NeFull.c:52-55), as thin wrappers over pareben_fit: with useDynLib pointed at this library the
// R wrappers EBelasticNet.Gaussian / EBelasticNet.Binomial (EBEN_orig/R) run unchanged on the GPU.  Like the originals
// they return nothing; a failure is reported on stderr (where the shimmed Rprintf of the reference writes) and leaves
// the outputs zeroed.
namespace {
void dot_c_fit(const char *name, double *BASIS, double *y, double lambda, double alpha, double *Beta, double *wald, double *intercept,
               int n, int k, int epis, int prior, double *extra, int beta_rows, int beta_cols)
{
    for (size_t i = 0, e = (size_t)beta_rows * beta_cols; i < e; i++) Beta[i] = 0;
    if (wald) wald[0] = 0;
    if (intercept) { intercept[0] = 0; if (prior == PAREBEN_BINOMIAL) intercept[1] = 0; }
    if (extra) extra[0] = 0;
    int dev = 0;
    if (const char *e = getenv("PAREBEN_DEVICE")) dev = atoi(e);
    pareben_problem *p = nullptr;
    int rc = pareben_problem_create(&p, dev, BASIS, n, k, y, nullptr, 0, epis, prior);
    int st = 0;
    if (rc == PAREBEN_OK) rc = pareben_fit(p, alpha, lambda, Beta, wald, intercept, extra, &st);
    if (p) pareben_problem_destroy(p);
    if (rc != PAREBEN_OK) fprintf(stderr, "%s (libpareben): error %d: %s\n", name, rc, pareben_last_error());
    else if (st != 0) fprintf(stderr, "%s (libpareben): fit finished with status %d\n", name, st);
}
}  // namespace

extern "C" void elasticNetLinearNeMainEff(double *BASIS, double *y, double *a_lambda, double *b_Alpha, double *Beta, double *wald,
                                          double *intercept, int *n, int *kdim, int *verb, double *residual)
{
    (void)verb;
    dot_c_fit("elasticNetLinearNeMainEff", BASIS, y, *a_lambda, *b_Alpha, Beta, wald, intercept, *n, *kdim, 0, PAREBEN_GAUSSIAN, residual, *kdim, 4);
}

extern "C" void elasticNetLinearNeEpisEff(double *BASIS, double *y, double *a_lambda, double *b_Alpha, double *Beta, double *wald,
                                          double *intercept, int *n, int *kdim, int *verb, double *residual)
{
    (void)verb;
    const int k = *kdim;
    dot_c_fit("elasticNetLinearNeEpisEff", BASIS, y, *a_lambda, *b_Alpha, Beta, wald, intercept, *n, k, 1, PAREBEN_GAUSSIAN, residual,
              (int)((long long)k * (k + 1) / 2), 5);
}

extern "C" void ElasticNetBinaryNEmainEff(double *BASIS, double *Targets, double *a_Lambda, double *b_Alpha, double *logLIKELIHOOD,
                                          double *Beta, double *wald, double *intercept, int *n, int *kdim, int *VB, int *bMax)
{
    (void)VB; (void)bMax;                     // bMax = k for main effects (EBelasticNet.Binomial.R:30): the table is k x 4
    dot_c_fit("ElasticNetBinaryNEmainEff", BASIS, Targets, *a_Lambda, *b_Alpha, Beta, wald, intercept, *n, *kdim, 0, PAREBEN_BINOMIAL,
              logLIKELIHOOD, *kdim, 4);
}

extern "C" void ElasticNetBinaryNEfull(double *BASIS, double *Targets, double *a_Lambda, double *b_Alpha, double *logLIKELIHOOD,
                                       double *Beta, double *wald, double *intercept, int *n, int *kdim, int *VB, int *bMax)
{
    (void)VB; (void)bMax;                     // bMax = 2k for Epis (EBelasticNet.Binomial.R:8): the table is 2k x 4, compact
    dot_c_fit("ElasticNetBinaryNEfull", BASIS, Targets, *a_Lambda, *b_Alpha, Beta, wald, intercept, *n, *kdim, 1, PAREBEN_BINOMIAL,
              logLIKELIHOOD, 2 * *kdim, 4);
}

extern "C" int pareben_lambda_max(pareben_problem *p, double *lambda_max)
{
    if (!p || !lambda_max) return fail(PAREBEN_EINVAL, "pareben_lambda_max: bad argument");
    try {
        CU(cudaSetDevice(p->device));
        // GetLambdaMax works on ALL rows (R/BuildGrid.R:5-32): build a row-major copy once.
        const int n = p->n, k = p->k;
        std::vector<double> y(n);
        CU(cudaMemcpy(y.data(), p->d_y, sizeof(double) * n, cudaMemcpyDeviceToHost));
        long double s = 0; for (double v : y) s += v;
        long double mean = s / n, t = 0; for (double v : y) t += (v - mean);
        mean += t / n;
        std::vector<double> centred(n), resp(n);
        long double ss = 0;
        for (int i = 0; i < n; i++) { centred[i] = (double)(y[i] - (double)mean); ss += (long double)centred[i] * centred[i]; }
        const double nrm = std::sqrt((double)ss);
        for (int i = 0; i < n; i++) resp[i] = centred[i] / nrm;
        // scratch comes from the problem's pooled allocations (returned to the pool with the problem; nothing to leak on error)
        double *d_rows_x = p->dalloc<double>((size_t)n * k), *d_resp = p->dalloc<double>(n);
        int *d_rows = p->dalloc<int>(n);
        std::vector<int> rows(n); for (int i = 0; i < n; i++) rows[i] = i;
        CU(cudaMemcpy(d_rows, rows.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
        gather_rows_kernel<<<dim3((n + 31) / 32, (k + 31) / 32), dim3(32, 8), 0, p->stream>>>(p->d_Xcol, n, k, d_rows, n, d_rows_x);
        double best = std::log(1.1);
        auto pass = [&](int c0, int c1, const std::vector<double> &r, bool epis) {
            const int nb = (c1 - c0 + 255) / 256;
            if (nb <= 0) return;
            CU(cudaMemcpyAsync(d_resp, r.data(), sizeof(double) * n, cudaMemcpyHostToDevice, p->stream));
            double *d_max = p->dalloc<double>(nb);
            if (epis) lambda_max_kernel<true><<<nb, 256, 0, p->stream>>>(d_rows_x, n, k, c0, c1, d_resp, d_max);
            else lambda_max_kernel<false><<<nb, 256, 0, p->stream>>>(d_rows_x, n, k, c0, c1, d_resp, d_max);
            CU(cudaGetLastError());
            std::vector<double> hm(nb);
            CU(cudaMemcpyAsync(hm.data(), d_max, sizeof(double) * nb, cudaMemcpyDeviceToHost, p->stream));
            CU(cudaStreamSynchronize(p->stream));
            for (double v : hm) if (v > best) best = v;
        };
        pass(0, k, resp, false);                       // main effects against the normalised response (:14-19)
        if (p->epis) pass(k, p->kc, centred, true);    // pairs against the UN-normalised centred response (:24-27)
        *lambda_max = best;
    } catch (std::pair<int, std::string> &e) {
        return fail(e.first, e.second);
    }
    return PAREBEN_OK;
}

extern "C" int pareben_sl_filter(pareben_problem *p, double tau_main, double tau_pair, int capacity, int *cand, double *stat,
                                 int *n_kept)
{
    if (!p || !n_kept || capacity < 0) return fail(PAREBEN_EINVAL, "pareben_sl_filter: bad argument");
    try {
        CU(cudaSetDevice(p->device));
        const int n = p->n, k = p->k;
        std::vector<double> y(n), ys(n);
        CU(cudaMemcpy(y.data(), p->d_y, sizeof(double) * n, cudaMemcpyDeviceToHost));
        long double s = 0; for (double v : y) s += v;
        long double mean = s / n, t = 0; for (double v : y) t += (v - mean);
        mean += t / n;                                                     // R's two-pass mean
        long double ss = 0; for (double v : y) ss += ((long double)v - mean) * ((long double)v - mean);
        const double sd = std::sqrt((double)(ss / (n - 1)));
        for (int i = 0; i < n; i++) ys[i] = (double)(y[i] - (double)mean) / sd;
        double *d_rows_x = p->dalloc<double>((size_t)n * k), *d_ys = p->dalloc<double>(n);
        int *d_rows = p->dalloc<int>(n);
        std::vector<int> rows(n); for (int i = 0; i < n; i++) rows[i] = i;
        CU(cudaMemcpy(d_rows, rows.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
        CU(cudaMemcpyAsync(d_ys, ys.data(), sizeof(double) * n, cudaMemcpyHostToDevice, p->stream));
        gather_rows_kernel<<<dim3((n + 31) / 32, (k + 31) / 32), dim3(32, 8), 0, p->stream>>>(p->d_Xcol, n, k, d_rows, n, d_rows_x);
        const int chunk = 1 << 22;
        double *d_stat = p->dalloc<double>(chunk);
        std::vector<double> h_stat(chunk);
        long long kept = 0;
        const int c_total = p->epis ? p->kc : k;
        for (int c0 = 0; c0 < c_total; ) {
            // a chunk never straddles the main-effect / pair boundary (different thresholds, different column rule)
            const bool pairs = c0 >= k;
            const int c1 = std::min(pairs ? c_total : k, c0 + chunk);
            const int nb = (c1 - c0 + 255) / 256;
            if (pairs) sl_stat_kernel<true><<<nb, 256, 0, p->stream>>>(d_rows_x, n, k, c0, c1, d_ys, d_stat);
            else sl_stat_kernel<false><<<nb, 256, 0, p->stream>>>(d_rows_x, n, k, c0, c1, d_ys, d_stat);
            CU(cudaGetLastError());
            CU(cudaMemcpyAsync(h_stat.data(), d_stat, sizeof(double) * (c1 - c0), cudaMemcpyDeviceToHost, p->stream));
            CU(cudaStreamSynchronize(p->stream));
            const double tau = pairs ? tau_pair : tau_main;
            for (int c = c0; c < c1; c++) {
                const double v = h_stat[c - c0];
                if (v > tau) {
                    if (kept < capacity) { if (cand) cand[kept] = c; if (stat) stat[kept] = v; }
                    kept++;
                }
            }
            c0 = c1;
        }
        *n_kept = (int)std::min<long long>(kept, 0x7fffffff);
    } catch (std::pair<int, std::string> &e) {
        return fail(e.first, e.second);
    }
    return PAREBEN_OK;
}

// experiments only (timing build, -DPAREBEN_PHASE_TIMING; absent from the product library): cycles per phase summed over
// blocks and over the four kernel variants.  out: PH_COUNT cycle totals then PH_COUNT call counts.
#ifdef PAREBEN_PHASE_TIMING
extern "C" int pareben_phase_cycles(unsigned long long *out, int reset)
{
    unsigned long long acc[2 * PH_COUNT] = {0}, one[2 * PH_COUNT];
    void (*fn[4])(unsigned long long *, int, unsigned long long *, unsigned long long *, int *, int) = {timing_gm, timing_ge, timing_bm, timing_be};
    for (int i = 0; i < 4; i++) {
        for (int j = 0; j < 2 * PH_COUNT; j++) one[j] = 0;
        fn[i](one, reset, nullptr, nullptr, nullptr, 0);
        for (int j = 0; j < 2 * PH_COUNT; j++) acc[j] += one[j];
    }
    if (out) for (int j = 0; j < 2 * PH_COUNT; j++) out[j] = acc[j];
    return PH_COUNT;
}

// experiments only: per-fit start/end (%globaltimer ns) and block id of the last launch of variant
// `which` (0 gm, 1 ge, 2 bm, 3 be).
extern "C" int pareben_fit_trace(int which, unsigned long long *t0, unsigned long long *t1, int *block, int n)
{
    void (*fn[4])(unsigned long long *, int, unsigned long long *, unsigned long long *, int *, int) = {timing_gm, timing_ge, timing_bm, timing_be};
    if (which < 0 || which > 3) return 0;
    fn[which](nullptr, 0, t0, t1, block, n);
    return n;
}
#endif  // PAREBEN_PHASE_TIMING

extern "C" int pareben_set_mode(int mode)
{
    if (mode < 0 || mode > 2) return fail(PAREBEN_EINVAL, "pareben_set_mode: mode must be 0 (auto), 1 (cached) or 2 (streaming)");
    g_mode = mode;
    return PAREBEN_OK;
}

extern "C" int pareben_is_streaming(pareben_problem *p) { return p && p->streaming ? 1 : 0; }

extern "C" int pareben_last_stream_counters(pareben_problem *p, double *scan_ms, double *scan_flops, int *scan_launches, int *rounds)
{
    if (!p) return fail(PAREBEN_EINVAL, "null problem");
    if (scan_ms) *scan_ms = p->last_scan_ms;
    if (scan_flops) *scan_flops = p->last_scan_flops;
    if (scan_launches) *scan_launches = p->last_scan_launches;
    if (rounds) *rounds = p->last_rounds;
    return PAREBEN_OK;
}

extern "C" int pareben_last_gram_info(pareben_problem *p, int *in_use, double *avoided_flops, double *build_ms)
{
    if (!p) return fail(PAREBEN_EINVAL, "null problem");
    if (in_use) *in_use = p->gram_state == 1 ? 1 : 0;
    if (avoided_flops) *avoided_flops = p->last_avoided;
    if (build_ms) *build_ms = p->gram_ms;
    return PAREBEN_OK;
}

extern "C" int pareben_last_counters(pareben_problem *p, double *flops, double *kernel_ms, int *launches)
{
    if (!p) return fail(PAREBEN_EINVAL, "null problem");
    if (flops) *flops = p->last_flops;
    if (kernel_ms) *kernel_ms = p->last_ms;
    if (launches) *launches = p->last_launches;
    return PAREBEN_OK;
}

// FP64 peak probes used by bench.py for the roofline denominator (MEASURED_PEAKS.json has no
// FP64 entry).  which: 0 = DFMA (CUDA cores), 1 = DMMA (mma.sync m8n8k4 f64).
extern "C" int pareben_measure_fp64_peak(int device, int which, double *tflops)
{
    if (!tflops) return fail(PAREBEN_EINVAL, "null output");
    if (pareben_device_count() <= device || device < 0) return fail(PAREBEN_ENODEVICE, "no usable CUDA device");
    try {
        CU(cudaSetDevice(device));
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, device));
        const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 15;
        double *d = nullptr;
        CU(cudaMalloc(&d, sizeof(double) * blocks * threads));
        cudaEvent_t e0, e1;
        CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
        double best = 0;
        for (int rep = 0; rep < 5; rep++) {
            CU(cudaEventRecord(e0));
            if (which == 0) dfma_peak_kernel<<<blocks, threads>>>(d, iters);
            else dmma_peak_kernel<<<blocks, threads>>>(d, iters);
            CU(cudaEventRecord(e1));
            CU(cudaEventSynchronize(e1));
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, e0, e1));
            double fl = which == 0 ? 2.0 * 8 * iters * (double)blocks * threads
                                   : 2.0 * 8 * 8 * 4 * 4 * iters * (double)blocks * (threads / 32);
            if (rep > 0) best = std::max(best, fl / (ms * 1e-3) / 1e12);
        }
        cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
        *tflops = best;
    } catch (std::pair<int, std::string> &e) {
        return fail(e.first, e.second);
    }
    return PAREBEN_OK;
}
