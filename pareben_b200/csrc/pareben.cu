// pareben.cu -- host side of libpareben.so: problem upload, per-fold layout kernels, the
// persistent batched-fit launch, and the extern "C" entry points declared in include/pareben.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -fmad=false --shared ...
// (-fmad=false keeps the scalar decision formulas un-contracted like the reference's x86 build;
//  the hot loops use explicit fma()).
#include "../../include/pareben.h"
#include "common.cuh"
#include "tc_contract.cuh"
#include "layout.cuh"
#include "fit_launch.h"
#include "stream_launch.h"

#include <algorithm>
#include <map>
#include <new>
#include <tuple>
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

// out[t * ld_out + r] = y[t * n + rows[r]] for response t = blockIdx.y (columns of an n x n_targets matrix)
__global__ void gather_vec_kernel(const double *__restrict__ y, int n, const int *__restrict__ rows, int nrows,
                                  double *__restrict__ out, size_t ld_out)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < nrows) out[blockIdx.y * ld_out + r] = y[(size_t)blockIdx.y * n + rows[r]];
}

// lambda_max pieces (R/BuildGrid.R:5-32) for T responses in one pass over the candidates: lmax[t] = max(lmax[t], max over
// candidates c of x_c' r_t / ||x_c||), r_t = resp + t * N.  A thread owns a candidate and holds TT accumulators, one per
// response of the current tile; the tile's responses are staged in shared memory LM_ROWS rows at a time and read as
// broadcasts, so each value x of the candidate column feeds TT FMAs.  For every (candidate, response) the FMA chain is
// z = fma(x_h, r_h, z) over h = 0..N-1 from z = 0, and ||x_c||^2 = fma(x_h, x_h, nn) once per candidate: a response's
// value does not depend on T or on which tile it falls in.  Only positive maxima matter to the caller (it starts from
// log(1.1)), and a positive double's bit pattern orders like its value, so the block maxima meet in lmax with atomicMax.
constexpr int LM_THREADS = 256, LM_ROWS = 64;
template <bool EPIS, int TT>
__global__ void __launch_bounds__(LM_THREADS) lambda_max_multi_kernel(const double *__restrict__ X, int N, int K, int c_begin,
                                                                      int c_end, const double *__restrict__ resp, int T,
                                                                      double *__restrict__ lmax)
{
    __shared__ __align__(16) double s_r[LM_ROWS][TT];
    __shared__ double red[LM_THREADS / 32][TT];
    const int c = c_begin + blockIdx.x * LM_THREADS + threadIdx.x;
    const bool live = c < c_end;
    const Cand<EPIS> cd(live ? c : c_begin, K);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double nn = 0;
    for (int t0 = 0; t0 < T; t0 += TT) {
        double z[TT];
#pragma unroll
        for (int j = 0; j < TT; j++) z[j] = 0;
        for (int h0 = 0; h0 < N; h0 += LM_ROWS) {
            const int nh = min(LM_ROWS, N - h0);
            __syncthreads();
            for (int i = threadIdx.x; i < LM_ROWS * TT; i += LM_THREADS) {
                const int hh = i / TT, j = i % TT;
                s_r[hh][j] = (t0 + j < T && hh < nh) ? resp[(size_t)(t0 + j) * N + h0 + hh] : 0.0;
            }
            __syncthreads();
            if (live) {
                for (int hh = 0; hh < nh; hh++) {
                    const double x = cd.at(X + (size_t)(h0 + hh) * K);
#pragma unroll
                    for (int j = 0; j < TT; j++) z[j] = fma(x, s_r[hh][j], z[j]);
                    if (t0 == 0) nn = fma(x, x, nn);
                }
            }
        }
        const double rn = live && nn > 0 ? sqrt(nn) : 0.0;
#pragma unroll
        for (int j = 0; j < TT; j++) {
            double v = rn > 0 ? z[j] / rn : -1e300;
            for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
            if (lane == 0) red[wid][j] = v;
        }
        __syncthreads();
        if (threadIdx.x < TT && t0 + (int)threadIdx.x < T) {
            double m = red[0][threadIdx.x];
            for (int w = 1; w < LM_THREADS / 32; w++) m = fmax(m, red[w][threadIdx.x]);
            if (m > 0) atomicMax(reinterpret_cast<unsigned long long *>(lmax + t0 + threadIdx.x), (unsigned long long)__double_as_longlong(m));
        }
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
    int tc = 0;                          // the folds carry the int8 operand images of the tensor-core contraction (FoldData::Xtc)
    int n = 0, k = 0, kc = 0, n_folds = 0, epis = 0, prior = 0, cap = 0, nmax = 0, min_ntr = 0;
    int n_targets = 1;                   // responses sharing the design (pareben_problem_create_multi)
    int sm_count = 0;
    std::vector<PoolEntry> allocs;       // every device buffer of this problem (returned to the pool on destroy)
    FoldData *d_folds = nullptr;
    // [n_targets][n_folds + 1] (Problem::folds): h_folds[f] are response 0's records, whose design-side pointers every
    // response shares; whatever changes a design-side field changes it in all n_targets records of the fold
    std::vector<FoldData> h_folds;
    double *d_Xcol = nullptr, *d_y = nullptr;     // full data, column-major: X n x k, y n x n_targets (kept for lambda_max)
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
    double last_tc_calls = 0;            // score contractions the last call ran on the int8 tensor cores
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

// basis cap of the cached kernels: the reference's basisMax, bounded (PAREBEN_BASIS_CAP, default 1024) so that the
// per-block slab stays reasonable
static int cached_cap(const pareben_problem *p)
{
    int cap = reference_basis_max(p->min_ntr, p->k, p->kc, p->epis, p->prior);
    const char *env_cap = getenv("PAREBEN_BASIS_CAP");
    int hard = env_cap ? atoi(env_cap) : 1024;
    if (hard < 2) hard = 2;
    if (p->prior == PAREBEN_BINOMIAL) cap += 1;       // slot 0 is the intercept
    return std::max(2, std::min(cap, hard));
}

// The per-block work slabs are only needed by the fit kernel: they are sized and allocated at the first
// pareben_run_fits / pareben_fit of a problem (lambda_max and the single-locus prefilter never touch them, and an
// Epis problem's candidate cache can be far larger than those two need).  Throws like the CU() macro.
static void ensure_slabs(pareben_problem *p)
{
    if (p->d_slabs) return;
    p->cap = cached_cap(p);

    // persistent grid: blocks per SM limited by memory for slabs
    p->slab_stride = slab_bytes(p->cap, p->nmax, p->kc, p->tc);
    // resident blocks per SM of the kernel variant this problem will launch (asked once per variant:
    // the occupancy query, like cudaMemGetInfo below, costs up to tens of milliseconds)
    int per_sm = 1;
    {
        // Block size: measured on B200 (config 2 / bundled Gaussian): 256 threads x 2 blocks per SM beats
        // 128 x 4 (-5 % / -43 %) and 64 x 8 (-40 % / -70 %) (measured with an earlier build that had a run-time block size).
        p->threads = FIT_THREADS_HOST;     // sweep_regs() and the fused gram_pipe() run only at exactly 256 threads
        static int occ_cache[5] = {0, 0, 0, 0, 0};
        int &occ = occ_cache[p->tc ? 4 : (p->prior == PAREBEN_BINOMIAL ? 2 : 0) + (p->epis ? 1 : 0)];
        if (!occ) {
            cudaError_t e;
            if (p->prior == PAREBEN_GAUSSIAN) e = p->epis ? occupancy_ge(&occ, p->threads) : occupancy_gm(&occ, p->threads);
            else e = p->epis ? occupancy_be(&occ, p->threads) : p->tc ? occupancy_bt(&occ, p->threads) : occupancy_bm(&occ, p->threads);
            CU(e);
        }
        per_sm = std::max(1, occ);
        // The occupancy calculator counts one block per SM for any kernel that contains a tensor-memory allocation.  Two blocks
        // of the tensor-core variant fit its registers and shared memory and take 256 of the SM's 512 TMEM columns each
        // (tc_contract.cuh); measured resident and running side by side on B200.
        if (p->tc) per_sm = std::max(per_sm, 2);
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
    const int nf1 = p->n_folds + 1;
    for (int f : need) {
        double *C = p->dalloc<double>(bytes_per_fold / sizeof(double));
        for (int t = 0; t < p->n_targets; t++) p->h_folds[(size_t)t * nf1 + f].C = C;
    }
    int *d_list = p->dalloc<int>(need.size() + 1);           // fold list + the work counter (small, kept with the problem)
    std::vector<int> h_list(need);
    h_list.push_back(0);
    CU(cudaMemcpyAsync(d_list, h_list.data(), sizeof(int) * h_list.size(), cudaMemcpyHostToDevice, p->stream));
    CU(cudaMemcpyAsync(p->d_folds, p->h_folds.data(), sizeof(FoldData) * p->h_folds.size(), cudaMemcpyHostToDevice, p->stream));
    Problem P;
    P.N = p->n; P.K = p->k; P.Kc = p->kc; P.n_folds = p->n_folds; P.epis = p->epis; P.prior = p->prior;
    P.cap = p->cap; P.nmax = p->nmax; P.tc = p->tc; P.folds = p->d_folds;
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

extern "C" int pareben_problem_create_multi(pareben_problem **out, int device, const double *basis, int n, int k,
                                            const double *targets, int n_targets, const int *fold_id, int n_folds, int epis,
                                            int prior)
{
    if (!out || !basis || !targets || n < 2 || k < 1 || n_targets < 1 || n_folds < 0 || (n_folds > 0 && !fold_id))
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
        p->n = n; p->k = k; p->epis = epis; p->prior = prior; p->n_folds = n_folds; p->n_targets = n_targets;
        p->kc = epis ? (int)((long long)k * (k + 1) / 2) : k;
        p->streaming = want_streaming(p->kc, prior);
        if (p->streaming && n_folds + 1 > STREAM_MAX_FOLDS) throw std::make_pair((int)PAREBEN_EINVAL, std::string("streaming mode supports at most 255 folds"));
        CU(cudaStreamCreate(&p->stream));
        CU(cudaEventCreate(&p->ev0)); CU(cudaEventCreate(&p->ev1));

        p->d_Xcol = p->dalloc<double>((size_t)n * k);
        p->d_y = p->dalloc<double>((size_t)n * n_targets);
        CU(cudaMemcpyAsync(p->d_Xcol, basis, sizeof(double) * n * k, cudaMemcpyHostToDevice, p->stream));
        CU(cudaMemcpyAsync(p->d_y, targets, sizeof(double) * n * n_targets, cudaMemcpyHostToDevice, p->stream));

        // Genotype-coded designs (every entry an integer in [-127, 127], e.g. {-1, 0, 1}) also get an
        // int8 copy of the training matrices: the score contraction reads 1 byte instead of 8 per
        // element and widens in registers (exact).
        bool small_int = true;
        double max_abs = 0;
        for (size_t i = 0, e = (size_t)n * k; small_int && i < e; i++) {
            const double v = basis[i];
            if (!(v >= -127.0 && v <= 127.0) || v != (double)(int)v) small_int = false;
            max_abs = std::max(max_abs, std::fabs(v));
        }
        // Binomial main-effect fits on such designs with |x| <= 11 (x^2 fits int8) run the score contraction on the int8
        // tensor cores (tc_contract.cuh); every other design keeps the FP64 contraction.  The int32 sums of one digit plane
        // are bounded by rows x max|x|^2 x 64, which must stay below 2^31 (about 277,000 training rows at |x| = 11).
        p->tc = small_int && max_abs <= 11.0 && (double)n * max_abs * max_abs * 64.0 < 2147483648.0 && !epis &&
                prior == PAREBEN_BINOMIAL && !p->streaming;
        lap("stream/events/h2d enqueue/scan");
        // row lists per fold: index 0 = all rows (only materialised when n_folds == 0)
        const int nf = n_folds;
        p->h_folds.assign((size_t)n_targets * (nf + 1), FoldData{});
        std::vector<size_t> ld_y(2 * (nf + 1), 0);      // per fold: stride of the responses' training / test vectors
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
            // responses of the fold: one vector per response, each starting on a 256-byte boundary like its own allocation would
            ld_y[2 * f] = ((size_t)F.ntr + 31) & ~(size_t)31; ld_y[2 * f + 1] = ((size_t)F.nte + 31) & ~(size_t)31;
            double *Xtr = p->dalloc<double>((size_t)F.ntr * k), *ytr = p->dalloc<double>(ld_y[2 * f] * n_targets);
            double *Xte = p->dalloc<double>((size_t)F.nte * k), *yte = p->dalloc<double>(ld_y[2 * f + 1] * n_targets);
            double *scale = p->streaming ? nullptr : p->dalloc<double>(p->kc);     // streaming: norms are computed on the fly
            dim3 blk(32, 8);
            gather_rows_kernel<<<dim3((F.ntr + 31) / 32, (k + 31) / 32), blk, 0, p->stream>>>(p->d_Xcol, n, k, d_rows, F.ntr, Xtr);
            for (int t0 = 0; t0 < n_targets; t0 += 65535) {          // grid.y: one response each
                const unsigned nt = (unsigned)std::min(65535, n_targets - t0);
                gather_vec_kernel<<<dim3((F.ntr + 255) / 256, nt), 256, 0, p->stream>>>(p->d_y + (size_t)t0 * n, n, d_rows, F.ntr,
                                                                                         ytr + t0 * ld_y[2 * f], ld_y[2 * f]);
                if (F.nte > 0)
                    gather_vec_kernel<<<dim3((F.nte + 255) / 256, nt), 256, 0, p->stream>>>(p->d_y + (size_t)t0 * n, n, d_rows + F.ntr, F.nte,
                                                                                             yte + t0 * ld_y[2 * f + 1], ld_y[2 * f + 1]);
            }
            if (F.nte > 0)
                gather_rows_kernel<<<dim3((F.nte + 31) / 32, (k + 31) / 32), blk, 0, p->stream>>>(p->d_Xcol, n, k, d_rows + F.ntr, F.nte, Xte);
            if (scale) {
                if (epis) scales_kernel<true><<<(p->kc + 255) / 256, 256, 0, p->stream>>>(Xtr, F.ntr, k, p->kc, scale);
                else scales_kernel<false><<<(p->kc + 255) / 256, 256, 0, p->stream>>>(Xtr, F.ntr, k, p->kc, scale);
            }
            F.Xtr = Xtr; F.ytr = ytr; F.Xte = Xte; F.yte = yte; F.scale = scale; F.Xtr8 = nullptr;
            F.XT8 = nullptr; F.XTd = nullptr; F.C = nullptr; F.Xtc = nullptr; F.Xtcsq = nullptr;
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
            if (p->tc) {
                const int nst = (F.ntr + TC_KS - 1) / TC_KS, ntile = (k + TC_TILE - 1) / TC_TILE;
                const size_t bytes = (size_t)ntile * nst * TC_A_BYTES;
                int8_t *img = p->dalloc<int8_t>(2 * bytes);
                tc_image_kernel<<<(int)std::min<size_t>(1024, (bytes + 255) / 256), 256, 0, p->stream>>>(Xtr, F.ntr, k, nst, ntile, img, img + bytes);
                F.Xtc = img; F.Xtcsq = img + bytes;
            }
        }
        CU(cudaGetLastError());
        // the other responses' records: response 0's design side, their own ytr / yte
        for (int t = 1; t < n_targets; t++)
            for (int f = 0; f <= nf; f++) {
                FoldData &R = p->h_folds[(size_t)t * (nf + 1) + f];
                R = p->h_folds[f];
                if (R.ytr) { R.ytr += t * ld_y[2 * f]; R.yte += t * ld_y[2 * f + 1]; }
            }
        lap("per-fold layout (enqueue)");
        p->d_folds = p->dalloc<FoldData>(p->h_folds.size());
        CU(cudaMemcpyAsync(p->d_folds, p->h_folds.data(), sizeof(FoldData) * p->h_folds.size(), cudaMemcpyHostToDevice, p->stream));

        p->min_ntr = min_ntr;
        p->d_flops = p->dalloc<double>(3);
        CU(cudaStreamSynchronize(p->stream));
        lap("final sync");
    } catch (std::pair<int, std::string> &e) {
        delete p;
        return fail(e.first, e.second);
    }
    *out = p;
    return PAREBEN_OK;
}

extern "C" int pareben_problem_create(pareben_problem **out, int device, const double *basis, int n, int k,
                                      const double *target, const int *fold_id, int n_folds, int epis, int prior)
{
    return pareben_problem_create_multi(out, device, basis, n, k, target, 1, fold_id, n_folds, epis, prior);
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

// Full-model records of a launch's fits (FitOutputs::m_out ..): fit o has m(o) effects, used(o)[i] / beta(o)[i] / var(o)[i]
// for i < m(o), and scalars(o)[0..3].  The device buffer is one allocation of bytes(n, ld), doubles first, and comes back
// into `host` with one copy.
struct DumpBuffers {
    int n = 0, ld = 0;                   // records, record stride (the basis cap of the launch)
    std::vector<char> host;
    static size_t bytes(size_t n, int ld) { return n * ((2 * (size_t)ld + 4) * sizeof(double) + (1 + (size_t)ld) * sizeof(int)); }
    // point out's record arrays into a buffer of bytes(n, ld) bytes
    static void carve(char *base, size_t n, int ld, FitOutputs &out)
    {
        out.beta_out = reinterpret_cast<double *>(base); out.var_out = out.beta_out + n * ld; out.scalars_out = out.var_out + n * ld;
        out.m_out = reinterpret_cast<int *>(out.scalars_out + 4 * n); out.used_out = out.m_out + n; out.dump_ld = ld;
    }
    // size the host side for n records of stride ld (throws std::bad_alloc like any host allocation)
    void resize(int n_, int ld_) { n = n_; ld = ld_; host.assign(bytes(n, ld), 0); }
    FitOutputs view() { FitOutputs o; carve(host.data(), n, ld, o); return o; }
    int m(int o) { return view().m_out[o]; }
    const int *used(int o) { return view().used_out + (size_t)o * ld; }
    const double *beta(int o) { return view().beta_out + (size_t)o * ld; }
    const double *var(int o) { return view().var_out + (size_t)o * ld; }
    const double *scalars(int o) { return view().scalars_out + 4 * (size_t)o; }
    // record j of src into record i of this (same stride)
    void copy_from(int i, DumpBuffers &src, int j)
    {
        FitOutputs d = view(), s = src.view();
        d.m_out[i] = s.m_out[j];
        memcpy(d.used_out + (size_t)i * ld, s.used_out + (size_t)j * ld, sizeof(int) * ld);
        memcpy(d.beta_out + (size_t)i * ld, s.beta_out + (size_t)j * ld, sizeof(double) * ld);
        memcpy(d.var_out + (size_t)i * ld, s.var_out + (size_t)j * ld, sizeof(double) * ld);
        memcpy(d.scalars_out + 4 * (size_t)i, s.scalars_out + 4 * (size_t)j, sizeof(double) * 4);
    }
};

// Streaming mode (stream.cuh): every fit keeps only its active set; all fits advance in lock-step rounds of
//   stream_advance_kernel (one block per fit)  ->  stream_scan_kernel (one dense contraction per fold for all waiting fits)
// until no fit is waiting for a scan.  One 4-byte-per-fold read-back per round tells the host when to stop.
constexpr int STREAM_LIST_CAP = 4096;

// device bytes of one streaming fit's state at basis cap c (the layout run_fits_streaming carves)
size_t stream_fit_bytes(const pareben_problem *p, int c)
{
    const size_t LD = phi_ld(p->nmax), lc = STREAM_LIST_CAP;
    const size_t dbl = (size_t)4 * c * c + LD * c + (size_t)12 * (c + 1) + (size_t)4 * p->nmax + 2 * lc + 16;
    const size_t ints = (size_t)2 * c + (size_t)4 * (c + lc) + lc + 16;
    return ((dbl * 8 + ints * 4) + 255) & ~(size_t)255;
}

// the largest basis cap a streaming call can get: the reference's basisMax, bounded by PAREBEN_BASIS_CAP
int stream_cap_bound(const pareben_problem *p)
{
    const int cap = reference_basis_max(p->min_ntr, p->k, p->kc, p->epis, p->prior);
    const char *env_cap = getenv("PAREBEN_BASIS_CAP");
    return std::max(2, std::min(cap, env_cap ? atoi(env_cap) : 1024));
}

// basis cap of a streaming call whose largest response has fits_per_target fits: stream_cap_bound, lowered to what that
// many active sets may occupy.  It depends on the fits of one response, never on the number of responses, so each
// response's fits end as they would in a single-response call.
int stream_cap(const pareben_problem *p, long long fits_per_target, size_t free_b)
{
    int cap = stream_cap_bound(p);
    while (cap > 16 && stream_fit_bytes(p, cap) * (size_t)fits_per_target > free_b / 2) cap = cap * 3 / 4;
    return cap;
}

int run_fits_streaming(pareben_problem *p, int n_fits, const int *target, const int *fold, const double *alpha, const double *lambda,
                       double *fold_err, int *status, int *n_selected, int *n_iter, DumpBuffers *dump, int cap)
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
        const int list_cap = STREAM_LIST_CAP;
        const int LD = phi_ld(p->nmax);
        p->cap = cap;
        const size_t stride = stream_fit_bytes(p, cap);
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
            f.fold = fold[i]; f.target = target[i]; f.out_index = i; f.lambda = lambda[i]; f.alpha_en = alpha[i]; f.phase = SP_START;
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
        out.dump_ld = 0;
        out.flops = p->d_flops;
        char *d_dump = nullptr;
        if (dump) {
            dump->resize(n_fits, cap);
            d_dump = (char *)tmp_alloc(DumpBuffers::bytes(n_fits, cap));
            DumpBuffers::carve(d_dump, n_fits, cap, out);
        }
        Problem P;
        P.N = p->n; P.K = p->k; P.Kc = p->kc; P.n_folds = p->n_folds; P.epis = p->epis; P.prior = p->prior;
        P.cap = cap; P.nmax = p->nmax; P.tc = p->tc; P.folds = p->d_folds;
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
        if (dump) CU(cudaMemcpyAsync(dump->host.data(), d_dump, dump->host.size(), cudaMemcpyDeviceToHost, p->stream));
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
        cudaEventDestroy(es0); cudaEventDestroy(es1);
        for (auto &q : scratch) pool_give(p->device, q.first, q.second);
    } catch (std::pair<int, std::string> &e) {
        if (es0) cudaEventDestroy(es0);
        if (es1) cudaEventDestroy(es1);
        for (auto &q : scratch) pool_give(p->device, q.first, q.second);
        return fail(e.first, e.second);
    } catch (std::bad_alloc &) {
        if (es0) cudaEventDestroy(es0);
        if (es1) cudaEventDestroy(es1);
        for (auto &q : scratch) pool_give(p->device, q.first, q.second);
        return fail(PAREBEN_ENOMEM, "host allocation of the fit records failed");
    }
    return PAREBEN_OK;
}

// Streaming call: the basis cap comes from the largest share of the fits that one response has (stream_cap).  When the
// states of all fits do not fit in device memory at that cap, the responses run in waves of whole responses.
int run_fits_streaming_waves(pareben_problem *p, int n_fits, const int *target, const int *fold, const double *alpha,
                             const double *lambda, double *fold_err, int *status, int *n_selected, int *n_iter, DumpBuffers *dump)
{
    std::vector<long long> per_t(p->n_targets, 0);
    for (int i = 0; i < n_fits; i++) per_t[target[i]]++;
    size_t free_b = 0, total_b = 0;
    cudaError_t e = cudaSetDevice(p->device);
    if (e == cudaSuccess) e = cudaMemGetInfo(&free_b, &total_b);
    if (e != cudaSuccess) return fail(PAREBEN_ECUDA, std::string("cudaMemGetInfo failed: ") + cudaGetErrorString(e));
    free_b += pool_parked(p->device);
    const int cap = stream_cap(p, *std::max_element(per_t.begin(), per_t.end()), free_b);
    const long long budget = std::max<long long>(1, (long long)(free_b / 2 / stream_fit_bytes(p, cap)));
    if (n_fits <= budget)
        return run_fits_streaming(p, n_fits, target, fold, alpha, lambda, fold_err, status, n_selected, n_iter, dump, cap);
    if (dump) {
        try { dump->resize(n_fits, cap); } catch (std::bad_alloc &) { return fail(PAREBEN_ENOMEM, "host allocation of the fit records failed"); }
    }
    DumpBuffers wave_dump;                 // each wave's records, moved into `dump` at the wave's fit numbers
    double ms = 0, flops = 0, scan_ms = 0, scan_flops = 0;
    int launches = 0, scans = 0, rounds = 0;
    for (int t0 = 0; t0 < p->n_targets;) {
        long long cnt = per_t[t0];
        int t1 = t0 + 1;
        while (t1 < p->n_targets && cnt + per_t[t1] <= budget) cnt += per_t[t1++];
        std::vector<int> idx;
        for (int i = 0; i < n_fits; i++) if (target[i] >= t0 && target[i] < t1) idx.push_back(i);
        t0 = t1;
        if (idx.empty()) continue;
        const int m = (int)idx.size();
        std::vector<int> tg(m), fd(m), st(m), ns(m), it(m);
        std::vector<double> a(m), l(m), err(m);
        for (int j = 0; j < m; j++) { tg[j] = target[idx[j]]; fd[j] = fold[idx[j]]; a[j] = alpha[idx[j]]; l[j] = lambda[idx[j]]; }
        const int rc = run_fits_streaming(p, m, tg.data(), fd.data(), a.data(), l.data(), err.data(), st.data(), ns.data(), it.data(),
                                          dump ? &wave_dump : nullptr, cap);
        if (rc != PAREBEN_OK) return rc;
        for (int j = 0; j < m; j++) {
            if (dump) dump->copy_from(idx[j], wave_dump, j);
            if (fold_err) fold_err[idx[j]] = err[j];
            if (status) status[idx[j]] = st[j];
            if (n_selected) n_selected[idx[j]] = ns[j];
            if (n_iter) n_iter[idx[j]] = it[j];
        }
        ms += p->last_ms; flops += p->last_flops; launches += p->last_launches;
        scan_ms += p->last_scan_ms; scan_flops += p->last_scan_flops; scans += p->last_scan_launches; rounds += p->last_rounds;
    }
    p->last_ms = ms; p->last_flops = flops; p->last_launches = launches;
    p->last_scan_ms = scan_ms; p->last_scan_flops = scan_flops; p->last_scan_launches = scans; p->last_rounds = rounds;
    return PAREBEN_OK;
}

// target: response of each fit (0 .. n_targets - 1); null = response 0 for every fit
int run_fits_impl(pareben_problem *p, int n_fits, const int *target, const int *fold, const double *alpha, const double *lambda,
                  double *fold_err, int *status, int *n_selected, int *n_iter, DumpBuffers *dump)
{
    if (!p || n_fits < 0 || (n_fits > 0 && (!fold || !alpha || !lambda))) return fail(PAREBEN_EINVAL, "pareben_run_fits: bad argument");
    if (n_fits == 0) return PAREBEN_OK;
    std::vector<int> target0;
    if (!target) { target0.assign(n_fits, 0); target = target0.data(); }
    for (int i = 0; i < n_fits; i++)
        if (target[i] < 0 || target[i] >= p->n_targets) return fail(PAREBEN_EINVAL, "pareben_run_fits: target index out of range");
    if (p->streaming) return run_fits_streaming_waves(p, n_fits, target, fold, alpha, lambda, fold_err, status, n_selected, n_iter, dump);
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
        // groups: fits of one response that share (alpha, lambda) -- one row of the reference's ParameterGrid -- differ
        // only in the fold and cost about the same; the device scheduler prices a group by its first finished fit
        // (fit_kernel.cuh).  Another response's fits at the same point can cost quite differently, so they form their own group.
        std::map<std::tuple<int, double, double>, int> group_of;
        for (int i = 0; i < n_fits; i++) {
            if (fold[i] < 0 || fold[i] > p->n_folds || (p->n_folds > 0 && fold[i] == 0) || !p->h_folds[fold[i]].Xtr)
                return fail(PAREBEN_EINVAL, "pareben_run_fits: fold label not available in this problem");
            const auto key = std::make_tuple(target[i], alpha[i], lambda[i]);
            auto it = group_of.find(key);
            if (it == group_of.end()) it = group_of.emplace(key, (int)group_of.size()).first;
            tasks[i] = FitTask{fold[i], target[i], alpha[i], lambda[i], i, it->second};
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
        CU(cudaMemsetAsync(p->d_flops, 0, 3 * sizeof(double), p->stream));
        FitOutputs out;
        out.fold_err = d_err; out.status = d_ints; out.n_selected = d_ints + n_fits; out.n_iter = d_ints + 2 * n_fits;
        out.m_out = nullptr; out.used_out = nullptr; out.beta_out = nullptr; out.var_out = nullptr; out.scalars_out = nullptr;
        out.dump_ld = 0;
        out.flops = p->d_flops;
        char *d_dump = nullptr;
        if (dump) {
            dump->resize(n_fits, p->cap);
            d_dump = (char *)tmp_alloc(DumpBuffers::bytes(n_fits, p->cap));
            DumpBuffers::carve(d_dump, n_fits, p->cap, out);
        }
        Problem P;
        P.N = p->n; P.K = p->k; P.Kc = p->kc; P.n_folds = p->n_folds; P.epis = p->epis; P.prior = p->prior;
        P.cap = p->cap; P.nmax = p->nmax; P.tc = p->tc; P.folds = p->d_folds;
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
            CU((p->epis ? launch_fit_be : p->tc ? launch_fit_bt : launch_fit_bm)(grid, p->threads, p->stream, P, v, d_tasks, n_fits, sched, p->d_slabs, p->slab_stride, out));
        CU(cudaEventRecord(p->ev1, p->stream));
        std::vector<int> h_ints(3 * (size_t)n_fits);
        std::vector<double> h_err(n_fits);
        CU(cudaMemcpyAsync(h_err.data(), d_err, sizeof(double) * n_fits, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaMemcpyAsync(h_ints.data(), d_ints, sizeof(int) * 3 * n_fits, cudaMemcpyDeviceToHost, p->stream));
        double h_flops2[3] = {0, 0, 0};
        CU(cudaMemcpyAsync(h_flops2, p->d_flops, 3 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        if (dump) CU(cudaMemcpyAsync(dump->host.data(), d_dump, dump->host.size(), cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        const double h_flops = h_flops2[0];
        p->last_avoided = h_flops2[1];
        p->last_tc_calls = h_flops2[2];
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, p->ev0, p->ev1));
        p->last_ms = ms + p->gram_ms; p->last_flops = h_flops; p->last_launches = 1 + p->gram_launches;      // a call that had to build C pays for it
        for (int i = 0; i < n_fits; i++) {
            if (fold_err) fold_err[i] = h_err[i];
            if (status) status[i] = h_ints[i];
            if (n_selected) n_selected[i] = h_ints[n_fits + i];
            if (n_iter) n_iter[i] = h_ints[2 * (size_t)n_fits + i];
        }
        for (int i = 0; i < ns; i++) pool_give(p->device, scratch[i], scratch_bytes[i]);
    } catch (std::pair<int, std::string> &e) {
        for (int i = 0; i < ns; i++) pool_give(p->device, scratch[i], scratch_bytes[i]);
        return fail(e.first, e.second);
    } catch (std::bad_alloc &) {
        for (int i = 0; i < ns; i++) pool_give(p->device, scratch[i], scratch_bytes[i]);
        return fail(PAREBEN_ENOMEM, "host allocation of the fit records failed");
    }
    return PAREBEN_OK;
}

}  // namespace

extern "C" int pareben_run_fits(pareben_problem *p, int n_fits, const int *fold, const double *alpha,
                                const double *lambda, double *fold_err, int *status, int *n_selected, int *n_iter)
{
    return run_fits_impl(p, n_fits, nullptr, fold, alpha, lambda, fold_err, status, n_selected, n_iter, nullptr);
}

extern "C" int pareben_run_fits_multi(pareben_problem *p, int n_fits, const int *target, const int *fold, const double *alpha,
                                      const double *lambda, double *fold_err, int *status, int *n_selected, int *n_iter)
{
    if (n_fits > 0 && !target) return fail(PAREBEN_EINVAL, "pareben_run_fits_multi: bad argument");
    return run_fits_impl(p, n_fits, target, fold, alpha, lambda, fold_err, status, n_selected, n_iter, nullptr);
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

// One sub-shard of a grid call on one device: upload, lay out, run, scatter into the caller's tables.  Responses, grid
// points and folds are numbered as in pareben_cv_grid_multi.
int cv_grid_on_device(const double *basis, int n, int k, const double *targets, int n_targets, const int *fold_id, int n_folds,
                      const double *alpha, const double *lambda, int n_grid, int epis, int prior, int device,
                      int shard, int n_shards, double *fold_err, int *status, int *n_selected)
{
    const int rows = n_targets * n_grid, total = rows * n_folds;
    std::vector<int> mine(total);
    int m = 0;
    pareben_shard_plan(lambda, rows, n_folds, shard, n_shards, mine.data(), &m);
    if (m == 0) return PAREBEN_OK;
    pareben_problem *p = nullptr;
    const bool timing = getenv("PAREBEN_TIMING") != nullptr;
    auto t0 = std::chrono::steady_clock::now();
    int rc = pareben_problem_create_multi(&p, device, basis, n, k, targets, n_targets, fold_id, n_folds, epis, prior);
    if (rc != PAREBEN_OK) return rc;
    auto t1 = std::chrono::steady_clock::now();
    std::vector<int> tg(m), fold(m), st(m), ns(m);
    std::vector<double> a(m), l(m), err(m);
    for (int i = 0; i < m; i++) {
        const int fit = mine[i], row = fit / n_folds;
        tg[i] = row / n_grid; fold[i] = fit % n_folds + 1; a[i] = alpha[row]; l[i] = lambda[row];
    }
    p->grid_fits_hint = total;
    rc = run_fits_impl(p, m, tg.data(), fold.data(), a.data(), l.data(), err.data(), st.data(), ns.data(), nullptr, nullptr);
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
extern "C" int pareben_cv_grid_multi(const double *basis, int n, int k, const double *targets, int n_targets, const int *fold_id,
                                     int n_folds, const double *alpha, const double *lambda, int n_grid, int epis,
                                     int prior, int n_devices, int device, int shard, int n_shards, double *fold_err,
                                     int *status, int *n_selected)
{
    if (n_folds < 1 || n_grid < 1 || n_targets < 1 || !alpha || !lambda || !fold_err) return fail(PAREBEN_EINVAL, "pareben_cv_grid: bad argument");
    if ((long long)n_targets * n_grid * n_folds > 0x7fffffffLL) return fail(PAREBEN_EINVAL, "pareben_cv_grid: more than 2^31 - 1 fits");
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail(PAREBEN_EINVAL, "pareben_cv_grid: bad shard");
    const int visible = pareben_device_count();
    if (visible < 1) return fail(PAREBEN_ENODEVICE, "no usable CUDA device");
    if (n_devices == 0) n_devices = visible - device;                 // 0 = every device from `device` on
    if (device < 0 || n_devices < 1 || device + n_devices > visible) return fail(PAREBEN_ENODEVICE, "pareben_cv_grid: device range not available");
    if (n_devices == 1)
        return cv_grid_on_device(basis, n, k, targets, n_targets, fold_id, n_folds, alpha, lambda, n_grid, epis, prior, device,
                                 shard, n_shards, fold_err, status, n_selected);
    std::vector<int> rcs(n_devices, PAREBEN_OK);
    std::vector<std::string> msgs(n_devices);
    std::vector<std::thread> workers;
    for (int d = 0; d < n_devices; d++)
        workers.emplace_back([&, d] {
            rcs[d] = cv_grid_on_device(basis, n, k, targets, n_targets, fold_id, n_folds, alpha, lambda, n_grid, epis, prior, device + d,
                                       shard * n_devices + d, n_shards * n_devices, fold_err, status, n_selected);
            if (rcs[d] != PAREBEN_OK) msgs[d] = g_err;                // g_err is thread-local: carry the text back
        });
    for (std::thread &w : workers) w.join();
    for (int d = 0; d < n_devices; d++)
        if (rcs[d] != PAREBEN_OK) return fail(rcs[d], "device " + std::to_string(device + d) + ": " + msgs[d]);
    return PAREBEN_OK;
}

extern "C" int pareben_cv_grid(const double *basis, int n, int k, const double *target, const int *fold_id,
                               int n_folds, const double *alpha, const double *lambda, int n_grid, int epis,
                               int prior, int n_devices, int device, int shard, int n_shards, double *fold_err,
                               int *status, int *n_selected)
{
    return pareben_cv_grid_multi(basis, n, k, target, 1, fold_id, n_folds, alpha, lambda, n_grid, epis, prior, n_devices, device,
                                 shard, n_shards, fold_err, status, n_selected);
}

namespace {

// Bound on the effects of one fit's record: the cached kernels' basis cap (the one in use once the slabs exist), or the
// largest cap a streaming call can get; the binomial intercept slot is not an effect.
int max_effects_of(const pareben_problem *p)
{
    if (p->streaming) return stream_cap_bound(p);
    const int cap = p->d_slabs ? p->cap : cached_cap(p);
    return p->prior == PAREBEN_BINOMIAL ? cap - 1 : cap;
}

}  // namespace

extern "C" int pareben_max_effects(pareben_problem *p, int *max_effects)
{
    if (!p || !max_effects) return fail(PAREBEN_EINVAL, "pareben_max_effects: bad argument");
    *max_effects = max_effects_of(p);
    return PAREBEN_OK;
}

extern "C" int pareben_fit_batch(pareben_problem *p, int n_fits, const int *target, const int *fold, const double *alpha,
                                 const double *lambda, int max_effects, int *n_effects, int *cand, double *beta, double *var,
                                 double *scalars, int *status, double *fold_err)
{
    if (!p || n_fits < 0 || (n_fits > 0 && (!target || !fold || !alpha || !lambda)))
        return fail(PAREBEN_EINVAL, "pareben_fit_batch: bad argument");
    if (n_fits == 0) return PAREBEN_OK;
    if (max_effects < max_effects_of(p))
        return fail(PAREBEN_EINVAL, "pareben_fit_batch: max_effects is below pareben_max_effects (" + std::to_string(max_effects_of(p)) + ")");
    if (max_effects > 0 && (!n_effects || !cand || !beta)) return fail(PAREBEN_EINVAL, "pareben_fit_batch: n_effects, cand and beta are required");
    DumpBuffers dump;
    std::vector<int> st;
    std::vector<double> err;
    try { st.resize(n_fits); err.resize(n_fits); } catch (std::bad_alloc &) { return fail(PAREBEN_ENOMEM, "pareben_fit_batch: host allocation failed"); }
    const int rc = run_fits_impl(p, n_fits, target, fold, alpha, lambda, err.data(), st.data(), nullptr, nullptr, &dump);
    if (rc != PAREBEN_OK) return rc;
    for (int i = 0; i < n_fits; i++)
        if (dump.m(i) < 0 || dump.m(i) > max_effects) return fail(PAREBEN_ECUDA, "pareben_fit_batch: a record has more effects than its stride");
    const size_t me = (size_t)max_effects;
    for (int i = 0; i < n_fits; i++) {
        const int M = dump.m(i);
        if (n_effects) n_effects[i] = M;
        if (cand) { std::copy(dump.used(i), dump.used(i) + M, cand + i * me); std::fill(cand + i * me + M, cand + (i + 1) * me, 0); }
        if (beta) { std::copy(dump.beta(i), dump.beta(i) + M, beta + i * me); std::fill(beta + i * me + M, beta + (i + 1) * me, 0.0); }
        if (var) { std::copy(dump.var(i), dump.var(i) + M, var + i * me); std::fill(var + i * me + M, var + (i + 1) * me, 0.0); }
        if (scalars) std::copy(dump.scalars(i), dump.scalars(i) + 4, scalars + 4 * (size_t)i);
        if (status) status[i] = st[i];
        if (fold_err) fold_err[i] = fold[i] == 0 ? 0.0 : err[i];      // an all-rows fit has no held-out rows to score
    }
    return PAREBEN_OK;
}

// The one-fit case of pareben_fit_batch, expanded into the reference's table layouts.
extern "C" int pareben_fit(pareben_problem *p, double alpha, double lambda, double *beta_table, double *wald,
                           double *intercept, double *extra, int *status)
{
    if (!p || !beta_table) return fail(PAREBEN_EINVAL, "pareben_fit: bad argument");
    if (p->n_folds != 0) return fail(PAREBEN_EINVAL, "pareben_fit needs a problem created with n_folds == 0");
    if (p->n_targets != 1) return fail(PAREBEN_EINVAL, "pareben_fit needs a problem with one response");
    int me = 0;
    pareben_max_effects(p, &me);
    std::vector<int> used(me);           // one record: candidate ids in Used order, mu/scale, sigma_ii/scale^2
    std::vector<double> beta(me), var(me);
    double sc[4] = {0, 0, 0, 0};
    const int target = 0, fold = 0;
    int M = 0, st = 0;
    const int rc = pareben_fit_batch(p, 1, &target, &fold, &alpha, &lambda, me, &M, used.data(), beta.data(), var.data(), sc, &st, nullptr);
    if (rc != PAREBEN_OK) return rc;
    const int k = p->k, kc = p->kc;
    if (p->prior == PAREBEN_GAUSSIAN) {
        const int ncol = p->epis ? 5 : 4;
        // loci columns (MainEff.c:87-91, NeFull2.c:100-134)
        for (int c = 0; c < k; c++) { beta_table[c] = c + 1; beta_table[(size_t)kc + c] = c + 1; }
        if (p->epis) { size_t kk = k; for (int i = 0; i < k - 1; i++) for (int j = i + 1; j < k; j++, kk++) { beta_table[kk] = i + 1; beta_table[(size_t)kc + kk] = j + 1; } }
        for (size_t z = (size_t)2 * kc; z < (size_t)ncol * kc; z++) beta_table[z] = 0;
        for (int i = 0; i < M; i++) {
            const int c = used[i] - 1;
            beta_table[(size_t)2 * kc + c] = beta[i];
            beta_table[(size_t)3 * kc + c] = var[i];
            if (p->epis) beta_table[(size_t)4 * kc + c] = used[i];
        }
        if (intercept) intercept[0] = sc[1];
    } else {
        if (!p->epis) {      // k x 4 indexed by column id (NEmainEff.c:270-291, 364-371)
            for (int c = 0; c < k; c++) { beta_table[c] = c + 1; beta_table[(size_t)k + c] = c + 1; beta_table[(size_t)2 * k + c] = 0; beta_table[(size_t)3 * k + c] = 0; }
            for (int i = 0; i < M; i++) { const int c = used[i] - 1; beta_table[(size_t)2 * k + c] = beta[i]; beta_table[(size_t)3 * k + c] = var[i]; }
        } else {             // compact 2k x 4 in Used order with decoded loci (NeFull.c:168-208)
            const int rows = 2 * k;
            for (size_t z = 0; z < (size_t)4 * rows; z++) beta_table[z] = 0;
            for (int i = 0; i < M && i < rows; i++) {
                const int c = used[i] - 1;
                int li = c, lj = c;
                if (c >= k) { long long pp = (long long)c - k; int ii = 0; while ((long long)(ii + 1) * (2LL * k - (ii + 1) - 1) / 2 <= pp) ii++; li = ii; lj = (int)(pp - (long long)ii * (2LL * k - ii - 1) / 2) + ii + 1; }
                beta_table[i] = li + 1; beta_table[(size_t)rows + i] = lj + 1;
                beta_table[(size_t)2 * rows + i] = beta[i]; beta_table[(size_t)3 * rows + i] = var[i];
            }
        }
        if (intercept) { intercept[0] = sc[1]; intercept[1] = sc[2]; }
    }
    if (wald) wald[0] = sc[0];
    if (extra) extra[0] = sc[3];
    if (status) status[0] = st;
    return PAREBEN_OK;
}

// The grid call on a problem that is already resident (one upload serves BuildGrid's lambda_max, the grid and any
// LocalSearch refinement): same table layout and shard assignment as pareben_cv_grid_multi.
extern "C" int pareben_problem_cv_grid_multi(pareben_problem *p, const double *alpha, const double *lambda, int n_grid, int shard,
                                             int n_shards, double *fold_err, int *status, int *n_selected)
{
    if (!p || !alpha || !lambda || !fold_err || n_grid < 1) return fail(PAREBEN_EINVAL, "pareben_problem_cv_grid: bad argument");
    if (p->n_folds < 1) return fail(PAREBEN_EINVAL, "pareben_problem_cv_grid needs a problem created with folds");
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail(PAREBEN_EINVAL, "pareben_problem_cv_grid: bad shard");
    if ((long long)p->n_targets * n_grid * p->n_folds > 0x7fffffffLL) return fail(PAREBEN_EINVAL, "pareben_problem_cv_grid: more than 2^31 - 1 fits");
    const int nf = p->n_folds, rows = p->n_targets * n_grid, total = rows * nf;
    std::vector<int> mine(total);
    int m = 0;
    int rc = pareben_shard_plan(lambda, rows, nf, shard, n_shards, mine.data(), &m);
    if (rc != PAREBEN_OK || m == 0) return rc;
    std::vector<int> tg(m), fold(m), st(m), ns(m);
    std::vector<double> a(m), l(m), err(m);
    for (int i = 0; i < m; i++) {
        const int row = mine[i] / nf;
        tg[i] = row / n_grid; fold[i] = mine[i] % nf + 1; a[i] = alpha[row]; l[i] = lambda[row];
    }
    p->grid_fits_hint = total;
    rc = run_fits_impl(p, m, tg.data(), fold.data(), a.data(), l.data(), err.data(), st.data(), ns.data(), nullptr, nullptr);
    p->grid_fits_hint = 0;
    if (rc != PAREBEN_OK) return rc;
    for (int i = 0; i < m; i++) {
        fold_err[mine[i]] = err[i];
        if (status) status[mine[i]] = st[i];
        if (n_selected) n_selected[mine[i]] = ns[i];
    }
    return PAREBEN_OK;
}

extern "C" int pareben_problem_cv_grid(pareben_problem *p, const double *alpha, const double *lambda, int n_grid, int shard,
                                       int n_shards, double *fold_err, int *status, int *n_selected)
{
    if (p && p->n_targets != 1) return fail(PAREBEN_EINVAL, "pareben_problem_cv_grid: the problem holds several responses (use pareben_problem_cv_grid_multi)");
    return pareben_problem_cv_grid_multi(p, alpha, lambda, n_grid, shard, n_shards, fold_err, status, n_selected);
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

namespace {
template <bool EPIS>
void launch_lambda_max(int T, int nb, cudaStream_t s, const double *X, int n, int k, int c0, int c1, const double *resp, double *out)
{   // response tile: 1 (a single response keeps the FMA pipe for itself), else the smallest of 4 / 8 / 16 that covers T
    if (T == 1) lambda_max_multi_kernel<EPIS, 1><<<nb, LM_THREADS, 0, s>>>(X, n, k, c0, c1, resp, T, out);
    else if (T <= 4) lambda_max_multi_kernel<EPIS, 4><<<nb, LM_THREADS, 0, s>>>(X, n, k, c0, c1, resp, T, out);
    else if (T <= 8) lambda_max_multi_kernel<EPIS, 8><<<nb, LM_THREADS, 0, s>>>(X, n, k, c0, c1, resp, T, out);
    else lambda_max_multi_kernel<EPIS, 16><<<nb, LM_THREADS, 0, s>>>(X, n, k, c0, c1, resp, T, out);
}
}  // namespace

extern "C" int pareben_lambda_max_multi(pareben_problem *p, double *lambda_max)
{
    if (!p || !lambda_max) return fail(PAREBEN_EINVAL, "pareben_lambda_max: bad argument");
    try {
        CU(cudaSetDevice(p->device));
        // GetLambdaMax works on ALL rows (R/BuildGrid.R:5-32): build a row-major copy once.
        const int n = p->n, k = p->k, T = p->n_targets;
        std::vector<double> y((size_t)n * T), centred((size_t)n * T), resp((size_t)n * T);
        CU(cudaMemcpy(y.data(), p->d_y, sizeof(double) * n * T, cudaMemcpyDeviceToHost));
        for (int r = 0; r < T; r++) {
            const double *yr = y.data() + (size_t)r * n;
            double *cr = centred.data() + (size_t)r * n, *rr = resp.data() + (size_t)r * n;
            long double s = 0; for (int i = 0; i < n; i++) s += yr[i];
            long double mean = s / n, t = 0; for (int i = 0; i < n; i++) t += (yr[i] - mean);
            mean += t / n;
            long double ss = 0;
            for (int i = 0; i < n; i++) { cr[i] = (double)(yr[i] - (double)mean); ss += (long double)cr[i] * cr[i]; }
            const double nrm = std::sqrt((double)ss);
            for (int i = 0; i < n; i++) rr[i] = cr[i] / nrm;
        }
        // scratch comes from the problem's pooled allocations (returned to the pool with the problem; nothing to leak on error)
        double *d_rows_x = p->dalloc<double>((size_t)n * k), *d_resp = p->dalloc<double>((size_t)n * T);
        double *d_max = p->dalloc<double>(T);
        int *d_rows = p->dalloc<int>(n);
        std::vector<int> rows(n); for (int i = 0; i < n; i++) rows[i] = i;
        CU(cudaMemcpy(d_rows, rows.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
        CU(cudaMemsetAsync(d_max, 0, sizeof(double) * T, p->stream));
        gather_rows_kernel<<<dim3((n + 31) / 32, (k + 31) / 32), dim3(32, 8), 0, p->stream>>>(p->d_Xcol, n, k, d_rows, n, d_rows_x);
        auto pass = [&](int c0, int c1, const std::vector<double> &r, bool epis) {
            const int nb = (c1 - c0 + LM_THREADS - 1) / LM_THREADS;
            if (nb <= 0) return;
            CU(cudaMemcpyAsync(d_resp, r.data(), sizeof(double) * n * T, cudaMemcpyHostToDevice, p->stream));
            (epis ? launch_lambda_max<true> : launch_lambda_max<false>)(T, nb, p->stream, d_rows_x, n, k, c0, c1, d_resp, d_max);
            CU(cudaGetLastError());
            CU(cudaStreamSynchronize(p->stream));      // r may be the next pass's source
        };
        pass(0, k, resp, false);                       // main effects against the normalised response (:14-19)
        if (p->epis) pass(k, p->kc, centred, true);    // pairs against the UN-normalised centred response (:24-27)
        std::vector<double> hm(T);
        CU(cudaMemcpyAsync(hm.data(), d_max, sizeof(double) * T, cudaMemcpyDeviceToHost, p->stream));
        CU(cudaStreamSynchronize(p->stream));
        const double floor_ = std::log(1.1);
        for (int r = 0; r < T; r++) lambda_max[r] = hm[r] > floor_ ? hm[r] : floor_;
    } catch (std::pair<int, std::string> &e) {
        return fail(e.first, e.second);
    }
    return PAREBEN_OK;
}

extern "C" int pareben_lambda_max(pareben_problem *p, double *lambda_max)
{
    if (p && p->n_targets != 1) return fail(PAREBEN_EINVAL, "pareben_lambda_max: the problem holds several responses (use pareben_lambda_max_multi)");
    return pareben_lambda_max_multi(p, lambda_max);
}

extern "C" int pareben_sl_filter(pareben_problem *p, double tau_main, double tau_pair, int capacity, int *cand, double *stat,
                                 int *n_kept)
{
    if (!p || !n_kept || capacity < 0) return fail(PAREBEN_EINVAL, "pareben_sl_filter: bad argument");
    if (p->n_targets != 1) return fail(PAREBEN_EINVAL, "pareben_sl_filter needs a problem with one response");
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
// blocks and over the five kernel variants.  out: PH_COUNT cycle totals then PH_COUNT call counts.
#ifdef PAREBEN_PHASE_TIMING
extern "C" int pareben_phase_cycles(unsigned long long *out, int reset)
{
    unsigned long long acc[2 * PH_COUNT] = {0}, one[2 * PH_COUNT];
    void (*fn[5])(unsigned long long *, int, unsigned long long *, unsigned long long *, int *, int) = {timing_gm, timing_ge, timing_bm, timing_be, timing_bt};
    for (int i = 0; i < 5; i++) {
        for (int j = 0; j < 2 * PH_COUNT; j++) one[j] = 0;
        fn[i](one, reset, nullptr, nullptr, nullptr, 0);
        for (int j = 0; j < 2 * PH_COUNT; j++) acc[j] += one[j];
    }
    if (out) for (int j = 0; j < 2 * PH_COUNT; j++) out[j] = acc[j];
    return PH_COUNT;
}

// experiments only: per-fit start/end (%globaltimer ns) and block id of the last launch of variant
// `which` (0 gm, 1 ge, 2 bm, 3 be, 4 bt).
extern "C" int pareben_fit_trace(int which, unsigned long long *t0, unsigned long long *t1, int *block, int n)
{
    void (*fn[5])(unsigned long long *, int, unsigned long long *, unsigned long long *, int *, int) = {timing_gm, timing_ge, timing_bm, timing_be, timing_bt};
    if (which < 0 || which > 4) return 0;
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

extern "C" int pareben_last_contraction_info(pareben_problem *p, int *tensor_core, double *tc_contractions)
{
    if (!p) return fail(PAREBEN_EINVAL, "null problem");
    if (tensor_core) *tensor_core = p->tc;
    if (tc_contractions) *tc_contractions = p->last_tc_calls;
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
