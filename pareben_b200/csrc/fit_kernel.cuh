// fit_kernel.cuh -- the persistent batched-fit kernel and its per-variant host launchers.
// Each of the four (Epis, prior) variants is compiled in its own translation unit (fit_gm.cu,
// fit_ge.cu, fit_bm.cu, fit_be.cu) so that the build runs four ptxas jobs in parallel; the host
// side (pareben.cu) reaches them through the plain functions declared in fit_launch.h.
#pragma once
#include "common.cuh"
#include "gauss_fit.cuh"
#include "binom_fit.cuh"
#include "fit_launch.h"

namespace pareben {

// the persistent batched-fit kernel: one block = one fit at a time, fits pulled from a queue
#ifndef PAREBEN_MIN_BLOCKS
#define PAREBEN_MIN_BLOCKS 2
#endif
constexpr int FIT_THREADS = FIT_T;     // compile-time maximum (register budget: 2 x 256 or 4 x 128 threads per SM)

constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int SWEEP_DOUBLES = SWEEP_SMEM_M * SWEEP_SMEM_M + 2 * SWEEP_SMEM_M;
constexpr int QUAD_DOUBLES = cmax(2 * QT * LDS_V + 784, cmax(4096 + 1040, GRAM_PIPE_DOUBLES));
constexpr int S_BUF_DOUBLES = cmax(cmax(cmax(SWEEP_DOUBLES, SWEEP_PANEL_DOUBLES), cmax(SV_DOUBLES, COL_MAX_ROWS)), cmax(GRAM_DOUBLES, QUAD_DOUBLES));
constexpr size_t S_BUF_BYTES = (size_t)S_BUF_DOUBLES * sizeof(double);

__device__ inline unsigned long long sched_now()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// Longest-predicted-first task selection with on-line cost learning.  Fit cost varies > 100x over the grid and does
// not follow lambda alone (it peaks where the active set and the iteration count are both large), so a queue in a fixed
// order leaves most SMs idle behind a few long fits started late.  Here a block that needs work scans the unclaimed
// tasks and takes the one with the largest predicted cost:
//   * a group (grid point) none of whose fits has started: top priority, in host order (rising lambda) -- every
//     group gets a pilot as early as possible;
//   * a group whose pilot is still running: the pilot's elapsed time so far (a lower bound that keeps growing, so
//     the siblings of long fits are pulled forward while the pilot is still busy);
//   * a group with a finished fit: the longest finished duration.
// The first pull of a block is its own index (tasks arrive with the pilots first), which avoids a start-up stampede.
// The result table does not depend on the schedule: every fit is computed by one block on its own.
__device__ inline int next_task(const FitTask *__restrict__ tasks, int n_tasks, const Sched &sd, bool first, const Scratch &sc,
                                int *s_pick)
{
    const int T = blockDim.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
    volatile int *taken = sd.taken;
    volatile unsigned long long *cost = sd.cost, *tstart = sd.t_start;
    for (int attempt = 0;; attempt++) {
        int pick = -1;
        if (first && attempt == 0) {
            pick = (int)blockIdx.x < n_tasks ? (int)blockIdx.x : -1;
        } else {
            const unsigned long long now = sched_now();
            unsigned long long bp = 0; int bi = 0x7fffffff;
            for (int i = threadIdx.x; i < n_tasks; i += T) {
                if (taken[i]) continue;
                const int g = tasks[i].group;
                const unsigned long long c = cost[g], t0 = tstart[g];
                unsigned long long prio;
                if (c) prio = c + 1;
                else if (t0) prio = (now > t0 ? now - t0 : 0) + 1;
                else prio = (1ull << 62) - (unsigned long long)i;
                if (prio > bp || (prio == bp && i < bi)) { bp = prio; bi = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long p2 = __shfl_xor_sync(0xffffffffu, bp, o);
                const int i2 = __shfl_xor_sync(0xffffffffu, bi, o);
                if (p2 > bp || (p2 == bp && i2 < bi)) { bp = p2; bi = i2; }
            }
            __syncthreads();
            unsigned long long *redp = reinterpret_cast<unsigned long long *>(sc.red);
            if (lane == 0) { redp[wid] = bp; sc.redi[wid] = bi; }
            __syncthreads();
            bp = 0; bi = 0x7fffffff;
            for (int w = 0; w < nw; w++) {
                const unsigned long long p2 = redp[w]; const int i2 = sc.redi[w];
                if (p2 > bp || (p2 == bp && i2 < bi)) { bp = p2; bi = i2; }
            }
            pick = bp ? bi : -1;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int got = -1;
            if (pick >= 0) {
                if (atomicCAS(sd.taken + pick, 0, 1) == 0) {
                    got = pick;
                    atomicCAS(sd.t_start + tasks[pick].group, 0ull, sched_now());
                } else got = -2;                                   // lost the race: look again
            }
            *s_pick = got;
        }
        __syncthreads();
        const int got = *s_pick;
        if (got != -2) return got;
    }
}

template <bool EPIS, bool BINOMIAL>
__global__ void __launch_bounds__(FIT_THREADS, PAREBEN_MIN_BLOCKS)
eben_fit_kernel(Problem P, Variant v, const FitTask *__restrict__ tasks, int n_tasks, Sched sched, char *slabs,
                size_t slab_stride, FitOutputs out)
{
    // One shared buffer (dynamic: it exceeds the 48 KB static limit), used by phases that never overlap: the
    // cp.async ring of the contraction, the resident SIGMA tile of the quadratic forms, the Gram partial tiles
    // and the pivot columns of the register sweep.
    extern __shared__ __align__(32) double s_buf[];
    double *sV = s_buf;
    __shared__ double red[66];
    __shared__ int redi[66];
    __shared__ int s_task;
    Scratch sc{red, redi, s_buf};
    for (bool first = true;; first = false) {
        const int ti = next_task(tasks, n_tasks, sched, first, sc, &s_task);
        if (ti < 0) break;
        const FitTask task = tasks[ti];
        const unsigned long long t_fit0 = sched_now();
        const FoldData F = P.folds[task.fold];
        Slab s = carve_slab(slabs + (size_t)blockIdx.x * slab_stride, P.cap, P.nmax, P.Kc);
#ifdef PAREBEN_PHASE_TIMING
        if (threadIdx.x == 0 && task.out_index < FIT_TRACE_MAX) { g_fit_t0[task.out_index] = global_ns(); g_fit_block[task.out_index] = blockIdx.x; }
#endif
        if (BINOMIAL) binom_fit<EPIS>(P, F, v, s, task.lambda, task.alpha, task, out, sV, sc);
        else gauss_fit<EPIS>(P, F, v, s, task.lambda, task.alpha, task, out, sV, sc);
        if (threadIdx.x == 0) atomicMax(sched.cost + task.group, sched_now() - t_fit0 + 1);
#ifdef PAREBEN_PHASE_TIMING
        if (threadIdx.x == 0 && task.out_index < FIT_TRACE_MAX) g_fit_t1[task.out_index] = global_ns();
#endif
    }
}


// Gram organisation of the Gaussian fits (FoldData::C): row p of C is the cache row x_c' phi_p / s_c of candidate p as
// basis, for every candidate -- what CacheBP* (MainEff.c:1144-1201) and ActionAdd* (:1608-1618) compute again for every
// basis of every fit although it depends on the fold alone.  One launch builds the rows of all listed folds: a block
// takes 32 candidates at a time, writes their normalised columns (exactly the column an add would build, :1590-1606 /
// NeFull2.c:277-290) into its own slab's PHI and runs the same tensor-core contraction a fit runs at the top of an outer
// iteration, with C's rows as destinations.  2 N Kc^2 flops per fold, once per problem.
constexpr int GRAM_CHUNK = 8 * NT_MAX;

template <bool EPIS>
__global__ void __launch_bounds__(FIT_THREADS, PAREBEN_MIN_BLOCKS)
fold_gram_kernel(Problem P, const int *__restrict__ fold_list, int n_fold_list, char *slabs, size_t slab_stride, int *next_item)
{
    extern __shared__ __align__(32) double s_buf[];
    __shared__ int s_item;
    const int K = P.K, Kc = P.Kc, T = blockDim.x;
    const int chunks = (Kc + GRAM_CHUNK - 1) / GRAM_CHUNK;
    const int n_items = chunks * n_fold_list;
    Slab s = carve_slab(slabs + (size_t)blockIdx.x * slab_stride, P.cap, P.nmax, Kc);
    const int rpb = min(GRAM_CHUNK, P.cap);            // right-hand sides per contraction: the slab's PHI holds `cap` columns
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_item = atomicAdd(next_item, 1);
        __syncthreads();
        const int item = s_item;
        if (item >= n_items) break;
        const FoldData F = P.folds[fold_list[item / chunks]];
        const int N = F.ntr, LD = phi_ld(N);
        const int p_begin = (item % chunks) * GRAM_CHUNK, p_end = min(p_begin + GRAM_CHUNK, Kc);
        for (int p0 = p_begin; p0 < p_end; p0 += rpb) {
            const int R = min(rpb, p_end - p0);
            __syncthreads();
            for (int r = threadIdx.x & 31; r < R; r += 32) {             // a lane owns a column: one decode, coalesced row reads
                Cand<EPIS> cd(p0 + r, K);
                const double sc_p = F.scale[p0 + r], isc = 1 / sc_p;
                const bool pair = cd.i != cd.j;
                double *col = s.phi + (size_t)r * LD;
                for (int h = threadIdx.x >> 5; h < LD; h += T >> 5) {
                    double val = 0.0;
                    if (h < N) { const double x = cd.at(F.Xtr + (size_t)h * K); val = pair ? x / sc_p : x * isc; }
                    col[h] = val;
                }
            }
            __syncthreads();
            contract_x<EPIS>(F, K, Kc, R, R,
                [&](int r) -> const double * { return s.phi + (size_t)r * LD; },
                [&](int r, bool &dv) -> double * { dv = true; return F.C + (size_t)(p0 + r) * Kc; }, s_buf);
        }
    }
}

template <bool EPIS>
inline cudaError_t launch_gram_variant(int grid, int threads, cudaStream_t stream, const Problem &P, const int *fold_list,
                                       int n_fold_list, char *slabs, size_t slab_stride, int *next_item)
{
    cudaError_t e = cudaFuncSetAttribute(fold_gram_kernel<EPIS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S_BUF_BYTES);
    if (e != cudaSuccess) return e;
    fold_gram_kernel<EPIS><<<grid, threads, S_BUF_BYTES, stream>>>(P, fold_list, n_fold_list, slabs, slab_stride, next_item);
    return cudaGetLastError();
}

template <bool EPIS, bool BINOMIAL>
inline cudaError_t launch_fit_variant(int grid, int threads, cudaStream_t stream, const Problem &P, const Variant &v,
                                      const FitTask *tasks, int n_tasks, const Sched &sched, char *slabs, size_t slab_stride,
                                      const FitOutputs &out)
{
    cudaError_t e = cudaFuncSetAttribute(eben_fit_kernel<EPIS, BINOMIAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S_BUF_BYTES);
    if (e != cudaSuccess) return e;
    eben_fit_kernel<EPIS, BINOMIAL><<<grid, threads, S_BUF_BYTES, stream>>>(P, v, tasks, n_tasks, sched, slabs, slab_stride, out);
    return cudaGetLastError();
}

template <bool EPIS, bool BINOMIAL>
inline cudaError_t occupancy_variant(int *blocks_per_sm, int threads)
{
    cudaError_t e = cudaFuncSetAttribute(eben_fit_kernel<EPIS, BINOMIAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S_BUF_BYTES);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, eben_fit_kernel<EPIS, BINOMIAL>, threads, S_BUF_BYTES);
}

// experiments only (timing build): copy out / reset this translation unit's phase counters and fit trace
inline void timing_variant(unsigned long long *cycles_calls, int reset, unsigned long long *t0, unsigned long long *t1, int *block, int n)
{
#ifdef PAREBEN_PHASE_TIMING
    if (cycles_calls) { cudaMemcpyFromSymbol(cycles_calls, g_phase_cycles, sizeof(unsigned long long) * PH_COUNT);
                        cudaMemcpyFromSymbol(cycles_calls + PH_COUNT, g_phase_calls, sizeof(unsigned long long) * PH_COUNT); }
    if (reset) { unsigned long long z[PH_COUNT] = {0}; cudaMemcpyToSymbol(g_phase_cycles, z, sizeof z); cudaMemcpyToSymbol(g_phase_calls, z, sizeof z); }
    if (t0 && n > 0) {
        if (n > FIT_TRACE_MAX) n = FIT_TRACE_MAX;
        cudaMemcpyFromSymbol(t0, g_fit_t0, sizeof(unsigned long long) * n);
        cudaMemcpyFromSymbol(t1, g_fit_t1, sizeof(unsigned long long) * n);
        cudaMemcpyFromSymbol(block, g_fit_block, sizeof(int) * n);
    }
#else
    (void)cycles_calls; (void)reset; (void)t0; (void)t1; (void)block; (void)n;
#endif
}

}  // namespace pareben

#define PAREBEN_DEFINE_VARIANT(NAME, EPIS, BINOMIAL)                                                                      \
    namespace pareben {                                                                                                   \
    cudaError_t launch_fit_##NAME(int grid, int threads, cudaStream_t stream, const Problem &P, const Variant &v,        \
                                  const FitTask *tasks, int n_tasks, const Sched &sched, char *slabs, size_t slab_stride,         \
                                  const FitOutputs &out)                                                                  \
    { return launch_fit_variant<EPIS, BINOMIAL>(grid, threads, stream, P, v, tasks, n_tasks, sched, slabs, slab_stride, out); } \
    cudaError_t occupancy_##NAME(int *blocks_per_sm, int threads) { return occupancy_variant<EPIS, BINOMIAL>(blocks_per_sm, threads); } \
    void timing_##NAME(unsigned long long *cc, int reset, unsigned long long *t0, unsigned long long *t1, int *block, int n) \
    { timing_variant(cc, reset, t0, t1, block, n); }                                                                      \
    }

#define PAREBEN_DEFINE_GRAM(NAME, EPIS)                                                                                   \
    namespace pareben {                                                                                                   \
    cudaError_t launch_gram_##NAME(int grid, int threads, cudaStream_t stream, const Problem &P, const int *fold_list,   \
                                   int n_fold_list, char *slabs, size_t slab_stride, int *next_item)                      \
    { return launch_gram_variant<EPIS>(grid, threads, stream, P, fold_list, n_fold_list, slabs, slab_stride, next_item); } \
    }
