// common.cuh -- shared device-side definitions for the batched EBEN fit kernels (sm_100a).
//
// Execution model: ONE thread block runs ONE complete EBEN fit (one (fold, alpha, lambda)
// point of R/CrossValidate.R's grid) from initialisation to hold-out error, entirely on the
// device; a grid of persistent blocks (a multiple of the 148 SMs) pulls fits from an atomic
// queue ordered by expected cost.  All blocks share the per-fold training matrices, which are
// small enough to stay resident in the 126 MB L2, so the score contractions stream them from
// L2 rather than HBM.  Per-fit state (active-set inverse, candidate cache, statistics) lives
// in a per-block slab of global memory plus shared memory for the hot vectors.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

namespace pareben {

enum : int { ACT_REEST = 0, ACT_ADD = 1, ACT_DEL = -1, ACT_TERM = 10, ACT_NONE = -10 };

// status bits, mirrored in include/pareben.h
enum : int { ST_CAP = 1, ST_NOT_PD = 2, ST_NONFINITE = 4, ST_ITER_MAX = 8 };

// Constants that differ between the four reference translation units (SURVEY.md Appendix A).
struct Variant {
    int epis;
    int binomial;
    double n_add;            // block threshold factor
    double ml_delta;         // minimum worthwhile delta-ML
    double reest_tol;        // |dlog alpha| below which a lone re-estimate terminates
    double init_alpha_max;
    double init_alpha_min;
};

struct FoldData {
    const double *Xtr;       // [ntr][K] row-major training rows
    const int8_t *Xtr8;      // same matrix as int8 when every entry is a small integer (genotype codes), else null
    const double *ytr;       // [ntr]
    const double *Xte;       // [nte][K] row-major held-out rows
    const double *yte;       // [nte]
    const double *scale;     // [Kc] column norms of the training rows (1 where the column is all zero)
    // column-major (transposed) copies for the tensor-core contraction: column k at XT + k*ldt, rows zero-padded
    // to ldt (a multiple of 64).  Exactly one of the two is non-null (int8 when Xtr8 is).
    const int8_t *XT8;
    const double *XTd;
    int ldt;
    int ntr, nte;
    // Gaussian fits, "Gram" organisation (null otherwise): C[p][c] = x_c' phi_p / s_c for EVERY candidate p, i.e. the
    // row the reference's CacheBP* (MainEff.c:1144-1201) would compute for basis p.  It depends on the fold only -- not
    // on alpha, lambda or the solver's state -- so it is built once per fold (fold_gram_kernel) and shared by all fits.
    double *C;
    // Binomial main-effect fits on designs of integers with |x| <= 11 (null otherwise): the transposed training matrix and
    // its elementwise square as int8 operand images of the tensor-core score contraction (tc_contract.cuh), zero-padded
    // to whole 128-candidate tiles and 32-row stages.
    const int8_t *Xtc, *Xtcsq;
};

struct Problem {
    int N, K, Kc, n_folds, epis, prior;
    int cap;                 // basis cap actually used (<= the reference's basisMax)
    int nmax;                // max ntr over folds
    int tc;                  // 1 when the folds carry the int8 operand images (FoldData::Xtc): the slabs then hold digit planes
    // [n_targets][n_folds + 1]; fold index 0 = all rows, f = rows with fold_id != f.  The records of one fold differ
    // only in ytr / yte (one response each) and share every design-side buffer, so whatever depends on the design alone
    // (the Gram build, the streaming scan) indexes folds[f], the records of response 0.
    const FoldData *folds;
};

// target: the response the fit trains on; its data are P.folds[target * (n_folds + 1) + fold] (see Problem::folds)
struct FitTask { int fold, target; double alpha, lambda; int out_index; int group; };

// Device-side scheduler state of one launch (see next_task() in fit_kernel.cuh).  Fits that differ only in the
// fold (same alpha, lambda: one row of the reference's ParameterGrid, R/CrossValidate.R:66) form a group and
// cost about the same, so the first fit of a group to run is the pilot that prices its siblings.
struct Sched {
    int *taken;                      // [n_tasks] 0 = free, 1 = claimed
    unsigned long long *t_start;     // [n_groups] %globaltimer at which the group's first fit started (0 = none yet)
    unsigned long long *cost;        // [n_groups] longest finished fit of the group in ns (0 = none yet)
};

struct FitOutputs {
    double *fold_err;        // [n] indexed by out_index
    int *status, *n_selected, *n_iter;
    // optional full-model dump for pareben_fit (batch of 1)
    int *m_out; int *used_out; double *beta_out; double *var_out; double *scalars_out; // wald, intercept0, intercept1, extra
    double *flops;           // three accumulators (atomicAdd): [0] model flops (SURVEY 8d), [1] the part the Gram organisation avoided,
                             // [2] score contractions run on the int8 tensor cores
};

// Per-block slab carved out of one big allocation.
struct Slab {
    double *sigma, *sigma_new, *H;      // cap*cap each
    double *ptp;                        // cap*cap (leading dimension cap): PHI'PHI of the Gaussian fit, maintained incrementally
    double *phi;                        // phi_ld(nmax) * cap, column-major (column j at phi + j*phi_ld(N), pad rows zero)
    double *phit;                       // (nmax + 32) * PHIT_LD: row-major copy of the first PHIT_LD active columns (binomial IRLS)
    double *G;                          // cap * Kc: physical rows, row r at G + r*Kc
    double *xt, *S_in, *Q_in, *S_out, *Q_out, *dml, *aroot;   // Kc each
    double *t, *e, *phinew, *w1, *w2;   // nmax each
    double *mu, *alpha, *gamma, *tmp, *u, *colk;  // cap (+1) each
    int *used, *grow;                   // cap
    int *unused, *upos, *amap, *action, *block;   // Kc each
    int8_t *planes;                     // digit planes of the tensor-core contraction (tc_planes_bytes), or null
};

// Each of the three cap x cap matrices is over-allocated to (cap + 32) x (cap + 8), rounded to a
// multiple of 4 doubles, so that either SIGMA buffer can hold the zero-padded copy (rows to a multiple
// of 32, columns to a multiple of 8) that quad_forms() streams into shared memory.
__host__ __device__ inline size_t sig_elems(int cap) { return (((size_t)(cap + 32) * (cap + 8)) + 3) & ~(size_t)3; }

// leading dimension of the column-major active-column matrix PHI: rows padded to a multiple of 4 so that a lane
// can fetch four consecutive rows of a column with 16-byte loads (the pad rows are kept at zero)
__host__ __device__ inline int phi_ld(int n) { return (n + 3) & ~3; }
constexpr int PHIT_LD = 64;       // row-major copy of the first 64 active columns (binomial IRLS Gram matrix)

__host__ __device__ inline size_t slab_doubles(int cap, int nmax, int Kc)
{
    return 3 * sig_elems(cap) + (((size_t)cap * cap + 3) & ~(size_t)3) + (size_t)phi_ld(nmax) * cap + (size_t)(nmax + 32) * PHIT_LD + (size_t)cap * Kc + (size_t)7 * Kc + (size_t)5 * nmax +
           (size_t)7 * (cap + 1);
}
__host__ __device__ inline size_t slab_ints(int cap, int Kc) { return (((size_t)2 * cap + (size_t)5 * Kc) + 3) & ~(size_t)3; }
__host__ __device__ inline size_t slab_base_bytes(int cap, int nmax, int Kc)
{
    size_t b = slab_doubles(cap, nmax, Kc) * 8 + slab_ints(cap, Kc) * 4;
    return (b + 255) & ~(size_t)255;
}
// right-hand-side digit planes of the tensor-core contraction: 8 planes x 30 columns x the training rows rounded up to 32
__host__ __device__ inline size_t tc_planes_bytes(int nmax) { return (size_t)30 * 8 * (size_t)((nmax + 31) & ~31); }
__host__ __device__ inline size_t slab_bytes(int cap, int nmax, int Kc, int tc)
{
    return slab_base_bytes(cap, nmax, Kc) + (tc ? (tc_planes_bytes(nmax) + 255) & ~(size_t)255 : 0);
}

__device__ inline Slab carve_slab(char *base, int cap, int nmax, int Kc, int tc)
{
    Slab s;
    double *d = reinterpret_cast<double *>(base);
    s.sigma = d; d += sig_elems(cap);
    s.sigma_new = d; d += sig_elems(cap);
    s.H = d; d += sig_elems(cap);
    s.ptp = d; d += ((size_t)cap * cap + 3) & ~(size_t)3;          // keeps the arrays behind it 32-byte aligned
    s.phit = d; d += (size_t)(nmax + 32) * PHIT_LD;
    s.phi = d; d += (size_t)phi_ld(nmax) * cap;
    s.G = d; d += (size_t)cap * Kc;
    s.xt = d; d += Kc; s.S_in = d; d += Kc; s.Q_in = d; d += Kc; s.S_out = d; d += Kc; s.Q_out = d; d += Kc;
    s.dml = d; d += Kc; s.aroot = d; d += Kc;
    s.t = d; d += nmax; s.e = d; d += nmax; s.phinew = d; d += nmax; s.w1 = d; d += nmax; s.w2 = d; d += nmax;
    s.mu = d; d += cap + 1; s.alpha = d; d += cap + 1; s.gamma = d; d += cap + 1;
    s.tmp = d; d += cap + 1; s.u = d; d += cap + 1; s.colk = d; d += 2 * (cap + 1);
    int *i = reinterpret_cast<int *>(d);
    s.used = i; i += cap; s.grow = i; i += cap;
    s.unused = i; i += Kc; s.upos = i; i += Kc; s.amap = i; i += Kc; s.action = i; i += Kc; s.block = i; i += Kc;
    s.planes = tc ? reinterpret_cast<int8_t *>(base + slab_base_bytes(cap, nmax, Kc)) : nullptr;
    return s;
}

// ------------------------------------------------------------------------------------------
// Optional per-phase cycle accounting (compile with -DPAREBEN_PHASE_TIMING; experiments only).
enum : int { PH_VFILL = 0, PH_CONTRACT, PH_QUAD, PH_GRAM, PH_SWEEP, PH_IRLS_OTHER, PH_DELTA_ML, PH_ACTIONS, PH_LOGLIK, PH_OTHER, PH_COUNT };
#ifdef PAREBEN_PHASE_TIMING
static __device__ unsigned long long g_phase_cycles[PH_COUNT];
static __device__ unsigned long long g_phase_calls[PH_COUNT];
struct PhaseTimer {
    long long t0; int ph;
    __device__ inline PhaseTimer(int p) : ph(p) { __syncthreads(); t0 = clock64(); if (threadIdx.x == 0) atomicAdd(&g_phase_calls[p], 1ULL); }
    __device__ inline ~PhaseTimer() { __syncthreads(); if (threadIdx.x == 0) atomicAdd(&g_phase_cycles[ph], (unsigned long long)(clock64() - t0)); }
};
#define PHASE(p) PhaseTimer phase_timer_##p(p)
constexpr int FIT_TRACE_MAX = 1 << 16;
static __device__ unsigned long long g_fit_t0[FIT_TRACE_MAX], g_fit_t1[FIT_TRACE_MAX];   // %globaltimer (ns) per fit
static __device__ int g_fit_block[FIT_TRACE_MAX];
__device__ inline unsigned long long global_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#else
#define PHASE(p) do { } while (0)
#endif

// ------------------------------------------------------------------------------------------
// mbarrier and bulk-copy (TMA) helpers
__device__ inline unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ inline void mbar_init(unsigned long long *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ inline void mbar_arrive(unsigned long long *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ inline void mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ inline void mbar_wait(unsigned long long *bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy executed by the TMA unit (SASS: UBLKCP), completion counted in bytes on `bar`
__device__ inline void bulk_load(void *dst_smem, const void *src_gmem, unsigned bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------
// block-level primitives.  `red` is a shared scratch of >= 33 doubles, `redi` >= 33 ints.
struct TcState;
struct Scratch {
    double *red; int *redi; double *sweep; /* SWEEP_SMEM_M^2 + 2*SWEEP_SMEM_M doubles, or null */
    TcState *tc;                           // tensor-core contraction state (binomial main-effect kernel with Problem::tc), or null
};

__device__ inline double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ inline double block_sum(double v, const Scratch &sc)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();                       // protect scratch from the previous use
    if (lane == 0) sc.red[wid] = v;
    __syncthreads();
    double tot = 0;
    for (int w = 0; w < nw; w++) tot += sc.red[w];   // same order in every thread -> identical result
    return tot;
}

__device__ inline void block_sum2(double &a, double &b, const Scratch &sc)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    a = warp_sum(a); b = warp_sum(b);
    __syncthreads();
    if (lane == 0) { sc.red[wid] = a; sc.red[32 + wid] = b; }
    __syncthreads();
    double ta = 0, tb = 0;
    for (int w = 0; w < nw; w++) { ta += sc.red[w]; tb += sc.red[32 + w]; }
    a = ta; b = tb;
}

// argmax of (val, key): largest val, ties -> smallest key.  Only val > 0 competes (the reference's
// scans start from 0 with a strict '>').  Returns arg (0 when nothing is positive) and the max.
__device__ inline void block_argmax(double val, int key, int arg, const Scratch &sc, double &best, int &best_arg)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double v2 = __shfl_xor_sync(0xffffffffu, val, o);
        int k2 = __shfl_xor_sync(0xffffffffu, key, o);
        int a2 = __shfl_xor_sync(0xffffffffu, arg, o);
        if (v2 > val || (v2 == val && k2 < key)) { val = v2; key = k2; arg = a2; }
    }
    __syncthreads();
    if (lane == 0) { sc.red[wid] = val; sc.redi[wid] = key; sc.redi[32 + wid] = arg; }
    __syncthreads();
    double bv = 0; int bk = 0x7fffffff, ba = 0;
    for (int w = 0; w < nw; w++) {
        double v2 = sc.red[w]; int k2 = sc.redi[w], a2 = sc.redi[32 + w];
        if (v2 > bv || (v2 == bv && v2 > 0 && k2 < bk)) { bv = v2; bk = k2; ba = a2; }
    }
    best = bv; best_arg = ba;
}

// Ordered compaction: list[] receives, in ascending order, every c in [0,n) with pred(c);
// pos[c] (optional) receives its position.  Values stored are c + store_offset.
template <class Pred>
__device__ inline int block_compact(int n, Pred pred, int *list, int *pos, int store_offset, const Scratch &sc)
{
    const int T = blockDim.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
    int base = 0;
    for (int c0 = 0; c0 < n; c0 += T) {
        const int c = c0 + threadIdx.x;
        const bool f = c < n && pred(c);
        const unsigned m = __ballot_sync(0xffffffffu, f);
        __syncthreads();
        if (lane == 0) sc.redi[wid] = __popc(m);
        __syncthreads();
        int off = 0, tot = 0;
        for (int w = 0; w < nw; w++) { int v = sc.redi[w]; if (w < wid) off += v; tot += v; }
        if (f) {
            int p = base + off + __popc(m & ((1u << lane) - 1u));
            list[p] = c + store_offset;
            if (pos) pos[c] = p;
        }
        base += tot;
    }
    __syncthreads();
    return base;
}

// Candidate id -> loci.  Main effects: (c, c).  Pairs are enumerated i<j row-major after the K
// main effects (NeFull2.c:115-134): c = K + i*(2K-i-1)/2 + (j-i-1).
__device__ inline void decode_candidate(int c, int K, int &i, int &j)
{
    if (c < K) { i = j = c; return; }
    long long p = (long long)c - K;
    double kk = 2.0 * K - 1.0;
    long long ii = (long long)floor((kk - sqrt(kk * kk - 8.0 * (double)p)) * 0.5);
    if (ii < 0) ii = 0;
    while (ii > 0 && ii * (2LL * K - ii - 1) / 2 > p) ii--;
    while ((ii + 1) * (2LL * K - (ii + 1) - 1) / 2 <= p) ii++;
    i = (int)ii;
    j = (int)(p - ii * (2LL * K - ii - 1) / 2) + i + 1;
}

template <bool EPIS>
struct Cand {
    int i, j;
    __device__ inline Cand(int c, int K) { if (EPIS) decode_candidate(c, K, i, j); else i = j = c; }
    __device__ inline double at(const double *Xrow) const
    {
        if (EPIS) return i == j ? Xrow[i] : Xrow[i] * Xrow[j];
        return Xrow[i];
    }
    // int -> double without the (quarter-rate) I2F conversion: 2^52 + 2^31 + v is representable and its
    // low word is 0x80000000 ^ v, so one XOR and one FP64 subtract give v exactly.
    static __device__ inline double small_int_to_double(int v)
    {
        return __hiloint2double(0x43300000, (int)(0x80000000u ^ (unsigned)v)) - 4503601774854144.0;
    }
    static __device__ inline int sbyte(int w, int b) { return (int)(int8_t)((unsigned)w >> (8 * b)); }
    // element b (0..3) of a 4-row packed word pair loaded from the transposed int8 matrix
    // (one I2F.F64.S8 with a byte selector per main-effect value: the conversion pipe is otherwise idle next to the DMMAs)
    __device__ inline double from_words(int wi, int wj, int b) const
    {
        if (EPIS && i != j) return (double)(sbyte(wi, b) * sbyte(wj, b));
        return (double)(signed char)((unsigned)wi >> (8 * b));
    }
    __device__ inline double at(const int8_t *Xrow) const      // exact: |x| <= 127, products <= 2^14
    {
        if (EPIS) return small_int_to_double(i == j ? (int)Xrow[i] : (int)Xrow[i] * (int)Xrow[j]);
        return small_int_to_double((int)Xrow[i]);
    }
};

}  // namespace pareben
