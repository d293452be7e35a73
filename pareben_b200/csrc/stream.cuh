// stream.cuh -- streaming-Kc mode: EBEN fits whose candidate set is too large for a per-fit cache
// (BASELINE config 5: K = 20,000 loci -> Kc = 200,010,000 main + pair candidates).
//
// The cached kernel (fit_kernel.cuh) keeps, per fit, the reference's BASIS_PHI cache (one row of Kc doubles per
// active basis, NeFull2.c:350-365) plus six Kc-length statistic arrays; at Kc = 2e8 that is 1.6 GB per active
// basis per fit and neither the reference nor that kernel can run.  Here a fit keeps ONLY its active set
// (PHI, SIGMA, mu, alpha, PHI'PHI) and the per-candidate statistics are recomputed from it whenever the solver
// asks for them:
//
//     Q_c = beta_s * phi_c' e'            e' = t - PHI mu - d          (one N-vector per fit)
//     S_c = beta_s - beta_s^2 g_c' SIGMA g_c,   g_c = PHI' phi_c
//
// which are the quantities the reference maintains incrementally (FullStat NeFull2.c:1063-1196 followed by the
// rank-1 corrections of the add / delete / re-estimate actions :1407-1640).  Two details make the recomputed
// values equal to the reference's to rounding, not just approximately:
//   * d accumulates mu'_j phi_j for every basis deleted since the last FullStat: the reference's delete
//     truncates the weight to an int (`int Mujj`, MainEff.c:1746) and drops the remainder, so its Q array is
//     consistent with a residual that still carries that remainder;
//   * beta_s is the noise precision of the last FullStat: a noise update that moves log(beta) by less than 1e-6
//     changes beta but not the statistic arrays (:716-727).
// (scripts/stream_equivalence.py demonstrates both on the CPU oracle.)
//
// An out-of-model candidate can only ever be ADDed, and only when a = S - Q^2 + 2 l1 + l2 < 0 (fEBDeltaML,
// NeFull2.c:1227-1404) -- impossible unless Q^2 > 2 l1 + l2 because S > 0.  So one pass needs Q for every
// candidate but S only for the few that pass this exact screen.  All fits that share a fold advance in
// lock-step rounds:
//
//   stream_advance_kernel   one block per fit: consume the previous scan (in-model statistics, decision,
//                           block of actions, noise update, outer-loop bookkeeping) up to the next point where
//                           the reference calls fEBDeltaML, then publish e' as one column of the fold's
//                           right-hand-side matrix E;
//   stream_scan_kernel      ONE dense FP64 contraction  X_fold' * E  for all waiting fits of every fold on the
//                           FP64 tensor cores (DMMA m8n8k4): candidate columns -- pair products x_i * x_j are
//                           generated in registers from the int8 loci -- against E tiles that the TMA unit
//                           streams into shared memory (cp.async.bulk + mbarrier
//                           ring).  The epilogue screens, and for survivors computes S, the closed-form
//                           delta-ML and appends to the fit's ADD list; nothing of length Kc is ever stored.
#pragma once
#include "common.cuh"
#include "eben_step.cuh"

namespace pareben {

enum : int { ST_LIST = 16 };                 // streaming mode: a fit's ADD list overflowed (mirrored in include/pareben.h)
enum : int { SP_START = 0, SP_WAIT = 1, SP_DONE = 2 };

constexpr int SK = 64;                       // rows per shared-memory stage of E
constexpr int SN = 64;                       // right-hand sides (fits) per tile
constexpr int SLD = SK + 4;                  // leading dimension of a staged column: == 4 (mod 16) doubles -> conflict-free B fragments
constexpr int STAGE_D = SN * SLD;            // doubles per stage (34,816 bytes: one bulk copy)
constexpr int SCAN_STAGES = 4;
constexpr int SCAN_CT = 128;                 // candidates per work item: 8 consumer warps x 16
constexpr int SCAN_WARPS = 8;                // two per scheduler: up to 255 registers each
constexpr int SCAN_THREADS = 32 * SCAN_WARPS;
constexpr int STREAM_MAX_FOLDS = 256;
constexpr int ADV_THREADS = 256;

struct StreamFit {
    // task
    int fold, target, out_index;           // target: response index, as FitTask::target
    double lambda, alpha_en;
    // control state of the solver between two rounds (the loop-carried scalars of gauss_fit())
    int phase;
    int iter, i_iter, selected, ini_removed, n_update, jj, it_max, initial, M, status;
    int n_hidden, hidden[4];                // candidates in neither Used nor Unused until the next outer iteration (see the delete action)
    int stats_valid;                        // nothing has touched the statistic arrays since the last fEBDeltaML: the next one sees the same S, Q
    double beta, beta_s, b, vk, vk0, err, residvar, var_y, flops;
    // scan interface (meaningful while phase == SP_WAIT)
    int slot, cls;                          // right-hand-side slot within the (fold, class) this round
    double l1, l2, ml_delta, n_add, s_lb;
    unsigned long long runmax;              // bit pattern of the largest ADD delta-ML seen so far this round (0 = none)
    int n_list, any_add;
    // per-fit arrays
    double *sigma, *sigma_new, *H, *ptp, *phi;
    double *mu, *alpha, *gamma, *tmp, *u, *colk, *ascale, *s_in, *q_in, *dml_in, *aroot_in;
    double *t, *e, *d, *phinew;
    int *used, *act_in, *blk_c, *blk_src;
    int *list_c; double *list_dml, *list_aroot;
};

// The scan's per-element test is ONE comparison, z^2 > thr[slot] * ||x_c||^2, with thr the tightest exact bound known:
//   screen 1:  Q^2 > 2 l1 + l2 is necessary for a < 0 because S > 0 (fEBDeltaML, NeFull2.c:1290-1345);
//   screen 2:  delta-ML is L(S, Q) = sup_r f(r; S, Q) with df/dS < 0 < df/dQ^2, and S >= s_lb = 1 / (1/beta_s + sum_j 1/alpha_j)
//              (C^-1 >= lambda_min(C^-1) I, unit columns): L(s_lb, Q) bounds a candidate's delta-ML from above and is
//              increasing in Q^2, so "L could reach `need`" is Q^2 >= q2_threshold(need), found by bisection -- once per fit
//              per round for need = ml_delta, and again whenever a survivor raises the fit's best delta-ML
//              (need = n_add * best; thr only ever grows: atomicMax on its bit pattern).
__device__ inline double lub_of(double q2, double sl, double l1, double l2)
{   // upper bound of delta-ML at Q^2 = q2; +inf where the closed form cannot be evaluated (keeps the candidate)
    if (!(add_a(sl, q2, l1, l2) < 0)) return 0.0;
    double r, L;
    if (!add_root(sl, q2, l1, l2, r, L)) return INFINITY;
    if (!(r > 0)) return INFINITY;
    return L == L ? L : INFINITY;
}

__device__ inline double q2_threshold(double need, double sl, double l1, double l2)
{   // largest q2 known to have lub_of(q2) < need (every Q^2 at or below it is rejected)
    double lo = sl + 2 * l1 + l2;
    if (!(need > 0)) return lo;
    double hi = 2 * lo + 4 * need + 1e-300;
    for (int it = 0; it < 400 && lub_of(hi, sl, l1, l2) < need; it++) hi *= 2;
    for (int it = 0; it < 40; it++) {                 // lo only has to be a valid rejection bound: 2^-40 of the bracket is plenty
        const double mid = 0.5 * (lo + hi);
        if (lub_of(mid, sl, l1, l2) >= need) hi = mid; else lo = mid;
    }
    return lo * (1 - 1e-12);
}

// Right-hand-side classes.  Every waiting fit brings its residual e' as one right-hand-side column:
//   class 1 (A)   M = 1 and the basis is the initial one (candidate 1: the state of every fit of a large-lambda grid
//                 point and of every fit's first pass, MainEff.c:1003-1090): its column phi_0 is the same vector for all
//                 of them and rides ONCE per tile, in column 0, so the contraction also delivers g = phi_0' x_c for every
//                 candidate and the epilogue computes S EXACTLY instead of bounding it; 63 fits per tile;
//   class 0 (B)   every other fit: one column per fit, the s_lb bound, survivors finished by a warp each.
// The per-element test stays ONE comparison in both classes: with u = beta_s g'SIGMA g in [0, 1), S = beta_s (1 - u), and
// T[k] is the Q^2 threshold valid for u <= 2^-k (S >= max(s_lb, beta_s (1 - 2^-k))), k = 0..7.  Class B, which has no g,
// compares against T[0] (S >= s_lb); class A picks its bucket from u.  Nearly every candidate of a genotype design has
// u < 1/128 (k = 7), where the bound is within 1 % of its exact S.
struct ScanSlot { double bs, sig, l1, l2, s_lb, T[8]; };
constexpr int STREAM_CLASSES = 2;
__host__ __device__ inline int class_fits_per_tile(int cls) { return cls == 1 ? SN - 1 : SN; }

__device__ inline void slot_thresholds(ScanSlot *sp, double need, double thr_basic, bool use_bound)
{   // T[k] (in z^2 / ssq units) for `need`; only ever raised (atomicMax on the bit pattern: positive doubles are monotone)
    double sk_prev = -1, q2_prev = 0;
    for (int k = 0; k < 8; k++) {
        double sk = sp->bs * (1 - exp2(-(double)k));
        if (sk < sp->s_lb) sk = sp->s_lb;
        sk *= 1 - 1e-9;
        double q2 = thr_basic;
        if (use_bound) {
            const double q2t = sk == sk_prev ? q2_prev : q2_threshold(need, sk, sp->l1, sp->l2);      // buckets below s_lb share one bound
            sk_prev = sk; q2_prev = q2t;
            if (q2t > q2) q2 = q2t;
        }
        const double t = q2 / (sp->bs * sp->bs);
        if (t == t && t > 0) atomicMax(reinterpret_cast<unsigned long long *>(&sp->T[k]), (unsigned long long)__double_as_longlong(t));
    }
}

// Per-(fold, class) view of the lock-step round: index STREAM_CLASSES * fold + class.
struct StreamFold {
    double *E;                  // [rhs tile][stage][SN][SLD] staged right-hand sides of this round
    ScanSlot *par;              // [slot] (slot = first column of the fit within the class' tiles)
    int *slot_fit;              // [slot] fit index
    int max_slots;
};

struct StreamShared {
    StreamFold *folds;          // [STREAM_CLASSES * (n_folds + 1)]
    int *n_slots;               // [STREAM_CLASSES * (n_folds + 1)] fits waiting this round (advance kernel: atomicAdd; host: reset)
    int list_cap;
    double *warp_scratch;       // [scan blocks][SCAN_WARPS][cap]
    double *flops;
};

__host__ __device__ inline size_t e_tile_doubles(int ldt) { return (size_t)(ldt / SK) * STAGE_D; }

}  // namespace pareben
