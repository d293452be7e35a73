// eben_step.cuh -- the steps of the EBEN iteration that the cached Gaussian (gauss_fit.cuh), cached binomial
// (binom_fit.cuh) and streaming (stream_fit.cuh, stream_scan.cuh) solvers share.  Each step exists once, with the
// floating-point operations of the reference in its order, quirks included: a rule changed here changes every solver.
// What looks alike but rounds differently (the add's SIGMA * tmp, the intercept and noise updates, the S/Q corrections)
// stays with its solver.
#pragma once
#include "common.cuh"
#include "linalg.cuh"
#include <type_traits>

namespace pareben {

// ---- fEBDeltaML's closed form (MainEff.c:1417-1497, NeFull2.c:1290-1345, NEmainEff.c:2101-2170) ----
// so and q2 = Q^2 are a candidate's statistics with the in-model correction applied; l1 = lambda alpha_en,
// l2 = lambda (1 - alpha_en).  add_a: the leading coefficient a of the ADD's quadratic (a < 0 is necessary for an ADD).
// add_root: the root r of an ADD (alpha = r + l2) and its gain L, defined only where a < 0 and dl > 0, which it returns.
__device__ __forceinline__ double add_a(double so, double q2, double l1, double l2)
{
    return so - q2 + 2 * l1 + l2;
}

__device__ __forceinline__ bool add_root(double so, double q2, double l1, double l2, double &r, double &L)
{
    const double a = add_a(so, q2, l1, l2);
    const double b = (so + l2) * (so + 4 * l1 + l2);
    const double gm = 2 * l1 * (so + l2) * (so + l2);
    const double dl = b * b - 4 * a * gm;
    if (!(a < 0 && dl > 0)) return false;
    r = (-b - sqrt(dl)) / (2 * a);
    L = (log(r / (r + so + l2)) + q2 / (r + so + l2)) * 0.5 - l1 / r;
    return true;
}

// gain of re-estimating an active basis from alpha to r + l2
__device__ __forceinline__ double reest_gain(double so, double q2, double l1, double l2, double r, double alpha)
{
    const double o = alpha - l2;
    return 0.5 * (log(r * (o + so + l2) / (o * (r + so + l2))) +
                  q2 * (1 / (r + so + l2) - 1 / (o + so + l2))) -
           l1 * (1 / r - 1 / o);
}

// gain of deleting an active basis with prior alpha
__device__ __forceinline__ double delete_gain(double so, double q2, double l1, double l2, double alpha)
{
    const double o = alpha - l2;
    const double L = (log(o / (o + so + l2)) + q2 / (o + so + l2)) * 0.5 - l1 / o;
    return -L;
}

__device__ inline void refresh_out(const Slab &s, int M, int Kc)
{   // S_out/Q_out = S_in/Q_in, with the in-model correction (MainEff.c:664-671, 1320-1338)
    for (int c = threadIdx.x; c < Kc; c += blockDim.x) {
        double si = s.S_in[c], qi = s.Q_in[c];
        const int i = s.amap[c];
        if (i >= 0) {
            const double a = s.alpha[i];
            const double den = a - si;
            qi = a * qi / den;
            si = a * si / den;
        }
        s.S_out[c] = si; s.Q_out[c] = qi;
    }
    __syncthreads();
}

struct Decision { double best; int nu; int any_delete; };

// M = number of active effects (the binomial intercept is not counted).
template <bool EPIS, bool BINOM>
__device__ inline Decision delta_ml(Slab &s, int M, int N, int Kc, double lambda,
                                    double alpha_en, double residual, double var_y, int iter, int i_iter,
                                    const Scratch &sc)
{   // fEBDeltaML* (MainEff.c:1372-1582; NeFull2.c:1227-1404; NEmainEff.c:2063-2238; NeFull.c:1775-1950)
    PHASE(PH_DELTA_ML);
    const double l1 = lambda * alpha_en, l2 = lambda * (1 - alpha_en);
    int prio_add = 0, prio_del = 0;
    if (M < 10) { prio_add = 1; prio_del = 0; }
    if (M > 100 || (!EPIS && M >= N) || (!BINOM && residual <= var_y * 0.1)) { prio_add = 0; prio_del = 1; }
    double lbest = 0; int lkey = 0x7fffffff, larg = 0;
    int f_add = 0, f_del = 0;
    for (int c = threadIdx.x; c < Kc; c += blockDim.x) {
        const int i = s.amap[c];
        if (i == -2) { s.dml[c] = 0; s.action[c] = ACT_NONE; continue; }      // in neither Used nor Unused (see the delete action)
        const double so = s.S_out[c], qo = s.Q_out[c], q2 = qo * qo;
        double d_ml = 0; int act = ACT_NONE;
        double r, L;
        if (add_root(so, q2, l1, l2, r, L)) {
            if (L > 0) {
                s.aroot[c] = r + l2;
                if (i >= 0) {
                    act = ACT_REEST;
                    d_ml = reest_gain(so, q2, l1, l2, r, s.alpha[i]);
                } else {
                    act = ACT_ADD;
                    d_ml = L;
                    if (!EPIS && !BINOM) f_add = 1;   // only the Gaussian main-effect file ever sets anyToAdd (:1484)
                }
            }
        } else if (i >= 0 && M > 1) {
            f_del = 1;
            act = ACT_DEL;
            d_ml = delete_gain(so, q2, l1, l2, s.alpha[i]);
        }
        s.dml[c] = d_ml; s.action[c] = act;
        const int key = i >= 0 ? i : M + s.upos[c];    // visiting order of the reference's two scans
        if (d_ml > lbest || (d_ml == lbest && d_ml > 0 && key < lkey)) { lbest = d_ml; lkey = key; larg = c; }
    }
    const int any_add = __syncthreads_or(f_add);
    const int any_del = __syncthreads_or(f_del);
    Decision out;
    out.any_delete = any_del;
    bool rescan = false;
    if ((any_add && prio_add) || (any_del && prio_del)) {        // :1527-1556
        for (int c = threadIdx.x; c < Kc; c += blockDim.x) {
            const int act = s.action[c];
            if (act == ACT_REEST) s.dml[c] = 0;
            else if (act == ACT_DEL) { if (any_add && prio_add && !prio_del) s.dml[c] = 0; }
            else if (act == ACT_ADD) { if (any_del && prio_del && !prio_add) s.dml[c] = 0; }
        }
        rescan = true;
    }
    if (!EPIS && !BINOM && ((!any_add && iter == 1 && i_iter < 10) || (!any_add && residual >= var_y * 0.95))) {   // :1557-1577
        for (int c = threadIdx.x; c < Kc; c += blockDim.x) if (s.action[c] == ACT_DEL) s.dml[c] = 0;
        rescan = true;
    }
    if (rescan) {       // rescans run in ascending candidate order
        lbest = 0; lkey = 0x7fffffff; larg = 0;
        for (int c = threadIdx.x; c < Kc; c += blockDim.x) {
            const double d = s.dml[c];
            if (d > lbest) { lbest = d; lkey = c; larg = c; }
        }
    }
    block_argmax(lbest, lkey, larg, sc, out.best, out.nu);
    return out;
}

// The block of actions that follows fEBDeltaML (MainEff.c:426-474, NEmainEff.c:559-607): the forced delete of the
// initial basis, or every candidate whose delta-ML reaches the cutoff (a single one when the best is a delete), in
// s.block.  n_eff counts the active effects (not the binomial intercept).  Returns the block's length; 0 when nothing
// is worthwhile, which terminates (selected = ACT_TERM).
__device__ __forceinline__ int choose_block(Slab &s, const Variant &v, const Decision &d, int n_eff, int Kc, int initial,
                                            int &selected, int &ini_removed, const Scratch &sc)
{
    int nu = d.nu, n_update = 0;
    if (selected == ACT_TERM && !ini_removed && n_eff > 1) nu = -1;         // :426-430
    if (nu == -1 && ini_removed) {
    } else if (nu == -1 && !ini_removed && n_eff > 1) {                      // :437-446
        nu = initial - 1;
        __syncthreads();
        if (threadIdx.x == 0) { s.action[nu] = ACT_DEL; s.block[0] = nu; }
        __syncthreads();
        n_update = 1; ini_removed = 1; selected = ACT_DEL;
    } else {
        const int best_is_add = s.action[nu] == ACT_ADD, best_is_del = s.action[nu] == ACT_DEL;
        double cutoff = d.best * (best_is_add ? v.n_add : 1.0);
        if (cutoff < v.ml_delta) cutoff = v.ml_delta;
        n_update = block_compact(Kc, [&](int c) { return s.dml[c] >= cutoff; }, s.block, nullptr, 0, sc);
        if (best_is_del && n_update > 1) n_update = 1;                       // :474
    }
    if (n_update == 0) selected = ACT_TERM;
    return n_update;
}

// Slot jj of candidate nu for a re-estimate or delete.  The reference searches Used and silently keeps the previous jj
// when the search fails (the forced removal of an initial basis that a regular delete already took out, MainEff.c:498-509,
// NEmainEff.c:629-636).  Keep that, but never index outside the n_eff active effects.
__device__ __forceinline__ void find_slot(const Slab &s, int nu, int n_eff, int &jj, int &selected, int &status)
{
    if (selected != ACT_REEST && selected != ACT_DEL) return;
    const int a = s.amap[nu];
    if (a >= 0) jj = a;
    if (jj < 0 || jj >= n_eff) { status |= ST_NOT_PD; selected = ACT_TERM; }
}

// ---- SIGMA and mu after an action (ActionRes/Add/Del: MainEff.c:553-596, 1585-1822; NEmainEff.c:830-1203) ----
// SIGMA is M x M with leading dimension M; the updated matrix goes to sigma_new, which never aliases it (restrict: the
// loads of an unrolled column run ahead of its stores).  Warps own columns, lanes rows: no integer division.

// re-estimate of slot j:  SIGMA' = SIGMA - kappa s_j s_j',  mu += -mu_j kappa s_j
__device__ __forceinline__ void sigma_reest(const double *__restrict__ sigma, double *__restrict__ sigma_new, int M, int j, double kappa)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int c = wid; c < M; c += nw) {
        const double kj = sigma[j * M + c];
#pragma unroll 4
        for (int i = lane; i < M; i += 32) {
            const int idx = c * M + i;
            sigma_new[idx] = sigma[idx] - kappa * sigma[j * M + i] * kj;
        }
    }
}

__device__ __forceinline__ void mu_reest(double *mu, int M, const double *sj, double mujj, double kappa)
{
    for (int i = threadIdx.x; i < M; i += blockDim.x) mu[i] += -mujj * kappa * sj[i];
}

// add of slot M:  SIGMA' = [SIGMA + s_ii u u', -s_ii u; -s_ii u', s_ii]  ((M+1) x (M+1)),  u = SIGMA * (beta) PHI' phi_new
__device__ __forceinline__ void sigma_add(const double *__restrict__ sigma, double *__restrict__ sigma_new, int M,
                                          const double *__restrict__ u, double s_ii)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int M1 = M + 1;
    for (int j = wid; j < M1; j += nw) {
        const double uj = u[min(j, M - 1)];
#pragma unroll 4
        for (int i = lane; i < M1; i += 32) {
            double val;
            if (i < M && j < M) val = sigma[j * M + i] + (s_ii * u[i]) * uj;
            else if (i == M && j == M) val = s_ii;
            else val = -s_ii * u[i < M ? i : j];
            sigma_new[j * M1 + i] = val;
        }
    }
}

__device__ __forceinline__ void mu_add(double *mu, int M, const double *u, double mu_i)
{
    for (int i = threadIdx.x; i < M; i += blockDim.x) mu[i] += -mu_i * u[i];
    if (threadIdx.x == 0) mu[M] = mu_i;
}

// delete of slot j: the Schur downdate, the last row and column moved into slot j ((M-1) x (M-1), :1754-1776).  The
// reference rounds the update term two ways:
//   QUOTIENT_FIRST   s - (s_i / s_jj) * s_j   MainEff.c, NeFull2.c, NeFull.c:1612
//   otherwise        s - s_i * s_j / s_jj     NEmainEff.c:1069
// q (QUOTIENT_FIRST only): M doubles of scratch that take the quotients s_i / s_jj first -- one division per row instead
// of per entry, behind one more barrier; a literal nullptr divides per entry (the same quotients, bit for bit).
template <bool QUOTIENT_FIRST, class Q>
__device__ __forceinline__ void sigma_delete(const double *__restrict__ sigma, double *__restrict__ sigma_new, int M, int j, Q q)
{
    constexpr bool ROW_QUOTIENTS = QUOTIENT_FIRST && !std::is_same<Q, std::nullptr_t>::value;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const double *sj = sigma + j * M;
    const double sjj = sj[j];
    if constexpr (ROW_QUOTIENTS) {
        for (int i = threadIdx.x; i < M; i += blockDim.x) q[i] = sj[i] / sjj;
        __syncthreads();
    }
    const int lastj = M - 1;
    for (int c = wid; c < lastj; c += nw) {
        const int sjx = (c == j) ? lastj : c;
        const double sjv = sj[sjx];
#pragma unroll 4
        for (int i = lane; i < lastj; i += 32) {
            const int si = (i == j) ? lastj : i;
            double v;
            if constexpr (!QUOTIENT_FIRST) v = sigma[sjx * M + si] - sj[si] * sjv / sjj;
            else if constexpr (ROW_QUOTIENTS) v = sigma[sjx * M + si] - q[si] * sjv;
            else v = sigma[sjx * M + si] - sj[si] / sjj * sjv;
            sigma_new[c * lastj + i] = v;
        }
    }
}

// mujj: the deleted slot's weight as the reference holds it (an `int Mujj` in the Gaussian files, MainEff.c:1746-1747)
__device__ __forceinline__ void mu_delete(double *mu, int M, const double *sj, double sjj, double mujj)
{
    for (int i = threadIdx.x; i < M; i += blockDim.x) mu[i] = mu[i] - mujj * sj[i] / sjj;
}

// PHI'PHI (leading dimension cap) after a delete: the last row and column into slot jj
__device__ __forceinline__ void ptp_move_last(double *ptp, int cap, int jj, int lastj)
{
    if (jj == lastj) return;
    for (int i = threadIdx.x; i < lastj; i += blockDim.x) {
        if (i == jj) ptp[(size_t)jj * cap + jj] = ptp[(size_t)lastj * cap + lastj];
        else { ptp[(size_t)i * cap + jj] = ptp[(size_t)i * cap + lastj]; ptp[(size_t)jj * cap + i] = ptp[(size_t)lastj * cap + i]; }
    }
}

// ---- the Gaussian solver's start and hold-out score (cached and streaming) ----
// initialisation (MainEff.c:1003-1090): beta from the variance of t, alpha_0 of the initial basis phi in closed form,
// clamped to init_alpha_max
template <bool EPIS>
__device__ __forceinline__ void gauss_start(const double *phi, const double *t, int N, const Variant &v, double &beta,
                                            double *alpha, const Scratch &sc)
{
    const double var = block_var(t, N, sc);
    if (!EPIS) beta = 1 / (var * 0.01 + 1e-10);
    else { double sd = sqrt(var); if (sd < 1e-6) sd = 1e-6; beta = 1 / ((sd * 0.1) * (sd * 0.1)); }
    double p = 0, q = 0;
    for (int h = threadIdx.x; h < N; h += blockDim.x) { p = fma(phi[h], phi[h], p); q = fma(phi[h], t[h], q); }
    block_sum2(p, q, sc);
    p *= beta; q *= beta;
    double a = p * p / (q * q - p);
    if (a < 0) a = v.init_alpha_max;
    if (a > v.init_alpha_max) a = v.init_alpha_max;
    if (threadIdx.x == 0) alpha[0] = a;
}

// hold-out sum of squared errors (R/GetModelError.R:6-32) of the model (b, mu on `used`): Beta[,3] = mu / norm(i) into
// tmp (:221), norm(i) being the column norm of active slot i.  nsel = number of non-zero weights.
template <bool EPIS, class Norm>
__device__ __forceinline__ double gauss_holdout_sse(const FoldData &F, int K, int M, const double *mu, const int *used, double b,
                                                    double *tmp, Norm norm, int &nsel, int &status, const Scratch &sc)
{
    const int T = blockDim.x;
    __syncthreads();
    for (int i = threadIdx.x; i < M; i += T) tmp[i] = mu[i] / norm(i);
    __syncthreads();
    double sse = 0;
    for (int h = threadIdx.x; h < F.nte; h += T) {
        const double *xr = F.Xte + (size_t)h * K;
        double pred = 0;
        for (int i = 0; i < M; i++) {
            const double w = tmp[i];
            if (w != 0) { Cand<EPIS> cd(used[i] - 1, K); pred = fma(cd.at(xr), w, pred); }
        }
        const double r = F.yte[h] - (b + pred);
        sse = fma(r, r, sse);
    }
    sse = block_sum(sse, sc);
    nsel = 0;
    for (int i = 0; i < M; i++) nsel += tmp[i] != 0;
    if (!isfinite(sse)) status |= ST_NONFINITE;
    return sse;
}

// ---- what a fit reports (thread 0) ----
// flops[1] collects work the SURVEY 8d model counts but the Gram organisation did not execute, flops[2] the score
// contractions run on the int8 tensor cores
__device__ __forceinline__ void write_fit_outputs(const FitOutputs &out, int o, double err, int status, int nsel, int iter,
                                                  double flops, double avoided, double tc_calls)
{
    if (out.fold_err) out.fold_err[o] = err;
    if (out.status) out.status[o] = status;
    if (out.n_selected) out.n_selected[o] = nsel;
    if (out.n_iter) out.n_iter[o] = iter;
    if (out.flops) {
        atomicAdd(out.flops, flops);
        if (avoided > 0) atomicAdd(out.flops + 1, avoided);
        if (tc_calls > 0) atomicAdd(out.flops + 2, tc_calls);
    }
}

// full-model record of fit o (pareben_fit_batch): the M slots of mu / SIGMA / H, effects from slot `first` on (the
// binomial intercept is slot 0), norm(k) the column norm of effect k; scalars: the Wald score mu'H mu with H read at
// leading dimension M (MainEff.c:206-215), then s1, s2, s3
template <class Norm>
__device__ __forceinline__ void write_record(const FitOutputs &out, int o, int M, int first, const double *mu, const double *H,
                                             const double *sigma, const int *used, Norm norm, double s1, double s2, double s3)
{
    out.m_out[o] = M - first;
    double wd = 0;
    for (int i = 0; i < M; i++) {
        double z = 0;
        for (int j = 0; j < M; j++) z += mu[j] * H[i * M + j];
        wd += z * mu[i];
    }
    const size_t r = (size_t)o * out.dump_ld;
    for (int i = first; i < M; i++) {
        const int k = i - first;
        const double sc = norm(k);
        out.used_out[r + k] = used[k];
        out.beta_out[r + k] = mu[i] / sc;
        out.var_out[r + k] = sigma[i * M + i] / (sc * sc);
    }
    out.scalars_out[4 * (size_t)o + 0] = wd; out.scalars_out[4 * (size_t)o + 1] = s1;
    out.scalars_out[4 * (size_t)o + 2] = s2; out.scalars_out[4 * (size_t)o + 3] = s3;
}

}  // namespace pareben
