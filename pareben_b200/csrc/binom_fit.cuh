// binom_fit.cuh -- one Binomial (logistic) EBEN fit per thread block (main-effect and Epis).
//
// Device re-design of the reference's logistic solver; behaviour follows
//   /root/reference/EBEN_orig/src/ElasticNetBinaryNEmainEff.c (entry :236-389, inner solver
//   :397-827, ActionAdd :830-1003, ActionDel :1010-1121, ActionRes :1127-1203, init :1215-1406,
//   FullStat :1633-1803, PostMode/IRLS :1808-2010, DeltaML :2063-2238) and
//   ElasticNetBinaryNeFull.c for Epis (same skeleton; clamps and constants per SURVEY.md App. A),
// followed by the hold-out score of /root/reference/R/GetModelError.R:34-57.
// Differences in kind, not in result:
//  * FullStat's per-candidate vector BASIS'B PHI (:1693-1702) is computed once as a blocked
//    contraction and KEPT as a cache G for the block of actions that follows; the reference
//    recomputes it from scratch inside every action (:967-987, 1040-1058, 1171-1194) even though
//    the IRLS weights B cannot change until the next FullStat.
//  * the S/Q corrections of the LAST action of a block are skipped: FullStat overwrites S and Q
//    immediately afterwards (:749-762), so they are dead in the reference too.
//  * dgelsy on the N x 2 start-up regression is a closed-form pivoted QR; dpotrf/dpotri is the
//    in-block symmetric sweep.
#pragma once
#include "common.cuh"
#include "contract.cuh"
#include "linalg.cuh"
#include "tc_contract.cuh"
#include "eben_step.cuh"

namespace pareben {

struct BinomState {
    int M;            // intercept + active effects
    int n_unused;
    int status;
    double flops;
    double tc_calls;  // score contractions run on the int8 tensor cores
    bool at_mode;     // the last FullStat's posterior mode stopped on the gradient test at a point it had evaluated itself
};

// z = sum_j phi_j[h] mu[j] and z2 = the same for row h2, j ascending: two rows per thread keep twice the loads of the
// L2-resident PHI in flight (the sums themselves are unchanged).
__device__ inline void phi_rows_dot(const double *__restrict__ phi, int LD, int M, const double *__restrict__ mu, int h, int h2,
                                    double &z, double &z2)
{
    const double *pa = phi + h, *pb = phi + h2;
    double a = 0, b = 0;
#pragma unroll 4
    for (int j = 0; j < M; j++) { const double m = mu[j]; a = fma(pa[(size_t)j * LD], m, a); b = fma(pb[(size_t)j * LD], m, b); }
    z = a; z2 = b;
}

// eta = PHI mu ; y = sigmoid(eta) ; returns the data error (NEmainEff.c:2013-2032)
__device__ inline double predictor_and_error(const Slab &s, int N, int M, const double *mu, const double *t,
                                             double *eta, double *yv, const Scratch &sc)
{
    double err = 0;
    const int LD = phi_ld(N);
    auto row = [&](int h, double z) {
        eta[h] = z;
        const double y = 1 / (1 + exp(-z));
        yv[h] = y;
        double e = 0;
        if (y != 0) e = e - t[h] * log(y);
        if (y != 1) e = e - (1 - t[h]) * log(1 - y);
        err += e;
    };
    const int T = blockDim.x;
    for (int h = threadIdx.x; h < N; h += 2 * T) {
        const int h2 = h + T;
        const bool two = h2 < N;
        double z, z2;
        phi_rows_dot(s.phi, LD, M, mu, h, two ? h2 : h, z, z2);
        row(h, z);
        if (two) row(h2, z2);
    }
    return block_sum(err, sc);
}

// Returns true when eta / yv in memory belong to the final mu (the last evaluation was an accepted one).  Sets b.at_mode
// when, in addition, the loop stopped on the gradient test after a positive definite inverse: mu is then a fixed point, and
// another call from the same mu and alpha repeats the last Newton step's arithmetic bit for bit and stops at once.
template <bool EPIS>
__device__ inline bool post_mode(Slab &s, BinomState &b, int N, const double *t, const Scratch &sc)
{   // fEBCatPostMode*: Newton steps with step halving (NEmainEff.c:1808-2010, NeFull.c:998-1152)
    PHASE(PH_IRLS_OTHER);      // includes the nested IRLS phases (subtract them when reading the counters)
    const int M = b.M, T = blockDim.x, LD = phi_ld(N);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
    double *yv = s.t, *e = s.e, *w = s.w1, *eta = s.w2, *g = s.gamma, *dmu = s.u, *mun = s.tmp;
    double derr, reg = 0;
    {
        PHASE(PH_IRLS_PRED);
        derr = predictor_and_error(s, N, M, s.mu, t, eta, yv, sc);
        for (int i = 1; i < M; i++) reg = reg + s.alpha[i - 1] * s.mu[i] * s.mu[i] / 2;
    }
    bool current = true;
    double total = reg + derr;
    bool converged = false, pd = true;
    for (int it = 0; it < 25; it++) {
        const double err_log = total;
        double g0 = 0, h0 = 0;
        {
            PHASE(PH_IRLS_DIR);
            for (int h = threadIdx.x; h < N; h += T) {
                double y = yv[h];
                if (EPIS) { if (y < 1e-5) y = 1e-5; if (y > (1 - 1e-5)) y = 1 - 1e-5; yv[h] = y; }     // NeFull.c:1049-1050
                const double eh = t[h] - y;
                e[h] = eh; g0 += eh;
                double bw = y * (1 - y);
                if (!EPIS) { if (bw < 1e-10) bw = 1e-5; if (bw > 1e10) bw = 1e5; }                      // NEmainEff.c:1880-1882
                else { if (bw < 1e-5) bw = 1e-3; if (bw > 1e5) bw = 1e3; }                              // NeFull.c:1054-1055
                w[h] = bw; h0 += bw;
            }
            block_sum2(g0, h0, sc);
            if (threadIdx.x == 0) g[0] = g0;
            (void)h0;
            __syncthreads();
        }
        // gradient g_j = phi_j'e - alpha_j mu_j (one warp per column), then the Hessian PHI'B PHI + diag(0, alpha)
        // as a tiled Gram matrix; column 0 of PHI is the intercept's all-ones column, so H(0, k) = sum w phi_k
        // and H(0, 0) = sum w come out of the same pass (:1887-1919).
        const bool fused = M <= PHIT_LD && blockDim.x == 256;     // the Gram pass below also produces PHI'e
        if (!fused)
        for (int j = 1 + wid; j < M; j += 2 * nw) {             // two columns per warp: twice the loads in flight
            const int j2 = j + nw;
            const bool two = j2 < M;
            const double *ph = s.phi + (size_t)j * LD, *ph2 = s.phi + (size_t)(two ? j2 : j) * LD;
            double gj = 0, gj2 = 0;
#pragma unroll 4
            for (int h = lane; h < N; h += 32) { const double eh = e[h]; gj = fma(ph[h], eh, gj); gj2 = fma(ph2[h], eh, gj2); }
            gj = warp_sum(gj); gj2 = warp_sum(gj2);
            if (lane == 0) { g[j] = gj - s.alpha[j - 1] * s.mu[j]; if (two) g[j2] = gj2 - s.alpha[j2 - 1] * s.mu[j2]; }
        }
        auto put = [&](int j, int k, double z) {
            if (j == k && j > 0) z += s.alpha[k - 1];
            s.H[k * M + j] = z; s.H[j * M + k] = z;
        };
        if (fused) gram_pipe(s.phit, N, M, w, sc.sweep, put, e, [&](int j, double z) { if (j >= 1) g[j] = z - s.alpha[j - 1] * s.mu[j]; });   // row-major copy, pipelined
        else gram_mma(s.phi, N, LD, M, w, sc.sweep, put);
        {
            PHASE(PH_IRLS_COPY);
            for (int idx = threadIdx.x; idx < M * M; idx += T) s.sigma[idx] = s.H[idx];
            __syncthreads();
        }
        pd = spd_inverse_sweep(s.sigma, M, s.colk, sc, sc.sweep);
        if (!pd) b.status |= ST_NOT_PD;
        int cnt = 0;
        {
            PHASE(PH_IRLS_DIR);
            for (int j = EPIS ? 0 : 1; j < M; j++) cnt += fabs(g[j]) < 1e-6;
            for (int k = threadIdx.x; k < M; k += T) {
                double z = 0;
                for (int L = 0; L < M; L++) z = fma(s.sigma[L * M + k], g[L], z);
                dmu[k] = z;
            }
            __syncthreads();
        }
        if (cnt == (EPIS ? M : M - 1)) { converged = true; break; }
        double step = 1;
        PHASE(PH_IRLS_PRED);
        while (step > 1.0 / 256) {
            for (int j = threadIdx.x; j < M; j += T) mun[j] = s.mu[j] + step * dmu[j];
            __syncthreads();
            derr = predictor_and_error(s, N, M, mun, t, eta, yv, sc);
            current = false;
            reg = 0;
            for (int j = 1; j < M; j++) reg = reg + s.alpha[j - 1] * mun[j] * mun[j] / 2;
            total = derr + reg;
            if (total >= err_log) step = step / 2;
            else {
                __syncthreads();
                for (int j = threadIdx.x; j < M; j += T) s.mu[j] = mun[j];
                step = 0;
                current = true;
            }
            __syncthreads();
        }
    }
    b.at_mode = converged && current && pd;
    return current;                        // (IRLS work is not counted in the score-pass model)
}

template <bool EPIS, bool TC>
__device__ inline void binom_full_stat(const Problem &P, const FoldData &F, Slab &s, BinomState &b, double *sV,
                                       const Scratch &sc)
{   // fEBCatFullStat* (NEmainEff.c:1633-1803, NeFull.c:848-993)
    const int N = F.ntr, K = P.K, Kc = P.Kc, T = blockDim.x, LD = phi_ld(N);
    const double *t = F.ytr, *scale = F.scale;
    const bool current = post_mode<EPIS>(s, b, N, t, sc);
    const int M = b.M;
    double *yv = s.t, *e = s.e, *w = s.w1, *eta = s.w2;
    if (!EPIS && current) {
        // the posterior mode's last evaluation was at the final mu: predictor and probabilities are already in memory
        // (the Epis variant clamps the stored probabilities in place, NeFull.c:1049-1050, so it recomputes)
        for (int h = threadIdx.x; h < N; h += T) e[h] = t[h] - yv[h];
    } else
    for (int h = threadIdx.x; h < N; h += 2 * T) {
        const int h2 = h + T;
        const bool two = h2 < N;
        double z, z2;
        phi_rows_dot(s.phi, LD, M, s.mu, h, two ? h2 : h, z, z2);
        { eta[h] = z; const double y = 1 / (1 + exp(-z)); yv[h] = y; e[h] = t[h] - y; }
        if (two) { eta[h2] = z2; const double y = 1 / (1 + exp(-z2)); yv[h2] = y; e[h2] = t[h2] - y; }
    }
    __syncthreads();
    // One pass over the shared training matrix gives, per candidate c,
    //   bb = sum_h w[h] x_c[h]^2                        (BBsquare, :1728-1729)   -> S_in
    //   ze = sum_h x_c[h] e[h]                          (tempZE,  :1731-1732)    -> Q_in
    //   G[p][c] = sum_h x_c[h] phi_p[h] w[h] / s_c      (BPvector, :1693-1702)   -- kept as the action cache
    // on the int8 tensor cores where the fold carries their operand images (tc_contract.cuh), else in FP64 (DMMA)
    auto phi_col = [&](int r) -> const double * { return s.phi + (size_t)r * LD; };
    auto g_row = [&](int r, bool &dv) -> double * { dv = true; return s.G + (size_t)s.grow[r] * Kc; };
    if constexpr (TC) { tc_contract(F, Kc, M, phi_col, g_row, w, e, s.S_in, s.Q_in, s.planes, sV, *sc.tc); b.tc_calls += 1; }
    else contract_x<EPIS>(F, K, Kc, M, M, phi_col, g_row, sV, w, e, s.S_in, s.Q_in);
    quad_forms(s, s.sigma, s.sigma_new, M, Kc, nullptr, sc.sweep, [&](int c, double quad, double) {
        const double sc_c = scale[c];
        s.S_in[c] = s.S_in[c] / (sc_c * sc_c) - quad;
        s.Q_in[c] = s.Q_in[c] / sc_c;
    });
    if (threadIdx.x == 0) b.flops += 2.0 * N * (double)Kc * (M + 2) + (double)Kc * (2.0 * M * M + M);     // SURVEY 8d model: w, e and the M columns
    refresh_out(s, M - 1, Kc);
}

// TC: the score contraction runs on the int8 tensor cores (tc_contract.cuh; main effects, FoldData::Xtc present)
template <bool EPIS, bool TC>
__device__ void binom_fit(const Problem &P, const FoldData &F, const Variant &v, Slab &s, double lambda,
                          double alpha_en, const FitTask &task, const FitOutputs &out, double *sV, const Scratch &sc)
{
    const int N = F.ntr, K = P.K, Kc = P.Kc, cap = P.cap, T = blockDim.x, LD = phi_ld(N);   // cap counts the intercept slot
    const double *X = F.Xtr, *t = F.ytr, *scale = F.scale;
    BinomState b; b.M = 2; b.n_unused = 0; b.status = 0; b.flops = 0; b.tc_calls = 0; b.at_mode = false;
    for (int j = threadIdx.x; j < cap + 1; j += T) { if (j < cap) s.grow[j] = j; s.alpha[j] = 0; s.mu[j] = 0; }
    __syncthreads();
    double vk = 1e-30, vk0, err = 1000, loglik = 0;
    int iter = 0;
    while (iter < 100 && err > 1e-8) {                                        // NEmainEff.c:329-344
        iter++;
        vk0 = vk;
        // ------------------------- inner solver (fEBBinaryMex*, :397-827) -------------------------
        int ini_removed = 1;
        if (iter <= 1) {                                                      // initialisation, :1239-1385
            ini_removed = 0;
            b.M = 2;
            if (threadIdx.x == 0) s.used[0] = 1;
            const double sc0 = scale[0], isc = 1 / sc0;
            for (int h = N + threadIdx.x; h < LD; h += T) { s.phi[h] = 0; s.phi[(size_t)LD + h] = 0; }      // pad rows stay zero
            for (int h = threadIdx.x; h < N; h += T) {
                s.phi[h] = 1;
                const double x = X[(size_t)h * K];
                const double p1 = EPIS ? x / sc0 : x * isc;                   // NeFull.c:93 vs NEmainEff.c:1347-1350
                s.phi[(size_t)LD + h] = p1;
                double *pr = s.phit + (size_t)h * PHIT_LD;                    // row-major copy for the IRLS Gram matrix
                pr[0] = 1; pr[1] = p1;
                for (int j = 2; j < PHIT_LD; j++) pr[j] = 0;
            }
            __syncthreads();
            // least squares of [1 phi] on the pseudo-logits (dgelsy with rcond 1e-5, :1366-1370):
            // pivoted QR with the ones column leading (its norm sqrt(N) >= ||phi|| = 1)
            const double *ph = s.phi + LD;
            double sphi = 0, sz = 0;
            for (int h = threadIdx.x; h < N; h += T) {
                const double tp = 2 * t[h] - 1, pp = (tp * 0.9 + 1) / 2;
                const double z = log(pp / (1 - pp));
                s.e[h] = z;
                sphi += ph[h]; sz += z;
            }
            block_sum2(sphi, sz, sc);
            const double r11 = sqrt((double)N), r12 = sphi / r11, c1 = sz / r11;
            double r22 = 0, c2 = 0;
            for (int h = threadIdx.x; h < N; h += T) { const double vv = ph[h] - r12 / r11; r22 = fma(vv, vv, r22); c2 = fma(vv, s.e[h], c2); }
            block_sum2(r22, c2, sc);
            r22 = sqrt(r22);
            const double f = r11 * r11 + r12 * r12 + r22 * r22, dd = r11 * r22;
            const double disc = sqrt(fmax(f * f - 4 * dd * dd, 0.0));
            const double smax = sqrt((f + disc) / 2), smin = smax > 0 ? fabs(dd) / smax : 0;
            double w0, w1;
            if (r22 > 0 && smax * 1e-5 <= smin) { w1 = c2 / (r22 * r22); w0 = (c1 - r12 * w1) / r11; }
            else { const double den = r11 * r11 + r12 * r12; w0 = r11 * c1 / den; w1 = r12 * c1 / den; }
            double a = w1 == 0 ? 1 : 1 / (w1 * w1);
            if (a < v.init_alpha_min) a = v.init_alpha_min;
            if (a > v.init_alpha_max) a = v.init_alpha_max;
            __syncthreads();
            if (threadIdx.x == 0) { s.mu[0] = w0; s.mu[1] = w1; s.alpha[0] = a; }
        }
        __syncthreads();
        for (int c = threadIdx.x; c < Kc; c += T) s.amap[c] = -1;
        __syncthreads();
        for (int j = threadIdx.x; j < b.M - 1; j += T) s.amap[s.used[j] - 1] = j;
        __syncthreads();
        b.n_unused = block_compact(Kc, [&](int c) { return s.amap[c] < 0; }, s.unused, s.upos, 1, sc);
        const int initial = s.used[0];
        // Every block of actions ends with a FullStat and nothing changes mu, alpha or PHI after it, so at iter > 1 the
        // state is that of the last FullStat.  If its posterior mode stopped at a fixed point, FullStat would reproduce
        // w, e, SIGMA, G, S_in and Q_in bit for bit: it is skipped (main effects; the Epis variant clamps the stored
        // probabilities in place and recomputes them).  S_out/Q_out are refreshed as FullStat would (amap was rebuilt).
        if (EPIS || iter <= 1 || !b.at_mode) binom_full_stat<EPIS, TC>(P, F, s, b, sV, sc);
        else {
            if (threadIdx.x == 0) {   // counted as binom_full_stat counts it, and reported as not executed (out.flops[1])
                const double f = 2.0 * N * (double)Kc * (b.M + 2) + (double)Kc * (2.0 * b.M * b.M + b.M);
                b.flops += f;
                if (out.flops) atomicAdd(out.flops + 1, f);
            }
            refresh_out(s, b.M - 1, Kc);
        }
        int selected = ACT_NONE, last = 0, n_update = 0, jj = -1, i_iter = 0;
        const int it_max = iter == 1 ? 10 : 100;
        loglik = 1e-30;
        while (!last) {
            i_iter++;
            const double logl0 = loglik;
            Decision d = delta_ml<EPIS, true>(s, b.M - 1, N, Kc, lambda, alpha_en, 0.0, 0.0, iter, i_iter, sc);
            n_update = choose_block(s, v, d, b.M - 1, Kc, initial, selected, ini_removed, sc);
            for (int iu = 0; iu < n_update; iu++) {
                __syncthreads();
                const int nu = s.block[iu];
                selected = s.action[nu];
                const double new_alpha = s.aroot[nu];
                { PHASE(PH_ACTIONS);
                const bool need_sq = iu != n_update - 1;      // S/Q only matter to later actions of this block
                find_slot(s, nu, b.M - 1, jj, selected, b.status);
                if (selected == ACT_REEST && fabs(log(new_alpha) - log(s.alpha[jj])) <= v.reest_tol && !d.any_delete)
                    selected = ACT_TERM;                                          // :663-670
                const int M = b.M;
                if (selected == ACT_REEST) {                                      // ActionRes*, :1127-1203
                    const int j1 = jj + 1;
                    const double old = s.alpha[jj];
                    const double kappa = 1.0 / (s.sigma[j1 * M + j1] + 1.0 / (new_alpha - old));
                    const double mujj = s.mu[j1];
                    const double *sj = s.sigma + j1 * M;
                    __syncthreads();
                    if (threadIdx.x == 0) s.alpha[jj] = new_alpha;
                    mu_reest(s.mu, M, sj, mujj, kappa);
                    sigma_reest(s.sigma, s.sigma_new, M, j1, kappa);
                    __syncthreads();
                    { double *tp = s.sigma; s.sigma = s.sigma_new; s.sigma_new = tp; }
                    if (need_sq) {   // reads the UPDATED row j1 (the copy precedes the loop, :1166, 1191)
                        const double *sn = s.sigma + j1 * M;
                        cache_dot(s, M, Kc, sn, [&](int c, double z) {
                            s.S_in[c] += z * z * kappa;
                            s.Q_in[c] += mujj * kappa * z;
                        });
                        if (threadIdx.x == 0) b.flops += 2.0 * Kc * (double)M;
                    }
                } else if (selected == ACT_ADD) {                                 // ActionAdd*, :830-1003
                    const int n_used = M - 1;
                    if (n_used + 1 > cap - 1) { b.status |= ST_CAP; selected = ACT_TERM; }
                    else {
                        {
                            Cand<EPIS> cd(nu, K);
                            const double sc_nu = scale[nu], isc = 1 / sc_nu;
                            for (int h = threadIdx.x; h < N; h += T) {
                                const double x = cd.at(X + (size_t)h * K);
                                s.phinew[h] = EPIS ? x / sc_nu : x * isc;         // NeFull.c:253-262 vs NEmainEff.c:643-646
                            }
                        }
                        __syncthreads();
                        const int grow_new = s.grow[M];
                        if (need_sq) {
                            contract_x<EPIS>(F, K, Kc, 1, 0,
                                [&](int) -> const double * { return s.phinew; },
                                [&](int, bool &dv) -> double * { dv = true; return s.G + (size_t)grow_new * Kc; }, sV, s.w1);
                        }
                        {   // tmp = PHI' (w o phi_new), one warp per active column
                            const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
                            for (int i = wid; i < M; i += nw) {
                                const double *p = s.phi + (size_t)i * LD;
                                double z = 0;
                                for (int h = lane; h < N; h += 32) z = fma(p[h], s.w1[h] * s.phinew[h], z);
                                z = warp_sum(z);
                                if (lane == 0) s.tmp[i] = z;
                            }
                        }
                        __syncthreads();
                        for (int i = threadIdx.x; i < M; i += T) {
                            double z = 0;
                            for (int j = 0; j < M; j++) z = fma(s.sigma[i * M + j], s.tmp[j], z);
                            s.u[i] = z;
                        }
                        for (int h = N + threadIdx.x; h < LD; h += T) s.phi[(size_t)M * LD + h] = 0;
                        for (int h = threadIdx.x; h < N; h += T) {
                            s.phi[(size_t)M * LD + h] = s.phinew[h];
                            if (M < PHIT_LD) s.phit[(size_t)h * PHIT_LD + M] = s.phinew[h];
                        }
                        const double s_ii = 1.0 / (new_alpha + s.S_in[nu]);
                        const double mu_i = s_ii * s.Q_in[nu];
                        __syncthreads();
                        if (threadIdx.x == 0) s.alpha[n_used] = new_alpha;
                        mu_add(s.mu, M, s.u, mu_i);
                        sigma_add(s.sigma, s.sigma_new, M, s.u, s_ii);
                        if (need_sq) {
                            cache_dot(s, M, Kc, s.u, [&](int c, double z) {
                                const double mci = s.G[(size_t)grow_new * Kc + c] - z;
                                s.S_in[c] -= mci * mci * s_ii;
                                s.Q_in[c] -= mu_i * mci;
                            });
                        }
                        __syncthreads();
                        if (threadIdx.x == 0) {
                            s.used[n_used] = nu + 1;
                            s.amap[nu] = n_used;
                            const int p = s.upos[nu], nun = b.n_unused - 1;
                            if (p < nun) { const int lastc = s.unused[nun] - 1; s.unused[p] = lastc + 1; s.upos[lastc] = p; }
                            if (need_sq) b.flops += 2.0 * N * (double)Kc + 2.0 * Kc * (double)M;
                        }
                        { double *tp = s.sigma; s.sigma = s.sigma_new; s.sigma_new = tp; }
                        b.n_unused--;
                        b.M = M + 1;
                    }
                } else if (selected == ACT_DEL) {                                 // ActionDel*, :1010-1121
                    const int j1 = jj + 1, lastj = M - 1;
                    const double *sj = s.sigma + j1 * M;
                    const double sjj = sj[j1];
                    const double mujj = s.mu[j1];
                    const double al_last = s.alpha[lastj - 1];
                    __syncthreads();
                    if (need_sq) {
                        cache_dot(s, M, Kc, sj, [&](int c, double z) {
                            s.S_in[c] += z * z / sjj;
                            s.Q_in[c] += z * mujj / sjj;
                        });
                        if (threadIdx.x == 0) b.flops += 2.0 * Kc * (double)M;
                    }
                    sigma_delete<EPIS>(s.sigma, s.sigma_new, M, j1, nullptr);    // NeFull.c:1612 vs NEmainEff.c:1069
                    mu_delete(s.mu, M, sj, sjj, mujj);
                    for (int h = threadIdx.x; h < N; h += T) {
                        if (j1 != lastj) {
                            const double pv = s.phi[(size_t)lastj * LD + h];
                            s.phi[(size_t)j1 * LD + h] = pv;
                            if (j1 < PHIT_LD) s.phit[(size_t)h * PHIT_LD + j1] = pv;
                        }
                        if (lastj < PHIT_LD) s.phit[(size_t)h * PHIT_LD + lastj] = 0;     // vacated slot back to zero
                    }
                    __syncthreads();
                    if (threadIdx.x == 0) {
                        if (j1 != lastj) {
                            s.alpha[jj] = al_last;
                            s.mu[j1] = s.mu[lastj];
                            const int gr = s.grow[j1]; s.grow[j1] = s.grow[lastj]; s.grow[lastj] = gr;
                        }
                        const int moved = s.used[lastj - 1];
                        s.used[jj] = moved;
                        s.amap[nu] = -1;
                        if (jj != lastj - 1) s.amap[moved - 1] = jj;
                        s.unused[b.n_unused] = nu + 1; s.upos[nu] = b.n_unused;
                    }
                    { double *tp = s.sigma; s.sigma = s.sigma_new; s.sigma_new = tp; }
                    b.n_unused++;
                    b.M = M - 1;
                    if (nu + 1 == initial) ini_removed = 1;                       // :744
                }
                __syncthreads();
                }
                if (iu == n_update - 1) binom_full_stat<EPIS, TC>(P, F, s, b, sV, sc);          // after the last action of the block (:749-762)
            }
            if (selected == ACT_TERM && ini_removed) last = 1;
            if ((i_iter == it_max && b.M == 2) || i_iter > it_max) last = 1;
            if (i_iter == it_max) selected = ACT_TERM;
            {   // global log-likelihood and its relative change (:782-801)
                PHASE(PH_LOGLIK);
                // the linear predictor PHI mu is already in memory: FullStat left it in w2 after the posterior mode, and
                // mu has not changed since (every block of actions ends with a FullStat)
                const double *eta = s.w2;
                double ll = 0;
                for (int h = threadIdx.x; h < N; h += T) {
                    const double ez = exp(eta[h]);
                    ll += t[h] * log(ez / (1 + ez)) + (1 - t[h]) * log(1 / (1 + ez));
                }
                loglik = block_sum(ll, sc);
                const double dL = fabs((loglik - logl0) / logl0);
                if (dL < 1e-3) selected = ACT_TERM;
            }
        }
        {
            const int M = b.M;
            vk = 0;
            if (!EPIS) { for (int i = 0; i < M; i++) vk += fabs(s.alpha[i]); }        // dasum over m entries, one of them stale (:340)
            else { for (int i = 0; i < M - 1; i++) vk += s.alpha[i]; }                // NeFull.c:138-139
            err = fabs(vk - vk0) / M;
        }
    }
    if (iter >= 100) b.status |= ST_ITER_MAX;

    // ---------------- hold-out score (R/GetModelError.R:34-57) ----------------
    const int M = b.M;
    __syncthreads();
    for (int i = 1 + threadIdx.x; i < M; i += T) s.tmp[i] = s.mu[i] / scale[s.used[i - 1] - 1];
    __syncthreads();
    int nsel = 0;
    for (int i = 1; i < M; i++) nsel += s.tmp[i] != 0;
    double ll = 0;
    if (nsel > 0) {
        const double mu0 = s.mu[0];
        for (int h = threadIdx.x; h < F.nte; h += T) {
            const double *xr = F.Xte + (size_t)h * K;
            double pred = 0;
            for (int i = 1; i < M; i++) {
                const double wgt = s.tmp[i];
                if (wgt != 0) { Cand<EPIS> cd(s.used[i - 1] - 1, K); pred = fma(cd.at(xr), wgt, pred); }
            }
            double od = exp(mu0 + pred);
            if (od > 1e10) od = 1e5;
            if (od < 1e-10) od = 1e-5;
            ll += F.yte[h] * log(od / (1 + od)) + (1 - F.yte[h]) * log(1 / (1 + od));
        }
        ll = block_sum(ll, sc) / F.nte;
    }
    if (F.nte > 0 && !isfinite(ll)) b.status |= ST_NONFINITE;      // (no held-out rows in an all-rows fit: nothing to score)
    if (threadIdx.x == 0) {
        const int o = task.out_index;
        write_fit_outputs(out, o, ll, b.status, nsel, iter, b.flops, 0, b.tc_calls);
        if (out.m_out)            // slot 0 is the intercept
            write_record(out, o, M, 1, s.mu, s.H, s.sigma, s.used, [&](int k) { return scale[s.used[k] - 1]; }, s.mu[0], s.sigma[0], loglik);
    }
    __syncthreads();
}

}  // namespace pareben
