// gauss_fit.cuh -- one Gaussian EBEN fit per thread block (main-effect and Epis variants).
//
// Device re-design of the reference's Gaussian solver; behaviour follows
//   /root/reference/EBEN_orig/src/elasticNetLinearNeMainEff.c (entry :55-242, inner solver
//   :248-809, init :976-1108, CacheBP :1144-1201, FullStat :1209-1341, DeltaML :1372-1582,
//   ActionAdd :1585-1723, ActionDel :1725-1822, FinalUpdate :1841-1921)
//   and elasticNetLinearNeFull2.c for Epis (same skeleton, constants per SURVEY.md App. A),
// followed by the hold-out score of /root/reference/R/GetModelError.R:6-32.
// Differences in kind, not in result: the N x N matrix C_inv (:742-781) is never formed (only
// 1'C^-1 1 and 1'C^-1 y are needed, :172-188); the SPD inverse is an in-block symmetric sweep
// instead of dpotrf/dpotri; the candidate cache is stored as physical rows + a permutation;
// pair columns for Epis are generated on the fly from two loci and never stored.
#pragma once
#include "common.cuh"
#include "contract.cuh"
#include "linalg.cuh"
#include "eben_step.cuh"

namespace pareben {

struct GaussState {
    int M, n_unused, cap;
    double beta;
    int status;
    double flops;
    double avoided;          // the part of `flops` (SURVEY 8d model) that the Gram organisation did not execute
};

__device__ inline void posterior_mean(Slab &s, GaussState &g, int N)
{   // Mu = beta * SIGMA * PHI' t   (MainEff.c:1256-1280)
    // PHI' t needs no pass over PHI: column j of PHI is candidate used[j]'s normalised column, and x_c' t / s_c is
    // xt[c], computed for every candidate by the contraction at the top of the outer iteration (t has not changed since).
    const int M = g.M;
    (void)N;
    for (int j = threadIdx.x; j < M; j += blockDim.x) s.tmp[j] = s.xt[s.used[j] - 1];
    __syncthreads();
    for (int i = threadIdx.x; i < M; i += blockDim.x) s.mu[i] = sym_matvec_row(s.sigma, M, i, s.tmp) * g.beta;
    __syncthreads();
}

__device__ inline void full_stat(Slab &s, GaussState &g, int N, int Kc, bool first, const Scratch &sc)
{   // fEBLinearFullStat* (MainEff.c:1209-1341)
    const int M = g.M;
    if (first) {                                                    // :1236-1246
        double h = 0;
        for (int k = threadIdx.x; k < N; k += blockDim.x) h = fma(s.phi[k], s.phi[k], h);
        h = block_sum(h, sc);
        if (threadIdx.x == 0) { s.ptp[0] = h; s.H[0] = h * g.beta + s.alpha[0]; s.sigma[0] = 1.0 / s.H[0]; }
        __syncthreads();
    }
    posterior_mean(s, g, N);
    for (int i = 1 + threadIdx.x; i < M; i += blockDim.x) s.gamma[i] = 1.0 - s.sigma[i * M + i] * s.alpha[i];
    const double beta = g.beta;
    __syncthreads();
    quad_forms(s, s.sigma, s.sigma_new, M, Kc, s.mu, sc.sweep, [&](int c, double quad, double gm) {
        s.S_in[c] = beta - beta * quad * beta;
        s.Q_in[c] = beta * (s.xt[c] - gm);
    });
    if (threadIdx.x == 0) g.flops += (double)Kc * (2.0 * M * M + 2.0 * M);
    refresh_out(s, M, Kc);
}

__device__ inline bool final_update(Slab &s, GaussState &g, int N, const Scratch &sc, bool keep_H)
{   // FinalUpdate*: H = beta PHI'PHI + diag(alpha), SIGMA = H^-1, Mu  (MainEff.c:1841-1921)
    // PHI'PHI is not recomputed (the reference's dgemm, :1869-1874): it is kept up to date by the add and delete
    // actions -- a new column's products with the active columns are entries of the cache row the add has just
    // computed (G[new][c] = x_c' phi_new / s_c) -- so this is an M x M pass, not N x M x M.
    const int M = g.M, cap = g.cap;
    const double beta = g.beta;
    (void)N;
    for (int j = threadIdx.x >> 5; j < M; j += blockDim.x >> 5)
        for (int i = threadIdx.x & 31; i < M; i += 32) {
            double v = s.ptp[(size_t)j * cap + i] * beta;
            if (i == j) v += s.alpha[i];
            if (keep_H) s.H[j * M + i] = v;       // read by the Wald score of a full-model dump only (:206-215): a CV fit never writes it
            s.sigma[j * M + i] = v;
        }
    __syncthreads();
    const bool ok = spd_inverse_sweep(s.sigma, M, s.colk, sc, sc.sweep);
    posterior_mean(s, g, N);
    return ok;
}

// One complete Gaussian fit.  Every thread of the block executes this with identical scalars.
template <bool EPIS>
__device__ void gauss_fit(const Problem &P, const FoldData &F, const Variant &v, Slab &s, double lambda,
                          double alpha_en, const FitTask &task, const FitOutputs &out, double *sV,
                          const Scratch &sc)
{
    const int N = F.ntr, K = P.K, Kc = P.Kc, cap = P.cap, T = blockDim.x, LD = phi_ld(N);
    const int lane_ = threadIdx.x & 31, wid_ = threadIdx.x >> 5, nw_ = T >> 5;
    const double *X = F.Xtr, *y = F.ytr, *scale = F.scale;
    GaussState g; g.M = 1; g.n_unused = 0; g.cap = cap; g.beta = 0; g.status = 0; g.flops = 0; g.avoided = 0;
    // Gram organisation: the cache row of basis p is row p of the fold's shared matrix C (FoldData::C), so the cache is
    // never computed or stored per fit -- `grow[j]` simply holds the candidate id of active slot j, and every reader of
    // the cache (quadratic forms, S/Q corrections) streams rows that all fits of the fold share in L2.
    const bool gram = F.C != nullptr;
    if (gram) s.G = F.C;

    for (int j = threadIdx.x; j < cap; j += T) { s.grow[j] = j; s.alpha[j] = 0; s.mu[j] = 0; }
    double b = 0;
    for (int h = threadIdx.x; h < N; h += T) b += y[h];
    b = block_sum(b, sc) / N;
    const double var_y = block_var(y, N, sc);
    const double eps = var_y * 0.01;
    double residvar = 1e10, vk = 1e-30, vk0, err = 1000;
    int iter = 0;

    while (iter < 100 && err > 1e-8 && residvar >= eps) {          // MainEff.c:155-197
        iter++;
        vk0 = vk;
        for (int h = threadIdx.x; h < N; h += T) s.t[h] = y[h] - b;
        __syncthreads();
        const double vt = block_var(s.t, N, sc);                    // t is fixed for the whole inner solver (:705 recomputes it per noise update)
        double tt = 0;
        for (int h = threadIdx.x; h < N; h += T) tt = fma(s.t[h], s.t[h], tt);
        tt = block_sum(tt, sc);
        // ---------------- inner solver (LinearFastEmpBayes*, MainEff.c:248-809) ----------------
        int ini_removed = 1;
        if (iter <= 1) {                                             // initialisation, :1003-1090
            ini_removed = 0;
            g.M = 1;
            if (threadIdx.x == 0) s.used[0] = 1;
            const double isc = 1 / scale[0];
            for (int h = threadIdx.x; h < LD; h += T) s.phi[h] = h < N ? X[(size_t)h * K] * isc : 0.0;      // pad rows stay zero
            __syncthreads();
            gauss_start<EPIS>(s.phi, s.t, N, v, g.beta, s.alpha, sc);
        }
        __syncthreads();
        // Used -> amap; Unused rebuilt in ascending order (:1092-1107)
        for (int c = threadIdx.x; c < Kc; c += T) s.amap[c] = -1;
        for (int j = threadIdx.x; j < cap; j += T) s.gamma[j] = 0;       // gamma is Calloc'ed per call (:344)
        __syncthreads();
        for (int j = threadIdx.x; j < g.M; j += T) s.amap[s.used[j] - 1] = j;
        __syncthreads();
        g.n_unused = block_compact(Kc, [&](int c) { return s.amap[c] < 0; }, s.unused, s.upos, 1, sc);
        const int initial = s.used[0];
        // candidate cache G = PHI'X/s and xt = X't/s  (CacheBP*, :1144-1201)
        {
            const int M = g.M;
            if (gram)       // only xt depends on the fit (t = y - b); the M cache rows are rows of C
                contract_x<EPIS>(F, K, Kc, 1, 0,
                    [&](int) -> const double * { return s.t; },
                    [&](int, bool &dv) -> double * { dv = true; return s.xt; }, sV);
            else
                contract_x<EPIS>(F, K, Kc, M + 1, M,
                    [&](int r) -> const double * { return r < M ? s.phi + (size_t)r * LD : s.t; },
                    [&](int r, bool &dv) -> double * { dv = true; return r < M ? s.G + (size_t)s.grow[r] * Kc : s.xt; },
                    sV);
            if (threadIdx.x == 0) { g.flops += 2.0 * N * (double)Kc * (M + 1); if (gram) g.avoided += 2.0 * N * (double)Kc * M; }     // the SURVEY 8d model of this step
        }
        int i_iter = 0;
        full_stat(s, g, N, Kc, iter == 1, sc);
        int selected = ACT_NONE, last = 0, n_update = 0, jj = -1;
        const int it_max = iter == 1 ? 10 : 100;
        while (!last) {
            i_iter++;
            Decision d = delta_ml<EPIS, false>(s, g.M, N, Kc, lambda, alpha_en, residvar, var_y, iter, i_iter, sc);
            n_update = choose_block(s, v, d, g.M, Kc, initial, selected, ini_removed, sc);
            for (int iu = 0; iu < n_update; iu++) {
                __syncthreads();
                const int nu = s.block[iu];
                selected = s.action[nu];
                const double new_alpha = s.aroot[nu];
                find_slot(s, nu, g.M, jj, selected, g.status);
                if (selected == ACT_REEST && fabs(log(new_alpha) - log(s.alpha[jj])) <= v.reest_tol && !d.any_delete)
                    selected = ACT_TERM;                                       // :541-549
                const int M = g.M;
                bool updated = false;
                { PHASE(PH_ACTIONS);
                if (selected == ACT_REEST) {                                   // :553-596
                    const double old = s.alpha[jj];
                    const double kappa = 1.0 / (s.sigma[jj * M + jj] + 1.0 / (new_alpha - old));
                    const double mujj = s.mu[jj];
                    const double *sj = s.sigma + jj * M;
                    __syncthreads();
                    if (threadIdx.x == 0) s.alpha[jj] = new_alpha;
                    mu_reest(s.mu, M, sj, mujj, kappa);
                    sigma_reest(s.sigma, s.sigma_new, M, jj, kappa);
                    const double beta = g.beta;
                    cache_dot(s, M, Kc, sj, [&](int c, double z) {
                        const double bz = beta * z;
                        s.S_in[c] += bz * bz * kappa;
                        s.Q_in[c] += beta * mujj * kappa * z;
                    });
                    if (threadIdx.x == 0) g.flops += 2.0 * Kc * (double)M;
                    updated = true;
                } else if (selected == ACT_ADD) {                              // ActionAdd*, :1585-1723
                    if (M + 1 > cap) { g.status |= ST_CAP; selected = ACT_TERM; }
                    else {
                        // new normalised column (on the fly for pairs)
                        {
                            Cand<EPIS> cd(nu, K);
                            const double sc_nu = scale[nu], isc = 1 / sc_nu;
                            const bool pair = cd.i != cd.j;     // pairs are divided, main effects scaled by 1/s (NeFull2.c:277-290)
                            for (int h = threadIdx.x; h < N; h += T) {
                                const double x = cd.at(X + (size_t)h * K);
                                s.phinew[h] = pair ? x / sc_nu : x * isc;
                            }
                        }
                        __syncthreads();
                        const int grow_new = gram ? nu : s.grow[M];
                        if (gram) { if (threadIdx.x == 0) s.grow[M] = nu; }          // row nu of C is the new cache row
                        else
                        contract_x<EPIS>(F, K, Kc, 1, 0,
                            [&](int) -> const double * { return s.phinew; },
                            [&](int, bool &dv) -> double * { dv = true; return s.G + (size_t)grow_new * Kc; }, sV);
                        // tmp = beta PHI' phi_new: the entries are already in the cache row just computed
                        // (G[new][c] = x_c' phi_new / s_c), at the active candidates
                        __syncthreads();
                        for (int j = threadIdx.x; j < M; j += T) {
                            const double pj = s.G[(size_t)grow_new * Kc + s.used[j] - 1];      // phi_j' phi_new
                            s.tmp[j] = g.beta * pj;
                            s.ptp[(size_t)j * cap + M] = pj; s.ptp[(size_t)M * cap + j] = pj;
                        }
                        if (threadIdx.x == 0) s.ptp[(size_t)M * cap + M] = s.G[(size_t)grow_new * Kc + nu];
                        __syncthreads();
                        for (int i = threadIdx.x; i < M; i += T) s.u[i] = sym_matvec_row(s.sigma, M, i, s.tmp);
                        for (int h = threadIdx.x; h < LD; h += T) s.phi[(size_t)M * LD + h] = h < N ? s.phinew[h] : 0.0;
                        const double s_ii = 1.0 / (new_alpha + s.S_in[nu]);
                        const double mu_i = s_ii * s.Q_in[nu];
                        __syncthreads();
                        if (threadIdx.x == 0) { s.alpha[M] = new_alpha; }
                        mu_add(s.mu, M, s.u, mu_i);
                        sigma_add(s.sigma, s.sigma_new, M, s.u, s_ii);
                        const double beta = g.beta;
                        cache_dot(s, M, Kc, s.u, [&](int c, double z) {
                            const double mci = beta * s.G[(size_t)grow_new * Kc + c] - beta * z;
                            s.S_in[c] -= mci * mci * s_ii;
                            s.Q_in[c] -= mu_i * mci;
                        });
                        __syncthreads();
                        if (threadIdx.x == 0) {
                            s.used[M] = nu + 1;
                            s.amap[nu] = M;
                            const int p = s.upos[nu], nun = g.n_unused - 1;   // Unused: swap-with-last (:621-625)
                            if (p < nun) { const int lastc = s.unused[nun] - 1; s.unused[p] = lastc + 1; s.upos[lastc] = p; }
                            g.flops += 2.0 * N * (double)Kc + 2.0 * Kc * (double)M;
                            if (gram) g.avoided += 2.0 * N * (double)Kc;
                        }
                        g.n_unused--;
                        g.M = M + 1;
                        updated = true;
                    }
                } else if (selected == ACT_DEL) {                              // ActionDel*, :1725-1822
                    const int lastj = M - 1;
                    const int mujj = (int)s.mu[jj];                            // `int Mujj` truncation (:1746-1747)
                    const double *sj = s.sigma + jj * M;
                    const double sjj = sj[jj];
                    const double al_last = s.alpha[lastj];
                    __syncthreads();
                    mu_delete(s.mu, M, sj, sjj, mujj);
                    for (int h = threadIdx.x; h < N; h += T) s.phi[(size_t)jj * LD + h] = s.phi[(size_t)lastj * LD + h];
                    ptp_move_last(s.ptp, cap, jj, lastj);
                    sigma_delete<true>(s.sigma, s.sigma_new, M, jj, s.colk);
                    const double beta = g.beta;
                    cache_dot(s, M, Kc, sj, [&](int c, double z) {
                        const double bz = beta * z;
                        s.S_in[c] += bz * bz / sjj;
                        s.Q_in[c] += beta * z * mujj / sjj;
                    });
                    __syncthreads();
                    if (threadIdx.x == 0) {
                        s.alpha[jj] = al_last;
                        // mu[jj] must be the *updated* last entry
                        s.mu[jj] = s.mu[lastj];
                        const int gr = s.grow[jj]; s.grow[jj] = s.grow[lastj]; s.grow[lastj] = gr;
                        const int moved = s.used[lastj];
                        // The basis that leaves is the one in slot jj.  That is candidate nu, except in the forced
                        // removal of an initial basis that a regular delete has already taken out (:437-446): the
                        // reference's search of Used then fails, jj keeps its previous value and ANOTHER basis is
                        // dropped -- while it is candidate nu that is appended to Unused (:621-625).  The dropped one
                        // is then in neither list: no scan sees it until Unused is rebuilt at the next outer
                        // iteration (:1092-1107).  amap = -2 reproduces that.
                        const int dropped = s.used[jj] - 1;
                        s.used[jj] = moved;
                        s.amap[dropped] = dropped == nu ? -1 : -2;
                        if (jj != lastj) s.amap[moved - 1] = jj;
                        s.unused[g.n_unused] = nu + 1; s.upos[nu] = g.n_unused;
                        g.flops += 2.0 * Kc * (double)M;
                    }
                    g.n_unused++;
                    g.M = M - 1;
                    updated = true;
                }
                __syncthreads();
                }
                if (updated) {                                                 // :657-681
                    PHASE(PH_OTHER);
                    double *tmpp = s.sigma; s.sigma = s.sigma_new; s.sigma_new = tmpp;
                    refresh_out(s, g.M, Kc);
                    const int Mn = g.M;
                    for (int i = threadIdx.x; i < Mn; i += T) s.gamma[i] = 1 - s.alpha[i] * s.sigma[i * Mn + i];
                    __syncthreads();
                }
            }
            if (selected == ACT_TERM || i_iter <= 10 || i_iter % 5 == 0 || n_update >= 2) {      // :685-729
                const int M = g.M;
                double ee = 0;
                { PHASE(PH_LOGLIK);
                // ||t - PHI mu||^2 = t't - 2 mu'(PHI't) + mu'(PHI'PHI)mu: PHI't is xt at the active candidates and PHI'PHI is
                // kept by the actions, so the residual costs M^2 instead of a pass over the N x M matrix PHI (the
                // cancellation costs a factor t't / ee <= 100 in relative accuracy -- the outer loop stops at 1 % -- of 1e-16)
                double part = 0;
                for (int j = wid_; j < M; j += nw_) {
                    const double *pr = s.ptp + (size_t)j * cap;
                    double z = 0;
                    for (int i = lane_; i < M; i += 32) z = fma(pr[i], s.mu[i], z);
                    z = warp_sum(z);
                    if (lane_ == 0) part += s.mu[j] * (z - 2 * s.xt[s.used[j] - 1]);
                }
                ee = tt + block_sum(part, sc);
                }
                double sg = 0;
                for (int i = 0; i < M; i++) sg += s.gamma[i];
                const double beta_old = g.beta;
                g.beta = (N - sg) / ee;
                if (g.beta > 1e6 / vt) g.beta = 1e6 / vt;
                if (fabs(log(g.beta) - log(beta_old)) > 1e-6) {
                    if (!final_update(s, g, N, sc, out.m_out != nullptr)) g.status |= ST_NOT_PD;
                    if (selected != ACT_TERM) full_stat(s, g, N, Kc, false, sc);
                }
            }
            if (selected == ACT_TERM && ini_removed) last = 1;
            if ((i_iter == it_max && g.M == 1) || i_iter > it_max) last = 1;
            if (i_iter == it_max) selected = ACT_TERM;
        }
        // ---------------- intercept update: b = 1'C^-1 y / (1'C^-1 1 [+1e-10]) ----------------
        {
            const int M = g.M;
            const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
            for (int j = wid; j < M; j += nw) {
                const double *p = s.phi + (size_t)j * LD;
                double a1 = 0, ay = 0;
                for (int h = lane; h < N; h += 32) { a1 += p[h]; ay = fma(p[h], y[h], ay); }
                a1 = warp_sum(a1); ay = warp_sum(ay);
                if (lane == 0) { s.tmp[j] = a1; s.u[j] = ay; }
            }
            __syncthreads();
            double q11 = 0, q1y = 0, sy = 0;
            for (int j = threadIdx.x; j < M; j += T) {
                const double z = sym_matvec_row(s.sigma, M, j, s.tmp);
                q11 = fma(z, s.tmp[j], q11); q1y = fma(z, s.u[j], q1y);
            }
            block_sum2(q11, q1y, sc);
            for (int h = threadIdx.x; h < N; h += T) sy += y[h];
            sy = block_sum(sy, sc);
            const double cinv = g.beta * N - g.beta * g.beta * q11;
            const double cinvy = g.beta * sy - g.beta * g.beta * q1y;
            b = EPIS ? cinvy / cinv : cinvy / (cinv + 1e-10);                      // MainEff.c:188 vs NeFull2.c:202
            vk = 0;
            for (int i = 0; i < M; i++) vk += s.alpha[i];
            err = fabs(vk - vk0) / M;
            residvar = 1 / (g.beta + 1e-10);
        }
    }
    if (iter >= 100) g.status |= ST_ITER_MAX;

    // ---------------- hold-out score (R/GetModelError.R:6-32) ----------------
    const int M = g.M;
    auto norm = [&](int i) { return scale[s.used[i] - 1]; };
    int nsel;
    const double sse = gauss_holdout_sse<EPIS>(F, K, M, s.mu, s.used, b, s.tmp, norm, nsel, g.status, sc);
    if (threadIdx.x == 0) {
        const int o = task.out_index;
        write_fit_outputs(out, o, sse, g.status, nsel, iter, g.flops, g.avoided, 0);
        if (out.m_out) write_record(out, o, M, 0, s.mu, s.H, s.sigma, s.used, norm, b, 0, 1 / (g.beta + 1e-10));
    }
    __syncthreads();
}

}  // namespace pareben
