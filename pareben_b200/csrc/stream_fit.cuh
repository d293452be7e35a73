// stream_fit.cuh -- streaming mode, the per-fit half: one thread block advances one Gaussian EBEN fit from the
// results of the last score scan to the next point where the solver needs per-candidate statistics (the call of
// fEBDeltaML at the top of every inner iteration, MainEff.c:420 / NeFull2.c:437), then publishes its residual
// e' = t - PHI mu - d as a column of the fold's right-hand-side matrix and returns.  The control flow is
// gauss_fit()'s (gauss_fit.cuh; reference MainEff.c:124-197 outer loop, :248-809 inner solver) cut at that one
// point: the loop-carried scalars live in StreamFit between launches.  What differs from the cached kernel:
//   * no candidate cache, no Kc-length arrays: the statistics of the IN-model candidates are recomputed here from
//     PHI'PHI, SIGMA, mu (O(M^3) per iteration), those of the out-of-model candidates by stream_scan_kernel;
//   * an ADD recomputes S and Q of the candidate it adds at the moment it is applied (earlier actions of the same
//     block have changed them, exactly as the reference's incremental corrections would have);
//   * column norms are computed when a column enters the model (exact sums for genotype codes).
#pragma once
#include "stream.cuh"
#include "linalg.cuh"
#include "eben_step.cuh"

namespace pareben {

// raw candidate column c over the training rows -> out[h], and its norm (1 when all zero; MainEff.c:96-98)
template <bool EPIS>
__device__ inline double stream_column(const FoldData &F, int K, int c, double *out, const Scratch &sc)
{
    const int N = F.ntr, T = blockDim.x;
    Cand<EPIS> cd(c, K);
    double z = 0;
    for (int h = threadIdx.x; h < N; h += T) {
        const double x = F.Xtr8 ? cd.at(F.Xtr8 + (size_t)h * K) : cd.at(F.Xtr + (size_t)h * K);
        out[h] = x;
        z = fma(x, x, z);
    }
    z = block_sum(z, sc);
    if (z == 0) z = 1;
    return sqrt(z);
}

// out[j] = sum_h phi_j[h] * v[h], j < M (a warp per column, fixed-order warp reduction)
__device__ inline void phi_t_vec(const double *phi, int N, int LD, int M, const double *v, double *out)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int j = wid; j < M; j += nw) {
        const double *p = phi + (size_t)j * LD;
        double z = 0;
        for (int h = lane; h < N; h += 32) z = fma(p[h], v[h], z);
        z = warp_sum(z);
        if (lane == 0) out[j] = z;
    }
    __syncthreads();
}

// e[h] = t[h] - sum_j phi_j[h] mu_j - (d ? d[h] : 0); returns sum e^2
__device__ inline double stream_residual(const StreamFit &s, int N, int LD, int M, const double *d, double *e, const Scratch &sc)
{
    double ee = 0;
    for (int h = threadIdx.x; h < N; h += blockDim.x) {
        double pm = 0;
        for (int j = 0; j < M; j++) pm = fma(s.phi[(size_t)j * LD + h], s.mu[j], pm);
        double r = s.t[h] - pm;
        if (d) r -= d[h];
        e[h] = r;
        ee = fma(r, r, ee);
    }
    return block_sum(ee, sc);
}

// Mu = beta * SIGMA * PHI' t (MainEff.c:1256-1280)
__device__ inline void stream_posterior_mean(StreamFit &s, int N, int LD, int M, double beta)
{
    phi_t_vec(s.phi, N, LD, M, s.t, s.tmp);
    for (int i = threadIdx.x; i < M; i += blockDim.x) {
        double z = 0;
        for (int j = 0; j < M; j++) z = fma(s.sigma[j * M + i], s.tmp[j], z);
        s.mu[i] = z * beta;
    }
    __syncthreads();
}

template <bool EPIS>
__global__ void __launch_bounds__(ADV_THREADS)
stream_advance_kernel(Problem P, Variant v, StreamFit *fits, int n_fits, StreamShared sh, FitOutputs out)
{
    extern __shared__ __align__(32) double s_buf[];           // SWEEP_PANEL_DOUBLES
    __shared__ double red[66];
    __shared__ int redi[66];
    __shared__ int s_slot;
    Scratch sc{red, redi, s_buf, nullptr};
    if ((int)blockIdx.x >= n_fits) return;
    StreamFit &G = fits[blockIdx.x];
    if (G.phase == SP_DONE) return;
    StreamFit s = G;                                          // local copy: pointers and scalars (written back at the end)
    const FoldData F = P.folds[s.target * (P.n_folds + 1) + s.fold];
    const int N = F.ntr, K = P.K, cap = P.cap, T = blockDim.x, LD = phi_ld(N);
    const int lane_ = threadIdx.x & 31, wid_ = threadIdx.x >> 5, nw_ = T >> 5;
    const double *y = F.ytr;
    const double lambda = s.lambda, alpha_en = s.alpha_en;
    const double l1 = lambda * alpha_en, l2 = lambda * (1 - alpha_en);
    bool resume = s.phase == SP_WAIT;
    int last = 0;
    double eps;

    if (!resume) {
        s.M = 1; s.beta = 0; s.beta_s = 0; s.status = 0; s.flops = 0;
        for (int j = threadIdx.x; j < cap; j += T) { s.alpha[j] = 0; s.mu[j] = 0; }
        double b = 0;
        for (int h = threadIdx.x; h < N; h += T) b += y[h];
        s.b = block_sum(b, sc) / N;
        s.var_y = block_var(y, N, sc);
        s.residvar = 1e10; s.vk = 1e-30; s.vk0 = 0; s.err = 1000; s.iter = 0;
    }
    eps = s.var_y * 0.01;

    for (;;) {
        if (!resume) {
            if (!(s.iter < 100 && s.err > 1e-8 && s.residvar >= eps)) break;          // MainEff.c:155
            s.iter++;
            s.vk0 = s.vk;
            for (int h = threadIdx.x; h < N; h += T) { s.t[h] = y[h] - s.b; s.d[h] = 0; }
            __syncthreads();
            s.ini_removed = 1;
            if (s.iter <= 1) {                                                        // initialisation, :1003-1090
                s.ini_removed = 0;
                s.M = 1;
                if (threadIdx.x == 0) s.used[0] = 1;
                const double sc0 = stream_column<EPIS>(F, K, 0, s.phinew, sc);
                const double isc = 1 / sc0;
                __syncthreads();
                if (threadIdx.x == 0) s.ascale[0] = sc0;
                for (int h = threadIdx.x; h < LD; h += T) s.phi[h] = h < N ? s.phinew[h] * isc : 0.0;
                __syncthreads();
                gauss_start<EPIS>(s.phi, s.t, N, v, s.beta, s.alpha, sc);
            }
            __syncthreads();
            for (int j = threadIdx.x; j < cap; j += T) s.gamma[j] = 0;               // gamma is Calloc'ed per call (:344)
            __syncthreads();
            s.initial = s.used[0];
            // FullStat (:1209-1341) minus the per-candidate part
            if (s.iter == 1) {
                double h = 0;
                for (int k = threadIdx.x; k < N; k += T) h = fma(s.phi[k], s.phi[k], h);
                h = block_sum(h, sc);
                if (threadIdx.x == 0) { s.ptp[0] = h; s.H[0] = h * s.beta + s.alpha[0]; s.sigma[0] = 1.0 / s.H[0]; }
                __syncthreads();
            }
            stream_posterior_mean(s, N, LD, s.M, s.beta);
            for (int i = 1 + threadIdx.x; i < s.M; i += T) s.gamma[i] = 1.0 - s.sigma[i * s.M + i] * s.alpha[i];
            __syncthreads();
            s.beta_s = s.beta;
            s.stats_valid = 0;                                                        // CacheBP + FullStat: everything is recomputed
            s.n_hidden = 0;                                                           // Unused is rebuilt from Used (:1092-1107)
            s.i_iter = 0; s.selected = ACT_NONE; s.n_update = 0; s.jj = -1;
            s.it_max = s.iter == 1 ? 10 : 100;
        }
        // ---------------- inner solver, one pass per scan ----------------
        for (;;) {
            // An iteration that applied no action and did not re-base the statistics leaves the reference's S/Q arrays
            // untouched (even when FinalUpdate has meanwhile replaced SIGMA and Mu, :716-727): its next fEBDeltaML sees
            // exactly what the last one saw.  Only a change asks for a new scan.
            const bool reuse = !resume && s.stats_valid;
            if (!resume && !reuse) {
                // request: publish e' and the screens, hand the fit to the scan kernel
                (void)stream_residual(s, N, LD, s.M, s.d, s.e, sc);
                // right-hand-side class (stream.cuh): a fit on the initial basis brings phi_0 along
                const int cls = (s.M == 1 && s.used[0] == 1) ? 1 : 0;
                const int vf = STREAM_CLASSES * s.fold + cls;
                if (threadIdx.x == 0) s_slot = atomicAdd(sh.n_slots + vf, 1);
                __syncthreads();
                const int idx = s_slot, per = class_fits_per_tile(cls);
                const int slot = (idx / per) * SN + (cls == 1 ? 1 + idx % per : idx % per);
                const StreamFold SF = sh.folds[vf];
                double *Et = SF.E + (size_t)(slot / SN) * e_tile_doubles(F.ldt);
                double *E = Et + (size_t)(slot % SN) * SLD;
                for (int h = threadIdx.x; h < F.ldt; h += T) {
                    const size_t o = (size_t)(h / SK) * STAGE_D + (h % SK);
                    E[o] = h < N ? s.e[h] : 0.0;
                    if (cls == 1) Et[o] = h < N ? s.phi[h] : 0.0;          // every fit of the tile writes the same bytes
                }
                if (threadIdx.x == 0) {
                    double thr_q2 = (2 * l1 + l2) * (1 - 1e-6) - 1e-10 * s.beta_s;       // Q^2 must exceed S + 2 l1 + l2 > this
                    if (!(thr_q2 > 0)) thr_q2 = 0;
                    double inv = 1 / s.beta_s;
                    for (int j = 0; j < s.M; j++) inv += 1 / s.alpha[j];
                    double s_lb = 1 / inv - 1e-4 * s.beta_s;                             // slack: SIGMA follows beta to 1e-6 only
                    if (!(s_lb > 0)) s_lb = 0;
                    ScanSlot *sp = SF.par + slot;
                    sp->bs = s.beta_s; sp->sig = s.sigma[0]; sp->l1 = l1; sp->l2 = l2; sp->s_lb = s_lb;
                    for (int k = 0; k < 8; k++) sp->T[k] = 0;
                    // (main effects keep screen 1 only: anyToAdd needs every a < 0)
                    slot_thresholds(sp, v.ml_delta * (1 - 1e-9), thr_q2, EPIS);
                    s.s_lb = s_lb;
                    SF.slot_fit[slot] = blockIdx.x;
                    s.slot = slot; s.cls = cls; s.l1 = l1; s.l2 = l2; s.ml_delta = v.ml_delta; s.n_add = v.n_add;
                    s.runmax = 0ull; s.n_list = 0; s.any_add = 0;
                    s.phase = SP_WAIT;
                    s.flops += 2.0 * N * (double)P.Kc;
                    G = s;
                }
                return;
            }
            resume = false;
            s.i_iter++;
            const int M0 = s.M;
            // ---- statistics of the in-model candidates: g_j = column j of PHI'PHI ----
            if (!reuse) {
            (void)stream_residual(s, N, LD, M0, s.d, s.e, sc);
            phi_t_vec(s.phi, N, LD, M0, s.e, s.q_in);                    // phi_j' e'
            for (int j = wid_; j < M0; j += nw_) {
                double quad = 0;
                for (int i = lane_; i < M0; i += 32) {
                    double z = 0;
                    for (int k = 0; k < M0; k++) z = fma(s.sigma[(size_t)k * M0 + i], s.ptp[(size_t)j * cap + k], z);
                    quad = fma(z, s.ptp[(size_t)j * cap + i], quad);
                }
                quad = warp_sum(quad);
                if (lane_ == 0) s.s_in[j] = s.beta_s - s.beta_s * quad * s.beta_s;
            }
            }
            s.stats_valid = 1;
            __syncthreads();
            // ---- fEBDeltaML (MainEff.c:1372-1582): in-model here, out-of-model from the scan's list ----
            int prio_add = 0, prio_del = 0;
            if (M0 < 10) { prio_add = 1; prio_del = 0; }
            if (M0 > 100 || (!EPIS && M0 >= N) || (s.residvar <= s.var_y * 0.1)) { prio_add = 0; prio_del = 1; }
            int f_del = 0;
            for (int j = threadIdx.x; j < M0; j += T) {
                const double si = s.s_in[j], qi = s.beta_s * s.q_in[j];
                const double aj = s.alpha[j];
                const double den = aj - si;
                const double qo = aj * qi / den, so = aj * si / den, q2 = qo * qo;
                double d_ml = 0; int act = ACT_NONE;
                double r, L;
                if (add_root(so, q2, l1, l2, r, L)) {
                    if (L > 0) {
                        s.aroot_in[j] = r + l2;
                        act = ACT_REEST;
                        d_ml = reest_gain(so, q2, l1, l2, r, aj);
                    }
                } else if (M0 > 1) {
                    f_del = 1;
                    act = ACT_DEL;
                    d_ml = delete_gain(so, q2, l1, l2, aj);
                }
                s.dml_in[j] = d_ml; s.act_in[j] = act;
            }
            const int any_del = __syncthreads_or(f_del);
            const int any_add = (!EPIS) ? s.any_add : 0;               // only the Gaussian main-effect file ever sets anyToAdd (:1484)
            int n_list = s.n_list;
            if (n_list > sh.list_cap) { n_list = sh.list_cap; s.status |= ST_LIST; }
            bool zero_reest = false, zero_del = false, zero_add = false;
            if ((any_add && prio_add) || (any_del && prio_del)) {        // :1527-1556
                zero_reest = true;
                if (any_add && prio_add && !prio_del) zero_del = true;
                if (any_del && prio_del && !prio_add) zero_add = true;
            }
            if (!EPIS && ((!any_add && s.iter == 1 && s.i_iter < 10) || (!any_add && s.residvar >= s.var_y * 0.95))) zero_del = true;   // :1557-1577
            __syncthreads();
            for (int j = threadIdx.x; j < M0; j += T) {
                const int act = s.act_in[j];
                if ((act == ACT_REEST && zero_reest) || (act == ACT_DEL && zero_del)) s.dml_in[j] = 0;
            }
            __syncthreads();
            // best over both sets; only its value and its action matter downstream (ties: in-model first, as the
            // reference's first scan visits Used before Unused; the rescans run in ascending id and can only differ
            // from this on an exact tie between an add and an in-model action)
            double lbest = 0; int lkey = 0x7fffffff, larg = 0;
            for (int j = threadIdx.x; j < M0; j += T) {
                const double d = s.dml_in[j];
                if (d > lbest || (d == lbest && d > 0 && j < lkey)) { lbest = d; lkey = j; larg = s.act_in[j]; }
            }
            if (!zero_add)
                for (int i = threadIdx.x; i < n_list; i += T) {
                    const double d = s.list_dml[i];
                    const int key = M0 + 1;                                // after every in-model candidate
                    if (d > lbest || (d == lbest && d > 0 && key < lkey)) { lbest = d; lkey = key; larg = ACT_ADD; }
                }
            double best; int best_act;
            block_argmax(lbest, lkey, larg, sc, best, best_act);
            int nu_none = !(best > 0);                                     // the reference's nu stays at its initial value
            int worthwhile;
            int n_update = 0;
            if (s.selected == ACT_TERM && !s.ini_removed && s.M > 1) nu_none = 2;           // nu = -1, :426-430
            if (nu_none == 2 && s.ini_removed) { worthwhile = 0; s.selected = ACT_TERM; }
            else if (nu_none == 2 && !s.ini_removed && s.M > 1) {                          // :437-446
                worthwhile = 1;
                __syncthreads();
                if (threadIdx.x == 0) { s.blk_c[0] = s.initial - 1; s.blk_src[0] = -1; }    // forced delete of the initial basis
                __syncthreads();
                n_update = 1; s.ini_removed = 1; s.selected = ACT_DEL;
            } else {
                worthwhile = 1;
                // nothing positive: the reference reads action[nu = 0]; whatever it finds, the cutoff is ml_delta and the block empty
                const int best_is_add = best > 0 && best_act == ACT_ADD;
                const int best_is_del = best > 0 && best_act == ACT_DEL;
                double cutoff = best * (best_is_add ? v.n_add : 1.0);
                if (cutoff < v.ml_delta) cutoff = v.ml_delta;
                // block = in-model entries and list entries with dml >= cutoff, ascending candidate id
                __syncthreads();
                if (threadIdx.x == 0) {
                    int n = 0;
                    for (int j = 0; j < M0; j++) if (s.dml_in[j] >= cutoff) { s.blk_c[n] = s.used[j] - 1; s.blk_src[n] = -1 - j; n++; }
                    if (!zero_add)
                        for (int i = 0; i < n_list; i++) if (s.list_dml[i] >= cutoff) { s.blk_c[n] = s.list_c[i]; s.blk_src[n] = i; n++; }
                    redi[64] = n;
                }
                __syncthreads();
                n_update = redi[64];
                // rank sort by candidate id (ids are distinct); the sorted block goes to the upper half of blk_*
                __syncthreads();
                for (int a = threadIdx.x; a < n_update; a += T) {
                    const int ca = s.blk_c[a];
                    int rank = 0;
                    for (int b = 0; b < n_update; b++) rank += s.blk_c[b] < ca;
                    s.blk_c[n_update + rank] = ca; s.blk_src[n_update + rank] = s.blk_src[a];
                }
                __syncthreads();
                for (int a = threadIdx.x; a < n_update; a += T) { s.blk_c[a] = s.blk_c[n_update + a]; s.blk_src[a] = s.blk_src[n_update + a]; }
                __syncthreads();
                if (best_is_del && n_update > 1) n_update = 1;                             // :474
                if (n_update == 0) worthwhile = 0;
            }
            if (!worthwhile) s.selected = ACT_TERM;
            if (worthwhile) {
                for (int iu = 0; iu < n_update; iu++) {
                    __syncthreads();
                    const int nu = s.blk_c[iu];
                    const int src = s.blk_src[iu];
                    double new_alpha = 0;
                    if (src >= 0) { s.selected = ACT_ADD; new_alpha = s.list_aroot[src]; }
                    else if (src == -1 && s.selected == ACT_DEL && n_update == 1 && s.blk_c[0] == s.initial - 1 && nu_none == 2) { /* forced delete */ }
                    else { s.selected = s.act_in[-1 - src]; new_alpha = s.aroot_in[-1 - src]; }
                    if (s.selected == ACT_REEST || s.selected == ACT_DEL) {
                        // position of nu in Used NOW (earlier actions of this block may have moved it); a failed search
                        // keeps the previous jj like the reference (:498-509), but never indexes outside the active set
                        int found = -1;
                        for (int j = threadIdx.x; j < s.M; j += T) if (s.used[j] - 1 == nu) found = j;
                        __syncthreads();
                        if (threadIdx.x == 0) redi[65] = -1;
                        __syncthreads();
                        if (found >= 0) redi[65] = found;
                        __syncthreads();
                        if (redi[65] >= 0) s.jj = redi[65];
                        if (s.jj < 0 || s.jj >= s.M) { s.status |= ST_NOT_PD; s.selected = ACT_TERM; }
                    }
                    const int jj = s.jj;
                    if (s.selected == ACT_REEST && fabs(log(new_alpha) - log(s.alpha[jj])) <= v.reest_tol && !any_del)
                        s.selected = ACT_TERM;                                             // :541-549
                    const int M = s.M;
                    bool updated = false;
                    if (s.selected == ACT_REEST) {                                         // :553-596
                        const double old = s.alpha[jj];
                        const double kappa = 1.0 / (s.sigma[jj * M + jj] + 1.0 / (new_alpha - old));
                        const double mujj = s.mu[jj];
                        const double *sj = s.sigma + jj * M;
                        __syncthreads();
                        if (threadIdx.x == 0) s.alpha[jj] = new_alpha;
                        sigma_reest(s.sigma, s.sigma_new, M, jj, kappa);
                        mu_reest(s.mu, M, sj, mujj, kappa);
                        updated = true;
                    } else if (s.selected == ACT_ADD) {                                    // ActionAdd*, :1585-1723
                        if (M + 1 > cap) { s.status |= ST_CAP; s.selected = ACT_TERM; }
                        else {
                            const double sc_nu = stream_column<EPIS>(F, K, nu, s.phinew, sc);
                            {
                                Cand<EPIS> cd(nu, K);
                                const double isc = 1 / sc_nu;
                                const bool pair = cd.i != cd.j;     // pairs are divided, main effects scaled by 1/s (NeFull2.c:277-290)
                                __syncthreads();
                                // raw x' phi_new / s (the cache entry G[new][nu] of the reference) before the column is normalised
                                double pp = 0;
                                for (int h = threadIdx.x; h < N; h += T) {
                                    const double x = s.phinew[h];
                                    const double ph = pair ? x / sc_nu : x * isc;
                                    pp = fma(x, ph, pp);
                                    s.phinew[h] = ph;
                                }
                                pp = block_sum(pp, sc);
                                if (threadIdx.x == 0) s.ptp[(size_t)M * cap + M] = pp / sc_nu;
                            }
                            __syncthreads();
                            // g = PHI' phi_new; current S and Q of nu
                            phi_t_vec(s.phi, N, LD, M, s.phinew, s.u);                     // u <- g for now
                            (void)stream_residual(s, N, LD, M, s.d, s.e, sc);
                            double qn = 0;
                            for (int h = threadIdx.x; h < N; h += T) qn = fma(s.phinew[h], s.e[h], qn);
                            qn = block_sum(qn, sc);
                            double quad = 0;
                            for (int i = threadIdx.x; i < M; i += T) {
                                double z = 0;
                                for (int k = 0; k < M; k++) z = fma(s.sigma[(size_t)k * M + i], s.u[k], z);
                                quad = fma(z, s.u[i], quad);
                            }
                            quad = block_sum(quad, sc);
                            const double S_nu = s.beta_s - s.beta_s * quad * s.beta_s;
                            const double Q_nu = s.beta_s * qn;
                            for (int j = threadIdx.x; j < M; j += T) {
                                const double pj = s.u[j];                                   // phi_j' phi_new
                                s.tmp[j] = s.beta * pj;
                                s.ptp[(size_t)j * cap + M] = pj; s.ptp[(size_t)M * cap + j] = pj;
                            }
                            __syncthreads();
                            for (int i = threadIdx.x; i < M; i += T) {
                                double z = 0;
                                for (int j = 0; j < M; j++) z = fma(s.sigma[i * M + j], s.tmp[j], z);
                                s.colk[i] = z;
                            }
                            __syncthreads();
                            for (int i = threadIdx.x; i < M; i += T) s.u[i] = s.colk[i];
                            for (int h = threadIdx.x; h < LD; h += T) s.phi[(size_t)M * LD + h] = h < N ? s.phinew[h] : 0.0;
                            const double s_ii = 1.0 / (new_alpha + S_nu);
                            const double mu_i = s_ii * Q_nu;
                            __syncthreads();
                            if (threadIdx.x == 0) { s.alpha[M] = new_alpha; s.ascale[M] = sc_nu; }
                            mu_add(s.mu, M, s.u, mu_i);
                            sigma_add(s.sigma, s.sigma_new, M, s.u, s_ii);
                            __syncthreads();
                            if (threadIdx.x == 0) s.used[M] = nu + 1;
                            s.M = M + 1;
                            updated = true;
                        }
                    } else if (s.selected == ACT_DEL) {                                    // ActionDel*, :1725-1822
                        const int lastj = M - 1;
                        const int mujj = (int)s.mu[jj];                                    // `int Mujj` truncation (:1746-1747)
                        const double *sj = s.sigma + jj * M;
                        const double sjj = sj[jj];
                        const double al_last = s.alpha[lastj], sc_last = s.ascale[lastj];
                        __syncthreads();
                        mu_delete(s.mu, M, sj, sjj, mujj);
                        __syncthreads();
                        // the remainder of the deleted weight stays in the reference's Q array: carry it in d
                        const double mu_drop = s.mu[jj];
                        for (int h = threadIdx.x; h < N; h += T) {
                            s.d[h] = fma(mu_drop, s.phi[(size_t)jj * LD + h], s.d[h]);
                            s.phi[(size_t)jj * LD + h] = s.phi[(size_t)lastj * LD + h];
                        }
                        ptp_move_last(s.ptp, cap, jj, lastj);
                        sigma_delete<true>(s.sigma, s.sigma_new, M, jj, s.colk);
                        __syncthreads();
                        // the basis that leaves is the one in slot jj: not candidate nu when the forced removal's search of Used
                        // failed (gauss_fit.cuh, delete action) -- it is then in neither list until the next outer iteration
                        const int dropped = s.used[jj] - 1;
                        __syncthreads();
                        if (dropped != nu && s.n_hidden < 4) { s.hidden[s.n_hidden] = dropped; s.n_hidden++; }
                        if (threadIdx.x == 0) {
                            s.alpha[jj] = al_last; s.ascale[jj] = sc_last;
                            s.mu[jj] = s.mu[lastj];
                            s.used[jj] = s.used[lastj];
                        }
                        s.M = M - 1;
                        updated = true;
                    }
                    __syncthreads();
                    if (updated) {                                                         // :657-681
                        s.stats_valid = 0;
                        double *tmpp = s.sigma; s.sigma = s.sigma_new; s.sigma_new = tmpp;
                        const int Mn = s.M;
                        for (int i = threadIdx.x; i < Mn; i += T) s.gamma[i] = 1 - s.alpha[i] * s.sigma[i * Mn + i];
                        __syncthreads();
                    }
                }
            }
            s.n_update = n_update;
            if (s.selected == ACT_TERM || s.i_iter <= 10 || s.i_iter % 5 == 0 || n_update >= 2) {      // :685-729
                const int M = s.M;
                const double ee = stream_residual(s, N, LD, M, nullptr, s.e, sc);
                double sg = 0;
                for (int i = 0; i < M; i++) sg += s.gamma[i];
                const double beta_old = s.beta;
                s.beta = (N - sg) / ee;
                const double vt = block_var(s.t, N, sc);
                if (s.beta > 1e6 / vt) s.beta = 1e6 / vt;
                if (fabs(log(s.beta) - log(beta_old)) > 1e-6) {
                    // FinalUpdate* (:1841-1921): H = beta PHI'PHI + diag(alpha), SIGMA = H^-1, Mu
                    for (int j = wid_; j < M; j += nw_)
                        for (int i = lane_; i < M; i += 32) {
                            double val = s.ptp[(size_t)j * cap + i] * s.beta;
                            if (i == j) val += s.alpha[i];
                            s.H[j * M + i] = val; s.sigma[j * M + i] = val;
                        }
                    __syncthreads();
                    if (!spd_inverse_sweep(s.sigma, M, s.colk, sc, sc.sweep)) s.status |= ST_NOT_PD;
                    stream_posterior_mean(s, N, LD, M, s.beta);
                    // the FullStat that follows (unless terminating) re-bases the statistic arrays on the new beta; the
                    // terminating case leaves the reference's arrays as they were
                    if (s.selected != ACT_TERM) {
                        s.beta_s = s.beta;
                        s.stats_valid = 0;
                        for (int h = threadIdx.x; h < N; h += T) s.d[h] = 0;
                        for (int i = 1 + threadIdx.x; i < M; i += T) s.gamma[i] = 1.0 - s.sigma[i * M + i] * s.alpha[i];
                    }
                    __syncthreads();
                }
            }
            if (s.selected == ACT_TERM && s.ini_removed) last = 1;
            if ((s.i_iter == s.it_max && s.M == 1) || s.i_iter > s.it_max) last = 1;
            if (s.i_iter == s.it_max) s.selected = ACT_TERM;
            if (last) break;
        }
        last = 0;
        // ---------------- intercept update: b = 1'C^-1 y / (1'C^-1 1 [+1e-10]) ----------------
        {
            const int M = s.M;
            for (int j = wid_; j < M; j += nw_) {
                const double *p = s.phi + (size_t)j * LD;
                double a1 = 0, ay = 0;
                for (int h = lane_; h < N; h += 32) { a1 += p[h]; ay = fma(p[h], y[h], ay); }
                a1 = warp_sum(a1); ay = warp_sum(ay);
                if (lane_ == 0) { s.tmp[j] = a1; s.u[j] = ay; }
            }
            __syncthreads();
            double q11 = 0, q1y = 0, sy = 0;
            for (int j = threadIdx.x; j < M; j += T) {
                double z = 0;
                for (int k = 0; k < M; k++) z = fma(s.sigma[j * M + k], s.tmp[k], z);
                q11 = fma(z, s.tmp[j], q11); q1y = fma(z, s.u[j], q1y);
            }
            block_sum2(q11, q1y, sc);
            for (int h = threadIdx.x; h < N; h += T) sy += y[h];
            sy = block_sum(sy, sc);
            const double cinv = s.beta * N - s.beta * s.beta * q11;
            const double cinvy = s.beta * sy - s.beta * s.beta * q1y;
            s.b = EPIS ? cinvy / cinv : cinvy / (cinv + 1e-10);                            // MainEff.c:188 vs NeFull2.c:202
            s.vk = 0;
            for (int i = 0; i < M; i++) s.vk += s.alpha[i];
            s.err = fabs(s.vk - s.vk0) / M;
            s.residvar = 1 / (s.beta + 1e-10);
        }
    }
    if (s.iter >= 100) s.status |= ST_ITER_MAX;

    // ---------------- hold-out score (R/GetModelError.R:6-32) ----------------
    const int M = s.M;
    auto norm = [&](int i) { return s.ascale[i]; };
    int nsel;
    const double sse = gauss_holdout_sse<EPIS>(F, K, M, s.mu, s.used, s.b, s.tmp, norm, nsel, s.status, sc);
    if (threadIdx.x == 0) {
        const int o = s.out_index;
        write_fit_outputs(out, o, sse, s.status, nsel, s.iter, s.flops, 0, 0);
        if (out.m_out) write_record(out, o, M, 0, s.mu, s.H, s.sigma, s.used, norm, s.b, 0, 1 / (s.beta + 1e-10));
        s.phase = SP_DONE;
        G = s;
    }
}

}  // namespace pareben
