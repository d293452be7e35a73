// stream_scan.cuh -- the streaming-mode score contraction: for every fold, Z = X_fold' * E on the FP64 tensor
// cores, screened and reduced in the epilogue (see stream.cuh).  Replaces, for Kc too large to cache,
// CacheBP + FullStat + the scan over Unused of fEBDeltaML (NeFull2.c:998-1055, 1063-1196, 1227-1404).
//
// Work item = (rhs tile of 64 fits of one fold, tile of 128 consecutive candidates); items are dealt to a
// persistent grid in a fixed stride, so consecutive blocks work on consecutive candidate tiles of the same E tile
// (E tile and X rows are L2 hits).  Inside a block:
//   * E travels by the TMA unit: per stage ONE cp.async.bulk of 34,816 bytes -- a [64 fits][68] column-major slab of E
//     that the advance kernel wrote in exactly this shape -- into a 4-deep shared-memory ring, completion on the
//     stage's `full` mbarrier, re-use gated by its `empty` mbarrier (8 warp arrivals).  Lane 0 of warp 0 issues the
//     copy of stage g + 3 just before the block consumes stage g (a ninth, dedicated producer warp would put three
//     warps on one scheduler and cap every warp at 168 registers: measured, the main loop then spills);
//   * all 8 warps are consumers, 16 candidates x 64 fits each = 2 x 8 DMMA tiles (64 accumulator registers); 8-column
//     tiles past the last waiting fit are skipped.  The A
//     operand never touches shared memory: a lane reads one 32-bit word per locus per 16 rows from the transposed,
//     row-permuted int8 matrix (position 4a+b holds row 4b+a, so the word IS the lane's element of four k-steps),
//     forms the pair product in integer registers, converts once and feeds 8 DMMAs with it; words are requested a
//     whole stage (4 groups) ahead.  The column's squared norm rides along (x^2 summed per lane, exact for genotype
//     codes), so no Kc-length scale array exists either.
//   * no block-wide barrier anywhere in the main loop: the ring and the item sequence run on across items.
// Epilogue (per warp, on its own): two exact screens (ScanSlot, stream.cuh); a survivor is processed by the whole warp:
// g = PHI_fit' phi_c, S = beta_s - beta_s^2 g'SIGMA g, Q = beta_s z / ||x_c||, the closed-form root / delta-ML, and
// an append to the fit's ADD list when it is within n_add of the fit's running maximum (a superset of the final block;
// the advance kernel filters with the exact cutoff and sorts, so the result does not depend on the schedule).
#pragma once
#include "stream.cuh"
#include "contract.cuh"
#include "eben_step.cuh"

namespace pareben {

// physical position of row h inside the transposed matrices (rows of every group of 16 permuted, see transpose_pad_kernel)
__device__ inline int perm_row(int h) { return (h & ~15) | ((h & 3) << 2) | ((h >> 2) & 3); }

// raw (unscaled) value of candidate (i, j) at training row h, from the transposed matrices
__device__ inline double xt_value(const FoldData &F, int i, int j, int h)
{
    const int rp = perm_row(h);
    if (F.XT8) {
        const int a = F.XT8[(size_t)i * F.ldt + rp];
        return (double)(i == j ? a : a * (int)F.XT8[(size_t)j * F.ldt + rp]);
    }
    const double a = F.XTd[(size_t)i * F.ldt + rp];
    return i == j ? a : a * F.XTd[(size_t)j * F.ldt + rp];
}

// fEBDeltaML for ONE out-of-model candidate with exact statistics (so, qo) (NeFull2.c:1290-1345 / MainEff.c:1417-1497),
// executed by one lane: the ADD's delta-ML goes to the fit's list when it is within n_add of the running maximum.
// Returns the delta-ML when it became the fit's new best (the caller then tightens its screen), else 0.
template <bool GAUSS_MAIN>
__device__ inline double scan_decide(StreamFit *fit, int c, double so, double qo, int list_cap)
{
    const double l1 = fit->l1, l2 = fit->l2;
    for (int h = 0; h < fit->n_hidden; h++) if (fit->hidden[h] == c) return 0.0;       // in neither Used nor Unused
    double r = 0, L = 0;
    if (!add_root(so, qo * qo, l1, l2, r, L)) return 0.0;
    if (!(L > 0)) return 0.0;
    if (GAUSS_MAIN) fit->any_add = 1;
    if (!(L >= fit->ml_delta)) return 0.0;
    const unsigned long long bits = (unsigned long long)__double_as_longlong(L);      // L > 0: the bit pattern is monotone
    const unsigned long long old = atomicMax(&fit->runmax, bits);
    const double cur = __longlong_as_double((long long)(old > bits ? old : bits));
    if (L >= cur * fit->n_add) {
        const int p = atomicAdd(&fit->n_list, 1);
        if (p < list_cap) { fit->list_c[p] = c; fit->list_dml[p] = L; fit->list_aroot[p] = r + l2; }
    }
    return bits > old ? L : 0.0;
}

// One survivor, processed by a whole warp: exact S, Q, the closed-form delta-ML, list append.
template <bool EPIS, bool GAUSS_MAIN>
__device__ inline void scan_survivor(const FoldData &F, int K, int c, double z_raw, double ssq, StreamFit *fit, ScanSlot *sp,
                                     int list_cap, double *g /* per-warp scratch, cap doubles */)
{
    const int lane = threadIdx.x & 31;
    const int M = fit->M, N = F.ntr, LD = phi_ld(N);
    int inmodel = 0;
    for (int j = lane; j < M; j += 32) inmodel |= (fit->used[j] - 1 == c);
    if (__any_sync(0xffffffffu, inmodel)) return;
    Cand<EPIS> cd(c, K);
    const double scale = ssq == 0.0 ? 1.0 : sqrt(ssq);
    const double *phi = fit->phi;
    for (int j0 = 0; j0 < M; j0 += 4) {
        double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
        const double *p0 = phi + (size_t)j0 * LD;
        const double *p1 = phi + (size_t)min(j0 + 1, M - 1) * LD, *p2 = phi + (size_t)min(j0 + 2, M - 1) * LD, *p3 = phi + (size_t)min(j0 + 3, M - 1) * LD;
#pragma unroll 4
        for (int h = lane; h < N; h += 32) {
            const double x = xt_value(F, cd.i, cd.j, h);
            a0 = fma(x, p0[h], a0); a1 = fma(x, p1[h], a1); a2 = fma(x, p2[h], a2); a3 = fma(x, p3[h], a3);
        }
        a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2); a3 = warp_sum(a3);
        if (lane == 0) {
            g[j0] = a0 / scale;
            if (j0 + 1 < M) g[j0 + 1] = a1 / scale;
            if (j0 + 2 < M) g[j0 + 2] = a2 / scale;
            if (j0 + 3 < M) g[j0 + 3] = a3 / scale;
        }
    }
    __syncwarp();
    const double *sigma = fit->sigma;
    double quad = 0;
    for (int i = lane; i < M; i += 32) {
        double z = 0;
        for (int j = 0; j < M; j++) z = fma(sigma[(size_t)j * M + i], g[j], z);
        quad = fma(z, g[i], quad);
    }
    quad = warp_sum(quad);
    __syncwarp();
    const double bs = fit->beta_s;
    const double so = bs - bs * quad * bs;
    const double qo = bs * (z_raw / scale);
    if (lane == 0) {
        const double L = scan_decide<GAUSS_MAIN>(fit, c, so, qo, list_cap);
        if (!GAUSS_MAIN && L > 0) {
            // a new best: no candidate whose delta-ML bound stays below n_add * best can enter the block any more
            const double need = L * fit->n_add * (1 - 1e-9);
            if (need > fit->ml_delta) slot_thresholds(sp, need, 0.0, true);
        }
    }
}

// Cheap form of the per-element test of class A: u (= beta_s g'SIGMA g, here from un-normalised products and a
// reciprocal, inflated by 1e-6 so that it can only over-estimate) picks the bucket, one comparison decides.
__device__ inline bool bucket_pass(const ScanSlot *sp, double z2, double ssq, double u)
{
    u *= 1 + 1e-6;
    int kb = 7;
    if (u >= 0.0078125) { kb = -ilogb(u) - 1; kb = kb < 0 ? 0 : (kb > 7 ? 7 : kb); }
    return z2 > sp->T[kb] * ssq;
}

// Class A: the contraction has delivered g_raw = x_c' phi_0 for the fit's one active column, so the candidate's
// statistics are exact here (FullStat's formulas, NeFull2.c:1150-1185: bp = G'SIGMA, quad = bp'G, with SIGMA = sp->sig), one lane.
template <bool GAUSS_MAIN>
__device__ inline void scan_exact_a(StreamFit *fit, ScanSlot *sp, int c, double z, double ssq, double g_raw, int list_cap)
{
    const double scale = sqrt(ssq), bs = sp->bs;
    const double g = g_raw / scale;
    const double quad = fma(fma(g, sp->sig, 0.0), g, 0.0);
    const double u = bs * quad;
    int kb = 7;
    if (u >= 0.0078125) { kb = -ilogb(u) - 1; kb = kb < 0 ? 0 : (kb > 7 ? 7 : kb); }
    if (!(z * z > sp->T[kb] * ssq)) return;                     // S >= beta_s (1 - 2^-kb): its delta-ML cannot reach the cutoff
    if (fit->used[0] - 1 == c) return;
    const double so = bs - bs * quad * bs, qo = bs * (z / scale);
    const double L = scan_decide<GAUSS_MAIN>(fit, c, so, qo, list_cap);
    if (!GAUSS_MAIN && L > 0) {
        const double need = L * fit->n_add * (1 - 1e-9);
        if (need > fit->ml_delta) slot_thresholds(sp, need, 0.0, true);
    }
}

template <bool EPIS, bool GAUSS_MAIN>
__global__ void __launch_bounds__(SCAN_THREADS, 1)
stream_scan_kernel(Problem P, StreamFit *fits, StreamShared sh)
{
    extern __shared__ __align__(128) double s_ring[];                 // SCAN_STAGES x STAGE_D doubles
    __shared__ unsigned long long s_full[SCAN_STAGES], s_empty[SCAN_STAGES];
    __shared__ int s_prefix[STREAM_CLASSES * STREAM_MAX_FOLDS + 2];   // rhs tiles before (fold, class)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int K = P.K, Kc = P.Kc, nf1 = STREAM_CLASSES * (P.n_folds + 1);
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int f = 0; f < nf1; f++) { s_prefix[f] = tot; const int per = class_fits_per_tile(f % STREAM_CLASSES); tot += (sh.n_slots[f] + per - 1) / per; }
        s_prefix[nf1] = tot;
        for (int s = 0; s < SCAN_STAGES; s++) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], SCAN_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int n_rt_total = s_prefix[nf1];
    const long long n_ct = ((long long)Kc + SCAN_CT - 1) / SCAN_CT;
    const long long n_items = n_ct * n_rt_total;
    auto locate = [&](long long item, int &f, int &rt, long long &ct) {
        const int prt = (int)(item / n_ct);
        ct = item - (long long)prt * n_ct;
        f = 0;
        while (s_prefix[f + 1] <= prt) f++;
        rt = prt - s_prefix[f];
    };

    // ---------------- producer cursor (used by lane 0 of warp 0 only) ----------------
    long long p_item = blockIdx.x;
    int p_st = 0, p_nstage = 0;
    const double *p_src = nullptr;
    unsigned p_stage = 0, p_par = 1;                                  // a fresh `empty` barrier passes a wait on parity 1
    auto produce_one = [&]() {
        if (p_item >= n_items) return;
        if (p_st == 0) {
            int f, rt; long long ct;
            locate(p_item, f, rt, ct);
            const int ldt = P.folds[f / STREAM_CLASSES].ldt;
            p_nstage = ldt / SK;
            p_src = sh.folds[f].E + (size_t)rt * e_tile_doubles(ldt);
        }
        mbar_wait(&s_empty[p_stage], p_par);
        mbar_expect_tx(&s_full[p_stage], STAGE_D * 8);
        bulk_load(s_ring + (size_t)p_stage * STAGE_D, p_src + (size_t)p_st * STAGE_D, STAGE_D * 8, &s_full[p_stage]);
        if (++p_stage == SCAN_STAGES) { p_stage = 0; p_par ^= 1; }
        if (++p_st == p_nstage) { p_st = 0; p_item += gridDim.x; }
    };
    const bool producer = threadIdx.x == 0;
    if (producer)
        for (int d = 0; d < SCAN_STAGES - 1; d++) produce_one();

    // ---------------- consumers ----------------
    const int gm = lane >> 2, gk = lane & 3;
    unsigned stage = 0, par = 0;
    double *scratch = sh.warp_scratch + ((size_t)blockIdx.x * SCAN_WARPS + wid) * P.cap;
    for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
        int f, rt; long long ct;
        locate(item, f, rt, ct);                                        // f = STREAM_CLASSES * fold + class
        const FoldData F = P.folds[f / STREAM_CLASSES];
        const int cls = f % STREAM_CLASSES;
        const int N = F.ntr, ldt = F.ldt, nstage = ldt / SK;
        const int8_t *__restrict__ X8 = F.XT8;
        const double *__restrict__ Xd = F.XTd;
        const long long cbase = ct * SCAN_CT + wid * 16;
        const int c0 = (int)min(cbase + gm, (long long)Kc - 1), c1 = (int)min(cbase + 8 + gm, (long long)Kc - 1);
        // loci of this lane's two candidates; the second is 8 ids further on, usually in the same row of the pair
        // enumeration (c = K + i (2K - i - 1) / 2 + (j - i - 1), NeFull2.c:115-134), so it is stepped instead of decoded
        Cand<EPIS> cd0(c0, K), cd1 = cd0;
        if (!EPIS || c1 < K || c0 < K) cd1 = Cand<EPIS>(c1, K);
        else if (c1 != c0) {
            int i1 = cd0.i, j1 = cd0.j + (c1 - c0);
            while (j1 > K - 1) { j1 -= K - 1 - i1; i1++; j1 += 1; }      // past the end of row i1: continue in row i1 + 1 at its first pair
            cd1.i = i1; cd1.j = j1;
        }
        double acc[2][8][2];
#pragma unroll
        for (int t = 0; t < 2; t++)
#pragma unroll
            for (int n = 0; n < 8; n++) { acc[t][n][0] = 0.0; acc[t][n][1] = 0.0; }
        double ssq0 = 0.0, ssq1 = 0.0;
        // raw words of the next four groups of 16 rows (slot = group index within its stage)
        int wn[4][2][2];
        double xv[2][4];
        const int8_t *pa0 = X8 + (size_t)cd0.i * ldt + 4 * gk, *pa1 = X8 + (size_t)cd1.i * ldt + 4 * gk;
        const int8_t *pj0 = X8 + (size_t)cd0.j * ldt + 4 * gk, *pj1 = X8 + (size_t)cd1.j * ldt + 4 * gk;
        auto fetch8 = [&](int slot, int grp) {
            const int h = min(16 * grp, ldt - 16);
            wn[slot][0][0] = *reinterpret_cast<const int *>(pa0 + h);
            wn[slot][1][0] = *reinterpret_cast<const int *>(pa1 + h);
            if (EPIS) {
                wn[slot][0][1] = *reinterpret_cast<const int *>(pj0 + h);
                wn[slot][1][1] = *reinterpret_cast<const int *>(pj1 + h);
            }
        };
        auto make_current = [&](int slot, int grp) {
            if (X8) {
#pragma unroll
                for (int ks = 0; ks < 4; ks++) {
                    xv[0][ks] = cd0.from_words(wn[slot][0][0], EPIS ? wn[slot][0][1] : 0, ks);
                    xv[1][ks] = cd1.from_words(wn[slot][1][0], EPIS ? wn[slot][1][1] : 0, ks);
                }
                fetch8(slot, grp + 4);
            } else {
                const int h = min(16 * grp, ldt - 16) + 4 * gk;
                const double2 *p0 = reinterpret_cast<const double2 *>(Xd + (size_t)cd0.i * ldt + h);
                const double2 *p1 = reinterpret_cast<const double2 *>(Xd + (size_t)cd1.i * ldt + h);
                const double2 a = p0[0], b = p0[1], c = p1[0], d = p1[1];
                xv[0][0] = a.x; xv[0][1] = a.y; xv[0][2] = b.x; xv[0][3] = b.y;
                xv[1][0] = c.x; xv[1][1] = c.y; xv[1][2] = d.x; xv[1][3] = d.y;
                if (EPIS) {
                    if (cd0.i != cd0.j) {
                        const double2 *q0 = reinterpret_cast<const double2 *>(Xd + (size_t)cd0.j * ldt + h);
                        const double2 e = q0[0], ff = q0[1];
                        xv[0][0] *= e.x; xv[0][1] *= e.y; xv[0][2] *= ff.x; xv[0][3] *= ff.y;
                    }
                    if (cd1.i != cd1.j) {
                        const double2 *q1 = reinterpret_cast<const double2 *>(Xd + (size_t)cd1.j * ldt + h);
                        const double2 e = q1[0], ff = q1[1];
                        xv[1][0] *= e.x; xv[1][1] *= e.y; xv[1][2] *= ff.x; xv[1][3] *= ff.y;
                    }
                }
            }
        };
        if (X8) {
#pragma unroll
            for (int d = 0; d < 4; d++) fetch8(d, d);
        }
        const int n_wait = sh.n_slots[f];
        const int fits_here = min(class_fits_per_tile(cls), n_wait - rt * class_fits_per_tile(cls));
        const int cols_live = cls == 1 ? 1 + fits_here : fits_here;
        const int nt_live = (cols_live + 7) >> 3;                        // 8-column tiles that hold a waiting fit
        for (int st = 0; st < nstage; st++) {
            if (producer) produce_one();                                // stage g + 3 (its slot was released by everyone at g - 1)
            __syncwarp();
            mbar_wait(&s_full[stage], par);
            const double *buf = s_ring + (size_t)stage * STAGE_D;
#pragma unroll
            for (int g = 0; g < 4; g++) {
                if (st * SK + 16 * g < N) {                            // uniform: whole groups past the last row are skipped
                    make_current(g, st * 4 + g);
#pragma unroll
                    for (int ks = 0; ks < 4; ks++) { ssq0 = fma(xv[0][ks], xv[0][ks], ssq0); ssq1 = fma(xv[1][ks], xv[1][ks], ssq1); }
                    const double *bcol = buf + gm * SLD + 16 * g + gk;
#pragma unroll
                    for (int ks = 0; ks < 4; ks++) {
                        double bf[8];
#pragma unroll
                        for (int n = 0; n < 8; n++) if (n < nt_live) bf[n] = bcol[8 * n * SLD + 4 * ks];
#pragma unroll
                        for (int n = 0; n < 8; n++)
                            if (n < nt_live) {
                                dmma(acc[0][n][0], acc[0][n][1], xv[0][ks], bf[n]);
                                dmma(acc[1][n][0], acc[1][n][1], xv[1][ks], bf[n]);
                            }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&s_empty[stage]);
            if (++stage == SCAN_STAGES) { stage = 0; par ^= 1; }
        }
        // ---------------- epilogue: screen, then the survivors one at a time with the whole warp ----------------
        ssq0 += __shfl_xor_sync(0xffffffffu, ssq0, 1); ssq0 += __shfl_xor_sync(0xffffffffu, ssq0, 2);
        ssq1 += __shfl_xor_sync(0xffffffffu, ssq1, 1); ssq1 += __shfl_xor_sync(0xffffffffu, ssq1, 2);
        const StreamFold SF = sh.folds[f];
        if (cls == 1) {
            // column 0 of the tile is phi_0: g = x_c' phi_0 sits in n-tile 0 of the lane with gk == 0
            const double g0 = __shfl_sync(0xffffffffu, acc[0][0][0], lane & ~3), g1 = __shfl_sync(0xffffffffu, acc[1][0][0], lane & ~3);
#pragma unroll
            for (int t = 0; t < 2; t++) {
                const long long cl = cbase + 8 * t + gm;
                const double ssq = t == 0 ? ssq0 : ssq1;
                const double graw = t == 0 ? g0 : g1;
                const double rho2 = ssq > 0 ? graw * graw * (1.0 / ssq) : 0.0;
#pragma unroll
                for (int n = 0; n < 8; n++)
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const int col = 8 * n + 2 * gk + i;
                        if (cl < Kc && col >= 1 && col < cols_live) {
                            ScanSlot *sp = SF.par + rt * SN + col;
                            const double z = acc[t][n][i];
                            if (bucket_pass(sp, z * z, ssq, sp->bs * sp->sig * rho2))
                                scan_exact_a<GAUSS_MAIN>(fits + SF.slot_fit[rt * SN + col], sp, (int)cl, z, ssq, graw, sh.list_cap);
                        }
                    }
            }
            continue;
        }
#pragma unroll
        for (int t = 0; t < 2; t++) {
            const long long cl = cbase + 8 * t + gm;
            const double ssq = t == 0 ? ssq0 : ssq1;
#pragma unroll
            for (int n = 0; n < 8; n++)
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    const int slot = rt * SN + 8 * n + 2 * gk + i;
                    const double z = acc[t][n][i];
                    bool pass = false;
                    if (cl < Kc && slot < rt * SN + cols_live) pass = z * z > SF.par[slot].T[0] * ssq;     // strict: z = 0 can never be added
                    unsigned mask = __ballot_sync(0xffffffffu, pass);
                    while (mask) {
                        const int src = __ffs(mask) - 1;
                        mask &= mask - 1;
                        const int sc = __shfl_sync(0xffffffffu, (int)cl, src);
                        const int sslot = __shfl_sync(0xffffffffu, slot, src);
                        const double sz = __shfl_sync(0xffffffffu, z, src);
                        const double sq = __shfl_sync(0xffffffffu, ssq, src);
                        scan_survivor<EPIS, GAUSS_MAIN>(F, K, sc, sz, sq, fits + SF.slot_fit[sslot], SF.par + sslot, sh.list_cap, scratch);
                    }
                }
        }
    }
}

}  // namespace pareben
