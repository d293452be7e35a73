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
#include <cuda_pipeline.h>

namespace pareben {

struct GaussState {
    int M, n_unused, cap;
    double beta;
    int status;
    double flops;
    double avoided;          // the part of `flops` (SURVEY 8d model) that the Gram organisation did not execute
};

// ---- contraction: out(r, c) = sum_h x_c[h] * V_r[h]  for r in [0,R), c in [0,Kc) -------------
// The right-hand sides V_r are columns that already exist in memory (the active columns of PHI, the
// residual vector); nothing is materialised for a contraction.  Three code paths:
//
//  * contract_mma (R > SIMT_R_MAX): FP64 tensor-core path, mma.sync.m8n8k4.f64 (DMMA).  A warp owns
//    16 candidates (two 8-row A tiles) x up to 32 right-hand sides (four 8-column B tiles) and keeps the
//    16 x 32 accumulator block in registers.  A: one 32-bit word of the transposed int8 training matrix
//    per lane per 16 rows (or four doubles), two groups ahead in a register ring; B: 32-row tiles copied
//    by cp.async straight from the sources into a 3-stage shared-memory ring, conflict-free 8-byte
//    fragment loads; one barrier per stage.  A thread-per-candidate DFMA loop needs one 8-byte shared
//    operand per FMA and is capped at 25 % of the FP64 peak by the 128 B/clk shared-memory return path;
//    the DMMA form needs 1/8 of that traffic.
//  * contract_col (R == 1, the new column of an add): a warp per candidate, see below.
//  * contract_simt (2 <= R <= SIMT_R_MAX): one candidate per thread, RCS accumulators in registers.
//
// Every (r, c) is summed in an order that depends only on the row index, with identical arithmetic for
// every candidate, so exact duplicate columns tie exactly (SURVEY.md fact 8).
constexpr int KT = 32;            // rows per shared-memory stage of the contraction (two groups of 16; 64 is faster in isolation,
                                  // but its shared memory comes out of the L1 that the latency-bound phases live on)
constexpr int QT = 32;            // rows per stage of the row-major tiles (quadratic forms)
constexpr int NT_MAX = 4;         // 8-column B tiles per pass (32 right-hand sides): 16 x 32 accumulators = 32 registers, no spills
constexpr int MT = 2;             // 8-candidate A tiles per warp
constexpr int LDS_V = 68;         // leading dimension of a row-major staged tile (quadratic forms): == 4 (mod 16) doubles -> conflict-free B fragments
constexpr int SIMT_R_MAX = 4;
constexpr int RCS = 4;            // accumulators per thread in the SIMT path
constexpr int PF = 8;             // rows of X prefetched per group (SIMT path)
constexpr int FIT_T = 256;        // threads per block (the tile-production loops are unrolled for it)

// a / b given r = 1/b (correctly rounded): quotient estimate plus one FMA residual correction -- the tail of the
// division routine without its reciprocal iteration; used where one divisor serves many dividends.
__device__ inline double div_by(double a, double b, double r)
{
    const double q = a * r;
    return fma(fma(-q, b, a), r, q);
}

__device__ inline void dmma(double &d0, double &d1, double a, double b)
{
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// QT rows x ncol doubles (ncol a multiple of 2) of a row-major matrix V -> dst (leading dimension ldd), 16 bytes per
// cp.async (the SIGMA tiles of the DMMA quadratic forms).  PERM stores the rows of every group of 16 permuted
// (row 4a + b at position 4b + a); unused at present.
template <bool PERM>
__device__ inline void stage_tile(double *dst, int ldd, const double *__restrict__ V, int ldv, int h0, int r0, int ncol)
{
    const int ch = ncol >> 1;                  // 16-byte chunks per row
    for (int idx = threadIdx.x; idx < QT * ch; idx += blockDim.x) {
        const int h = idx / ch, q = idx - h * ch;
        const int hp = PERM ? ((h & ~15) | ((h & 3) << 2) | ((h >> 2) & 3)) : h;
        __pipeline_memcpy_async(dst + hp * ldd + 2 * q, V + (size_t)(h0 + h) * ldv + r0 + 2 * q, 16);
    }
    __pipeline_commit();
}

// One pass over the rows for NT 8-column tiles of right-hand sides starting at column r0, all candidates.
//   col(r)      base pointer of right-hand side r: N doubles, contiguous in the row index.  `n_aligned` of the
//               leading columns (the active columns of PHI: 16-byte aligned, pad rows zero) are copied with
//               16-byte cp.async, the rest (plain vectors) with 8-byte copies; rows >= N are zero-filled.
//   wv, ev      binomial only (else null): row weights w[h] and residuals e[h].  The A operand is then x*w and
//               two more sums per candidate ride along on the CUDA cores: bb = sum_h w x^2 and ze = sum_h x e.
//   dest(r, div)  destination row of right-hand side r (element c at dest[c]); div = divide by scale[c]
// Stages of KT rows are streamed through an NSTG-deep cp.async ring (no registers, the copies of two later
// stages are in flight while one is consumed; one barrier per stage).  Tiles are stored column-major with
// leading dimension LDS_C == 4 (mod 16) doubles, which makes the B-fragment loads bank-conflict free.
constexpr int NSTG = 3;
constexpr int LDS_C = KT + 4;
constexpr int STAGE_DOUBLES = 8 * NT_MAX * LDS_C + 2 * KT;       // tile + w + e
constexpr int SV_DOUBLES = NSTG * STAGE_DOUBLES;

template <int NT, bool EPIS, class Col, class Dest>
__device__ inline void mma_pass(const FoldData &F, int K, int Kc, int R, int r0, int n_aligned, Col col, Dest dest, double *sV,
                                const double *__restrict__ wv, const double *__restrict__ ev, double *bb_out, double *ze_out)
{
    const int N = F.ntr, ldt = F.ldt;
    const int8_t *__restrict__ X8 = F.XT8;
    const double *__restrict__ Xd = F.XTd;
    const int T = blockDim.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
    const int gm = lane >> 2, gk = lane & 3;                  // fragment coordinates of this lane
    const int nstage = (N + KT - 1) / KT, Np = nstage * KT;
    const int n_mtile = (Kc + 7) >> 3;
    const int per_round = nw * MT;
    const int nround = (n_mtile + per_round - 1) / per_round;
    const bool weighted = wv != nullptr;
    const int ncol = min(8 * NT, R - r0);                     // live columns of this pass (the rest of the tile is zeroed once)
    auto issue_stage = [&](int st) {
#ifdef MB_NO_STAGE
        if (false) {
#else
        if (st < nstage) {
#endif
            double *dst = sV + (st % NSTG) * STAGE_DOUBLES;
            const int h0 = st * KT;
            // aligned columns: KT/2 16-byte chunks each
            const int na = max(0, min(ncol, n_aligned - r0));
            for (int idx = threadIdx.x; idx < na * (KT / 2); idx += T) {
                const int c = idx / (KT / 2), q = idx - c * (KT / 2), h = h0 + 2 * q;
                const double *src = col(r0 + c);
                __pipeline_memcpy_async(dst + c * LDS_C + 2 * q, src + min(h, N - 1 & ~1), 16, h < N ? 0 : 16);
            }
            // plain vectors: 8-byte copies
            for (int idx = threadIdx.x; idx < (ncol - na) * KT; idx += T) {
                const int c = na + idx / KT, q = idx & (KT - 1), h = h0 + q;
                const double *src = col(r0 + c);
                __pipeline_memcpy_async(dst + c * LDS_C + q, src + min(h, N - 1), 8, h < N ? 0 : 8);
            }
            if (weighted) {
                double *wd = dst + 8 * NT_MAX * LDS_C;
                for (int idx = threadIdx.x; idx < 2 * KT; idx += T) {     // (w[h], e[h]) interleaved: one 16-byte load per row
                    const int q = idx >> 1, h = h0 + q;
                    __pipeline_memcpy_async(wd + idx, ((idx & 1) ? ev : wv) + min(h, N - 1), 8, h < N ? 0 : 8);
                }
            }
        }
        __pipeline_commit();
    };
    // columns past the last live one are read by the fragment loads of the final 8-column tile: zero them once
    for (int idx = threadIdx.x; idx < NSTG * (8 * NT - ncol) * KT; idx += T) {
        const int sgi = idx / ((8 * NT - ncol) * KT), rem = idx - sgi * ((8 * NT - ncol) * KT);
        sV[sgi * STAGE_DOUBLES + (ncol + rem / KT) * LDS_C + (rem & (KT - 1))] = 0.0;
    }
    for (int rd = 0; rd < nround; rd++) {
        // this warp's two tiles: mt0 and mt0 + nw, so that a short last round is spread over all warps
        const int mt0 = rd * per_round + wid;
        const bool live = mt0 < n_mtile;
        Cand<EPIS> cd0(min(mt0 * 8 + gm, Kc - 1), K), cd1(min((mt0 + nw) * 8 + gm, Kc - 1), K);
        double acc[MT][NT][2];
#pragma unroll
        for (int t = 0; t < MT; t++)
#pragma unroll
            for (int n = 0; n < NT; n++) { acc[t][n][0] = 0.0; acc[t][n][1] = 0.0; }
        double bb0 = 0.0, bb1 = 0.0, ze0 = 0.0, ze1 = 0.0;
        // A fragments of one group of 16 rows.  The transposed training matrix is stored with the rows of every
        // group permuted (physical position 4a + b holds row 4b + a), so the 32-bit word (or the four doubles) at
        // positions 4*gk .. 4*gk+3 holds rows gk, gk+4, gk+8, gk+12: exactly this lane's element of the four k-steps.
        // int8: the raw words of the next NG groups sit in a ring (slot = group index within its stage: static indices,
        // no register moves); a slot is converted to doubles when its group becomes current and refilled at once with the
        // group NG ahead, so every load has NG - 1 groups of DMMAs (> 1500 cycles) to land.  f64: loaded one group ahead.
        constexpr int NG = KT / 16;                            // groups per stage == ring slots
        double xv[MT][4];
        int wn[NG][MT][2];
        const int8_t *pa0 = X8 + (size_t)cd0.i * ldt + 4 * gk, *pa1 = X8 + (size_t)cd1.i * ldt + 4 * gk;
        const int8_t *pj0 = X8 + (size_t)cd0.j * ldt + 4 * gk, *pj1 = X8 + (size_t)cd1.j * ldt + 4 * gk;
        auto fetch8 = [&](int slot, int grp) {
            const int h = min(16 * grp, Np - 16);
            wn[slot][0][0] = *reinterpret_cast<const int *>(pa0 + h);
            wn[slot][1][0] = *reinterpret_cast<const int *>(pa1 + h);
            if (EPIS) {
                wn[slot][0][1] = *reinterpret_cast<const int *>(pj0 + h);
                wn[slot][1][1] = *reinterpret_cast<const int *>(pj1 + h);
            }
        };
        // make group `grp` current (xv), then start the loads of group grp + NG into the slot just freed
        auto advance = [&](int slot, int grp) {
#ifdef MB_NO_A
            if (true) { for (int ks = 0; ks < 4; ks++) { xv[0][ks] = 1.0 + gk; xv[1][ks] = 2.0 + gm; } return; }
#endif
            if (X8) {
#pragma unroll
                for (int ks = 0; ks < 4; ks++) {
                    xv[0][ks] = cd0.from_words(wn[slot][0][0], EPIS ? wn[slot][0][1] : 0, ks);
                    xv[1][ks] = cd1.from_words(wn[slot][1][0], EPIS ? wn[slot][1][1] : 0, ks);
                }
                fetch8(slot, grp + NG);
            } else {
                const int h = min(16 * grp, Np - 16) + 4 * gk;
                const double2 *p0 = reinterpret_cast<const double2 *>(Xd + (size_t)cd0.i * ldt + h);
                const double2 *p1 = reinterpret_cast<const double2 *>(Xd + (size_t)cd1.i * ldt + h);
                const double2 a = p0[0], b = p0[1], c = p1[0], d = p1[1];
                xv[0][0] = a.x; xv[0][1] = a.y; xv[0][2] = b.x; xv[0][3] = b.y;
                xv[1][0] = c.x; xv[1][1] = c.y; xv[1][2] = d.x; xv[1][3] = d.y;
                if (EPIS) {
                    if (cd0.i != cd0.j) {
                        const double2 *q0 = reinterpret_cast<const double2 *>(Xd + (size_t)cd0.j * ldt + h);
                        const double2 e = q0[0], f = q0[1];
                        xv[0][0] *= e.x; xv[0][1] *= e.y; xv[0][2] *= f.x; xv[0][3] *= f.y;
                    }
                    if (cd1.i != cd1.j) {
                        const double2 *q1 = reinterpret_cast<const double2 *>(Xd + (size_t)cd1.j * ldt + h);
                        const double2 e = q1[0], f = q1[1];
                        xv[1][0] *= e.x; xv[1][1] *= e.y; xv[1][2] *= f.x; xv[1][3] *= f.y;
                    }
                }
            }
        };
        if (rd == 0) {
            __syncthreads();                                   // the ring is free (previous pass / phase fully consumed)
#pragma unroll
            for (int d = 0; d < NSTG - 1; d++) issue_stage(d);
        }
        if (live) {
            if (X8) {
#pragma unroll
                for (int d = 0; d < NG; d++) fetch8(d, d);
            }
            advance(0, 0);
        }
        for (int st = 0; st < nstage; st++) {
            __pipeline_wait_prior(NSTG - 2);                   // stage st has landed (for this thread's copies)
#ifndef MB_NO_BARRIER
            __syncthreads();                                   // ... and for everyone's; stage st-1 is fully consumed
#endif
            issue_stage(st + NSTG - 1);
            const double *buf = sV + (st % NSTG) * STAGE_DOUBLES;
            const double *wrow = buf + 8 * NT_MAX * LDS_C;
            if (live) {
#pragma unroll
                for (int g = 0; g < NG; g++) {
                    if (st * KT + 16 * g >= N) break;          // block-uniform: whole groups past the last row are skipped
                    // group prologue: everything the CUDA cores have to do for these 16 rows (row weights into the A
                    // operand, the two ride-along sums), so that the 8*NT DMMAs below issue back to back
                    double aw0[4], aw1[4];
#pragma unroll
                    for (int ks = 0; ks < 4; ks++) {
                        const int hl = 16 * g + 4 * ks + gk;
                        double a0 = xv[0][ks], a1 = xv[1][ks];
                        if (weighted) {
                            const double2 we = *reinterpret_cast<const double2 *>(wrow + 2 * hl);
                            const double w = we.x, e = we.y;
                            ze0 = fma(a0, e, ze0); ze1 = fma(a1, e, ze1);
                            const double x0 = a0, x1 = a1;
                            a0 *= w; a1 *= w;
                            bb0 = fma(a0, x0, bb0); bb1 = fma(a1, x1, bb1);          // (x w) x: one multiply fewer than (x x) w, identical for genotype codes
                        }
                        aw0[ks] = a0; aw1[ks] = a1;
                    }
                    const double *bcol = buf + gm * LDS_C + 16 * g + gk;
                    double bc[NT], bn[NT];
#pragma unroll
                    for (int n = 0; n < NT; n++) bc[n] = bcol[8 * n * LDS_C];
#pragma unroll
                    for (int ks = 0; ks < 4; ks++) {
                        if (ks < 3) {
#pragma unroll
                            for (int n = 0; n < NT; n++) bn[n] = bcol[8 * n * LDS_C + 4 * (ks + 1)];
                        }
#pragma unroll
                        for (int n = 0; n < NT; n++) {
                            dmma(acc[0][n][0], acc[0][n][1], aw0[ks], bc[n]);
                            dmma(acc[1][n][0], acc[1][n][1], aw1[ks], bc[n]);
                        }
#pragma unroll
                        for (int n = 0; n < NT; n++) bc[n] = bn[n];
                    }
                    advance((g + 1) % NG, st * NG + g + 1);             // the slot index is a compile-time constant
                }
            }
        }
        __pipeline_wait_prior(0);
        // every round streams the same tiles: start the next round's first stages before this round's stores
        __syncthreads();
        if (rd + 1 < nround) {
#pragma unroll
            for (int d = 0; d < NSTG - 1; d++) issue_stage(d);
        }
        if (live) {
            if (weighted && r0 == 0) {
                bb0 += __shfl_xor_sync(0xffffffffu, bb0, 1); bb0 += __shfl_xor_sync(0xffffffffu, bb0, 2);
                bb1 += __shfl_xor_sync(0xffffffffu, bb1, 1); bb1 += __shfl_xor_sync(0xffffffffu, bb1, 2);
                ze0 += __shfl_xor_sync(0xffffffffu, ze0, 1); ze0 += __shfl_xor_sync(0xffffffffu, ze0, 2);
                ze1 += __shfl_xor_sync(0xffffffffu, ze1, 1); ze1 += __shfl_xor_sync(0xffffffffu, ze1, 2);
                if (gk == 0) {
                    const int ca = mt0 * 8 + gm, cb = (mt0 + nw) * 8 + gm;
                    if (ca < Kc) { bb_out[ca] = bb0; ze_out[ca] = ze0; }
                    if (cb < Kc) { bb_out[cb] = bb1; ze_out[cb] = ze1; }
                }
            }
#ifdef MB_NO_EPILOGUE
            if (acc[0][0][0] == 1.2345e-300)
#endif
            {
            // destination rows first (their look-ups are independent loads), then divide and store
            double *rowp[NT][2];
            bool rdiv[NT][2];
#pragma unroll
            for (int n = 0; n < NT; n++)
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    const int r = r0 + 8 * n + 2 * gk + i;
                    rdiv[n][i] = false;
                    rowp[n][i] = r < R ? dest(r, rdiv[n][i]) : nullptr;
                }
#pragma unroll
            for (int t = 0; t < MT; t++) {
                const int c = (mt0 + t * nw) * 8 + gm;
                if (c < Kc) {
                    const double sc = F.scale[c], isc = 1.0 / sc;
#pragma unroll
                    for (int n = 0; n < NT; n++)
#pragma unroll
                        for (int i = 0; i < 2; i++)
                            if (rowp[n][i]) rowp[n][i][c] = rdiv[n][i] ? div_by(acc[t][n][i], sc, isc) : acc[t][n][i];
                }
            }
            }
        }
    }
    __syncthreads();
}

template <bool EPIS, class Col, class Dest>
__device__ inline void contract_mma(const FoldData &F, int K, int Kc, int R, int n_aligned, Col col, Dest dest, double *sV,
                                    const double *wv = nullptr, const double *ev = nullptr, double *bb_out = nullptr, double *ze_out = nullptr)
{
    const int Rp = (R + 7) & ~7;
    __syncthreads();
    PHASE(PH_CONTRACT);
    for (int r0 = 0; r0 < Rp; r0 += 8 * NT_MAX) {
        const int nt = min(NT_MAX, (Rp - r0) >> 3);
        switch (nt) {
        case 1: mma_pass<1, EPIS>(F, K, Kc, R, r0, n_aligned, col, dest, sV, wv, ev, bb_out, ze_out); break;
        case 2: mma_pass<2, EPIS>(F, K, Kc, R, r0, n_aligned, col, dest, sV, wv, ev, bb_out, ze_out); break;
        case 3: mma_pass<3, EPIS>(F, K, Kc, R, r0, n_aligned, col, dest, sV, wv, ev, bb_out, ze_out); break;
        default: mma_pass<4, EPIS>(F, K, Kc, R, r0, n_aligned, col, dest, sV, wv, ev, bb_out, ze_out); break;
        }
    }
}

// R <= RCS right-hand sides (the single new column of an add): one candidate per thread, the right-hand
// sides of up to SIMT_ROWS rows held in shared memory (row-major, RCS per row) and broadcast with 32-byte loads.
constexpr int SIMT_ROWS = (2 * QT * LDS_V) / RCS;

template <bool EPIS, class XT, class ColVal, class Dest>
__device__ inline void contract_simt(const XT *__restrict__ X, int N, int K, int Kc, int R, ColVal colval,
                                     Dest dest, const double *__restrict__ scale, double *sV, bool sq_first)
{
    const int T = blockDim.x;
    __syncthreads();
    PHASE(PH_CONTRACT);
    for (int hb = 0; hb < N; hb += SIMT_ROWS) {
        const int nh = min(SIMT_ROWS, N - hb);
        __syncthreads();
        for (int idx = threadIdx.x; idx < nh * RCS; idx += T) {
            const int h = idx % nh, r = idx / nh;                         // row fastest: coalesced reads of the sources
            sV[h * RCS + r] = r < R ? colval(r, hb + h) : 0.0;
        }
        __syncthreads();
        for (int c0 = 0; c0 < Kc; c0 += T) {
            const int c = c0 + threadIdx.x;
            if (c >= Kc) continue;
            Cand<EPIS> cd(c, K);
            double acc[RCS];
#pragma unroll
            for (int r = 0; r < RCS; r++) acc[r] = 0.0;
            double xv[PF];
#pragma unroll
            for (int i = 0; i < PF; i++) xv[i] = cd.at(X + (size_t)min(hb + i, N - 1) * K);
            for (int hh = 0; hh < nh; hh += PF) {
                double xn[PF];
#pragma unroll
                for (int i = 0; i < PF; i++) xn[i] = cd.at(X + (size_t)min(hb + hh + PF + i, N - 1) * K);
#pragma unroll
                for (int i = 0; i < PF; i++) {
                    if (hh + i < nh) {
                        const double x = xv[i];
                        const double4 a = *reinterpret_cast<const double4 *>(sV + (hh + i) * RCS);
                        acc[0] = fma(sq_first ? x * x : x, a.x, acc[0]);
                        acc[1] = fma(x, a.y, acc[1]);
                        acc[2] = fma(x, a.z, acc[2]);
                        acc[3] = fma(x, a.w, acc[3]);
                    }
                }
#pragma unroll
                for (int i = 0; i < PF; i++) xv[i] = xn[i];
            }
            const double sc = scale[c];
#pragma unroll
            for (int r = 0; r < RCS; r++) {
                if (r < R) {
                    bool dv = false;
                    double *row = dest(r, dv);
                    // row chunks after the first accumulate onto the stored partial sum (un-scaled until the last chunk)
                    double v = acc[r];
                    if (hb > 0) v += row[c];
                    row[c] = (dv && hb + nh >= N) ? v / sc : v;
                }
            }
        }
    }
    __syncthreads();
}

// One right-hand side (the new column of an add, the most frequent contraction of a Gaussian fit): a WARP per
// candidate over the transposed training matrix.  The right-hand side sits in shared memory in the matrix's
// permuted row order; a lane takes 4 consecutive positions per 128 (one 32-bit word of int8 codes, or four
// doubles), keeps one partial sum per position and the warp combines them in a fixed order -- 4x fewer
// instructions than a thread per candidate, and the loads of two candidates are in flight together.
// Same arithmetic sequence for every candidate (duplicates tie exactly).
constexpr int COL_MAX_ROWS = 5120;

template <bool EPIS, class ColVal, class Dest>
__device__ inline void contract_col(const FoldData &F, int K, int Kc, ColVal colval, Dest dest, double *sV)
{
    const int N = F.ntr, ldt = F.ldt, T = blockDim.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
    const int8_t *__restrict__ X8 = F.XT8;
    const double *__restrict__ Xd = F.XTd;
    __syncthreads();
    PHASE(PH_CONTRACT);
    for (int pos = threadIdx.x; pos < ldt; pos += T) {
        const int h = (pos & ~15) | ((pos & 3) << 2) | ((pos >> 2) & 3);          // row stored at this position (see mma_pass)
        sV[pos] = h < N ? colval(0, h) : 0.0;
    }
    __syncthreads();
    bool dv = false;
    double *row = dest(0, dv);
    // int8: all the words a lane needs from both candidates for 1024 positions are requested before the first is used
    // (up to 32 loads in flight per lane: the matrix comes from L2, a dependent load per 128 positions would pay its
    // latency eight times per candidate); f64: one 128-position step at a time.
    constexpr int CH = 8;
    auto accumulate = [&](const Cand<EPIS> &cd, int wi, int wj, int p4, double (&z)[4]) {
        const double4 v = *reinterpret_cast<const double4 *>(sV + p4);
        z[0] = fma(cd.from_words(wi, wj, 0), v.x, z[0]); z[1] = fma(cd.from_words(wi, wj, 1), v.y, z[1]);
        z[2] = fma(cd.from_words(wi, wj, 2), v.z, z[2]); z[3] = fma(cd.from_words(wi, wj, 3), v.w, z[3]);
    };
    auto partial_f64 = [&](const Cand<EPIS> &cd, int p4, double (&z)[4]) {
        const double4 v = *reinterpret_cast<const double4 *>(sV + p4);
        const double2 *pi = reinterpret_cast<const double2 *>(Xd + (size_t)cd.i * ldt + p4);
        const double2 a = pi[0], c = pi[1];
        double x[4] = {a.x, a.y, c.x, c.y};
        if (EPIS && cd.i != cd.j) {
            const double2 *pj = reinterpret_cast<const double2 *>(Xd + (size_t)cd.j * ldt + p4);
            const double2 e = pj[0], f = pj[1];
            x[0] *= e.x; x[1] *= e.y; x[2] *= f.x; x[3] *= f.y;
        }
        z[0] = fma(x[0], v.x, z[0]); z[1] = fma(x[1], v.y, z[1]); z[2] = fma(x[2], v.z, z[2]); z[3] = fma(x[3], v.w, z[3]);
    };
    for (int c0 = wid; c0 < Kc; c0 += 2 * nw) {
        const int c1 = c0 + nw;
        const bool two = c1 < Kc;
        Cand<EPIS> cda(c0, K), cdb(two ? c1 : c0, K);
        double za[4] = {0.0, 0.0, 0.0, 0.0}, zb[4] = {0.0, 0.0, 0.0, 0.0};
        if (X8) {
            const int8_t *ai = X8 + (size_t)cda.i * ldt, *aj = X8 + (size_t)cda.j * ldt;
            const int8_t *bi = X8 + (size_t)cdb.i * ldt, *bj = X8 + (size_t)cdb.j * ldt;
            const bool pa = EPIS && cda.i != cda.j, pb = EPIS && cdb.i != cdb.j;
            for (int base = 4 * lane; base < ldt; base += 128 * CH) {
                int wai[CH], waj[CH], wbi[CH], wbj[CH];
#pragma unroll
                for (int u = 0; u < CH; u++) {
                    const int p4 = base + 128 * u;
                    const bool in = p4 < ldt;
                    wai[u] = in ? *reinterpret_cast<const int *>(ai + p4) : 0;
                    wbi[u] = in ? *reinterpret_cast<const int *>(bi + p4) : 0;
                    waj[u] = (in && pa) ? *reinterpret_cast<const int *>(aj + p4) : 0;
                    wbj[u] = (in && pb) ? *reinterpret_cast<const int *>(bj + p4) : 0;
                }
#pragma unroll
                for (int u = 0; u < CH; u++) {
                    const int p4 = base + 128 * u;
                    if (p4 < ldt) { accumulate(cda, wai[u], waj[u], p4, za); accumulate(cdb, wbi[u], wbj[u], p4, zb); }
                }
            }
        } else {
            for (int p4 = 4 * lane; p4 < ldt; p4 += 128) { partial_f64(cda, p4, za); partial_f64(cdb, p4, zb); }
        }
        const double ta = warp_sum((za[0] + za[1]) + (za[2] + za[3])), tb = warp_sum((zb[0] + zb[1]) + (zb[2] + zb[3]));
        if (lane == 0) {
            row[c0] = dv ? ta / F.scale[c0] : ta;
            if (two) row[c1] = dv ? tb / F.scale[c1] : tb;
        }
    }
    __syncthreads();
}

// Dispatch on the number of right-hand sides (and, in the SIMT path, on the storage type of the training matrix).
//   col(r)        base pointer of right-hand side r (see mma_pass); the first n_aligned are 16-byte aligned columns
//   dest(r, div)  destination row of right-hand side r; div set when the result is divided by the column norm
//   wv            optional row weights folded into the product (binomial); the SIMT path applies them per row
template <bool EPIS, class Col, class Dest>
__device__ inline void contract_x(const FoldData &F, int K, int Kc, int R, int n_aligned, Col col, Dest dest, double *sV,
                                  const double *wv = nullptr, const double *ev = nullptr, double *bb_out = nullptr, double *ze_out = nullptr)
{
    if (R == 1 && !bb_out && F.ldt <= COL_MAX_ROWS) {
        contract_col<EPIS>(F, K, Kc, [&](int r, int h) { const double v = col(r)[h]; return wv ? v * wv[h] : v; }, dest, sV);
    } else if (R <= SIMT_R_MAX && !bb_out) {
        auto colval = [&](int r, int h) { const double v = col(r)[h]; return wv ? v * wv[h] : v; };
        if (F.Xtr8) contract_simt<EPIS, int8_t>(F.Xtr8, F.ntr, K, Kc, R, colval, dest, F.scale, sV, false);
        else contract_simt<EPIS, double>(F.Xtr, F.ntr, K, Kc, R, colval, dest, F.scale, sV, false);
    } else {
        contract_mma<EPIS>(F, K, Kc, R, n_aligned, col, dest, sV, wv, ev, bb_out, ze_out);
    }
}

// SIMT form of the quadratic forms, used while the active set is small (M <= QUAD_SIMT_M): measured faster than the
// tensor-core form there (the DMMA form wins by 3-4x at M ~ 200).
// Quadratic forms of the candidate cache against the active-set inverse:
//   quad[c] = g_c' SIGMA g_c,  lin[c] = g_c' v      with g_c = G[:, c]   (FullStat*, MainEff.c:1291-1316)
// SIGMA is first copied to a padded layout (leading dimension ldp, multiple of 8, in `sigp`) so a
// thread reads 8 consecutive entries of a row with two 32-byte loads; z_p accumulates over j in
// ascending order and quad over p in ascending order, as the reference's loops do.
template <int PW, class Emit>       // PW = z accumulators per candidate: the cache rows are re-read M / PW times
__device__ inline void quad_forms_simt(const Slab &s, const double *sigma, double *sigp_global, int M, int Kc, const double *v,
                                  double *smem /* >= 4096 + 1040 doubles */, Emit emit)
{
    PHASE(PH_QUAD);
    const int T = blockDim.x;
    const int ldp = (M + PW - 1) / PW * PW;
    // padded copy sigp[j][p] = SIGMA(p, j): in shared memory when it fits (M <= 64), else in the spare SIGMA buffer
    double *sigp = (M * ldp <= 4096) ? smem : sigp_global;
    size_t *rowoff = reinterpret_cast<size_t *>(smem + 4096);          // G row offsets: no dependent index load in the hot loop
    __syncthreads();
    // SIGMA is symmetric: g'SIGMA g = sum_p g_p (SIGMA_pp g_p + 2 sum_{j<p} SIGMA_pj g_j), so only the lower triangle is
    // multiplied (off-diagonal entries doubled -- exact -- and the upper triangle of the copy zero): half the FMAs
    for (int idx = threadIdx.x; idx < M * ldp; idx += T) {
        const int j = idx / ldp, p = idx - j * ldp;
        sigp[idx] = (p < M && j <= p) ? (j < p ? 2.0 * sigma[p * M + j] : sigma[p * M + j]) : 0.0;
    }
    const bool off_smem = M <= 1040;
    if (off_smem) for (int j = threadIdx.x; j < M; j += T) rowoff[j] = (size_t)s.grow[j] * Kc;
    __syncthreads();
    auto roff = [&](int j) -> size_t { return off_smem ? rowoff[j] : (size_t)s.grow[j] * Kc; };
    // two candidates per thread share every SIGMA row fetched; four G rows are loaded ahead of their FMAs
    for (int c0 = 0; c0 < Kc; c0 += 2 * T) {
        const int ca = c0 + threadIdx.x, cb = ca + T;
        const bool la = ca < Kc, lb = cb < Kc;
        const int xa = la ? ca : 0, xb = lb ? cb : 0;
        double quad_a = 0, lin_a = 0, quad_b = 0, lin_b = 0;
        for (int p0 = 0; p0 < M; p0 += PW) {
            double za[PW], zb[PW];
#pragma unroll
            for (int q = 0; q < PW; q++) { za[q] = 0.0; zb[q] = 0.0; }
            const int jend = min(M, p0 + PW);             // rows j > p hold zeros
            for (int j = 0; j < jend; j += 4) {
                double ga[4], gb[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const size_t o = roff(min(j + u, M - 1));
                    ga[u] = s.G[o + xa]; gb[u] = s.G[o + xb];
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    if (j + u < jend) {
                        const double4 *row = reinterpret_cast<const double4 *>(sigp + (size_t)(j + u) * ldp + p0);
#pragma unroll
                        for (int q4 = 0; q4 < PW / 4; q4++) {
                            const double4 a = row[q4];
                            za[4 * q4 + 0] = fma(ga[u], a.x, za[4 * q4 + 0]); za[4 * q4 + 1] = fma(ga[u], a.y, za[4 * q4 + 1]);
                            za[4 * q4 + 2] = fma(ga[u], a.z, za[4 * q4 + 2]); za[4 * q4 + 3] = fma(ga[u], a.w, za[4 * q4 + 3]);
                            zb[4 * q4 + 0] = fma(gb[u], a.x, zb[4 * q4 + 0]); zb[4 * q4 + 1] = fma(gb[u], a.y, zb[4 * q4 + 1]);
                            zb[4 * q4 + 2] = fma(gb[u], a.z, zb[4 * q4 + 2]); zb[4 * q4 + 3] = fma(gb[u], a.w, zb[4 * q4 + 3]);
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < PW; q++) {
                if (p0 + q < M) {
                    const size_t o = roff(p0 + q);
                    const double gpa = s.G[o + xa], gpb = s.G[o + xb];
                    quad_a = fma(za[q], gpa, quad_a); quad_b = fma(zb[q], gpb, quad_b);
                    if (v) { lin_a = fma(gpa, v[p0 + q], lin_a); lin_b = fma(gpb, v[p0 + q], lin_b); }
                }
            }
        }
        if (la) emit(ca, quad_a, lin_a);
        if (lb) emit(cb, quad_b, lin_b);
    }
    __syncthreads();
}


// Quadratic forms of the candidate cache against the active-set inverse:
//   quad[c] = g_c' SIGMA g_c,  lin[c] = g_c' v      with g_c = G[:, c]   (FullStat*, MainEff.c:1291-1316)
// Tensor-core form: Z = G' SIGMA is a (Kc x M) x (M x M) product -- A fragments are 8 candidates x 4 cache
// rows read straight from G (through the row permutation), B fragments come from a zero-padded copy of
// SIGMA in shared memory -- and quad[c] = sum_p Z[c][p] G[p][c] is folded into the accumulator epilogue.
// For M <= 2*QT the padded SIGMA stays resident in shared memory for the whole call; larger matrices are
// streamed through the same double buffer in 64-column chunks from a padded copy in the spare SIGMA buffer.
// Every candidate goes through the identical sequence of operations (duplicate columns tie exactly).
template <int NT>
__device__ inline void quad_chunk(const double *__restrict__ G, const size_t *rowoff, const int *grow, int M, int Kc,
                                  const double *__restrict__ sigp, int ldp, int p0, double *sV, bool resident,
                                  bool live, int c0, int c1, const double *__restrict__ v, double (&q)[MT], double (&l)[MT])
{
    const int lane = threadIdx.x & 31;
    const int gm = lane >> 2, gk = lane & 3;
    const int jlim = min(M, p0 + 8 * NT);                   // lower triangle only (see quad_forms_mma): rows j > p hold zeros
    const int nstage = (jlim + QT - 1) / QT;
    auto roff = [&](int j) -> size_t { return rowoff ? rowoff[j] : (size_t)grow[j] * Kc; };
    double acc[MT][NT][2];
#pragma unroll
    for (int t = 0; t < MT; t++)
#pragma unroll
        for (int n = 0; n < NT; n++) { acc[t][n][0] = 0.0; acc[t][n][1] = 0.0; }
    double xv[MT][4], xn[MT][4], xn2[MT][4];                // cache rows come from L2: two groups (32 rows) in flight
    auto fetch = [&](double (&x)[MT][4], int jb) {
#pragma unroll
        for (int ks = 0; ks < 4; ks++) {
            const size_t o = roff(min(jb + 4 * ks + gk, M - 1));
            x[0][ks] = G[o + c0];
            x[1][ks] = G[o + c1];
        }
    };
    if (!resident) stage_tile<false>(sV, LDS_V, sigp, ldp, 0, p0, 8 * NT);
    if (live) { fetch(xv, 0); fetch(xn, 16); }
    if (!resident) { __pipeline_wait_prior(0); __syncthreads(); }
    for (int st = 0; st < nstage; st++) {
        const double *buf = sV + (st & 1) * (QT * LDS_V);
        if (!resident && st + 1 < nstage) stage_tile<false>(sV + ((st + 1) & 1) * (QT * LDS_V), LDS_V, sigp, ldp, (st + 1) * QT, p0, 8 * NT);
        if (live) {
#pragma unroll
            for (int g = 0; g < QT / 16; g++) {
                if (st * QT + 16 * g < jlim) {                 // warp-uniform: groups past the last contributing cache row are skipped
                    fetch(xn2, st * QT + 16 * (g + 2));
#pragma unroll
                    for (int ks = 0; ks < 4; ks++) {
                        const double *brow = buf + (16 * g + 4 * ks + gk) * LDS_V + gm + (resident ? p0 : 0);   // the resident tile holds every column
                        double b[NT];
#pragma unroll
                        for (int n = 0; n < NT; n++) b[n] = brow[8 * n];
#pragma unroll
                        for (int n = 0; n < NT; n++) {
                            dmma(acc[0][n][0], acc[0][n][1], xv[0][ks], b[n]);
                            dmma(acc[1][n][0], acc[1][n][1], xv[1][ks], b[n]);
                        }
                    }
#pragma unroll
                    for (int ks = 0; ks < 4; ks++) { xv[0][ks] = xn[0][ks]; xv[1][ks] = xn[1][ks]; xn[0][ks] = xn2[0][ks]; xn[1][ks] = xn2[1][ks]; }
                }
            }
        }
        if (!resident) { __pipeline_wait_prior(0); __syncthreads(); }
    }
    if (live) {
#pragma unroll
        for (int n = 0; n < NT; n++)
#pragma unroll
            for (int i = 0; i < 2; i++) {
                const int pp = p0 + 8 * n + 2 * gk + i;
                if (pp < M) {
                    const size_t o = roff(pp);
                    const double g0 = G[o + c0], g1 = G[o + c1];
                    q[0] = fma(acc[0][n][i], g0, q[0]);
                    q[1] = fma(acc[1][n][i], g1, q[1]);
                    if (v) { const double vp = v[pp]; l[0] = fma(g0, vp, l[0]); l[1] = fma(g1, vp, l[1]); }
                }
            }
    }
}

template <class Emit>
__device__ inline void quad_forms_mma(const Slab &s, const double *sigma, double *sigp_global, int M, int Kc, const double *v,
                                      double *smem /* >= 2*QT*LDS_V + 784 doubles */, Emit emit)
{
    PHASE(PH_QUAD);
    const int T = blockDim.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
    const int gm = lane >> 2, gk = lane & 3;
    const int ldp = (M + 7) & ~7, Mp = ((M + QT - 1) / QT) * QT;
    const bool resident = Mp <= 2 * QT;
    size_t *rowoff = M <= 784 ? reinterpret_cast<size_t *>(smem + 2 * QT * LDS_V) : nullptr;
    __syncthreads();
    // zero-padded copy sigp[j][p] of SIGMA's lower triangle, off-diagonal entries doubled (exact): SIGMA is symmetric, so
    // g'SIGMA g = sum_p g_p (SIGMA_pp g_p + 2 sum_{j<p} SIGMA_pj g_j) and a chunk of columns p only needs the cache rows
    // j <= p -- half the DMMAs.  Straight into the shared tile layout when resident.
    auto tri = [&](int j, int p) { return (p < M && j <= p) ? (j < p ? 2.0 * sigma[p * M + j] : sigma[p * M + j]) : 0.0; };
    if (resident) {
        for (int idx = threadIdx.x; idx < Mp * ldp; idx += T) {
            const int j = idx / ldp, p = idx - j * ldp;
            smem[j * LDS_V + p] = tri(j, p);
        }
    } else {
        for (int idx = threadIdx.x; idx < Mp * ldp; idx += T) {
            const int j = idx / ldp, p = idx - j * ldp;
            sigp_global[idx] = tri(j, p);
        }
    }
    if (rowoff) for (int j = threadIdx.x; j < M; j += T) rowoff[j] = (size_t)s.grow[j] * Kc;
    __syncthreads();
    const int n_mtile = (Kc + 7) >> 3;
    const int per_round = nw * MT;
    const int nround = (n_mtile + per_round - 1) / per_round;
    for (int rd = 0; rd < nround; rd++) {
        const int mt0 = rd * per_round + wid;
        const bool live = mt0 < n_mtile;
        const int ca = mt0 * 8 + gm, cb = (mt0 + nw) * 8 + gm;
        const int c0 = min(ca, Kc - 1), c1 = min(cb, Kc - 1);
        double q[MT] = {0.0, 0.0}, l[MT] = {0.0, 0.0};
        for (int p0 = 0; p0 < ldp; p0 += 8 * NT_MAX) {
            const int nt = min(NT_MAX, (ldp - p0) >> 3);
            switch (nt) {
            case 1: quad_chunk<1>(s.G, rowoff, s.grow, M, Kc, sigp_global, ldp, p0, smem, resident, live, c0, c1, v, q, l); break;
            case 2: quad_chunk<2>(s.G, rowoff, s.grow, M, Kc, sigp_global, ldp, p0, smem, resident, live, c0, c1, v, q, l); break;
            case 3: quad_chunk<3>(s.G, rowoff, s.grow, M, Kc, sigp_global, ldp, p0, smem, resident, live, c0, c1, v, q, l); break;
            default: quad_chunk<4>(s.G, rowoff, s.grow, M, Kc, sigp_global, ldp, p0, smem, resident, live, c0, c1, v, q, l); break;
            }
        }
        if (live) {
#pragma unroll
            for (int t = 0; t < MT; t++) {
                q[t] += __shfl_xor_sync(0xffffffffu, q[t], 1); q[t] += __shfl_xor_sync(0xffffffffu, q[t], 2);
                l[t] += __shfl_xor_sync(0xffffffffu, l[t], 1); l[t] += __shfl_xor_sync(0xffffffffu, l[t], 2);
            }
            if (gk == 0) {
                if (ca < Kc) emit(ca, q[0], l[0]);
                if (cb < Kc) emit(cb, q[1], l[1]);
            }
        }
    }
    __syncthreads();
}

constexpr int QUAD_SIMT_M = 64;
template <class Emit>
__device__ inline void quad_forms(const Slab &s, const double *sigma, double *sigp_global, int M, int Kc, const double *v,
                                  double *smem, Emit emit)
{
    if (M <= QUAD_SIMT_M) quad_forms_simt<8>(s, sigma, sigp_global, M, Kc, v, smem, emit);
    else quad_forms_mma(s, sigma, sigp_global, M, Kc, v, smem, emit);
}

// z[c] = sum_j G[row j][c] * vec[j], j ascending, for every candidate c (the S/Q corrections of the three actions,
// MainEff.c:577-587, 1699-1711, 1800-1808).  Two candidates per thread and four cache rows loaded ahead of their
// FMAs: the loads come from L2 and a plain loop keeps only one or two of them in flight.
template <class Emit>
__device__ inline void cache_dot(const Slab &s, int M, int Kc, const double *__restrict__ vec, Emit emit)
{
    const int T = blockDim.x;
    for (int c0 = threadIdx.x; c0 < Kc; c0 += 2 * T) {
        const int c1 = c0 + T;
        const bool two = c1 < Kc;
        const int cb = two ? c1 : c0;
        double za = 0, zb = 0;
        int j = 0;
        for (; j + 4 <= M; j += 4) {
            double ga[4], gb[4], v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const size_t o = (size_t)s.grow[j + u] * Kc;
                ga[u] = s.G[o + c0]; gb[u] = s.G[o + cb]; v[u] = vec[j + u];
            }
#pragma unroll
            for (int u = 0; u < 4; u++) { za = fma(ga[u], v[u], za); zb = fma(gb[u], v[u], zb); }
        }
        for (; j < M; j++) {
            const size_t o = (size_t)s.grow[j] * Kc;
            const double vj = vec[j];
            za = fma(s.G[o + c0], vj, za); zb = fma(s.G[o + cb], vj, zb);
        }
        emit(c0, za);
        if (two) emit(c1, zb);
    }
}

// dot products of active columns with a vector: out[i] = sum_h phi_i[h] * v[h], one warp per i.
__device__ inline void phi_dot(const double *phi, int N, int M, const double *v, double *out, double scale)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5, LD = phi_ld(N);
    for (int i = wid; i < M; i += 2 * nw) {                 // two columns per warp: twice the loads in flight, same sums
        const int i2 = i + nw;
        const bool two = i2 < M;
        const double *p = phi + (size_t)i * LD, *q = phi + (size_t)(two ? i2 : i) * LD;
        double za = 0, zb = 0;
#pragma unroll 4
        for (int h = lane; h < N; h += 32) { const double vv = v[h]; za = fma(p[h], vv, za); zb = fma(q[h], vv, zb); }
        za = warp_sum(za); zb = warp_sum(zb);
        if (lane == 0) { out[i] = za * scale; if (two) out[i2] = zb * scale; }
    }
    __syncthreads();
}

// In-place inverse of a symmetric positive-definite M x M matrix (leading dimension M) by the
// symmetric sweep operator.  Plays the role of dpotrf + dpotri (MainEff.c:1346-1369).  Returns
// false (to every thread) when a pivot is not positive.
//   * one barrier per pivot: the thread that rewrites entry (i, k+1) also publishes it as the next
//     pivot column (double-buffered in `colbuf`, 2*M doubles);
//   * warps own columns, lanes own rows (no integer division, conflict-free);
//   * when M <= SWEEP_SMEM_M the matrix is swept inside shared memory (`sm`) and copied back.
constexpr int SWEEP_SMEM_M = 64;

__device__ inline bool sweep_core(double *a, int M, double *colbuf)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    double *cur = colbuf, *nxt = colbuf + M;
    for (int i = threadIdx.x; i < M; i += blockDim.x) cur[i] = a[i];          // column 0
    __syncthreads();
    bool ok = true;
    for (int k = 0; k < M; k++) {
        const double d = cur[k];
        if (!(d > 0.0)) { ok = false; break; }        // uniform: every thread reads the same value
        const double dinv = 1.0 / d;
        for (int j = wid; j < M; j += nw) {
            const double cj = cur[j];
            double *col = a + (size_t)j * M;
            for (int i = lane; i < M; i += 32) {
                double v;
                if (i == k && j == k) v = -dinv;
                else if (i == k) v = cj * dinv;
                else if (j == k) v = cur[i] * dinv;
                else v = col[i] - (cur[i] * cj) * dinv;
                col[i] = v;
                if (j == k + 1) nxt[i] = v;
            }
        }
        __syncthreads();
        double *t = cur; cur = nxt; nxt = t;
    }
    return ok;
}

// Panel variant of sweep_core for matrices that do not fit in registers (M > SWEEP_SMEM_M): NB pivots per pass
// over the matrix instead of one.  Phase A sweeps the NB pivot columns themselves inside shared memory with the
// one-pivot formulas (saving each pivot's pre-update column C_p and reciprocal); phase B applies the NB rank-1
// updates to the rest of the matrix as ONE rank-NB update on the FP64 tensor cores:
//     a(i, j) -= sum_p C_p[i] * (C_p[j] / d_p)          8 x 8 tiles, two DMMAs per tile for NB = 8,
// lower triangle only, mirrored on store so the matrix stays exactly symmetric; the rows of the panel's pivots are
// the mirror image of the swept panel columns.  Global traffic and block barriers per element drop by NB and the
// update runs at tensor-core rate instead of ~7 instructions per element and pivot.
//   sm: SWEEP_PANEL_DOUBLES doubles
constexpr int SWEEP_PANEL_DOUBLES = 5120;

__device__ inline bool sweep_panel(double *a, int M, double *sm)
{
    // While the sweep runs only the LOWER triangle of `a` (element (i, j), i >= j, at a[j*M + i]) is kept current: the
    // rank-NB update reads and writes each entry once per panel instead of writing it twice (entry and mirror image) --
    // the matrix lives in L2, and with every block of the grid sweeping, L2 bandwidth is what a panel costs.  The upper
    // triangle is rebuilt (and the sign flipped) once at the end.  Returns with the NEGATED inverse's sign already
    // restored, i.e. a = inverse.
    const int T = blockDim.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = T >> 5;
    const int gm = lane >> 2, gk = lane & 3;
    const int Mp = ((M + 7) & ~7) + 4;                    // row stride of the panel arrays (tiles may read up to 7 past M)
    int NB = 8;
    while (NB > 2 && 2 * NB * Mp + NB > SWEEP_PANEL_DOUBLES) NB >>= 1;
    const int KS = (NB + 3) >> 2;                         // k-steps of the rank-NB update (NB = 2 is padded to 4 with zero rows)
    const int NBp = 4 * KS;
    double *Pn = sm, *C = sm + NBp * Mp, *dv = C + NBp * Mp;      // dv[p] = 1 / pivot p (0 for the padding rows)
    const int nt = (M + 7) >> 3;
    bool ok = true;
    for (int k0 = 0; k0 < M; k0 += NB) {
        const int nb = min(NB, M - k0);
        __syncthreads();
        // panel columns k0 .. k0+nb-1, all rows: rows above the diagonal come from the mirror-image entries
        for (int i = threadIdx.x; i < Mp; i += T) {       // a thread takes row i of all panel columns: NBp independent loads, no division
#pragma unroll
            for (int q = 0; q < 8; q++) {
                if (q < NBp) {
                    const int j = k0 + q;
                    const double v = (q < nb && i < M) ? (i >= j ? a[(size_t)j * M + i] : a[(size_t)i * M + j]) : 0.0;
                    Pn[q * Mp + i] = v;
                    C[q * Mp + i] = q == 0 ? v : 0.0;     // C_0 = the first pivot's column; rows past nb and entries past M contribute nothing to the update
                }
            }
        }
        if (threadIdx.x < NBp) dv[threadIdx.x] = 0.0;
        // phase A: the pivots of this panel, applied to the panel's own columns
        // (C_p, the pivot's pre-update column that phase B needs, is written by the warp that updates column p during pivot
        //  p - 1 -- C_0 by the load above -- so a pivot costs one barrier)
        for (int p = 0; p < nb; p++) {
            __syncthreads();
            const int k = k0 + p;
            const double *cp = C + p * Mp;
            const double d = cp[k];
            if (!(d > 0.0)) { ok = false; break; }        // uniform: every thread reads the same value
            const double dinv = 1.0 / d;
            if (threadIdx.x == 0) dv[p] = dinv;
            for (int q = wid; q < nb; q += nw) {              // a warp per panel column, lanes over rows (no integer division)
                const int j = k0 + q;
                const double cj = cp[j];
                const bool next_pivot = q == p + 1;
                for (int i = lane; i < M; i += 32) {
                    double v;
                    if (i == k && j == k) v = -dinv;
                    else if (i == k) v = cj * dinv;
                    else if (j == k) v = cp[i] * dinv;
                    else v = Pn[q * Mp + i] - (cp[i] * cj) * dinv;
                    Pn[q * Mp + i] = v;
                    if (next_pivot) C[q * Mp + i] = v;
                }
            }
        }
        if (!ok) break;
        __syncthreads();
        const double dv0 = dv[gk], dv1 = KS > 1 ? dv[4 + gk] : 0.0;     // B fragments are C_p[j] / d_p, formed on the fly
        // phase B: rank-nb update of the lower triangle.  The nt (nt + 1) / 2 tiles, row-major, are cut into one contiguous
        // range per warp (balanced to a tile); a warp works on PB tiles at a time: the tile's own entries come from L2 and a
        // single load -> DMMA -> store chain per warp would pay that latency once per tile.  Tiles that lie inside the
        // panel's own rows or columns are skipped: phase A has produced those entries and the write-back below stores them.
        constexpr int PB = 8;
        const int tp0 = k0 >> 3;                                         // NB = 8: tile row / column tp0 is the panel's
        const bool panel_aligned = NB == 8;                              // narrower panels share a tile with other columns: update everything
        const int ntile = nt * (nt + 1) / 2;
        const int t_begin = (int)((long long)ntile * wid / nw), t_end = (int)((long long)ntile * (wid + 1) / nw);
        int ti = (int)((sqrt(8.0 * t_begin + 1.0) - 1.0) * 0.5);
        while (ti * (ti + 1) / 2 > t_begin) ti--;
        while ((ti + 1) * (ti + 2) / 2 <= t_begin) ti++;
        int tj = t_begin - ti * (ti + 1) / 2;
        for (int tb = t_begin; tb < t_end; tb += PB) {
            int ti_[PB], tj_[PB];
            double c0[PB], c1[PB];
#pragma unroll
            for (int u = 0; u < PB; u++) {
                ti_[u] = ti; tj_[u] = tj;
                const bool lv = tb + u < t_end && !(panel_aligned && (ti == tp0 || tj == tp0));
                if (!lv) ti_[u] = -1;
                const int i = 8 * ti + gm, j0 = 8 * tj + 2 * gk;          // this lane's elements: (i, j0) and (i, j0 + 1)
                c0[u] = (lv && i < M && j0 < M) ? a[(size_t)j0 * M + i] : 0.0;
                c1[u] = (lv && i < M && j0 + 1 < M) ? a[(size_t)(j0 + 1) * M + i] : 0.0;
                if (++tj > ti) { ti++; tj = 0; }
            }
#pragma unroll
            for (int u = 0; u < PB; u++) {
                if (ti_[u] >= 0) {                                        // warp-uniform
                    dmma(c0[u], c1[u], -C[(gk) * Mp + 8 * ti_[u] + gm], C[(gk) * Mp + 8 * tj_[u] + gm] * dv0);
                    if (KS > 1) dmma(c0[u], c1[u], -C[(4 + gk) * Mp + 8 * ti_[u] + gm], C[(4 + gk) * Mp + 8 * tj_[u] + gm] * dv1);
                }
            }
#pragma unroll
            for (int u = 0; u < PB; u++) {
                if (ti_[u] >= 0) {
                    const int i = 8 * ti_[u] + gm, j0 = 8 * tj_[u] + 2 * gk;
                    if (i < M && j0 < M && i >= j0) a[(size_t)j0 * M + i] = c0[u];
                    if (i < M && j0 + 1 < M && i >= j0 + 1) a[(size_t)(j0 + 1) * M + i] = c1[u];
                }
            }
        }
        __syncthreads();
        // the panel's own columns: below the diagonal in place, above it at the mirror-image position (row k0+q of the
        // lower triangle)
        for (int q = 0; q < nb; q++) {
            const int j = k0 + q;
            for (int i = threadIdx.x; i < M; i += T) {
                const double v = Pn[q * Mp + i];
                if (i >= j) a[(size_t)j * M + i] = v;
                else if (i < k0) a[(size_t)i * M + j] = v;        // (k0 <= i < j: that entry is column i's, written by its own pass)
            }
        }
    }
    __syncthreads();
    // sign, and the upper triangle from the lower one: warps own columns j, lanes rows i >= j
    if (ok)
        for (int j = wid; j < M; j += nw)
            for (int i = j + lane; i < M; i += 32) {
                const double v = -a[(size_t)j * M + i];
                a[(size_t)j * M + i] = v;
                if (i != j) a[(size_t)i * M + j] = v;
            }
    __syncthreads();
    return ok;
}

// Register-resident variant for M <= 64 and 256 threads: thread (warp w, lane l) owns rows {l, l+32}
// x columns {w, w+8, ..., w+56} = 16 entries kept in registers across all M pivots; only the pivot
// column travels through shared memory (2 x 64 doubles, double-buffered), one barrier per pivot.
template <int NI>                                     // NI = 1: M <= 32, the second row block does not exist
__device__ inline bool sweep_regs(double *a, int M, double *colbuf /* 128 doubles of shared memory */)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double r[NI][8];
    {
        PHASE(PH_SWEEP_LS);
#pragma unroll
        for (int ii = 0; ii < NI; ii++)
#pragma unroll
            for (int jj = 0; jj < 8; jj++) {
                const int i = lane + 32 * ii, j = wid + 8 * jj;
                r[ii][jj] = (i < M && j < M) ? a[(size_t)j * M + i] : 0.0;
            }
    }
    double *cur = colbuf, *nxt = colbuf + 64;
    __syncthreads();
    if (wid == 0) {                                   // column 0 lives in warp 0 (jj = 0)
        cur[lane] = r[0][0];
        if (NI > 1) cur[lane + 32] = r[NI - 1][0];
    }
    __syncthreads();
    bool ok = true;
    for (int k = 0; k < M; k++) {
        const double d = cur[k];
        if (!(d > 0.0)) { ok = false; break; }
        const double dinv = 1.0 / d, ndinv = -dinv;
        const double ci0 = cur[lane], ci1 = NI > 1 ? cur[lane + 32] : 0.0;
        const int kn = k + 1;
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
            const int j = wid + 8 * jj;
            if (j < M) {                                  // warp-uniform: whole columns beyond M are skipped
                const double cj = cur[j];
                if (j == k) {                             // the pivot column (warp-uniform branch)
#pragma unroll
                    for (int ii = 0; ii < NI; ii++) {
                        const double ci = ii == 0 ? ci0 : ci1;
                        r[ii][jj] = lane + 32 * ii == k ? ndinv : ci * dinv;
                    }
                } else {                                  // the pivot row's entry, else the rank-1 update
                    const double cjd = cj * dinv;
#pragma unroll
                    for (int ii = 0; ii < NI; ii++) {
                        const double ci = ii == 0 ? ci0 : ci1;
                        const double u = fma(ci * cj, ndinv, r[ii][jj]);  // (ci*cj) is symmetric in (i, j): the result stays exactly symmetric
                        r[ii][jj] = lane + 32 * ii == k ? cjd : u;
                    }
                }
                if (j == kn) {                            // publish the next pivot's column
                    nxt[lane] = r[0][jj];
                    if (NI > 1) nxt[lane + 32] = r[NI - 1][jj];
                }
            }
        }
        __syncthreads();
        double *t = cur; cur = nxt; nxt = t;
    }
    if (ok) {
        PHASE(PH_SWEEP_LS);
#pragma unroll
        for (int ii = 0; ii < NI; ii++)
#pragma unroll
            for (int jj = 0; jj < 8; jj++) {
                const int i = lane + 32 * ii, j = wid + 8 * jj;
                if (i < M && j < M) a[(size_t)j * M + i] = -r[ii][jj];
            }
    }
    return ok;
}

__device__ inline bool spd_inverse_sweep(double *a, int M, double *colk, const Scratch &sc, double *sm = nullptr)
{
    PHASE(PH_SWEEP);
    const int T = blockDim.x;
    bool ok;
    if (sm && M <= SWEEP_SMEM_M && T == 256) {
        ok = M <= 32 ? sweep_regs<1>(a, M, sm) : sweep_regs<2>(a, M, sm);
    } else {
        // the panel arrays need 2 * 4 * (M rounded up to 8, + 4) doubles even at the narrowest panel: beyond that
        // (M > 632) the one-pivot sweep in global memory takes over
        const bool panel_fits = 8 * (((M + 7) & ~7) + 4) + 8 <= SWEEP_PANEL_DOUBLES;
        if (sm && panel_fits) ok = sweep_panel(a, M, sm);                                  // (restores the sign itself)
        else {
            ok = sweep_core(a, M, colk);                                                   // colk: 2*(cap+1) doubles in the slab
            if (ok) for (int idx = threadIdx.x; idx < M * M; idx += T) a[idx] = -a[idx];
        }
    }
    __syncthreads();
    return ok;
}

// Gram matrix of the active columns, H(j, k) = sum_h (phi_j[h] * w[h]) * phi_k[h]  for j <= k,
// w = nullptr meaning all ones.  This is FinalUpdate*'s PHI'PHI (MainEff.c:1869-1874) and the IRLS
// Hessian PHI'B PHI (NEmainEff.c:1911-1919, same (phi_j * beta) * phi_k order for the upper triangle
// the Cholesky reads).  Tensor-core form with no shared-memory staging and no barrier in the main loop:
// the upper triangle is cut into 16 x 16 blocks (2 x 2 DMMA tiles); a work item is one block over one
// contiguous range of rows; warps take items round-robin and read their A/B fragments (4 rows x 8 columns,
// one element per lane) straight from the column-major PHI, one k-step ahead of the DMMAs.  With few
// blocks (small M) the rows are split so that every warp has work, and the per-split partial tiles are
// combined through shared memory in a fixed order.
//   sm: GRAM_DOUBLES doubles.   out(j, k, value) is called exactly once per j <= k.
constexpr int GRAM_DOUBLES = 5120;

template <class Out>
__device__ inline void gram_mma(const double *__restrict__ phi, int N, int LD, int M, const double *__restrict__ w,
                                double *sm, Out out)
{
    PHASE(PH_GRAM);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int gm = lane >> 2, gk = lane & 3;
    const int nt = (M + 7) >> 3, ntb = (nt + 1) >> 1, P = ntb * (ntb + 1) / 2;
    const int ng = (N + 15) >> 4;                              // groups of 16 rows; lane gk owns rows 4*gk .. 4*gk+3 of a group
    int RS = 1;
    if (P < 2 * nw) RS = max(1, min(min((2 * nw + P - 1) / P, GRAM_DOUBLES / (256 * P)), ng / 2));
    const int items = P * RS, gsplit = (ng + RS - 1) / RS;
    __syncthreads();
    for (int item = wid; item < items; item += nw) {
        const int pb = item % P, sp = item / P;
        int Jb = 0, Kb = pb;
        { int rem = pb; while (rem >= ntb - Jb) { rem -= ntb - Jb; Jb++; } Kb = Jb + rem; }
        const bool diag = Jb == Kb;
        const int g0 = sp * gsplit, g1 = min(ng, g0 + gsplit);
        const double *pa0 = phi + (size_t)min(16 * Jb + gm, M - 1) * LD, *pa1 = phi + (size_t)min(16 * Jb + 8 + gm, M - 1) * LD;
        const double *pb0 = phi + (size_t)min(16 * Kb + gm, M - 1) * LD, *pb1 = phi + (size_t)min(16 * Kb + 8 + gm, M - 1) * LD;
        double acc[2][2][2];
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int b = 0; b < 2; b++) { acc[a][b][0] = 0.0; acc[a][b][1] = 0.0; }
        struct Frag { double a0[4], a1[4], b0[4], b1[4], ww[4]; };
        auto fetch = [&](int g, Frag &f) {
            const int h = 16 * g + 4 * gk, hc = min(h, LD - 4);     // whole quads past the padded column are clamped (weight 0)
            const double2 *q;
            q = reinterpret_cast<const double2 *>(pa0 + hc); { const double2 u = q[0], v2 = q[1]; f.a0[0] = u.x; f.a0[1] = u.y; f.a0[2] = v2.x; f.a0[3] = v2.y; }
            q = reinterpret_cast<const double2 *>(pa1 + hc); { const double2 u = q[0], v2 = q[1]; f.a1[0] = u.x; f.a1[1] = u.y; f.a1[2] = v2.x; f.a1[3] = v2.y; }
            if (!diag) {
                q = reinterpret_cast<const double2 *>(pb0 + hc); { const double2 u = q[0], v2 = q[1]; f.b0[0] = u.x; f.b0[1] = u.y; f.b0[2] = v2.x; f.b0[3] = v2.y; }
                q = reinterpret_cast<const double2 *>(pb1 + hc); { const double2 u = q[0], v2 = q[1]; f.b1[0] = u.x; f.b1[1] = u.y; f.b1[2] = v2.x; f.b1[3] = v2.y; }
            }
#pragma unroll
            for (int i = 0; i < 4; i++) f.ww[i] = (h + i < N) ? (w ? w[h + i] : 1.0) : 0.0;      // rows past N contribute nothing
        };
        Frag cur, nxt;
        if (g0 < g1) fetch(g0, cur);
        for (int g = g0; g < g1; g++) {
            fetch(min(g + 1, g1 - 1), nxt);
#pragma unroll
            for (int ks = 0; ks < 4; ks++) {
                const double wa0 = cur.a0[ks] * cur.ww[ks], wa1 = cur.a1[ks] * cur.ww[ks];
                const double b0 = diag ? cur.a0[ks] : cur.b0[ks], b1 = diag ? cur.a1[ks] : cur.b1[ks];
                dmma(acc[0][0][0], acc[0][0][1], wa0, b0);
                dmma(acc[0][1][0], acc[0][1][1], wa0, b1);
                if (!diag) dmma(acc[1][0][0], acc[1][0][1], wa1, b0);  // below the diagonal inside a diagonal block: not needed
                dmma(acc[1][1][0], acc[1][1][1], wa1, b1);
            }
            cur = nxt;
        }
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int b = 0; b < 2; b++)
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    if (RS == 1) {
                        const int j = 16 * Jb + 8 * a + gm, k = 16 * Kb + 8 * b + 2 * gk + i;
                        if (j < M && k < M && j <= k) out(j, k, acc[a][b][i]);
                    } else {
                        sm[(size_t)item * 256 + (a * 2 + b) * 64 + gm * 8 + 2 * gk + i] = acc[a][b][i];
                    }
                }
    }
    if (RS > 1) {
        __syncthreads();
        for (int idx = threadIdx.x; idx < P * 256; idx += blockDim.x) {
            const int pb = idx >> 8, e = idx & 255, tile = e >> 6, a = tile >> 1, b = tile & 1, m = (e >> 3) & 7, n = e & 7;
            int Jb = 0, Kb = pb;
            { int rem = pb; while (rem >= ntb - Jb) { rem -= ntb - Jb; Jb++; } Kb = Jb + rem; }
            const int j = 16 * Jb + 8 * a + m, k = 16 * Kb + 8 * b + n;
            if (j < M && k < M && j <= k) {
                double z = 0.0;
                for (int sp = 0; sp < RS; sp++) z += sm[(size_t)(sp * P + pb) * 256 + e];
                out(j, k, z);
            }
        }
    }
    __syncthreads();
}

// Pipelined Gram matrix for at most 64 active columns, from the ROW-major copy PHIt (leading dimension
// PHIT_LD = 64):  H(j, k) = sum_h (phit[h][j] * w[h]) * phit[h][k],  j <= k.
// Tiles of 32 rows (16 KB) are streamed with cp.async, double-buffered, so the copy of tile t+1
// overlaps the FMAs of tile t and there is one barrier per tile (gram_tiled pays two barriers and
// an exposed global load per tile).  Register blocks, row splitting and the fixed-order combination
// of partial sums are as in gram_tiled.   smem: 2 * 32 * 64 + 64 doubles (w tiles).
constexpr int GP_ROWS = 32;
constexpr int GRAM_PIPE_DOUBLES = 2 * GP_ROWS * PHIT_LD + 8 * GP_ROWS;

//   ev / outg (optional): the same pass also yields PHI' ev -- the IRLS gradient's data term -- column by column
//   (accumulated by the threads that own the diagonal blocks), saving a separate pass over PHI.
template <class Out, class OutG>
__device__ inline void gram_pipe(const double *__restrict__ phit, int N, int M, const double *__restrict__ w,
                                 double *sm, Out out, const double *__restrict__ ev, OutG outg)
{
    PHASE(PH_GRAM);
    const int T = blockDim.x;
    const int NC = M <= 32 ? 32 : 64, TR = M <= 32 ? 2 * GP_ROWS : GP_ROWS;   // narrow matrices: half the columns, twice the rows per tile (half the barriers)
    double *tiles = sm, *wt = sm + 2 * GP_ROWS * PHIT_LD, *et = wt + 4 * GP_ROWS;
    const int ntile = (N + TR - 1) / TR;
    const int nb = (M + 3) >> 2, nblk = nb * (nb + 1) / 2;
    const int nsplit = max(1, min(min(T, 256) / nblk, 8));
    const int blk = threadIdx.x % nblk, split = threadIdx.x / nblk;
    const bool active = threadIdx.x < nblk * nsplit;
    int bj = 0, bk = blk;
    { int rem = blk; while (rem >= nb - bj) { rem -= nb - bj; bj++; } bk = bj + rem; }
    const int rps = (TR + nsplit - 1) / nsplit;                 // rows of a tile per split
    const int cpr = NC / 2;                                     // 16-byte pieces per row
    auto stage = [&](int t) {
        if (t < ntile) {
            double *dst = tiles + (t & 1) * (GP_ROWS * PHIT_LD);
            const int h0 = t * TR;
            for (int idx = threadIdx.x; idx < TR * cpr; idx += T) {
                const int hl = idx / cpr, q = idx - hl * cpr;
                __pipeline_memcpy_async(dst + hl * NC + 2 * q, phit + (size_t)min(h0 + hl, N - 1) * PHIT_LD + 2 * q, 16);
            }
            if (threadIdx.x < TR) {                              // w and ev ride in the same cp.async group (zero past N):
                const int h = h0 + (int)threadIdx.x;              // a plain load here would stall these warps for an L2 round
                double *wd = wt + (t & 1) * 2 * GP_ROWS + threadIdx.x;    // trip per tile, and the next barrier waits for them
                if (w) __pipeline_memcpy_async(wd, w + min(h, N - 1), 8, h < N ? 0 : 8);
                else *wd = h < N ? 1.0 : 0.0;
                if (ev) __pipeline_memcpy_async(et + (t & 1) * 2 * GP_ROWS + threadIdx.x, ev + min(h, N - 1), 8, h < N ? 0 : 8);
            }
        }
        __pipeline_commit();
    };
    const bool grad = ev != nullptr && bj == bk;
    double ge[4] = {0.0, 0.0, 0.0, 0.0};
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
    __syncthreads();
    stage(0);
    for (int t = 0; t < ntile; t++) {
        __pipeline_wait_prior(0);
        __syncthreads();                                         // tile t visible; everyone finished tile t-1
        stage(t + 1);
        if (active) {
            const double *tile = tiles + (t & 1) * (GP_ROWS * PHIT_LD), *wv = wt + (t & 1) * 2 * GP_ROWS;
            const int hb = split * rps, he = min(hb + rps, TR);
#pragma unroll 2
            for (int hl = hb; hl < he; hl++) {
                const double4 a4 = *reinterpret_cast<const double4 *>(tile + hl * NC + 4 * bj);
                const double4 b4 = *reinterpret_cast<const double4 *>(tile + hl * NC + 4 * bk);
                const double ww = wv[hl];                        // rows past N carry weight 0
                const double av[4] = {a4.x * ww, a4.y * ww, a4.z * ww, a4.w * ww}, bv[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int a = 0; a < 4; a++)
#pragma unroll
                    for (int b = 0; b < 4; b++) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
                if (grad) {
                    const double eh = et[(t & 1) * 2 * GP_ROWS + hl];
                    ge[0] = fma(a4.x, eh, ge[0]); ge[1] = fma(a4.y, eh, ge[1]); ge[2] = fma(a4.z, eh, ge[2]); ge[3] = fma(a4.w, eh, ge[3]);
                }
            }
        }
    }
    __pipeline_wait_prior(0);
    __syncthreads();                                             // tiles are dead: reuse the buffer for the partial sums
    if (active) {
        double *dst = sm + ((size_t)split * nblk + blk) * 16;
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int b = 0; b < 4; b++) dst[a * 4 + b] = acc[a][b];
    }
    __syncthreads();
    for (int idx = threadIdx.x; idx < nblk * 16; idx += T) {
        const int b2 = idx >> 4, e = idx & 15, a = e >> 2, b = e & 3;
        double z = 0.0;
        for (int sp = 0; sp < nsplit; sp++) z += sm[((size_t)sp * nblk + b2) * 16 + e];
        int cj = 0, ck = b2;
        { int rem = b2; while (rem >= nb - cj) { rem -= nb - cj; cj++; } ck = cj + rem; }
        const int j = 4 * cj + a, k = 4 * ck + b;
        if (j < M && k < M && j <= k) out(j, k, z);
    }
    __syncthreads();
    if (ev) {                                                    // the gradient's partial sums, combined the same way
        if (active && grad) {
            double *dst = sm + ((size_t)split * nb + bj) * 4;
            dst[0] = ge[0]; dst[1] = ge[1]; dst[2] = ge[2]; dst[3] = ge[3];
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < nb * 4; idx += T) {
            double z = 0.0;
            for (int sp = 0; sp < nsplit; sp++) z += sm[((size_t)sp * nb + (idx >> 2)) * 4 + (idx & 3)];
            if (idx < M) outg(idx, z);
        }
        __syncthreads();
    }
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

__device__ inline double block_var(const double *t, int N, const Scratch &sc)
{   // varTargets (MainEff.c:1826-1838)
    double m = 0;
    for (int h = threadIdx.x; h < N; h += blockDim.x) m += t[h];
    m = block_sum(m, sc) / N;
    double v = 0;
    for (int h = threadIdx.x; h < N; h += blockDim.x) { double d = t[h] - m; v = fma(d, d, v); }
    return block_sum(v, sc) / (N - 1);
}

// (A v)[i] for a symmetric M x M matrix stored with leading dimension M: the thread walks COLUMN i (a warp's loads coalesce)
// in four interleaved chains, so that sixteen loads of the L2-resident matrix are in flight instead of four behind one
// dependent FMA chain; the chains are combined in a fixed order.
__device__ inline double sym_matvec_row(const double *__restrict__ A, int M, int i, const double *__restrict__ v)
{
    double z0 = 0, z1 = 0, z2 = 0, z3 = 0;
    int j = 0;
#pragma unroll 4
    for (; j + 4 <= M; j += 4) {
        z0 = fma(A[(size_t)j * M + i], v[j], z0);
        z1 = fma(A[(size_t)(j + 1) * M + i], v[j + 1], z1);
        z2 = fma(A[(size_t)(j + 2) * M + i], v[j + 2], z2);
        z3 = fma(A[(size_t)(j + 3) * M + i], v[j + 3], z3);
    }
    for (; j < M; j++) z0 = fma(A[(size_t)j * M + i], v[j], z0);
    return (z0 + z1) + (z2 + z3);
}

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
        const double so = s.S_out[c], qo = s.Q_out[c];
        double d_ml = 0; int act = ACT_NONE;
        const double a = so - qo * qo + 2 * l1 + l2;
        const double b = (so + l2) * (so + 4 * l1 + l2);
        const double gm = 2 * l1 * (so + l2) * (so + l2);
        const double dl = b * b - 4 * a * gm;
        if (a < 0 && dl > 0) {
            const double r = (-b - sqrt(dl)) / (2 * a);
            const double L = (log(r / (r + so + l2)) + qo * qo / (r + so + l2)) * 0.5 - l1 / r;
            if (L > 0) {
                s.aroot[c] = r + l2;
                if (i >= 0) {
                    act = ACT_REEST;
                    const double o = s.alpha[i] - l2;
                    d_ml = 0.5 * (log(r * (o + so + l2) / (o * (r + so + l2))) +
                                  qo * qo * (1 / (r + so + l2) - 1 / (o + so + l2))) -
                           l1 * (1 / r - 1 / o);
                } else {
                    act = ACT_ADD;
                    d_ml = L;
                    if (!EPIS && !BINOM) f_add = 1;   // only the Gaussian main-effect file ever sets anyToAdd (:1484)
                }
            }
        } else if (i >= 0 && M > 1) {
            f_del = 1;
            act = ACT_DEL;
            const double o = s.alpha[i] - l2;
            const double L = (log(o / (o + so + l2)) + qo * qo / (o + so + l2)) * 0.5 - l1 / o;
            d_ml = -L;
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
            const double var = block_var(s.t, N, sc);
            if (!EPIS) g.beta = 1 / (var * 0.01 + 1e-10);
            else { double sd = sqrt(var); if (sd < 1e-6) sd = 1e-6; g.beta = 1 / ((sd * 0.1) * (sd * 0.1)); }
            double p = 0, q = 0;
            for (int h = threadIdx.x; h < N; h += T) { p = fma(s.phi[h], s.phi[h], p); q = fma(s.phi[h], s.t[h], q); }
            block_sum2(p, q, sc);
            p *= g.beta; q *= g.beta;
            double a = p * p / (q * q - p);
            if (a < 0) a = v.init_alpha_max;
            if (a > v.init_alpha_max) a = v.init_alpha_max;
            if (threadIdx.x == 0) s.alpha[0] = a;
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
            int nu = d.nu, worthwhile;
            if (selected == ACT_TERM && !ini_removed && g.M > 1) nu = -1;          // :426-430
            if (nu == -1 && ini_removed) { worthwhile = 0; selected = ACT_TERM; }
            else if (nu == -1 && !ini_removed && g.M > 1) {                        // :437-446
                worthwhile = 1; nu = initial - 1;
                __syncthreads();
                if (threadIdx.x == 0) { s.action[nu] = ACT_DEL; s.block[0] = nu; }
                __syncthreads();
                n_update = 1; ini_removed = 1; selected = ACT_DEL;
            } else {
                worthwhile = 1;
                const int best_is_add = s.action[nu] == ACT_ADD;
                double cutoff = d.best * (best_is_add ? v.n_add : 1.0);
                if (cutoff < v.ml_delta) cutoff = v.ml_delta;
                const int best_is_del = s.action[nu] == ACT_DEL;
                n_update = block_compact(Kc, [&](int c) { return s.dml[c] >= cutoff; }, s.block, nullptr, 0, sc);
                if (best_is_del && n_update > 1) n_update = 1;                     // :474
                if (n_update == 0) worthwhile = 0;
            }
            if (!worthwhile) selected = ACT_TERM;
            if (worthwhile) {
                for (int iu = 0; iu < n_update; iu++) {
                    __syncthreads();
                    nu = s.block[iu];
                    selected = s.action[nu];
                    const double new_alpha = s.aroot[nu];
                    if (selected == ACT_REEST || selected == ACT_DEL) {
                        // The reference searches Used for nu and silently keeps the previous jj when the
                        // search fails (forced removal of an initial basis that a regular delete already
                        // took out, :498-509).  Keep that, but never index outside the active set.
                        const int a = s.amap[nu];
                        if (a >= 0) jj = a;
                        if (jj < 0 || jj >= g.M) { g.status |= ST_NOT_PD; selected = ACT_TERM; }
                    }
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
                        for (int i = threadIdx.x; i < M; i += T) s.mu[i] += -mujj * kappa * sj[i];
                        {   // (restrict: the two SIGMA buffers never alias, so the loads of an unrolled row run ahead of its stores)
                            const double *__restrict__ sg = s.sigma; double *__restrict__ sn = s.sigma_new;
                            for (int j = wid_; j < M; j += nw_) {                // warps own columns, lanes rows: no integer division
                                const double kj = sg[jj * M + j];
#pragma unroll 4
                                for (int i = lane_; i < M; i += 32) {
                                    const int idx = j * M + i;
                                    sn[idx] = sg[idx] - kappa * sg[jj * M + i] * kj;
                                }
                            }
                        }
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
                            for (int i = threadIdx.x; i < M; i += T) s.mu[i] += -mu_i * s.u[i];
                            if (threadIdx.x == 0) s.mu[M] = mu_i;
                            const int M1 = M + 1;
                            {
                                const double *__restrict__ sg = s.sigma; double *__restrict__ sn = s.sigma_new;
                                const double *__restrict__ uu = s.u;
                                for (int j = wid_; j < M1; j += nw_) {
                                    const double uj = uu[min(j, M - 1)];
#pragma unroll 4
                                    for (int i = lane_; i < M1; i += 32) {
                                        double val;
                                        if (i < M && j < M) val = sg[j * M + i] + (s_ii * uu[i]) * uj;
                                        else if (i == M && j == M) val = s_ii;
                                        else val = -s_ii * uu[i < M ? i : j];
                                        sn[j * M1 + i] = val;
                                    }
                                }
                            }
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
                        for (int i = threadIdx.x; i < M; i += T) {
                            double m = s.mu[i] - mujj * sj[i] / sjj;
                            s.mu[i] = m;
                        }
                        for (int h = threadIdx.x; h < N; h += T) s.phi[(size_t)jj * LD + h] = s.phi[(size_t)lastj * LD + h];
                        if (jj != lastj) {                                         // PHI'PHI: last row/column into slot jj
                            for (int i = threadIdx.x; i < lastj; i += T) {
                                if (i == jj) s.ptp[(size_t)jj * cap + jj] = s.ptp[(size_t)lastj * cap + lastj];
                                else { s.ptp[(size_t)i * cap + jj] = s.ptp[(size_t)i * cap + lastj]; s.ptp[(size_t)jj * cap + i] = s.ptp[(size_t)lastj * cap + i]; }
                            }
                        }
                        // Schur downdate, then move the last row/column into slot jj (:1754-1776)
                        for (int i = threadIdx.x; i < M; i += T) s.colk[i] = sj[i] / sjj;      // one division per row, not per entry
                        __syncthreads();
                        {
                            const double *__restrict__ sg = s.sigma; double *__restrict__ sn = s.sigma_new;
                            const double *__restrict__ ck = s.colk;
                            for (int j = wid_; j < lastj; j += nw_) {
                                const int sjx = (j == jj) ? lastj : j;
                                const double sjv = sg[jj * M + sjx];
#pragma unroll 4
                                for (int i = lane_; i < lastj; i += 32) {
                                    const int si = (i == jj) ? lastj : i;
                                    sn[j * lastj + i] = sg[sjx * M + si] - ck[si] * sjv;
                                }
                            }
                        }
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
    __syncthreads();
    for (int i = threadIdx.x; i < M; i += T) s.tmp[i] = s.mu[i] / scale[s.used[i] - 1];   // Beta[,3] (:221)
    __syncthreads();
    double sse = 0;
    for (int h = threadIdx.x; h < F.nte; h += T) {
        const double *xr = F.Xte + (size_t)h * K;
        double pred = 0;
        for (int i = 0; i < M; i++) {
            const double w = s.tmp[i];
            if (w != 0) { Cand<EPIS> cd(s.used[i] - 1, K); pred = fma(cd.at(xr), w, pred); }
        }
        const double r = F.yte[h] - (b + pred);
        sse = fma(r, r, sse);
    }
    sse = block_sum(sse, sc);
    int nsel = 0;
    for (int i = 0; i < M; i++) nsel += s.tmp[i] != 0;
    if (!isfinite(sse)) g.status |= ST_NONFINITE;
    if (threadIdx.x == 0) {
        const int o = task.out_index;
        if (out.fold_err) out.fold_err[o] = sse;
        if (out.status) out.status[o] = g.status;
        if (out.n_selected) out.n_selected[o] = nsel;
        if (out.n_iter) out.n_iter[o] = iter;
        if (out.flops) { atomicAdd(out.flops, g.flops); if (g.avoided > 0) atomicAdd(out.flops + 1, g.avoided); }
        if (out.m_out) {          // full-model record of fit o (pareben_fit_batch)
            out.m_out[o] = M;
            double wd = 0;        // Wald score mu'H mu with H read at leading dimension M (:206-215)
            for (int i = 0; i < M; i++) {
                double z = 0;
                for (int j = 0; j < M; j++) z += s.mu[j] * s.H[i * M + j];
                wd += z * s.mu[i];
            }
            const size_t r = (size_t)o * out.dump_ld;
            for (int i = 0; i < M; i++) {
                const int c = s.used[i] - 1;
                out.used_out[r + i] = s.used[i];
                out.beta_out[r + i] = s.mu[i] / scale[c];
                out.var_out[r + i] = s.sigma[i * M + i] / (scale[c] * scale[c]);
            }
            out.scalars_out[4 * (size_t)o + 0] = wd; out.scalars_out[4 * (size_t)o + 1] = b;
            out.scalars_out[4 * (size_t)o + 2] = 0;
            out.scalars_out[4 * (size_t)o + 3] = 1 / (g.beta + 1e-10);
        }
    }
    __syncthreads();
}

}  // namespace pareben
