// contract.cuh -- the candidate contractions every EBEN solver runs: X' V against the training matrix (DMMA,
// SIMT and warp-per-candidate forms), the quadratic forms of the candidate cache against SIGMA, and cache_dot.
#pragma once
#include "common.cuh"
#include <cuda_pipeline.h>

namespace pareben {

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
// cp.async (the SIGMA tiles of the DMMA quadratic forms).
__device__ inline void stage_tile(double *dst, int ldd, const double *__restrict__ V, int ldv, int h0, int r0, int ncol)
{
    const int ch = ncol >> 1;                  // 16-byte chunks per row
    for (int idx = threadIdx.x; idx < QT * ch; idx += blockDim.x) {
        const int h = idx / ch, q = idx - h * ch;
        __pipeline_memcpy_async(dst + h * ldd + 2 * q, V + (size_t)(h0 + h) * ldv + r0 + 2 * q, 16);
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
        if (st < nstage) {
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
            __syncthreads();                                   // ... and for everyone's; stage st-1 is fully consumed
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
    if (!resident) stage_tile(sV, LDS_V, sigp, ldp, 0, p0, 8 * NT);
    if (live) { fetch(xv, 0); fetch(xn, 16); }
    if (!resident) { __pipeline_wait_prior(0); __syncthreads(); }
    for (int st = 0; st < nstage; st++) {
        const double *buf = sV + (st & 1) * (QT * LDS_V);
        if (!resident && st + 1 < nstage) stage_tile(sV + ((st + 1) & 1) * (QT * LDS_V), LDS_V, sigp, ldp, (st + 1) * QT, p0, 8 * NT);
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

}  // namespace pareben
