// linalg.cuh -- the dense linear algebra of the EBEN solvers on the active set: the SPD inverse by the symmetric
// sweep, the Gram matrices PHI'B PHI, the symmetric matrix-vector product and the block variance.
#pragma once
#include "common.cuh"
#include "contract.cuh"

namespace pareben {

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
// overlaps the FMAs of tile t and there is one barrier per tile.  Threads own 4 x 4 register blocks
// of the upper triangle, rows are split among the threads left over, and the partial sums are
// combined in a fixed order.   smem: 2 * 32 * 64 + 64 doubles (w tiles).
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

}  // namespace pareben
