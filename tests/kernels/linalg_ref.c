/* linalg_ref.c -- bit-exact C restatements of the dense linear algebra kernels of gauss_fit.cuh whose arithmetic is plain
 * IEEE double in a fixed order.  Built by the tests with gcc -O2 -std=c11 -ffp-contract=off (no contraction: every
 * multiply and add rounds where the kernel's do, and fma() from libm is the correctly rounded fused operation the kernels'
 * fma() is; the library is compiled with -fmad=false for the same reason).
 *
 *   ref_sweep_regs    sweep_regs<1/2> and the sign flip of its write-back: v = fma(ci*cj, -1/d, r), pivot by pivot
 *   ref_sweep_core    sweep_core, then spd_inverse_sweep's negation: v = col[i] - (cur[i]*cj)*dinv, unfused
 *   ref_quad_simt     quad_forms_simt<8>: the doubled lower triangle read at sigma[p*M + j], 8-column chunks cut at jend
 *   ref_gram_pipe     gram_pipe: 4 x 4 register blocks, row splits, per-split FMA order, fixed-order combination, gradient
 *   ref_cache_dot     cache_dot: one FMA chain per candidate, cache rows ascending
 *   ref_sym_matvec    sym_matvec_row: four interleaved chains, combined as (z0 + z1) + (z2 + z3)
 *
 * Matrices are column-major with leading dimension M (element (i, j) at [j*M + i]) unless stated otherwise; the candidate
 * cache G is passed by logical row (row j of Kc at G + j*Kc), since the physical row map changes no arithmetic.
 * The sweeps return 1, or 0 as soon as a pivot is not positive (a is then left partly swept).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

int ref_sweep_regs(double *a, int M)
{
    double *cur = malloc(sizeof(double) * M);
    int ok = 1;
    for (int k = 0; k < M && ok; k++) {
        for (int i = 0; i < M; i++) cur[i] = a[(size_t)k * M + i];          /* column k before pivot k */
        const double d = cur[k];
        if (!(d > 0.0)) { ok = 0; break; }
        const double dinv = 1.0 / d, ndinv = -dinv;
        for (int j = 0; j < M; j++) {
            const double cj = cur[j];
            for (int i = 0; i < M; i++) {
                const double ci = cur[i];
                double v;
                if (i == k && j == k) v = ndinv;
                else if (i == k) v = cj * dinv;
                else if (j == k) v = ci * dinv;
                else v = fma(ci * cj, ndinv, a[(size_t)j * M + i]);
                a[(size_t)j * M + i] = v;
            }
        }
    }
    if (ok)
        for (size_t idx = 0; idx < (size_t)M * M; idx++) a[idx] = -a[idx];
    free(cur);
    return ok;
}

int ref_sweep_core(double *a, int M)
{
    double *cur = malloc(sizeof(double) * M);
    int ok = 1;
    for (int k = 0; k < M && ok; k++) {
        for (int i = 0; i < M; i++) cur[i] = a[(size_t)k * M + i];
        const double d = cur[k];
        if (!(d > 0.0)) { ok = 0; break; }
        const double dinv = 1.0 / d;
        for (int j = 0; j < M; j++) {
            const double cj = cur[j];
            for (int i = 0; i < M; i++) {
                double v;
                if (i == k && j == k) v = -dinv;
                else if (i == k) v = cj * dinv;
                else if (j == k) v = cur[i] * dinv;
                else v = a[(size_t)j * M + i] - (cur[i] * cj) * dinv;
                a[(size_t)j * M + i] = v;
            }
        }
    }
    if (ok)
        for (size_t idx = 0; idx < (size_t)M * M; idx++) a[idx] = -a[idx];
    free(cur);
    return ok;
}

/* v may be null (lin is then 0) */
void ref_quad_simt(int M, int Kc, const double *G, const double *sigma, const double *v, double *quad, double *lin)
{
    enum { PW = 8 };
    const int ldp = (M + PW - 1) / PW * PW;
    double *sigp = malloc(sizeof(double) * (size_t)M * ldp);
    for (int j = 0; j < M; j++)
        for (int p = 0; p < ldp; p++)
            sigp[(size_t)j * ldp + p] = (p < M && j <= p) ? (j < p ? 2.0 * sigma[(size_t)p * M + j] : sigma[(size_t)p * M + j]) : 0.0;
    for (int c = 0; c < Kc; c++) {
        double q = 0, l = 0;
        for (int p0 = 0; p0 < M; p0 += PW) {
            double z[PW] = {0};
            const int jend = M < p0 + PW ? M : p0 + PW;
            for (int j = 0; j < jend; j++) {
                const double g = G[(size_t)j * Kc + c];
                for (int t = 0; t < PW; t++) z[t] = fma(g, sigp[(size_t)j * ldp + p0 + t], z[t]);
            }
            for (int t = 0; t < PW; t++)
                if (p0 + t < M) {
                    const double gp = G[(size_t)(p0 + t) * Kc + c];
                    q = fma(z[t], gp, q);
                    if (v) l = fma(gp, v[p0 + t], l);
                }
        }
        quad[c] = q; lin[c] = l;
    }
    free(sigp);
}

/* phi: M x N (column j contiguous), w: N or null (ones), ev: N or null.  T: threads of the block.
 * Out: H[j*M + k] for j <= k (other entries untouched), g[j] = (PHI'ev)_j when ev is given. */
void ref_gram_pipe(int N, int M, const double *phi, const double *w, const double *ev, int T, double *H, double *g)
{
    enum { GP_ROWS = 32 };
    const int TR = M <= 32 ? 2 * GP_ROWS : GP_ROWS;
    const int ntile = (N + TR - 1) / TR;
    const int nb = (M + 3) >> 2, nblk = nb * (nb + 1) / 2;
    int nsplit = (T < 256 ? T : 256) / nblk;
    if (nsplit > 8) nsplit = 8;
    if (nsplit < 1) nsplit = 1;
    const int rps = (TR + nsplit - 1) / nsplit;
    double *part = calloc((size_t)nsplit * nblk * 16, sizeof(double));
    double *gpart = calloc((size_t)nsplit * nb * 4, sizeof(double));
    /* column c of row h as the staged tile holds it: rows past N are row N - 1 (weight 0), columns past M zero */
    #define X(h, c) ((c) < M ? phi[(size_t)(c) * N + ((h) < N ? (h) : N - 1)] : 0.0)
    for (int blk = 0; blk < nblk; blk++) {
        int bj = 0, bk = blk;
        { int rem = blk; while (rem >= nb - bj) { rem -= nb - bj; bj++; } bk = bj + rem; }
        for (int sp = 0; sp < nsplit; sp++) {
            double acc[4][4] = {{0}}, ge[4] = {0};
            for (int t = 0; t < ntile; t++) {
                const int hb = sp * rps, he = hb + rps < TR ? hb + rps : TR;
                for (int hl = hb; hl < he; hl++) {
                    const int h = t * TR + hl;
                    const double ww = h < N ? (w ? w[h] : 1.0) : 0.0;
                    double av[4], bv[4], ax[4];
                    for (int a = 0; a < 4; a++) { ax[a] = X(h, 4 * bj + a); av[a] = ax[a] * ww; bv[a] = X(h, 4 * bk + a); }
                    for (int a = 0; a < 4; a++)
                        for (int b = 0; b < 4; b++) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
                    if (ev && bj == bk) {
                        const double eh = h < N ? ev[h] : 0.0;
                        for (int a = 0; a < 4; a++) ge[a] = fma(ax[a], eh, ge[a]);
                    }
                }
            }
            memcpy(part + ((size_t)sp * nblk + blk) * 16, acc, sizeof(acc));
            if (bj == bk) memcpy(gpart + ((size_t)sp * nb + bj) * 4, ge, sizeof(ge));
        }
    }
    #undef X
    for (int blk = 0; blk < nblk; blk++) {
        int cj = 0, ck = blk;
        { int rem = blk; while (rem >= nb - cj) { rem -= nb - cj; cj++; } ck = cj + rem; }
        for (int e = 0; e < 16; e++) {
            double z = 0.0;
            for (int sp = 0; sp < nsplit; sp++) z += part[((size_t)sp * nblk + blk) * 16 + e];
            const int j = 4 * cj + (e >> 2), k = 4 * ck + (e & 3);
            if (j < M && k < M && j <= k) H[(size_t)j * M + k] = z;
        }
    }
    if (ev)
        for (int idx = 0; idx < nb * 4 && idx < M; idx++) {
            double z = 0.0;
            for (int sp = 0; sp < nsplit; sp++) z += gpart[((size_t)sp * nb + (idx >> 2)) * 4 + (idx & 3)];
            g[idx] = z;
        }
    free(part);
    free(gpart);
}

void ref_cache_dot(int M, int Kc, const double *G, const double *vec, double *z)
{
    for (int c = 0; c < Kc; c++) {
        double s = 0;
        for (int j = 0; j < M; j++) s = fma(G[(size_t)j * Kc + c], vec[j], s);
        z[c] = s;
    }
}

void ref_sym_matvec(int M, const double *A, const double *v, double *z)
{
    for (int i = 0; i < M; i++) {
        double z0 = 0, z1 = 0, z2 = 0, z3 = 0;
        int j = 0;
        for (; j + 4 <= M; j += 4) {
            z0 = fma(A[(size_t)j * M + i], v[j], z0);
            z1 = fma(A[(size_t)(j + 1) * M + i], v[j + 1], z1);
            z2 = fma(A[(size_t)(j + 2) * M + i], v[j + 2], z2);
            z3 = fma(A[(size_t)(j + 3) * M + i], v[j + 3], z3);
        }
        for (; j < M; j++) z0 = fma(A[(size_t)j * M + i], v[j], z0);
        z[i] = (z0 + z1) + (z2 + z3);
    }
}
