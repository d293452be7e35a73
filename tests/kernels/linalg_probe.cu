// linalg_probe.cu -- test-only entry points into the dense linear algebra of a fit (linalg.cuh, contract.cuh), built by
// tests/test_gpu_linalg_kernels.py into its own shared library (libpareben.so gains nothing).
//
// Each entry copies host arrays into guarded device buffers (probe_call.cuh), runs ONE block with the fit kernels'
// resources (launch bounds, FIT_T threads, S_BUF_BYTES of dynamic shared memory, s_buf as the sweep / Gram / quadratic-form
// scratch, as eben_fit_kernel passes it) on a private stream, copies the results back and frees every device buffer before
// it returns, on success and on failure alike.  The emit and out callbacks count their calls with atomicAdd, so a test can
// check that every candidate and every pair j <= k is emitted exactly once.
//
//   probe_sweep       spd_inverse_sweep(a, M, colk, sc, s_buf): a (M x M) in place, ok as every thread returned it
//   probe_quad        quad_forms: quad[c] = g_c' SIGMA g_c, lin[c] = g_c' v, G read through the physical row map grow
//   probe_gram        gram_pipe (row-major PHIt, with the gradient PHI'ev) or gram_mma (column-major PHI)
//   probe_cache_dot   cache_dot: z[c] = sum_j G[grow[j]][c] vec[j]
//   probe_sym_matvec  sym_matvec_row for every row i < M
//   probe_constant    the dispatch constants the kernels choose their paths by
//
// Return value: 0, -1 for arguments the kernel does not accept, -2 when a kernel wrote into a guard region
// (probe_last_error says which), or a positive cudaError_t.
#include "../../pareben_b200/csrc/common.cuh"
#include "../../pareben_b200/csrc/contract.cuh"
#include "../../pareben_b200/csrc/linalg.cuh"
#include "../../pareben_b200/csrc/fit_kernel.cuh"
#include "probe_call.cuh"

#include <cstring>
#include <vector>

using namespace pareben;
using probe::bad;
using probe::Call;

namespace {

#define PROBE_KERNEL __global__ void __launch_bounds__(FIT_THREADS, PAREBEN_MIN_BLOCKS)

PROBE_KERNEL probe_sweep_kernel(double *a, int M, double *colk, int *ok)
{
    extern __shared__ __align__(32) double s_buf[];
    __shared__ double red[66];
    __shared__ int redi[66];
    Scratch sc{red, redi, s_buf, nullptr};
    const bool r = spd_inverse_sweep(a, M, colk, sc, sc.sweep);
    ok[threadIdx.x] = r ? 1 : 0;
}

PROBE_KERNEL probe_quad_kernel(double *G, int *grow, int M, int Kc, const double *sigma, double *sigp, const double *v,
                               double *quad, double *lin, int *cnt)
{
    extern __shared__ __align__(32) double s_buf[];
    Slab s{};
    s.G = G; s.grow = grow;
    quad_forms(s, sigma, sigp, M, Kc, v, s_buf, [&](int c, double q, double l) {
        quad[c] = q; lin[c] = l; atomicAdd(cnt + c, 1);
    });
}

PROBE_KERNEL probe_gram_pipe_kernel(const double *phit, int N, int M, const double *w, const double *ev, double *H, int *cntH,
                                    double *g, int *cntg)
{
    extern __shared__ __align__(32) double s_buf[];
    gram_pipe(phit, N, M, w, s_buf, [&](int j, int k, double z) { H[(size_t)j * M + k] = z; atomicAdd(cntH + (size_t)j * M + k, 1); },
              ev, [&](int j, double z) { g[j] = z; atomicAdd(cntg + j, 1); });
}

PROBE_KERNEL probe_gram_mma_kernel(const double *phi, int N, int LD, int M, const double *w, double *H, int *cntH)
{
    extern __shared__ __align__(32) double s_buf[];
    gram_mma(phi, N, LD, M, w, s_buf, [&](int j, int k, double z) { H[(size_t)j * M + k] = z; atomicAdd(cntH + (size_t)j * M + k, 1); });
}

PROBE_KERNEL probe_cache_dot_kernel(double *G, int *grow, int M, int Kc, const double *vec, double *out, int *cnt)
{
    Slab s{};
    s.G = G; s.grow = grow;
    cache_dot(s, M, Kc, vec, [&](int c, double z) { out[c] = z; atomicAdd(cnt + c, 1); });
}

PROBE_KERNEL probe_sym_matvec_kernel(const double *A, int M, const double *v, double *out)
{
    for (int i = threadIdx.x; i < M; i += blockDim.x) out[i] = sym_matvec_row(A, M, i, v);
}

template <class Kern, class... Args>
void launch(Call &cl, Kern kern, Args... args)
{
    if (cl.err) return;
    if (!cl.note(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S_BUF_BYTES))) return;
    kern<<<1, FIT_T, S_BUF_BYTES, cl.stream>>>(args...);
    cl.note(cudaGetLastError());
}

// the candidate cache as a fit stores it: nphys physical rows of Kc, logical row j at physical row grow[j]
bool valid_rows(int M, int nphys, const int *grow)
{
    std::vector<char> seen(nphys, 0);
    for (int j = 0; j < M; j++) {
        if (grow[j] < 0 || grow[j] >= nphys || seen[grow[j]]) return false;
        seen[grow[j]] = 1;
    }
    return true;
}

}  // namespace

extern "C" const char *probe_last_error(void) { return probe::last_error().c_str(); }

extern "C" int probe_device_count(void)
{
    int n = 0;
    return cudaGetDeviceCount(&n) == cudaSuccess ? n : 0;
}

// the constants the dispatch of these kernels depends on (-1 for an unknown name)
extern "C" long long probe_constant(const char *name)
{
    struct { const char *n; long long v; } tab[] = {
        {"SWEEP_SMEM_M", SWEEP_SMEM_M}, {"SWEEP_PANEL_DOUBLES", SWEEP_PANEL_DOUBLES}, {"QUAD_SIMT_M", QUAD_SIMT_M},
        {"QT", QT}, {"PHIT_LD", PHIT_LD}, {"FIT_T", FIT_T}, {"NT_MAX", NT_MAX}, {"MT", MT},
        {"S_BUF_BYTES", (long long)S_BUF_BYTES}, {"GP_ROWS", GP_ROWS},
    };
    for (const auto &e : tab)
        if (!std::strcmp(e.n, name)) return e.v;
    return -1;
}

// a: M x M (column-major, leading dimension M), overwritten as the kernel leaves it.  ok: FIT_T flags.
// colk holds 2 (M + 1) doubles, as in a slab with cap = M.
extern "C" int probe_sweep(int M, double *a, int *ok)
{
    if (M < 1 || !a || !ok) return bad("probe_sweep: bad argument");
    Call cl;
    double *d_a = cl.upload_guarded(a, (size_t)M * M, "a");
    double *d_colk = cl.guarded<double>(2 * ((size_t)M + 1), "colk");
    int *d_ok = cl.guarded<int>(FIT_T, "ok");
    launch(cl, probe_sweep_kernel, d_a, M, d_colk, d_ok);
    cl.download(a, d_a, (size_t)M * M);
    cl.download(ok, d_ok, FIT_T);
    return cl.finish();
}

// Gphys: nphys x Kc physical rows (logical row j at grow[j]); sigma: M x M; v: M, or null.  The spare SIGMA buffer holds
// sig_elems(M) doubles, as in a slab with cap = M.  Out: quad, lin [Kc], cnt [Kc] = emit calls per candidate.
extern "C" int probe_quad(int M, int Kc, int nphys, const int *grow, const double *Gphys, const double *sigma, const double *v,
                          double *quad, double *lin, int *cnt)
{
    if (M < 1 || Kc < 1 || nphys < M || !grow || !Gphys || !sigma || !quad || !lin || !cnt || !valid_rows(M, nphys, grow))
        return bad("probe_quad: bad argument");
    Call cl;
    double *d_G = cl.upload_guarded(Gphys, (size_t)nphys * Kc, "G");
    int *d_grow = cl.upload_guarded(grow, M, "grow");
    const double *d_sigma = cl.upload_guarded(sigma, (size_t)M * M, "sigma");
    double *d_sigp = cl.guarded<double>(sig_elems(M), "spare sigma");
    const double *d_v = v ? cl.upload_guarded(v, M, "v") : nullptr;
    double *d_q = cl.guarded<double>(Kc, "quad"), *d_l = cl.guarded<double>(Kc, "lin");
    int *d_cnt = cl.guarded<int>(Kc, "emit count", 0);
    launch(cl, probe_quad_kernel, d_G, d_grow, M, Kc, d_sigma, d_sigp, d_v, d_q, d_l, d_cnt);
    cl.download(quad, d_q, Kc);
    cl.download(lin, d_l, Kc);
    cl.download(cnt, d_cnt, Kc);
    return cl.finish();
}

// phi: M x N (column j = active column j, N rows); w: N or null (all ones); ev: N or null (gram_pipe only).
// use_mma = 0: gram_pipe from the row-major copy PHIt, (N + 32) rows of PHIT_LD (columns >= M zero, rows >= N never read:
// NaN); 1: gram_mma from the column-major PHI, leading dimension phi_ld(N), pad rows zero.
// Out: H [M][M] at j*M + k for j <= k, cntH [M][M] = out calls per entry, g [M] and cntg [M] (ev only).
extern "C" int probe_gram(int use_mma, int N, int M, const double *phi, const double *w, const double *ev, double *H, int *cntH,
                          double *g, int *cntg)
{
    if (N < 1 || M < 1 || !phi || !H || !cntH || (ev && (use_mma || !g || !cntg))) return bad("probe_gram: bad argument");
    if (!use_mma && (M > PHIT_LD || FIT_T != 256)) return bad("probe_gram: gram_pipe takes at most PHIT_LD columns and 256 threads");
    Call cl;
    const double *d_w = w ? cl.upload_guarded(w, N, "w") : nullptr;
    double *d_H = cl.guarded<double>((size_t)M * M, "H");
    int *d_cH = cl.guarded<int>((size_t)M * M, "out count", 0);
    if (!use_mma) {
        const size_t rows = (size_t)N + 32;
        std::vector<double> pt(rows * PHIT_LD, 0.0);
        for (size_t h = N; h < rows; h++)
            for (int j = 0; j < PHIT_LD; j++) pt[h * PHIT_LD + j] = NAN;
        for (int j = 0; j < M; j++)
            for (int h = 0; h < N; h++) pt[(size_t)h * PHIT_LD + j] = phi[(size_t)j * N + h];
        const double *d_pt = cl.upload_guarded(pt.data(), pt.size(), "phit");
        const double *d_ev = ev ? cl.upload_guarded(ev, N, "ev") : nullptr;
        double *d_g = cl.guarded<double>(M, "g");
        int *d_cg = cl.guarded<int>(M, "outg count", 0);
        launch(cl, probe_gram_pipe_kernel, d_pt, N, M, d_w, d_ev, d_H, d_cH, d_g, d_cg);
        if (ev) { cl.download(g, d_g, M); cl.download(cntg, d_cg, M); }
    } else {
        const int LD = phi_ld(N);
        std::vector<double> pc((size_t)LD * M, 0.0);
        for (int j = 0; j < M; j++) std::memcpy(pc.data() + (size_t)j * LD, phi + (size_t)j * N, sizeof(double) * N);
        const double *d_pc = cl.upload_guarded(pc.data(), pc.size(), "phi");
        launch(cl, probe_gram_mma_kernel, d_pc, N, LD, M, d_w, d_H, d_cH);
    }
    cl.download(H, d_H, (size_t)M * M);
    cl.download(cntH, d_cH, (size_t)M * M);
    return cl.finish();
}

// Gphys, grow as in probe_quad; vec: M.  Out: z [Kc], cnt [Kc].
extern "C" int probe_cache_dot(int M, int Kc, int nphys, const int *grow, const double *Gphys, const double *vec, double *z, int *cnt)
{
    if (M < 1 || Kc < 1 || nphys < M || !grow || !Gphys || !vec || !z || !cnt || !valid_rows(M, nphys, grow))
        return bad("probe_cache_dot: bad argument");
    Call cl;
    double *d_G = cl.upload_guarded(Gphys, (size_t)nphys * Kc, "G");
    int *d_grow = cl.upload_guarded(grow, M, "grow");
    const double *d_vec = cl.upload_guarded(vec, M, "vec");
    double *d_z = cl.guarded<double>(Kc, "z");
    int *d_cnt = cl.guarded<int>(Kc, "emit count", 0);
    launch(cl, probe_cache_dot_kernel, d_G, d_grow, M, Kc, d_vec, d_z, d_cnt);
    cl.download(z, d_z, Kc);
    cl.download(cnt, d_cnt, Kc);
    return cl.finish();
}

// A: M x M (leading dimension M); v: M.  Out: z [M], z[i] = sym_matvec_row(A, M, i, v).
extern "C" int probe_sym_matvec(int M, const double *A, const double *v, double *z)
{
    if (M < 1 || !A || !v || !z) return bad("probe_sym_matvec: bad argument");
    Call cl;
    const double *d_A = cl.upload_guarded(A, (size_t)M * M, "A");
    const double *d_v = cl.upload_guarded(v, M, "v");
    double *d_z = cl.guarded<double>(M, "z");
    launch(cl, probe_sym_matvec_kernel, d_A, M, d_v, d_z);
    cl.download(z, d_z, M);
    return cl.finish();
}
