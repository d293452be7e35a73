// contract_probe.cu -- test-only entry points into the two score contractions, built by
// tests/test_gpu_contract_kernels.py into its own shared library (libpareben.so gains nothing).
//
// Each entry takes host arrays, lays the training matrix out with the library's own layout kernels (layout.cuh) exactly
// as pareben_problem_create does, runs ONE block with the fit kernels' resources (launch bounds, FIT_T threads, S_BUF_BYTES
// of dynamic shared memory) on a private stream, copies the results back and frees every device buffer before it returns, on
// success and on failure alike.  The tensor-core kernel allocates its tensor memory with tc_open and gives it back with
// tc_close before it exits.
//
//   probe_tc          tc_contract (tc_contract.cuh): G[j][c] = x_c'(w o phi_j) / s_c for j < R, ze = X'e, bb = (X o X)'(w o phi_0)
//   probe_contract_x  contract_x (gauss_fit.cuh), the form chosen as a fit chooses it: by R, ldt and whether bb is wanted
//   probe_cand_map    Cand<true>: candidate index -> loci (i, j) of the Epis numbering
//
// Return value: 0, a negative number for arguments the contraction does not accept (probe_last_error says which), or a
// positive cudaError_t.
#include "../../pareben_b200/csrc/common.cuh"
#include "../../pareben_b200/csrc/gauss_fit.cuh"
#include "../../pareben_b200/csrc/tc_contract.cuh"
#include "../../pareben_b200/csrc/layout.cuh"
#include "../../pareben_b200/csrc/fit_kernel.cuh"

#include <cmath>
#include <string>
#include <vector>

using namespace pareben;

namespace {

std::string g_err;

// device buffers and the stream of one call, released in the destructor whatever path the call leaves by
struct Call {
    cudaStream_t stream = nullptr;
    std::vector<void *> bufs;
    cudaError_t err = cudaSuccess;
    Call() { note(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)); }
    ~Call()
    {
        if (stream) cudaStreamSynchronize(stream);
        for (void *p : bufs) cudaFree(p);
        if (stream) cudaStreamDestroy(stream);
    }
    bool note(cudaError_t e)
    {
        if (e != cudaSuccess && err == cudaSuccess) { err = e; g_err = cudaGetErrorString(e); }
        return err == cudaSuccess;
    }
    template <class T>
    T *alloc(size_t n)
    {
        void *p = nullptr;
        if (!note(cudaMalloc(&p, n * sizeof(T) + 16))) return nullptr;
        bufs.push_back(p);
        note(cudaMemsetAsync(p, 0, n * sizeof(T) + 16, stream));
        return static_cast<T *>(p);
    }
    template <class T>
    T *upload(const T *h, size_t n)
    {
        T *d = alloc<T>(n);
        if (d && h && n) note(cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, stream));
        return d;
    }
    template <class T>
    void download(T *h, const T *d, size_t n)
    {
        if (h && d && n && err == cudaSuccess) note(cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, stream));
    }
    int finish()
    {
        if (err == cudaSuccess) note(cudaGetLastError());
        if (err == cudaSuccess) note(cudaStreamSynchronize(stream));
        return (int)err;
    }
};

int bad(const char *msg) { g_err = msg; return -1; }

// the design as pareben_problem_create sees it: every entry an integer in [-127, 127], and the largest magnitude
bool small_int_design(const double *X, size_t n, double &max_abs)
{
    bool small_int = true;
    max_abs = 0;
    for (size_t i = 0; small_int && i < n; i++) {
        const double v = X[i];
        if (!(v >= -127.0 && v <= 127.0) || v != (double)(int)v) small_int = false;
        max_abs = std::max(max_abs, std::fabs(v));
    }
    return small_int;
}

// The training-side fields of a FoldData, built with the layout kernels and launch shapes of pareben_problem_create.
FoldData layout_fold(Call &cl, const double *X, int N, int K, int Kc, bool epis, bool int8, bool tc)
{
    FoldData F{};
    const double *Xtr = cl.upload(X, (size_t)N * K);
    double *scale = cl.alloc<double>(Kc);
    if (!cl.err) {
        if (epis) scales_kernel<true><<<(Kc + 255) / 256, 256, 0, cl.stream>>>(Xtr, N, K, Kc, scale);
        else scales_kernel<false><<<(Kc + 255) / 256, 256, 0, cl.stream>>>(Xtr, N, K, Kc, scale);
    }
    F.Xtr = Xtr; F.scale = scale; F.ntr = N;
    F.ldt = (N + 63) & ~63;
    const dim3 blk(32, 8), tg((F.ldt + 31) / 32, (K + 31) / 32);
    if (int8) {
        int8_t *t8 = cl.alloc<int8_t>((size_t)F.ldt * K + 16);
        int8_t *x8 = cl.alloc<int8_t>((size_t)N * K + 16);
        if (!cl.err) {
            transpose_pad_kernel<int8_t><<<tg, blk, 0, cl.stream>>>(Xtr, N, K, F.ldt, t8);
            to_int8_kernel<<<std::min<size_t>(1024, ((size_t)N * K + 255) / 256), 256, 0, cl.stream>>>(Xtr, (size_t)N * K, x8);
        }
        F.XT8 = t8; F.Xtr8 = x8;
    } else {
        double *td = cl.alloc<double>((size_t)F.ldt * K + 4);
        if (!cl.err) transpose_pad_kernel<double><<<tg, blk, 0, cl.stream>>>(Xtr, N, K, F.ldt, td);
        F.XTd = td;
    }
    if (tc) {
        const int nst = (N + TC_KS - 1) / TC_KS, ntile = (K + TC_TILE - 1) / TC_TILE;
        const size_t bytes = (size_t)ntile * nst * TC_A_BYTES;
        int8_t *img = cl.alloc<int8_t>(2 * bytes);
        if (!cl.err)
            tc_image_kernel<<<(int)std::min<size_t>(1024, (bytes + 255) / 256), 256, 0, cl.stream>>>(Xtr, N, K, nst, ntile, img, img + bytes);
        F.Xtc = img; F.Xtcsq = img + bytes;
    }
    cl.note(cudaGetLastError());
    return F;
}

__global__ void __launch_bounds__(FIT_THREADS, PAREBEN_MIN_BLOCKS) probe_tc_kernel(FoldData F, int Kc, int R, const double *phi, int ldphi,
                                                         const double *w, const double *e, double *G, double *bb,
                                                         double *ze, int8_t *planes)
{
    extern __shared__ __align__(32) double s_buf[];
    __shared__ TcState tcs;
    tc_open(tcs);
    tc_contract(F, Kc, R, [&](int j) -> const double * { return phi + (size_t)j * ldphi; },
                [&](int j, bool &dv) -> double * { dv = true; return G + (size_t)j * Kc; }, w, e, bb, ze, planes, s_buf, tcs);
    tc_close(tcs);
}

// right-hand sides r < n_aligned: 16-byte aligned PHI columns (leading dimension phi_ld(N), pad rows zero); the others:
// plain vectors of N doubles that start 8 bytes past a 16-byte boundary, as the 8-byte copy path sees them
template <bool EPIS>
__global__ void __launch_bounds__(FIT_THREADS, PAREBEN_MIN_BLOCKS) probe_contract_x_kernel(FoldData F, int K, int Kc, int R, int n_aligned,
                                                                 const double *acols, const double *ucols, const double *w,
                                                                 const double *e, double *G, double *bb, double *ze)
{
    extern __shared__ __align__(32) double s_buf[];
    const int N = F.ntr, LD = phi_ld(N);
    contract_x<EPIS>(F, K, Kc, R, n_aligned,
                     [&](int r) -> const double * { return r < n_aligned ? acols + (size_t)r * LD : ucols + (size_t)(r - n_aligned) * N; },
                     [&](int r, bool &dv) -> double * { dv = true; return G + (size_t)r * Kc; }, s_buf, w, e, bb, ze);
}

__global__ void probe_cand_kernel(int K, int Kc, int *I, int *J)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < Kc) { Cand<true> cd(c, K); I[c] = cd.i; J[c] = cd.j; }
}

template <class Kern>
bool launch_setup(Call &cl, Kern kern)
{
    return cl.note(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S_BUF_BYTES));
}

}  // namespace

extern "C" const char *probe_last_error(void) { return g_err.c_str(); }

// X: [N][K] row-major training rows (integers, |x| <= 11, N max|x|^2 64 < 2^31: the host predicate of the tensor-core
// path).  phi: [R][N], column 0 all ones in a fit (bb reuses column 0's digit planes).  w, e: [N].
// Out: G [R][K], bb [K], ze [K], scale [K] (the column norms the kernel divided by).
extern "C" int probe_tc(int N, int K, const double *X, int R, const double *phi, const double *w, const double *e,
                        double *G, double *bb, double *ze, double *scale)
{
    if (N < 1 || K < 1 || R < 0 || !X || !w || !e || (R > 0 && !phi)) return bad("probe_tc: bad argument");
    double max_abs = 0;
    if (!small_int_design(X, (size_t)N * K, max_abs) || max_abs > 11.0 || (double)N * max_abs * max_abs * 64.0 >= 2147483648.0)
        return bad("probe_tc: the design is outside the tensor-core path (integers, |x| <= 11, N max|x|^2 64 < 2^31)");
    Call cl;
    FoldData F = layout_fold(cl, X, N, K, K, false, true, true);
    const int ld = phi_ld(N);
    double *d_phi = cl.alloc<double>((size_t)std::max(R, 1) * ld);
    for (int j = 0; j < R && !cl.err; j++) cl.note(cudaMemcpyAsync(d_phi + (size_t)j * ld, phi + (size_t)j * N, sizeof(double) * N, cudaMemcpyHostToDevice, cl.stream));
    const double *d_w = cl.upload(w, N), *d_e = cl.upload(e, N);
    double *d_G = cl.alloc<double>((size_t)std::max(R, 1) * K), *d_bb = cl.alloc<double>(K), *d_ze = cl.alloc<double>(K);
    int8_t *d_planes = cl.alloc<int8_t>(tc_planes_bytes(N));
    if (!cl.err && launch_setup(cl, probe_tc_kernel))
        probe_tc_kernel<<<1, FIT_T, S_BUF_BYTES, cl.stream>>>(F, K, R, d_phi, ld, d_w, d_e, d_G, d_bb, d_ze, d_planes);
    cl.note(cudaGetLastError());
    cl.download(G, d_G, (size_t)R * K);
    cl.download(bb, d_bb, K);
    cl.download(ze, d_ze, K);
    cl.download(scale, F.scale, K);
    return cl.finish();
}

// X: [N][K] row-major training rows; epis: candidates are the K main effects and the K(K-1)/2 pairs (Cand<true>).
// The int8 operand variant runs when every entry is an integer in [-127, 127] and force_f64 is 0, the f64 one otherwise.
// cols: [R][N]; the first n_aligned go through the 16-byte copy path, the rest through the 8-byte one.
// w (optional) weights the right-hand sides (binomial); want_bb (needs w and e) asks for bb = sum x^2 w and ze = X'e,
// which only the DMMA form computes.  Out: G [R][Kc], bb [Kc], ze [Kc] (when want_bb), scale [Kc].
extern "C" int probe_contract_x(int N, int K, int epis, int force_f64, int n_aligned, const double *X, int R,
                                const double *cols, const double *w, const double *e, int want_bb, double *G, double *bb,
                                double *ze, double *scale)
{
    if (N < 2 || K < 1 || R < 1 || !X || !cols || n_aligned < 0 || n_aligned > R) return bad("probe_contract_x: bad argument");
    if (epis && (long long)K * (K + 1) / 2 > 0x7fffffffLL) return bad("probe_contract_x: K(K+1)/2 exceeds int32");
    if (want_bb && (!w || !e)) return bad("probe_contract_x: bb and ze need w and e");
    // the weighted DMMA form always stores bb and ze (a fit asks for them whenever it weights more than SIMT_R_MAX sides)
    if (w && !want_bb && R > SIMT_R_MAX) return bad("probe_contract_x: weighted contractions of more than 4 right-hand sides store bb");
    const int Kc = epis ? (int)((long long)K * (K + 1) / 2) : K;
    double max_abs = 0;
    const bool int8 = small_int_design(X, (size_t)N * K, max_abs) && !force_f64;
    Call cl;
    FoldData F = layout_fold(cl, X, N, K, Kc, epis != 0, int8, false);
    const int ld = phi_ld(N);
    double *d_a = cl.alloc<double>((size_t)std::max(n_aligned, 1) * ld);
    double *d_u = cl.alloc<double>((size_t)(R - n_aligned) * N + 2) + 1;
    for (int r = 0; r < R && !cl.err; r++) {
        double *dst = r < n_aligned ? d_a + (size_t)r * ld : d_u + (size_t)(r - n_aligned) * N;
        cl.note(cudaMemcpyAsync(dst, cols + (size_t)r * N, sizeof(double) * N, cudaMemcpyHostToDevice, cl.stream));
    }
    const double *d_w = w ? cl.upload(w, N) : nullptr, *d_e = (w && e) ? cl.upload(e, N) : nullptr;
    double *d_G = cl.alloc<double>((size_t)R * Kc);
    double *d_bb = want_bb ? cl.alloc<double>(Kc) : nullptr, *d_ze = want_bb ? cl.alloc<double>(Kc) : nullptr;
    if (!cl.err) {
        if (epis) {
            if (launch_setup(cl, probe_contract_x_kernel<true>))
                probe_contract_x_kernel<true><<<1, FIT_T, S_BUF_BYTES, cl.stream>>>(F, K, Kc, R, n_aligned, d_a, d_u, d_w, d_e, d_G, d_bb, d_ze);
        } else {
            if (launch_setup(cl, probe_contract_x_kernel<false>))
                probe_contract_x_kernel<false><<<1, FIT_T, S_BUF_BYTES, cl.stream>>>(F, K, Kc, R, n_aligned, d_a, d_u, d_w, d_e, d_G, d_bb, d_ze);
        }
    }
    cl.note(cudaGetLastError());
    cl.download(G, d_G, (size_t)R * Kc);
    if (want_bb) { cl.download(bb, d_bb, Kc); cl.download(ze, d_ze, Kc); }
    cl.download(scale, F.scale, Kc);
    return cl.finish();
}

// I[c], J[c] for c < Kc = K(K+1)/2: the loci of Epis candidate c as the contraction kernels decode it
extern "C" int probe_cand_map(int K, int Kc, int *I, int *J)
{
    if (K < 1 || Kc < 1 || !I || !J) return bad("probe_cand_map: bad argument");
    Call cl;
    int *d_I = cl.alloc<int>(Kc), *d_J = cl.alloc<int>(Kc);
    if (!cl.err) probe_cand_kernel<<<(Kc + 255) / 256, 256, 0, cl.stream>>>(K, Kc, d_I, d_J);
    cl.note(cudaGetLastError());
    cl.download(I, d_I, Kc);
    cl.download(J, d_J, Kc);
    return cl.finish();
}

// the launch resources of the probes (those of the fit kernels)
extern "C" void probe_resources(int *threads, long long *smem_bytes)
{
    *threads = FIT_T;
    *smem_bytes = (long long)S_BUF_BYTES;
}
