// mb_tc.cu -- isolated microbenchmark and exactness check of the tcgen05 INT8 score contraction (tc_contract.cuh).
// Config-2 shape: 481 candidates, 400 training rows of {-1, 0, 1} codes, M + 1 in {8, 32, 64} right-hand-side columns,
// two 256-thread blocks per SM on every SM.  Reports cycles per call of the digit extraction alone and of the whole
// contraction (extraction + MMA pass + epilogue), and checks G, bb and ze against a long-double host evaluation with the
// bound N 2^-57 max|b| max|x| (+ the FP64 rounding of the scaling steps).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -std=c++17 -I../../pareben_b200/csrc -o mb_tc mb_tc.cu
#include "tc_contract.cuh"
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <random>

using namespace pareben;

__global__ void __launch_bounds__(256, 2) mb_kernel(FoldData F, int Kc, int M, int reps, const double *phi, int LD,
                                                    const double *w, const double *e, char *slabs, size_t slab_stride,
                                                    double *G, double *bb, double *ze, unsigned long long *cyc)
{
    extern __shared__ __align__(32) double s_buf[];
    __shared__ TcState tcs;
    tc_open(tcs);
    int8_t *planes = reinterpret_cast<int8_t *>(slabs + (size_t)blockIdx.x * slab_stride);
    const int N = F.ntr, nst = (N + TC_KS - 1) / TC_KS;
    double *bscale = s_buf + TC_RING_BYTES / 8;
    const bool out = blockIdx.x == 0;
    double *Gb = out ? G : G + (size_t)M * Kc, *bbb = out ? bb : bb + Kc, *zeb = out ? ze : ze + Kc;   // block 0 writes the checked copy
    auto col = [&](int r) -> const double * { return phi + (size_t)r * LD; };
    auto dest = [&](int r, bool &dv) -> double * { dv = true; return Gb + (size_t)r * Kc; };
    long long t0 = clock64();
    for (int i = 0; i < reps; i++) {
        for (int j0 = 0; j0 < M + 1; j0 += TC_COLS)
            tc_digits(j0, min(TC_COLS, M + 1 - j0), N, nst, M, col, w, e, planes, bscale, s_buf);
        __syncthreads();
    }
    long long t1 = clock64();
    for (int i = 0; i < reps; i++) tc_contract(F, Kc, M, col, dest, w, e, bbb, zeb, planes, s_buf, tcs);
    long long t2 = clock64();
    if (threadIdx.x == 0) { atomicAdd(&cyc[0], (unsigned long long)(t1 - t0)); atomicAdd(&cyc[1], (unsigned long long)(t2 - t1)); }
    tc_close(tcs);
}

__global__ void image_kernel(const int8_t *X, int nrows, int K, int nst, int ntile, int8_t *img, int8_t *sq)
{
    const int cols = ntile * TC_TILE;
    const size_t n = (size_t)cols * nst * TC_KS;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cols), h = (int)(i / cols);
        const int x = (c < K && h < nrows) ? X[(size_t)h * K + c] : 0;
        const size_t o = tc_image_offset(c, h, nst);
        img[o] = (int8_t)x; sq[o] = (int8_t)(x * x);
    }
}

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

int main()
{
    const int N = 400, K = 481, reps = 20, LD = (N + 3) & ~3, nst = (N + TC_KS - 1) / TC_KS, ntile = (K + TC_TILE - 1) / TC_TILE;
    int sms = 0; CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, 0));
    printf("device %s, %d SMs; N %d, Kc %d, %d blocks x 256 threads, %d calls per block\n", prop.name, sms, N, K, 2 * sms, reps);
    std::mt19937_64 rng(7);
    std::vector<int8_t> X((size_t)N * K);
    for (auto &x : X) x = (int8_t)((int)(rng() % 3) - 1);
    for (int h = 0; h < N; h++) X[(size_t)h * K + 17] = 0;            // an all-zero column
    std::vector<double> scale(K);
    for (int c = 0; c < K; c++) { double s = 0; for (int h = 0; h < N; h++) s += X[(size_t)h * K + c] * X[(size_t)h * K + c]; scale[c] = s > 0 ? std::sqrt(s) : 1; }
    std::uniform_real_distribution<double> U(-1, 1);
    const int Mmax = 63;
    std::vector<double> phi((size_t)LD * Mmax, 0.0), w(N), e(N);
    for (int h = 0; h < N; h++) { phi[h] = 1; w[h] = 0.25 * (0.02 + 0.98 * (U(rng) + 1) / 2); e[h] = U(rng) * 0.9; }
    for (int r = 1; r < Mmax; r++) for (int h = 0; h < N; h++) phi[(size_t)r * LD + h] = U(rng) * std::ldexp(1.0, (int)(rng() % 9) - 4);
    int8_t *dX, *dimg; double *dphi, *dw, *de, *dscale, *dG, *dbb, *dze; char *dslab; unsigned long long *dcyc;
    const size_t img_bytes = (size_t)ntile * nst * TC_A_BYTES, slab_stride = (tc_planes_bytes(N) + 255) & ~(size_t)255;
    CK(cudaMalloc(&dX, X.size())); CK(cudaMalloc(&dimg, 2 * img_bytes));
    CK(cudaMalloc(&dphi, phi.size() * 8)); CK(cudaMalloc(&dw, N * 8)); CK(cudaMalloc(&de, N * 8)); CK(cudaMalloc(&dscale, K * 8));
    CK(cudaMalloc(&dG, (size_t)2 * Mmax * K * 8)); CK(cudaMalloc(&dbb, 2 * K * 8)); CK(cudaMalloc(&dze, 2 * K * 8));
    CK(cudaMalloc(&dslab, slab_stride * 2 * sms)); CK(cudaMalloc(&dcyc, 16));
    CK(cudaMemcpy(dX, X.data(), X.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dphi, phi.data(), phi.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dw, w.data(), N * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(de, e.data(), N * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dscale, scale.data(), K * 8, cudaMemcpyHostToDevice));
    image_kernel<<<256, 256>>>(dX, N, K, nst, ntile, dimg, dimg + img_bytes);
    FoldData F{};
    F.ntr = N; F.scale = dscale; F.Xtc = dimg; F.Xtcsq = dimg + img_bytes;
    const int smem = TC_SMEM_BYTES;
    CK(cudaFuncSetAttribute(mb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int fails = 0;
    for (int Mp1 : {8, 32, 64}) {
        const int M = Mp1 - 1;
        CK(cudaMemset(dcyc, 0, 16));
        mb_kernel<<<2 * sms, 256, smem>>>(F, K, M, reps, dphi, LD, dw, de, dslab, slab_stride, dG, dbb, dze, dcyc);
        CK(cudaGetLastError()); CK(cudaDeviceSynchronize());
        unsigned long long cyc[2]; CK(cudaMemcpy(cyc, dcyc, 16, cudaMemcpyDeviceToHost));
        const double calls = 2.0 * sms * reps;
        std::vector<double> G((size_t)M * K), bb(K), ze(K);
        CK(cudaMemcpy(G.data(), dG, G.size() * 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(bb.data(), dbb, K * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(ze.data(), dze, K * 8, cudaMemcpyDeviceToHost));
        double worst = 0;      // largest error in units of the bound
        auto check = [&](double got, long double ref, double bound) { const double r = (double)fabsl((long double)got - ref) / bound; if (!(r <= 1)) fails++; if (r > worst || r != r) worst = r; };
        for (int c = 0; c < K; c++) {
            for (int r = 0; r <= M + 1; r++) {
                long double s = 0; double mb = 0;
                for (int h = 0; h < N; h++) {
                    const double b = r < M ? w[h] * phi[(size_t)r * LD + h] : r == M ? e[h] : w[h];
                    const int x = X[(size_t)h * K + c], xx = r == M + 1 ? x * x : x;
                    s += (long double)xx * b; mb = std::max(mb, std::fabs(b));
                }
                const double bound = N * std::ldexp(1.0, -57) * mb * 2 + std::fabs((double)s) * std::ldexp(1.0, -51) + 1e-300;
                if (r < M) check(G[(size_t)r * K + c], s / scale[c], bound / scale[c] + std::fabs((double)(s / scale[c])) * std::ldexp(1.0, -52));
                else if (r == M) check(ze[c], s, bound);
                else check(bb[c], s, bound);
            }
        }
        printf("M+1 = %2d: digits %8.0f cycles/call, whole contraction %8.0f cycles/call (MMA pass + epilogue %8.0f); "
               "max error / bound %.3f\n", Mp1, cyc[0] / calls, cyc[1] / calls, (cyc[1] - (double)cyc[0]) / calls, worst);
    }
    printf(fails ? "FAIL: %d values outside the bound\n" : "PASS%.0d\n", fails);
    return fails ? 1 : 0;
}
