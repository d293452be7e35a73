// mb_linalg.cu -- the binomial IRLS Newton step's dense linear algebra alone: gram_pipe (Hessian PHI'B PHI and the
// gradient PHI'e from the row-major PHIt) and the register sweep (spd_inverse_sweep, M <= 64), with one block per SM
// slot (2 x 148 blocks of FIT_T threads, S_BUF_BYTES of shared memory, as the fit kernel runs), N = 400 rows.
// Each block repeats Gram -> H + diag(0, alpha) -> sweep REPS times on its own data; thread 0 reads clock64 around
// each phase behind a barrier.  Prints cycles per call for M in {8, 24, 40, 56}.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -std=c++17 -o mb_linalg mb_linalg.cu
#include "../../pareben_b200/csrc/common.cuh"
#include "../../pareben_b200/csrc/gauss_fit.cuh"
#include "../../pareben_b200/csrc/fit_kernel.cuh"
#include <cstdio>
#include <vector>

using namespace pareben;

constexpr int REPS = 40;

__global__ void __launch_bounds__(FIT_THREADS, PAREBEN_MIN_BLOCKS)
mb_kernel(const double *phit, const double *w, const double *e, const double *alpha, int N, int M, double *Hall,
          double *sigall, double *colkall, unsigned long long *cyc)
{
    extern __shared__ __align__(32) double s_buf[];
    __shared__ double red[66];
    __shared__ int redi[66];
    Scratch sc{red, redi, s_buf, nullptr};
    double *H = Hall + (size_t)blockIdx.x * 64 * 64, *sigma = sigall + (size_t)blockIdx.x * 64 * 64;
    double *colk = colkall + (size_t)blockIdx.x * 130;
    unsigned long long cg = 0, cs = 0;
    for (int rep = 0; rep < REPS; rep++) {
        __syncthreads();
        long long t0 = clock64();
        gram_pipe(phit, N, M, w, sc.sweep, [&](int j, int k, double z) {
            if (j == k && j > 0) z += alpha[k - 1];
            H[k * M + j] = z; H[j * M + k] = z;
        }, e, [&](int, double) {});
        for (int idx = threadIdx.x; idx < M * M; idx += blockDim.x) sigma[idx] = H[idx];
        __syncthreads();
        long long t1 = clock64();
        spd_inverse_sweep(sigma, M, colk, sc, sc.sweep);
        __syncthreads();
        long long t2 = clock64();
        cg += t1 - t0; cs += t2 - t1;
    }
    if (threadIdx.x == 0) { cyc[2 * blockIdx.x] = cg; cyc[2 * blockIdx.x + 1] = cs; }
}

int main()
{
    int dev = 0, nsm = 0;
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, dev);
    const int N = 400, grid = 2 * nsm;
    std::vector<double> pt((size_t)(N + 32) * PHIT_LD, 0.0), w(N), e(N), alpha(64);
    unsigned s = 12345u;
    auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (double)(s >> 8) / 16777216.0; };
    for (int h = 0; h < N; h++) {
        pt[(size_t)h * PHIT_LD] = 1.0;
        for (int j = 1; j < PHIT_LD; j++) pt[(size_t)h * PHIT_LD + j] = (double)((int)(rnd() * 3) - 1);
        const double y = rnd();
        w[h] = y * (1 - y) + 0.01; e[h] = rnd() - 0.5;
    }
    for (int j = 0; j < 64; j++) alpha[j] = 0.5 + rnd();
    double *d_pt, *d_w, *d_e, *d_a, *d_H, *d_s, *d_c;
    unsigned long long *d_cyc;
    cudaMalloc(&d_pt, pt.size() * 8); cudaMalloc(&d_w, N * 8); cudaMalloc(&d_e, N * 8); cudaMalloc(&d_a, 64 * 8);
    cudaMalloc(&d_H, (size_t)grid * 4096 * 8); cudaMalloc(&d_s, (size_t)grid * 4096 * 8); cudaMalloc(&d_c, (size_t)grid * 130 * 8);
    cudaMalloc(&d_cyc, (size_t)grid * 2 * 8);
    cudaMemcpy(d_pt, pt.data(), pt.size() * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(d_w, w.data(), N * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(d_e, e.data(), N * 8, cudaMemcpyHostToDevice);
    cudaMemcpy(d_a, alpha.data(), 64 * 8, cudaMemcpyHostToDevice);
    cudaFuncSetAttribute(mb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S_BUF_BYTES);
    printf("# %s, %d SMs, %d blocks x %d threads, N = %d, %d calls per block\n", prop.name, nsm, grid, FIT_T, N, REPS);
    printf("#  M   gram_pipe + H copy (cycles/call)   register sweep (cycles/call)\n");
    for (int M : {8, 24, 40, 56}) {
        std::vector<unsigned long long> cyc((size_t)grid * 2);
        for (int pass = 0; pass < 2; pass++)           // the first pass warms up
            mb_kernel<<<grid, FIT_T, S_BUF_BYTES>>>(d_pt, d_w, d_e, d_a, N, M, d_H, d_s, d_c, d_cyc);
        cudaError_t err = cudaDeviceSynchronize();
        if (err != cudaSuccess) { printf("error: %s\n", cudaGetErrorString(err)); return 1; }
        cudaMemcpy(cyc.data(), d_cyc, cyc.size() * 8, cudaMemcpyDeviceToHost);
        double g = 0, sw = 0;
        for (int b = 0; b < grid; b++) { g += cyc[2 * b]; sw += cyc[2 * b + 1]; }
        printf("%4d   %12.0f   %12.0f\n", M, g / grid / REPS, sw / grid / REPS);
    }
    return 0;
}
