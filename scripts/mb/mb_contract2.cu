// Microbenchmark of the tensor-core contraction in isolation (experiments only).
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -std=c++17 -I../../pareben_b200/csrc -o mb_contract2 mb_contract2.cu
#include "contract.cuh"
#include <cstdio>
#include <cstdlib>
#include <vector>
using namespace pareben;

__global__ void __launch_bounds__(256, 2)
mb_kernel(FoldData F, int K, int Kc, int M, int LD, double *phi_all, double *G_all, double *vec_all, int reps, long long *cycles, int weighted)
{
    extern __shared__ __align__(32) double s_buf[];
    double *phi = phi_all + (size_t)blockIdx.x * M * LD;
    double *G = G_all + (size_t)blockIdx.x * (M + 2) * Kc;
    double *w = vec_all + (size_t)blockIdx.x * 2 * LD, *e = w + LD;
    __syncthreads();
    const long long t0 = clock64();
    for (int r = 0; r < reps; r++) {
        contract_x<false>(F, K, Kc, M, M,
            [&](int c) -> const double * { return phi + (size_t)c * LD; },
            [&](int c, bool &dv) -> double * { dv = true; return G + (size_t)c * Kc; },
            s_buf, weighted ? w : nullptr, weighted ? e : nullptr, weighted ? G + (size_t)M * Kc : nullptr, weighted ? G + (size_t)(M + 1) * Kc : nullptr);
    }
    __syncthreads();
    if (threadIdx.x == 0) cycles[blockIdx.x] = clock64() - t0;
}

int main(int argc, char **argv)
{
    const int N = argc > 1 ? atoi(argv[1]) : 400, K = argc > 2 ? atoi(argv[2]) : 481, M = argc > 3 ? atoi(argv[3]) : 30;
    const int blocks = argc > 4 ? atoi(argv[4]) : 296, reps = argc > 5 ? atoi(argv[5]) : 20, weighted = argc > 6 ? atoi(argv[6]) : 1;
    const int Kc = K, LD = phi_ld(N), ldt = (N + 31) & ~31;
    std::vector<int8_t> xt((size_t)K * ldt, 0), xr((size_t)N * K);
    for (int k = 0; k < K; k++) for (int h = 0; h < N; h++) { int8_t v = (int8_t)(rand() % 3 - 1); xt[(size_t)k * ldt + h] = v; xr[(size_t)h * K + k] = v; }
    int8_t *d_xt, *d_xr; double *d_scale, *d_phi, *d_G, *d_vec; long long *d_cyc;
    cudaMalloc(&d_xt, xt.size()); cudaMalloc(&d_xr, xr.size()); cudaMalloc(&d_scale, sizeof(double) * Kc);
    cudaMemcpy(d_xt, xt.data(), xt.size(), cudaMemcpyHostToDevice); cudaMemcpy(d_xr, xr.data(), xr.size(), cudaMemcpyHostToDevice);
    std::vector<double> ones(Kc, 1.5); cudaMemcpy(d_scale, ones.data(), sizeof(double) * Kc, cudaMemcpyHostToDevice);
    std::vector<double> ph((size_t)blocks * M * LD); for (auto &v : ph) v = (rand() % 1000) * 1e-3;
    cudaMalloc(&d_phi, sizeof(double) * ph.size()); cudaMemcpy(d_phi, ph.data(), sizeof(double) * ph.size(), cudaMemcpyHostToDevice);
    cudaMalloc(&d_G, sizeof(double) * (size_t)blocks * (M + 2) * Kc);
    std::vector<double> vv((size_t)blocks * 2 * LD, 0.25); cudaMalloc(&d_vec, sizeof(double) * vv.size()); cudaMemcpy(d_vec, vv.data(), sizeof(double) * vv.size(), cudaMemcpyHostToDevice);
    cudaMalloc(&d_cyc, sizeof(long long) * blocks);
    FoldData F{}; F.Xtr = nullptr; F.Xtr8 = d_xr; F.XT8 = d_xt; F.XTd = nullptr; F.ldt = ldt; F.ntr = N; F.nte = 0; F.scale = d_scale;
    const size_t smem = (size_t)(SV_DOUBLES > 5200 ? SV_DOUBLES : 5200) * sizeof(double);
    cudaFuncSetAttribute(mb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int it = 0; it < 2; it++) {
        cudaEventRecord(e0);
        mb_kernel<<<blocks, 256, smem>>>(F, K, Kc, M, LD, d_phi, d_G, d_vec, reps, d_cyc, weighted);
        cudaEventRecord(e1); cudaEventSynchronize(e1);
    }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    std::vector<long long> cyc(blocks); cudaMemcpy(cyc.data(), d_cyc, sizeof(long long) * blocks, cudaMemcpyDeviceToHost);
    double avg = 0; for (auto c : cyc) avg += c; avg /= blocks * (double)reps;
    const double fma = (double)N * Kc * M, flops = 2 * fma * blocks * reps;
    printf("N=%d K=%d M=%d blocks=%d weighted=%d: %.0f cycles/call/block, %.3f ms total, %.2f TFLOP/s (alg), err=%s\n", N, K, M, blocks, weighted, avg, ms,
           flops / (ms * 1e-3) / 1e12, cudaGetErrorString(cudaGetLastError()));
    return 0;
}
