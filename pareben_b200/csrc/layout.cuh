// layout.cuh -- the per-fold layout kernels that turn a row-major training matrix into the operands of the score
// contractions: the transposed, row-permuted copy (FoldData::XT8 / XTd), the int8 copy (Xtr8), the tensor-core operand
// images (Xtc / Xtcsq) and the column norms (scale).  pareben_problem_create launches them; the kernel tests
// (tests/kernels/contract_probe.cu) build their FoldData with the same kernels.
#pragma once
#include "common.cuh"
#include "tc_contract.cuh"

namespace {

__global__ void to_int8_kernel(const double *__restrict__ in, size_t n, int8_t *__restrict__ out)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (int8_t)in[i];
}

// The int8 operand images of the tensor-core contraction (tc_contract.cuh): X' and X o X' in the UMMA canonical K-major
// layout, [128-candidate tile][32-row stage], zero-padded to whole tiles and stages.
__global__ void tc_image_kernel(const double *__restrict__ X, int nrows, int K, int nst, int ntile, int8_t *__restrict__ img,
                                int8_t *__restrict__ sq)
{
    const int cols = ntile * pareben::TC_TILE;
    const size_t n = (size_t)cols * nst * pareben::TC_KS;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % cols), h = (int)(i / cols);
        const int x = (c < K && h < nrows) ? (int)X[(size_t)h * K + c] : 0;
        const size_t o = pareben::tc_image_offset(c, h, nst);
        img[o] = (int8_t)x; sq[o] = (int8_t)(x * x);
    }
}

// Transposed, row-padded copy of a row-major matrix: out[k*ldt + r] = X[r*K + k] (zero for r >= nrows), as int8 or f64.
template <class T>
__global__ void transpose_pad_kernel(const double *__restrict__ X, int nrows, int K, int ldt, T *__restrict__ out)
{
    __shared__ double tile[32][33];
    const int r0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
    for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
        const int r = r0 + rr, k = k0 + threadIdx.x;
        tile[rr][threadIdx.x] = (r < nrows && k < K) ? X[(size_t)r * K + k] : 0.0;
    }
    __syncthreads();
    for (int kk = threadIdx.y; kk < 32; kk += blockDim.y) {
        const int r = r0 + threadIdx.x, k = k0 + kk;
        // rows of every group of 16 are stored permuted: physical position 4a + b holds row 4b + a (see mma_pass)
        const int rp = (r & ~15) | ((r & 3) << 2) | ((r >> 2) & 3);
        if (r < ldt && k < K) out[(size_t)k * ldt + rp] = (T)tile[threadIdx.x][kk];
    }
}

// scale[c] = sqrt(sum_h x_c[h]^2), 1 when the column is all zero (MainEff.c:87-99, NeFull2.c:100-135)
template <bool EPIS>
__global__ void scales_kernel(const double *__restrict__ X, int N, int K, int Kc, double *__restrict__ scale)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= Kc) return;
    pareben::Cand<EPIS> cd(c, K);
    double z = 0;
    for (int h = 0; h < N; h++) { const double x = cd.at(X + (size_t)h * K); z = fma(x, x, z); }
    if (z == 0) z = 1;
    scale[c] = sqrt(z);
}

}  // namespace
