// fit_launch.h -- host-callable entry points of the five kernel translation units.
#pragma once
#include "common.cuh"

namespace pareben {

constexpr int FIT_THREADS_HOST = 256;

#define PAREBEN_DECLARE_VARIANT(NAME)                                                                                     \
    cudaError_t launch_fit_##NAME(int grid, int threads, cudaStream_t stream, const Problem &P, const Variant &v,        \
                                  const FitTask *tasks, int n_tasks, const Sched &sched, char *slabs, size_t slab_stride,  \
                                  const FitOutputs &out);                                                                 \
    cudaError_t occupancy_##NAME(int *blocks_per_sm, int threads);                                                        \
    void timing_##NAME(unsigned long long *cc, int reset, unsigned long long *t0, unsigned long long *t1, int *block, int n);

PAREBEN_DECLARE_VARIANT(gm)   // Gaussian, main effects
PAREBEN_DECLARE_VARIANT(ge)   // Gaussian, Epis
PAREBEN_DECLARE_VARIANT(bm)   // binomial, main effects
PAREBEN_DECLARE_VARIANT(be)   // binomial, Epis
PAREBEN_DECLARE_VARIANT(bt)   // binomial, main effects, score contraction on the int8 tensor cores (Problem::tc)

// Gaussian only: build FoldData::C for the listed folds (fold_gram_kernel, fit_kernel.cuh)
cudaError_t launch_gram_gm(int grid, int threads, cudaStream_t stream, const Problem &P, const int *fold_list, int n_fold_list,
                           char *slabs, size_t slab_stride, int *next_item);
cudaError_t launch_gram_ge(int grid, int threads, cudaStream_t stream, const Problem &P, const int *fold_list, int n_fold_list,
                           char *slabs, size_t slab_stride, int *next_item);

}  // namespace pareben
