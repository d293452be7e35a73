/* pareben.h -- C-ABI of the B200-native EBEN cross-validation hot path (libpareben.so).
 *
 * Drop-in boundary.  The reference reaches its numerical core through R's `.C` interface, one
 * call per (fold, alpha, lambda) fit, fanned out by foreach/%dopar%:
 *     R/CrossValidate.R:66-70,88-92  ->  R/TestModel.R:20,28  ->
 *     EBEN_orig/R/EBelasticNet.Gaussian.R:16-28,39-51 / EBelasticNet.Binomial.R:12-25,33-46  ->
 *     void elasticNetLinearNeMainEff(...)   EBEN_orig/src/elasticNetLinearNeMainEff.c:55-57
 *     void elasticNetLinearNeEpisEff(...)   EBEN_orig/src/elasticNetLinearNeFull2.c:57-58
 *     void ElasticNetBinaryNEmainEff(...)   EBEN_orig/src/ElasticNetBinaryNEmainEff.c:236-238
 *     void ElasticNetBinaryNEfull(...)      EBEN_orig/src/ElasticNetBinaryNeFull.c:52-55
 * and scores every fit in R (R/GetModelError.R:6-59).  This library replaces that whole
 * fan-out by ONE grid-level call (pareben_cv_grid) plus a batch-of-1 entry (pareben_fit) that
 * returns the same outputs, in the same layouts, as the four `.C` symbols, so the R wrappers'
 * post-processing (EBelasticNet.Gaussian.R:56-98) keeps working unchanged.
 *
 * Conventions: plain pointers and sizes only; caller owns every host buffer; matrices are
 * column-major doubles exactly as `as.double(BASIS)` hands them to `.C`; the library owns all
 * device memory.  Every function returns 0 on success or a negative PAREBEN_E* code, with
 * text available from pareben_last_error().  Nothing here ever runs a fit on the CPU: without
 * a CUDA device the calls fail with PAREBEN_ENODEVICE.
 */
#ifndef PAREBEN_H
#define PAREBEN_H

#ifdef __cplusplus
extern "C" {
#endif

#define PAREBEN_VERSION 2

/* prior (R: prior = "gaussian" | "binomial", R/CrossValidate.R:65,87) */
#define PAREBEN_GAUSSIAN 0
#define PAREBEN_BINOMIAL 1

/* error codes */
#define PAREBEN_OK          0
#define PAREBEN_EINVAL     -1   /* bad argument */
#define PAREBEN_ENODEVICE  -2   /* no usable CUDA device */
#define PAREBEN_ECUDA      -3   /* CUDA runtime failure (see pareben_last_error) */
#define PAREBEN_ENOMEM     -4   /* device or host allocation failed */
#define PAREBEN_EUNSUPPORTED -5 /* variant not built yet */

/* per-fit status bits (0 = clean).  The reference has no error channel: these are the cases in
 * which it prints and carries on (MainEff.c:605-611, 1352-1362; NEmainEff.c:692-695). */
#define PAREBEN_FIT_BASIS_CAP   1   /* active set reached the basis cap; further additions dropped */
#define PAREBEN_FIT_NOT_PD      2   /* a Hessian was not positive definite */
#define PAREBEN_FIT_NONFINITE   4   /* non-finite hold-out error */
#define PAREBEN_FIT_ITER_MAX    8   /* outer loop hit its 100-iteration limit */
#define PAREBEN_FIT_LIST_CAP   16   /* streaming mode: more than 4096 candidates tied within n_add of the best addition */

typedef struct pareben_problem pareben_problem;

/* Upload one CrossValidate problem to `device` and prepare the per-fold training/test matrices
 * and column norms there (replaces the per-task row subsetting of R/TestModel.R:11-17 and the
 * `Scales` loops at MainEff.c:87-99 / NeFull2.c:100-135).
 *   basis    n x k column-major        target  length n (binomial: 0/1)
 *   fold_id  length n, values 1..n_folds (R/AssignToFolds.R); n_folds == 0 means "no hold-out":
 *            a single pseudo-fold 0 that trains on all rows (used by pareben_fit)
 *   epis     0: Epis="no", 1: Epis="yes" (k(k+1)/2 candidates, pair columns generated on the fly) */
int pareben_problem_create(pareben_problem **out, int device, const double *basis, int n, int k,
                           const double *target, const int *fold_id, int n_folds, int epis, int prior);
void pareben_problem_destroy(pareben_problem *p);

/* Several responses, one design (QTL traits measured on the same genotypes, permuted copies of one response):
 * pareben_problem_create with targets an n x n_targets column-major matrix, one response per column.  The design-side
 * data (per-fold training matrices, column norms, Gram matrices, streaming buffers) exist once and serve every response;
 * only the training and test vectors are kept per (response, fold).  Every fit of such a problem gives bitwise the result
 * of the same fit on a problem created with that response alone.  pareben_problem_create is the n_targets = 1 case.
 * pareben_fit, pareben_lambda_max, pareben_sl_filter and pareben_problem_cv_grid fail with PAREBEN_EINVAL on a problem
 * with n_targets > 1 (use the _multi calls; the final model of a response is fitted on a single-response problem). */
int pareben_problem_create_multi(pareben_problem **out, int device, const double *basis, int n, int k,
                                 const double *targets, int n_targets, const int *fold_id, int n_folds, int epis, int prior);

/* The library keeps one per-device work buffer alive between calls (allocating several GB per
 * CrossValidate would dominate small problems); this releases it. */
void pareben_release_cache(void);

/* Run n_fits independent EBEN fits in one batched launch.  Fit i trains on the rows whose fold
 * label differs from fold[i] (1-based; 0 = all rows) with hyper-parameters (alpha[i], lambda[i])
 * and is scored on the held-out rows as R/GetModelError.R does: Gaussian -> sum of squared
 * errors, binomial -> mean Bernoulli log-likelihood with the odds clamp of :52-55.
 * Outputs (each length n_fits, any may be NULL): fold_err, status (PAREBEN_FIT_* bits),
 * n_selected (number of non-zero effects), n_iter (outer iterations). */
int pareben_run_fits(pareben_problem *p, int n_fits, const int *fold, const double *alpha,
                     const double *lambda, double *fold_err, int *status, int *n_selected, int *n_iter);

/* pareben_run_fits for a problem with several responses: fit i trains on response target[i] (0 .. n_targets - 1).
 * Fits of every response share one launch (cached kernels) or the same lock-step rounds and scans (streaming mode); when
 * the streaming states of all fits do not fit in device memory, whole responses run in successive waves. */
int pareben_run_fits_multi(pareben_problem *p, int n_fits, const int *target, const int *fold, const double *alpha,
                           const double *lambda, double *fold_err, int *status, int *n_selected, int *n_iter);

/* One-shot grid call with host buffers: the replacement for the foreach loop of
 * R/CrossValidate.R:66-70 / 88-92.  Grid point g (alpha[g], lambda[g]) x fold f (1..n_folds)
 * is fit number g*n_folds + (f-1).  fold_err/status/n_selected are n_grid*n_folds, grid-major,
 * fold-minor -- the row order of Results.Detail.
 * Devices: the call drives n_devices GPUs, `device` .. `device + n_devices - 1` (n_devices = 0: every
 * visible device from `device` on), one internal worker thread per GPU, BASIS uploaded once per
 * GPU; it returns when all of them have written their entries (the in-library gather).  This is
 * what a single R process uses to fan one grid over the box (the reference fans the 400 rows over
 * all registered workers from one call, R/CrossValidate.R:66-70).
 * Shards (one process per GPU, e.g. torchrun / doMPI-style launches): fits are ordered by falling
 * expected cost (rising lambda) and dealt round-robin over n_shards * n_devices; this call computes
 * shard `shard` and writes ONLY those entries of the outputs (pass shard 0, n_shards 1 for
 * everything).  The caller merges shards -- a 32 KB gather at nFolds = 10, the `.combine = rbind`
 * of the reference.  Each fit is computed by exactly one thread block with a schedule-independent
 * summation order, so the table is bitwise identical for any device / shard count. */
int pareben_cv_grid(const double *basis, int n, int k, const double *target, const int *fold_id,
                    int n_folds, const double *alpha, const double *lambda, int n_grid, int epis,
                    int prior, int n_devices, int device, int shard, int n_shards, double *fold_err,
                    int *status, int *n_selected);

/* pareben_cv_grid on a problem that is already resident (created with folds): BuildGrid's pareben_lambda_max, the
 * grid and a LocalSearch refinement then share ONE upload and one set of per-fold layouts.  Same outputs, same shard rule. */
int pareben_problem_cv_grid(pareben_problem *p, const double *alpha, const double *lambda, int n_grid, int shard,
                            int n_shards, double *fold_err, int *status, int *n_selected);

/* pareben_cv_grid / pareben_problem_cv_grid for n_targets responses (targets n x n_targets column-major).  alpha and lambda
 * are n_targets x n_grid, response-major (entry t * n_grid + g: each response has its own grid, from its own lambda_max);
 * the tables are response-major, then grid, then fold: fit (t * n_grid + g) * n_folds + (f - 1).  That is the numbering of
 * pareben_cv_grid on n_targets * n_grid grid points with the flattened lambda, and shards are dealt by pareben_shard_plan on
 * exactly that (n_grid' = n_targets * n_grid).  One upload and one set of per-fold layouts per device serve all responses. */
int pareben_cv_grid_multi(const double *basis, int n, int k, const double *targets, int n_targets, const int *fold_id,
                          int n_folds, const double *alpha, const double *lambda, int n_grid, int epis, int prior,
                          int n_devices, int device, int shard, int n_shards, double *fold_err, int *status, int *n_selected);
int pareben_problem_cv_grid_multi(pareben_problem *p, const double *alpha, const double *lambda, int n_grid, int shard,
                                  int n_shards, double *fold_err, int *status, int *n_selected);

/* The shard assignment pareben_cv_grid uses, exposed for the host layer and tests (host-only
 * logic, needs no device): writes the ascending fit numbers of `shard` into fit_index
 * (capacity n_grid*n_folds) and their count into n_mine. */
int pareben_shard_plan(const double *lambda, int n_grid, int n_folds, int shard, int n_shards,
                       int *fit_index, int *n_mine);

/* Batch-of-1 fit on all rows of a problem created with n_folds == 0: the `.C` outputs.
 *   beta_table  gaussian main: k x 4, gaussian epis: k(k+1)/2 x 5, binomial main: k x 4,
 *               binomial epis: 2k x 4 -- column-major, same cell meaning as `Beta` in the
 *               reference entry points (loc1, loc2, mu/scale, sigma_ii/scale^2[, used id])
 *   wald[1], intercept[1 gaussian | 2 binomial], extra[1] = residual variance (gaussian,
 *   MainEff.c:227) or log-likelihood (binomial, NEmainEff.c:805). */
int pareben_fit(pareben_problem *p, double alpha, double lambda, double *beta_table, double *wald,
                double *intercept, double *extra, int *status);

/* EBEN's own four `.C` entry points, same names, argument lists and output layouts, as wrappers over
 * pareben_problem_create + pareben_fit: an R session that loads this library in place of EBEN's (useDynLib / PACKAGE
 * swapped) runs EBelasticNet.Gaussian / EBelasticNet.Binomial unchanged.  Replaces
 *   EBEN_orig/src/elasticNetLinearNeMainEff.c:55-57     EBEN_orig/src/elasticNetLinearNeFull2.c:57-58
 *   EBEN_orig/src/ElasticNetBinaryNEmainEff.c:236-238   EBEN_orig/src/ElasticNetBinaryNeFull.c:52-55
 * (call sites EBEN_orig/R/EBelasticNet.Gaussian.R:16-28,39-51, EBelasticNet.Binomial.R:12-25,33-46).  Device:
 * environment variable PAREBEN_DEVICE (default 0).  void like the originals; failures are reported on stderr. */
void elasticNetLinearNeMainEff(double *BASIS, double *y, double *a_lambda, double *b_Alpha, double *Beta, double *wald,
                               double *intercept, int *n, int *kdim, int *verb, double *residual);
void elasticNetLinearNeEpisEff(double *BASIS, double *y, double *a_lambda, double *b_Alpha, double *Beta, double *wald,
                               double *intercept, int *n, int *kdim, int *verb, double *residual);
void ElasticNetBinaryNEmainEff(double *BASIS, double *Targets, double *a_Lambda, double *b_Alpha, double *logLIKELIHOOD,
                               double *Beta, double *wald, double *intercept, int *n, int *kdim, int *VB, int *bMax);
void ElasticNetBinaryNEfull(double *BASIS, double *Targets, double *a_Lambda, double *b_Alpha, double *logLIKELIHOOD,
                            double *Beta, double *wald, double *intercept, int *n, int *kdim, int *VB, int *bMax);

/* lambda_max of R/BuildGrid.R:5-32 (before the x10), computed on the device for the problem's
 * full data; epis taken from the problem. */
int pareben_lambda_max(pareben_problem *p, double *lambda_max);
/* pareben_lambda_max of every response of the problem (lambda_max[n_targets]) in one pass over the candidates; each value
 * is bitwise the one pareben_lambda_max gives on a problem holding that response alone. */
int pareben_lambda_max_multi(pareben_problem *p, double *lambda_max);

/* Single-locus prefilter of the published workflow, the step before CrossValidate
 * (paper_materials/Real Data Analysis/SL_filter.R:17-52): standardise the response and every candidate column with
 * R's scale() (centre, divide by the n-1 standard deviation) and keep the candidates whose statistic
 * |ys' xs| / n exceeds a threshold -- tau_main for the k main-effect columns (:21) and, when the problem was created
 * with epis = 1, tau_pair for the k(k-1)/2 products x_i*x_j, i < j (:28-39).  Candidates are numbered as everywhere
 * in this library (0..k-1 main effects, then pairs row-major in i < j); the kept ones are written in ascending order
 * to cand[] / stat[] (each of capacity entries, either may be NULL) and their number to n_kept (which may exceed
 * capacity: call again with a larger buffer).  Constant columns (sd = 0) are never kept, as in R (NaN > tau is FALSE). */
int pareben_sl_filter(pareben_problem *p, double tau_main, double tau_pair, int capacity, int *cand, double *stat,
                      int *n_kept);

/* Work counters of the last pareben_run_fits on this problem, for roofline accounting
 * (SURVEY.md 8d): algorithmic FP64 flops of the contraction/statistics phases, kernel
 * milliseconds measured with CUDA events on the launch stream, launches issued. */
int pareben_last_counters(pareben_problem *p, double *flops, double *kernel_ms, int *launches);
/* Gram organisation of the Gaussian cached kernels.  The candidate-cache row of a basis (CacheBP*,
 * /root/reference/EBEN_orig/src/elasticNetLinearNeMainEff.c:1144-1201; ActionAdd* :1608-1618) depends on the fold only, so
 * the library builds it once per fold for every candidate (8 Kc^2 bytes per fold, when that fits in half of the free
 * device memory and the call has enough fits to amortise 2 N Kc^2 flops per fold; PAREBEN_GRAM=0 / 1 overrides the work
 * test) and all fits of the fold share it.  in_use: 1 when the problem runs that way; avoided_flops: the part of
 * pareben_last_counters' model flops that the last call did not have to execute; build_ms: time the last call spent
 * building the matrices (0 once they exist; it is included in that call's kernel_ms). */
int pareben_last_gram_info(pareben_problem *p, int *in_use, double *avoided_flops, double *build_ms);
/* Score contraction of the binomial main-effect fits (FullStat, ElasticNetBinaryNEmainEff.c:1693-1735).  tensor_core: 1 when
 * the problem computes it on the int8 tensor cores (every design entry an integer with |x| <= 11, exact to FP64 rounding),
 * 0 when on the FP64 path; tc_contractions: how many contractions the last pareben_run_fits ran on the tensor cores. */
int pareben_last_contraction_info(pareben_problem *p, int *tensor_core, double *tc_contractions);

/* Solver organisation.  mode 0 (default) = automatic, 1 = cached kernel, 2 = streaming kernels.
 * The cached kernel keeps the reference's per-fit candidate cache (BASIS_PHI, one row of Kc doubles per active basis,
 * NeFull2.c:350-365) in device memory; the streaming kernels keep only the active set and recompute the per-candidate
 * statistics by one dense contraction per fold for all fits at once -- the only form that exists at
 * Kc = k(k+1)/2 = 2e8 (BASELINE config 5), where the reference itself cannot allocate.  Automatic = streaming above
 * 4,000,000 candidates (PAREBEN_STREAM_KC), Gaussian prior only.  The setting is read by pareben_problem_create. */
int pareben_set_mode(int mode);
int pareben_is_streaming(pareben_problem *p);
/* Streaming mode's share of the last pareben_run_fits: summed CUDA-event time and algorithmic flops
 * (2 x training rows x candidates per waiting fit) of the score-contraction launches, their number, and the rounds. */
int pareben_last_stream_counters(pareben_problem *p, double *scan_ms, double *scan_flops, int *scan_launches, int *rounds);

/* FP64 peak probes for the roofline denominator (MEASURED_PEAKS.json carries no FP64 figure):
 * which = 0 -> DFMA chains on the CUDA cores, 1 -> DMMA (mma.sync.m8n8k4.f64). */
int pareben_measure_fp64_peak(int device, int which, double *tflops);

int pareben_device_count(void);
const char *pareben_last_error(void);
int pareben_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PAREBEN_H */
