"""pareben_b200 -- B200-native (sm_100a CUDA) implementation of parEBEN's cross-validation hot path.

Public surface mirrors the reference R package (same names and arguments):
CrossValidate, BuildGrid, GetLambdaMax, AssignToFolds, LocalSearch, plus the final-model
wrappers EBelasticNet_Gaussian / EBelasticNet_Binomial.  All numerics run in libpareben.so
(pareben_b200/csrc, C-ABI in include/pareben.h); there is no CPU implementation here.
"""
from ._lib import (FIT_BASIS_CAP, FIT_ITER_MAX, FIT_LIST_CAP, FIT_NONFINITE, FIT_NOT_PD, MODE_AUTO, MODE_CACHED,  # noqa: F401
                   MODE_STREAMING, ParebenError, Problem, cv_grid, cv_grid_multi, default_device, device_count, load,
                   measure_fp64_peak, release_cache, set_mode, shard_plan)
from .cross_validate import (AssignToFolds, BuildGrid, CrossValidate, CrossValidateMulti, EBelasticNet_Binomial,  # noqa: F401
                             EBelasticNet_Gaussian, GetLambdaMax, LocalSearch, SLFilter)
