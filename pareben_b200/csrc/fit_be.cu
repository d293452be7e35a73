// fit_be.cu -- eben_fit_kernel<EPIS=true, BINOMIAL=true> and its launcher (see fit_kernel.cuh).
#include "fit_kernel.cuh"
PAREBEN_DEFINE_VARIANT(be, true, true, false)
