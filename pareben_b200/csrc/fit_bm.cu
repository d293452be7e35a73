// fit_bm.cu -- eben_fit_kernel<EPIS=false, BINOMIAL=true> and its launcher (see fit_kernel.cuh).
#include "fit_kernel.cuh"
PAREBEN_DEFINE_VARIANT(bm, false, true, false)
