// fit_gm.cu -- eben_fit_kernel<EPIS=false, BINOMIAL=false> and its launcher (see fit_kernel.cuh).
#include "fit_kernel.cuh"
PAREBEN_DEFINE_VARIANT(gm, false, false, false)
PAREBEN_DEFINE_GRAM(gm, false)
