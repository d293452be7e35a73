// fit_ge.cu -- eben_fit_kernel<EPIS=true, BINOMIAL=false> and its launcher (see fit_kernel.cuh).
#include "fit_kernel.cuh"
PAREBEN_DEFINE_VARIANT(ge, true, false, false)
PAREBEN_DEFINE_GRAM(ge, true)
