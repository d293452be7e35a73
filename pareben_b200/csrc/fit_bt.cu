// fit_bt.cu -- eben_fit_kernel<EPIS=false, BINOMIAL=true, TC=true> (score contraction on the int8 tensor cores,
// tc_contract.cuh) and its launcher (see fit_kernel.cuh).
#include "fit_kernel.cuh"
PAREBEN_DEFINE_VARIANT(bt, false, true, true)
