// instantiations of sweep_kernel<Scalar32, C, T, FAST=0, MULTI=0> -- STREAM: symbols read from global memory
#include "sweep_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_SWEEP(sweep_lookup_s32_f0_m0_st, Scalar32, false, false, true)
}
