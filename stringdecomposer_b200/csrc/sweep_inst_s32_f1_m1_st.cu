// instantiations of sweep_kernel<Scalar32, C, T, FAST=1, MULTI=1> -- STREAM: symbols read from global memory
#include "sweep_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_SWEEP(sweep_lookup_s32_f1_m1_st, Scalar32, true, true, true)
}
