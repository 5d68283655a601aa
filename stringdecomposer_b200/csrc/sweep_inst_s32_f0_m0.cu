// instantiations of sweep_kernel<Scalar32, C, T, FAST=0, MULTI=0>
#include "sweep_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_SWEEP(sweep_lookup_s32_f0_m0, Scalar32, false, false, false)
}
