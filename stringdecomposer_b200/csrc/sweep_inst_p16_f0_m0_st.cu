// instantiations of sweep_kernel<Packed16, C, T, FAST=0, MULTI=0> -- STREAM: symbols read from global memory
#include "sweep_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_SWEEP(sweep_lookup_p16_f0_m0_st, Packed16, false, false, true)
}
