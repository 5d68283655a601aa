// instantiations of sweep_kernel<Packed16, C, T, FAST=1, MULTI=0> -- STREAM: symbols read from global memory
#include "sweep_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_SWEEP(sweep_lookup_p16_f1_m0_st, Packed16, true, false, true)
}
