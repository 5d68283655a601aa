// instantiations of sweep_kernel<Packed16, C, T, FAST=1, MULTI=1> -- STREAM: symbols read from global memory
#include "sweep_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_SWEEP(sweep_lookup_p16_f1_m1_st, Packed16, true, true, true)
}
