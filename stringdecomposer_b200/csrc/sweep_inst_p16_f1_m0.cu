// instantiations of sweep_kernel<Packed16, C, T, FAST=1, MULTI=0>
#include "sweep_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_SWEEP(sweep_lookup_p16_f1_m0, Packed16, true, false, false)
}
