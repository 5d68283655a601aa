// instantiations of sweep_kernel<Packed16, C, T, FAST=1, MULTI=1>
#include "sweep_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_SWEEP(sweep_lookup_p16_f1_m1, Packed16, true, true, false)
}
