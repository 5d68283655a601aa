// explicit instantiations of the deferred-jump sweep, s32 policy -- ST: symbols read from global memory
#include "sweep_lat_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_LAT(sweep_lat_lookup_s32_st, Scalar32, true)
}
