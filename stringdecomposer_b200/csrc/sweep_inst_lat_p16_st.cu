// explicit instantiations of the deferred-jump sweep, packed s16x2 policy -- ST: symbols read from global memory
#include "sweep_lat_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_LAT(sweep_lat_lookup_p16_st, Packed16, true)
}
