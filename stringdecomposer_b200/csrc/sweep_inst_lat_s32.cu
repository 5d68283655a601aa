// explicit instantiations of the deferred-jump sweep, s32 policy
#include "sweep_lat_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_LAT(sweep_lat_lookup_s32, Scalar32, false)
}
