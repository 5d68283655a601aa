// explicit instantiations of the deferred-jump sweep, packed s16x2 policy (+ the instrumented twins)
#include "sweep_lat_kernel.cuh"
namespace sdb {
SD_INSTANTIATE_LAT(sweep_lat_lookup_p16, Packed16, false)
const void *sweep_lat_timing_lookup_p16(const Geometry &g)
{
    const int C = g.C, T = g.T, W = g.scanw;
    SD_LAT_PICK(Packed16, 6, 32, true, false) SD_LAT_PICK(Packed16, 12, 16, true, false)
    return nullptr;
}
}
