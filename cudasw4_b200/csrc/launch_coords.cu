// Launcher of the alignment-coordinate passes (kernels_coords.cuh).
#include "launch.hpp"

namespace sw4 {

cudaError_t launch_coords(bool reverse, const CoordParams& prm, int groups, cudaStream_t stream) {
    if (groups <= 0) return cudaSuccess;
    if (reverse) sw_coords_kernel<true><<<groups, kCoordThreads, 0, stream>>>(prm);
    else sw_coords_kernel<false><<<groups, kCoordThreads, 0, stream>>>(prm);
    return cudaGetLastError();
}

}  // namespace sw4
