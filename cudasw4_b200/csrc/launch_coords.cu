// Launchers of the alignment-coordinate passes, the traceback pass and the walk (kernels_coords.cuh).
#include "launch.hpp"

namespace sw4 {

cudaError_t launch_coords(bool reverse, const CoordParams& prm, int groups, cudaStream_t stream) {
    if (groups <= 0) return cudaSuccess;
    if (reverse) sw_coords_kernel<true><<<groups, kCoordThreads, 0, stream>>>(prm);
    else sw_coords_kernel<false><<<groups, kCoordThreads, 0, stream>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_coords_trace(const CoordParams& prm, int groups, cudaStream_t stream) {
    if (groups <= 0) return cudaSuccess;
    sw_coords_trace_kernel<><<<groups, kCoordThreads, 0, stream>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_coords_walk(const CoordParams& prm, cudaStream_t stream) {
    if (prm.numItems <= 0) return cudaSuccess;
    sw_coords_walk_kernel<><<<(prm.numItems + kWalkThreads - 1) / kWalkThreads, kWalkThreads, 0, stream>>>(prm);
    return cudaGetLastError();
}

}  // namespace sw4
