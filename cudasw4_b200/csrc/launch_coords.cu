// Launchers of the alignment-coordinate passes, the traceback pass and the walk (kernels_coords.cuh).
#include "launch.hpp"

namespace sw4 {

cudaError_t launch_coords(bool reverse, const CoordParams& prm, int groups, cudaStream_t stream, const int8_t* pssm) {
    if (groups <= 0) return cudaSuccess;
    if (pssm) {
        if (reverse) sw_coords_pssm_kernel<true><<<groups, kCoordThreads, 0, stream>>>(prm, pssm);
        else sw_coords_pssm_kernel<false><<<groups, kCoordThreads, 0, stream>>>(prm, pssm);
    } else {
        if (reverse) sw_coords_kernel<true><<<groups, kCoordThreads, 0, stream>>>(prm);
        else sw_coords_kernel<false><<<groups, kCoordThreads, 0, stream>>>(prm);
    }
    return cudaGetLastError();
}

cudaError_t launch_coords_trace(const CoordParams& prm, int groups, cudaStream_t stream, const int8_t* pssm) {
    if (groups <= 0) return cudaSuccess;
    if (pssm) sw_coords_trace_pssm_kernel<><<<groups, kCoordThreads, 0, stream>>>(prm, pssm);
    else sw_coords_trace_kernel<><<<groups, kCoordThreads, 0, stream>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_coords_walk(const CoordParams& prm, cudaStream_t stream, const int8_t* pssm) {
    if (prm.numItems <= 0) return cudaSuccess;
    const int blocks = (prm.numItems + kWalkThreads - 1) / kWalkThreads;
    if (pssm) sw_coords_walk_pssm_kernel<><<<blocks, kWalkThreads, 0, stream>>>(prm, pssm);
    else sw_coords_walk_kernel<><<<blocks, kWalkThreads, 0, stream>>>(prm);
    return cudaGetLastError();
}

}  // namespace sw4
