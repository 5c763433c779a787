// Launchers of the profile construction (profile.cuh).
#include "profile.cuh"

namespace sw4 {

cudaError_t launch_profile_scatter(const CoordParams& prm, const int* msaRow, uint8_t* msa, int m, cudaStream_t stream) {
    if (prm.numItems <= 0 || m <= 0) return cudaSuccess;
    const int blocks = (prm.numItems + kProfileThreads - 1) / kProfileThreads;
    profile_scatter_kernel<><<<blocks, kProfileThreads, 0, stream>>>(prm, msaRow, msa, m);
    return cudaGetLastError();
}

cudaError_t launch_profile_build(const ProfileParams& prm, cudaStream_t stream, int* launches) {
    if (prm.m <= 0) return cudaSuccess;
    const int colBlocks = (prm.m + kProfileThreads - 1) / kProfileThreads;
    profile_columns_kernel<><<<colBlocks, kProfileThreads, 0, stream>>>(prm);
    profile_weights_kernel<><<<prm.rows, kProfileThreads, 0, stream>>>(prm);
    profile_scores_kernel<><<<colBlocks, kProfileThreads, 0, stream>>>(prm);
    *launches += 3;
    return cudaGetLastError();
}

}  // namespace sw4
