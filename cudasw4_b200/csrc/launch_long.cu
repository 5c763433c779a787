// Launchers of the CTA-wide array kernels (kernels_s16_long.cuh, kernels_s32_long.cuh) and of the one-subject-per-warp
// exact 32-bit kernel (kernels_s32.cuh).
#include <cstdlib>
#include "launch.hpp"

namespace sw4 {

template <int GAPS>
static cudaError_t launch_s16_long_gaps(const S16LongParams& prm, int grid, cudaStream_t stream) {
    static bool configured[64] = {};
    cudaError_t e = ensure_smem_attr(sw_s16_long_kernel<GAPS>, s16_long_smem_bytes(kLongMaxWarps), configured);
    if (e != cudaSuccess) return e;
    sw_s16_long_kernel<GAPS><<<grid, prm.warps * 32, s16_long_smem_bytes(prm.warps), stream>>>(prm);
    return cudaGetLastError();
}
cudaError_t launch_s16_long(const S16LongParams& prm, int grid, cudaStream_t stream) {
    static const bool generic = getenv("SW4_NO_GAP_SETS") != nullptr;
    switch (generic ? 0 : s16_gap_set_for(prm.gop2, prm.gex2)) {
        case 1: return launch_s16_long_gaps<1>(prm, grid, stream);
        case 2: return launch_s16_long_gaps<2>(prm, grid, stream);
        case 3: return launch_s16_long_gaps<3>(prm, grid, stream);
        default: return launch_s16_long_gaps<0>(prm, grid, stream);
    }
}

template <int GAPS>
static cudaError_t launch_s16_long2_gaps(const S16Long2Params& prm, int grid, cudaStream_t stream) {
    static bool configured[64] = {};
    cudaError_t e = ensure_smem_attr(sw_s16_long2_kernel<GAPS>, s16_long2_smem_bytes(kLong2MaxW), configured);
    if (e != cudaSuccess) return e;
    sw_s16_long2_kernel<GAPS><<<grid, kLong2Warps * 32, s16_long2_smem_bytes(prm.warps), stream>>>(prm);
    return cudaGetLastError();
}
cudaError_t launch_s16_long2(const S16Long2Params& prm, int grid, cudaStream_t stream) {
    static const bool generic = getenv("SW4_NO_GAP_SETS") != nullptr;
    switch (generic ? 0 : s16_gap_set_for(prm.gop2, prm.gex2)) {
        case 1: return launch_s16_long2_gaps<1>(prm, grid, stream);
        case 2: return launch_s16_long2_gaps<2>(prm, grid, stream);
        case 3: return launch_s16_long2_gaps<3>(prm, grid, stream);
        default: return launch_s16_long2_gaps<0>(prm, grid, stream);
    }
}

template <int GAPS>
static cudaError_t launch_s32_long_gaps(const S32LongParams& prm, int grid, cudaStream_t stream) {
    static bool configured[64] = {};
    cudaError_t e = ensure_smem_attr(sw_s32_long_kernel<GAPS>, s32_long_smem_bytes(kLongMaxWarps), configured);
    if (e != cudaSuccess) return e;
    sw_s32_long_kernel<GAPS><<<grid, prm.warps * 32, s32_long_smem_bytes(prm.warps), stream>>>(prm);
    return cudaGetLastError();
}
cudaError_t launch_s32_long(const S32LongParams& prm, int grid, cudaStream_t stream) {
    static const bool generic = getenv("SW4_NO_GAP_SETS") != nullptr;
    if (!generic && prm.gop == -11 && prm.gex == -1) return launch_s32_long_gaps<1>(prm, grid, stream);
    return launch_s32_long_gaps<0>(prm, grid, stream);
}

cudaError_t launch_s32(const S32Params& prm, int blocks, cudaStream_t stream) {
    sw_s32_kernel<0><<<blocks, kS32Threads, 0, stream>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_s32_pssm(const S32Params& prm, const int32_t* prof, int profStride, int blocks, cudaStream_t stream) {
    sw_s32_pssm_kernel<0><<<blocks, kS32Threads, 0, stream>>>(prm, prof, profStride);
    return cudaGetLastError();
}

}  // namespace sw4
