// Host-callable launchers of the score kernels. The kernels are heavily unrolled templates (one instantiation per
// length class); they are compiled in their own translation units (launch_*.cu) so that the host engine and the
// kernel families build in parallel and a change in one does not recompile the others.
#pragma once
#include <cuda_runtime.h>

#include "kernels_s16.cuh"
#include "kernels_s16_wide.cuh"
#include "kernels_s16_long.cuh"
#include "kernels_s16_long2.cuh"
#include "kernels_s32.cuh"
#include "kernels_s32_long.cuh"
#include "kernels_coords.cuh"

namespace sw4 {

// two-rows-per-step kernel, subjects <= 512 (R = 4, 6, ..., 32); cudaErrorInvalidValue for an unknown R
cudaError_t launch_s16(int R, const S16Params& prm, int grid, cudaStream_t stream);
// the same kernel in its multi-segment form (items of several 16 x R-column segments, R = 18..32)
cudaError_t launch_s16_multi(int R, const S16Params& prm, int grid, cudaStream_t stream);
// full-warp one-row-per-step kernel, 513..1024 (R = 18..32) and the multi-segment class (R = 32, multi)
cudaError_t launch_s16_wide(int R, bool multi, const S16WideParams& prm, int grid, cudaStream_t stream);
// CTA-wide systolic arrays for long subjects (blockDim = 32 * prm.warps)
cudaError_t launch_s16_long(const S16LongParams& prm, int grid, cudaStream_t stream);
cudaError_t launch_s32_long(const S32LongParams& prm, int grid, cudaStream_t stream);
// the same arrays at two query rows per step (16 / prm.warps arrays of prm.warps warps per 512-thread CTA)
cudaError_t launch_s16_long2(const S16Long2Params& prm, int grid, cudaStream_t stream);
// exact 32-bit wavefront, one subject per warp
cudaError_t launch_s32(const S32Params& prm, int blocks, cudaStream_t stream);
// its PSSM form: scores from the int32 plane of the query profile (prof = profile + 483 * profStride)
cudaError_t launch_s32_pssm(const S32Params& prm, const int32_t* prof, int profStride, int blocks, cudaStream_t stream);
// alignment coordinates: pass 1 (ends) or pass 2 (begins), one CTA per CoordGroup. The coordinate and traceback
// launchers take a PSSM query's [qlen][21] device table as `pssm` (nullptr: a sequence query scored with prm.matrix).
cudaError_t launch_coords(bool reverse, const CoordParams& prm, int groups, cudaStream_t stream, const int8_t* pssm = nullptr);
// alignment traceback: pass 3 (directions over each rectangle, one CTA per CoordGroup), then the walk (prm.numItems pairs)
cudaError_t launch_coords_trace(const CoordParams& prm, int groups, cudaStream_t stream, const int8_t* pssm = nullptr);
cudaError_t launch_coords_walk(const CoordParams& prm, cudaStream_t stream, const int8_t* pssm = nullptr);

// CTAs are launched as clusters of 2 whenever the grid is even: the two SMs of a TPC share an instruction cache, and
// with many different (large, heavily unrolled) kernels resident at once it pays to give both SMs the same code.
template <class Kernel, class Params>
inline cudaError_t launch_clustered(Kernel kernel, const Params& prm, int grid, int threads, int smemBytes, cudaStream_t stream) {
    static const bool noCluster = getenv("SW4_NO_CLUSTER") != nullptr;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = (size_t)smemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (grid % 2 == 0 && !noCluster) ? 2 : 1;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, prm);
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device)
template <class Kernel>
inline cudaError_t ensure_smem_attr(Kernel kernel, int smemBytes, bool (&configured)[64]) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (!configured[dev & 63]) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smemBytes);
        if (e != cudaSuccess) return e;
        configured[dev & 63] = true;
    }
    return cudaSuccess;
}

}  // namespace sw4
