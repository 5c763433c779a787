// Test harness of the device top-k (cudasw4_b200/csrc/topk.cuh). TEST INFRASTRUCTURE: compiled on first use by
// tests/topk_harness.py into the system's temporary directory. It runs the engine's own dispatch (topk_enqueue) on
// scores given by the host, with the scratch sized by the same helpers the engine uses.
#include <cstdint>
#include <cuda_runtime.h>

#include "../cudasw4_b200/csrc/topk.cuh"

using namespace sw4;

extern "C" int topk_h_shift_for(long long maxScore) { return topk_shift_for(maxScore); }
extern "C" int topk_h_pass1_blocks(long long n, int k, int smCount) { return topk_pass1_blocks(n, k, smCount); }
extern "C" int topk_h_uses_large_path(int k) { return topk_uses_large_path(k) ? 1 : 0; }
extern "C" int topk_h_max_candidates() { return kTopkMaxCandidates; }
extern "C" int topk_h_large_blocks() { return kTopkLargeBlocks; }
extern "C" int topk_h_sm_count() {  // of device 0, or -1 without one
    int v = 0;
    return cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, 0) == cudaSuccess ? v : -1;
}

// Top-k of scores[0..n) through topk_enqueue. The outputs (k entries each, and *outCount) are first set to a poison
// value on the device, so entries the kernels leave unwritten show up. *launches receives topk_enqueue's return value.
// Returns 0, the CUDA error code, or -1 when topk_enqueue refused maxScore.
extern "C" int topk_h_run(const int32_t* scores, long long n, int k, long long maxScore, int smCount, const int32_t* globalIds,
                          int32_t* outScores, int32_t* outIds, int* outCount, int* launches) {
    int32_t *dScores = nullptr, *dIds = nullptr, *dOutScores = nullptr, *dOutIds = nullptr;
    int *dCount = nullptr, *dWork = nullptr;
    TopkCand* dCand = nullptr;
    unsigned long long* dKeys = nullptr;
    cudaStream_t stream = nullptr;
    int rc = -1;
    *launches = 0;
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; return e == cudaSuccess; };
    if (ok(topk_configure()) && ok(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)) &&
        ok(cudaMalloc(&dScores, (size_t)n * sizeof(int32_t))) &&
        (!globalIds || ok(cudaMalloc(&dIds, (size_t)n * sizeof(int32_t)))) &&
        ok(cudaMalloc(&dOutScores, (size_t)k * sizeof(int32_t))) && ok(cudaMalloc(&dOutIds, (size_t)k * sizeof(int32_t))) &&
        ok(cudaMalloc(&dCount, sizeof(int))) && ok(cudaMalloc(&dCand, (size_t)kTopkMaxCandidates * sizeof(TopkCand))) &&
        ok(cudaMalloc(&dWork, topk_large_work_ints() * sizeof(int))) &&
        ok(cudaMalloc(&dKeys, (size_t)topk_large_num_keys(k) * sizeof(unsigned long long))) &&
        ok(cudaMemcpyAsync(dScores, scores, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, stream)) &&
        (!globalIds || ok(cudaMemcpyAsync(dIds, globalIds, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, stream))) &&
        ok(cudaMemsetAsync(dOutScores, 0x5a, (size_t)k * sizeof(int32_t), stream)) &&
        ok(cudaMemsetAsync(dOutIds, 0x5a, (size_t)k * sizeof(int32_t), stream)) &&
        ok(cudaMemsetAsync(dCount, 0x5a, sizeof(int), stream))) {
        *launches = topk_enqueue(dScores, n, k, maxScore, smCount, dIds, dCand, dWork, dKeys, dOutScores, dOutIds, dCount, stream);
        if (ok(cudaGetLastError()) &&
            ok(cudaMemcpyAsync(outScores, dOutScores, (size_t)k * sizeof(int32_t), cudaMemcpyDeviceToHost, stream)) &&
            ok(cudaMemcpyAsync(outIds, dOutIds, (size_t)k * sizeof(int32_t), cudaMemcpyDeviceToHost, stream)) &&
            ok(cudaMemcpyAsync(outCount, dCount, sizeof(int), cudaMemcpyDeviceToHost, stream)) && ok(cudaStreamSynchronize(stream)))
            rc = *launches < 0 ? -1 : 0;
    }
    for (void* p : {(void*)dScores, (void*)dIds, (void*)dOutScores, (void*)dOutIds, (void*)dCount, (void*)dCand, (void*)dWork,
                    (void*)dKeys})
        if (p) cudaFree(p);
    if (stream) cudaStreamDestroy(stream);
    return e != cudaSuccess ? (int)e : rc;
}
