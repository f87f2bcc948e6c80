// Developer tool: resident CTAs per SM of every bucketed NMS kernel at the shared memory its launches use
// (cudaOccupancyMaxActiveBlocksPerMultiprocessor).  Built and run by tools/nms_two_per_sm.py; one JSON line per kernel.
#include <cstdarg>
#include <cstdio>

#include "nms_bucket.cu"

namespace frr {
std::atomic<uint64_t> g_launches{0};
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vfprintf(stderr, fmt, ap);
    va_end(ap);
    fputc('\n', stderr);
}
}  // namespace frr

template <int kThreads, int S>
static int report() {
    constexpr int kYBins = frr::bk_ybins(kThreads, S);
    auto kern = frr::nms_bucket_kernel<kThreads, kYBins>;
    const size_t smem = frr::nms_bucket_smem_bytes(kThreads, S);
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    cudaFuncAttributes fa;
    FRR_CUDA(cudaFuncGetAttributes(&fa, kern));
    int blocks = 0;
    FRR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, kern, kThreads, smem));
    printf("{\"kernel\": \"nms_bucket_kernel<%d, %d>\", \"dynamic_smem\": %zu, \"registers\": %d, \"local_bytes\": %zu, "
           "\"ctas_per_sm\": %d}\n", kThreads, kYBins, smem, fa.numRegs, fa.localSizeBytes, blocks);
    return 0;
}

int main() {
    if (report<256, 1>() || report<512, 1>() || report<1024, 1>() || report<1024, 8>()) return 1;
    return 0;
}
