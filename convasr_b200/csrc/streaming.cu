// Batched copies of the streaming acoustic model (convasr_b200/streaming.py).
//
// A stream keeps, per activation of the inference plan, a linear buffer of the frames later launches still read.  Every
// call gathers those rows of all streams into the batched input window of each launch, appends the new final rows to
// every stream's buffer and, when a buffer fills up, moves its live rows back to the front.  All three are lists of
// contiguous byte ranges, one list per launch of stream_copy_kernel.
#include "common.cuh"
#include "../../include/convasr_b200.h"
#include <atomic>

namespace cab {
extern std::atomic<int64_t> g_launch_count;

// jobs: [n][3] int64 (dst, src, bytes); src 0 = zero fill; 16-byte aligned pointers and sizes; ranges of one launch
// do not overlap.  blockIdx.y = job
__global__ void __launch_bounds__(256) stream_copy_kernel(const int64_t* __restrict__ jobs) {
    const int64_t* j = jobs + 3 * (size_t)blockIdx.y;
    uint4* dst = reinterpret_cast<uint4*>(j[0]);
    const uint4* src = reinterpret_cast<const uint4*>(j[1]);
    const int64_t n = j[2] >> 4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        dst[i] = src != nullptr ? src[i] : make_uint4(0u, 0u, 0u, 0u);
}
}  // namespace cab

using namespace cab;

extern "C" int cab_stream_copy(const int64_t* jobs, int n_jobs, int64_t max_bytes, cab_stream_t stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    CAB_CHECK_ARG(n_jobs >= 0 && n_jobs <= 65535, "n_jobs=%d out of [0, 65535]", n_jobs);
    CAB_CHECK_ARG(max_bytes >= 0 && max_bytes % 16 == 0, "max_bytes=%lld must be a non-negative multiple of 16", (long long)max_bytes);
    if (n_jobs == 0 || max_bytes == 0) return 0;
    CAB_CHECK_ARG(jobs != nullptr && (reinterpret_cast<uintptr_t>(jobs) & 7) == 0, "jobs must be an 8-byte aligned device array");
    const int64_t vec = max_bytes / 16;
    const unsigned gx = (unsigned)(vec < 256 * 16 ? (vec + 255) / 256 : 16);
    stream_copy_kernel<<<dim3(gx, (unsigned)n_jobs), 256, 0, stream>>>(jobs);
    CAB_CHECK_LAUNCH();
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return 0;
}
