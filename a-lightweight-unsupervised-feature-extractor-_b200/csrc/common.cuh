// Shared host/device helpers for libb200track (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "b200track.h"

namespace b200 {

extern thread_local char g_err[512];
extern std::atomic<int64_t> g_launches;

int fail(int code, const char* fmt, ...);
int scratch_pool(cudaMemPool_t* out);       // private per-device pool for stream-ordered scratch (api.cu)

inline int check_launch(const char* what) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(B200_ECUDA, "%s: %s", what, cudaGetErrorString(e));
    return B200_OK;
}

// Launches kern with programmatic stream serialisation when pdl is set, and as clusters of cluster_x CTAs when
// cluster_x > 0 (a cluster attribute of size 1 is still an attribute: the launch is not the same as one without).
// Errors surface in check_launch().
template <typename Kern, typename... Args>
inline void launch_ex(Kern kern, dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, int cluster_x,
                      Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    unsigned n = 0;
    if (pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n++].val.programmaticStreamSerializationAllowed = 1;
    }
    if (cluster_x > 0) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n++].val.clusterDim = {(unsigned)cluster_x, 1, 1};
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    (void)cudaLaunchKernelEx(&cfg, kern, args...);
}

#define B200_CUDA(expr)                                                                  \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess)                                                           \
            return ::b200::fail(B200_ECUDA, "%s: %s", #expr, cudaGetErrorString(_e));    \
    } while (0)

#define B200_REQUIRE(cond, ...)                                                          \
    do {                                                                                 \
        if (!(cond)) return ::b200::fail(B200_EINVAL, __VA_ARGS__);                      \
    } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

constexpr int kWarp = 32;
constexpr int kSMs = 148;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace b200
