// Cost operators of the C ABI: build_C_app_topk and bbox/conf/total cost.  Math in assoc_cost.cuh.
#include "assoc_cost.cuh"

namespace b200 {
int app_cost_tc(const float* bank, const int32_t* bank_len, const float* fallback, const float* det, int M, int N, int T,
                int topk, int use_topk_mean, float* C_app, int ldc, cudaStream_t st);      // app_cost_tc.cu
namespace {

__global__ void __launch_bounds__(cost::kThreads)
app_cost_kernel(const float* __restrict__ bank, const int32_t* __restrict__ bank_len,
                const float* __restrict__ fallback, const float* __restrict__ det, int N, int T, int topk,
                int topk_mean, float* __restrict__ C_app, int ldc) {
    extern __shared__ __align__(16) float smem[];
    const int i = blockIdx.y, j0 = blockIdx.x * cost::kTileN;
    int len = min(bank_len[i], T);
    const float* rows = bank + (size_t)i * T * cost::kD;
    if (len <= 0 && fallback) {                 // mainTracking.py:180-182: the EMA stands in as a 1-row bank
        rows = fallback + (size_t)i * cost::kD;
        len = 1;
    }
    const int j = j0 + threadIdx.x;
    if (len <= 0 || topk <= 0) {                // :183-186 and :197-199: a row of ones
        if (threadIdx.x < cost::kTileN && j < N) C_app[(size_t)i * ldc + j] = 1.0f;
        return;
    }
    const float c = cost::app_cost_tile<true>(rows, len, det, N, j0, topk, topk_mean != 0, smem);
    if (threadIdx.x < cost::kTileN && j < N) C_app[(size_t)i * ldc + j] = c;
}

__global__ void __launch_bounds__(256)
pair_cost_kernel(const float* __restrict__ C_app, const float* __restrict__ bp, const float* __restrict__ bc,
                 const float* __restrict__ cp, const float* __restrict__ cc, int M, int N, cost::PairWeights w,
                 float* C_total, float* C_bbox, float* C_center, float* C_scale, float* C_conf, int ldc) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= N) return;
    float p[4], c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { p[k] = bp[(size_t)i * 4 + k]; c[k] = bc[(size_t)j * 4 + k]; }
    const size_t o = (size_t)i * ldc + j;
    const cost::PairCost r = cost::pair_cost(p, c, cp[i], cc[j], w, C_app ? C_app[o] : 0.0f);
    if (C_total) C_total[o] = r.total;
    if (C_bbox) C_bbox[o] = r.bbox;
    if (C_center) C_center[o] = r.center;
    if (C_scale) C_scale[o] = r.scale;
    if (C_conf) C_conf[o] = r.conf;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" int b200_app_cost_topk_f32(const float* bank, const int32_t* bank_len, const float* fallback,
                                      const float* det, int M, int N, int T, int topk, int use_topk_mean,
                                      float* C_app, int ldc, void* stream) {
    B200_REQUIRE(M >= 0 && N >= 0, "app_cost: negative size");
    if (M == 0 || N == 0) return B200_OK;
    B200_REQUIRE(T >= 1 && T <= cost::kMaxBank, "app_cost: bank depth %d outside [1,%d]", T, cost::kMaxBank);
    B200_REQUIRE(bank && bank_len && det && C_app, "app_cost: null pointer");
    B200_REQUIRE(ldc >= N, "app_cost: ldc < N");
    B200_REQUIRE(M <= 65535, "app_cost: M too large");
    // large launches are a real GEMM: bf16x3-split tensor-core kernel (app_cost_tc.cu); problems under 64 x 64 and
    // banks deeper than its 32 rows keep the float32 FFMA kernel below
    const int rc = app_cost_tc(bank, bank_len, fallback, det, M, N, T, topk, use_topk_mean, C_app, ldc, as_stream(stream));
    if (rc != 1) return rc;
    static bool configured[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    if (!configured[dev]) {
        B200_CUDA(cudaFuncSetAttribute(app_cost_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)cost::smem_bytes(cost::kMaxBank)));
        configured[dev] = true;
    }
    dim3 grid((N + cost::kTileN - 1) / cost::kTileN, M);
    app_cost_kernel<<<grid, cost::kThreads, cost::smem_bytes(T), as_stream(stream)>>>(
        bank, bank_len, fallback, det, N, T, topk, use_topk_mean, C_app, ldc);
    return check_launch("app_cost_kernel");
}

extern "C" int b200_pair_cost_f32(const float* C_app, const float* boxes_prev, const float* boxes_cur,
                                  const float* conf_prev, const float* conf_cur, int M, int N, float w_app,
                                  float w_bbox, float w_conf, float alpha, float beta, float conf_eps,
                                  float* C_total, float* C_bbox, float* C_center, float* C_scale, float* C_conf,
                                  int ldc, void* stream) {
    B200_REQUIRE(M >= 0 && N >= 0, "pair_cost: negative size");
    if (M == 0 || N == 0) return B200_OK;
    B200_REQUIRE(boxes_prev && boxes_cur && conf_prev && conf_cur, "pair_cost: null pointer");
    B200_REQUIRE(ldc >= N && M <= 65535, "pair_cost: bad ldc / M");
    cost::PairWeights w{w_app, w_bbox, w_conf, alpha, beta, conf_eps};
    dim3 grid((N + 255) / 256, M);
    pair_cost_kernel<<<grid, 256, 0, as_stream(stream)>>>(C_app, boxes_prev, boxes_cur, conf_prev, conf_cur, M, N, w,
                                                         C_total, C_bbox, C_center, C_scale, C_conf, ldc);
    return check_launch("pair_cost_kernel");
}
