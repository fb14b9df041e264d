// Shared device helpers for the rorl_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define RORL_OK 0
#define RORL_ERR_SHAPE (-1)
#define RORL_ERR_ALIGN (-2)
#define RORL_ERR_ARG (-3)
#define RORL_ERR_WORKSPACE (-4)

// A launch error is reported as 1000 + cudaError_t (see include/rorl_b200.h).
#define RORL_RETURN_LAUNCH()                              \
    do {                                                  \
        cudaError_t _e = cudaGetLastError();              \
        return _e == cudaSuccess ? RORL_OK : 1000 + (int)_e; \
    } while (0)

namespace rorl {

__device__ __forceinline__ float ex2f(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2f(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcpf(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// sigmoid / tanh / softplus built from ex2 + rcp (2 MUFU each): ~1e-7 relative, far inside the
// 1e-3 parity budget, unlike tanh.approx (2^-11).
__device__ __forceinline__ float sigmoidf_fast(float x) {
    return rcpf(1.0f + ex2f(-x * kLog2e));
}
__device__ __forceinline__ float tanhf_fast(float x) {
    // tanh(x) = 2*sigmoid(2x) - 1, evaluated so that large |x| saturates cleanly.
    float e = ex2f(-2.0f * kLog2e * fabsf(x));
    float t = (1.0f - e) * rcpf(1.0f + e);
    return copysignf(t, x);
}
// torch.nn.functional.softplus(beta=1, threshold=20)
__device__ __forceinline__ float softplusf_fast(float x) {
    if (x > 20.0f) return x;
    float e = ex2f(x * kLog2e);
    // log1p(e): for tiny e use e - e^2/2 to keep relative accuracy
    if (e < 1e-4f) return e - 0.5f * e * e;
    return lg2f(1.0f + e) * kLn2;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, bool valid) {
    uint32_t s = (uint32_t)__cvta_generic_to_shared(smem_dst);
    int sz = valid ? 16 : 0;  // src-size 0 => zero-fill, no global access
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem_src), "r"(sz));
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src, bool valid) {
    uint32_t s = (uint32_t)__cvta_generic_to_shared(smem_dst);
    int sz = valid ? 4 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(s), "l"(gmem_src), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N));
}

// ---- mbarrier (shared-memory transaction barrier) helpers ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void st_cs_f4(float4* p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- persistent thread-block-cluster recurrences (csrc/gru.cu, csrc/lstm.cu) ----
// Launch a 1-D grid of nclusters clusters of cl CTAs each; returns RORL_OK or 1000 + cudaError_t.
template <typename Kern, typename Params>
static int launch_cluster(Kern kern, const Params& p, int cl, int nthreads, int nclusters, cudaStream_t stream) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(cl * nclusters));
    cfg.blockDim = dim3((unsigned)nthreads);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cl;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, p);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return 1000 + (int)e;
    }
    return RORL_OK;
}

// batch rows per cluster: smallest power of two that fits the batch into <= max_clusters clusters
static inline int pick_bg(int64_t B, int max_clusters) {
    int bg = 1;
    while (bg < 4 && (B + bg - 1) / bg > max_clusters) bg <<= 1;
    return bg;
}

}  // namespace rorl
