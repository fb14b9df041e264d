// Trajectory gather: builds the zero-padded, nest-stacked [rows, Lmax, F] batch and the [rows, Lmax]
// valid indicator of NestedMemoryArray.sample_trajs from a device-resident fp32 ring buffer, following
// a host-computed placement plan (ref: offpolicy_rnn/buffers/transition_buffer/
// nested_replay_memory.py:103-185; exact layout in SURVEY.md App. A):
//   batch[row, ptr+skip : ptr+skip+len, :]      = ring[src : src+len, :]                  (:160)
//   batch[row, ptr+skip-1, dst_cols]            = ring[src, src_cols]   (pre-step targets)  (:162)
//   batch[row, ptr : ptr+skip, start_col]       = 1                                        (:164)
//   valid[row, ptr+skip : ptr+skip+len]         = ring[src : src+len, mask_col]            (:165)
//   batch[row, row_end[row] :, start_col]       = 1                                        (:171)
// Pure byte movement: a trajectory is one contiguous run in both source and destination, so the
// copy is float4-vectorised when F*len and the offsets allow, scalar otherwise.  Bit-exact.
#include "common.cuh"

namespace rorl {

constexpr int kGatherThreads = 256;
constexpr int kGatherChunk = 8192;  // floats per CTA

__global__ void __launch_bounds__(kGatherThreads) traj_gather_kernel(
    const float* __restrict__ ring, int F, const int64_t* __restrict__ plan, const int32_t* __restrict__ colmap,
    float* __restrict__ batch, float* __restrict__ valid, int64_t Lmax, int skip) {
    const int64_t src = plan[blockIdx.x * 4 + 0], row = plan[blockIdx.x * 4 + 1], ptr = plan[blockIdx.x * 4 + 2],
                  len = plan[blockIdx.x * 4 + 3];
    const int start_col = colmap[0], mask_col = colmap[1], npairs = colmap[2];
    const int64_t total = len * F;
    const float* s = ring + src * F;
    float* d = batch + (row * Lmax + ptr + skip) * F;
    const int64_t e0 = (int64_t)blockIdx.y * kGatherChunk;
    if (e0 < total) {
        const int64_t e1 = min(total, e0 + (int64_t)kGatherChunk);
        const bool vec = ((reinterpret_cast<uintptr_t>(s + e0) | reinterpret_cast<uintptr_t>(d + e0)) & 15) == 0;
        if (vec) {
            const int64_t n4 = (e1 - e0) / 4;
            for (int64_t i = threadIdx.x; i < n4; i += kGatherThreads)
                reinterpret_cast<float4*>(d + e0)[i] = reinterpret_cast<const float4*>(s + e0)[i];
            for (int64_t e = e0 + n4 * 4 + threadIdx.x; e < e1; e += kGatherThreads) d[e] = s[e];
        } else {
            for (int64_t e = e0 + threadIdx.x; e < e1; e += kGatherThreads) d[e] = s[e];
        }
        // valid indicator for the steps whose first element falls in this chunk
        const int64_t s0 = (e0 + F - 1) / F, s1 = (e1 + F - 1) / F;
        for (int64_t st = s0 + threadIdx.x; st < s1 && st < len; st += kGatherThreads)
            valid[row * Lmax + ptr + skip + st] = s[st * F + mask_col];
    }
    if (blockIdx.y == 0) {
        for (int i = threadIdx.x; i < skip; i += kGatherThreads) batch[(row * Lmax + ptr + i) * F + start_col] = 1.0f;
        float* pre = batch + (row * Lmax + ptr + skip - 1) * F;
        for (int i = threadIdx.x; i < npairs; i += kGatherThreads) pre[colmap[3 + 2 * i]] = s[colmap[3 + 2 * i + 1]];
    }
}

__global__ void __launch_bounds__(kGatherThreads) traj_tail_kernel(const int64_t* __restrict__ row_end, int F,
                                                                    int start_col, float* __restrict__ batch,
                                                                    int64_t Lmax) {
    const int64_t row = blockIdx.x;
    for (int64_t t = row_end[row] + threadIdx.x; t < Lmax; t += kGatherThreads)
        batch[(row * Lmax + t) * F + start_col] = 1.0f;
}

}  // namespace rorl

using namespace rorl;

extern "C" {

// plan: device int64[ntraj*4 + rows] = (src_start, row, ptr, len) per placed trajectory, then row_end per row.
// colmap: device int32[3 + 2*npairs] = {start_col, mask_col, npairs, (dst_col, src_col)...}; start_col_host is
// the same start column, passed by value for the tail kernel.  max_len = longest trajectory in the plan.
int rorl_traj_gather(const float* ring, int64_t F, const int64_t* plan, int64_t ntraj, const int32_t* colmap,
                     int64_t start_col_host, float* batch, float* valid, int64_t rows, int64_t Lmax, int64_t skip,
                     int64_t max_len, cudaStream_t stream) {
    if (!ring || !plan || !colmap || !batch || !valid) return RORL_ERR_ARG;
    if (F <= 0 || ntraj <= 0 || rows <= 0 || Lmax <= 0 || skip < 1 || max_len <= 0 || ntraj > (1 << 30)) return RORL_ERR_SHAPE;
    cudaMemsetAsync(batch, 0, sizeof(float) * (size_t)rows * Lmax * F, stream);
    cudaMemsetAsync(valid, 0, sizeof(float) * (size_t)rows * Lmax, stream);
    int64_t chunks = (max_len * F + kGatherChunk - 1) / kGatherChunk;
    if (chunks > 65535) return RORL_ERR_SHAPE;
    dim3 grid((unsigned)ntraj, (unsigned)chunks);
    traj_gather_kernel<<<grid, kGatherThreads, 0, stream>>>(ring, (int)F, plan, colmap, batch, valid, Lmax, (int)skip);
    traj_tail_kernel<<<(unsigned)rows, kGatherThreads, 0, stream>>>(plan + ntraj * 4, (int)F, (int)start_col_host, batch, Lmax);
    RORL_RETURN_LAUNCH();
}

int rorl_abi_version(void) { return 6; }   // 6: rorl_gemm_tn / rorl_gemm_nt take passes 2 and 4 only (the TF32 forms are gone); K % 4 for every form

}  // extern "C"
