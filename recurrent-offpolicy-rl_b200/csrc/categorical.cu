// Categorical policy head of the discrete-action SAC policy, forward and backward, one kernel each (sm_100a).
//
// Replaces the ATen chain of ContextualSACDiscretePolicy.process_model_out and its autograd graph
// (ref: offpolicy_rnn/policy_value_models/contextual_sac_discrete_policy.py:106-111):
//   s = softmax(z);  p = (s + 0.01) / sum_a (s + 0.01);  logp = log p
//   mode   = argmax_a p, the first index winning ties (torch.argmax)
//   sample = the first a with cumsum(p)[a] > u * sum(p)   (inverse-CDF draw from one uniform u per row)
// Backward, the closed form of autograd through those ops.  With T = sum_a (s + 0.01) (= 1 + 0.01 A up to rounding):
//   dL/dp = d_logp / p;  dL/ds_a = (dL/dp_a) / T - sum_b (dL/dp_b) p_b / T.
// The second term is the same for every a, and the softmax Jacobian (dz = s * (g - sum s g)) removes any constant added
// to g, so the gradient through the renormalising sum vanishes and
//   dz = s * (v - sum_a s v),   v = d_logp / p / T              (exact up to rounding).
// The backward recomputes s, p and T from the logits; nothing is saved.
//
// One warp per row.  Lane l holds the contiguous columns [l K, l K + K), K = ceil(A / 32) <= 8, so the prefix sum of the
// inverse-CDF search is a per-lane running sum plus one warp scan.  All reductions are fixed-order warp shuffles: the
// kernels are deterministic, use no atomics and no host synchronisation.  Precise expf / logf: logp enters the losses.
#include "common.cuh"

namespace rorl {

constexpr int kCatRowsPerBlock = 8;   // 256 threads
constexpr int kCatPer = 8;            // columns per lane at the largest A (256)
constexpr float kCatFloor = 0.01f;    // exploration floor (ref :108-109)

// A butterfly warp sum leaves each lane with its own association order; every lane takes lane 0's sum, so that equal
// logits in different lanes get bit-equal probabilities (ties stay ties for the argmax).
__device__ __forceinline__ float warp_sum_uniform(float v) { return __shfl_sync(0xffffffffu, warp_sum(v), 0); }

// s (softmax) and p (floored, renormalised) of one row, columns [lane K, lane K + K); invalid slots hold 0.  tsum = T.
__device__ __forceinline__ void cat_row(const float* __restrict__ z, int A, int K, int lane, float (&s)[kCatPer],
                                        float (&p)[kCatPer], float& tsum) {
    const int a0 = lane * K;
    float mx = -INFINITY;
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) {
        s[k] = (k < K && a0 + k < A) ? z[a0 + k] : -INFINITY;
        mx = fmaxf(mx, s[k]);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) {
        s[k] = (k < K && a0 + k < A) ? expf(s[k] - mx) : 0.f;
        sum += s[k];
    }
    sum = warp_sum_uniform(sum);
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) {
        const bool ok = k < K && a0 + k < A;
        s[k] = ok ? s[k] / sum : 0.f;
        p[k] = ok ? s[k] + kCatFloor : 0.f;
        t += p[k];
    }
    tsum = warp_sum_uniform(t);
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) p[k] = p[k] / tsum;   // invalid slots stay 0
}

__global__ void __launch_bounds__(kCatRowsPerBlock * 32) categorical_fwd_kernel(
    const float* __restrict__ logits, int64_t ld, const float* __restrict__ u, float* __restrict__ probs,
    float* __restrict__ logp, float* __restrict__ mode, float* __restrict__ sample, int64_t M, int A) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kCatRowsPerBlock + (threadIdx.x >> 5);
    if (row >= M) return;                      // whole warps leave together
    const int K = (A + 31) >> 5, a0 = lane * K;
    float s[kCatPer], p[kCatPer], tsum;
    cat_row(logits + row * ld, A, K, lane, s, p, tsum);
    float best = -INFINITY;
    int arg = A;
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) {
        const int a = a0 + k;
        if (k < K && a < A) {
            probs[row * A + a] = p[k];
            logp[row * A + a] = logf(p[k]);
            if (p[k] > best) { best = p[k]; arg = a; }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {         // (larger p, then smaller index) wins
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
    }
    if (lane == 0) mode[row] = (float)arg;
    if (u == nullptr) return;
    float run = 0.f;
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) run += p[k];
    float incl = run;                          // inclusive scan of the lane totals
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    const float total = __shfl_sync(0xffffffffu, incl, 31);
    float c = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) c = 0.f;
    const float thr = u[row] * total;
    int first = A;
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) {
        const int a = a0 + k;
        c += p[k];
        if (k < K && a < A && first == A && c > thr) first = a;
    }
    first = __reduce_min_sync(0xffffffffu, first);
    if (lane == 0) sample[row] = (float)(first < A ? first : A - 1);   // u * total rounded up to total: the last action
}

__global__ void __launch_bounds__(kCatRowsPerBlock * 32) categorical_bwd_kernel(
    const float* __restrict__ logits, int64_t ld, const float* __restrict__ d_logp, float* __restrict__ d_logits, int64_t M,
    int A) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kCatRowsPerBlock + (threadIdx.x >> 5);
    if (row >= M) return;
    const int K = (A + 31) >> 5, a0 = lane * K;
    float s[kCatPer], p[kCatPer], tsum;
    cat_row(logits + row * ld, A, K, lane, s, p, tsum);
    float v[kCatPer], dot = 0.f;
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) {
        const int a = a0 + k;
        v[k] = (k < K && a < A) ? d_logp[row * A + a] / p[k] / tsum : 0.f;
        dot = fmaf(s[k], v[k], dot);
    }
    dot = warp_sum_uniform(dot);
#pragma unroll
    for (int k = 0; k < kCatPer; ++k) {
        const int a = a0 + k;
        if (k < K && a < A) d_logits[row * A + a] = s[k] * (v[k] - dot);
    }
}

static inline unsigned cat_grid(int64_t M) { return (unsigned)((M + kCatRowsPerBlock - 1) / kCatRowsPerBlock); }

}  // namespace rorl

using namespace rorl;

extern "C" {

int rorl_categorical_fwd(const float* logits, int64_t ld, const float* u, float* probs, float* logp, float* mode,
                         float* sample, int64_t M, int64_t A, cudaStream_t stream) {
    if (!logits || !probs || !logp || !mode || (u && !sample)) return RORL_ERR_ARG;
    if (M < 0 || A < 1 || A > 256 || ld < A) return RORL_ERR_SHAPE;
    if (M == 0) return RORL_OK;
    categorical_fwd_kernel<<<cat_grid(M), kCatRowsPerBlock * 32, 0, stream>>>(logits, ld, u, probs, logp, mode, sample, M,
                                                                              (int)A);
    RORL_RETURN_LAUNCH();
}

int rorl_categorical_bwd(const float* logits, int64_t ld, const float* d_logp, float* d_logits, int64_t M, int64_t A,
                         cudaStream_t stream) {
    if (!logits || !d_logp || !d_logits) return RORL_ERR_ARG;
    if (M < 0 || A < 1 || A > 256 || ld < A) return RORL_ERR_SHAPE;
    if (M == 0) return RORL_OK;
    categorical_bwd_kernel<<<cat_grid(M), kCatRowsPerBlock * 32, 0, stream>>>(logits, ld, d_logp, d_logits, M, (int)A);
    RORL_RETURN_LAUNCH();
}

}  // extern "C"
