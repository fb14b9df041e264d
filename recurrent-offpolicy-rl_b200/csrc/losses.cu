// Fused target-Q / masked-TD / actor / entropy reductions over the valid-step mask.
// Replaces the chains of small ATen kernels and .item() syncs in
//   _target_Q            (ref: offpolicy_rnn/algorithm/sac_full_length_rnn_ensembleQ.py:83-103,
//                         REDQ subset sac_full_length_rnn_redq.py:28-32, TD3 td3_full_length_rnn_ensembleQ.py:23-46)
//   QValueGuard          (ref: offpolicy_rnn/utility/q_value_guard.py:22-38)
//   _Q_loss/_policy_loss/_alpha_loss/_mask_mean (ref: sac_full_length_rnn_ensembleQ.py:80-132,
//                         REDQ mean aggregate sac_full_length_rnn_redq.py:46)
//
// Every kernel is a deterministic two-level reduction: CTAs write partials to `work`, the last CTA
// to finish (ticket counter at the end of `work`) folds them in index order and resets the ticket,
// so the kernels are CUDA-graph replayable and need no host round trip.  The guard state lives on
// the device as double[4] = {min, max, initialised, decay}: the reference keeps it in Python floats
// (double), and the clamp bounds are cast to fp32 exactly where torch.clamp casts them.
#include "common.cuh"
#include <float.h>

namespace rorl {

constexpr int kLossThreads = 256;
constexpr int kLossMaxBlocks = 296;

__device__ __forceinline__ int loss_nblocks_dev() { return gridDim.x; }

// Block-reduce K values with op (0 = sum, 1 = min, 2 = max); result valid in thread 0.
template <int K>
__device__ __forceinline__ void block_reduce(float (&v)[K], const int (&op)[K], float* sbuf) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        float x = v[k];
        x = op[k] == 0 ? warp_sum(x) : (op[k] == 1 ? warp_min(x) : warp_max(x));
        if (lane == 0) sbuf[k * 8 + warp] = x;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float x = sbuf[k * 8];
            for (int w = 1; w < kLossThreads / 32; ++w) {
                float y = sbuf[k * 8 + w];
                x = op[k] == 0 ? x + y : (op[k] == 1 ? fminf(x, y) : fmaxf(x, y));
            }
            v[k] = x;
        }
    }
}

// Publish this CTA's partials; returns true (in thread 0 only) for the last CTA, with v = totals.
template <int K>
__device__ __forceinline__ bool grid_reduce(float (&v)[K], const int (&op)[K], float* work, float* sbuf) {
    block_reduce<K>(v, op, sbuf);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(work + kLossMaxBlocks * 8);
    bool last = false;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) work[blockIdx.x * 8 + k] = v[k];
        __threadfence();
        unsigned int t = atomicAdd(ticket, 1u);
        last = (t == gridDim.x - 1);
        if (last) {
            __threadfence();
#pragma unroll
            for (int k = 0; k < K; ++k) {
                float x = op[k] == 0 ? 0.f : (op[k] == 1 ? FLT_MAX : -FLT_MAX);
                for (unsigned int bI = 0; bI < gridDim.x; ++bI) {
                    float y = __ldcg(work + bI * 8 + k);
                    x = op[k] == 0 ? x + y : (op[k] == 1 ? fminf(x, y) : fmaxf(x, y));
                }
                v[k] = x;
            }
            *ticket = 0u;
        }
    }
    return last;
}

__global__ void __launch_bounds__(kLossThreads) target_minq_kernel(
    const float* __restrict__ q, const int32_t* __restrict__ sel, int nsel, int64_t M,
    const float* __restrict__ logp, const float* __restrict__ log_alpha, float* __restrict__ m, double* guard,
    float* work) {
    __shared__ float sbuf[64];
    const float alpha = (logp != nullptr) ? expf(log_alpha[0]) : 0.f;
    float v[2] = {FLT_MAX, -FLT_MAX};
    for (int64_t i = (int64_t)blockIdx.x * kLossThreads + threadIdx.x; i < M; i += (int64_t)gridDim.x * kLossThreads) {
        float mn = FLT_MAX;
        for (int s = 0; s < nsel; ++s) mn = fminf(mn, q[(int64_t)sel[s] * M + i]);
        if (logp) mn = mn - alpha * logp[i];
        m[i] = mn;
        v[0] = fminf(v[0], mn);
        v[1] = fmaxf(v[1], mn);
    }
    const int op[2] = {1, 2};
    if (grid_reduce<2>(v, op, work, sbuf)) {
        if (guard[2] == 0.0) {   // first clamp() call initialises the bounds from the tensor itself
            guard[0] = (double)v[0];
            guard[1] = (double)v[1];
            guard[2] = 1.0;
        }
    }
}

__global__ void __launch_bounds__(kLossThreads) target_finish_kernel(
    const float* __restrict__ m, const float* __restrict__ reward, const float* __restrict__ done,
    const float* __restrict__ timeout, const float* __restrict__ mask, float gamma, float* __restrict__ y,
    double* guard, float* __restrict__ stats, float* work, int64_t M) {
    __shared__ float sbuf[64];
    const float lo = (float)guard[0], hi = (float)guard[1];
    float v[4] = {FLT_MAX, -FLT_MAX, 0.f, 0.f};   // min(y*mask), max(y*mask), max|y|, sum(mask)
    for (int64_t i = (int64_t)blockIdx.x * kLossThreads + threadIdx.x; i < M; i += (int64_t)gridDim.x * kLossThreads) {
        float dn = (timeout != nullptr && timeout[i] > 0.f) ? 0.f : done[i];
        float c = fminf(fmaxf(m[i], lo), hi);
        float yy = reward[i] + (1.0f - dn) * gamma * c;
        y[i] = yy;
        float ym = yy * mask[i];
        v[0] = fminf(v[0], ym);
        v[1] = fmaxf(v[1], ym);
        v[2] = fmaxf(v[2], fabsf(yy));
        v[3] += mask[i];
    }
    const int op[4] = {1, 2, 2, 0};
    if (grid_reduce<4>(v, op, work, sbuf)) {
        const double vmin = (double)v[0], vmax = (double)v[1], decay = guard[3];
        double gmin = fmin(guard[0], vmin), gmax = fmax(guard[1], vmax);
        if (decay < 1.0) {
            gmin = decay * gmin + (1.0 - decay) * vmin;
            gmax = decay * gmax + (1.0 - decay) * vmax;
        }
        guard[0] = gmin;
        guard[1] = gmax;
        stats[0] = v[2];
        stats[1] = v[3];
    }
}

__global__ void __launch_bounds__(kLossThreads) q_loss_kernel(
    const float* __restrict__ q, const float* __restrict__ y, const float* __restrict__ mask,
    const float* __restrict__ nvalid, float* __restrict__ loss, float* __restrict__ dq, float* work, int E, int64_t M) {
    __shared__ float sbuf[64];
    const float inv = 1.0f / nvalid[0];
    float v[1] = {0.f};
    for (int64_t i = (int64_t)blockIdx.x * kLossThreads + threadIdx.x; i < M; i += (int64_t)gridDim.x * kLossThreads) {
        const float yy = y[i], mk = mask[i];
        float s = 0.f;
        for (int e = 0; e < E; ++e) {
            float df = q[(int64_t)e * M + i] - yy;
            s = fmaf(df, df, s);
            dq[(int64_t)e * M + i] = 2.0f * mk * df * inv;
        }
        v[0] = fmaf(s, mk, v[0]);
    }
    const int op[1] = {0};
    if (grid_reduce<1>(v, op, work, sbuf)) loss[0] = v[0] * inv;
}

__global__ void __launch_bounds__(kLossThreads) actor_loss_kernel(
    const float* __restrict__ q, const float* __restrict__ logp, const float* __restrict__ mask,
    const float* __restrict__ nvalid, const float* __restrict__ log_alpha, float target_entropy, int mode,
    float* __restrict__ out, float* __restrict__ dq, float* __restrict__ dlogp, float* work, int E, int64_t M) {
    __shared__ float sbuf[64];
    const float inv = 1.0f / nvalid[0];
    const float la = log_alpha ? log_alpha[0] : 0.f;
    const float alpha = logp ? expf(la) : 0.f;
    float v[3] = {0.f, 0.f, 0.f};   // sum mask*(alpha*logp - agg), sum mask*logp, sum mask*(logp + H)
    for (int64_t i = (int64_t)blockIdx.x * kLossThreads + threadIdx.x; i < M; i += (int64_t)gridDim.x * kLossThreads) {
        const float mk = mask[i];
        float agg;
        if (mode == 0) {
            int arg = 0;
            agg = q[i];
            for (int e = 1; e < E; ++e) {
                float qq = q[(int64_t)e * M + i];
                if (qq < agg) { agg = qq; arg = e; }
            }
            for (int e = 0; e < E; ++e) dq[(int64_t)e * M + i] = (e == arg) ? -mk * inv : 0.f;
        } else {
            float s = 0.f;
            for (int e = 0; e < E; ++e) s += q[(int64_t)e * M + i];
            agg = s / (float)E;
            const float gq = -mk * inv / (float)E;
            for (int e = 0; e < E; ++e) dq[(int64_t)e * M + i] = gq;
        }
        float lp = 0.f;
        if (logp) {
            lp = logp[i];
            dlogp[i] = alpha * mk * inv;
        }
        v[0] = fmaf(mk, alpha * lp - agg, v[0]);
        v[1] = fmaf(mk, lp, v[1]);
        v[2] = fmaf(mk, lp + target_entropy, v[2]);
    }
    const int op[3] = {0, 0, 0};
    if (grid_reduce<3>(v, op, work, sbuf)) {
        out[0] = v[0] * inv;
        out[1] = v[1] * inv;
        out[2] = -la * (v[2] * inv);
        out[3] = -(v[2] * inv);
    }
}

// Discrete actions ([E, M, A] Q, [M, A] log-probabilities): one warp per row i, lanes over the actions, so that each
// row's expectation over actions is one fixed-order warp sum.  Rows are strided over the warps of the grid.
constexpr int kLossWarps = kLossThreads / 32;

__global__ void __launch_bounds__(kLossThreads) discrete_target_expect_kernel(
    const float* __restrict__ q, const int32_t* __restrict__ sel, int nsel, int64_t M, int A,
    const float* __restrict__ logp, const float* __restrict__ log_alpha, float* __restrict__ m, double* guard, float* work) {
    __shared__ float sbuf[64];
    const int lane = threadIdx.x & 31;
    const float alpha = expf(log_alpha[0]);
    float v[2] = {FLT_MAX, -FLT_MAX};
    for (int64_t i = (int64_t)blockIdx.x * kLossWarps + (threadIdx.x >> 5); i < M; i += (int64_t)gridDim.x * kLossWarps) {
        float acc = 0.f;
        for (int a = lane; a < A; a += 32) {
            float mn = FLT_MAX;
            for (int s = 0; s < nsel; ++s) mn = fminf(mn, q[((int64_t)sel[s] * M + i) * A + a]);
            const float lp = logp[i * A + a];
            acc = fmaf(mn - alpha * lp, expf(lp), acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) {   // lanes hold the sum in different association orders: lane 0's is the one written
            m[i] = acc;
            v[0] = fminf(v[0], acc);
            v[1] = fmaxf(v[1], acc);
        }
    }
    const int op[2] = {1, 2};
    if (grid_reduce<2>(v, op, work, sbuf)) {
        if (guard[2] == 0.0) {   // first clamp() call initialises the bounds from the tensor itself
            guard[0] = (double)v[0];
            guard[1] = (double)v[1];
            guard[2] = 1.0;
        }
    }
}

__global__ void __launch_bounds__(kLossThreads) discrete_actor_loss_kernel(
    const float* __restrict__ q, const float* __restrict__ logp, const float* __restrict__ mask,
    const float* __restrict__ nvalid, const float* __restrict__ log_alpha, int mode, float* __restrict__ out,
    float* __restrict__ dlogp, float* work, int E, int64_t M, int A) {
    __shared__ float sbuf[64];
    const int lane = threadIdx.x & 31;
    const float inv = 1.0f / nvalid[0];
    const float alpha = expf(log_alpha[0]);
    float v[2] = {0.f, 0.f};   // sum_i mask_i sum_a p (alpha logp - agg), sum_i mask_i sum_a p logp
    for (int64_t i = (int64_t)blockIdx.x * kLossWarps + (threadIdx.x >> 5); i < M; i += (int64_t)gridDim.x * kLossWarps) {
        const float mk = mask[i];
        const float g = mk * inv;
        float r = 0.f, h = 0.f;
        for (int a = lane; a < A; a += 32) {
            float agg;
            if (mode == 0) {
                agg = q[i * A + a];
                for (int e = 1; e < E; ++e) agg = fminf(agg, q[((int64_t)e * M + i) * A + a]);
            } else {
                float s = 0.f;
                for (int e = 0; e < E; ++e) s += q[((int64_t)e * M + i) * A + a];
                agg = s / (float)E;
            }
            const float lp = logp[i * A + a], p = expf(lp);
            const float t = alpha * lp - agg;
            r = fmaf(p, t, r);
            h = fmaf(p, lp, h);
            dlogp[i * A + a] = g * p * (t + alpha);
        }
        r = warp_sum(r);
        h = warp_sum(h);
        if (lane == 0) {
            v[0] = fmaf(mk, r, v[0]);
            v[1] = fmaf(mk, h, v[1]);
        }
    }
    const int op[2] = {0, 0};
    if (grid_reduce<2>(v, op, work, sbuf)) {
        out[0] = v[0] * inv;
        out[1] = v[1] * inv;
    }
}

__global__ void __launch_bounds__(kLossThreads) sumsq_kernel(const float* __restrict__ p, int64_t n, float* out,
                                                              float* work) {
    __shared__ float sbuf[64];
    float v[1] = {0.f};
    for (int64_t i = (int64_t)blockIdx.x * kLossThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kLossThreads)
        v[0] = fmaf(p[i], p[i], v[0]);
    const int op[1] = {0};
    if (grid_reduce<1>(v, op, work, sbuf)) out[0] = v[0];
}

static int loss_grid(int64_t M) {
    int64_t nb = (M + kLossThreads - 1) / kLossThreads;
    if (nb > kLossMaxBlocks) nb = kLossMaxBlocks;
    if (nb < 1) nb = 1;
    return (int)nb;
}

static int loss_grid_rows(int64_t M) { return loss_grid((M + kLossWarps - 1) / kLossWarps * kLossThreads); }

}  // namespace rorl

using namespace rorl;

extern "C" {

int64_t rorl_loss_work_floats(int64_t /*M*/) { return kLossMaxBlocks * 8 + 4; }

int rorl_target_minq(const float* q, const int32_t* sel, int64_t nsel, int64_t E, int64_t M, const float* logp,
                     const float* log_alpha, float* m, double* guard, float* work, cudaStream_t stream) {
    if (!q || !sel || !m || !guard || !work) return RORL_ERR_ARG;
    if (logp && !log_alpha) return RORL_ERR_ARG;
    if (nsel <= 0 || nsel > E || M <= 0) return RORL_ERR_SHAPE;
    target_minq_kernel<<<loss_grid(M), kLossThreads, 0, stream>>>(q, sel, (int)nsel, M, logp, log_alpha, m, guard, work);
    RORL_RETURN_LAUNCH();
}

int rorl_target_finish(const float* m, const float* reward, const float* done, const float* timeout,
                       const float* mask, float gamma, float* y, double* guard, float* stats, float* work,
                       int64_t M, cudaStream_t stream) {
    if (!m || !reward || !done || !mask || !y || !guard || !stats || !work) return RORL_ERR_ARG;
    if (M <= 0) return RORL_ERR_SHAPE;
    target_finish_kernel<<<loss_grid(M), kLossThreads, 0, stream>>>(m, reward, done, timeout, mask, gamma, y, guard,
                                                                   stats, work, M);
    RORL_RETURN_LAUNCH();
}

int rorl_q_loss_fwd_bwd(const float* q, const float* y, const float* mask, const float* nvalid, float* loss,
                        float* dq, float* work, int64_t E, int64_t M, cudaStream_t stream) {
    if (!q || !y || !mask || !nvalid || !loss || !dq || !work) return RORL_ERR_ARG;
    if (E <= 0 || M <= 0) return RORL_ERR_SHAPE;
    q_loss_kernel<<<loss_grid(M), kLossThreads, 0, stream>>>(q, y, mask, nvalid, loss, dq, work, (int)E, M);
    RORL_RETURN_LAUNCH();
}

int rorl_actor_loss_fwd_bwd(const float* q, const float* logp, const float* mask, const float* nvalid,
                            const float* log_alpha, float target_entropy, int mode, float* out, float* dq,
                            float* dlogp, float* work, int64_t E, int64_t M, cudaStream_t stream) {
    if (!q || !mask || !nvalid || !out || !dq || !work) return RORL_ERR_ARG;
    if (logp && (!dlogp || !log_alpha)) return RORL_ERR_ARG;
    if (E <= 0 || M <= 0 || (mode != 0 && mode != 1)) return RORL_ERR_SHAPE;
    actor_loss_kernel<<<loss_grid(M), kLossThreads, 0, stream>>>(q, logp, mask, nvalid, log_alpha, target_entropy, mode,
                                                                out, dq, dlogp, work, (int)E, M);
    RORL_RETURN_LAUNCH();
}

int rorl_discrete_target_expect(const float* q, const int32_t* sel, int64_t nsel, int64_t E, int64_t M, int64_t A,
                                const float* logp, const float* log_alpha, float* m, double* guard, float* work,
                                cudaStream_t stream) {
    if (!q || !sel || !logp || !log_alpha || !m || !guard || !work) return RORL_ERR_ARG;
    if (nsel <= 0 || nsel > E || M <= 0 || A < 1 || A > 256) return RORL_ERR_SHAPE;
    discrete_target_expect_kernel<<<loss_grid_rows(M), kLossThreads, 0, stream>>>(q, sel, (int)nsel, M, (int)A, logp,
                                                                                  log_alpha, m, guard, work);
    RORL_RETURN_LAUNCH();
}

int rorl_discrete_actor_loss_fwd_bwd(const float* q, const float* logp, const float* mask, const float* nvalid,
                                     const float* log_alpha, int mode, float* out, float* dlogp, float* work, int64_t E,
                                     int64_t M, int64_t A, cudaStream_t stream) {
    if (!q || !logp || !mask || !nvalid || !log_alpha || !out || !dlogp || !work) return RORL_ERR_ARG;
    if (E <= 0 || M <= 0 || A < 1 || A > 256 || (mode != 0 && mode != 1)) return RORL_ERR_SHAPE;
    discrete_actor_loss_kernel<<<loss_grid_rows(M), kLossThreads, 0, stream>>>(q, logp, mask, nvalid, log_alpha, mode, out,
                                                                               dlogp, work, (int)E, M, (int)A);
    RORL_RETURN_LAUNCH();
}

int rorl_sumsq(const float* p, int64_t n, float* out, float* work, cudaStream_t stream) {
    if (!p || !out || !work) return RORL_ERR_ARG;
    if (n <= 0) return RORL_ERR_SHAPE;
    sumsq_kernel<<<loss_grid(n), kLossThreads, 0, stream>>>(p, n, out, work);
    RORL_RETURN_LAUNCH();
}

}  // extern "C"
