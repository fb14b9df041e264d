// Decode-step kernels: what one environment step of the policy (L = 1, a handful of rows) runs (sm_100a).
//
// rorl_small_linear: y[g][m, n] = act(bias[g][n] + sum_k x[g][m, k] W[g](n, k)) for M <= 64 rows in true fp32 on the FMA
// pipe.  A 128-row tensor-core tile would compute one to a few real rows there, and cuBLAS picks a different kernel per
// shape.  Here every weight is read once, coalesced, while the x rows sit in shared memory, tiled along K:
//   layout 0 (nn.Linear, W [N, K]): one warp per output column, lane l takes k = l, l + 32, ... in increasing order, then
//     a fixed xor-butterfly over the 32 lanes;
//   layout 1 (EnsembleLinear, W [G, K, N]): lane <-> output column, the block's 4 warps take interleaved k (k % 4), then
//     their partial sums are added in warp order.
// The summation order along K is a property of the block shape only, never of the grid: results are deterministic.
//
// rorl_mamba_step_conv / rorl_mamba_step_ssm: the smamba mixer's single-step path (ref: smamba/mamba.py Mamba.step):
//   conv: window <- roll left + append xs;  u = silu(sum_j window[j] w[j] + b)       one thread per (row, channel)
//   ssm:  delta = softplus(x_dbl[:R] . Wdt[d] + b_dt[d]);  A = -exp(A_log)
//         h <- exp(delta A) h + delta u B;  y = (C . h + D u) silu(z)               one warp per (row, channel), lane <-> n
// The carried window / state may be updated in place (in == out) or written to a new buffer.
#include "common.cuh"

namespace rorl {

constexpr int kSlKt0 = 128;   // layout 0: K-tile of the staged x rows
constexpr int kSlKt1 = 32;    // layout 1: K-tile of the staged x rows
constexpr int kSlWarps1 = 4;  // layout 1: warps splitting K inside a block

__device__ __forceinline__ float elu_exact(float v) { return v > 0.f ? v : expm1f(v); }

template <int MT>
__global__ void __launch_bounds__(256) small_linear_nk_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ W,
                                                              const float* __restrict__ bias, float* __restrict__ y, int64_t ldy,
                                                              int M, int N, int K, int elu) {
    __shared__ float xs[MT][kSlKt0];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = blockIdx.x * 8 + warp;
    const float* w = W + (int64_t)(n < N ? n : 0) * K;
    float acc[MT];
#pragma unroll
    for (int m = 0; m < MT; ++m) acc[m] = 0.f;
    for (int k0 = 0; k0 < K; k0 += kSlKt0) {
        const int kt = min(kSlKt0, K - k0);
        __syncthreads();
        for (int i = threadIdx.x; i < MT * kSlKt0; i += 256) {
            const int m = i / kSlKt0, k = i % kSlKt0;
            xs[m][k] = (m < M && k < kt) ? x[(int64_t)m * ldx + k0 + k] : 0.f;
        }
        __syncthreads();
        if (n < N) {
#pragma unroll
            for (int j = 0; j < kSlKt0 / 32; ++j) {
                const int k = lane + 32 * j;
                if (k < kt) {
                    const float wv = __ldg(w + k0 + k);
#pragma unroll
                    for (int m = 0; m < MT; ++m) acc[m] = fmaf(xs[m][k], wv, acc[m]);
                }
            }
        }
    }
    if (n >= N) return;
#pragma unroll
    for (int m = 0; m < MT; ++m) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[m] += __shfl_xor_sync(0xffffffffu, acc[m], o);
    }
    const float b = bias ? bias[n] : 0.f;
#pragma unroll
    for (int m = 0; m < MT; ++m) {
        if (m < M && (m & 31) == lane) {
            const float v = acc[m] + b;
            y[(int64_t)m * ldy + n] = elu ? elu_exact(v) : v;
        }
    }
}

template <int MT>
__global__ void __launch_bounds__(128) small_linear_gkn_kernel(const float* __restrict__ x, int64_t ldx, int64_t x_gstride,
                                                               const float* __restrict__ W, const float* __restrict__ bias,
                                                               float* __restrict__ y, int64_t ldy, int M, int N, int K, int elu) {
    __shared__ float xs[MT][kSlKt1];
    __shared__ float part[kSlWarps1][MT][32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.y;
    const int n = blockIdx.x * 32 + lane;
    const float* xg = x + (int64_t)g * x_gstride;
    const float* wg = W + (int64_t)g * K * N;
    float acc[MT];
#pragma unroll
    for (int m = 0; m < MT; ++m) acc[m] = 0.f;
    for (int k0 = 0; k0 < K; k0 += kSlKt1) {
        const int kt = min(kSlKt1, K - k0);
        __syncthreads();
        for (int i = threadIdx.x; i < MT * kSlKt1; i += 128) {
            const int m = i / kSlKt1, k = i % kSlKt1;
            xs[m][k] = (m < M && k < kt) ? xg[(int64_t)m * ldx + k0 + k] : 0.f;
        }
        __syncthreads();
        if (n < N) {
            for (int k = warp; k < kt; k += kSlWarps1) {
                const float wv = __ldg(wg + (int64_t)(k0 + k) * N + n);
#pragma unroll
                for (int m = 0; m < MT; ++m) acc[m] = fmaf(xs[m][k], wv, acc[m]);
            }
        }
    }
#pragma unroll
    for (int m = 0; m < MT; ++m) part[warp][m][lane] = acc[m];
    __syncthreads();
    const float b = (bias && n < N) ? bias[(int64_t)g * N + n] : 0.f;
    for (int m = warp; m < M; m += kSlWarps1) {
        if (n >= N) break;
        float v = part[0][m][lane];
#pragma unroll
        for (int w = 1; w < kSlWarps1; ++w) v += part[w][m][lane];
        v += b;
        y[((int64_t)g * M + m) * ldy + n] = elu ? elu_exact(v) : v;
    }
}

template <int MT>
static void launch_small_linear(const float* x, int64_t ldx, int64_t x_gstride, const float* W, const float* bias, float* y,
                                int64_t ldy, int M, int N, int K, int G, int layout, int elu, cudaStream_t s) {
    if (layout == 0) {
        small_linear_nk_kernel<MT><<<(unsigned)((N + 7) / 8), 256, 0, s>>>(x, ldx, W, bias, y, ldy, M, N, K, elu);
    } else {
        dim3 grid((unsigned)((N + 31) / 32), (unsigned)G);
        small_linear_gkn_kernel<MT><<<grid, 128, 0, s>>>(x, ldx, x_gstride, W, bias, y, ldy, M, N, K, elu);
    }
}

__device__ __forceinline__ float silu_exact(float v) { return v / (1.f + expf(-v)); }
__device__ __forceinline__ float softplus_exact(float v) { return v > 20.f ? v : log1pf(expf(v)); }

__global__ void __launch_bounds__(256) mamba_step_conv_kernel(const float* __restrict__ xz, int64_t ld_xz, const float* __restrict__ w,
                                                              const float* __restrict__ b, const float* win_in, int64_t ld_in,
                                                              float* win_out, int64_t ld_out, float* __restrict__ u, int B, int D,
                                                              int Kc) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= (int64_t)B * D) return;
    const int r = (int)(i / D), d = (int)(i % D);
    const float* src = win_in + (int64_t)r * ld_in + (int64_t)d * Kc;
    float* dst = win_out + (int64_t)r * ld_out + (int64_t)d * Kc;
    const float* wd = w + (int64_t)d * Kc;
    float acc = 0.f;
    // read position j + 1 before writing position j: safe when src == dst
    for (int j = 0; j + 1 < Kc; ++j) {
        const float v = src[j + 1];
        acc = fmaf(v, wd[j], acc);
        dst[j] = v;
    }
    const float xn = xz[(int64_t)r * ld_xz + d];
    acc = fmaf(xn, wd[Kc - 1], acc);
    dst[Kc - 1] = xn;
    if (b) acc += b[d];
    u[i] = silu_exact(acc);
}

__global__ void __launch_bounds__(256) mamba_step_ssm_kernel(const float* __restrict__ u, const float* __restrict__ xdbl, int64_t ld_xdbl,
                                                             const float* __restrict__ z, int64_t ld_z, const float* __restrict__ wdt,
                                                             const float* __restrict__ bdt, const float* __restrict__ a_log,
                                                             const float* __restrict__ dskip, const float* h_in, int64_t ld_hin,
                                                             float* h_out, int64_t ld_hout, float* __restrict__ y, int B, int D,
                                                             int R, int Ns) {
    const int64_t wi = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wi >= (int64_t)B * D) return;
    const int r = (int)(wi / D), d = (int)(wi % D);
    const float* xr = xdbl + (int64_t)r * ld_xdbl;
    const float* wd = wdt + (int64_t)d * R;
    float dr = 0.f;
    for (int k = 0; k < R; ++k) dr = fmaf(xr[k], wd[k], dr);
    const float delta = softplus_exact(dr + bdt[d]);
    const float uv = u[wi];
    const float du = delta * uv;
    const float* hs = h_in + (int64_t)r * ld_hin + (int64_t)d * Ns;
    float* hd = h_out + (int64_t)r * ld_hout + (int64_t)d * Ns;
    const float* al = a_log + (int64_t)d * Ns;
    float acc = 0.f;
    for (int n = lane; n < Ns; n += 32) {
        const float a = -expf(al[n]);
        const float h = fmaf(expf(delta * a), hs[n], du * xr[R + n]);
        hd[n] = h;
        acc = fmaf(xr[R + Ns + n], h, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
        const float out = fmaf(dskip ? dskip[d] : 0.f, uv, acc);
        y[wi] = out * silu_exact(z[(int64_t)r * ld_z + d]);
    }
}

}  // namespace rorl

using namespace rorl;

extern "C" {

int rorl_small_linear(const float* x, int64_t ldx, int64_t x_gstride, const float* W, const float* bias, float* y, int64_t ldy,
                      int64_t M, int64_t N, int64_t K, int64_t G, int layout, int elu, cudaStream_t stream) {
    if (!x || !W || !y) return RORL_ERR_ARG;
    if (layout != 0 && layout != 1) return RORL_ERR_ARG;
    if (M < 1 || M > 64 || N < 1 || K < 1 || G < 1 || G > 65535 || N > (1 << 30) || K > (1 << 30)) return RORL_ERR_SHAPE;
    if (layout == 0 && (G != 1 || x_gstride != 0)) return RORL_ERR_ARG;
    if (ldx < K || ldy < N || x_gstride < 0) return RORL_ERR_SHAPE;
    const int m = (int)M, n = (int)N, k = (int)K, g = (int)G;
    if (m <= 1)
        launch_small_linear<1>(x, ldx, x_gstride, W, bias, y, ldy, m, n, k, g, layout, elu, stream);
    else if (m <= 4)
        launch_small_linear<4>(x, ldx, x_gstride, W, bias, y, ldy, m, n, k, g, layout, elu, stream);
    else if (m <= 16)
        launch_small_linear<16>(x, ldx, x_gstride, W, bias, y, ldy, m, n, k, g, layout, elu, stream);
    else
        launch_small_linear<64>(x, ldx, x_gstride, W, bias, y, ldy, m, n, k, g, layout, elu, stream);
    RORL_RETURN_LAUNCH();
}

int rorl_mamba_step_conv(const float* xz, int64_t ld_xz, const float* conv_w, const float* conv_b, const float* win_in,
                         int64_t ld_win_in, float* win_out, int64_t ld_win_out, float* u, int64_t B, int64_t D, int64_t Kc,
                         cudaStream_t stream) {
    if (!xz || !conv_w || !win_in || !win_out || !u) return RORL_ERR_ARG;
    if (B < 1 || D < 1 || Kc < 1 || Kc > 1024 || B * D > ((int64_t)1 << 31)) return RORL_ERR_SHAPE;
    if (ld_xz < D || ld_win_in < D * Kc || ld_win_out < D * Kc) return RORL_ERR_SHAPE;
    const int64_t n = B * D;
    mamba_step_conv_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(xz, ld_xz, conv_w, conv_b, win_in, ld_win_in, win_out,
                                                                            ld_win_out, u, (int)B, (int)D, (int)Kc);
    RORL_RETURN_LAUNCH();
}

int rorl_mamba_step_ssm(const float* u, const float* x_dbl, int64_t ld_xdbl, const float* z, int64_t ld_z, const float* dt_w,
                        const float* dt_b, const float* A_log, const float* Dskip, const float* h_in, int64_t ld_h_in, float* h_out,
                        int64_t ld_h_out, float* y, int64_t B, int64_t D, int64_t R, int64_t Ns, cudaStream_t stream) {
    if (!u || !x_dbl || !z || !dt_w || !dt_b || !A_log || !h_in || !h_out || !y) return RORL_ERR_ARG;
    if (B < 1 || D < 1 || R < 1 || Ns < 1 || Ns > 4096 || R > 4096 || B * D > ((int64_t)1 << 26)) return RORL_ERR_SHAPE;
    if (ld_xdbl < R + 2 * Ns || ld_z < D || ld_h_in < D * Ns || ld_h_out < D * Ns) return RORL_ERR_SHAPE;
    const int64_t threads = B * D * 32;
    mamba_step_ssm_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(u, x_dbl, ld_xdbl, z, ld_z, dt_w, dt_b, A_log, Dskip,
                                                                                 h_in, ld_h_in, h_out, ld_h_out, y, (int)B, (int)D,
                                                                                 (int)R, (int)Ns);
    RORL_RETURN_LAUNCH();
}

}  // extern "C"
