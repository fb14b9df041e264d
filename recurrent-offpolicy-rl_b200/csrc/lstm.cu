// LSTM recurrence as a PERSISTENT thread-block-cluster kernel, forward and backward, sm_100a.
//
//   gates = gi + W_hh h + b_hh   (gi = x W_ih^T + b_ih; gate order i, f, g, o as in torch.nn.LSTM)
//   i = sigmoid(a_i)  f = sigmoid(a_f)  g = tanh(a_g)  o = sigmoid(a_o)
//   c' = f * c + i * g            h' = o * tanh(c')
//
// Replaces torch.nn.LSTM(in, H, batch_first=True) on the `lstm` encoder path (ref: offpolicy_rnn/models/rnn_base.py,
// layer table entry 'lstm'; cuDNN on GPU, ATen loop on CPU).  gi for all steps is ONE tensor-core GEMM up front
// (csrc/gemm_bf16.cu); this file is the L dependent steps that remain.
//
// Design.  W_hh is 4H x H fp32 = 1 MiB at H = 256, four times one SM's shared memory and four times its register
// file.  The GRU's split (csrc/gru.cu: 64 units per CTA) would need a whole register file per CTA for weights alone,
// so the LSTM halves the units per CTA: a cluster of CL = H / 32 CTAs (8 at H = 256, the portable maximum) owns
// W_hh, CTA `rank` owns hidden units [32 rank, 32 rank + 32), and its 512 threads are 32 units x 16 K-slices.
// Thread (unit j, slice ks) keeps the 4 x H/16 weights W_h{i,f,g,o}[j, ks*H/16 ...] in registers (64 at H = 256)
// for the whole sequence.  Per step, as in the GRU:
//   (1) every thread multiplies its weight slice with h_{t-1} (a warp is 32 units x one K-slice, so the h read is a
//       shared-memory broadcast) and leaves 4 x BG partial sums in shared memory;
//   (2) __syncthreads; 32 x BG owner threads add the 16 partials, apply the gates, keep c_t in a register, write h_t
//       and the saved activations to HBM and push h_t into every CTA of the cluster through distributed shared memory;
//   (3) one cluster barrier publishes h_t; h is double buffered, so that is the only cluster-wide sync per step.
// One cluster serves BG batch rows; the number of clusters comes from cudaOccupancyMaxActiveClusters (8-CTA
// clusters must fit inside a GPC, so fewer are co-resident than 148 / 8).
//
// Backward walks the steps in reverse with the transposed product dh_{t-1} = W_hh^T da_t in the same shape: thread
// (unit j, slice ks) keeps W_hh[ks*4H/16 ..., j] (64 registers), and the broadcast vector is da_t = d(gates) [4H].
// It emits da [B, L, 4H] (= d gi) plus dh0, dc0; the weight gradients are GEMMs over all steps (host side).
// No atomics anywhere: every sum has a fixed order, so graph replays are bit-identical to eager launches.
#include "common.cuh"
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace rorl {

template <int H_>
struct LstmCfg {
    static constexpr int H = H_;
    static constexpr int UNITS = H_ >= 32 ? 32 : H_;          // hidden units per CTA
    static constexpr int KS = H_ >= 64 ? 16 : H_ / 4;         // K slices per unit
    static constexpr int NT = UNITS * KS;                     // threads per CTA (512 at H >= 64)
    static constexpr int CL = H_ / UNITS;                     // CTAs per cluster
    static_assert(H_ % UNITS == 0 && (H_ / KS) % 4 == 0 && (4 * H_ / KS) % 4 == 0, "unsupported hidden size");
};

struct LstmFwdParams {
    const float *gi, *w_hh, *b_hh, *h0, *c0;
    float *out, *save, *h_last, *c_last;
    int B, L, nclusters;
};

template <int H, int BG>
__global__ void __launch_bounds__(LstmCfg<H>::NT, 1) lstm_fwd_kernel(const LstmFwdParams p) {
    constexpr int CL = LstmCfg<H>::CL, UN = LstmCfg<H>::UNITS, KS = LstmCfg<H>::KS, NT = LstmCfg<H>::NT;
    constexpr int KW = H / KS;                       // k's per slice
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int cid = blockIdx.x / CL;
    const int tid = threadIdx.x;
    const int jl = tid % UN, ks = tid / UN;
    const int j = rank * UN + jl;

    __shared__ __align__(16) float h_s[2][BG][H];
    __shared__ float part[KS][4][BG][UN];

    float w[4][KW];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const float4* src = reinterpret_cast<const float4*>(p.w_hh + ((size_t)(g * H + j)) * H + ks * KW);
#pragma unroll
        for (int q = 0; q < KW / 4; ++q) {
            float4 v = __ldg(src + q);
            w[g][4 * q] = v.x; w[g][4 * q + 1] = v.y; w[g][4 * q + 2] = v.z; w[g][4 * q + 3] = v.w;
        }
    }
    const bool fin = tid < UN * BG;                  // owner thread of (row fb, unit j)
    const int fb = tid / UN;
    float bh[4] = {0.f, 0.f, 0.f, 0.f};
    if (fin && p.b_hh) {
#pragma unroll
        for (int g = 0; g < 4; ++g) bh[g] = p.b_hh[g * H + j];
    }
    float* peer_h[CL];
#pragma unroll
    for (int r = 0; r < CL; ++r) peer_h[r] = cluster.map_shared_rank(&h_s[0][0][0], r);

    const int L = p.L;
    for (int bg = cid; bg * BG < p.B; bg += p.nclusters) {
        const int b = bg * BG + fb;
        const bool bvalid = fin && b < p.B;
        for (int i = tid; i < BG * H; i += NT) {
            int bb = bg * BG + i / H;
            h_s[0][i / H][i % H] = (p.h0 && bb < p.B) ? p.h0[(size_t)bb * H + (i % H)] : 0.f;
        }
        float hprev = (bvalid && p.h0) ? p.h0[(size_t)b * H + j] : 0.f;
        float cprev = (bvalid && p.c0) ? p.c0[(size_t)b * H + j] : 0.f;
        cluster.sync();
        int cur = 0;
        for (int t = 0; t < L; ++t) {
            float xg[4] = {0.f, 0.f, 0.f, 0.f};
            if (bvalid) {
                const float* g = p.gi + ((size_t)b * L + t) * (4 * H) + j;
#pragma unroll
                for (int q = 0; q < 4; ++q) xg[q] = __ldg(g + q * H);
            }
            float acc[4][BG];
#pragma unroll
            for (int bb = 0; bb < BG; ++bb) {
                acc[0][bb] = acc[1][bb] = acc[2][bb] = acc[3][bb] = 0.f;
                const float4* hv = reinterpret_cast<const float4*>(&h_s[cur][bb][ks * KW]);
#pragma unroll
                for (int q = 0; q < KW / 4; ++q) {
                    const float4 x = hv[q];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        acc[g][bb] = fmaf(w[g][4 * q], x.x, acc[g][bb]);
                        acc[g][bb] = fmaf(w[g][4 * q + 1], x.y, acc[g][bb]);
                        acc[g][bb] = fmaf(w[g][4 * q + 2], x.z, acc[g][bb]);
                        acc[g][bb] = fmaf(w[g][4 * q + 3], x.w, acc[g][bb]);
                    }
                }
            }
#pragma unroll
            for (int bb = 0; bb < BG; ++bb) {
#pragma unroll
                for (int g = 0; g < 4; ++g) part[ks][g][bb][jl] = acc[g][bb];
            }
            __syncthreads();
            if (fin) {
                float s[4];
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    float a = bh[g] + xg[g];
#pragma unroll
                    for (int k = 0; k < KS; ++k) a += part[k][g][fb][jl];
                    s[g] = a;
                }
                const float ig = sigmoidf_fast(s[0]);
                const float fg = sigmoidf_fast(s[1]);
                const float gg = tanhf_fast(s[2]);
                const float og = sigmoidf_fast(s[3]);
                const float cn = fmaf(fg, cprev, ig * gg);
                const float hn = og * tanhf_fast(cn);
                cprev = cn;
                hprev = hn;
                if (bvalid) {
                    const size_t o = (size_t)b * L + t;
                    p.out[o * H + j] = hn;
                    if (p.save) {
                        float* sv = p.save + o * (5 * H) + j;
                        sv[0] = ig; sv[H] = fg; sv[2 * H] = gg; sv[3 * H] = og; sv[4 * H] = cn;
                    }
                }
                const int off = ((cur ^ 1) * BG + fb) * H + j;
#pragma unroll
                for (int rr = 0; rr < CL; ++rr) peer_h[rr][off] = hn;
            }
            cluster.sync();
            cur ^= 1;
        }
        if (bvalid && p.h_last) p.h_last[(size_t)b * H + j] = hprev;
        if (bvalid && p.c_last) p.c_last[(size_t)b * H + j] = cprev;
    }
}

struct LstmBwdParams {
    const float *dout, *dh_last, *dc_last, *w_hh, *save, *c0;
    float *dgates, *dh0, *dc0;
    int B, L, nclusters;
};

template <int H, int BG>
__global__ void __launch_bounds__(LstmCfg<H>::NT, 1) lstm_bwd_kernel(const LstmBwdParams p) {
    constexpr int CL = LstmCfg<H>::CL, UN = LstmCfg<H>::UNITS, KS = LstmCfg<H>::KS;
    constexpr int KW = 4 * H / KS;                   // rows of W_hh per slice
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int cid = blockIdx.x / CL;
    const int tid = threadIdx.x;
    const int jl = tid % UN, ks = tid / UN;
    const int j = rank * UN + jl;

    __shared__ __align__(16) float v_s[2][BG][4 * H];
    __shared__ float part[KS][BG][UN];

    float w[KW];                                     // W_hh[ks*KW + i][j]
#pragma unroll
    for (int i = 0; i < KW; ++i) w[i] = __ldg(p.w_hh + (size_t)(ks * KW + i) * H + j);

    const bool fin = tid < UN * BG;
    const int fb = tid / UN;
    float* peer_v[CL];
#pragma unroll
    for (int r = 0; r < CL; ++r) peer_v[r] = cluster.map_shared_rank(&v_s[0][0][0], r);

    const int L = p.L;
    for (int bg = cid; bg * BG < p.B; bg += p.nclusters) {
        const int b = bg * BG + fb;
        const bool bvalid = fin && b < p.B;
        float dh_in = (bvalid && p.dh_last) ? p.dh_last[(size_t)b * H + j] : 0.f;   // dL/dh_{L-1} from h_n
        float dc = (bvalid && p.dc_last) ? p.dc_last[(size_t)b * H + j] : 0.f;      // carried dL/dc_t
        bool have_part = false;
        int nxt = 0;
        cluster.sync();      // previous batch group fully drained before v_s / part are reused
        for (int t = L - 1; t >= 0; --t) {
            if (fin) {
                float dho = 0.f, ig = 0.f, fg = 0.f, gg = 0.f, og = 0.f, cc = 0.f, cp = 0.f;
                if (bvalid) {
                    const size_t o = (size_t)b * L + t;
                    dho = __ldg(p.dout + o * H + j);
                    const float* sv = p.save + o * (5 * H) + j;
                    ig = __ldg(sv); fg = __ldg(sv + H); gg = __ldg(sv + 2 * H); og = __ldg(sv + 3 * H); cc = __ldg(sv + 4 * H);
                    cp = t > 0 ? __ldg(sv - 5 * H + 4 * H) : (p.c0 ? __ldg(p.c0 + (size_t)b * H + j) : 0.f);
                }
                float dh = dho + dh_in;
                dh_in = 0.f;
                if (have_part) {
#pragma unroll
                    for (int k = 0; k < KS; ++k) dh += part[k][fb][jl];
                }
                const float tc = tanhf_fast(cc);
                const float dao = dh * tc * og * (1.f - og);
                dc = fmaf(dh * og, 1.f - tc * tc, dc);
                const float dai = dc * gg * ig * (1.f - ig);
                const float daf = dc * cp * fg * (1.f - fg);
                const float dag = dc * ig * (1.f - gg * gg);
                dc *= fg;
                if (bvalid) {
                    float* g = p.dgates + ((size_t)b * L + t) * (4 * H) + j;
                    g[0] = dai; g[H] = daf; g[2 * H] = dag; g[3 * H] = dao;
                }
                const int off = (nxt * BG + fb) * (4 * H) + j;
#pragma unroll
                for (int rr = 0; rr < CL; ++rr) {
                    peer_v[rr][off] = dai;
                    peer_v[rr][off + H] = daf;
                    peer_v[rr][off + 2 * H] = dag;
                    peer_v[rr][off + 3 * H] = dao;
                }
            }
            cluster.sync();
#pragma unroll
            for (int bb = 0; bb < BG; ++bb) {
                float a0 = 0.f, a1 = 0.f;
                const float4* vv = reinterpret_cast<const float4*>(&v_s[nxt][bb][ks * KW]);
#pragma unroll
                for (int q = 0; q < KW / 4; ++q) {
                    const float4 x = vv[q];
                    a0 = fmaf(w[4 * q], x.x, a0);
                    a1 = fmaf(w[4 * q + 1], x.y, a1);
                    a0 = fmaf(w[4 * q + 2], x.z, a0);
                    a1 = fmaf(w[4 * q + 3], x.w, a1);
                }
                part[ks][bb][jl] = a0 + a1;
            }
            __syncthreads();
            have_part = true;
            nxt ^= 1;
        }
        if (fin) {
            float d = dh_in;
            if (have_part) {
#pragma unroll
                for (int k = 0; k < KS; ++k) d += part[k][fb][jl];
            }
            if (bvalid && p.dh0) p.dh0[(size_t)b * H + j] = d;
            if (bvalid && p.dc0) p.dc0[(size_t)b * H + j] = dc;
        }
    }
}

// Clusters of this kernel that fit on the device at once (queried once per kernel instance; 0 = query failed).
template <typename Kern>
static int max_active_clusters(Kern kern, int cl, int nthreads) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)cl);
    cfg.blockDim = dim3((unsigned)nthreads);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cl;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

// Launch kernel<H, BG> for the BG that fits the batch into the co-resident clusters (the BG = 4 instance is the one
// queried: all three use the same threads, and its shared memory is the largest).
template <int H, typename Params, typename K1, typename K2, typename K4>
static int launch_lstm(Params& p, K1 k1, K2 k2, K4 k4, int& cached_clusters, cudaStream_t stream) {
    constexpr int cl = LstmCfg<H>::CL, nt = LstmCfg<H>::NT;
    if (cached_clusters <= 0) {
        cached_clusters = max_active_clusters(k4, cl, nt);
        if (cached_clusters <= 0) return 1000 + (int)cudaErrorLaunchOutOfResources;
    }
    const int max_clusters = cached_clusters;
    const int bg = pick_bg(p.B, max_clusters);
    const int ngroups = (p.B + bg - 1) / bg;
    p.nclusters = ngroups < max_clusters ? ngroups : max_clusters;
    switch (bg) {
        case 1: return launch_cluster(k1, p, cl, nt, p.nclusters, stream);
        case 2: return launch_cluster(k2, p, cl, nt, p.nclusters, stream);
        default: return launch_cluster(k4, p, cl, nt, p.nclusters, stream);
    }
}

template <int H>
static int lstm_fwd_h(LstmFwdParams& p, cudaStream_t stream) {
    static int clusters = 0;
    return launch_lstm<H>(p, lstm_fwd_kernel<H, 1>, lstm_fwd_kernel<H, 2>, lstm_fwd_kernel<H, 4>, clusters, stream);
}

template <int H>
static int lstm_bwd_h(LstmBwdParams& p, cudaStream_t stream) {
    static int clusters = 0;
    return launch_lstm<H>(p, lstm_bwd_kernel<H, 1>, lstm_bwd_kernel<H, 2>, lstm_bwd_kernel<H, 4>, clusters, stream);
}

}  // namespace rorl

using namespace rorl;

static bool lstm_h_ok(int64_t H) { return H == 256 || H == 128 || H == 64 || H == 32 || H == 16; }

extern "C" {

int rorl_lstm_save_floats_per_step(int64_t H) { return (int)(5 * H); }

int rorl_lstm_fwd(const float* gi, const float* w_hh, const float* b_hh, const float* h0, const float* c0, float* out,
                  float* save, float* h_last, float* c_last, int64_t B, int64_t L, int64_t H, cudaStream_t stream) {
    if (!gi || !w_hh || !out) return RORL_ERR_ARG;
    if (B <= 0 || L <= 0 || !lstm_h_ok(H)) return RORL_ERR_SHAPE;
    if ((reinterpret_cast<uintptr_t>(w_hh) & 15) != 0) return RORL_ERR_ALIGN;
    LstmFwdParams p;
    p.gi = gi; p.w_hh = w_hh; p.b_hh = b_hh; p.h0 = h0; p.c0 = c0;
    p.out = out; p.save = save; p.h_last = h_last; p.c_last = c_last;
    p.B = (int)B; p.L = (int)L; p.nclusters = 1;
    switch (H) {
        case 256: return lstm_fwd_h<256>(p, stream);
        case 128: return lstm_fwd_h<128>(p, stream);
        case 64: return lstm_fwd_h<64>(p, stream);
        case 32: return lstm_fwd_h<32>(p, stream);
        default: return lstm_fwd_h<16>(p, stream);
    }
}

int rorl_lstm_bwd(const float* dout, const float* dh_last, const float* dc_last, const float* w_hh, const float* save,
                  const float* c0, float* dgates, float* dh0, float* dc0, int64_t B, int64_t L, int64_t H,
                  cudaStream_t stream) {
    if (!dout || !w_hh || !save || !dgates) return RORL_ERR_ARG;
    if (B <= 0 || L <= 0 || !lstm_h_ok(H)) return RORL_ERR_SHAPE;
    LstmBwdParams p;
    p.dout = dout; p.dh_last = dh_last; p.dc_last = dc_last; p.w_hh = w_hh; p.save = save; p.c0 = c0;
    p.dgates = dgates; p.dh0 = dh0; p.dc0 = dc0;
    p.B = (int)B; p.L = (int)L; p.nclusters = 1;
    switch (H) {
        case 256: return lstm_bwd_h<256>(p, stream);
        case 128: return lstm_bwd_h<128>(p, stream);
        case 64: return lstm_bwd_h<64>(p, stream);
        case 32: return lstm_bwd_h<32>(p, stream);
        default: return lstm_bwd_h<16>(p, stream);
    }
}

}  // extern "C"
