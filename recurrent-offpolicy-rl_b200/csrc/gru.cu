// GRU recurrence as a PERSISTENT thread-block-cluster kernel, forward and backward, sm_100a.
//
//   r = sigmoid(gi_r + W_hr h + b_hr)      z = sigmoid(gi_z + W_hz h + b_hz)
//   n = tanh(gi_n + r * (W_hn h + b_hn))   h' = (1 - z) * n + z * h
//
// Replaces torch.nn.GRU(256, 256, batch_first=True) on the `gru` encoder path
// (ref: offpolicy_rnn/models/rnn_base.py:59,245-247,454; cuDNN on GPU, ATen loop on CPU).
// gi = x W_ih^T + b_ih for all steps is ONE tensor-core GEMM up front (csrc/gemm_bf16.cu); this file is
// the L dependent steps that remain.
//
// Design.  W_hh is 3H x H fp32 = 786 KB at H = 256: more than one SM's shared memory, so a cluster
// of CL = H / 64 CTAs owns it, and it lives in REGISTERS, not shared memory: CTA `rank` owns hidden
// units [64 rank, 64 rank + 64); its 512 threads are 64 units x 8 K-slices, and thread (unit j,
// slice ks) keeps the 3 x H/8 weights W_h{r,z,n}[j, ks*H/8 ...] (96 registers at H = 256) for the
// whole sequence.  One cluster serves BG batch rows; the grid is ceil(B / BG) clusters, so B = 32
// rows keep 128 SMs busy.  Per step:
//   (1) every thread multiplies its weight slice with h_{t-1} (read from shared memory as a warp
//       broadcast: a warp is 32 units x one K-slice) and leaves 3 x BG partial sums in shared memory;
//   (2) __syncthreads; 64 x BG "owner" threads add the 8 partials, apply the gates, write h_t and the
//       saved gates to HBM, and push h_t into the h buffer of every CTA of the cluster through
//       distributed shared memory;
//   (3) one cluster barrier (release/acquire) publishes h_t.  The h buffer is double buffered, so
//       that barrier is the only cluster-wide synchronisation per step.
// The step is latency bound (one dependent chain of 1002 steps): the roofline is us/step, not GB/s.
//
// Backward walks the steps in reverse with the transposed product dh_{t-1} += W_hh^T dgh_t in the
// same shape: thread (unit j, slice ks) keeps W_hh[ks*3H/8 ..., j] (96 registers), the broadcast
// vector is dgh_t = (da_r, da_z, r * da_n) [3H].  It emits dgi [B, L, 3H] and d(gh_n) [B, L, H];
// the weight gradients are two tensor-core GEMMs over all steps afterwards (host side).
#include "common.cuh"
#include <cstdlib>
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

namespace rorl {

// Shape of one configuration: H hidden units split over CL = H / UNITS CTAs of NT = UNITS * KS threads.
template <int H_>
struct GruCfg {
    static constexpr int H = H_;
    static constexpr int UNITS = H_ >= 64 ? 64 : H_;          // hidden units per CTA
    static constexpr int KS = H_ >= 32 ? 8 : 4;               // K slices per unit
    static constexpr int NT = UNITS * KS;                     // threads per CTA (512 at H >= 64)
    static constexpr int CL = H_ / UNITS;                     // CTAs per cluster
    static_assert(H_ % UNITS == 0 && (H_ / KS) % 4 == 0 && (3 * H_ / KS) % 4 == 0, "unsupported hidden size");
};

struct GruFwdParams {
    const float *gi, *w_hh, *b_hh, *h0;
    float *out, *save, *h_last;
    int B, L, nclusters;
};

template <int H, int BG>
__global__ void __launch_bounds__(GruCfg<H>::NT, 1) gru_fwd_kernel(const GruFwdParams p) {
    constexpr int CL = GruCfg<H>::CL, kGruUnits = GruCfg<H>::UNITS, kGruKS = GruCfg<H>::KS, kGruThreads = GruCfg<H>::NT;
    constexpr int KW = H / kGruKS;                   // k's per slice
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int cid = blockIdx.x / CL;
    const int tid = threadIdx.x;
    const int jl = tid % kGruUnits, ks = tid / kGruUnits;
    const int j = rank * kGruUnits + jl;

    __shared__ __align__(16) float h_s[2][BG][H];
    __shared__ float part[kGruKS][3][BG][kGruUnits];

    float w[3][KW];
#pragma unroll
    for (int g = 0; g < 3; ++g) {
        const float4* src = reinterpret_cast<const float4*>(p.w_hh + ((size_t)(g * H + j)) * H + ks * KW);
#pragma unroll
        for (int q = 0; q < KW / 4; ++q) {
            float4 v = __ldg(src + q);
            w[g][4 * q] = v.x; w[g][4 * q + 1] = v.y; w[g][4 * q + 2] = v.z; w[g][4 * q + 3] = v.w;
        }
    }
    const bool fin = tid < kGruUnits * BG;           // owner thread of (row fb, unit j)
    const int fb = tid / kGruUnits;
    float bh[3] = {0.f, 0.f, 0.f};
    if (fin && p.b_hh) {
#pragma unroll
        for (int g = 0; g < 3; ++g) bh[g] = p.b_hh[g * H + j];
    }
    float* peer_h[CL];
#pragma unroll
    for (int r = 0; r < CL; ++r) peer_h[r] = cluster.map_shared_rank(&h_s[0][0][0], r);

    const int L = p.L;
    for (int bg = cid; bg * BG < p.B; bg += p.nclusters) {
        const int b = bg * BG + fb;
        const bool bvalid = fin && b < p.B;
        // initial state into buffer 0 of this CTA (every CTA loads the full vector itself)
        for (int i = tid; i < BG * H; i += kGruThreads) {
            int bb = bg * BG + i / H;
            h_s[0][i / H][i % H] = (p.h0 && bb < p.B) ? p.h0[(size_t)bb * H + (i % H)] : 0.f;
        }
        float hprev = (bvalid && p.h0) ? p.h0[(size_t)b * H + j] : 0.f;
        cluster.sync();
        int cur = 0;
        for (int t = 0; t < L; ++t) {
            float gr = 0.f, gz = 0.f, gn = 0.f;
            if (bvalid) {
                const float* g = p.gi + ((size_t)b * L + t) * (3 * H) + j;
                gr = __ldg(g); gz = __ldg(g + H); gn = __ldg(g + 2 * H);
            }
            float acc[3][BG];
#pragma unroll
            for (int bb = 0; bb < BG; ++bb) {
                acc[0][bb] = acc[1][bb] = acc[2][bb] = 0.f;
                const float4* hv = reinterpret_cast<const float4*>(&h_s[cur][bb][ks * KW]);
#pragma unroll
                for (int q = 0; q < KW / 4; ++q) {
                    const float4 x = hv[q];
#pragma unroll
                    for (int g = 0; g < 3; ++g) {
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
                for (int g = 0; g < 3; ++g) part[ks][g][bb][jl] = acc[g][bb];
            }
            __syncthreads();
            if (fin) {
                float s[3];
#pragma unroll
                for (int g = 0; g < 3; ++g) {
                    float a = bh[g];
#pragma unroll
                    for (int k = 0; k < kGruKS; ++k) a += part[k][g][fb][jl];
                    s[g] = a;
                }
                const float r = sigmoidf_fast(gr + s[0]);
                const float z = sigmoidf_fast(gz + s[1]);
                const float n = tanhf_fast(fmaf(r, s[2], gn));
                const float hn = fmaf(z, hprev - n, n);          // (1 - z) n + z h
                hprev = hn;
                if (bvalid) {
                    const size_t o = (size_t)b * L + t;
                    p.out[o * H + j] = hn;
                    if (p.save) {
                        float* sv = p.save + o * (4 * H) + j;
                        sv[0] = r; sv[H] = z; sv[2 * H] = n; sv[3 * H] = s[2];
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
    }
}

struct GruBwdParams {
    const float *dout, *dh_last, *w_hh, *save, *out, *h0;
    float *dgi, *dghn, *dh0;
    int B, L, nclusters;
};

template <int H, int BG>
__global__ void __launch_bounds__(GruCfg<H>::NT, 1) gru_bwd_kernel(const GruBwdParams p) {
    constexpr int CL = GruCfg<H>::CL, kGruUnits = GruCfg<H>::UNITS, kGruKS = GruCfg<H>::KS;
    constexpr int KW = 3 * H / kGruKS;               // rows of W_hh per slice
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int cid = blockIdx.x / CL;
    const int tid = threadIdx.x;
    const int jl = tid % kGruUnits, ks = tid / kGruUnits;
    const int j = rank * kGruUnits + jl;

    __shared__ __align__(16) float v_s[2][BG][3 * H];
    __shared__ float part[kGruKS][BG][kGruUnits];

    float w[KW];                                     // W_hh[ks*KW + i][j]
#pragma unroll
    for (int i = 0; i < KW; ++i) w[i] = __ldg(p.w_hh + (size_t)(ks * KW + i) * H + j);

    const bool fin = tid < kGruUnits * BG;
    const int fb = tid / kGruUnits;
    float* peer_v[CL];
#pragma unroll
    for (int r = 0; r < CL; ++r) peer_v[r] = cluster.map_shared_rank(&v_s[0][0][0], r);

    const int L = p.L;
    for (int bg = cid; bg * BG < p.B; bg += p.nclusters) {
        const int b = bg * BG + fb;
        const bool bvalid = fin && b < p.B;
        float dh_rec = (bvalid && p.dh_last) ? p.dh_last[(size_t)b * H + j] : 0.f;   // direct part of dL/dh_t
        bool have_part = false;
        int nxt = 0;
        cluster.sync();      // previous batch group fully drained before v_s / part are reused
        for (int t = L - 1; t >= 0; --t) {
            if (fin) {
                float dho = 0.f, r = 0.f, z = 0.f, n = 0.f, ghn = 0.f, hp = 0.f;
                if (bvalid) {
                    const size_t o = (size_t)b * L + t;
                    dho = __ldg(p.dout + o * H + j);
                    const float* sv = p.save + o * (4 * H) + j;
                    r = __ldg(sv); z = __ldg(sv + H); n = __ldg(sv + 2 * H); ghn = __ldg(sv + 3 * H);
                    hp = t > 0 ? __ldg(p.out + (o - 1) * H + j) : (p.h0 ? __ldg(p.h0 + (size_t)b * H + j) : 0.f);
                }
                float dh = dho + dh_rec;
                if (have_part) {
#pragma unroll
                    for (int k = 0; k < kGruKS; ++k) dh += part[k][fb][jl];
                }
                const float dn = dh * (1.f - z);
                const float dz = dh * (hp - n);
                dh_rec = dh * z;
                const float dan = dn * (1.f - n * n);
                const float dar = dan * ghn * r * (1.f - r);
                const float daz = dz * z * (1.f - z);
                const float dgn = dan * r;
                if (bvalid) {
                    const size_t o = (size_t)b * L + t;
                    float* g = p.dgi + o * (3 * H) + j;
                    g[0] = dar; g[H] = daz; g[2 * H] = dan;
                    p.dghn[o * H + j] = dgn;
                }
                const int off = (nxt * BG + fb) * (3 * H) + j;
#pragma unroll
                for (int rr = 0; rr < CL; ++rr) {
                    peer_v[rr][off] = dar;
                    peer_v[rr][off + H] = daz;
                    peer_v[rr][off + 2 * H] = dgn;
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
            float d = dh_rec;
            if (have_part) {
#pragma unroll
                for (int k = 0; k < kGruKS; ++k) d += part[k][fb][jl];
            }
            if (bvalid && p.dh0) p.dh0[(size_t)b * H + j] = d;
        }
    }
}

}  // namespace rorl

using namespace rorl;

static bool gru_h_ok(int64_t H) { return H == 256 || H == 128 || H == 64 || H == 32 || H == 16; }

// SMs the FORWARD recurrence may occupy (rorl_gru_set_fwd_sms; default all): the update runs two independent context
// encoders side by side on two streams, and a recurrence that takes every SM cannot overlap with the other one.  With
// half the SMs a cluster serves two batch rows at B = 32: 1.9 instead of 1.36 us per step, but two at a time.
static int g_gru_fwd_sms = 148;
static int gru_fwd_sms() { return g_gru_fwd_sms; }

template <int H>
static int gru_fwd_h(GruFwdParams& p, cudaStream_t stream) {
    constexpr int cl = GruCfg<H>::CL;
    const int max_clusters = gru_fwd_sms() / cl > 0 ? gru_fwd_sms() / cl : 1;
    const int bg = pick_bg(p.B, max_clusters);
    const int ngroups = (p.B + bg - 1) / bg;
    p.nclusters = ngroups < max_clusters ? ngroups : max_clusters;
    switch (bg) {
        case 1: return launch_cluster(gru_fwd_kernel<H, 1>, p, cl, GruCfg<H>::NT, p.nclusters, stream);
        case 2: return launch_cluster(gru_fwd_kernel<H, 2>, p, cl, GruCfg<H>::NT, p.nclusters, stream);
        default: return launch_cluster(gru_fwd_kernel<H, 4>, p, cl, GruCfg<H>::NT, p.nclusters, stream);
    }
}

template <int H>
static int gru_bwd_h(GruBwdParams& p, cudaStream_t stream) {
    constexpr int cl = GruCfg<H>::CL;
    const int max_clusters = 148 / cl;
    const int bg = pick_bg(p.B, max_clusters);
    const int ngroups = (p.B + bg - 1) / bg;
    p.nclusters = ngroups < max_clusters ? ngroups : max_clusters;
    switch (bg) {
        case 1: return launch_cluster(gru_bwd_kernel<H, 1>, p, cl, GruCfg<H>::NT, p.nclusters, stream);
        case 2: return launch_cluster(gru_bwd_kernel<H, 2>, p, cl, GruCfg<H>::NT, p.nclusters, stream);
        default: return launch_cluster(gru_bwd_kernel<H, 4>, p, cl, GruCfg<H>::NT, p.nclusters, stream);
    }
}

extern "C" {

int rorl_gru_set_fwd_sms(int sms) {
    g_gru_fwd_sms = (sms >= 4 && sms <= 148) ? sms : 148;
    return g_gru_fwd_sms;
}

int rorl_gru_save_floats_per_step(int64_t H) { return (int)(4 * H); }

int rorl_gru_fwd(const float* gi, const float* w_hh, const float* b_hh, const float* h0, float* out, float* save,
                 float* h_last, int64_t B, int64_t L, int64_t H, cudaStream_t stream) {
    if (!gi || !w_hh || !out) return RORL_ERR_ARG;
    if (B <= 0 || L <= 0 || !gru_h_ok(H)) return RORL_ERR_SHAPE;
    if ((reinterpret_cast<uintptr_t>(w_hh) & 15) != 0) return RORL_ERR_ALIGN;
    GruFwdParams p;
    p.gi = gi; p.w_hh = w_hh; p.b_hh = b_hh; p.h0 = h0; p.out = out; p.save = save; p.h_last = h_last;
    p.B = (int)B; p.L = (int)L; p.nclusters = 1;
    switch (H) {
        case 256: return gru_fwd_h<256>(p, stream);
        case 128: return gru_fwd_h<128>(p, stream);
        case 64: return gru_fwd_h<64>(p, stream);
        case 32: return gru_fwd_h<32>(p, stream);
        default: return gru_fwd_h<16>(p, stream);
    }
}

int rorl_gru_bwd(const float* dout, const float* dh_last, const float* w_hh, const float* save, const float* out,
                 const float* h0, float* dgi, float* dghn, float* dh0, int64_t B, int64_t L, int64_t H,
                 cudaStream_t stream) {
    if (!dout || !w_hh || !save || !out || !dgi || !dghn) return RORL_ERR_ARG;
    if (B <= 0 || L <= 0 || !gru_h_ok(H)) return RORL_ERR_SHAPE;
    GruBwdParams p;
    p.dout = dout; p.dh_last = dh_last; p.w_hh = w_hh; p.save = save; p.out = out; p.h0 = h0;
    p.dgi = dgi; p.dghn = dghn; p.dh0 = dh0;
    p.B = (int)B; p.L = (int)L; p.nclusters = 1;
    switch (H) {
        case 256: return gru_bwd_h<256>(p, stream);
        case 128: return gru_bwd_h<128>(p, stream);
        case 64: return gru_bwd_h<64>(p, stream);
        case 32: return gru_bwd_h<32>(p, stream);
        default: return gru_bwd_h<16>(p, stream);
    }
}

}  // extern "C"
