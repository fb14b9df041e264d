// Causal variable-length attention with ALiBi on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), every head
// dimension hd that is a multiple of 8 from 8 to 128, bf16 operands / fp32 accumulation, forward and backward.
//
// Replaces flash_attn_varlen_qkvpacked_func(qkv[T, 3, H, hd], cu_seqlens, max_seqlen, p, softmax_scale, causal=True,
// alibi_slopes) as called by flash_attn's MHA inside the cgpt encoder layer (ref:
// offpolicy_rnn/models/flash_attention/TransformerFlashAttention.py:65-85; bf16 autocast :80-82; sequences come from
// unpad_input_for_concatenated_sequences :104-112).  score_ij = softmax_scale * q_i.k_j - slope_h * (i - j), j <= i.
//
// Layout decision: every tcgen05.mma operand is a K-major SWIZZLE_128B tile fetched by TMA.  Every operand is padded
// along d to DP = 64 (hd <= 64) or DP = 128 (64 < hd <= 128) with zero columns, which add exact zeros to every fp32
// accumulator; the epilogues write only the hd real columns.  A 128-byte swizzle row holds 64 bf16, so a DP = 128
// tile is two swizzle atoms along d: the d-contractions (Q K^T, dO V^T) step through both, and the TMA boxes are
// loaded at d = 0 and d = 64.  Products that contract over tokens (P.V, dS.K, dS^T.Q, P^T.dO) need the token axis
// contiguous, so rorl_attn_prep writes, next to the row-major bf16 copies [T, H, DP], transposed copies [H, DP, Tp]
// (token-contiguous).  That costs one extra pass over 33 MB per tensor (hd 64) and removes every in-kernel
// transposition and every MN-major descriptor.
//
// Forward: CTA = (128-query tile of one sequence, head); 4 softmax warps (thread = one query row = one TMEM lane)
// + 1 issuer warp (one thread drives TMA and tcgen05.mma).  Two passes over the key tiles j <= i: pass A computes the
// row maximum and the normaliser from S = Q K^T in TMEM (no O to rescale), pass B recomputes S, writes
// P = exp2(s - m) / l as bf16 into a swizzled shared tile and accumulates O += P V in TMEM.  lse is kept for the
// backward.  The exponentials (2 per score) bound the kernel: 256 M ex2 per call at 32 x 1001 tokens, ~55 us.
// DP = 64 fits two CTAs per SM (97 KiB of shared memory each), DP = 128 one (161 KiB).
//
// Backward: one kernel template, run twice.  Row side = queries gives dQ; row side = keys gives dK and dV.  Per
// 64-column sub-tile: S and dP by two MMAs into TMEM, p = exp2(s - lse), dS = p (dP - D) scale in registers, bf16
// tiles of dS (and P) in shared memory, then dQ += dS K or dK += dS^T Q, dV += P^T dO from the transposed copies.
// Deterministic: every output element is produced by exactly one CTA, no atomics.  DP = 128 takes 231 552 B of
// shared memory and 384 TMEM columns (allocated as 512), one CTA per SM.
#include "tc.cuh"
#include <cuda_bf16.h>

namespace rorl {

__host__ __device__ constexpr bool attn_head_dim_ok(long long hd) { return hd >= 8 && hd <= 128 && hd % 8 == 0; }
// padded head dimension of the bf16 operand copies
__host__ __device__ constexpr int attn_dp(long long hd) { return hd <= 64 ? 64 : 128; }

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}

// ---------------------------------------------------------------------------------------------------------------
// prep: fp32 source rows [*, nsec, H, hd] (row stride ld_tok floats) -> bf16 row-major [nsec][T, H, DP] and transposed
// [nsec][H, DP, Tp] in ATTENTION TOKEN SPACE, zero in columns hd .. DP-1: token t of that space is source row gmap[t]
// (-1 = zero padding slot).  TMA needs 16-byte aligned inner coordinates, i.e. sequence starts that are multiples of 8
// tokens in the token-contiguous copies, so the caller lays the sequences out on 8-token boundaries
// (kernels.attention_tiles) and the gather happens here.  Optionally D[h, t] = sum_d src[gmap[t], h, d] * o[gmap[t], h, d]
// over the hd real columns (nsec == 1).  Block = 64 tokens x DP columns of one head.
// ---------------------------------------------------------------------------------------------------------------
template <int DP>
__global__ void __launch_bounds__(256) attn_prep_kernel(const float* __restrict__ src, long long ld_tok, int H, int hd, int T, int Tp,
                                                        const int* __restrict__ gmap, __nv_bfloat16* __restrict__ rm,
                                                        __nv_bfloat16* __restrict__ tr, const float* __restrict__ o, long long ld_o,
                                                        float* __restrict__ Dout) {
    constexpr int C4 = DP / 4, RPP = 256 / C4;          // float4 columns per row, rows per pass
    __shared__ float tile[64][DP + 1];
    const int t0 = blockIdx.x * 64, h = blockIdx.y, sec = blockIdx.z;
    const int tid = threadIdx.x;
    const int r = tid / C4, c4 = tid % C4;
    const bool real = c4 * 4 < hd;                      // hd % 8 == 0: a float4 is all real or all padding
#pragma unroll
    for (int rr = 0; rr < 64 / RPP; ++rr) {
        const int row = r + RPP * rr, t = t0 + row;
        const int ts = t < T ? (gmap ? gmap[t] : t) : -1;       // source row of attention-space token t (-1: padding slot)
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ts >= 0 && real) v = *reinterpret_cast<const float4*>(src + (size_t)ts * ld_tok + ((size_t)sec * H + h) * hd + c4 * 4);
        tile[row][c4 * 4] = v.x; tile[row][c4 * 4 + 1] = v.y; tile[row][c4 * 4 + 2] = v.z; tile[row][c4 * 4 + 3] = v.w;
        if (rm != nullptr && t < T) {
            uint2 pk = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
            *reinterpret_cast<uint2*>(rm + ((size_t)sec * T + t) * H * DP + (size_t)h * DP + c4 * 4) = pk;
        }
        if (o != nullptr) {
            float d = 0.f;
            if (ts >= 0 && real) {
                const float4 ov = *reinterpret_cast<const float4*>(o + (size_t)ts * ld_o + (size_t)h * hd + c4 * 4);
                d = v.x * ov.x + v.y * ov.y + v.z * ov.z + v.w * ov.w;
            }
#pragma unroll
            for (int m = C4 / 2; m >= 1; m >>= 1) d += __shfl_xor_sync(0xffffffffu, d, m);
            if (c4 == 0 && t < Tp) Dout[(size_t)h * Tp + t] = d;
        }
    }
    if (tr == nullptr) return;
    __syncthreads();
    const int tq = tid & 3;
#pragma unroll
    for (int dh = 0; dh < DP / 64; ++dh) {
        const int d = dh * 64 + (tid >> 2);
        uint32_t pk[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) pk[i] = pack_bf16(tile[tq * 16 + 2 * i][d], tile[tq * 16 + 2 * i + 1][d]);
        __nv_bfloat16* dst = tr + (((size_t)sec * H + h) * DP + d) * Tp + t0 + tq * 16;
        *reinterpret_cast<uint4*>(dst) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        *reinterpret_cast<uint4*>(dst + 8) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
    }
}

// fp32 [32 columns] of one TMEM row -> dst[0 .. ncols), ncols a multiple of 4 (float4 stores; none for ncols <= 0)
__device__ __forceinline__ void store_cols(float* dst, const uint32_t (&x)[32], int ncols) {
#pragma unroll
    for (int q = 0; q < 8; ++q)
        if (q * 4 < ncols)
            *reinterpret_cast<float4*>(dst + q * 4) =
                make_float4(__uint_as_float(x[4 * q]), __uint_as_float(x[4 * q + 1]), __uint_as_float(x[4 * q + 2]), __uint_as_float(x[4 * q + 3]));
}

// K-major SWIZZLE_128B tile of 128-byte rows: byte offset of 16-byte chunk `ch` (0..7) of row `r`
__device__ __forceinline__ uint32_t sw128(int r, int ch) { return (uint32_t)(r * 128 + ((ch ^ (r & 7)) << 4)); }

struct AttnParams {
    const int4* tiles;          // (first attention-space token of the sequence, length, 128-row tile index, first OUTPUT row)
    const float* slopes;        // [H] ALiBi slopes
    float c1;                   // softmax_scale * log2(e)
    float scale;                // softmax_scale
    int H, hd, T, Tp;               // hd: real head dimension (output columns per head)
    // forward
    float* O; long long ld_o; float* lse;
    // backward
    const float* lse_in; const float* D;
    float* out1; float* out2; long long ld_out;
    // dropout: keep if 16 random bits >= drop_thr (= round(p * 65536)); survivors are scaled by drop_scale = 1 / (1 - p)
    const long long* seed_ptr; uint32_t salt; uint32_t drop_thr; float drop_scale;
};

// Attention-probability dropout (flash-attn's `dropout_p`, active in training mode; ref:
// TransformerFlashAttention.py:65-70 builds MHA(dropout=p)): P_d = P * keep / (1 - p) before the P.V product.  The keep
// bit of (head, query, key) is a counter-based hash of the pair's ABSOLUTE token indices, the per-call seed (a device
// scalar, so captured graphs draw fresh masks on every replay) and the head, evaluated identically in the forward and
// in both backward kernels.  16 random bits per element (two elements per 32-bit hash).  flash-attn's own Philox
// stream cannot be reproduced outside its kernels (SURVEY.md App. A), so parity for p > 0 is statistical; the mask
// function is restated in tests/test_attn_gpu.py to check the kernels against an explicit-mask reference.
__device__ __forceinline__ uint32_t drop_mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ uint32_t drop_head_seed(const long long* seed_ptr, uint32_t salt, int h) {
    const unsigned long long s = (unsigned long long)seed_ptr[0] * 0x9E3779B97F4A7C15ull;
    return drop_mix32((uint32_t)(s >> 32) ^ (uint32_t)s ^ salt ^ ((uint32_t)h * 0x85ebca6bu));
}
// keep factor of (query token qa, key token ka), absolute indices in attention token space
__device__ __forceinline__ float drop_factor(uint32_t hseed, int qa, int ka, int halfT, uint32_t thr, float inv_keep) {
    const uint32_t r = drop_mix32(hseed + (uint32_t)qa * (uint32_t)halfT + (uint32_t)(ka >> 1));
    const uint32_t u16 = (ka & 1) ? (r >> 16) : (r & 0xFFFFu);
    return u16 >= thr ? inv_keep : 0.f;
}

constexpr int kAttnThreads = 160;

// ---------------------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------------------
// a 128-row x DP bf16 tile (Q, one K stage, one 128-token V^T tile): DP / 64 swizzle atoms of 16 KiB along d
__host__ __device__ constexpr int fwd_tile_bytes(int DP) { return 256 * DP; }
__host__ __device__ constexpr int fwd_smem(int DP) { return 4 * fwd_tile_bytes(DP) /*Q, 2 K, Vt*/ + 32768 /*P*/ + 1024 /*align*/ + 128 /*barriers*/; }

template <int DP, bool DROP>
__global__ void __launch_bounds__(kAttnThreads, DP == 64 ? 2 : 1)
attn_fwd_kernel(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                const __grid_constant__ CUtensorMap mapVt, const AttnParams p) {
    constexpr uint32_t TB = fwd_tile_bytes(DP);
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t sQ = base, sK = base + TB, sVt = base + 3 * TB, sP = base + 4 * TB;
    uint8_t* sP_ptr = base_ptr + 4 * TB;
    const uint32_t bars = base + 4 * TB + 32768;
    const uint32_t bar_q = bars, bar_k0 = bars + 8, bar_vt = bars + 24, bar_sfull = bars + 32, bar_sfree = bars + 40,
                   bar_pfull = bars + 48, bar_pvdone = bars + 56;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(base_ptr + 4 * TB + 32768 + 64);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int4 tl = p.tiles[blockIdx.x];
    const int tok0 = tl.x, len = tl.y, qt = tl.z, out0 = tl.w, h = blockIdx.y;
    const int nk = qt + 1, total = 2 * nk;

    if (threadIdx.x == 0) {
        mbar_init(bar_q, 1); mbar_init(bar_k0, 1); mbar_init(bar_k0 + 8, 1); mbar_init(bar_vt, 1);
        mbar_init(bar_sfull, 1); mbar_init(bar_sfree, 4); mbar_init(bar_pfull, 4); mbar_init(bar_pvdone, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tS = tmem_base, tO = tmem_base + 128;

    if (warp == 4) {
        if (lane == 0) {
            const uint32_t idS = idesc_bf16(128, 128), idO = idesc_bf16(128, DP);
            mbar_expect_tx(bar_q, TB);
#pragma unroll
            for (int a = 0; a < DP / 64; ++a) tma_load_3d(sQ + a * 16384, &mapQ, bar_q, a * 64, tok0 + qt * 128, h);
            mbar_expect_tx(bar_k0, TB);
#pragma unroll
            for (int a = 0; a < DP / 64; ++a) tma_load_3d(sK + a * 16384, &mapK, bar_k0, a * 64, tok0, h);
            mbar_wait(bar_q, 0);
            for (int n = 0; n < total; ++n) {
                const int s = n & 1, kt = n % nk, nb = n - nk;
                const bool isB = n >= nk;
                mbar_wait(bar_k0 + 8 * s, (n >> 1) & 1);
                if (n >= 1) mbar_wait(bar_sfree, (n - 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < DP / 16; ++ks) {
                    const uint64_t aQ = make_kmajor_desc(sQ + (ks >> 2) * 16384), bK = make_kmajor_desc(sK + s * TB + (ks >> 2) * 16384);
                    umma_bf16(tS, aQ + (uint64_t)((ks & 3) * 2), bK + (uint64_t)((ks & 3) * 2), idS, ks ? 1u : 0u);
                }
                umma_commit(bar_sfull);
                if (isB && nb >= 1) mbar_wait(bar_pvdone, (nb - 1) & 1);
                if (isB) {
                    mbar_expect_tx(bar_vt, TB);
                    tma_load_3d(sVt, &mapVt, bar_vt, tok0 + kt * 128, 0, h);
                    tma_load_3d(sVt + TB / 2, &mapVt, bar_vt, tok0 + kt * 128 + 64, 0, h);
                }
                if (n + 1 < total) {
                    const int ktn = (n + 1) % nk;
                    mbar_expect_tx(bar_k0 + 8 * (s ^ 1), TB);
#pragma unroll
                    for (int a = 0; a < DP / 64; ++a)
                        tma_load_3d(sK + (s ^ 1) * TB + a * 16384, &mapK, bar_k0 + 8 * (s ^ 1), a * 64, tok0 + ktn * 128, h);
                }
                if (isB) {
                    mbar_wait(bar_vt, nb & 1);
                    mbar_wait(bar_pfull, nb & 1);
                    tc_fence_after();
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks) {
                        const uint64_t aP = make_kmajor_desc(sP + (ks >> 2) * 16384) + (uint64_t)((ks & 3) * 2);
                        const uint64_t bV = make_kmajor_desc(sVt + (ks >> 2) * (TB / 2)) + (uint64_t)((ks & 3) * 2);
                        umma_bf16(tO, aP, bV, idO, (nb | ks) ? 1u : 0u);
                    }
                    umma_commit(bar_pvdone);
                }
            }
        }
    } else {
        // ------------------------------------------------------------------ softmax warps: thread = query row
        const int r = threadIdx.x;
        const int i = qt * 128 + r;                       // query index inside the sequence
        const float c2 = p.slopes[h] * kLog2e;
        const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
        const uint32_t hseed = DROP ? drop_head_seed(p.seed_ptr, p.salt, h) : 0u;
        const int halfT = (p.Tp + 1) >> 1;
        float m = -1e30f, l = 0.f, inv_l = 0.f;
        for (int n = 0; n < total; ++n) {
            const int kt = n % nk, nb = n - nk;
            const bool isB = n >= nk;
            mbar_wait(bar_sfull, n & 1);
            tc_fence_after();
            if (isB && nb >= 1) mbar_wait(bar_pvdone, (nb - 1) & 1);
#pragma unroll 1
            for (int c = 0; c < 4; ++c) {
                uint32_t x[32];
                tmem_ld32(tS + lane_base + c * 32, x);
                tmem_ld_wait();
                const int j0 = kt * 128 + c * 32;
                float s2[32];
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) {
                    const int j = j0 + jj;
                    const float v = fmaf(__uint_as_float(x[jj]), p.c1, -c2 * (float)(i - j));
                    s2[jj] = (j > i) ? -INFINITY : v;
                }
                if (!isB) {
                    float cm = m;
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) cm = fmaxf(cm, s2[jj]);
                    float acc = 0.f;
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) acc += ex2f(s2[jj] - cm);
                    l = fmaf(l, ex2f(m - cm), acc);
                    m = cm;
                } else {
                    uint32_t pk[16];
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) {
                        float p0 = ex2f(s2[2 * jj] - m) * inv_l, p1 = ex2f(s2[2 * jj + 1] - m) * inv_l;
                        if (DROP) {
                            p0 *= drop_factor(hseed, tok0 + i, tok0 + j0 + 2 * jj, halfT, p.drop_thr, p.drop_scale);
                            p1 *= drop_factor(hseed, tok0 + i, tok0 + j0 + 2 * jj + 1, halfT, p.drop_thr, p.drop_scale);
                        }
                        pk[jj] = pack_bf16(p0, p1);
                    }
                    uint8_t* blk = sP_ptr + (c >> 1) * 16384;
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        *reinterpret_cast<uint4*>(blk + sw128(r, (c & 1) * 4 + q)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_sfree);
            if (isB) {
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_pfull);
            }
            if (n == nk - 1) inv_l = 1.0f / l;
        }
        mbar_wait(bar_pvdone, (nk - 1) & 1);
        tc_fence_after();
        const bool valid = i < len;
        float* orow = p.O + (size_t)(out0 + i) * p.ld_o + (size_t)h * p.hd;
#pragma unroll 1
        for (int c = 0; c < DP / 32; ++c) {
            uint32_t x[32];
            tmem_ld32(tO + lane_base + c * 32, x);
            tmem_ld_wait();
            if (valid) store_cols(orow + c * 32, x, p.hd - c * 32);
        }
        if (valid && p.lse != nullptr) p.lse[(size_t)h * p.Tp + tok0 + i] = m + lg2f(l);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256));
    }
}

// ---------------------------------------------------------------------------------------------------------------
// backward half: rows = 128 queries (KSIDE = false: dQ) or 128 keys (KSIDE = true: dK, dV); columns in sub-tiles of 64
// ---------------------------------------------------------------------------------------------------------------
// R / RG: 128 rows x DP (DP / 64 swizzle atoms of 16 KiB along d); a stage holds C, CG (64 rows x DP, atoms of 8 KiB)
// and Ct, CGt (DP rows x 64 tokens), CB bytes each
__host__ __device__ constexpr int bwd_row_bytes(int DP) { return 256 * DP; }
__host__ __device__ constexpr int bwd_col_bytes(int DP) { return 128 * DP; }
__host__ __device__ constexpr int bwd_smem(int DP) {
    return 2 * bwd_row_bytes(DP) /*R, RG*/ + 2 * 4 * bwd_col_bytes(DP) /*stages*/ + 2 * 16384 /*P, dS*/ + 1024 /*lse, D of the columns*/ +
           1024 /*align*/ + 128 /*barriers*/;
}
// TMEM: S and dP 64 columns each, the two accumulators DP each (a power of two is allocated)
__host__ __device__ constexpr int bwd_tmem_cols(int DP) { return DP == 64 ? 256 : 512; }

template <int DP, bool KSIDE, bool DROP>
__global__ void __launch_bounds__(kAttnThreads, 1)
attn_bwd_kernel(const __grid_constant__ CUtensorMap mapR, const __grid_constant__ CUtensorMap mapRG,
                const __grid_constant__ CUtensorMap mapC, const __grid_constant__ CUtensorMap mapCG,
                const __grid_constant__ CUtensorMap mapCt, const __grid_constant__ CUtensorMap mapCGt, const AttnParams p) {
    constexpr uint32_t RB = bwd_row_bytes(DP), CB = bwd_col_bytes(DP);
    constexpr uint32_t kTmemCols = bwd_tmem_cols(DP);
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t sR = base, sRG = base + RB, sStage = base + 2 * RB, sP = base + 2 * RB + 8 * CB, sdS = sP + 16384;
    uint8_t* sP_ptr = base_ptr + 2 * RB + 8 * CB;
    uint8_t* sdS_ptr = sP_ptr + 16384;
    float* s_col = reinterpret_cast<float*>(sP_ptr + 32768);       // [2][2][64]: lse, D of the columns
    const uint32_t bars = sP + 32768 + 1024;
    const uint32_t bar_r = bars, bar_full0 = bars + 8, bar_sdfull = bars + 24, bar_sdfree = bars + 32, bar_pdfull = bars + 40,
                   bar_outdone = bars + 48;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(sP_ptr + 32768 + 1024 + 64);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int4 tl = p.tiles[blockIdx.x];
    const int tok0 = tl.x, len = tl.y, rt = tl.z, out0 = tl.w, h = blockIdx.y;
    // column sub-tiles (64 wide): queries side walks keys 0 .. end of its diagonal tile; key side walks queries from
    // its own first row to the end of the sequence
    const int cs0 = KSIDE ? 2 * rt : 0;
    const int cs1 = KSIDE ? (len + 63) / 64 : min(2 * (rt + 1), (len + 63) / 64);
    const int total = cs1 - cs0;

    if (threadIdx.x == 0) {
        mbar_init(bar_r, 1); mbar_init(bar_full0, 1); mbar_init(bar_full0 + 8, 1);
        mbar_init(bar_sdfull, 1); mbar_init(bar_sdfree, 4); mbar_init(bar_pdfull, 4); mbar_init(bar_outdone, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tS = tmem_base, tdP = tmem_base + 64, tO1 = tmem_base + 128, tO2 = tmem_base + 128 + DP;

    if (warp == 4) {
        if (lane == 0 && total > 0) {
            const uint32_t id64 = idesc_bf16(128, 64), idO = idesc_bf16(128, DP);
            constexpr uint32_t kStageBytesB = (KSIDE ? 4u : 3u) * CB;
            auto load_stage = [&](int n) {
                const int s = n & 1, ctok = tok0 + (cs0 + n) * 64;
                const uint32_t st = sStage + s * 4 * CB, bar = bar_full0 + 8 * s;
                mbar_expect_tx(bar, kStageBytesB);
#pragma unroll
                for (int a = 0; a < DP / 64; ++a) {
                    tma_load_3d(st + a * 8192, &mapC, bar, a * 64, ctok, h);
                    tma_load_3d(st + CB + a * 8192, &mapCG, bar, a * 64, ctok, h);
                }
                tma_load_3d(st + 2 * CB, &mapCt, bar, ctok, 0, h);
                if (KSIDE) tma_load_3d(st + 3 * CB, &mapCGt, bar, ctok, 0, h);
            };
            mbar_expect_tx(bar_r, 2 * RB);
#pragma unroll
            for (int a = 0; a < DP / 64; ++a) {
                tma_load_3d(sR + a * 16384, &mapR, bar_r, a * 64, tok0 + rt * 128, h);
                tma_load_3d(sRG + a * 16384, &mapRG, bar_r, a * 64, tok0 + rt * 128, h);
            }
            load_stage(0);
            mbar_wait(bar_r, 0);
            for (int n = 0; n < total; ++n) {
                const int s = n & 1;
                const uint32_t st = sStage + s * 4 * CB;
                mbar_wait(bar_full0 + 8 * s, (n >> 1) & 1);
                if (n >= 1) mbar_wait(bar_sdfree, (n - 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int ks = 0; ks < DP / 16; ++ks) {
                    const uint64_t aR = make_kmajor_desc(sR + (ks >> 2) * 16384), bC = make_kmajor_desc(st + (ks >> 2) * 8192);
                    umma_bf16(tS, aR + (uint64_t)((ks & 3) * 2), bC + (uint64_t)((ks & 3) * 2), id64, ks ? 1u : 0u);
                }
#pragma unroll
                for (int ks = 0; ks < DP / 16; ++ks) {
                    const uint64_t aRG = make_kmajor_desc(sRG + (ks >> 2) * 16384), bCG = make_kmajor_desc(st + CB + (ks >> 2) * 8192);
                    umma_bf16(tdP, aRG + (uint64_t)((ks & 3) * 2), bCG + (uint64_t)((ks & 3) * 2), id64, ks ? 1u : 0u);
                }
                umma_commit(bar_sdfull);
                if (n >= 1) mbar_wait(bar_outdone, (n - 1) & 1);       // stage s^1 and the P / dS tiles are free again
                if (n + 1 < total) load_stage(n + 1);
                mbar_wait(bar_pdfull, n & 1);
                tc_fence_after();
                const uint64_t adS = make_kmajor_desc(sdS), aP = make_kmajor_desc(sP);
                const uint64_t bCt = make_kmajor_desc(st + 2 * CB), bCGt = make_kmajor_desc(st + 3 * CB);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) umma_bf16(tO1, adS + (uint64_t)(ks * 2), bCt + (uint64_t)(ks * 2), idO, (n | ks) ? 1u : 0u);
                if (KSIDE) {
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) umma_bf16(tO2, aP + (uint64_t)(ks * 2), bCGt + (uint64_t)(ks * 2), idO, (n | ks) ? 1u : 0u);
                }
                umma_commit(bar_outdone);
            }
        }
    } else {
        const int r = threadIdx.x;
        const int ri = rt * 128 + r;                      // row index inside the sequence (query or key)
        const float c2 = p.slopes[h] * kLog2e;
        const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
        float lse_r = 0.f, D_r = 0.f;
        const uint32_t hseed = DROP ? drop_head_seed(p.seed_ptr, p.salt, h) : 0u;
        const int halfT = (p.Tp + 1) >> 1;
        if (!KSIDE && ri < len) {
            lse_r = p.lse_in[(size_t)h * p.Tp + tok0 + ri];
            D_r = p.D[(size_t)h * p.Tp + tok0 + ri];
        }
        for (int n = 0; n < total; ++n) {
            const int c0 = (cs0 + n) * 64;               // first column index inside the sequence
            if (KSIDE) {
                float* sc = s_col + (n & 1) * 128;
                if (r < 64) {
                    const int qi = c0 + r;
                    sc[r] = qi < len ? p.lse_in[(size_t)h * p.Tp + tok0 + qi] : 0.f;
                    sc[64 + r] = qi < len ? p.D[(size_t)h * p.Tp + tok0 + qi] : 0.f;
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
            }
            mbar_wait(bar_sdfull, n & 1);
            tc_fence_after();
            if (n >= 1) mbar_wait(bar_outdone, (n - 1) & 1);
            const float* sc = s_col + (n & 1) * 128;
#pragma unroll 1
            for (int c = 0; c < 2; ++c) {
                uint32_t xs[32], xd[32];
                tmem_ld32(tS + lane_base + c * 32, xs);
                tmem_ld32(tdP + lane_base + c * 32, xd);
                tmem_ld_wait();
                uint32_t pk_p[16], pk_d[16];
#pragma unroll
                for (int jj = 0; jj < 32; jj += 2) {
                    float pv[2], dv[2];
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int ci = c0 + c * 32 + jj + e;          // column index inside the sequence
                        const int qi = KSIDE ? ci : ri, kj = KSIDE ? ri : ci;
                        const float lse_q = KSIDE ? sc[c * 32 + jj + e] : lse_r;
                        const float D_q = KSIDE ? sc[64 + c * 32 + jj + e] : D_r;
                        const float s2 = fmaf(__uint_as_float(xs[jj + e]), p.c1, -c2 * (float)(qi - kj));
                        const bool dead = kj > qi || qi >= len;
                        const float pe = dead ? 0.f : ex2f(s2 - lse_q);
                        const float mk = DROP ? drop_factor(hseed, tok0 + qi, tok0 + kj, halfT, p.drop_thr, p.drop_scale) : 1.f;
                        pv[e] = pe * mk;                                               // dropped probabilities (for dV)
                        dv[e] = pe * (__uint_as_float(xd[jj + e]) * mk - D_q) * p.scale;   // dS = P (dP_d M / (1-p) - D)
                    }
                    pk_p[jj >> 1] = pack_bf16(pv[0], pv[1]);
                    pk_d[jj >> 1] = pack_bf16(dv[0], dv[1]);
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    *reinterpret_cast<uint4*>(sdS_ptr + sw128(r, c * 4 + q)) = make_uint4(pk_d[4 * q], pk_d[4 * q + 1], pk_d[4 * q + 2], pk_d[4 * q + 3]);
                    if (KSIDE)
                        *reinterpret_cast<uint4*>(sP_ptr + sw128(r, c * 4 + q)) = make_uint4(pk_p[4 * q], pk_p[4 * q + 1], pk_p[4 * q + 2], pk_p[4 * q + 3]);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_sdfree);
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_pdfull);
        }
        if (total > 0) {
            mbar_wait(bar_outdone, (total - 1) & 1);
            tc_fence_after();
        }
        const bool valid = ri < len;
        float* o1 = p.out1 + (size_t)(out0 + ri) * p.ld_out + (size_t)h * p.hd;
        float* o2 = KSIDE ? p.out2 + (size_t)(out0 + ri) * p.ld_out + (size_t)h * p.hd : nullptr;
        constexpr int nc = DP / 32;                      // 32-column chunks of each accumulator
#pragma unroll 1
        for (int c = 0; c < (KSIDE ? 2 : 1) * nc; ++c) {
            const int cc = c & (nc - 1);
            uint32_t x[32];
            if (total > 0) {
                tmem_ld32((c < nc ? tO1 : tO2) + lane_base + cc * 32, x);
                tmem_ld_wait();
            } else {
#pragma unroll
                for (int q = 0; q < 32; ++q) x[q] = 0u;
            }
            if (valid) store_cols((c < nc ? o1 : o2) + cc * 32, x, p.hd - cc * 32);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols));
    }
}

// row-major bf16 [T, H, DP]: dims (d, token, head); box = 64 d (one swizzle row) x `rows` tokens of one head
static int map_rm(CUtensorMap* m, const void* ptr, int H, int DP, int T, int rows) {
    const unsigned long long dims[3] = {(unsigned long long)DP, (unsigned long long)T, (unsigned long long)H};
    const unsigned long long strides[2] = {(unsigned long long)H * DP * 2ull, (unsigned long long)DP * 2ull};
    const unsigned box[3] = {64u, (unsigned)rows, 1u};
    return make_map3(m, ptr, true, dims, strides, box);
}
// transposed bf16 [H, DP, Tp]: dims (token, d, head); box = 64 tokens x DP d of one head
static int map_tr(CUtensorMap* m, const void* ptr, int H, int DP, int Tp) {
    const unsigned long long dims[3] = {(unsigned long long)Tp, (unsigned long long)DP, (unsigned long long)H};
    const unsigned long long strides[2] = {(unsigned long long)Tp * 2ull, (unsigned long long)Tp * DP * 2ull};
    const unsigned box[3] = {64u, (unsigned)DP, 1u};
    return make_map3(m, ptr, true, dims, strides, box);
}

template <int DP>
static void attn_attrs() {
    static bool once = false;
    if (!once) {
        cudaFuncSetAttribute(attn_fwd_kernel<DP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd_smem(DP));
        cudaFuncSetAttribute(attn_fwd_kernel<DP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd_smem(DP));
        cudaFuncSetAttribute(attn_bwd_kernel<DP, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_smem(DP));
        cudaFuncSetAttribute(attn_bwd_kernel<DP, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_smem(DP));
        cudaFuncSetAttribute(attn_bwd_kernel<DP, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_smem(DP));
        cudaFuncSetAttribute(attn_bwd_kernel<DP, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd_smem(DP));
        once = true;
    }
}

template <int DP>
static int attn_fwd_launch(const void* q_rm, const void* k_rm, const void* v_tr, const int32_t* tiles, int64_t ntiles,
                           const float* slopes, float softmax_scale, float* O, int64_t ld_o, float* lse, int64_t H, int64_t hd,
                           int64_t T, int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt, cudaStream_t stream) {
    CUtensorMap mQ, mK, mVt;
    int rc = map_rm(&mQ, q_rm, (int)H, DP, (int)T, 128);
    if (!rc) rc = map_rm(&mK, k_rm, (int)H, DP, (int)T, 128);
    if (!rc) rc = map_tr(&mVt, v_tr, (int)H, DP, (int)Tp);
    if (rc) return rc;
    attn_attrs<DP>();
    AttnParams p = {};
    p.tiles = reinterpret_cast<const int4*>(tiles); p.slopes = slopes; p.c1 = softmax_scale * kLog2e; p.scale = softmax_scale;
    p.H = (int)H; p.hd = (int)hd; p.T = (int)T; p.Tp = (int)Tp; p.O = O; p.ld_o = ld_o; p.lse = lse;
    dim3 grid((unsigned)ntiles, (unsigned)H);
    if (dropout_p > 0.f) {
        p.seed_ptr = reinterpret_cast<const long long*>(seed); p.salt = (uint32_t)salt;
        p.drop_thr = (uint32_t)(dropout_p * 65536.0f + 0.5f); p.drop_scale = 1.0f / (1.0f - dropout_p);
        attn_fwd_kernel<DP, true><<<grid, kAttnThreads, fwd_smem(DP), stream>>>(mQ, mK, mVt, p);
    } else {
        attn_fwd_kernel<DP, false><<<grid, kAttnThreads, fwd_smem(DP), stream>>>(mQ, mK, mVt, p);
    }
    RORL_RETURN_LAUNCH();
}

template <int DP>
static int attn_bwd_launch(const void* q_rm, const void* k_rm, const void* v_rm, const void* do_rm, const void* q_tr,
                           const void* k_tr, const void* do_tr, const float* lse, const float* D, const int32_t* tiles,
                           int64_t ntiles, const float* slopes, float softmax_scale, float* dq, float* dk, float* dv,
                           int64_t ld_d, int64_t H, int64_t hd, int64_t T, int64_t Tp, float dropout_p, const int64_t* seed,
                           int64_t salt, cudaStream_t stream) {
    CUtensorMap mQ128, mK128, mV128, mdO128, mQ64, mK64, mV64, mdO64, mQt, mKt, mdOt;
    int rc = map_rm(&mQ128, q_rm, (int)H, DP, (int)T, 128);
    if (!rc) rc = map_rm(&mK128, k_rm, (int)H, DP, (int)T, 128);
    if (!rc) rc = map_rm(&mV128, v_rm, (int)H, DP, (int)T, 128);
    if (!rc) rc = map_rm(&mdO128, do_rm, (int)H, DP, (int)T, 128);
    if (!rc) rc = map_rm(&mQ64, q_rm, (int)H, DP, (int)T, 64);
    if (!rc) rc = map_rm(&mK64, k_rm, (int)H, DP, (int)T, 64);
    if (!rc) rc = map_rm(&mV64, v_rm, (int)H, DP, (int)T, 64);
    if (!rc) rc = map_rm(&mdO64, do_rm, (int)H, DP, (int)T, 64);
    if (!rc) rc = map_tr(&mQt, q_tr, (int)H, DP, (int)Tp);
    if (!rc) rc = map_tr(&mKt, k_tr, (int)H, DP, (int)Tp);
    if (!rc) rc = map_tr(&mdOt, do_tr, (int)H, DP, (int)Tp);
    if (rc) return rc;
    attn_attrs<DP>();
    AttnParams p = {};
    p.tiles = reinterpret_cast<const int4*>(tiles); p.slopes = slopes; p.c1 = softmax_scale * kLog2e; p.scale = softmax_scale;
    p.H = (int)H; p.hd = (int)hd; p.T = (int)T; p.Tp = (int)Tp; p.lse_in = lse; p.D = D; p.ld_out = ld_d;
    dim3 grid((unsigned)ntiles, (unsigned)H);
    const bool drop = dropout_p > 0.f;
    if (drop) {
        p.seed_ptr = reinterpret_cast<const long long*>(seed); p.salt = (uint32_t)salt;
        p.drop_thr = (uint32_t)(dropout_p * 65536.0f + 0.5f); p.drop_scale = 1.0f / (1.0f - dropout_p);
    }
    constexpr int smem = bwd_smem(DP);
    p.out1 = dq; p.out2 = nullptr;
    if (drop) attn_bwd_kernel<DP, false, true><<<grid, kAttnThreads, smem, stream>>>(mQ128, mdO128, mK64, mV64, mKt, mKt, p);
    else attn_bwd_kernel<DP, false, false><<<grid, kAttnThreads, smem, stream>>>(mQ128, mdO128, mK64, mV64, mKt, mKt, p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return 1000 + (int)e;
    p.out1 = dk; p.out2 = dv;
    if (drop) attn_bwd_kernel<DP, true, true><<<grid, kAttnThreads, smem, stream>>>(mK128, mV128, mQ64, mdO64, mQt, mdOt, p);
    else attn_bwd_kernel<DP, true, false><<<grid, kAttnThreads, smem, stream>>>(mK128, mV128, mQ64, mdO64, mQt, mdOt, p);
    RORL_RETURN_LAUNCH();
}

}  // namespace rorl

using namespace rorl;

extern "C" {

int rorl_attn_prep_hd(const float* src, int64_t ld_tok, int64_t nsec, int64_t H, int64_t T, int64_t Tp, const int32_t* gmap,
                      void* rm_bf16, void* tr_bf16, const float* o, int64_t ld_o, float* Dout, int64_t head_dim,
                      cudaStream_t stream) {
    if (!src || (!rm_bf16 && !tr_bf16 && !Dout)) return RORL_ERR_ARG;
    if (nsec <= 0 || H <= 0 || T <= 0 || Tp < T || Tp % 64 || !attn_head_dim_ok(head_dim)) return RORL_ERR_SHAPE;
    if (ld_tok % 4 || (o && ld_o % 4) || (o && (!Dout || nsec != 1))) return RORL_ERR_ALIGN;
    dim3 grid((unsigned)(Tp / 64), (unsigned)H, (unsigned)nsec);
    if (attn_dp(head_dim) == 64)
        attn_prep_kernel<64><<<grid, 256, 0, stream>>>(src, (long long)ld_tok, (int)H, (int)head_dim, (int)T, (int)Tp, gmap,
                                                       (__nv_bfloat16*)rm_bf16, (__nv_bfloat16*)tr_bf16, o, (long long)ld_o, Dout);
    else
        attn_prep_kernel<128><<<grid, 256, 0, stream>>>(src, (long long)ld_tok, (int)H, (int)head_dim, (int)T, (int)Tp, gmap,
                                                        (__nv_bfloat16*)rm_bf16, (__nv_bfloat16*)tr_bf16, o, (long long)ld_o, Dout);
    RORL_RETURN_LAUNCH();
}

int rorl_attn_prep(const float* src, int64_t ld_tok, int64_t nsec, int64_t H, int64_t T, int64_t Tp, const int32_t* gmap,
                   void* rm_bf16, void* tr_bf16, const float* o, int64_t ld_o, float* Dout, cudaStream_t stream) {
    return rorl_attn_prep_hd(src, ld_tok, nsec, H, T, Tp, gmap, rm_bf16, tr_bf16, o, ld_o, Dout, 64, stream);
}

int rorl_attn_fwd_hd(const void* q_rm, const void* k_rm, const void* v_tr, const int32_t* tiles, int64_t ntiles,
                     const float* slopes, float softmax_scale, float* O, int64_t ld_o, float* lse, int64_t H, int64_t T,
                     int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt, int64_t head_dim, cudaStream_t stream) {
    if (!q_rm || !k_rm || !v_tr || !tiles || !slopes || !O) return RORL_ERR_ARG;
    if (dropout_p < 0.f || dropout_p >= 1.f || (dropout_p > 0.f && !seed)) return RORL_ERR_ARG;
    if (ntiles <= 0 || H <= 0 || T <= 0 || Tp % 64 || ld_o % 4 || !attn_head_dim_ok(head_dim)) return RORL_ERR_SHAPE;
    return attn_dp(head_dim) == 64
               ? attn_fwd_launch<64>(q_rm, k_rm, v_tr, tiles, ntiles, slopes, softmax_scale, O, ld_o, lse, H, head_dim, T, Tp,
                                     dropout_p, seed, salt, stream)
               : attn_fwd_launch<128>(q_rm, k_rm, v_tr, tiles, ntiles, slopes, softmax_scale, O, ld_o, lse, H, head_dim, T, Tp,
                                      dropout_p, seed, salt, stream);
}

int rorl_attn_fwd(const void* q_rm, const void* k_rm, const void* v_tr, const int32_t* tiles, int64_t ntiles,
                  const float* slopes, float softmax_scale, float* O, int64_t ld_o, float* lse, int64_t H, int64_t T,
                  int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt, cudaStream_t stream) {
    return rorl_attn_fwd_hd(q_rm, k_rm, v_tr, tiles, ntiles, slopes, softmax_scale, O, ld_o, lse, H, T, Tp, dropout_p, seed, salt, 64, stream);
}

int rorl_attn_bwd_hd(const void* q_rm, const void* k_rm, const void* v_rm, const void* do_rm, const void* q_tr,
                     const void* k_tr, const void* do_tr, const float* lse, const float* D, const int32_t* tiles,
                     int64_t ntiles, const float* slopes, float softmax_scale, float* dq, float* dk, float* dv,
                     int64_t ld_d, int64_t H, int64_t T, int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt,
                     int64_t head_dim, cudaStream_t stream) {
    if (!q_rm || !k_rm || !v_rm || !do_rm || !q_tr || !k_tr || !do_tr || !lse || !D || !tiles || !slopes || !dq || !dk || !dv)
        return RORL_ERR_ARG;
    if (dropout_p < 0.f || dropout_p >= 1.f || (dropout_p > 0.f && !seed)) return RORL_ERR_ARG;
    if (ntiles <= 0 || H <= 0 || T <= 0 || Tp % 64 || ld_d % 4 || !attn_head_dim_ok(head_dim)) return RORL_ERR_SHAPE;
    return attn_dp(head_dim) == 64
               ? attn_bwd_launch<64>(q_rm, k_rm, v_rm, do_rm, q_tr, k_tr, do_tr, lse, D, tiles, ntiles, slopes, softmax_scale, dq,
                                     dk, dv, ld_d, H, head_dim, T, Tp, dropout_p, seed, salt, stream)
               : attn_bwd_launch<128>(q_rm, k_rm, v_rm, do_rm, q_tr, k_tr, do_tr, lse, D, tiles, ntiles, slopes, softmax_scale, dq,
                                      dk, dv, ld_d, H, head_dim, T, Tp, dropout_p, seed, salt, stream);
}

int rorl_attn_bwd(const void* q_rm, const void* k_rm, const void* v_rm, const void* do_rm, const void* q_tr,
                  const void* k_tr, const void* do_tr, const float* lse, const float* D, const int32_t* tiles,
                  int64_t ntiles, const float* slopes, float softmax_scale, float* dq, float* dk, float* dv,
                  int64_t ld_d, int64_t H, int64_t T, int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt,
                  cudaStream_t stream) {
    return rorl_attn_bwd_hd(q_rm, k_rm, v_rm, do_rm, q_tr, k_tr, do_tr, lse, D, tiles, ntiles, slopes, softmax_scale, dq, dk, dv,
                            ld_d, H, T, Tp, dropout_p, seed, salt, 64, stream);
}

}  // extern "C"
