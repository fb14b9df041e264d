// tcgen05 GEMM with fp32 parity from a two-term bf16 split ("bf16x3"), sm_100a.
//
//   D[g][M, N] = act( A[g][M, K] * B[g][N, K]^T + bias[g][N] )        g = 0..G-1 (ensemble members)
//
// Replaces the cuBLAS fp32 SGEMMs behind nn.Linear / EnsembleLinear on the update path (ref:
// offpolicy_rnn/models/ensemble_linear_model.py:36-49 einsum -> bmm; smamba in/x/dt/out_proj, ref:
// offpolicy_rnn/models/smamba/mamba.py:176,231-233,252).  The reference runs these in true fp32 (TF32 is never enabled
// there), so one low-precision MMA per product is not enough for the 1e-3 parity budget: every fp32 operand element is
// split as x = hi + lo with hi = bf16(x), lo = bf16(x - hi) (16 mantissa bits kept; the dropped lo*lo term and the
// representation remainder are ~2^-17 relative) and the product is accumulated as lo*hi + hi*lo + hi*hi on
// tcgen05.mma.kind::f16 into the fp32 TMEM accumulator (passes = 2).  passes = 4 issues the hi*hi term alone: what a
// layer the reference runs under bf16 autocast computes.
// Structure (one persistent CTA per SM, 14 warps), two decoupled shared-memory rings:
//   warp 0      TMA producer: raw fp32 A tiles (SWIZZLE_128B, 32 fp32 of K per row) into the RAW ring, and the B operand's
//               bf16 hi / lo tiles (pre-split once per call by split_bf16_kernel: B is the small, endlessly re-read
//               operand -- the weights) straight into the SPLIT ring (SWIZZLE_64B, 64 B of K per row)
//   warps 2-5   splitters: raw fp32 A -> bf16 hi / lo tiles in the same K-major SWIZZLE_64B layout of the SPLIT ring;
//               the raw stage is released to the producer as soon as it has been read, not when the MMAs that use
//               its split copy retire.  (ncu on the first version, which split both operands in the kernel: shared-
//               memory wavefronts -- splitter 768 + tensor core 576 + epilogue 260 per stage -- were the bound, l1tex
//               data pipe 69 % busy with the tensor pipe at 30 %; B was two thirds of the splitter's traffic.)
//   warp 1      MMA issuer: 2 k-steps x 3 tcgen05.mma.kind::f16 (M128 x N{128,256} x K16) per split stage
//   warps 6-13  epilogue: two warps per TMEM lane quarter, each owning half of the accumulator's 32-column chunks:
//               tcgen05.ld, + bias, ELU / GELU, shared-memory transposition, 128-B-row global stores; overlaps the next
//               tile's main loop (double-buffered TMEM).  One warp per scheduler was latency bound (ncu: the epilogue,
//               not the MMA, set the tile time), hence eight
// K only has to be a multiple of 4: B's split copy pads its rows to Kp = K rounded up to 8 (16-byte rows for the
// tensor map) while the map's extent stays K, so TMA zero-fills columns K..Kp-1 and the padding is never written or read.
#include "common.cuh"
#include "tc.cuh"
#include <cuda_bf16.h>

namespace rorl {

constexpr int kBfBM = 128, kBfBK = 32;
constexpr int kBfThreads = 448;
constexpr int kBfEpiWarps = 8;
constexpr int kBfStaging = kBfEpiWarps * 32 * 128;

template <int BN, bool MN = false>
struct BfCfg {
    static constexpr int kRawA = kBfBM * kBfBK * 4;               // 16 KiB
    static constexpr int kRaw = MN ? kRawA + BN * kBfBK * 4 : kRawA;   // TN: the raw ring holds A only; NT: both operands
    static constexpr int kHalfA = kBfBM * kBfBK * 2;              // one bf16 tile of A (hi or lo): 8 KiB
    static constexpr int kHalfB = BN * kBfBK * 2;
    static constexpr int kSplit = 2 * (kHalfA + kHalfB);          // A_hi | A_lo | B_hi | B_lo
    static constexpr int kRawStages = MN ? 3 : (BN == 256 ? 3 : 4);
    static constexpr int kSplitStages = MN ? 3 : (BN == 256 ? 3 : 4);
    static constexpr int kSmem = kRawStages * kRaw + kSplitStages * kSplit + kBfStaging + 1024 + 256;
};

struct BfParams {
    float* D;
    float* Dpre;
    const float* bias;
    int M, N, K, G;
    long long ldd, strideD, strideBias;
    int a_batched, b_batched, act, reduce_g;
    int accum;                  // TN form: D += result (read-modify-write in the epilogue's coalesced row stores)
    int single;                 // hi * hi only: one bf16 MMA per k-step (what a bf16-autocast layer of the reference computes)
    int splits;                 // NT variant: split-K factor; partial s is written at D + s * strideSplit
    long long strideSplit;
};

// exact GELU (torch.nn.GELU default, erf form): the cgpt FFN's activation (ref: TransformerFlashAttention.py:43-57)
__device__ __forceinline__ float bf_gelu(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float bf_elu1(float x) {
    const float e = ex2f(fminf(x, 0.f) * kLog2e) - 1.0f;
    return x > 0.f ? x : e;
}

// 8 fp32 -> 8 bf16 hi (packed in a uint4) and 8 bf16 lo
__device__ __forceinline__ void split8(const float4& a, const float4& b, uint4& hi, uint4& lo) {
    auto two = [](float x, float y, uint32_t& h, uint32_t& l) {
        const __nv_bfloat162 hh = __floats2bfloat162_rn(x, y);
        h = *reinterpret_cast<const uint32_t*>(&hh);
        const float rx = x - __uint_as_float(h << 16);
        const float ry = y - __uint_as_float(h & 0xFFFF0000u);
        const __nv_bfloat162 ll = __floats2bfloat162_rn(rx, ry);
        l = *reinterpret_cast<const uint32_t*>(&ll);
    };
    two(a.x, a.y, hi.x, lo.x);
    two(a.z, a.w, hi.y, lo.y);
    two(b.x, b.y, hi.z, lo.z);
    two(b.z, b.w, hi.w, lo.w);
}

// MN = false: TN form (both operands K-major; B pre-split, see above).  MN = true: weight-gradient form, both operands
// row-major with the REDUCTION over rows (MN-major): TMA delivers each operand as 4 boxes of [32 reduction rows][32 MN
// columns]; the splitters transpose while they split (kind::f16 multiplies K-major operands), writing K-major
// SWIZZLE_64B bf16 rows (row = MN index, 32 reduction values = 64 B) into the split ring -- a separate buffer, so no
// in-place hazard and no block barrier.  Split-K over the (very long) token dimension: partial s is written at
// D + s * strideSplit and the caller sums the partials (deterministic, no atomics).
template <int BN, bool MN, bool ACC = false>
__global__ void __launch_bounds__(kBfThreads, 1)
gemm_bf16x3_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapBhi,
                   const __grid_constant__ CUtensorMap mapBlo, const BfParams p) {
    static_assert(!MN || BN == 128, "the weight-gradient form uses 128 x 128 tiles");
    using Cfg = BfCfg<BN, MN>;
    constexpr int RS = Cfg::kRawStages, SS = Cfg::kSplitStages;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* base_ptr = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t split_base = base + RS * Cfg::kRaw;
    uint8_t* split_ptr = base_ptr + RS * Cfg::kRaw;
    uint8_t* staging = split_ptr + SS * Cfg::kSplit;
    const uint32_t bars = split_base + SS * Cfg::kSplit + kBfStaging;
    // barrier map (8 B each): raw_full[RS], raw_empty[RS], split_full[SS], split_empty[SS], tfull[2], tempty[2], tmem ptr
    auto bar_raw_full = [&](int s) { return bars + 8u * s; };
    auto bar_raw_empty = [&](int s) { return bars + 8u * (RS + s); };
    auto bar_split_full = [&](int s) { return bars + 8u * (2 * RS + s); };
    auto bar_split_empty = [&](int s) { return bars + 8u * (2 * RS + SS + s); };
    auto bar_tfull = [&](int a) { return bars + 8u * (2 * RS + 2 * SS + a); };
    auto bar_tempty = [&](int a) { return bars + 8u * (2 * RS + 2 * SS + 2 + a); };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(staging + kBfStaging + 8 * (2 * RS + 2 * SS + 4));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tilesM = (p.M + kBfBM - 1) / kBfBM, tilesN = (p.N + BN - 1) / BN;
    const int KTg = (p.K + kBfBK - 1) / kBfBK;
    const int nsplit = MN ? p.splits : 1;
    const int ntiles = tilesM * tilesN * (p.reduce_g ? 1 : p.G) * nsplit;
    const int KTs = (KTg + nsplit - 1) / nsplit;                                  // k-tiles per split (NT variant)
    const int KT = MN ? KTs : (p.reduce_g ? KTg * p.G : KTg);

    if (threadIdx.x == 0) {
        for (int s = 0; s < RS; ++s) {
            mbar_init(bar_raw_full(s), 1);
            mbar_init(bar_raw_empty(s), 4);
        }
        for (int s = 0; s < SS; ++s) {
            mbar_init(bar_split_full(s), MN ? 4 : 5);            // 4 splitter warps (+ the producer's expect_tx for B in the TN form)
            mbar_init(bar_split_empty(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(bar_tfull(a), 1);
            mbar_init(bar_tempty(a), kBfEpiWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(2 * BN));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (raw fp32 tiles)
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapBhi) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapBlo) : "memory");
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int tn = tile % tilesN, tm = (tile / tilesN) % tilesM;
                const int g = (tile / (tilesN * tilesM)) % p.G;
                const int sp = tile / (tilesN * tilesM * p.G);
                for (int kt = 0; kt < KT; ++kt, ++it) {
                    const int s = it % RS, ss = it % SS;
                    const int gg = p.reduce_g ? kt / KTg : g, kk = p.reduce_g ? kt % KTg : kt;
                    mbar_wait(bar_raw_empty(s), ((it / RS) & 1) ^ 1);
                    mbar_expect_tx(bar_raw_full(s), Cfg::kRaw);
                    if (MN) {
                        const int r0 = (sp * KTs + kt) * kBfBK;                  // rows beyond the tensor are zero-filled
                        const uint32_t st = base + s * Cfg::kRaw;
#pragma unroll
                        for (int bI = 0; bI < 4; ++bI) {
                            tma_load_3d(st + bI * 4096, &mapA, bar_raw_full(s), tm * kBfBM + 32 * bI, r0, p.a_batched ? g : 0);
                            tma_load_3d(st + Cfg::kRawA + bI * 4096, &mapBhi, bar_raw_full(s), tn * BN + 32 * bI, r0, p.b_batched ? g : 0);
                        }
                    } else {
                        tma_load_3d(base + s * Cfg::kRaw, &mapA, bar_raw_full(s), kk * kBfBK, tm * kBfBM, p.a_batched ? gg : 0);
                        mbar_wait(bar_split_empty(ss), ((it / SS) & 1) ^ 1);
                        mbar_expect_tx(bar_split_full(ss), 2 * Cfg::kHalfB);
                        const uint32_t sb = split_base + ss * Cfg::kSplit + 2 * Cfg::kHalfA;
                        tma_load_3d(sb, &mapBhi, bar_split_full(ss), kk * kBfBK, tn * BN, p.b_batched ? gg : 0);
                        tma_load_3d(sb + Cfg::kHalfB, &mapBlo, bar_split_full(ss), kk * kBfBK, tn * BN, p.b_batched ? gg : 0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            const uint32_t idesc = idesc_bf16(kBfBM, BN);
            uint32_t it = 0, tcount = 0;
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
                const int acc = tcount & 1;
                mbar_wait(bar_tempty(acc), ((tcount >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kt = 0; kt < KT; ++kt, ++it) {
                    const int s = it % SS;
                    mbar_wait(bar_split_full(s), (it / SS) & 1);
                    tc_fence_after();
                    const uint32_t st = split_base + s * Cfg::kSplit;
                    const uint64_t a_hi = make_kmajor_desc_sw64(st), a_lo = make_kmajor_desc_sw64(st + Cfg::kHalfA);
                    const uint64_t b_hi = make_kmajor_desc_sw64(st + 2 * Cfg::kHalfA);
                    const uint64_t b_lo = make_kmajor_desc_sw64(st + 2 * Cfg::kHalfA + Cfg::kHalfB);
#pragma unroll
                    for (int k = 0; k < kBfBK / 16; ++k) {
                        const uint64_t adv = (uint64_t)(k * 16 * 2 >> 4);       // 32 B per k-step inside the 64-B swizzle row
                        const uint32_t first = (kt | k) == 0 ? 0u : 1u;
                        if (!p.single) {
                            umma_bf16(tmem_d, a_lo + adv, b_hi + adv, idesc, first);
                            umma_bf16(tmem_d, a_hi + adv, b_lo + adv, idesc, 1u);
                        }
                        umma_bf16(tmem_d, a_hi + adv, b_hi + adv, idesc, p.single ? first : 1u);
                    }
                    umma_commit(bar_split_empty(s));
                }
                umma_commit(bar_tfull(acc));
            }
        }
    } else if (warp < 6) {
        // ------------------------------------------------------------------ splitters: fp32 raw -> bf16 hi / lo
        // item = (row r, pair j of 16-byte raw chunks): raw chunks 2j and 2j+1 of the row (8 fp32, chunk c sits at
        // physical chunk c ^ (r & 7) of the 128-byte row) become one 16-byte bf16 chunk j of the 64-byte bf16 row,
        // stored at physical chunk j ^ ((r >> 1) & 3) (SWIZZLE_64B: address bits 4-5 ^= bits 7-8).
        const int t = threadIdx.x - 64;                                          // 0..127
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            for (int kt = 0; kt < KT; ++kt, ++it) {
                const int rs = it % RS, ss = it % SS;
                mbar_wait(bar_raw_full(rs), (it / RS) & 1);
                mbar_wait(bar_split_empty(ss), ((it / SS) & 1) ^ 1);
                const uint8_t* raw = base_ptr + rs * Cfg::kRaw;
                uint8_t* sp = split_ptr + ss * Cfg::kSplit;
                if (MN) {
                    // thread = (32-column box blk, MN column mn of it = lane): for each of the 4 chunks of 8 reduction rows,
                    // 8 conflict-free LDS.32 down the column (a warp reads one 128-byte raw row per instruction), split,
                    // one 16-byte store per half into row blk * 32 + lane of the K-major bf16 tile
                    const int blk = t >> 5;
#pragma unroll
                    for (int op = 0; op < 2; ++op) {
                        const uint8_t* src = raw + op * Cfg::kRawA + blk * 4096;
                        const int mn = blk * 32 + lane;
                        uint8_t* drow = sp + (op ? 2 * Cfg::kHalfA : 0) + mn * 64;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            float v[8];
#pragma unroll
                            for (int rr = 0; rr < 8; ++rr) {
                                const int r = 8 * j + rr;
                                v[rr] = *reinterpret_cast<const float*>(src + r * 128 + ((((lane >> 2) ^ (r & 7)) << 4) | ((lane & 3) << 2)));
                            }
                            uint4 hi, lo;
                            split8(make_float4(v[0], v[1], v[2], v[3]), make_float4(v[4], v[5], v[6], v[7]), hi, lo);
                            uint8_t* dst = drow + ((j ^ ((mn >> 1) & 3)) << 4);
                            *reinterpret_cast<uint4*>(dst) = hi;
                            *reinterpret_cast<uint4*>(dst + (op ? Cfg::kHalfB : Cfg::kHalfA)) = lo;
                        }
                    }
                } else
#pragma unroll
                for (int i = 0; i < kBfBM * 4 / 128; ++i) {
                    const int idx = t + 128 * i;
                    const int r = idx >> 2, j = idx & 3;
                    const uint8_t* src = raw + r * 128;
                    const float4 v0 = *reinterpret_cast<const float4*>(src + (((2 * j) ^ (r & 7)) << 4));
                    const float4 v1 = *reinterpret_cast<const float4*>(src + (((2 * j + 1) ^ (r & 7)) << 4));
                    uint4 hi, lo;
                    split8(v0, v1, hi, lo);
                    uint8_t* dst = sp + r * 64 + ((j ^ ((r >> 1) & 3)) << 4);
                    *reinterpret_cast<uint4*>(dst) = hi;
                    *reinterpret_cast<uint4*>(dst + Cfg::kHalfA) = lo;
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(bar_split_full(ss));
                    mbar_arrive(bar_raw_empty(rs));
                }
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue
        const int q = warp & 3;
        const int hf = (warp - 6) >> 2;
        uint8_t* stg = staging + (warp - 6) * 4096;
        uint32_t tcount = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
            const int tn = tile % tilesN, tm = (tile / tilesN) % tilesM;
            const int g = (tile / (tilesN * tilesM)) % p.G;
            const int acc = tcount & 1;
            mbar_wait(bar_tfull(acc), (tcount >> 1) & 1);
            tc_fence_after();
            const int sp = tile / (tilesN * tilesM * p.G);
            const long long obase = (long long)g * p.strideD + (long long)sp * p.strideSplit;
            const int row0 = tm * kBfBM + q * 32;
            const float* bias = p.bias ? p.bias + (long long)g * p.strideBias : nullptr;
            auto flush = [&](const float4 (&o)[8], float* out, int col0, bool add) {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<float4*>(stg + lane * 128 + ((j ^ (lane & 7)) << 4)) = o[j];
                __syncwarp();
                // accumulate form: all eight addends are fetched before the first store -- loads interleaved with the
                // stores to the same buffer cannot be reordered by the compiler, which made the read-modify-write eight
                // dependent DRAM round trips per 32 x 32 block (ncu: 95 us for the K = 80 GEMM that takes 25 us without)
                float4 cin[ACC ? 8 : 1];
                if (ACC && add) {
#pragma unroll
                    for (int rr = 0; rr < 8; ++rr) {
                        const int grow = row0 + rr * 4 + (lane >> 3), col = col0 + (lane & 7) * 4;
                        cin[rr] = (grow < p.M && col < p.N)
                                      ? __ldcs(reinterpret_cast<const float4*>(out + obase + (long long)grow * p.ldd + col))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
#pragma unroll
                for (int rr = 0; rr < 8; ++rr) {
                    const int rloc = rr * 4 + (lane >> 3), ch = lane & 7;
                    float4 v = *reinterpret_cast<const float4*>(stg + rloc * 128 + ((ch ^ (rloc & 7)) << 4));
                    const int grow = row0 + rloc, col = col0 + ch * 4;
                    if (ACC && add) { v.x += cin[ACC ? rr : 0].x; v.y += cin[ACC ? rr : 0].y; v.z += cin[ACC ? rr : 0].z; v.w += cin[ACC ? rr : 0].w; }
                    if (grow < p.M && col < p.N)
                        *reinterpret_cast<float4*>(out + obase + (long long)grow * p.ldd + col) = v;
                }
                __syncwarp();
            };
            constexpr int kHalves = BN / 128;
#pragma unroll 1
            for (int half = 0; half < kHalves; ++half) {
                const int chunk0 = (BN / 64) * hf + 2 * half;
                uint32_t r[2][32];
#pragma unroll
                for (int cc = 0; cc < 2; ++cc)
                    tmem_ld32(tmem_base + acc * BN + (chunk0 + cc) * 32 + ((uint32_t)(q * 32) << 16), r[cc]);
                tmem_ld_wait();
                if (half == kHalves - 1) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_tempty(acc));
                }
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) {
                    const int col0 = tn * BN + (chunk0 + cc) * 32;
                    if (col0 >= p.N) break;
                    float4 o[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        o[j] = make_float4(__uint_as_float(r[cc][4 * j]), __uint_as_float(r[cc][4 * j + 1]), __uint_as_float(r[cc][4 * j + 2]),
                                           __uint_as_float(r[cc][4 * j + 3]));
                        if (bias && col0 + 4 * j < p.N) {
                            const float4 bv = __ldg(reinterpret_cast<const float4*>(bias + col0 + 4 * j));
                            o[j].x += bv.x; o[j].y += bv.y; o[j].z += bv.z; o[j].w += bv.w;
                        }
                    }
                    if (p.Dpre) flush(o, p.Dpre, col0, false);
                    if (p.act == 1) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) { o[j].x = bf_elu1(o[j].x); o[j].y = bf_elu1(o[j].y); o[j].z = bf_elu1(o[j].z); o[j].w = bf_elu1(o[j].w); }
                    } else if (p.act == 2) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) { o[j].x = bf_gelu(o[j].x); o[j].y = bf_gelu(o[j].y); o[j].z = bf_gelu(o[j].z); o[j].w = bf_gelu(o[j].w); }
                    }
                    flush(o, p.D, col0, p.accum != 0);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * BN));
    }
}

static int bf_sms() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaFuncSetAttribute(gemm_bf16x3_kernel<128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BfCfg<128>::kSmem);
        cudaFuncSetAttribute(gemm_bf16x3_kernel<256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BfCfg<256>::kSmem);
        cudaFuncSetAttribute(gemm_bf16x3_kernel<128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BfCfg<128, true>::kSmem);
        cudaFuncSetAttribute(gemm_bf16x3_kernel<128, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BfCfg<128>::kSmem);
        cudaFuncSetAttribute(gemm_bf16x3_kernel<256, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BfCfg<256>::kSmem);
    }
    return sms;
}

// Row stride (bf16 elements) of B's split copy: K rounded up to 8, so that every row is a 16-byte multiple as the tensor
// map requires.  The columns K..Kp-1 are never written: the map's extent is K and TMA zero-fills beyond it.
__host__ __device__ constexpr long long padded_k(long long K) { return (K + 7) & ~7LL; }

// fp32 [G][rows, cols] (row stride ld, group stride gs) -> bf16 hi / lo [G][rows, Kp] (Kp = padded_k(cols))
__global__ void __launch_bounds__(256) split_bf16_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ hi,
                                                         __nv_bfloat16* __restrict__ lo, int rows, int cols, long long ld, long long gs,
                                                         long long total4) {
    const long long Kp = padded_k(cols);
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total4; i += (long long)gridDim.x * 256) {
        const long long e = i * 4;
        const int c = (int)(e % cols);
        const long long rg = e / cols;
        const int r = (int)(rg % rows);
        const long long g = rg / rows;
        const long long o = rg * Kp + c;
        const float4 v = *reinterpret_cast<const float4*>(w + g * gs + (long long)r * ld + c);
        const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
        const uint32_t u0 = *reinterpret_cast<const uint32_t*>(&h0), u1 = *reinterpret_cast<const uint32_t*>(&h1);
        const __nv_bfloat162 l0 = __floats2bfloat162_rn(v.x - __uint_as_float(u0 << 16), v.y - __uint_as_float(u0 & 0xFFFF0000u));
        const __nv_bfloat162 l1 = __floats2bfloat162_rn(v.z - __uint_as_float(u1 << 16), v.w - __uint_as_float(u1 & 0xFFFF0000u));
        *reinterpret_cast<uint2*>(hi + o) = make_uint2(u0, u1);
        *reinterpret_cast<uint2*>(lo + o) = make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
    }
}

// the same from the TRANSPOSED source: fp32 [G][K rows, N cols] (row stride ld) -> bf16 hi / lo [G][N, Kp].  nn.Linear's
// input-gradient GEMM multiplies by W, not W^T; the K-major copy the MMA wants is made here instead of by an ATen transposition.
__global__ void __launch_bounds__(256) split_bf16_t_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ hi,
                                                           __nv_bfloat16* __restrict__ lo, int N, int K, long long ld, long long gs) {
    __shared__ float tile[32][33];
    const int n0 = blockIdx.x * 32, k0 = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const long long Kp = padded_k(K);
    w += (long long)blockIdx.z * gs;
    const long long obase = (long long)blockIdx.z * N * Kp;
    for (int j = ty; j < 32; j += 8) {
        const int k = k0 + j, n = n0 + tx;
        tile[j][tx] = (k < K && n < N) ? __ldg(w + (long long)k * ld + n) : 0.f;
    }
    __syncthreads();
    for (int j = ty; j < 32; j += 8) {
        const int n = n0 + j, k = k0 + tx;
        if (n < N && k < K) {
            const float x = tile[tx][j];
            const __nv_bfloat16 h = __float2bfloat16_rn(x);
            hi[obase + (long long)n * Kp + k] = h;
            lo[obase + (long long)n * Kp + k] = __float2bfloat16_rn(x - __bfloat162float(h));
        }
    }
}

// Many B operands in one launch: job j = one operand (G groups of [N, K], source either [N, K] rows or, transposed, [K, N]
// rows with row stride ld) -> its bf16 hi | lo copy in the layout rorl_gemm_tn reads.  grid = (32 x 32 tiles, jobs);
// the jobs table lives in device memory (it is static: weights sit in fixed arenas, the copies in persistent buffers).
struct SplitJob {
    const float* src;
    __nv_bfloat16* dst;          // hi [G][N][Kp] at dst, lo at dst + G * N * Kp
    int N, K, G, transposed;
    long long ld, gs;
};
__global__ void __launch_bounds__(256) split_bf16_multi_kernel(const SplitJob* __restrict__ jobs) {
    __shared__ float tile[32][33];
    const SplitJob jb = jobs[blockIdx.y];
    const int tn = (jb.N + 31) / 32, tk = (jb.K + 31) / 32;
    const long long ntile = (long long)tn * tk * jb.G;
    const long long Kp = padded_k(jb.K);
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    __nv_bfloat16* hi = jb.dst;
    __nv_bfloat16* lo = jb.dst + (long long)jb.G * jb.N * Kp;
    for (long long t = blockIdx.x; t < ntile; t += gridDim.x) {
        const int g = (int)(t / ((long long)tn * tk));
        const int rem = (int)(t % ((long long)tn * tk));
        const int n0 = (rem / tk) * 32, k0 = (rem % tk) * 32;
        const float* w = jb.src + (long long)g * jb.gs;
        const long long obase = (long long)g * jb.N * Kp;
        __syncthreads();
        for (int j = ty; j < 32; j += 8) {
            // tile[a][b]: a = n - n0, b = k - k0
            if (jb.transposed) {                   // source rows are k: read along n (contiguous), store transposed
                const int k = k0 + j, n = n0 + tx;
                tile[tx][j] = (k < jb.K && n < jb.N) ? __ldg(w + (long long)k * jb.ld + n) : 0.f;
            } else {
                const int n = n0 + j, k = k0 + tx;
                tile[j][tx] = (n < jb.N && k < jb.K) ? __ldg(w + (long long)n * jb.ld + k) : 0.f;
            }
        }
        __syncthreads();
        for (int j = ty; j < 32; j += 8) {
            const int n = n0 + j, k = k0 + tx;
            if (n < jb.N && k < jb.K) {
                const float x = tile[j][tx];
                const __nv_bfloat16 h = __float2bfloat16_rn(x);
                hi[obase + (long long)n * Kp + k] = h;
                lo[obase + (long long)n * Kp + k] = __float2bfloat16_rn(x - __bfloat162float(h));
            }
        }
    }
}

// 3-D map over a bf16 [batch][rows][cols] tensor with row stride ld elements (rows contiguous, batches rows * ld apart):
// box = 32 cols (64 B) x box_rows x 1, SWIZZLE_64B, elements beyond `cols` read as zero.
static int make_map_bf16(CUtensorMap* map, const void* ptr, long long rows, long long cols, long long ld, long long batch,
                         int box_rows) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return RORL_ERR_ARG;
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(batch > 0 ? batch : 1)};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)rows * ld * 2};
    cuuint32_t box[3] = {32, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? RORL_OK : RORL_ERR_ARG;
}

}  // namespace rorl

using namespace rorl;

extern "C" {

// D[g] = act(A[g] B[g]^T + bias[g]): contract in include/rorl_b200.h.  `work` receives B's bf16 hi | lo copy
// [GB][N][Kp] (GB = G if B is batched, else 1); transb bit 0: B is stored [K, N] (row stride ldb) and is transposed by
// the splitting pass; bit 1: `work` already holds the copy (rorl_split_bf16_multi).
int rorl_gemm_tn(const float* A, const float* B, const float* bias, float* D, float* Dpre, int64_t M, int64_t N, int64_t K, int64_t G,
                 int64_t lda, int64_t ldb, int64_t ldd, int64_t strideA, int64_t strideB, int64_t strideD,
                 int64_t strideBias, int act, int passes, int reduce_g, int transb, void* work, cudaStream_t stream) {
    if (!A || !B || !D) return RORL_ERR_ARG;
    if (passes != 2 && passes != 4) return RORL_ERR_ARG;         // two-term split (2) or its hi * hi term alone (4)
    if (transb & ~3) return RORL_ERR_ARG;
    if ((act & ~7) || (act & 3) == 3) return RORL_ERR_ARG;
    if (M <= 0 || N <= 0 || K <= 0 || G <= 0) return RORL_ERR_SHAPE;
    if (K % 4 || N % 4 || lda % 4 || ldb % 4 || ldd % 4 || strideA % 4 || strideB % 4 || strideD % 4 || strideBias % 4)
        return RORL_ERR_ALIGN;
    if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B) | reinterpret_cast<uintptr_t>(D) |
         reinterpret_cast<uintptr_t>(bias) | reinterpret_cast<uintptr_t>(Dpre)) & 15)
        return RORL_ERR_ALIGN;
    if (reduce_g && (!strideA || !strideB)) return RORL_ERR_ARG;
    if (!work || (reinterpret_cast<uintptr_t>(work) & 15)) return RORL_ERR_WORKSPACE;
    const int64_t GB = strideB ? G : 1, Kp = padded_k(K);
    __nv_bfloat16* bhi = reinterpret_cast<__nv_bfloat16*>(work);
    __nv_bfloat16* blo = bhi + GB * N * Kp;
    if (transb & 2) {
        // the caller keeps B's split copy up to date itself (rorl_split_bf16_multi after every weight change): nothing to do
    } else if (transb & 1) {
        dim3 grid((unsigned)((N + 31) / 32), (unsigned)((K + 31) / 32), (unsigned)GB);
        split_bf16_t_kernel<<<grid, 256, 0, stream>>>(B, bhi, blo, (int)N, (int)K, ldb, strideB);
    } else {
        const long long total4 = (long long)GB * N * K / 4;
        long long nb = (total4 + 255) / 256;
        if (nb > 148 * 4) nb = 148 * 4;
        split_bf16_kernel<<<(unsigned)nb, 256, 0, stream>>>(B, bhi, blo, (int)N, (int)K, ldb, strideB, total4);
    }
    CUtensorMap mapA, mapBhi, mapBlo;
    const bool wide = N > 128;                                   // 128 x 256 tiles read the A tile once for twice the columns
    const int bn = wide ? 256 : 128;
    int rc = make_map(&mapA, A, M, K, lda, strideA ? G : 1, strideA, kBfBM);
    if (rc) return rc;
    rc = make_map_bf16(&mapBhi, bhi, N, K, Kp, GB, bn);
    if (rc) return rc;
    rc = make_map_bf16(&mapBlo, blo, N, K, Kp, GB, bn);
    if (rc) return rc;
    BfParams p;
    p.D = D; p.Dpre = Dpre; p.bias = bias; p.M = (int)M; p.N = (int)N; p.K = (int)K; p.G = (int)G;
    p.ldd = ldd; p.strideD = strideD; p.strideBias = strideBias;
    p.a_batched = strideA != 0; p.b_batched = strideB != 0; p.act = act & 3; p.accum = (act & 4) != 0; p.reduce_g = reduce_g != 0;
    p.single = passes == 4;
    p.splits = 1; p.strideSplit = 0;
    const int sms = bf_sms();
    const long long tiles = ((M + kBfBM - 1) / kBfBM) * ((N + bn - 1) / bn) * (reduce_g ? 1 : G);
    const int grid = (int)(tiles < sms ? tiles : sms);
    if (wide && p.accum)
        gemm_bf16x3_kernel<256, false, true><<<grid, kBfThreads, BfCfg<256>::kSmem, stream>>>(mapA, mapBhi, mapBlo, p);
    else if (p.accum)
        gemm_bf16x3_kernel<128, false, true><<<grid, kBfThreads, BfCfg<128>::kSmem, stream>>>(mapA, mapBhi, mapBlo, p);
    else if (wide)
        gemm_bf16x3_kernel<256, false><<<grid, kBfThreads, BfCfg<256>::kSmem, stream>>>(mapA, mapBhi, mapBlo, p);
    else
        gemm_bf16x3_kernel<128, false><<<grid, kBfThreads, BfCfg<128>::kSmem, stream>>>(mapA, mapBhi, mapBlo, p);
    RORL_RETURN_LAUNCH();
}

// B operands whose split copy the CALLER maintains (transb bit 1 of rorl_gemm_tn): (re)build many of them in one launch.
int rorl_split_bf16_multi(const void* jobs, int64_t njobs, cudaStream_t stream) {
    if (!jobs && njobs > 0) return RORL_ERR_ARG;
    if (njobs < 0 || njobs > 65535) return RORL_ERR_SHAPE;
    if (njobs == 0) return RORL_OK;
    dim3 grid(64u, (unsigned)njobs);
    split_bf16_multi_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const SplitJob*>(jobs));
    RORL_RETURN_LAUNCH();
}

// bytes of `work` rorl_gemm_tn needs: B's bf16 hi | lo copies, [GB][N][Kp] each
int64_t rorl_gemm_tn_work_bytes(int64_t N, int64_t K, int64_t G, int64_t strideB, int passes) {
    if (passes != 2 && passes != 4) return RORL_ERR_ARG;
    return 2 * (strideB ? G : 1) * N * padded_k(K) * 2;
}

// Split-K factor rorl_gemm_nt uses for a [M x N] output reduced over R rows in G batches (the caller sizes D with it).
int rorl_gemm_nt_splits(int64_t M, int64_t N, int64_t R, int64_t G) {
    if (M <= 0 || N <= 0 || R <= 0 || G <= 0) return RORL_ERR_SHAPE;
    const long long tiles = ((M + kBfBM - 1) / kBfBM) * ((N + 127) / 128) * G;
    const long long kt = (R + kBfBK - 1) / kBfBK;
    long long s = (2 * 148 + tiles - 1) / tiles;
    const long long smax = kt / 4 > 0 ? kt / 4 : 1;
    if (s > smax) s = smax;
    if (s < 1) s = 1;
    return (int)s;
}

// D[s][g][M, N] = sum over the s-th slice of rows r of A[g][r, M]^T B[g][r, N]   (both operands MN-major: the
// reduction runs over ROWS).  Weight gradients: dW[n, k] = sum_m dY[m, n] X[m, k] with A = dY, B = X.
// splits must equal rorl_gemm_nt_splits(M, N, R, G); the caller sums the partials over s.
int rorl_gemm_nt(const float* A, const float* B, float* D, int64_t M, int64_t N, int64_t R, int64_t G, int64_t lda,
                 int64_t ldb, int64_t ldd, int64_t strideA, int64_t strideB, int64_t strideD, int64_t splits,
                 int64_t strideSplit, int passes, cudaStream_t stream) {
    if (!A || !B || !D) return RORL_ERR_ARG;
    if (passes != 2 && passes != 4) return RORL_ERR_ARG;
    if (M <= 0 || N <= 0 || R <= 0 || G <= 0 || splits <= 0) return RORL_ERR_SHAPE;
    if (M % 4 || N % 4 || lda % 4 || ldb % 4 || ldd % 4 || strideA % 4 || strideB % 4 || strideD % 4 || strideSplit % 4)
        return RORL_ERR_ALIGN;
    if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B) | reinterpret_cast<uintptr_t>(D)) & 15)
        return RORL_ERR_ALIGN;
    if (splits != rorl_gemm_nt_splits(M, N, R, G)) return RORL_ERR_ARG;
    CUtensorMap mapA, mapB;
    int rc = make_map(&mapA, A, R, M, lda, strideA ? G : 1, strideA, kBfBK);
    if (rc) return rc;
    rc = make_map(&mapB, B, R, N, ldb, strideB ? G : 1, strideB, kBfBK);
    if (rc) return rc;
    BfParams p;
    p.D = D; p.Dpre = nullptr; p.bias = nullptr; p.M = (int)M; p.N = (int)N; p.K = (int)R; p.G = (int)G;
    p.ldd = ldd; p.strideD = strideD; p.strideBias = 0;
    p.a_batched = strideA != 0; p.b_batched = strideB != 0; p.act = 0; p.accum = 0; p.reduce_g = 0; p.single = passes == 4;
    p.splits = (int)splits; p.strideSplit = strideSplit;
    const int sms = bf_sms();
    const long long tiles = ((M + kBfBM - 1) / kBfBM) * ((N + 127) / 128) * G * splits;
    const int grid = (int)(tiles < sms ? tiles : sms);
    gemm_bf16x3_kernel<128, true><<<grid, kBfThreads, BfCfg<128, true>::kSmem, stream>>>(mapA, mapB, mapB, p);
    RORL_RETURN_LAUNCH();
}

}  // extern "C"
