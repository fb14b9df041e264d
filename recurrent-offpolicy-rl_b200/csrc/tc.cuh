// tcgen05 / TMEM / TMA helpers shared by the tensor-core kernels (gemm_bf16.cu, attn.cu), sm_100a only.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace rorl {

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor: 8-row groups are 1024 B apart.
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);          // start address
    d |= (uint64_t)1 << 16;                            // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                  // stride byte offset
    d |= (uint64_t)1 << 46;                            // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                            // SWIZZLE_128B
    return d;
}
// K-major, SWIZZLE_64B (rows of 64 B = 32 bf16): 8-row groups are 512 B apart.
__device__ __forceinline__ uint64_t make_kmajor_desc_sw64(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)4 << 61;                            // SWIZZLE_64B
    return d;
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
// instruction descriptor, kind::f16 with bf16 operands, fp32 accumulate, both operands K-major
__device__ __forceinline__ uint32_t idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// 32 TMEM lanes (this warp's quarter) x 32 consecutive fp32 columns -> 32 registers per lane (lane = row)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

// 3-D map over a row-major [batch][rows][cols] fp32 tensor: box = 32 cols (128 B) x box_rows x 1, SWIZZLE_128B,
// out-of-bounds elements read as zero.
static inline int make_map(CUtensorMap* map, const float* ptr, long long rows, long long cols, long long ld, long long batch,
                    long long batch_stride, int box_rows) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return RORL_ERR_ARG;
    cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(batch > 0 ? batch : 1)};
    cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(batch > 1 ? batch_stride : rows * ld) * 4};
    cuuint32_t box[3] = {32, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? RORL_OK : RORL_ERR_ARG;
}


// General 3-D tiled map (bf16 or fp32 elements), SWIZZLE_128B: dims / strides innermost first, strides in BYTES for
// dimensions 1 and 2, box in elements.
static inline int make_map3(CUtensorMap* map, const void* ptr, bool bf16, const unsigned long long dims[3],
                            const unsigned long long strides_bytes[2], const unsigned box[3]) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return RORL_ERR_ARG;
    cuuint64_t d[3] = {dims[0], dims[1], dims[2]};
    cuuint64_t st[2] = {strides_bytes[0], strides_bytes[1]};
    cuuint32_t bx[3] = {box[0], box[1], box[2]};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), d, st,
                     bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? RORL_OK : RORL_ERR_ARG;
}

}  // namespace rorl
