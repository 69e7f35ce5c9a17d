// tcgen05 / TMA / mbarrier PTX helpers shared by the tensor-core kernels (sm_100a).
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace lpd {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    const uint32_t addr = smem_u32(bar);
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!ok);
}
// same, for the single-thread producer / issuer roles: back off between polls so the spin does not steal issue slots
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    const uint32_t addr = smem_u32(bar);
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(addr), "r"(parity)
            : "memory");
        if (ok) break;
        __nanosleep(40);
    }
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tmap, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Warp-convergent variants: the WHOLE warp executes these with identical operands and elect.sync inside the asm picks the
// issuing lane.  Control flow stays uniform, so ptxas emits ELECT + one predicated UTCHMMA / UTCBAR / UTMALDG; inside a
// divergent `if (lane == 0)` region it has to wrap every such instruction in an elect-and-loop sequence (9-10 instructions
// per MMA on the single issuing thread).
__device__ __forceinline__ void tc_mma_tf32_e(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit_e(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_2d_e(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_e(uint64_t* bar, uint32_t bytes) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}"
        ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, 128-byte swizzled operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);       // start address  [0,14)
    d |= (uint64_t)1 << 16;                            // leading byte offset (unused for swizzled K-major) [16,30)
    d |= (uint64_t)(1024 >> 4) << 32;                  // stride byte offset: 8 rows x 128 B [32,46)
    d |= (uint64_t)1 << 46;                            // descriptor version (Blackwell) [46,48)
    d |= (uint64_t)2 << 61;                            // SWIZZLE_128B [61,64)
    return d;
}

// MN-major operand tile of 32-bit elements built from TMA boxes {32 fp32 along M/N, k rows}.  For tf32 the only MN-major
// layout the tensor core accepts is "128B swizzle with a 32-byte atom" (layout type 1; TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B):
// rows of 128 B, 4-row atoms 512 B apart (stride byte offset), 32-element M/N groups one 32-row box = 4096 B apart
// (leading byte offset).
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(4096 >> 4) << 16;                  // leading byte offset: next 32 elements along M/N
    d |= (uint64_t)(512 >> 4) << 32;                   // stride byte offset: next 4 k-rows
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;                            // SWIZZLE_128B_BASE32B
    return d;
}

// kind::tf32, fp32 accumulate, A and B K-major
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {  // kind::tf32
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}


// host: resolve cuTensorMapEncodeTiled through the runtime (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D tensor [rows][cols] of fp32 or fp16 (type) with row pitch ld (elements), loaded in boxes of box_rows x box_cols;
// out-of-range box elements read as zero
inline int make_tmap(CUtensorMap* m, CUtensorMapDataType type, const void* base, long long rows, long long cols, long long ld,
                     int box_rows, int box_cols, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
    EncodeTiledFn enc = get_encode();
    if (!enc) { snprintf(g_last_error, sizeof(g_last_error), "cuTensorMapEncodeTiled entry point not found"); return LPD_ECUDA; }
    const size_t esize = type == CU_TENSOR_MAP_DATA_TYPE_FLOAT16 ? 2 : 4;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * esize};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, type, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { snprintf(g_last_error, sizeof(g_last_error), "cuTensorMapEncodeTiled failed: CUresult %d", (int)r); return LPD_ECUDA; }
    return LPD_OK;
}

}  // namespace tc
}  // namespace lpd
