// Tensor-core GEMM for sm_100a: TMA-fed, tcgen05.mma kind::tf32, fp32 accumulators in TMEM, fused
// per-column affine + activation epilogue.  "fast" arithmetic path for the dense 1x1-conv / matmul layers
// (reference lpdnet_model.py:249-262 conv stacks, PointNetVlad.py:48 soft-assignment) — fp32 operands are
// consumed as TF32 (10-bit mantissa) by the tensor core, products accumulate in fp32.
//
//     C[m][n] = act(scale[n] * sum_k A[m][k] * B[n][k] + shift[n])      A [M][K], B [N][K], both K-contiguous
//
// Persistent warp-specialised CTA (one per SM), 320 threads:
//   warp 0    TMA producer: cp.async.bulk.tensor 2-D boxes (128B swizzle) of A (128 x 32 fp32) and B (BN x 32 fp32)
//             into a STAGES-deep shared-memory ring, completion on mbarriers
//   warp 1    MMA issuer: one thread issues tcgen05.mma (M=128, N=BN, K=8) x4 per ring slot, tcgen05.commit
//             releases the slot; two accumulator stages in TMEM so the epilogue of tile i overlaps tile i+1
//   warps 2-9 epilogue (two per TMEM lane quarter, each owning half of the tile's columns): tcgen05.ld 32 lanes x
//             32 columns, raw accumulators transposed through an XOR-swizzled 4 KB per-warp staging buffer, then
//             affine + activation applied on the way out so that every st.global.v4 instruction writes four full
//             128-byte lines.  (TMA stores were measured slower here: they queue behind the producer's prefetch.)
//
// The same kernel also runs with FP16 operands (kind::f16, fp32 accumulation; template parameter TIN = __half): 64 halves per
// 128-byte shared-memory row, K = 16 per MMA — the byte geometry of the pipeline is unchanged — and can write its output as
// fp16 (OUT_HALF).  That is the "f16" precision mode of the eval path: operands rounded to nearest fp16 (11 significant
// bits, vs the 10-bit TRUNCATION kind::tf32 applies to fp32 operands), twice the tensor rate and half the operand bytes.
#include "tc_common.cuh"
#include <cuda_fp16.h>

namespace lpd {
namespace tc {

constexpr int BM = 128;      // UMMA M
constexpr int BK = 32;       // fp32 elements per smem row = 128 bytes = one swizzle span (fp16: 64 elements)
constexpr int UMMA_K = 8;    // tf32 (fp16: 16) — 32 bytes of K per MMA either way
constexpr int EPI_WARPS = 8;
constexpr int THREADS = 64 + 32 * EPI_WARPS;

struct Params {
    float* C = nullptr; int ldc = 0; int M = 0, N = 0, K = 0;
    const float* scale = nullptr; const float* shift = nullptr;
    float neg_slope = 1.f;   // act(v) = max(v, v * neg_slope), see act_neg_slope
    int tiles_m = 0, tiles_n = 0;
    int batch = 1; long long strideC = 0;   // TN: slice z contracts rows [z*K, (z+1)*K) of both operands into C + z*strideC
    int bM = 0, bN = 0;             // !TN, batch > 1: slice z multiplies rows [z*bM, ..) of A with rows [z*bN, ..) of B into C rows z*bM ..
    int accumulate = 0;             // !TN: C += result (the epilogue reads C)
    // EPI == 1 (BN == 64): row softmax of the affine result instead of the activation; C (fp32, may be null), a_h (fp16 copy, may
    // be null) and apart[row block of 32][64] = the column sums of every 32-row block (may be null)
    __half* a_h = nullptr; float* apart = nullptr;
};

// TN == false:  C[m][n] = sum_k A[m][k] B[n][k]      (both operands K-contiguous: "K-major" UMMA tiles)
// TN == true :  C[z][m][n] = sum_k A[z*K + k][m] B[z*K + k][n]   (both operands stored [k][m|n], i.e. "MN-major":
//               the weight-gradient / NetVLAD-aggregate contraction over the rows of two point-major maps).  An MN-major
//               operand tile (128B swizzle, 32-byte atom — the only MN-major layout kind::tf32 accepts) is a row of TMA boxes
//               {32 floats, 32 k-rows}: 4-row atoms 512 B apart (SBO), 32-element MN groups one box = 4096 B apart (LBO);
//               a K=8 MMA step advances the start address by two atoms (1024 B).
__device__ __forceinline__ void tc_mma_f16_e(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// kind::f16, fp16 operands (format 0), fp32 accumulate
__host__ __device__ constexpr uint32_t make_idesc_h(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// MN-major fp16 operand tile built from TMA boxes {64 halves along M/N (128 B), 64 k-rows}, plain 128B swizzle: 8-k-row atoms
// 1024 B apart (stride byte offset), 64-element M/N groups one box = 8192 B apart (leading byte offset)
__device__ __forceinline__ uint64_t make_smem_desc_mn_h(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(8192 >> 4) << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;                            // SWIZZLE_128B
    return d;
}

template <int BN, int STAGES, bool TN, typename TIN = float, bool OUT_HALF = false, int EPI = 0>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tf32_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, Params p) {
    constexpr bool HALF = sizeof(TIN) == 2;
    constexpr int BKE = HALF ? 2 * BK : BK;              // K elements per 128-byte shared-memory row / per ring slot
    constexpr int MNB = HALF ? 64 : 32;                  // TN: M/N elements per TMA box (128 bytes)
    constexpr uint32_t A_BYTES = BM * BK * 4, B_BYTES = BN * BK * 4, STAGE_BYTES = A_BYTES + B_BYTES;
    constexpr uint32_t TMEM_COLS = 2 * BN;  // two accumulator stages (power of two >= 32 for BN in {64,128,256})
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();       // 128B-swizzle atoms need 1024-byte aligned tiles
    float* cstage = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);          // [EPI_WARPS][32 rows][32 cols]
    uint64_t* full = reinterpret_cast<uint64_t*>(cstage + EPI_WARPS * 32 * 32);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float* xch = reinterpret_cast<float*>(tmem_slot + 2);       // EPI == 1: [2][4 quarters][2 halves][32 rows] row max / row sum
    static_assert(EPI == 0 || (BN == 64 && !TN && !OUT_HALF), "the softmax epilogue covers one 64-column tile");

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_kb = (p.K + BKE - 1) / BKE;
    const int tiles_mn = p.tiles_m * p.tiles_n;
    const int num_tiles = tiles_mn * p.batch;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        {   // whole warp, elect.sync picks the issuing lane (see tc_common.cuh)
            int stage = 0; uint32_t phase = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
                const int z = t / tiles_mn, tt = t % tiles_mn;
                const int m0 = (tt / p.tiles_n) * BM, n0 = (tt % p.tiles_n) * BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx_e(&full[stage], STAGE_BYTES);
                    uint8_t* sa = smem + stage * STAGE_BYTES;
                    if (TN) {
                        const int k0 = z * p.K + kb * BKE;        // boxes of {MNB elements, BKE k-rows}: 4096 B (fp32) / 8192 B (fp16)
#pragma unroll
                        for (int i = 0; i < BM / MNB; ++i) tma_load_2d_e(sa + i * (MNB * 128), &tmap_a, &full[stage], m0 + i * MNB, k0);
#pragma unroll
                        for (int i = 0; i < BN / MNB; ++i) tma_load_2d_e(sa + A_BYTES + i * (MNB * 128), &tmap_b, &full[stage], n0 + i * MNB, k0);
                    } else {
                        tma_load_2d_e(sa, &tmap_a, &full[stage], kb * BKE, z * p.bM + m0);
                        tma_load_2d_e(sa + A_BYTES, &tmap_b, &full[stage], kb * BKE, z * p.bN + n0);
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        {   // whole warp, elect.sync picks the issuing lane (see tc_common.cuh)
            constexpr uint32_t idesc = (HALF ? make_idesc_h(BM, BN) : make_idesc(BM, BN)) | (TN ? ((1u << 15) | (1u << 16)) : 0u);   // a_major / b_major = MN
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
                    if (TN && HALF) {
                        const uint64_t da = make_smem_desc_mn_h(sa), db = make_smem_desc_mn_h(sa + A_BYTES);
#pragma unroll
                        for (int k = 0; k < 4; ++k)                // 16 k-rows (2048 B) per K=16 step, 64 k-rows per slot
                            tc_mma_f16_e(tmem_d, da + (uint64_t)(k * 2048 >> 4), db + (uint64_t)(k * 2048 >> 4), idesc, (kb | k) != 0 ? 1u : 0u);
                    } else if (TN) {
                        const uint64_t da = make_smem_desc_mn(sa), db = make_smem_desc_mn(sa + A_BYTES);
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k)      // 8 k-rows (1024 B) per K=8 step
                            tc_mma_tf32_e(tmem_d, da + (uint64_t)(k * 1024 >> 4), db + (uint64_t)(k * 1024 >> 4), idesc,
                                        (kb | k) != 0 ? 1u : 0u);
                    } else {
                        const uint64_t da = make_smem_desc(sa), db = make_smem_desc(sa + A_BYTES);
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k) {    // 32 bytes of K per MMA: 8 tf32 or 16 fp16 elements
                            if (HALF) tc_mma_f16_e(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
                            else tc_mma_tf32_e(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
                        }
                    }
                    tc_commit_e(&empty[stage]);           // slot reusable once these MMAs have read it
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit_e(&tfull[acc]);                 // accumulator complete
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        const int q = warp & 3;                          // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;                // which half of the tile's column chunks this warp owns
        constexpr int CPW = BN / 64;                     // 32-column chunks per warp
        float* stg = cstage + (warp - 2) * (32 * 32);
        const int ch = lane & 7, rsub = lane >> 3;       // read-back role: 16-byte chunk within the row, row sub-index
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
            const int z = t / tiles_mn, tt = t % tiles_mn;
            const int m0 = (tt / p.tiles_n) * BM, n0 = (tt % p.tiles_n) * BN;
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const int row0 = m0 + q * 32;
            if constexpr (EPI == 1) {
                // softmax over the 64 columns of a row (NetVLAD soft assignment, PointNetVlad.py:48-59): lane = row; this warp holds
                // columns half*32 .. +31 of its 32 rows, the partner warp (same lane quarter) the other 32: row maximum and row sum
                // are exchanged through shared memory behind a 64-thread named barrier.
                if (row0 < p.M) {
                    uint32_t r[32];
                    tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + half * 32, r);
                    float v[32];
                    float mx = -INFINITY;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const int col = half * 32 + j;
                        const float sc = p.scale ? __ldg(p.scale + col) : 1.f, sh = p.shift ? __ldg(p.shift + col) : 0.f;
                        v[j] = fmaf(__uint_as_float(r[j]), sc, sh);
                        mx = fmaxf(mx, v[j]);
                    }
                    float* xmax = xch, *xsum = xch + 256;
                    xmax[(q * 2 + half) * 32 + lane] = mx;
                    asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
                    mx = fmaxf(mx, xmax[(q * 2 + (half ^ 1)) * 32 + lane]);
                    float sum = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) { v[j] = expf(v[j] - mx); sum += v[j]; }
                    xsum[(q * 2 + half) * 32 + lane] = sum;
                    asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");
                    const float tot = xsum[(q * 2) * 32 + lane] + xsum[(q * 2 + 1) * 32 + lane];   // same order in both warps
                    float* dst = stg + lane * 32;
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float4*>(dst + ((j ^ (lane & 7)) << 2)) =
                            make_float4(v[4 * j] / tot, v[4 * j + 1] / tot, v[4 * j + 2] / tot, v[4 * j + 3] / tot);
                    __syncwarp();
                    const int col = half * 32 + ch * 4;
                    const size_t goff = (size_t)row0 * 64 + col;
                    float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int rr = it * 4 + rsub;
                        const float4 o = *reinterpret_cast<const float4*>(stg + rr * 32 + ((ch ^ (rr & 7)) << 2));
                        if (row0 + rr < p.M) {
                            cs.x += o.x; cs.y += o.y; cs.z += o.z; cs.w += o.w;
                            if (p.C) *reinterpret_cast<float4*>(p.C + goff + (size_t)rr * 64) = o;
                            if (p.a_h) {
                                const __half2 h0 = __floats2half2_rn(o.x, o.y), h1 = __floats2half2_rn(o.z, o.w);
                                *reinterpret_cast<uint2*>(p.a_h + goff + (size_t)rr * 64) =
                                    make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
                            }
                        }
                    }
                    // column sums of the 32-row block: rows rsub, rsub + 4, ... were added above; now across the four rsub lanes
                    cs.x += __shfl_down_sync(kFull, cs.x, 16); cs.y += __shfl_down_sync(kFull, cs.y, 16);
                    cs.z += __shfl_down_sync(kFull, cs.z, 16); cs.w += __shfl_down_sync(kFull, cs.w, 16);
                    cs.x += __shfl_down_sync(kFull, cs.x, 8); cs.y += __shfl_down_sync(kFull, cs.y, 8);
                    cs.z += __shfl_down_sync(kFull, cs.z, 8); cs.w += __shfl_down_sync(kFull, cs.w, 8);
                    if (p.apart && lane < 8) *reinterpret_cast<float4*>(p.apart + (size_t)(row0 >> 5) * 64 + col) = cs;
                    __syncwarp();
                }
            } else {
#pragma unroll 1
            for (int i = 0; i < CPW; ++i) {
                const int c = half * CPW + i;
                const int col0 = n0 + c * 32;
                if (col0 >= p.N || row0 >= p.M) break;  // warp-uniform: the rest is out of range
                // accumulate mode: the old C values of this lane's 8 rows are requested before the accumulators are read, so
                // their latency overlaps the TMEM load and the staging pass instead of sitting in the store loop
                const int colp = col0 + ch * 4;
                float4 oldc[8];
                if (!TN && p.accumulate) {
                    const float* gold = p.C + (size_t)z * p.bM * p.ldc + (size_t)row0 * p.ldc + colp;
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int rr = it * 4 + rsub;
                        oldc[it] = (colp < p.N && row0 + rr < p.M) ? __ldg(reinterpret_cast<const float4*>(gold + (size_t)rr * p.ldc))
                                                                    : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                uint32_t r[32];
                tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + c * 32, r);
                float* dst = stg + lane * 32;
#pragma unroll
                for (int j = 0; j < 8; ++j)              // lane = row: raw accumulators, 16B chunk ^= row & 7
                    *reinterpret_cast<uint4*>(dst + ((j ^ (lane & 7)) << 2)) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                __syncwarp();
                const int col = col0 + ch * 4;           // this lane's 4 columns for the whole chunk
                const bool col_ok = col < p.N;           // N % 4 == 0
                float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
                if (col_ok) {
                    if (p.scale) sc = __ldg(reinterpret_cast<const float4*>(p.scale + col));
                    if (p.shift) sh = __ldg(reinterpret_cast<const float4*>(p.shift + col));
                }
                const size_t goff = (TN ? (size_t)z * p.strideC : (size_t)z * p.bM * p.ldc) + (size_t)row0 * p.ldc + col;
                float* gcol = p.C + goff;
                __half* hcol = reinterpret_cast<__half*>(p.C) + goff;          // OUT_HALF: C is an fp16 matrix (ldc in halves)
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    const int rr = it * 4 + rsub;
                    float4 v = *reinterpret_cast<const float4*>(stg + rr * 32 + ((ch ^ (rr & 7)) << 2));
                    v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y); v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
                    v.x = fmaxf(v.x, v.x * p.neg_slope); v.y = fmaxf(v.y, v.y * p.neg_slope);
                    v.z = fmaxf(v.z, v.z * p.neg_slope); v.w = fmaxf(v.w, v.w * p.neg_slope);
                    if (col_ok && row0 + rr < p.M) {
                        if (OUT_HALF) {
                            __half2 h0, h1;                                      // saturating: out-of-range values become +-65504, not inf
                            asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(*reinterpret_cast<uint32_t*>(&h0)) : "f"(v.y), "f"(v.x));
                            asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(*reinterpret_cast<uint32_t*>(&h1)) : "f"(v.w), "f"(v.z));
                            *reinterpret_cast<uint2*>(hcol + (size_t)rr * p.ldc) =
                                make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
                        } else {
                            float4* dstp = reinterpret_cast<float4*>(gcol + (size_t)rr * p.ldc);
                            if (!TN && p.accumulate) { const float4 o = oldc[it]; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
                            *dstp = v;
                        }
                    }
                }
                __syncwarp();                            // staging buffer is rewritten by the next chunk
            }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

template <int BN, int STAGES, bool TN = false, typename TIN = float, bool OUT_HALF = false, int EPI = 0>
static int launch(const CUtensorMap& ta, const CUtensorMap& tb, Params p, cudaStream_t st) {
    constexpr size_t smem = (size_t)STAGES * (BM * BK * 4 + BN * BK * 4) + EPI_WARPS * 32 * 32 * 4 + 256 + (EPI == 1 ? 2048 : 0);
    LPD_CUDA_CHECK(allow_smem(gemm_tf32_kernel<BN, STAGES, TN, TIN, OUT_HALF, EPI>, smem));
    int sms = 0;
    const int rc = sm_count(&sms);
    if (rc != LPD_OK) return rc;
    p.tiles_m = ceil_div(p.M, BM);
    p.tiles_n = ceil_div(p.N, BN);
    const long long tiles = (long long)p.tiles_m * p.tiles_n * p.batch;
    const int grid = (int)(tiles < sms ? tiles : sms);
    gemm_tf32_kernel<BN, STAGES, TN, TIN, OUT_HALF, EPI><<<grid, THREADS, smem, st>>>(ta, tb, p);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// CTA-PAIR form of the fp16 GEMM (cta_group::2) for the wide layers (N % 256 == 0, fp16 output: conv3 512 -> 1024 and the 128 ->
// 512 neighbour / centre projections of the f16 eval path).  In the single-CTA kernel above a 128 x 256 tile needs 4 KB of A and
// 8 KB of B out of shared memory per 128-clk MMA (96 B/clk) while TMA writes the same 96 B/clk and the fp32 staging of the epilogue
// adds 64 B/clk: 256 B/clk against the SM's 128 B/clk, which is exactly the 50 % tensor-pipe activity ncu shows for conv3.  Here the
// two CTAs of a cluster form ONE 256 x 256 tile: each CTA holds 128 rows of A and 128 of the 256 rows of W per stage (TMA ... .cta_group::2
// signalling the leader's mbarrier), the leader's elected lane issues tcgen05.mma.cta_group::2 (M = 256: each SM multiplies its A
// half with BOTH W halves), tcgen05.commit ... .multicast::cluster releases the ring slot / hands over the accumulator in both CTAs,
// and each CTA's epilogue drains its own 128 x 256 accumulator (TMEM -> affine + activation -> fp16 -> 4 KB staging -> full 128-byte
// lines).  Per SM: 64 B/clk operand reads + 64 B/clk TMA + 32 B/clk staging.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int H2_STAGES = 5;
constexpr int H2_MAXN = 2048;                           // columns whose epilogue scale / shift are kept in shared memory
constexpr uint32_t H2_A_BYTES = 128 * 128, H2_B_BYTES = 128 * 128, H2_STAGE_BYTES = H2_A_BYTES + H2_B_BYTES;
constexpr size_t H2_SMEM = (size_t)H2_STAGES * H2_STAGE_BYTES + EPI_WARPS * 32 * 128 + 2 * H2_MAXN * 4 + 256;

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// the address of the same shared-memory object in CTA `rank` of the cluster (shared::cluster window)
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void tma_load_2d_2sm_e(void* smem_dst, const CUtensorMap* tmap, uint32_t leader_bar, int c0, int c1) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc_mma_f16_2sm_e(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit_2sm_e(uint64_t* bar) {      // arrives on `bar` in BOTH CTAs of the pair
    asm volatile(
        "{\n\t.reg .pred q;\n\t.reg .b16 m;\n\t"
        "mov.b16 m, 3;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}"
        ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tc_mma_tf32_2sm_e(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// TIN = __half: fp16 operands (kind::f16, 64 K elements per 128-byte row); TIN = float: fp32 operands consumed as TF32 (32 per row)
// OUT32: fp32 output (the training path's plain conv / dgrad GEMMs); else fp16
template <typename TIN, bool OUT32 = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
gemm_h2_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, Params p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* cstage = smem + H2_STAGES * H2_STAGE_BYTES;                             // [EPI_WARPS][32 rows][128 B]
    float* ssc = reinterpret_cast<float*>(cstage + EPI_WARPS * 32 * 128);            // [H2_MAXN] epilogue scale, then shift
    float* ssh = ssc + H2_MAXN;
    uint64_t* full = reinterpret_cast<uint64_t*>(ssh + H2_MAXN);
    uint64_t* empty = full + H2_STAGES;
    uint64_t* tfull = empty + H2_STAGES;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < p.N; i += THREADS) {     // (made visible by the barriers below)
        ssc[i] = p.scale ? __ldg(p.scale + i) : 1.f;
        ssh[i] = p.shift ? __ldg(p.shift + i) : 0.f;
    }
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    constexpr bool HALF = sizeof(TIN) == 2;
    constexpr int BKE = HALF ? 64 : 32;                                             // K elements per ring slot
    const int num_kb = (p.K + BKE - 1) / BKE;
    const int num_tiles = p.tiles_m * p.tiles_n;                                    // 256 x 256 tiles of the pair
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
        for (int s = 0; s < H2_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 2 * EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {                                       // the same warp of both CTAs
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();                                       // (the CTA-level barrier is what racecheck models; the cluster barrier orders the pair)
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        int stage = 0; uint32_t phase = 0;
        for (int t = pair; t < num_tiles; t += npairs) {
            const int m0 = (t / p.tiles_n) * 256 + (int)rank * 128, n0 = (t % p.tiles_n) * 256 + (int)rank * 128;
            for (int kb = 0; kb < num_kb; ++kb) {
                mbar_wait(&empty[stage], phase ^ 1);
                if (leader) mbar_expect_tx_e(&full[stage], 2 * H2_STAGE_BYTES);      // the bytes of both CTAs land on the leader's barrier
                const uint32_t lbar = mapa_u32(smem_u32(&full[stage]), 0);
                uint8_t* sa = smem + stage * H2_STAGE_BYTES;
                tma_load_2d_2sm_e(sa, &tmap_a, lbar, kb * BKE, m0);
                tma_load_2d_2sm_e(sa + H2_A_BYTES, &tmap_b, lbar, kb * BKE, n0);
                if (++stage == H2_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (leader) {
            constexpr uint32_t idesc = HALF ? make_idesc_h(256, 256) : make_idesc(256, 256);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int t = pair; t < num_tiles; t += npairs) {
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * 256;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * H2_STAGE_BYTES);
                    const uint64_t da = make_smem_desc(sa), db = make_smem_desc(sa + H2_A_BYTES);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {              // 32 bytes of K per MMA: 16 fp16 or 8 tf32 elements
                        if (HALF) tc_mma_f16_2sm_e(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
                        else tc_mma_tf32_2sm_e(tmem_d, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    tc_commit_2sm_e(&empty[stage]);
                    if (++stage == H2_STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit_2sm_e(&tfull[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        const int q = warp & 3, half = (warp - 2) >> 2;
        uint8_t* stg = cstage + (warp - 2) * (32 * 128);
        const int ch = lane & 7, rsub = lane >> 3;
        __half* Cg = reinterpret_cast<__half*>(p.C);
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = pair; t < num_tiles; t += npairs) {
            const int m0 = (t / p.tiles_n) * 256 + (int)rank * 128, n0 = (t % p.tiles_n) * 256;
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const int row0 = m0 + q * 32;
            if constexpr (OUT32) {
                // fp32 output: four chunks of 32 columns (128 bytes per row), raw accumulators staged like the single-CTA kernel
                float* stgf = reinterpret_cast<float*>(stg);
#pragma unroll 1
                for (int i = 0; i < 4; ++i) {
                    const int c32 = half * 4 + i, col0 = n0 + c32 * 32;
                    if (row0 >= p.M) break;                 // warp-uniform
                    uint32_t r[32];
                    tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256 + c32 * 32, r);
                    float* dst = stgf + lane * 32;
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<uint4*>(dst + ((j ^ (lane & 7)) << 2)) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                    __syncwarp();
                    const int col = col0 + ch * 4;
                    const float4 sc = *reinterpret_cast<const float4*>(ssc + col), sh = *reinterpret_cast<const float4*>(ssh + col);
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int rr = it * 4 + rsub;
                        float4 v = *reinterpret_cast<const float4*>(stgf + rr * 32 + ((ch ^ (rr & 7)) << 2));
                        v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y); v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
                        v.x = fmaxf(v.x, v.x * p.neg_slope); v.y = fmaxf(v.y, v.y * p.neg_slope);
                        v.z = fmaxf(v.z, v.z * p.neg_slope); v.w = fmaxf(v.w, v.w * p.neg_slope);
                        if (row0 + rr < p.M) *reinterpret_cast<float4*>(p.C + (size_t)(row0 + rr) * p.ldc + col) = v;
                    }
                    __syncwarp();
                }
            } else
#pragma unroll 1
            for (int i = 0; i < 2; ++i) {
                const int c64 = half * 2 + i, col0 = n0 + c64 * 64;
                if (row0 >= p.M) break;                     // warp-uniform
                uint32_t pk[32];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    uint32_t r[32];
                    tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256 + c64 * 64 + h * 32, r);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int col = col0 + h * 32 + 4 * j;
                        const float4 sc = *reinterpret_cast<const float4*>(ssc + col), sh = *reinterpret_cast<const float4*>(ssh + col);   // warp broadcast
                        float v0 = fmaf(__uint_as_float(r[4 * j]), sc.x, sh.x), v1 = fmaf(__uint_as_float(r[4 * j + 1]), sc.y, sh.y);
                        float v2 = fmaf(__uint_as_float(r[4 * j + 2]), sc.z, sh.z), v3 = fmaf(__uint_as_float(r[4 * j + 3]), sc.w, sh.w);
                        v0 = fmaxf(v0, v0 * p.neg_slope); v1 = fmaxf(v1, v1 * p.neg_slope);
                        v2 = fmaxf(v2, v2 * p.neg_slope); v3 = fmaxf(v3, v3 * p.neg_slope);
                        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(pk[h * 16 + 2 * j]) : "f"(v1), "f"(v0));
                        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(pk[h * 16 + 2 * j + 1]) : "f"(v3), "f"(v2));
                    }
                }
                uint8_t* dst = stg + lane * 128;            // lane = row: 8 chunks of 16 B, chunk ^= row & 7
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<uint4*>(dst + ((j ^ (lane & 7)) << 4)) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                __syncwarp();
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                    const int rr = it * 4 + rsub;
                    const uint4 v = *reinterpret_cast<const uint4*>(stg + rr * 128 + ((ch ^ (rr & 7)) << 4));
                    if (row0 + rr < p.M) *reinterpret_cast<uint4*>(Cg + (size_t)(row0 + rr) * p.ldc + col0 + ch * 8) = v;
                }
                __syncwarp();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {                               // the accumulator stage is free again: tell the leader's MMA warp
                const uint32_t lbar = mapa_u32(smem_u32(&tempty[acc]), 0);
                asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(lbar) : "memory");
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    cluster_sync_all();                                    // nobody leaves while the peer may still read its shared memory / barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
    }
}

template <typename TIN, bool OUT32 = false>
static int launch_h2(const CUtensorMap& ta, const CUtensorMap& tb, Params p, cudaStream_t st) {
    LPD_CUDA_CHECK(allow_smem(gemm_h2_kernel<TIN, OUT32>, H2_SMEM));
    int sms = 0;
    const int rc = sm_count(&sms);
    if (rc != LPD_OK) return rc;
    p.tiles_m = ceil_div(p.M, 256);
    p.tiles_n = p.N / 256;
    const long long tiles = (long long)p.tiles_m * p.tiles_n;
    const long long pairs = sms / 2;
    const int grid = (int)(2 * (tiles < pairs ? tiles : pairs));
    gemm_h2_kernel<TIN, OUT32><<<grid, THREADS, H2_SMEM, st>>>(ta, tb, p);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

// One validated GEMM of the extern "C" entry points.  !tn: A [batch*M][K], B [batch*N][K]; tn: A [batch*K][M], B [batch*K][N].
struct GemmCall {
    const void* A = nullptr; int lda = 0;
    const void* B = nullptr; int ldb = 0;
    bool half = false;       // fp16 operands (kind::f16); else fp32 operands read as TF32
    bool tn = false;
    bool out_half = false;   // C is fp16
    bool softmax = false;    // EPI 1: row softmax over N == 64 columns
    Params p;
};

// the single-CTA kernel at tile width BN, with as many ring stages as its shared memory holds
template <typename TIN, bool TN, bool OUT_HALF>
static int launch_bn(int BN, const CUtensorMap& ta, const CUtensorMap& tb, const Params& p, cudaStream_t st) {
    if (BN == 64) return launch<64, 8, TN, TIN, OUT_HALF>(ta, tb, p, st);
    if (BN == 128) return launch<128, 6, TN, TIN, OUT_HALF>(ta, tb, p, st);
    return launch<256, 4, TN, TIN, OUT_HALF>(ta, tb, p, st);
}

template <typename TIN>
static int launch_form(const GemmCall& g, int BN, const CUtensorMap& ta, const CUtensorMap& tb, cudaStream_t st) {
    if (g.softmax) return launch<64, 8, false, TIN, false, 1>(ta, tb, g.p, st);
    if (g.tn) return launch_bn<TIN, true, false>(BN, ta, tb, g.p, st);
    if (g.out_half) return launch_bn<TIN, false, true>(BN, ta, tb, g.p, st);
    return launch_bn<TIN, false, false>(BN, ta, tb, g.p, st);
}

static int gemm_run(const GemmCall& g, cudaStream_t st) {
    int rc = require_sm100();
    if (rc != LPD_OK) return rc;
    const Params& p = g.p;
    // CTA-pair kernel: wide layers whose epilogue scale / shift fit its shared memory, with fp16 output (16-byte row stores) or
    // as one large fp32 product
    const bool pair = !g.tn && !g.softmax && (p.N % 256) == 0 && p.N <= H2_MAXN &&
                      (g.out_half ? (p.ldc % 8) == 0 : !g.half && p.batch == 1 && !p.accumulate && p.M >= 1024);
    const int BN = p.N <= 64 ? 64 : (p.N <= 128 ? 128 : 256);
    const CUtensorMapDataType type = g.half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    const int row = g.half ? 64 : 32;                       // elements per 128-byte shared-memory row
    CUtensorMap ta, tb;
    if (g.tn) {   // boxes {128 bytes along M / N, as many k-rows}; MN-major tf32 needs the 32-byte swizzle atom
        const long long rows = (long long)p.K * p.batch;
        const CUtensorMapSwizzle swz = g.half ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
        rc = make_tmap(&ta, type, g.A, rows, p.M, g.lda, row, row, swz);
        if (rc == LPD_OK) rc = make_tmap(&tb, type, g.B, rows, p.N, g.ldb, row, row, swz);
    } else {      // a CTA of the pair loads 128 of the 256 rows of B in its tile
        rc = make_tmap(&ta, type, g.A, (long long)p.batch * p.M, p.K, g.lda, BM, row);
        if (rc == LPD_OK) rc = make_tmap(&tb, type, g.B, (long long)p.batch * p.N, p.K, g.ldb, pair ? 128 : BN, row);
    }
    if (rc != LPD_OK) return rc;
    if (pair) {
        if (g.half) return launch_h2<__half>(ta, tb, p, st);
        return g.out_half ? launch_h2<float>(ta, tb, p, st) : launch_h2<float, true>(ta, tb, p, st);
    }
    return g.half ? launch_form<__half>(g, BN, ta, tb, st) : launch_form<float>(g, BN, ta, tb, st);
}

__global__ void __launch_bounds__(256)
f32_to_f16_kernel(const float* __restrict__ x, long long ldx, __half* __restrict__ y, long long ldy, long long rows, int cols) {
    const long long total = rows * cols;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / cols;
        const int c = (int)(e % cols);
        y[r * ldy + c] = __float2half_rn(x[r * ldx + c]);
    }
}

// x = hi + lo with hi = x truncated to TF32 (exactly what kind::tf32 reads of an fp32 operand) and lo = x - hi (exact in fp32).
// out holds three stacked copies: role 0 (A side) [hi; hi; lo], role 1 (B side) [hi; lo; hi], so that ONE TF32 contraction over
// the stacked axis accumulates hi.hi + hi.lo + lo.hi in fp32 ("3xTF32": ~2^-21 relative instead of 2^-10).
__global__ void __launch_bounds__(256)
split3_tf32_kernel(const float* __restrict__ x, long long n, float* __restrict__ out, int role) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const float v = x[e];
        const float hi = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
        const float lo = v - hi;
        out[e] = hi;
        out[n + e] = role ? lo : hi;
        out[2 * n + e] = role ? hi : lo;
    }
}

// the A side of the 3xTF32 hidden projection in one pass: v [B][R] (row-major descriptors) -> out [3][R][Bp] = the TRANSPOSED
// matrix split into [hi; hi; lo], columns B..Bp-1 zero.  32 x 32 shared-memory tiles: coalesced along R on the way in, along B out.
__global__ void __launch_bounds__(256)
transpose_split3_kernel(const float* __restrict__ v, int B, long long R, int Bp, float* __restrict__ out) {
    __shared__ float tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const long long r0 = (long long)blockIdx.x * 32;
    for (int b0 = 0; b0 < Bp; b0 += 32) {
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int b = b0 + ty + 8 * i;
            tile[ty + 8 * i][tx] = (b < B && r0 + tx < R) ? __ldg(v + (size_t)b * R + r0 + tx) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const long long r = r0 + ty + 8 * i;
            const int b = b0 + tx;
            if (r < R && b < Bp) {
                const float x = tile[tx][ty + 8 * i];
                const float hi = __uint_as_float(__float_as_uint(x) & 0xffffe000u);
                const size_t o = (size_t)r * Bp + b;
                out[o] = hi;
                out[(size_t)R * Bp + o] = hi;
                out[2 * (size_t)R * Bp + o] = x - hi;
            }
        }
    }
}

}  // namespace tc
}  // namespace lpd

extern "C" int lpd_transpose_split3(const float* v, int B, long long R, int Bp, float* out, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(v && out && B >= 1 && R >= 1 && Bp >= B && (Bp % 4) == 0);
    const long long blocks = (R + 31) / 32;
    LPD_REQUIRE(blocks <= 0x7fffffffLL);
    tc::transpose_split3_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(v, B, R, Bp, out);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_split3_tf32(const float* x, long long n, float* out, int role, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(x && out && n >= 1 && (role == 0 || role == 1));
    const long long blocks = (n + 255) / 256;
    tc::split3_tf32_kernel<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, as_stream(stream)>>>(x, n, out, role);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_f32_to_f16(const float* x, long long ldx, void* y, long long ldy, long long rows, int cols, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(x && y && rows >= 1 && cols >= 1 && ldx >= cols && ldy >= cols);
    const long long total = rows * cols;
    const long long blocks = (total + 255) / 256;
    tc::f32_to_f16_kernel<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, as_stream(stream)>>>(
        x, ldx, reinterpret_cast<__half*>(y), ldy, rows, cols);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_gemm_f16(const void* A, int lda, const void* W, int ldw, void* C, int ldc, int out_half,
                            int M, int N, int K, const float* scale, const float* shift, int act, float slope, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(A && W && C && M >= 1 && N >= 1 && K >= 1);
    LPD_REQUIRE(lda >= K && ldw >= K && ldc >= N);
    LPD_REQUIRE((lda % 8) == 0 && (ldw % 8) == 0 && (ldc % 4) == 0);          // 16-byte global strides (TMA), vector stores
    LPD_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)W & 15) == 0 && ((uintptr_t)C & 15) == 0);
    LPD_REQUIRE((N % 4) == 0);
    LPD_REQUIRE(act_is_slope(act, slope));
    tc::GemmCall g;
    g.A = A; g.lda = lda; g.B = W; g.ldb = ldw; g.half = true; g.out_half = out_half != 0;
    g.p.C = reinterpret_cast<float*>(C); g.p.ldc = ldc; g.p.M = M; g.p.N = N; g.p.K = K; g.p.scale = scale; g.p.shift = shift;
    g.p.neg_slope = act_neg_slope(act, slope);
    return tc::gemm_run(g, as_stream(stream));
}

extern "C" int lpd_gemm_f16_tn(const void* A, int lda, const void* B, int ldb, float* C, int ldc, long long strideC,
                               int M, int N, int K, int batch, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(A && B && C && M >= 1 && N >= 1 && K >= 1 && batch >= 1);
    LPD_REQUIRE(lda >= M && ldb >= N && ldc >= N);
    LPD_REQUIRE((lda % 8) == 0 && (ldb % 8) == 0 && (ldc % 4) == 0 && (strideC % 4) == 0);
    LPD_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0 && ((uintptr_t)C & 15) == 0);
    LPD_REQUIRE((N % 4) == 0);
    LPD_REQUIRE(batch == 1 || (K % 64) == 0);              // a slice's k-blocks must not run into the next slice
    tc::GemmCall g;
    g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.half = true; g.tn = true;
    g.p.C = C; g.p.ldc = ldc; g.p.M = M; g.p.N = N; g.p.K = K; g.p.batch = batch; g.p.strideC = strideC;
    return tc::gemm_run(g, as_stream(stream));
}

extern "C" int lpd_gemm_tf32_ex(const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                                int M, int N, int K, int batch, int accumulate, const float* scale, const float* shift, int act,
                                float slope, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(A && B && C && M >= 1 && N >= 1 && K >= 1 && batch >= 1);
    LPD_REQUIRE(lda >= K && ldb >= K && ldc >= N);
    LPD_REQUIRE((lda % 4) == 0 && (ldb % 4) == 0 && (ldc % 4) == 0);          // 16-byte global strides (TMA) / float4 stores
    LPD_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0 && ((uintptr_t)C & 15) == 0);
    LPD_REQUIRE((N % 4) == 0);
    LPD_REQUIRE(act_is_slope(act, slope));
    LPD_REQUIRE((long long)batch * M < (1ll << 31) && (long long)batch * N < (1ll << 31));
    tc::GemmCall g;
    g.A = A; g.lda = lda; g.B = B; g.ldb = ldb;
    g.p.C = C; g.p.ldc = ldc; g.p.M = M; g.p.N = N; g.p.K = K; g.p.scale = scale; g.p.shift = shift;
    g.p.neg_slope = act_neg_slope(act, slope);
    g.p.batch = batch; g.p.bM = batch > 1 ? M : 0; g.p.bN = batch > 1 ? N : 0; g.p.accumulate = accumulate ? 1 : 0;
    return tc::gemm_run(g, as_stream(stream));
}

extern "C" int lpd_gemm_tf32_out16(const float* A, int lda, const float* B, int ldb, void* C, int ldc, int M, int N, int K,
                                   const float* scale, const float* shift, int act, float slope, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(A && B && C && M >= 1 && N >= 1 && K >= 1);
    LPD_REQUIRE(lda >= K && ldb >= K && ldc >= N);
    LPD_REQUIRE((lda % 4) == 0 && (ldb % 4) == 0 && (ldc % 4) == 0 && (N % 4) == 0);
    LPD_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0 && ((uintptr_t)C & 7) == 0);
    LPD_REQUIRE(act_is_slope(act, slope));
    tc::GemmCall g;
    g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.out_half = true;
    g.p.C = reinterpret_cast<float*>(C); g.p.ldc = ldc; g.p.M = M; g.p.N = N; g.p.K = K; g.p.scale = scale; g.p.shift = shift;
    g.p.neg_slope = act_neg_slope(act, slope);
    return tc::gemm_run(g, as_stream(stream));
}

extern "C" int lpd_gemm_tf32(const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                             int M, int N, int K, const float* scale, const float* shift, int act, float slope,
                             void* stream) {
    return lpd_gemm_tf32_ex(A, lda, B, ldb, C, ldc, M, N, K, 1, 0, scale, shift, act, slope, stream);
}

extern "C" int lpd_gemm_tf32_tn(const float* A, int lda, const float* B, int ldb, float* C, int ldc, long long strideC,
                                int M, int N, int K, int batch, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(A && B && C && M >= 1 && N >= 1 && K >= 1 && batch >= 1);
    LPD_REQUIRE(lda >= M && ldb >= N && ldc >= N);
    LPD_REQUIRE((lda % 4) == 0 && (ldb % 4) == 0 && (ldc % 4) == 0 && (strideC % 4) == 0);
    LPD_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0 && ((uintptr_t)C & 15) == 0);
    LPD_REQUIRE((N % 4) == 0);
    LPD_REQUIRE(batch == 1 || (K % tc::BK) == 0);          // a slice's k-blocks must not run into the next slice
    tc::GemmCall g;
    g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.tn = true;
    g.p.C = C; g.p.ldc = ldc; g.p.M = M; g.p.N = N; g.p.K = K; g.p.batch = batch; g.p.strideC = strideC;
    return tc::gemm_run(g, as_stream(stream));
}

extern "C" int lpd_gemm_softmax64(const void* A, int a_f16, int lda, const void* W, int ldw, int M, int K, const float* scale,
                                  const float* shift, float* a32, void* a16, float* apart, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(A && W && M >= 1 && K >= 1 && (a32 || a16));
    LPD_REQUIRE(lda >= K && ldw >= K);
    const int al = a_f16 ? 8 : 4;
    LPD_REQUIRE((lda % al) == 0 && (ldw % al) == 0);
    LPD_REQUIRE(((uintptr_t)A & 15) == 0 && ((uintptr_t)W & 15) == 0 && ((uintptr_t)a32 & 15) == 0 && ((uintptr_t)a16 & 7) == 0 &&
                ((uintptr_t)apart & 15) == 0);
    tc::GemmCall g;
    g.A = A; g.lda = lda; g.B = W; g.ldb = ldw; g.half = a_f16 != 0; g.softmax = true;
    g.p.C = a32; g.p.ldc = 64; g.p.M = M; g.p.N = 64; g.p.K = K; g.p.scale = scale; g.p.shift = shift;
    g.p.a_h = reinterpret_cast<__half*>(a16); g.p.apart = apart;
    return tc::gemm_run(g, as_stream(stream));
}
