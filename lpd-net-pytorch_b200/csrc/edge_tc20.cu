// EdgeConv double layer on the tensor cores, specialised for the reference's own shape: k = 20 neighbours, C1 = C2 = 128
// (LPDNet convDG1 + max + convDG2 + max, reference util/lpdnet_model.py:246-252), first layer PRE-SCALED:
//     the folded BatchNorm of the first edge layer is applied by the per-point projection GEMM's epilogue
//     (p' = s1 * Wn f, q' = s1 * Wc f + t1), so an activated edge row is just  y1 = act(p'_j + q'_i).
// Same operand roles as edge_tc.cu (A = W2 resident in shared memory, B = the activated edge rows, one TMEM lane per output
// channel, the k edges of a point in consecutive accumulator columns).  What changes is the producer side, which bounded the
// generic kernel (54 instructions per gathered row, 60 % of all instructions, tensor pipe 19 % active):
//   * every point owns a 24-row slot of the 128-row edge tile (5 points per tile): slot bases are multiples of 8 rows, so the
//     128B-swizzle term of a row's store address depends on the neighbour number only and, with k a compile-time constant,
//     every store offset inside the unrolled loops is an immediate; rows 20-23 of a slot stay zero;
//   * no per-row predicates (k is known), no first-layer multiply-add (pre-scaled);
//   * TWO producer warps per point, each owning one half of the channels (16 lanes x float4 per row, two rows per warp
//     iteration): 20 producer warps in two groups of 10 (one group per shared-memory / TMEM stage) + 4 epilogue warps.
#include "tc_common.cuh"
#include <cuda_fp16.h>

namespace lpd {
namespace tc {

constexpr int D20_K = 20, D20_SLOT = 24, D20_PTS = 5, D20_C = 128;
constexpr int D20_EPI_WARPS = 4, D20_GROUP_WARPS = 2 * D20_PTS, D20_PROD_WARPS = 2 * D20_GROUP_WARPS;
constexpr int D20_THREADS = 32 * (D20_EPI_WARPS + D20_PROD_WARPS);
constexpr int D20_ALLOC_WARP = D20_EPI_WARPS;
constexpr int D20_ACC_STRIDE = 256;
constexpr uint32_t D20_KB_BYTES = 128 * 128;           // one 32-channel k-block of a 128-row operand tile
constexpr uint32_t D20_OP_BYTES = 4 * D20_KB_BYTES;    // a whole operand tile: 64 KB

struct Dg20Params {
    const float* p; const float* q; const int* idx;
    const float* s2; const float* t2;
    float* x1; float* x2;
    int ldp, ldq, ld1, ld2;
    long long total_pts; int N;
    float neg_slope;                  // act(v) = max(v, v * neg_slope)
    long long num_tiles;
};

__global__ void __launch_bounds__(D20_THREADS, 1)
edgeconv_dg20_tc_kernel(const __grid_constant__ CUtensorMap tmap_w2, Dg20Params P) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* w_s = smem;
    uint8_t* y_s = smem + D20_OP_BYTES;               // [2][OP_BYTES]
    uint64_t* wfull = reinterpret_cast<uint64_t*>(smem + 3 * D20_OP_BYTES);
    uint64_t* yfull = wfull + 1;
    uint64_t* yempty = yfull + 2;
    uint64_t* tfull = yempty + 2;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // zero both edge stages once: rows 20-23 of every slot and rows 120-127 are never written again
    for (uint32_t i = threadIdx.x; i < 2 * D20_OP_BYTES / 16; i += D20_THREADS)
        reinterpret_cast<uint4*>(y_s)[i] = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");

    if (warp == D20_ALLOC_WARP) {
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_w2)) : "memory");
            mbar_init(wfull, 1);
            for (int s = 0; s < 2; ++s) {
                mbar_init(&yfull[s], D20_GROUP_WARPS);
                mbar_init(&yempty[s], 1);
                mbar_init(&tfull[s], 1);
                mbar_init(&tempty[s], D20_EPI_WARPS);
            }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp >= D20_EPI_WARPS) {
        // ------------------------------ producers ------------------------------
        const int pwarp = warp - D20_EPI_WARPS;
        const int grp = pwarp / D20_GROUP_WARPS;                   // = the shared-memory / TMEM stage this warp fills
        const int gw = pwarp % D20_GROUP_WARPS;
        const int pl = gw >> 1, chalf = gw & 1;                    // point slot inside the tile, channel half
        const bool issuer = gw == 0;
        if (warp == D20_ALLOC_WARP && lane == 0) {
            mbar_expect_tx(wfull, D20_OP_BYTES);
            for (int kb2 = 0; kb2 < 4; ++kb2) tma_load_2d(w_s + kb2 * D20_KB_BYTES, &tmap_w2, wfull, kb2 * 32, 0);
        }
        constexpr uint32_t idesc = make_idesc(128, 128);
        const uint32_t w_addr = smem_u32(w_s);
        bool w_ready = false;
        const int sr = lane >> 4, lc = lane & 15;                  // row of the pair this lane works on, float4 index inside the half row
        const int ch = chalf * 64 + lc * 4;                        // first of this lane's 4 channels
        const int kb = ch >> 5, chunk = (ch >> 2) & 7;             // k-block and 16-byte chunk of those channels
        // store address of edge row m of this point:  slot base + m * 128 + ((chunk ^ (m & 7)) << 4), m = 2 i + sr:
        // (m & 7) = ((2 i) & 7) | sr, so chunk ^ (m & 7) = (chunk ^ sr) ^ ((2 i) & 7): four per-lane offsets, the rest immediates
        uint32_t xo[4];
#pragma unroll
        for (int b2 = 0; b2 < 4; ++b2) xo[b2] = (uint32_t)(((chunk ^ sr) ^ (2 * b2)) << 4);
        uint8_t* ybase = y_s + grp * D20_OP_BYTES + kb * D20_KB_BYTES + (pl * D20_SLOT + sr) * 128;
        const long long tstep = 2LL * gridDim.x;
        long long t = blockIdx.x + (long long)grp * gridDim.x;
        // software pipeline: the neighbour list and centre row of the NEXT tile's point are requested before waiting for the stage
        int nj = 0;
        float4 nq = make_float4(0.f, 0.f, 0.f, 0.f);
        auto prefetch = [&](long long tile) {
            const long long pt = tile * D20_PTS + pl;
            if (tile < P.num_tiles && pt < P.total_pts) {
                nj = (lane < D20_K) ? __ldg(P.idx + pt * D20_K + lane) : 0;
                nq = __ldg(reinterpret_cast<const float4*>(P.q + pt * P.ldq + ch));
            }
        };
        prefetch(t);
        const float slope = P.neg_slope;
        for (uint32_t it = 0; t < P.num_tiles; t += tstep, ++it) {
            const uint32_t ph = it & 1;
            const int myj = nj;
            const float4 qv = nq;
            const long long pt = t * D20_PTS + pl;
            prefetch(t + tstep);
            mbar_wait(&yempty[grp], ph ^ 1);
            if (pt < P.total_pts) {
                const float* pbase = P.p + (pt / P.N) * P.N * P.ldp + ch;      // row address = one 32-bit multiply-add on this base
                float4 best = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
#pragma unroll
                for (int h = 0; h < 2; ++h) {                                  // 2 x 5 row pairs: 5 gathers in flight per lane
                    float4 pv[5];
#pragma unroll
                    for (int u = 0; u < 5; ++u) {
                        const int j = __shfl_sync(kFull, myj, 2 * (5 * h + u) + sr);
                        pv[u] = __ldg(reinterpret_cast<const float4*>(pbase + (unsigned)(j * P.ldp)));
                    }
#pragma unroll
                    for (int u = 0; u < 5; ++u) {
                        const int i2 = 5 * h + u;                               // row pair: rows 2 i2 and 2 i2 + 1
                        best.x = fmaxf(best.x, pv[u].x); best.y = fmaxf(best.y, pv[u].y);
                        best.z = fmaxf(best.z, pv[u].z); best.w = fmaxf(best.w, pv[u].w);
                        float4 y;
                        y.x = pv[u].x + qv.x; y.y = pv[u].y + qv.y; y.z = pv[u].z + qv.z; y.w = pv[u].w + qv.w;
                        y.x = fmaxf(y.x, y.x * slope); y.y = fmaxf(y.y, y.y * slope);
                        y.z = fmaxf(y.z, y.z * slope); y.w = fmaxf(y.w, y.w * slope);
                        *reinterpret_cast<float4*>(ybase + i2 * 256 + xo[i2 & 3]) = y;
                    }
                }
                if (P.x1) {
                    // max_m act(p'_m + q') = act(max_m p'_m + q'): the activation is monotone
                    best.x = fmaxf(best.x, __shfl_xor_sync(kFull, best.x, 16)); best.y = fmaxf(best.y, __shfl_xor_sync(kFull, best.y, 16));
                    best.z = fmaxf(best.z, __shfl_xor_sync(kFull, best.z, 16)); best.w = fmaxf(best.w, __shfl_xor_sync(kFull, best.w, 16));
                    if (sr == 0) {
                        float4 o;
                        o.x = best.x + qv.x; o.y = best.y + qv.y; o.z = best.z + qv.z; o.w = best.w + qv.w;
                        o.x = fmaxf(o.x, o.x * slope); o.y = fmaxf(o.y, o.y * slope); o.z = fmaxf(o.z, o.z * slope); o.w = fmaxf(o.w, o.w * slope);
                        *reinterpret_cast<float4*>(P.x1 + pt * P.ld1 + ch) = o;
                    }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&yfull[grp]);
            if (issuer) {   // warp-uniform: the whole warp runs the issue sequence, elect.sync picks the lane (see tc_common.cuh)
                if (!w_ready) { mbar_wait(wfull, 0); w_ready = true; }
                mbar_wait(&tempty[grp], ph ^ 1);
                mbar_wait(&yfull[grp], ph);
                tc_fence_after();
                const uint32_t y_addr = smem_u32(y_s + grp * D20_OP_BYTES);
#pragma unroll
                for (int kb2 = 0; kb2 < 4; ++kb2) {
                    const uint64_t da = make_smem_desc(w_addr + kb2 * D20_KB_BYTES), db = make_smem_desc(y_addr + kb2 * D20_KB_BYTES);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        tc_mma_tf32_e(tmem_base + grp * D20_ACC_STRIDE, da + (uint64_t)(ks * 2), db + (uint64_t)(ks * 2), idesc,
                                      (kb2 | ks) != 0 ? 1u : 0u);
                }
                tc_commit_e(&yempty[grp]);
                tc_commit_e(&tfull[grp]);
            }
            __syncwarp();
        }
    } else {
        // ------------------------------ epilogue ------------------------------
        // BN (scale s2, shift t2) and the activation are monotone per channel, and a lane owns ONE channel, so
        //     max_m act(s2 * d_m + t2) = act(s2 * ext_m d_m + t2),  ext = max if s2 >= 0 else min            (exact in fp32)
        const int ch = warp * 32 + lane;               // output channel = TMEM lane
        const float s2 = __ldg(P.s2 + ch), t2 = __ldg(P.t2 + ch);
        long long t = blockIdx.x;
        for (uint32_t it = 0; t < P.num_tiles; t += gridDim.x, ++it) {
            const uint32_t s = it & 1, ph = (it >> 1) & 1;
            mbar_wait(&tfull[s], ph);
            tc_fence_after();
#pragma unroll 1
            for (int pl = 0; pl < D20_PTS; ++pl) {
                const long long pt = t * D20_PTS + pl;
                if (pt >= P.total_pts) break;
                const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + s * D20_ACC_STRIDE + pl * D20_SLOT;
                uint32_t r[20];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                    : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                      "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                    : "r"(taddr));
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]) : "r"(taddr + 16));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                float a4[4], b4[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { a4[u] = __uint_as_float(r[u]); b4[u] = a4[u]; }
#pragma unroll
                for (int j = 4; j < 20; j += 2) {
                    const float v0 = __uint_as_float(r[j]), v1 = __uint_as_float(r[j + 1]);
                    a4[(j >> 1) & 3] = fmaxf(fmaxf(a4[(j >> 1) & 3], v0), v1);
                    b4[(j >> 1) & 3] = fminf(fminf(b4[(j >> 1) & 3], v0), v1);
                }
                const float mx = fmaxf(fmaxf(a4[0], a4[1]), fmaxf(a4[2], a4[3]));
                const float mn = fminf(fminf(b4[0], b4[1]), fminf(b4[2], b4[3]));
                float v = fmaf(s2, s2 >= 0.f ? mx : mn, t2);
                v = fmaxf(v, v * P.neg_slope);
                P.x2[pt * P.ld2 + ch] = v;
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[s]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == D20_ALLOC_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// FP16 form ("f16" precision mode): p' / q' rows, W2, the activated edge rows and both outputs are fp16; the second edge layer
// runs on tcgen05 kind::f16 (fp32 accumulation).  A gathered row is 256 bytes instead of 512, an operand tile 32 KB instead of
// 64, and the first layer is three half2 instructions per two values (add, multiply by the slope, max).  Same roles: 4 epilogue
// warps + 2 groups of 10 producer warps (two per point, one 64-channel k-block each, FOUR rows per warp iteration).
// C = 64 (LPDNetOrign convDG2, reference util/lpdnet_model.py:98-107): one k-block, so ONE producer warp per point, and W2 is
// padded with zero rows to the M = 128 accumulator layout of the 128-channel form (TMEM lane = output channel): only epilogue
// warps 0 and 1 own output channels.  The padded half of each MMA is wasted, but the tensor pipe is not what bounds the kernel.
// ---------------------------------------------------------------------------------------------------------------------
constexpr uint32_t D20H_KB_BYTES = 128 * 128;          // one 64-channel k-block of a 128-row fp16 operand tile

struct Dg20hParams {
    const __half* p; const __half* q; const int* idx;
    const float* s2; const float* t2;
    __half* x1; __half* x2;
    int ldp, ldq, ld1, ld2;
    long long total_pts; int N;
    float neg_slope;
    long long num_tiles;
};

// KK = 20: 5 points x 24-row slots per 128-edge tile (the reference's k); KK = 32: 4 points x 32-row slots (the C5 stress shape).
// C = 128 or 64 channels in and out.
template <int KK, int C>
struct DgH {
    static constexpr int KBS = C / 64;                 // 64-channel k-blocks = producer warps per point
    static constexpr int SLOT = (KK + 7) / 8 * 8, PTS = 128 / SLOT, GROUP_WARPS = KBS * PTS, PROD_WARPS = 2 * GROUP_WARPS;
    static constexpr int THREADS = 32 * (D20_EPI_WARPS + PROD_WARPS), ROWQ = KK / 4;
    static constexpr int EPI_LIVE = C / 32;            // epilogue warps that own output channels
    static constexpr uint32_t OP_BYTES = KBS * D20H_KB_BYTES;
    static_assert(KK % 4 == 0 && KK <= 32 && PTS * SLOT <= 128, "edge tile geometry");
    static_assert(C == 64 || C == 128, "channel count");
};

template <int KK, int C>
__global__ void __launch_bounds__(DgH<KK, C>::THREADS, 1)
edgeconv_dg20_h_kernel(const __grid_constant__ CUtensorMap tmap_w2, Dg20hParams P) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    constexpr uint32_t D20H_OP_BYTES = DgH<KK, C>::OP_BYTES;
    constexpr int KBS = DgH<KK, C>::KBS, EPI_LIVE = DgH<KK, C>::EPI_LIVE;
    uint8_t* w_s = smem;
    uint8_t* y_s = smem + D20H_OP_BYTES;              // [2][OP_BYTES]
    uint64_t* wfull = reinterpret_cast<uint64_t*>(smem + 3 * D20H_OP_BYTES);
    uint64_t* yfull = wfull + 1;
    uint64_t* yempty = yfull + 2;
    uint64_t* tfull = yempty + 2;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    constexpr int D20_K = KK, D20_SLOT = DgH<KK, C>::SLOT, D20_PTS = DgH<KK, C>::PTS, D20_GROUP_WARPS = DgH<KK, C>::GROUP_WARPS, D20_THREADS = DgH<KK, C>::THREADS, ROWQ = DgH<KK, C>::ROWQ;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    for (uint32_t i = threadIdx.x; i < 2 * D20H_OP_BYTES / 16; i += D20_THREADS)
        reinterpret_cast<uint4*>(y_s)[i] = make_uint4(0, 0, 0, 0);
    if constexpr (C < 128) {                           // rows C..127 of the A tile (W2 padded to M = 128) are never loaded
        for (uint32_t i = threadIdx.x; i < (128 - C) * 128 / 16; i += D20_THREADS)
            reinterpret_cast<uint4*>(w_s + C * 128)[i] = make_uint4(0, 0, 0, 0);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == D20_ALLOC_WARP) {
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_w2)) : "memory");
            mbar_init(wfull, 1);
            for (int s = 0; s < 2; ++s) {
                mbar_init(&yfull[s], D20_GROUP_WARPS);
                mbar_init(&yempty[s], 1);
                mbar_init(&tfull[s], 1);
                mbar_init(&tempty[s], EPI_LIVE);
            }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp >= D20_EPI_WARPS) {
        const int pwarp = warp - D20_EPI_WARPS;
        const int grp = pwarp / D20_GROUP_WARPS, gw = pwarp % D20_GROUP_WARPS;
        const int pl = gw >> (KBS - 1), chalf = gw & (KBS - 1);    // point slot, 64-channel k-block
        const bool issuer = gw == 0;
        if (warp == D20_ALLOC_WARP && lane == 0) {
            mbar_expect_tx(wfull, C * C * 2);
            for (int kb2 = 0; kb2 < KBS; ++kb2) tma_load_2d(w_s + kb2 * D20H_KB_BYTES, &tmap_w2, wfull, kb2 * 64, 0);
        }
        // kind::f16, fp16 operands, fp32 accumulate, M = N = 128
        constexpr uint32_t idesc = (1u << 4) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        const uint32_t w_addr = smem_u32(w_s);
        bool w_ready = false;
        const int sr = lane >> 3, l8 = lane & 7;                   // row of the quadruple, 16-byte chunk (8 channels) inside the k-block
        const int ch = chalf * 64 + l8 * 8;
        // store address of edge row m = 4 i + sr:  slot base + m * 128 + ((l8 ^ (m & 7)) << 4),  (m & 7) = 4 (i & 1) + sr
        const uint32_t xo0 = (uint32_t)((l8 ^ sr) << 4), xo1 = (uint32_t)((l8 ^ sr ^ 4) << 4);
        uint8_t* ybase = y_s + grp * D20H_OP_BYTES + chalf * D20H_KB_BYTES + (pl * D20_SLOT + sr) * 128;
        const long long tstep = 2LL * gridDim.x;
        long long t = blockIdx.x + (long long)grp * gridDim.x;
        int nj = 0;
        uint4 nq = make_uint4(0u, 0u, 0u, 0u);
        auto prefetch = [&](long long tile) {
            const long long pt = tile * D20_PTS + pl;
            if (tile < P.num_tiles && pt < P.total_pts) {
                nj = (lane < D20_K) ? __ldg(P.idx + pt * D20_K + lane) : 0;
                nq = __ldg(reinterpret_cast<const uint4*>(P.q + pt * P.ldq + ch));
            }
        };
        prefetch(t);
        const __half2 slope2 = __float2half2_rn(P.neg_slope);
        const __half2 ninf = __float2half2_rn(-INFINITY);
        for (uint32_t it = 0; t < P.num_tiles; t += tstep, ++it) {
            const uint32_t ph = it & 1;
            const int myj = nj;
            const uint4 qraw = nq;
            const long long pt = t * D20_PTS + pl;
            // the neighbour rows of this tile are requested BEFORE the wait for the operand stage (the MMA of the group's previous
            // tile is still reading it): the gather latency runs under that MMA instead of after it
            uint4 pv[ROWQ];
            if (pt < P.total_pts) {
                const __half* pbase = P.p + (pt / P.N) * P.N * P.ldp + ch;
#pragma unroll
                for (int i = 0; i < ROWQ; ++i) {                                // all rows of the point in flight: KK / 4 per lane
                    const int j = __shfl_sync(kFull, myj, 4 * i + sr);
                    pv[i] = __ldg(reinterpret_cast<const uint4*>(pbase + (unsigned)(j * P.ldp)));
                }
            }
            prefetch(t + tstep);
            mbar_wait(&yempty[grp], ph ^ 1);
            uint4 x1v = make_uint4(0u, 0u, 0u, 0u);
            bool x1ok = false;
            if (pt < P.total_pts) {
                const __half2* qh = reinterpret_cast<const __half2*>(&qraw);
                __half2 best[4] = {ninf, ninf, ninf, ninf};
#pragma unroll
                for (int i = 0; i < ROWQ; ++i) {
                    const __half2* ph2 = reinterpret_cast<const __half2*>(&pv[i]);
                    uint4 y;
                    __half2* yh = reinterpret_cast<__half2*>(&y);
#pragma unroll
                    for (int v = 0; v < 4; ++v) {
                        best[v] = __hmax2(best[v], ph2[v]);
                        const __half2 z = __hadd2(ph2[v], qh[v]);
                        yh[v] = __hmax2(z, __hmul2(z, slope2));
                    }
                    *reinterpret_cast<uint4*>(ybase + i * 512 + ((i & 1) ? xo1 : xo0)) = y;
                }
                if (P.x1) {
                    uint4 o;
                    __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
                    for (int v = 0; v < 4; ++v) {
                        uint32_t b = *reinterpret_cast<uint32_t*>(&best[v]);
                        uint32_t o8 = __shfl_xor_sync(kFull, b, 8);
                        __half2 m2 = __hmax2(best[v], *reinterpret_cast<__half2*>(&o8));
                        b = *reinterpret_cast<uint32_t*>(&m2);
                        uint32_t o16 = __shfl_xor_sync(kFull, b, 16);
                        m2 = __hmax2(m2, *reinterpret_cast<__half2*>(&o16));
                        const __half2 z = __hadd2(m2, qh[v]);                   // max_m act(p'_m + q') = act(max_m p'_m + q')
                        oh[v] = __hmax2(z, __hmul2(z, slope2));
                    }
                    x1v = o; x1ok = sr == 0;
                }
            }
            // (the proxy fence compiles to MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC: it waits for every memory operation of the thread that
            // is still in flight, so the x1 store goes AFTER it instead of sitting in front of the operand hand-over)
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&yfull[grp]);
            if (x1ok) *reinterpret_cast<uint4*>(P.x1 + pt * P.ld1 + ch) = x1v;
            if (issuer) {
                if (!w_ready) { mbar_wait(wfull, 0); w_ready = true; }
                mbar_wait(&tempty[grp], ph ^ 1);
                mbar_wait(&yfull[grp], ph);
                tc_fence_after();
                const uint32_t y_addr = smem_u32(y_s + grp * D20H_OP_BYTES);
#pragma unroll
                for (int kb2 = 0; kb2 < KBS; ++kb2) {
                    const uint64_t da = make_smem_desc(w_addr + kb2 * D20H_KB_BYTES), db = make_smem_desc(y_addr + kb2 * D20H_KB_BYTES);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {             // 16 channels = 32 bytes per MMA
                        const uint32_t acc = (kb2 | ks) != 0 ? 1u : 0u;
                        asm volatile(
                            "{\n\t.reg .pred p, q;\n\t"
                            "setp.ne.b32 p, %4, 0;\n\t"
                            "elect.sync _|q, 0xffffffff;\n\t"
                            "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                            ::"r"(tmem_base + grp * D20_ACC_STRIDE), "l"(da + (uint64_t)(ks * 2)), "l"(db + (uint64_t)(ks * 2)), "r"(idesc), "r"(acc)
                            : "memory");
                    }
                }
                tc_commit_e(&yempty[grp]);
                tc_commit_e(&tfull[grp]);
            }
            __syncwarp();
        }
    } else if (warp < EPI_LIVE) {
        const int ch = warp * 32 + lane;
        const float s2 = __ldg(P.s2 + ch), t2 = __ldg(P.t2 + ch);
        long long t = blockIdx.x;
        for (uint32_t it = 0; t < P.num_tiles; t += gridDim.x, ++it) {
            const uint32_t s = it & 1, ph = (it >> 1) & 1;
            mbar_wait(&tfull[s], ph);
            tc_fence_after();
            // The accumulator columns of point pl + 1 are requested before point pl is reduced (a tcgen05.ld + wait per point left
            // the four epilogue warps ~1900 clk per tile, more than the producers need: ncu showed the producers spinning on the
            // operand stage for 18 % of their samples), and the accumulator stage is handed back as soon as the last point's
            // columns are in registers.
            const uint32_t tbase = tmem_base + ((uint32_t)(warp * 32) << 16) + s * D20_ACC_STRIDE;
            auto request = [&](int pl, uint32_t (&r)[KK]) {
                const uint32_t taddr = tbase + pl * D20_SLOT;
                if constexpr (KK == 20) {
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                        : "r"(taddr));
                    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]) : "r"(taddr + 16));
                } else {
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                        : "r"(taddr));
                }
            };
            auto reduce_store = [&](int pl, const uint32_t (&r)[KK]) {
                const long long pt = t * D20_PTS + pl;
                if (pt >= P.total_pts) return;
                float a4[4], b4[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { a4[u] = __uint_as_float(r[u]); b4[u] = a4[u]; }
#pragma unroll
                for (int j = 4; j < KK; j += 2) {
                    const float v0 = __uint_as_float(r[j]), v1 = __uint_as_float(r[j + 1]);
                    a4[(j >> 1) & 3] = fmaxf(fmaxf(a4[(j >> 1) & 3], v0), v1);
                    b4[(j >> 1) & 3] = fminf(fminf(b4[(j >> 1) & 3], v0), v1);
                }
                const float mx = fmaxf(fmaxf(a4[0], a4[1]), fmaxf(a4[2], a4[3]));
                const float mn = fminf(fminf(b4[0], b4[1]), fminf(b4[2], b4[3]));
                float v = fmaf(s2, s2 >= 0.f ? mx : mn, t2);
                v = fmaxf(v, v * P.neg_slope);
                // two channels per store: even lanes write their own and their right neighbour's value as one half2
                const float vn = __shfl_down_sync(kFull, v, 1);
                if ((lane & 1) == 0) {
                    __half2 h;
                    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(*reinterpret_cast<uint32_t*>(&h)) : "f"(vn), "f"(v));
                    *reinterpret_cast<__half2*>(P.x2 + pt * P.ld2 + ch) = h;
                }
            };
            uint32_t ra[KK], rb[KK];
            request(0, ra);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int pl = 0; pl < D20_PTS; ++pl) {
                const bool more = pl + 1 < D20_PTS;
                if (more) { if (pl & 1) request(pl + 1, ra); else request(pl + 1, rb); }
                else {                                         // every column of the stage is in registers: hand it back
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tempty[s]);
                }
                if (pl & 1) reduce_store(pl, rb); else reduce_store(pl, ra);
                if (more) asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == D20_ALLOC_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// called by lpd_edgeconv_dg_tf32 (edge_tc.cu) for k == 20, C1 == C2 == 128, s1 == t1 == NULL
int dg20_tc_run(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, const float* w2,
                const float* s2, const float* t2, float neg_slope, float* x1, int ld1, float* x2, int ld2, cudaStream_t st) {
    Dg20Params P;
    P.p = p; P.q = q; P.idx = idx; P.s2 = s2; P.t2 = t2; P.x1 = x1; P.x2 = x2;
    P.ldp = ldp; P.ldq = ldq; P.ld1 = ld1; P.ld2 = ld2; P.total_pts = (long long)B * N; P.N = N;
    P.neg_slope = neg_slope;
    P.num_tiles = (P.total_pts + D20_PTS - 1) / D20_PTS;
    CUtensorMap tw;
    int rc = make_tmap(&tw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w2, D20_C, D20_C, D20_C, 128, 32);
    if (rc != LPD_OK) return rc;
    constexpr size_t smem = 3 * (size_t)D20_OP_BYTES + 256;
    LPD_CUDA_CHECK(allow_smem(edgeconv_dg20_tc_kernel, smem));
    int sms = 0;
    rc = sm_count(&sms);
    if (rc != LPD_OK) return rc;
    const int grid = (int)(P.num_tiles < sms ? P.num_tiles : sms);
    edgeconv_dg20_tc_kernel<<<grid, D20_THREADS, smem, st>>>(tw, P);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

template <int KK, int C>
static int dgh_launch(const Dg20hParams& P, const CUtensorMap& tw, int grid, cudaStream_t st) {
    constexpr size_t smem = 3 * (size_t)DgH<KK, C>::OP_BYTES + 256;
    LPD_CUDA_CHECK(allow_smem(edgeconv_dg20_h_kernel<KK, C>, smem));
    edgeconv_dg20_h_kernel<KK, C><<<grid, DgH<KK, C>::THREADS, smem, st>>>(tw, P);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

}  // namespace tc
}  // namespace lpd

// C = 128 or 64 channels (p, q, W2 [C][C], x1, x2)
static int edgeconv_dgk_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N, int K, int C,
                            const void* w2, const float* s2, const float* t2, int act, float slope,
                            void* x1, int ld1, void* x2, int ld2, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(p && q && idx && w2 && s2 && t2 && x2 && B >= 1 && (K == 20 || K == 32) && N >= K);
    LPD_REQUIRE(ldp % 8 == 0 && ldq % 8 == 0 && ld2 % 2 == 0 && (!x1 || ld1 % 8 == 0));
    LPD_REQUIRE(ldp >= C && ldq >= C && ld2 >= C && (!x1 || ld1 >= C));
    LPD_REQUIRE((long long)N * ldp < (1ll << 31));
    LPD_REQUIRE(((uintptr_t)p & 15) == 0 && ((uintptr_t)q & 15) == 0 && ((uintptr_t)x1 & 15) == 0 && ((uintptr_t)x2 & 3) == 0 && ((uintptr_t)w2 & 15) == 0);
    LPD_REQUIRE(act_is_slope(act, slope));
    int rc = require_sm100();
    if (rc != LPD_OK) return rc;
    int sms = 0;
    rc = sm_count(&sms);
    if (rc != LPD_OK) return rc;
    tc::Dg20hParams P;
    P.p = reinterpret_cast<const __half*>(p); P.q = reinterpret_cast<const __half*>(q); P.idx = idx; P.s2 = s2; P.t2 = t2;
    P.x1 = reinterpret_cast<__half*>(x1); P.x2 = reinterpret_cast<__half*>(x2);
    P.ldp = ldp; P.ldq = ldq; P.ld1 = ld1; P.ld2 = ld2; P.total_pts = (long long)B * N; P.N = N;
    P.neg_slope = act_neg_slope(act, slope);
    const int pts = K == 32 ? tc::DgH<32, 128>::PTS : tc::DgH<20, 128>::PTS;
    P.num_tiles = (P.total_pts + pts - 1) / pts;
    CUtensorMap tw;   // W2 fp16 [C][C]: boxes of C rows x 64 halves
    rc = tc::make_tmap(&tw, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, w2, C, C, C, C, 64);
    if (rc != LPD_OK) return rc;
    const int grid = (int)(P.num_tiles < sms ? P.num_tiles : sms);
    cudaStream_t st = as_stream(stream);
    if (C == 128) return K == 32 ? tc::dgh_launch<32, 128>(P, tw, grid, st) : tc::dgh_launch<20, 128>(P, tw, grid, st);
    return K == 32 ? tc::dgh_launch<32, 64>(P, tw, grid, st) : tc::dgh_launch<20, 64>(P, tw, grid, st);
}

extern "C" int lpd_edgeconv_dg20_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N,
                                     const void* w2, const float* s2, const float* t2, int act, float slope,
                                     void* x1, int ld1, void* x2, int ld2, void* stream) {
    return edgeconv_dgk_f16(p, ldp, q, ldq, idx, B, N, 20, 128, w2, s2, t2, act, slope, x1, ld1, x2, ld2, stream);
}

extern "C" int lpd_edgeconv_dg32_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N,
                                     const void* w2, const float* s2, const float* t2, int act, float slope,
                                     void* x1, int ld1, void* x2, int ld2, void* stream) {
    return edgeconv_dgk_f16(p, ldp, q, ldq, idx, B, N, 32, 128, w2, s2, t2, act, slope, x1, ld1, x2, ld2, stream);
}

extern "C" int lpd_edgeconv_dg64_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N, int k,
                                     const void* w2, const float* s2, const float* t2, int act, float slope,
                                     void* x2, int ld2, void* stream) {
    return edgeconv_dgk_f16(p, ldp, q, ldq, idx, B, N, k, 64, w2, s2, t2, act, slope, nullptr, 0, x2, ld2, stream);
}
