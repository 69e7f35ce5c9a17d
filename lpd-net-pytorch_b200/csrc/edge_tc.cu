// EdgeConv double layer on the tensor cores (sm_100a): same contract as lpd_edgeconv_dg, "fast" (TF32) arithmetic
// for the second edge layer.  Replaces get_graph_feature + convDG1 + max + convDG2 + max, reference
// util/lpdnet_model.py:246-252 (and :98-101 for LPDNetOrign), without ever writing an edge tensor to HBM.
//
// Operand roles are chosen so that the max over the k neighbours is thread-local in the epilogue:
//     D[c2][e] = sum_c1 W2[c2][c1] * Y1[e][c1]          A = W2 (M = 128 output channels = TMEM lanes, resident in smem)
//                                                        B = Y1 (N = up to 128 edge rows = TMEM columns), K = C1
// so one TMEM lane holds one output channel and the k edges of a point are k consecutive accumulator columns.
//
// Persistent CTA, 16 warps (512 threads -> 128 registers per thread):
//   warps 0-3   epilogue: tcgen05.ld 32 columns at a point's first edge, folded BN + activation, max over its k
//               columns in registers, 128-byte coalesced store of x2 (lane = channel)
//   warps 4-15  producers, two groups of 6; the first warp of a group also loads W2 by TMA (group 0), owns the TMEM
//               allocation (group 0) and is the single-thread tcgen05.mma issuer of its group's stage;
//               two groups of 6 (group g fills shared-memory stage g, i.e. the CTA's even / odd tiles, so both
//               stages are gathered concurrently): per point gather the k neighbour rows of P (L2-resident, 10 rows in
//               flight per lane), y1 = act(s1 * (p_j + q_i) + t1) in fp32, running max -> x1, and st.shared of y1 rows
//               straight into the 128B-swizzled UMMA layout (generic-proxy writes are fenced to the async proxy before the
//               mbarrier arrive).  The gather is L2-latency bound: what matters is the number of rows in flight per SM.
#include "tc_common.cuh"

namespace lpd {
namespace tc {

constexpr int DG_EPI_WARPS = 4, DG_PROD_WARPS = 12, DG_GROUP_WARPS = DG_PROD_WARPS / 2;
constexpr int DG_ALLOC_WARP = DG_EPI_WARPS;      // first producer warp of group 0
constexpr int DG_THREADS = 32 * (DG_EPI_WARPS + DG_PROD_WARPS);
constexpr int DG_ROWS = 128;          // operand tile rows (both W2 and the edge tile)
constexpr int DG_ACC_STRIDE = 256;    // TMEM columns between the two accumulator stages

struct DgTcParams {
    const float* p; const float* q; const int* idx;
    const float* s1; const float* t1; const float* s2; const float* t2;
    float* x1; float* x2;
    int ldp, ldq, ld1, ld2;
    long long total_pts; int N, k, C2;
    float neg_slope;                  // act(v) = max(v, v * neg_slope)
    int pts_per_tile, n_mma;
    long long num_tiles;
};

template <int C1>
__global__ void __launch_bounds__(DG_THREADS, 1)
edgeconv_dg_tc_kernel(const __grid_constant__ CUtensorMap tmap_w2, DgTcParams P) {
    constexpr int KB = C1 / 32;                       // 128-byte k-blocks per operand row
    constexpr uint32_t KB_BYTES = DG_ROWS * 128;      // one k-block of a 128-row tile
    constexpr uint32_t OP_BYTES = KB * KB_BYTES;      // a whole operand tile (W2, or one stage of Y1)
    constexpr int LPR = C1 / 4;                       // lanes per edge row (float4 each)
    constexpr int RPI = 32 / LPR;                     // edge rows per warp iteration
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* w_s = smem;
    uint8_t* y_s = smem + OP_BYTES;                   // [2][OP_BYTES]
    uint64_t* wfull = reinterpret_cast<uint64_t*>(smem + 3 * OP_BYTES);
    uint64_t* yfull = wfull + 1;
    uint64_t* yempty = yfull + 2;
    uint64_t* tfull = yempty + 2;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int k = P.k, PTS = P.pts_per_tile;

    // zero both edge stages once: pad rows (beyond pts_per_tile * k) are never written again
    for (uint32_t i = threadIdx.x; i < 2 * OP_BYTES / 16; i += DG_THREADS)
        reinterpret_cast<uint4*>(y_s)[i] = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");

    if (warp == DG_ALLOC_WARP) {
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_w2)) : "memory");
            mbar_init(wfull, 1);
            for (int s = 0; s < 2; ++s) {
                mbar_init(&yfull[s], DG_GROUP_WARPS);
                mbar_init(&yempty[s], 1);
                mbar_init(&tfull[s], 1);
                mbar_init(&tempty[s], DG_EPI_WARPS);
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

    if (warp >= DG_EPI_WARPS) {
        // ------------------------------ producers ------------------------------
        const int pw = (warp - DG_EPI_WARPS) % DG_GROUP_WARPS;      // this warp's first point inside a tile
        const int grp = (warp - DG_EPI_WARPS) / DG_GROUP_WARPS;     // = the shared-memory / TMEM stage this warp fills
        const bool issuer = pw == 0;                                // this warp's lane 0 issues the group's MMAs
        if (warp == DG_ALLOC_WARP && lane == 0) {
            mbar_expect_tx(wfull, OP_BYTES);
            for (int kb2 = 0; kb2 < KB; ++kb2) tma_load_2d(w_s + kb2 * KB_BYTES, &tmap_w2, wfull, kb2 * 32, 0);
        }
        const uint32_t idesc = make_idesc(128, P.n_mma);
        const uint32_t w_addr = smem_u32(w_s);
        bool w_ready = false;
        const int sr = lane / LPR, lc = lane % LPR;    // sub-row of this lane within the iteration, 16-byte chunk index
        const int kb = lc >> 3, chunk = lc & 7;
        float s1[4], t1[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { s1[u] = __ldg(P.s1 + lc * 4 + u); t1[u] = __ldg(P.t1 + lc * 4 + u); }
        const long long tstep = 2LL * gridDim.x;       // this group's tiles: every other tile of the CTA
        long long t = blockIdx.x + (long long)grp * gridDim.x;
        // software pipeline: the neighbour list and centre row of this warp's first point of its NEXT tile are
        // requested before waiting for the stage, so the idx -> gather dependency is off the critical path
        int nj = 0;
        float4 nq = make_float4(0.f, 0.f, 0.f, 0.f);
        auto prefetch = [&](long long tile) {
            const long long pt = tile * PTS + pw;
            if (tile < P.num_tiles && pw < PTS && pt < P.total_pts) {
                nj = (lane < k) ? __ldg(P.idx + pt * k + lane) : 0;
                nq = __ldg(reinterpret_cast<const float4*>(P.q + pt * P.ldq + lc * 4));
            }
        };
        prefetch(t);
        uint8_t* ys = y_s + grp * OP_BYTES + kb * KB_BYTES;
        for (uint32_t it = 0; t < P.num_tiles; t += tstep, ++it) {
            const uint32_t ph = it & 1;
            const int cj = nj;
            const float4 cq = nq;
            prefetch(t + tstep);
            mbar_wait(&yempty[grp], ph ^ 1);
            for (int pl = pw; pl < PTS; pl += DG_GROUP_WARPS) {
                const long long pt = t * PTS + pl;
                if (pt >= P.total_pts) break;
                const long long cloud0 = (pt / P.N) * P.N;
                float4 qv = cq;
                int myj = cj;
                if (pl != pw) {
                    qv = __ldg(reinterpret_cast<const float4*>(P.q + pt * P.ldq + lc * 4));
                    myj = (lane < k) ? __ldg(P.idx + pt * k + lane) : 0;
                }
                float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
                const float* pbase = P.p + cloud0 * P.ldp + lc * 4;   // row address = one 32-bit multiply-add on this base
                constexpr int U = 10;                 // gathers in flight per lane
                for (int m0 = 0; m0 < k; m0 += U * RPI) {
                    float4 pv[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int m = m0 + u * RPI + sr;
                        const int j = __shfl_sync(kFull, myj, m & 31);
                        if (m < k) pv[u] = __ldg(reinterpret_cast<const float4*>(pbase + (unsigned)(j * P.ldp)));
                    }
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int m = m0 + u * RPI + sr;
                        if (m < k) {
                            float4 y;
                            y.x = fmaf(s1[0], pv[u].x + qv.x, t1[0]); y.y = fmaf(s1[1], pv[u].y + qv.y, t1[1]);
                            y.z = fmaf(s1[2], pv[u].z + qv.z, t1[2]); y.w = fmaf(s1[3], pv[u].w + qv.w, t1[3]);
                            y.x = fmaxf(y.x, y.x * P.neg_slope); y.y = fmaxf(y.y, y.y * P.neg_slope);
                            y.z = fmaxf(y.z, y.z * P.neg_slope); y.w = fmaxf(y.w, y.w * P.neg_slope);
                            best[0] = fmaxf(best[0], y.x); best[1] = fmaxf(best[1], y.y);
                            best[2] = fmaxf(best[2], y.z); best[3] = fmaxf(best[3], y.w);
                            const int e = pl * k + m;                                   // edge row inside the tile
                            *reinterpret_cast<float4*>(ys + e * 128 + ((chunk ^ (e & 7)) << 4)) = y;
                        }
                    }
                }
                if (P.x1) {
                    if (RPI == 2) {
#pragma unroll
                        for (int u = 0; u < 4; ++u) best[u] = fmaxf(best[u], __shfl_xor_sync(kFull, best[u], 16));
                    }
                    if (sr == 0) *reinterpret_cast<float4*>(P.x1 + pt * P.ld1 + lc * 4) = make_float4(best[0], best[1], best[2], best[3]);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&yfull[grp]);
            if (issuer) {   // warp-uniform: the whole warp runs the issue sequence, elect.sync picks the lane (see tc_common.cuh)
                // all six producer warps of the group run in lockstep on equal work, so this wait is short
                if (!w_ready) { mbar_wait(wfull, 0); w_ready = true; }
                mbar_wait(&tempty[grp], ph ^ 1);
                mbar_wait(&yfull[grp], ph);
                tc_fence_after();
                const uint32_t y_addr = smem_u32(y_s + grp * OP_BYTES);
#pragma unroll
                for (int kb2 = 0; kb2 < KB; ++kb2) {
                    const uint64_t da = make_smem_desc(w_addr + kb2 * KB_BYTES), db = make_smem_desc(y_addr + kb2 * KB_BYTES);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
                        tc_mma_tf32_e(tmem_base + grp * DG_ACC_STRIDE, da + (uint64_t)(ks * 2), db + (uint64_t)(ks * 2), idesc,
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
        // -> the per-edge work is a bare min/max over the k accumulator columns of the point (3-input FMNMX on sm_100).
        const int ch = warp * 32 + lane;               // output channel = TMEM lane
        const bool ch_ok = ch < P.C2;
        const float s2 = ch_ok ? __ldg(P.s2 + ch) : 0.f, t2 = ch_ok ? __ldg(P.t2 + ch) : 0.f;
        long long t = blockIdx.x;
        for (uint32_t it = 0; t < P.num_tiles; t += gridDim.x, ++it) {
            const uint32_t s = it & 1, ph = (it >> 1) & 1;
            mbar_wait(&tfull[s], ph);
            tc_fence_after();
            if (warp * 32 < P.C2) {
                for (int pl = 0; pl < PTS; ++pl) {
                    const long long pt = t * PTS + pl;
                    if (pt >= P.total_pts) break;
                    const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + s * DG_ACC_STRIDE + pl * k;
                    float mx, mn;
                    if (k == 20) {                      // the reference's k: exactly 16 + 4 columns, no masking
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
                        mx = fmaxf(fmaxf(a4[0], a4[1]), fmaxf(a4[2], a4[3]));
                        mn = fminf(fminf(b4[0], b4[1]), fminf(b4[2], b4[3]));
                    } else {
                        uint32_t r[32];
                        tc_ld32(taddr, r);
                        float a4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY}, b4[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float v = __uint_as_float(r[j]);
                            a4[j & 3] = fmaxf(a4[j & 3], j < k ? v : -INFINITY);
                            b4[j & 3] = fminf(b4[j & 3], j < k ? v : INFINITY);
                        }
                        mx = fmaxf(fmaxf(a4[0], a4[1]), fmaxf(a4[2], a4[3]));
                        mn = fminf(fminf(b4[0], b4[1]), fminf(b4[2], b4[3]));
                    }
                    float v = fmaf(s2, s2 >= 0.f ? mx : mn, t2);
                    v = fmaxf(v, v * P.neg_slope);
                    if (ch_ok) P.x2[pt * P.ld2 + ch] = v;
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[s]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == DG_ALLOC_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

template <int C1>
static int dg_tc_launch(const CUtensorMap& tw, DgTcParams P, cudaStream_t st) {
    constexpr size_t smem = 3 * (size_t)(C1 / 32) * DG_ROWS * 128 + 256;
    LPD_CUDA_CHECK(allow_smem(edgeconv_dg_tc_kernel<C1>, smem));
    int sms = 0;
    const int rc = sm_count(&sms);
    if (rc != LPD_OK) return rc;
    const int grid = (int)(P.num_tiles < sms ? P.num_tiles : sms);
    edgeconv_dg_tc_kernel<C1><<<grid, DG_THREADS, smem, st>>>(tw, P);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

int dg20_tc_run(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, const float* w2,
                const float* s2, const float* t2, float neg_slope, float* x1, int ld1, float* x2, int ld2, cudaStream_t st);

}  // namespace tc
}  // namespace lpd

extern "C" int lpd_edgeconv_dg_tf32(const float* p, int ldp, const float* q, int ldq,
                                    const int32_t* idx, int B, int N, int k, int C1, int C2,
                                    const float* s1, const float* t1, const float* w2,
                                    const float* s2, const float* t2, int act, float slope,
                                    float* x1, int ld1, float* x2, int ld2, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(p && q && idx && w2 && s2 && t2 && x2);
    LPD_REQUIRE((s1 && t1) || (!s1 && !t1 && k == 20 && C1 == 128 && C2 == 128));   // pre-scaled first layer: specialised kernel only
    LPD_REQUIRE(B >= 1 && N >= 1 && k >= 1 && k <= 32 && k <= N);
    LPD_REQUIRE((C1 == 128 && C2 == 128) || (C1 == 64 && C2 == 64));
    LPD_REQUIRE(ldp % 4 == 0 && ldq % 4 == 0 && (!x1 || ld1 % 4 == 0));
    LPD_REQUIRE(ldp >= C1 && ldq >= C1 && ld2 >= C2 && (!x1 || ld1 >= C1));
    LPD_REQUIRE((long long)N * ldp < (1ll << 31));          // cloud-local row offsets are 32-bit
    LPD_REQUIRE(((uintptr_t)p & 15) == 0 && ((uintptr_t)q & 15) == 0 && ((uintptr_t)x1 & 15) == 0 && ((uintptr_t)w2 & 15) == 0);
    LPD_REQUIRE(act_is_slope(act, slope));
    int rc = require_sm100();
    if (rc != LPD_OK) return rc;
    if (!s1)    // k = 20, 128 channels, first-layer BatchNorm already applied by the projection GEMM (edge_tc20.cu)
        return tc::dg20_tc_run(p, ldp, q, ldq, idx, B, N, w2, s2, t2, act_neg_slope(act, slope), x1, ld1, x2, ld2, as_stream(stream));
    tc::DgTcParams P;
    P.p = p; P.q = q; P.idx = idx; P.s1 = s1; P.t1 = t1; P.s2 = s2; P.t2 = t2; P.x1 = x1; P.x2 = x2;
    P.ldp = ldp; P.ldq = ldq; P.ld1 = ld1; P.ld2 = ld2; P.total_pts = (long long)B * N; P.N = N; P.k = k; P.C2 = C2;
    P.neg_slope = act_neg_slope(act, slope);
    P.pts_per_tile = tc::DG_ROWS / k;
    P.n_mma = (P.pts_per_tile * k + 15) / 16 * 16;
    P.num_tiles = (P.total_pts + P.pts_per_tile - 1) / P.pts_per_tile;
    CUtensorMap tw;   // rows beyond C2 are zero-filled by TMA
    rc = tc::make_tmap(&tw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w2, C2, C1, C1, tc::DG_ROWS, 32);
    if (rc != LPD_OK) return rc;
    cudaStream_t st = as_stream(stream);
    if (C1 == 128) return tc::dg_tc_launch<128>(tw, P, st);
    return tc::dg_tc_launch<64>(tw, P, st);
}
