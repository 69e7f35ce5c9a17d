// Feature-space kNN (C = 64) with the distance GEMM on the tensor cores and an EXACT result.
// Replaces knn() on the 64-channel feature map, reference util/lpdnet_model.py:246 -> :336 -> :317-326.
//
// Filter and refine (SURVEY.md H2), four launches on one stream:
//   1. knn_split_kernel     x -> X2 = [hi | lo] with hi = tf32(x), lo = tf32(x - hi)  (error-free split to 2^-22), the
//                           canonical squared norms xx_j (+inf padded) and the largest norm of every cloud.
//   2. knn_tc_kernel        tcgen05.mma kind::tf32, "3xTF32":  dot~ = Ahi.Blo + Alo.Bhi + Ahi.Bhi  accumulated in fp32 in
//                           TMEM (queries = TMEM lanes, 64 candidates = columns per stage).  Eight scan warps: warp w and
//                           warp w+4 share TMEM quadrant w and split every stage's columns in two halves, so each of the
//                           256 scan threads owns (one query row, one half of the candidate stream): score
//                           a_j = 2 dot~ - xx_j is compared against the thread's current L'-th best score; survivors
//                           (a register bit mask per 16 columns) replace the worst entry of the thread's unsorted
//                           candidate list (RowSelect, knn_select.cuh).  L' = 24 (k <= 24) or 32 (k <= 32) per half.
//                           The N x N matrix never leaves TMEM; the 2 L' candidates per row go to the workspace.
//   3. knn_refine_kernel    one warp per row: the L candidates are re-scored with the CANONICAL fp32 arithmetic of lpd_knn
//                           (fmaf chain, c ascending; pd = ((-xx_j) - (-2 dot)) - xx_i), sorted by (pd descending, index
//                           ascending) and the first k are written.  Every point outside the two half-lists has an
//                           approximate score <= tau (the larger of the two worst entries), so the lists provably hold the
//                           canonical top-k when
//                               tau + eps_i < pd_k + xx_i ,   eps_i = 2^-14 |x_i| max_j |x_j| + 2^-20 (xx_i + max_j xx_j)
//                           (>= 2.5x the summed worst-case error of the 3xTF32 gram and of the canonical chain).
//   4. rows that fail the test (masses of near-ties, e.g. duplicated points) flag their 64-row tile, which the exact
//      CUDA-core kernel (knn.cu) recomputes.  The result is bit-identical to lpd_knn whichever path produced a row.
#include "tc_common.cuh"
#include "knn_select.cuh"

namespace lpd {

int knn_simt64_flagged(const float* x, int B, int N, int k, void* idx, int idx_i64, const int* flags, cudaStream_t st);

namespace tc {

constexpr int KT_Q = 128;          // queries per work item (TMEM lanes)
constexpr int KT_C = 64;           // candidates per stage (TMEM columns)
constexpr int KT_SCAN_WARPS = 8;   // warps 0-7 scan/select (warp w: TMEM quadrant w % 4, column half w / 4)
constexpr int KT_THREADS = 320;    // + warp 8 TMA, warp 9 MMA
constexpr int KT_STRIDE = 257;     // list / queue words between slots: 256 (row, half) owners + 1 pad
constexpr int KT_BSTAGES = 3;      // shared-memory candidate stages (the TMA round trip is ~3 MMA stage times)
constexpr int KT_TSTAGES = 4;      // TMEM accumulator stages
constexpr int KT_XSLOTS = 8;       // candidate-norm slots (>= BSTAGES + TSTAGES)

struct KnnTcParams {
    const float* xxpad;    // [B][Npad] canonical squared norms, +inf padded
    float* cand_v;         // [B*N][2][L'] approximate scores of the surviving candidates of the two column halves
    int* cand_i;           // [B*N][2][L'] their cloud-local indices (INT_MAX = empty slot)
    int B, N, Npad;
    int qtiles, ctiles;    // per cloud
};

// Candidate tiles are streamed nearest-first in INDEX space around the query tile: 0, +1, -1, +2, -2, ... (mod ctiles, every
// tile exactly once).  The host modules feed clouds in spatial (grid-cell) order, so index-near candidates are space-near
// and, the features being smooth in space, feature-near: the lists' thresholds are almost final after the first few tiles
// and later candidates fail the cheap threshold test.  (Streaming from tile 0 instead is the WORST case for a cloud in
// spatial order: candidates improve monotonically and every one of them is inserted.)
__device__ __forceinline__ int ct_of(int s, int center, int ctiles) {
    const int d = (s + 1) >> 1;
    int ct = center + ((s & 1) ? d : -d);
    ct %= ctiles;
    return ct < 0 ? ct + ctiles : ct;
}

__device__ __forceinline__ float to_tf32(float v) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
    return __uint_as_float(r);
}

// one warp per point: hi / lo split, canonical squared norm (same fmaf chain as lpd_knn), per-cloud max norm
__global__ void __launch_bounds__(256)
knn_split_kernel(const float* __restrict__ x, int N, int Npad, float* __restrict__ x2, float* __restrict__ xxpad,
                 float* __restrict__ r2) {
    const int b = blockIdx.y;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= Npad) return;
    float v = INFINITY;
    if (n < N) {
        const float4* p = reinterpret_cast<const float4*>(x + ((size_t)b * N + n) * 64);
        float4* o = reinterpret_cast<float4*>(x2 + ((size_t)b * N + n) * 128);
        float acc = 0.f;
#pragma unroll
        for (int g = 0; g < 16; ++g) {
            const float4 t = __ldg(p + g);
            acc = __fmaf_rn(t.x, t.x, acc); acc = __fmaf_rn(t.y, t.y, acc);
            acc = __fmaf_rn(t.z, t.z, acc); acc = __fmaf_rn(t.w, t.w, acc);
            float4 hi, lo;
            hi.x = to_tf32(t.x); hi.y = to_tf32(t.y); hi.z = to_tf32(t.z); hi.w = to_tf32(t.w);
            lo.x = to_tf32(t.x - hi.x); lo.y = to_tf32(t.y - hi.y); lo.z = to_tf32(t.z - hi.z); lo.w = to_tf32(t.w - hi.w);
            o[g] = hi;
            o[16 + g] = lo;
        }
        v = acc;
        atomicMax(reinterpret_cast<int*>(r2 + b), __float_as_int(acc));   // acc >= 0: int order == float order
    }
    xxpad[(size_t)b * Npad + n] = v;
}

template <int GS, int QD>
struct KtSmem {
    static constexpr int L = 4 * GS;                      // candidates kept per (row, column half)
    static constexpr uint32_t A_KB = KT_Q * 128;          // one 32-channel k-block of the query tile
    static constexpr uint32_t B_KB = KT_C * 128;
    static constexpr uint32_t A_BYTES = 4 * A_KB;         // hi0 hi1 lo0 lo1
    static constexpr uint32_t B_BYTES = 4 * B_KB;
    static constexpr size_t off_b = A_BYTES;
    static constexpr size_t off_xs = off_b + KT_BSTAGES * B_BYTES;
    static constexpr size_t off_lv = off_xs + KT_XSLOTS * KT_C * 4;
    static constexpr size_t off_li = off_lv + (size_t)L * KT_STRIDE * 4;
    static constexpr size_t off_bar = (off_li + (size_t)L * KT_STRIDE * 4 + 7) / 8 * 8;
    static constexpr size_t total = off_bar + (2 + 2 * KT_BSTAGES + 2 * KT_TSTAGES) * 8 + 16;
    static_assert(total <= 227 * 1024, "knn_tc shared memory budget");
};

template <int GS, int QD>
__global__ void __launch_bounds__(KT_THREADS, 1)
knn_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, KnnTcParams P) {
    using S = KtSmem<GS, QD>;
    constexpr int L = S::L;
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* a_s = smem;
    uint8_t* b_s = smem + S::off_b;
    float* xs = reinterpret_cast<float*>(smem + S::off_xs);
    float* lv = reinterpret_cast<float*>(smem + S::off_lv);
    int* li = reinterpret_cast<int*>(smem + S::off_li);
    uint64_t* afull = reinterpret_cast<uint64_t*>(smem + S::off_bar);
    uint64_t* aempty = afull + 1;
    uint64_t* bfull = aempty + 1;
    uint64_t* bempty = bfull + KT_BSTAGES;
    uint64_t* tfull = bempty + KT_BSTAGES;
    uint64_t* tempty = tfull + KT_TSTAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + KT_TSTAGES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int items = P.B * P.qtiles;

    if (warp == 9) {
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
            mbar_init(afull, 1); mbar_init(aempty, 1);
            for (int s = 0; s < KT_BSTAGES; ++s) { mbar_init(&bfull[s], 1); mbar_init(&bempty[s], 1); }
            for (int s = 0; s < KT_TSTAGES; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], KT_SCAN_WARPS); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 8) {
        // ------------------------------ TMA producer ------------------------------
        if (lane == 0) {
            uint32_t tcount = 0, icount = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x, ++icount) {
                const int b = item / P.qtiles, q0 = (item % P.qtiles) * KT_Q;
                mbar_wait_sleep(aempty, (icount & 1) ^ 1);
                mbar_expect_tx(afull, S::A_BYTES);
#pragma unroll
                for (int kb = 0; kb < 4; ++kb) tma_load_2d(a_s + kb * S::A_KB, &tmap_a, afull, kb * 32, b * P.N + q0);
                for (int cs = 0; cs < P.ctiles; ++cs, ++tcount) {
                    const int ct = ct_of(cs, q0 / KT_C, P.ctiles);
                    const uint32_t s = tcount % KT_BSTAGES, ph = (tcount / KT_BSTAGES) & 1;
                    mbar_wait_sleep(&bempty[s], ph ^ 1);
                    mbar_expect_tx(&bfull[s], S::B_BYTES + KT_C * 4);
                    uint8_t* bs = b_s + s * S::B_BYTES;
#pragma unroll
                    for (int kb = 0; kb < 4; ++kb) tma_load_2d(bs + kb * S::B_KB, &tmap_b, &bfull[s], kb * 32, b * P.N + ct * KT_C);
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"(smem_u32(xs + (tcount % KT_XSLOTS) * KT_C)), "l"(P.xxpad + (size_t)b * P.Npad + ct * KT_C),
                                   "r"(KT_C * 4), "r"(smem_u32(&bfull[s])) : "memory");
                }
            }
        }
    } else if (warp == 9) {
        // ------------------------------ MMA issuer ------------------------------
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(KT_Q, KT_C);
            const uint32_t a_addr = smem_u32(a_s);
            uint32_t tcount = 0, icount = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x, ++icount) {
                mbar_wait_sleep(afull, icount & 1);
                for (int ct = 0; ct < P.ctiles; ++ct, ++tcount) {
                    const uint32_t s = tcount % KT_BSTAGES, ph = (tcount / KT_BSTAGES) & 1;
                    const uint32_t ts = tcount % KT_TSTAGES, tph = (tcount / KT_TSTAGES) & 1;
                    mbar_wait_sleep(&tempty[ts], tph ^ 1);
                    mbar_wait_sleep(&bfull[s], ph);
                    tc_fence_after();
                    const uint32_t b_addr = smem_u32(b_s + s * S::B_BYTES);
                    const uint32_t d = tmem_base + ts * KT_C;
                    uint32_t acc = 0;
                    // small terms first: Ahi.Blo, Alo.Bhi, then Ahi.Bhi  (k-blocks: 0,1 = hi ; 2,3 = lo)
#pragma unroll
                    for (int term = 0; term < 3; ++term) {
                        const int akb = (term == 1) ? 2 : 0, bkb = (term == 0) ? 2 : 0;
#pragma unroll
                        for (int kb = 0; kb < 2; ++kb) {
                            const uint64_t da = make_smem_desc(a_addr + (akb + kb) * S::A_KB);
                            const uint64_t db = make_smem_desc(b_addr + (bkb + kb) * S::B_KB);
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                tc_mma_tf32(d, da + (uint64_t)(ks * 2), db + (uint64_t)(ks * 2), idesc, acc);
                                acc = 1;
                            }
                        }
                    }
                    tc_commit(&bempty[s]);
                    tc_commit(&tfull[ts]);
                }
                tc_commit(aempty);   // all MMAs that read this query tile have completed when this arrives
            }
        }
    } else {
        // ------------------------------ scan + select: one (query row, column half) per thread ------------------------------
        const int quad = warp & 3, half = warp >> 2;
        const int own = half * KT_Q + quad * 32 + lane;   // this thread's column of the list / queue arrays
        RowSelect<GS, false, KT_STRIDE> sel;
        uint32_t tcount = 0;
        for (int item = blockIdx.x; item < items; item += gridDim.x) {
            const int b = item / P.qtiles, q0 = (item % P.qtiles) * KT_Q;
            sel.reset();
            for (int cs = 0; cs < P.ctiles; ++cs, ++tcount) {
                const int ct = ct_of(cs, q0 / KT_C, P.ctiles);
                const uint32_t ts = tcount % KT_TSTAGES, tph = (tcount / KT_TSTAGES) & 1;
                mbar_wait(&tfull[ts], tph);
                tc_fence_after();
                const float* xsj = xs + (tcount % KT_XSLOTS) * KT_C + half * 32;
                uint32_t r[32];
                tc_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + ts * KT_C + half * 32, r);
                // accumulator half fully read: hand the stage back before the selection work
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[ts]);
                const int jbase = ct * KT_C + half * 32;
#pragma unroll
                for (int sub = 0; sub < 32 / QD; ++sub) {
                    float a[QD];
                    float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
                    for (int j = 0; j < QD; j += 4) {
                        const float4 xx = *reinterpret_cast<const float4*>(xsj + sub * QD + j);   // warp broadcast
                        a[j + 0] = fmaf(2.f, __uint_as_float(r[sub * QD + j + 0]), -xx.x);
                        a[j + 1] = fmaf(2.f, __uint_as_float(r[sub * QD + j + 1]), -xx.y);
                        a[j + 2] = fmaf(2.f, __uint_as_float(r[sub * QD + j + 2]), -xx.z);
                        a[j + 3] = fmaf(2.f, __uint_as_float(r[sub * QD + j + 3]), -xx.w);
                        m4[0] = fmaxf(m4[0], a[j]); m4[1] = fmaxf(m4[1], a[j + 1]);
                        m4[2] = fmaxf(m4[2], a[j + 2]); m4[3] = fmaxf(m4[3], a[j + 3]);
                    }
                    const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
                    // survivors of this thread as a bit mask; they are inserted one per warp iteration (the list lives in
                    // shared memory, the scores stay in registers and are picked by a select tree on the bit index)
                    uint32_t mask = 0;
                    if (mx > sel.tau) {
#pragma unroll
                        for (int j = 0; j < QD; ++j) mask |= (a[j] > sel.tau) ? (1u << j) : 0u;
                    }
                    while (__any_sync(kFull, mask != 0)) {
                        if (mask) {
                            const int j = __ffs(mask) - 1;
                            mask &= mask - 1;
                            float t[QD];
#pragma unroll
                            for (int q = 0; q < QD; ++q) t[q] = a[q];
#pragma unroll
                            for (int w = QD / 2, bit = 0; w >= 1; w >>= 1, ++bit) {
                                const bool hi = (j >> bit) & 1;
#pragma unroll
                                for (int q = 0; q < w; ++q) t[q] = hi ? t[2 * q + 1] : t[2 * q];
                            }
                            sel.insert(lv, li, own, t[0], jbase + sub * QD + j);
                        }
                    }
                }
            }
            // ---------------- hand the L' candidates of every (row, half) to the refine kernel (coalesced rows) ----------------
            __syncwarp();
            for (int rl = 0; rl < 32; ++rl) {
                const int qrow = q0 + quad * 32 + rl;
                const int nfill = __shfl_sync(kFull, sel.filled, rl);
                if (qrow >= P.N) break;
                const size_t o = (((size_t)b * P.N + qrow) * 2 + half) * L;
                const int src = half * KT_Q + quad * 32 + rl;
                for (int s = lane; s < L; s += 32) {
                    const bool valid = s < nfill;
                    P.cand_v[o + s] = valid ? lv[s * KT_STRIDE + src] : -INFINITY;
                    P.cand_i[o + s] = valid ? li[s * KT_STRIDE + src] : INT_MAX;
                }
            }
            __syncwarp();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 9) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
    }
}

// one warp per query row: canonical re-score of its 2 L' candidates, exact sort, guarantee test
__global__ void __launch_bounds__(256)
knn_refine_kernel(const float* __restrict__ x, const float* __restrict__ xxpad, const float* __restrict__ r2,
                  const float* __restrict__ cand_v, const int* __restrict__ cand_i, int Lh, int B, int N, int Npad, int k,
                  void* __restrict__ idx_out, int idx_i64, int* __restrict__ flags) {
    constexpr int E = 2;
    const int lane = threadIdx.x & 31;
    const long long grow = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (grow >= (long long)B * N) return;
    const int b = (int)(grow / N), qi = (int)(grow % N);
    const int L = 2 * Lh;
    float av[E]; int id[E];
    float tmin[2] = {INFINITY, INFINITY};     // worst approximate score of each half-list
    bool hfull[2] = {true, true};             // half-list completely filled (otherwise it holds ALL candidates of its half)
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int s = e * 32 + lane;
        av[e] = -INFINITY; id[e] = INT_MAX;
        if (s < L) {
            av[e] = cand_v[grow * L + s];
            id[e] = cand_i[grow * L + s];
            const int h = s >= Lh;
            if (id[e] == INT_MAX || id[e] >= N) {
                id[e] = INT_MAX;
                if (h) hfull[1] = false; else hfull[0] = false;
            } else {
                if (h) tmin[1] = fminf(tmin[1], av[e]); else tmin[0] = fminf(tmin[0], av[e]);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tmin[0] = fminf(tmin[0], __shfl_xor_sync(kFull, tmin[0], o));
        tmin[1] = fminf(tmin[1], __shfl_xor_sync(kFull, tmin[1], o));
    }
    const bool full0 = __all_sync(kFull, hfull[0]), full1 = __all_sync(kFull, hfull[1]);
    // every candidate outside the lists scores <= tau; a half-list that never filled has no outsiders
    const float tau = fmaxf(full0 ? tmin[0] : -INFINITY, full1 ? tmin[1] : -INFINITY);
    const float xxi = __ldg(xxpad + (size_t)b * Npad + qi);
    const float rmax2 = __ldg(r2 + b);
    const float eps = 6.103515625e-5f * sqrtf(xxi) * sqrtf(rmax2) + 9.5367431640625e-7f * (xxi + rmax2);
    // prune: sort by approximate score; a candidate scoring below (k-th best approximate score) - 2 eps cannot be in the
    // canonical top-k (k candidates have canonical score >= a_k - eps, its own is < a_k - eps), so it is not re-scored
    warp_sort_desc<E>(av, id, lane);
    const float a_k = __shfl_sync(kFull, av[0], k - 1);
    const float cut = a_k - 2.f * eps;
    const float4* xi = reinterpret_cast<const float4*>(x + ((size_t)b * N + qi) * 64);
    float pd[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        pd[e] = -INFINITY;
        const bool keep = (id[e] != INT_MAX) && (av[e] >= cut);
        if (!keep) id[e] = INT_MAX;
        if (__any_sync(kFull, keep)) {
            if (keep) {
                const float4* xj = reinterpret_cast<const float4*>(x + ((size_t)b * N + id[e]) * 64);
                float dot = 0.f;
#pragma unroll
                for (int g = 0; g < 16; ++g) {
                    const float4 u = __ldg(xi + g), w = __ldg(xj + g);
                    dot = __fmaf_rn(u.x, w.x, dot); dot = __fmaf_rn(u.y, w.y, dot);
                    dot = __fmaf_rn(u.z, w.z, dot); dot = __fmaf_rn(u.w, w.w, dot);
                }
                const float xxj = __ldg(xxpad + (size_t)b * Npad + id[e]);
                const float t = -2.0f * dot;
                pd[e] = __fsub_rn(__fsub_rn(-xxj, t), xxi);
            }
        }
    }
    warp_sort_desc<E>(pd, id, lane);
    const float pd_k = __shfl_sync(kFull, pd[0], k - 1);   // k <= 32: always in the first register
    const bool ok = (tau == -INFINITY) || (tau + eps < pd_k + xxi);
    const size_t o = (size_t)grow * k;
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int g = e * 32 + lane;
        if (g < k) {
            if (idx_i64) reinterpret_cast<long long*>(idx_out)[o + g] = id[e];
            else reinterpret_cast<int*>(idx_out)[o + g] = id[e];
        }
    }
    if (!ok && lane == 0) flags[(size_t)b * ((N + 63) / 64) + qi / 64] = 1;
}

template <int GS, int QD>
static int knn_tc_launch(const CUtensorMap& ta, const CUtensorMap& tb, const KnnTcParams& P, cudaStream_t st) {
    const size_t smem = KtSmem<GS, QD>::total;
    LPD_CUDA_CHECK(allow_smem(knn_tc_kernel<GS, QD>, smem));
    int sms = 0;
    const int rc = sm_count(&sms);
    if (rc != LPD_OK) return rc;
    const int items = P.B * P.qtiles;
    knn_tc_kernel<GS, QD><<<items < sms ? items : sms, KT_THREADS, smem, st>>>(ta, tb, P);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct KnnWs {
    size_t off_xx, off_r2, off_flags, off_x2, off_cv, off_ci, total;
    int npad, L;
    KnnWs(int B, int N, int k) {
        npad = (N + 127) / 128 * 128;
        L = k <= 24 ? 48 : 64;      // 2 half-lists of 24 / 32
        size_t o = 0;
        off_xx = o; o = align_up(o + (size_t)B * npad * 4, 256);
        off_r2 = o; o += (size_t)B * 4;
        off_flags = o; o = align_up(o + (size_t)B * ((N + 63) / 64) * 4, 256);
        off_x2 = o; o = align_up(o + (size_t)B * N * 128 * 4, 256);
        off_cv = o; o = align_up(o + (size_t)B * N * L * 4, 256);
        off_ci = o; o = align_up(o + (size_t)B * N * L * 4, 256);
        total = o;
    }
};

}  // namespace tc
}  // namespace lpd

namespace lpd { namespace tc {
size_t knn2_workspace_bytes(int B, int N, int k);
size_t knn2_flags_offset(int B, int N, int k);
int knn2_run(const float* x, int B, int N, int k, void* idx, int idx_i64, void* workspace, size_t workspace_bytes, int mt,
             cudaStream_t st);
// 0 = single-pass 3xTF32 replace-worst filter (this file); 1 / 2 = two-pass fp16 threshold filter (knn_tc2.cu) with
// 128 / 256 query rows per work item; 3 = variant 1 with the query tile in tensor memory (TS-mode MMA).  Every variant returns the same (canonical) indices.
static int g_knn_variant = 1;
}}

extern "C" int lpd_knn_tc_variant(int v) {
    const int prev = lpd::tc::g_knn_variant;
    if (v >= 0 && v <= 3) lpd::tc::g_knn_variant = v;
    return prev;
}

extern "C" size_t lpd_knn_workspace_bytes(int B, int N, int C, int k) {
    if (B < 1 || N < 1 || C != 64 || k < 1 || k > 32) return 0;
    const size_t a = lpd::tc::KnnWs(B, N, k).total, b = lpd::tc::knn2_workspace_bytes(B, N, k);
    return a > b ? a : b;
}

extern "C" size_t lpd_knn_tc_flags_offset(int B, int N, int C, int k) {
    if (B < 1 || N < 1 || C != 64 || k < 1 || k > 32) return 0;
    return lpd::tc::g_knn_variant == 0 ? lpd::tc::KnnWs(B, N, k).off_flags : lpd::tc::knn2_flags_offset(B, N, k);
}

extern "C" int lpd_knn_tc(const float* x, int B, int N, int C, int k, void* idx, int idx_i64,
                          void* workspace, size_t workspace_bytes, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(x && idx && workspace);
    LPD_REQUIRE(B >= 1 && B <= 65535 && N >= 1 && C == 64 && k >= 1 && k <= 32 && k <= N);
    LPD_REQUIRE((long long)B * N < (1ll << 31) / 128);
    LPD_REQUIRE(((uintptr_t)x & 15) == 0 && ((uintptr_t)workspace & 255) == 0);
    const tc::KnnWs W(B, N, k);
    if (workspace_bytes < lpd_knn_workspace_bytes(B, N, C, k)) return LPD_EWORKSPACE;
    int rc = require_sm100();
    if (rc != LPD_OK) return rc;
    cudaStream_t st = as_stream(stream);
    if (tc::g_knn_variant != 0) return tc::knn2_run(x, B, N, k, idx, idx_i64, workspace, workspace_bytes, tc::g_knn_variant, st);
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    float* xxpad = reinterpret_cast<float*>(ws + W.off_xx);
    float* r2 = reinterpret_cast<float*>(ws + W.off_r2);
    int* flags = reinterpret_cast<int*>(ws + W.off_flags);
    float* x2 = reinterpret_cast<float*>(ws + W.off_x2);
    const int ftiles = (N + 63) / 64;
    LPD_CUDA_CHECK(cudaMemsetAsync(r2, 0, (size_t)B * sizeof(float), st));
    LPD_CUDA_CHECK(cudaMemsetAsync(flags, 0, (size_t)B * ftiles * sizeof(int), st));
    tc::knn_split_kernel<<<dim3(ceil_div(W.npad, 256), B), 256, 0, st>>>(x, N, W.npad, x2, xxpad, r2);
    LPD_LAUNCH_CHECK();
    CUtensorMap ta, tb;
    rc = tc::make_tmap(&ta, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, x2, (long long)B * N, 128, 128, tc::KT_Q, 32);
    if (rc != LPD_OK) return rc;
    rc = tc::make_tmap(&tb, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, x2, (long long)B * N, 128, 128, tc::KT_C, 32);
    if (rc != LPD_OK) return rc;
    tc::KnnTcParams P;
    P.xxpad = xxpad;
    P.cand_v = reinterpret_cast<float*>(ws + W.off_cv);
    P.cand_i = reinterpret_cast<int*>(ws + W.off_ci);
    P.B = B; P.N = N; P.Npad = W.npad; P.qtiles = ceil_div(N, tc::KT_Q); P.ctiles = ceil_div(N, tc::KT_C);
    rc = (W.L == 48) ? tc::knn_tc_launch<6, 16>(ta, tb, P, st) : tc::knn_tc_launch<8, 16>(ta, tb, P, st);
    if (rc != LPD_OK) return rc;
    const unsigned rblocks = (unsigned)(((long long)B * N + 7) / 8);
    tc::knn_refine_kernel<<<rblocks, 256, 0, st>>>(x, xxpad, r2, P.cand_v, P.cand_i, W.L / 2, B, N, W.npad, k, idx, idx_i64, flags);
    LPD_LAUNCH_CHECK();
    return knn_simt64_flagged(x, B, N, k, idx, idx_i64, flags, st);   // exact recompute of flagged 64-row tiles only
}
