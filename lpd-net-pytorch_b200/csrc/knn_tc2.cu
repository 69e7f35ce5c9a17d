// Feature-space kNN (C = 64), second tensor-core formulation: TWO-PASS THRESHOLD FILTER, fp16 gram, exact result.
// Replaces knn() on the 64-channel feature map, reference util/lpdnet_model.py:246 -> :336 -> :317-326.
//
// Why: the single-pass filter of knn_tc.cu keeps a per-row candidate list up to date while the gram streams by; the
// list updates (dependent shared-memory traffic, divergent) cost 4-5x the tensor work.  Here no list is ever maintained:
//
//   0. knn2_center_kernel   per cloud: mean feature mu and a power-of-two scale sigma so that (x - mu) * sigma fits fp16.
//      knn2_prep_kernel     per point: xh = fp16((x - mu) * sigma), centred norm nrm_j, canonical norm xx_j (fmaf chain of
//                           lpd_knn), per-cloud maxima of both, and the 16-column "K-extension" of the candidate operand
//                           (below).  Distances are translation invariant, so the centring only shrinks the operands (and
//                           with them the absolute rounding error of the fp16 gram).
//   1. knn2_tc_kernel       per work item (one cloud, 128*MT query rows) the candidates stream TWICE through tcgen05.mma
//                           kind::f16 (fp32 accumulation in TMEM), 128 candidates (two 64-point blocks) per stage.  Each
//                           stage is 4 MMAs over the 64 channels plus ONE MMA over the K-extension, whose operands
//                           ([2^6, 2^-5, 2^-14, 2^15, 0..] on the query side, three fp16 pieces of -sigma^2 nrm_j / 2 and a
//                           padding flag on the candidate side, no-swizzle core-matrix layout) make the tensor core itself
//                           deliver the finished score  t_ij = (sigma^2 / 2) (2 x'_i.x'_j - nrm_j)  with padded candidates
//                           at -2e9: the scan threads do no arithmetic on the scores, only comparisons.
//        pass 1  every scan thread (one query row, 32 storage positions of both blocks of a stage) keeps the running
//                maximum of each of its 32 positions: 64 "strided" groups per row (group = storage position inside the
//                64-block), no branches.  The k-th largest group maximum tau0 is a LOWER bound of the k-th best score of
//                the row (k distinct candidates reach it).  It is found with an in-register bitonic sort of the 32 maxima,
//                one exchange with the partner thread of the other 32 positions, and a bitonic merge.  Pass 1 also records,
//                per (warp, stage), D = min over the warp's 32 rows of (t_ii - best score of the row in the stage).
//        pass 2  the same stages again; a warp whose table entry says no row can reach its threshold does not even read the
//                accumulators (3 stages out of 4).  Otherwise every candidate with  t_ij >= tau0 - 2 eps_i  is appended to
//                the row's list in global memory (index only).  With |t_ij - (canonical score + const_i)| <= eps_i this set
//                provably holds the canonical top-k:  k candidates have canonical score >= tau0 - eps, so the canonical
//                k-th score is >= tau0 - eps, and everything at or above it has t_ij >= tau0 - 2 eps.  The set has ~1.4 k
//                members.
//      Column scrambling: the host modules feed clouds in grid-cell order, where the neighbours of a point sit at index
//      offsets that are near-multiples of the cell-row stride (64 points for N = 4096) and would pile up in the same
//      groups.  knn2_prep_kernel therefore stores every full 64-point block under its own affine permutation of the 64
//      positions (position = (a_t c + b_t) mod 64, a_t odd, hashed from the block number t); the scan maps hits back.
//      TIGHT (k > 24): the error bound is applied per candidate, e_ij = 2.5e-3 |x'_i| |x'_j| instead of its maximum over j:
//      pass 1 takes the maxima of the certified LOWER bounds t_ij - e_ij, pass 2 collects UPPER bounds t_ij + e_ij.
//   2. knn2_refine_kernel   one warp per row: canonical fp32 re-score of the collected candidates (the arithmetic of
//                           lpd_knn), rank by (pd descending, index ascending), first k written.
//   3. rows whose list overflowed (masses of near-ties, e.g. duplicated points) or whose cloud could not be scaled flag
//      their 64-row tile, which the exact CUDA-core kernel (knn.cu) recomputes.  Bit-identical to lpd_knn in every case.
//
// eps_i (in units of a = 2 x'_i.x'_j - nrm_j) = 2.5e-3 |x'_i| R' + 1.9e-6 (|x'_i| + R') / sigma + 2^-17 (xx_i + max xx) + 2^-18 R'^2:
//   * fp16 rounding of both operands (2^-11 relative each, 2^-25 absolute for subnormals; factor 2 of the score; 28 % spare);
//   * the fp32 accumulation of the tensor core including the K-extension (<= 2^-21 of the largest term per step);
//   * the WORST-CASE rounding of the canonical chain itself, which works on the UNcentred features: 64 fmaf steps give
//     |dot_fp32 - dot| <= 64 u |x_i||x_j| (u = 2^-24), doubled by the -2, plus <= 66 u per squared norm and the two
//     subtractions: <= 2^-17 (xx_i + max_j xx_j).  For features with a large common offset this term dominates and the
//     filter degrades to the exact fallback - the canonical fp32 ranking itself is ill-conditioned there.
//
// What bounds it (ncu, B200, 64 clouds x 4096): the accumulators are read from TMEM at 64 B/clk/SM (4.3 GB in pass 1 alone
// = 0.26 ms), and the MMA stream by itself (scan disabled) needs 0.31 ms: ~120 clk per 128 x 128 x 16 MMA, twice the
// tensor-pipe floor, whether the query tile comes from shared memory or from tensor memory (TS variant below: no gain) and
// whether consecutive MMAs share an accumulator or not.  N = 64 stages were worse (~90 clk per half-size MMA).  The
// single-thread roles issue through elect.sync (tc_common.cuh).
#include "tc_common.cuh"
#include <cuda_fp16.h>
#include <limits.h>
#include <stdlib.h>

namespace lpd {

int knn_simt64_list(const float* x, int B, int N, int k, void* idx, int idx_i64, const int* list, cudaStream_t st);

namespace tc {

constexpr int K2_C = 128;        // candidates per stage = two scrambled 64-blocks (TMEM columns per 128-row query tile);
                                 // tcgen05.mma with N = 64 ran at a third of its rate (per-instruction overhead), N = 128 does not
constexpr int K2_BSTAGES = 4;    // shared-memory candidate stages (16 + 4 KB each)
constexpr int K2_TCOLS = 512;    // TMEM columns used: 512 / (128 * MT) accumulator stages
constexpr int K2_XSLOTS = 12;    // candidate-norm slots (>= BSTAGES + TSTAGES + 3)
constexpr int K2_TBL = 128;      // candidate stages per cloud the pass-2 skip table covers (N <= 16384; beyond: no skipping)

struct Knn2Params {
    const float* nrmpad;   // [B][Npad] centred squared norms, +inf padded   (storage order, like the operand rows)
    const float* snpad;    // [B][Npad] their square roots, 0 padded          (storage order)
    const uint4* xh;       // [B*N][8] the fp16 operand rows (64 halves = 8 x 16 B), storage order (TS mode reads query rows)
    const uint4* ext;      // [B][Npad/64][128] K-extension rows of the candidate tiles (2 KB per tile, core-matrix layout)
    const float* xxpad;    // [B][Npad] canonical squared norms               (point order)
    const float* r2;       // [B] max canonical squared norm
    const float* r2c;      // [B] max centred squared norm
    const float* sc;       // [B][2] sigma, 2 / sigma^2  (NaN when the cloud cannot be scaled)
    int* cnt;              // [B*N][2] candidates found per (row, column half); > CAP = overflow
    int* cand;             // [B*N][2][CAP] cloud-local candidate indices
    int B, N, Npad, k;
    int qtiles, ctiles;    // per cloud
};

__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Warp-convergent issue: the WHOLE warp executes these with identical operands; elect.sync inside the asm picks the lane
// that issues.  The control flow stays uniform and ptxas emits ELECT + one predicated UTCHMMA / UTCBAR / UTMALDG instead
// of the elect-and-loop sequence it needs inside a divergent `if (lane == 0)` region (9-10 instructions per MMA there:
// the single issuing thread was the bottleneck of the whole kernel).  `leader` is unused (kept for call-site clarity).
__device__ __forceinline__ void tc_mma_f16_p(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate,
                                             uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tc_commit_p(uint64_t* bar, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(smem_u32(bar)), "r"(leader) : "memory");
}
__device__ __forceinline__ void tma_load_2d_p(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void bulk_load_p(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t}"
        ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "r"(leader) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_p(uint64_t* bar, uint32_t bytes, uint32_t leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}"
        ::"r"(smem_u32(bar)), "r"(bytes), "r"(leader) : "memory");
}
// the same with the A operand (query tile) in TENSOR MEMORY: lane = query row, 32-bit column c = fp16 elements (2c, 2c+1)
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_st4(uint32_t taddr, const uint4& v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                 ::"r"(taddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// kind::f16 with fp16 operands (format 0), fp32 accumulate, A and B K-major
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void named_bar(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// affine permutation of the 64 positions of candidate block t:  position = (a c + b) & 63,  a odd
__host__ __device__ __forceinline__ void block_perm(int t, int& a, int& b) {
    const uint32_t v = (uint32_t)(t + 1) * 2654435761u;
    a = (int)((v >> 8) & 63u) | 1;
    b = (int)((v >> 20) & 63u);
}
__host__ __device__ __forceinline__ int inv_mod64(int a) {   // a odd: a*a = 1 (mod 8); one Newton step doubles the bits
    return (a * (2 - a * a)) & 63;
}

// ---------------------------------------------------------------------------------------------------------------------
// 0a. per cloud: channel sums, minima and maxima.  K2_CSPLIT CTAs per cloud write partial results in a fixed order (no atomics:
// deterministic); knn2_prep_kernel folds them into the mean feature mu and the power-of-two fp16 scale sigma.
constexpr int K2_CSPLIT = 8;
__global__ void __launch_bounds__(256)
knn2_center_kernel(const float* __restrict__ x, int N, float* __restrict__ part) {
    __shared__ float4 red[3][256];
    __shared__ int sbad;
    const int b = blockIdx.y, sp = blockIdx.x, t = threadIdx.x, cg = t & 15, rl = t >> 4;
    const int chunk = (N + K2_CSPLIT - 1) / K2_CSPLIT;
    const int n0 = sp * chunk, n1 = min(N, n0 + chunk);
    const float4* xb = reinterpret_cast<const float4*>(x + (size_t)b * N * 64);
    if (t == 0) sbad = 0;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 lo = make_float4(INFINITY, INFINITY, INFINITY, INFINITY), hi = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    bool bad = false;                      // NaN / inf anywhere in the cloud must not be lost by fminf / fmaxf
    for (int n = n0 + rl; n < n1; n += 16) {
        const float4 v = __ldg(xb + (size_t)n * 16 + cg);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
        lo.x = fminf(lo.x, v.x); lo.y = fminf(lo.y, v.y); lo.z = fminf(lo.z, v.z); lo.w = fminf(lo.w, v.w);
        hi.x = fmaxf(hi.x, v.x); hi.y = fmaxf(hi.y, v.y); hi.z = fmaxf(hi.z, v.z); hi.w = fmaxf(hi.w, v.w);
        bad |= !(fabsf(v.x) <= 3.0e38f) || !(fabsf(v.y) <= 3.0e38f) || !(fabsf(v.z) <= 3.0e38f) || !(fabsf(v.w) <= 3.0e38f);
    }
    red[0][t] = s; red[1][t] = lo; red[2][t] = hi;
    __syncthreads();
    if (bad) sbad = 1;
    for (int o = 128; o >= 16; o >>= 1) {
        if (t < o) {
            const float4 a0 = red[0][t], c0 = red[0][t + o], a1 = red[1][t], c1 = red[1][t + o], a2 = red[2][t], c2 = red[2][t + o];
            red[0][t] = make_float4(a0.x + c0.x, a0.y + c0.y, a0.z + c0.z, a0.w + c0.w);
            red[1][t] = make_float4(fminf(a1.x, c1.x), fminf(a1.y, c1.y), fminf(a1.z, c1.z), fminf(a1.w, c1.w));
            red[2][t] = make_float4(fmaxf(a2.x, c2.x), fmaxf(a2.y, c2.y), fmaxf(a2.z, c2.z), fmaxf(a2.w, c2.w));
        }
        __syncthreads();
    }
    // partials of this CTA: [3][64] floats (sum, min, max) + the bad flag
    float* o = part + ((size_t)b * K2_CSPLIT + sp) * 196;
    if (t < 16) {
        reinterpret_cast<float4*>(o)[t] = red[0][t];
        reinterpret_cast<float4*>(o + 64)[t] = red[1][t];
        reinterpret_cast<float4*>(o + 128)[t] = red[2][t];
    }
    if (t == 0) o[192] = sbad ? 1.f : 0.f;
}

// folds the partials of one cloud: mean feature (shared memory, 64 floats) and fp16 scale (sigma, 2 / sigma^2; NaN = unusable cloud).
// Every CTA of the prep kernel does this redundantly (1.5 K floats out of L2) in the same order: same values everywhere.
__device__ __forceinline__ void knn2_fold_center(const float* __restrict__ part, int b, int N, float* mus, float* ssc, float* red) {
    const int t = threadIdx.x;
    if (t < 64) {
        const float* pb = part + (size_t)b * K2_CSPLIT * 196;
        float s = 0.f, lo = INFINITY, hi = -INFINITY, bad = 0.f;
#pragma unroll
        for (int sp = 0; sp < K2_CSPLIT; ++sp) {
            s += pb[sp * 196 + t];
            lo = fminf(lo, pb[sp * 196 + 64 + t]);
            hi = fmaxf(hi, pb[sp * 196 + 128 + t]);
            bad += pb[sp * 196 + 192];
        }
        const float m = s * (1.f / (float)N);
        mus[t] = m;
        float g = fmaxf(hi - m, m - lo);
        if (bad != 0.f || !(g <= 3.0e38f)) g = INFINITY;
        red[t] = g;
    }
    __syncthreads();
    if (t == 0) {
        float g = 0.f;
        for (int c = 0; c < 64; ++c) g = fmaxf(g, red[c]);
        float sigma = 1.f, c2 = 2.f;
        if (g > 0.f) {
            int e;
            frexpf(g, &e);             // g = f * 2^e, f in [0.5, 1)
            const int se = 8 - e;      // g * 2^se in [2^7, 2^8): the gram entries and sigma^2 nrm / 2 stay below 2^22
            if (!(g <= 3.0e38f) || se > 60 || se < -60) {
                sigma = 1.f; c2 = __int_as_float(0x7fc00000);   // NaN: nothing is collected, every tile falls back
            } else {
                sigma = ldexpf(1.f, se);
                c2 = ldexpf(2.f, -2 * se);
            }
        }
        ssc[0] = sigma; ssc[1] = c2;
    }
    __syncthreads();
}

// 0b. per point: fp16 centred operand row, both norms, per-cloud maxima.  One thread = one point (the canonical norm is a
// sequential fmaf chain), but the 256-byte input rows and the 128-byte output rows of a block travel through shared memory so that
// global memory only sees coalesced 16-byte accesses (a thread walking its own row touched 32 different lines per load instruction:
// 0.043 ms for 100 MB).
constexpr int K2_PREP_XS = 68;                         // staged input row stride in floats (conflict-free LDS.128 per thread)
constexpr int K2_PREP_HS = 9;                          // staged output row stride in uint4
constexpr size_t K2_PREP_SMEM = 256 * K2_PREP_XS * 4 + 256 * K2_PREP_HS * 16;
__global__ void __launch_bounds__(256)
knn2_prep_kernel(const float* __restrict__ x, const float* __restrict__ part, float* __restrict__ sc, int N, int Npad,
                 __half* __restrict__ xh, uint4* __restrict__ ext, float* __restrict__ xxpad, float* __restrict__ nrmpad,
                 float* __restrict__ snpad, float* __restrict__ r2, float* __restrict__ r2c) {
    __shared__ __align__(16) float mus_f[64];
    __shared__ float ssc[2], sred[64];
    extern __shared__ __align__(16) uint8_t prep_sm[];
    float* xs = reinterpret_cast<float*>(prep_sm);                               // [256][K2_PREP_XS]
    uint4* hs = reinterpret_cast<uint4*>(prep_sm + 256 * K2_PREP_XS * 4);        // [256][K2_PREP_HS], row = storage position
    const int b = blockIdx.y;
    const int n0 = blockIdx.x * 256;
    // the block's input rows, coalesced (in flight while the centre is folded)
    {
        const float4* src = reinterpret_cast<const float4*>(x + ((size_t)b * N + n0) * 64);
        const int rows = min(256, N - n0);
#pragma unroll 4
        for (int i = threadIdx.x; i < rows * 16; i += 256)
            *reinterpret_cast<float4*>(xs + (i >> 4) * K2_PREP_XS + (i & 15) * 4) = __ldg(src + i);
    }
    knn2_fold_center(part, b, N, mus_f, ssc, sred);                               // (ends with __syncthreads)
    const float4* mus = reinterpret_cast<const float4*>(mus_f);
    const float sigma = ssc[0];
    if (blockIdx.x == 0 && threadIdx.x == 0) { sc[2 * b] = sigma; sc[2 * b + 1] = ssc[1]; }
    const int n = n0 + threadIdx.x;
    float vxx = INFINITY, vn = INFINITY;
    int np = n;                                   // storage position of point n (scrambled inside full 64-blocks)
    if ((n | 63) < N) {
        int a, bb;
        block_perm(n >> 6, a, bb);
        np = (n & ~63) | (((n & 63) * a + bb) & 63);
    }
    if (n < N) {
        const float4* p = reinterpret_cast<const float4*>(xs + threadIdx.x * K2_PREP_XS);
        uint4* o = hs + (np - n0) * K2_PREP_HS;
        float acc = 0.f, accc = 0.f;
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            const float4 t0 = p[2 * g], t1 = p[2 * g + 1];
            acc = __fmaf_rn(t0.x, t0.x, acc); acc = __fmaf_rn(t0.y, t0.y, acc);
            acc = __fmaf_rn(t0.z, t0.z, acc); acc = __fmaf_rn(t0.w, t0.w, acc);
            acc = __fmaf_rn(t1.x, t1.x, acc); acc = __fmaf_rn(t1.y, t1.y, acc);
            acc = __fmaf_rn(t1.z, t1.z, acc); acc = __fmaf_rn(t1.w, t1.w, acc);
            const float4 m0 = mus[2 * g], m1 = mus[2 * g + 1];
            float c[8] = {t0.x - m0.x, t0.y - m0.y, t0.z - m0.z, t0.w - m0.w, t1.x - m1.x, t1.y - m1.y, t1.z - m1.z, t1.w - m1.w};
#pragma unroll
            for (int q = 0; q < 8; ++q) accc = __fmaf_rn(c[q], c[q], accc);
            uint32_t pk[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const __half2 h = __floats2half2_rn(c[2 * q] * sigma, c[2 * q + 1] * sigma);
                pk[q] = *reinterpret_cast<const uint32_t*>(&h);
            }
            o[g] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
        vxx = acc; vn = accc;
        atomicMax(reinterpret_cast<int*>(r2 + b), __float_as_int(acc));     // >= 0 (or NaN bits, harmless): int order == float order
        atomicMax(reinterpret_cast<int*>(r2c + b), __float_as_int(accc));
    }
    __syncthreads();
    {   // the block's operand rows in storage order, coalesced
        uint4* dst = reinterpret_cast<uint4*>(xh + ((size_t)b * N + n0) * 64);
        const int rows = min(256, N - n0);
#pragma unroll 4
        for (int i = threadIdx.x; i < rows * 8; i += 256) dst[i] = hs[(i >> 3) * K2_PREP_HS + (i & 7)];
    }
    // K-extension row of the candidate operand: the tensor core itself subtracts V = sigma^2 nrm / 2 from the gram entry,
    //   t_ij = sigma^2 x'_i.x'_j - V_j = (sigma^2 / 2) a_ij,   V = 2^6 B1 + 2^-5 B2 + 2^-14 B3  (three fp16 pieces, residual
    //   < 2^-15), against the constant query-side row [2^6, 2^-5, 2^-14, 2^15, 0...]; slot 3 pushes padded candidates to -2e9.
    {
        float b1 = 0.f, b2 = 0.f, b3 = 0.f, b4 = -60000.f;
        if (n < N) {
            const float V = 0.5f * (sigma * sigma) * vn;
            b1 = __half2float(__float2half_rn(V * 0.015625f));
            const float r1 = __fmaf_rn(-b1, 64.f, V);
            b2 = __half2float(__float2half_rn(r1 * 32.f));
            const float rr = __fmaf_rn(-b2, 0.03125f, r1);
            b3 = __half2float(__float2half_rn(rr * 16384.f));
            b4 = 0.f;
        }
        const __half2 h01 = __floats2half2_rn(-b1, -b2), h23 = __floats2half2_rn(-b3, b4);
        // no-swizzle K-major core-matrix layout of one 64-candidate tile (2 KB): 8-row groups 256 B apart, the two 8-column
        // core matrices of a group 128 B apart, 16 B per row inside a core matrix
        const int r = np & 63;
        uint4* e = ext + ((size_t)b * (Npad >> 6) + (np >> 6)) * 128 + (r >> 3) * 16 + (r & 7);
        e[0] = make_uint4(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23), 0u, 0u);
        e[8] = make_uint4(0u, 0u, 0u, 0u);
    }
    xxpad[(size_t)b * Npad + n] = vxx;            // canonical norms stay in point order (refine kernel)
    nrmpad[(size_t)b * Npad + np] = vn;           // centred norms follow the operand rows
    snpad[(size_t)b * Npad + np] = n < N ? sqrtf(vn) : 0.f;
}

// ---------------------------------------------------------------------------------------------------------------------
// in-register sorting networks over 32 values (all indices compile-time after unrolling)
__device__ __forceinline__ void cex_desc(float& a, float& b) {   // a >= b afterwards
    const float hi = fmaxf(a, b), lo = fminf(a, b);
    a = hi; b = lo;
}
__device__ __forceinline__ void bitonic_merge32_desc(float (&v)[32]) {
#pragma unroll
    for (int stride = 16; stride > 0; stride >>= 1) {
#pragma unroll
        for (int i = 0; i < 32; ++i)
            if ((i & stride) == 0) cex_desc(v[i], v[i | stride]);
    }
}
__device__ __forceinline__ void bitonic_sort32_desc(float (&v)[32]) {
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if ((i & stride) == 0) {
                    const bool desc = ((i & size) == 0) || (size == 32);
                    if (desc) cex_desc(v[i], v[i | stride]); else cex_desc(v[i | stride], v[i]);
                }
            }
        }
    }
}

// K-major operand WITHOUT swizzle (the 16-column K-extension): core matrices of 8 rows x 16 B, the two core matrices of
// a row group 128 B apart (leading byte offset), row groups 256 B apart (stride byte offset)
__device__ __forceinline__ uint64_t make_smem_desc_ext(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)(128 >> 4) << 16;
    d |= (uint64_t)(256 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    return d;                                              // layout type 0 = no swizzle
}
// two 32-column TMEM loads (columns c .. c+31 and c+64 .. c+95) in flight, one wait
__device__ __forceinline__ void tc_ld32x2(uint32_t taddr, uint32_t (&a)[32], uint32_t (&b)[32]) {
#define LPD_LD32(R, ADDR)                                                                                               \
    asm volatile(                                                                                                       \
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                       \
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                                       \
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                       \
        : "=r"(R[0]), "=r"(R[1]), "=r"(R[2]), "=r"(R[3]), "=r"(R[4]), "=r"(R[5]), "=r"(R[6]), "=r"(R[7]),              \
          "=r"(R[8]), "=r"(R[9]), "=r"(R[10]), "=r"(R[11]), "=r"(R[12]), "=r"(R[13]), "=r"(R[14]), "=r"(R[15]),        \
          "=r"(R[16]), "=r"(R[17]), "=r"(R[18]), "=r"(R[19]), "=r"(R[20]), "=r"(R[21]), "=r"(R[22]), "=r"(R[23]),      \
          "=r"(R[24]), "=r"(R[25]), "=r"(R[26]), "=r"(R[27]), "=r"(R[28]), "=r"(R[29]), "=r"(R[30]), "=r"(R[31])       \
        : "r"(ADDR))
    LPD_LD32(a, taddr);
    LPD_LD32(b, taddr + 64);
#undef LPD_LD32
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// order-preserving float -> signed int key (for the integer warp reductions); NaN maps above +inf
__device__ __forceinline__ int fkey(float v) {
    const int b = __float_as_int(v);
    return b ^ ((b >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

template <int MT, bool TS = false>
struct K2Smem {
    static constexpr int SCAN_THREADS = 256 * MT;
    static constexpr int TSTAGES = TS ? 3 : K2_TCOLS / (K2_C * MT);   // TS: columns 384.. hold the two query buffers
    static constexpr int EXS = SCAN_THREADS + 1;          // exchange-buffer row stride (words)
    static constexpr uint32_t A_TILE = 128 * 128;         // one 128-row query tile: 64 fp16 = 128 B per row
    static constexpr uint32_t A_BYTES = MT * A_TILE;
    static constexpr uint32_t B_BYTES = K2_C * 128;
    static constexpr uint32_t BX_BYTES = K2_C * 32;       // K-extension of a candidate tile
    static constexpr size_t off_b = TS ? 0 : 2 * A_BYTES; // two query buffers (next item prefetched); none in TS mode
    static constexpr size_t off_bx = off_b + K2_BSTAGES * B_BYTES;
    static constexpr size_t off_ax = off_bx + K2_BSTAGES * BX_BYTES;         // constant query-side extension, 128 rows
    static constexpr size_t off_xs = off_ax + 128 * 32;
    static constexpr size_t off_ex = off_xs + K2_XSLOTS * K2_C * 4;          // per slot: 64 root norms (TIGHT only)
    static constexpr size_t off_tbl = off_ex + (size_t)32 * EXS * 4;        // [scan warp][K2_TBL] pass-1 tile margins
    static constexpr size_t off_bar = (off_tbl + (size_t)8 * MT * K2_TBL * 4 + 7) / 8 * 8;
    static constexpr size_t total = off_bar + (4 + 2 * K2_BSTAGES + 2 * TSTAGES) * 8 + 16;
    static_assert(total <= 227 * 1024, "knn2 shared memory budget");
};

template <int MT, int CAP, bool TIGHT, bool TS>
__global__ void __launch_bounds__(256 * MT + 64, 1)
knn2_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, Knn2Params P) {
    static_assert(!TS || MT == 1, "TS mode: one 128-row query tile per item");
    using S = K2Smem<MT, TS>;
    constexpr int SCAN_WARPS = 8 * MT;
    constexpr uint32_t ACOL = 384;                       // TS: TMEM column of query buffer 0 (buffer 1 at + 64)
    constexpr int TCOLS = K2_C * MT;                       // TMEM columns per accumulator stage
    constexpr int K2_TSTAGES = S::TSTAGES;
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* a_s = smem;
    uint8_t* b_s = smem + S::off_b;
    uint8_t* bx_s = smem + S::off_bx;
    uint8_t* ax_s = smem + S::off_ax;
    float* xs = reinterpret_cast<float*>(smem + S::off_xs);
    float* ex = reinterpret_cast<float*>(smem + S::off_ex);
    int* tbl = reinterpret_cast<int*>(smem + S::off_tbl);
    uint64_t* afull = reinterpret_cast<uint64_t*>(smem + S::off_bar);   // [2]
    uint64_t* aempty = afull + 2;                                       // [2]
    uint64_t* bfull = aempty + 2;
    uint64_t* bempty = bfull + K2_BSTAGES;
    uint64_t* tfull = bempty + K2_BSTAGES;
    uint64_t* tempty = tfull + K2_TSTAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + K2_TSTAGES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int items = P.B * P.qtiles;
    const int nstages = 2 * P.ctiles;                      // per item: the candidate tiles twice
    const int full_blocks = P.N >> 6;                      // 64-blocks below this one are stored scrambled

    if (threadIdx.x < 128) {
        // constant query-side K-extension [2^6, 2^-5, 2^-14, 2^15, 0 ...] in the no-swizzle core-matrix layout
        const int r = threadIdx.x;
        const __half2 h01 = __floats2half2_rn(64.f, 0.03125f), h23 = __floats2half2_rn(6.103515625e-05f, 32768.f);
        uint4* e = reinterpret_cast<uint4*>(ax_s) + (r >> 3) * 16 + (r & 7);
        e[0] = make_uint4(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23), 0u, 0u);
        e[8] = make_uint4(0u, 0u, 0u, 0u);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core (async proxy) reads
    }
    if (warp == SCAN_WARPS + 1) {
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_a)) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap_b)) : "memory");
            for (int s = 0; s < 2; ++s) { mbar_init(&afull[s], TS ? SCAN_WARPS : 1); mbar_init(&aempty[s], 1); }
            for (int s = 0; s < K2_BSTAGES; ++s) { mbar_init(&bfull[s], 1); mbar_init(&bempty[s], 1); }
            for (int s = 0; s < K2_TSTAGES; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], SCAN_WARPS); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TS ? 512 : TCOLS * K2_TSTAGES) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == SCAN_WARPS) {
        // ------------------------------ TMA producer (whole warp, lane 0 issues) ------------------------------
        {
            const uint32_t leader = lane == 0;
            uint32_t tcount = 0, icount = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x, ++icount) {
                const int b = item / P.qtiles, q0 = (item % P.qtiles) * (128 * MT);
                const uint32_t ab = icount & 1, aph = (icount >> 1) & 1;
                if (!TS) {
                    mbar_wait_sleep(&aempty[ab], aph ^ 1);
                    mbar_expect_tx_p(&afull[ab], S::A_BYTES, leader);
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt)
                        tma_load_2d_p(a_s + ab * S::A_BYTES + mt * S::A_TILE, &tmap_a, &afull[ab], 0, b * P.N + q0 + mt * 128, leader);
                }
                const uint4* extb = P.ext + (size_t)b * (P.Npad >> 6) * 128;
                const float* snb = P.snpad + (size_t)b * P.Npad;
                uint32_t s = tcount % K2_BSTAGES, ph = (tcount / K2_BSTAGES) & 1, xsl = tcount % K2_XSLOTS;
                for (int cs = 0; cs < nstages; ++cs, ++tcount) {
                    const int ct = cs >= P.ctiles ? cs - P.ctiles : cs;
                    mbar_wait_sleep(&bempty[s], ph ^ 1);
                    mbar_expect_tx_p(&bfull[s], S::B_BYTES + S::BX_BYTES + (TIGHT ? K2_C * 4 : 0), leader);
                    tma_load_2d_p(b_s + s * S::B_BYTES, &tmap_b, &bfull[s], 0, b * P.N + ct * K2_C, leader);
                    bulk_load_p(bx_s + s * S::BX_BYTES, extb + (size_t)ct * 256, S::BX_BYTES, &bfull[s], leader);
                    if (TIGHT) bulk_load_p(xs + xsl * K2_C, snb + ct * K2_C, K2_C * 4, &bfull[s], leader);
                    if (++s == K2_BSTAGES) { s = 0; ph ^= 1; }
                    xsl = (xsl + 1) % K2_XSLOTS;
                }
            }
        }
    } else if (warp == SCAN_WARPS + 1) {
        // ------------------------------ MMA issuer (whole warp, lane 0 issues) ------------------------------
        {
            constexpr uint32_t idesc = make_idesc_f16(128, K2_C);
            const uint32_t leader = lane == 0;
            const uint64_t dax = make_smem_desc_ext(smem_u32(ax_s));
            uint32_t tcount = 0, icount = 0;
            for (int item = blockIdx.x; item < items; item += gridDim.x, ++icount) {
                const uint32_t ab = icount & 1, aph = (icount >> 1) & 1;
                mbar_wait_sleep(&afull[ab], aph);
                if (TS) tc_fence_after();
                const uint64_t da0 = make_smem_desc(smem_u32(a_s + ab * S::A_BYTES));
                const uint32_t ta0 = tmem_base + ACOL + ab * 64;        // TS: query rows in tensor memory
                uint32_t s = tcount % K2_BSTAGES, ph = (tcount / K2_BSTAGES) & 1;
                uint32_t ts = tcount % K2_TSTAGES, tph = (tcount / K2_TSTAGES) & 1;
                for (int cs = 0; cs < nstages; ++cs, ++tcount) {
                    mbar_wait(&tempty[ts], tph ^ 1);      // spin: __nanosleep wakes far too late for a 300-cycle stage
                    mbar_wait(&bfull[s], ph);
                    tc_fence_after();
                    const uint64_t db = make_smem_desc(smem_u32(b_s + s * S::B_BYTES));
                    const uint64_t dbx = make_smem_desc_ext(smem_u32(bx_s + s * S::BX_BYTES));
                    if (TS) {                               // A from tensor memory: 8 columns (16 fp16) per K step, extension at + 32
                        const uint32_t d = tmem_base + ts * TCOLS;
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) tc_mma_f16_ts(d, ta0 + ks * 8, db + (uint64_t)(ks * 2), idesc, ks ? 1u : 0u);
                        tc_mma_f16_ts(d, ta0 + 32, dbx, idesc, 1u);
                    } else {
                        // K = 64 = 4 x 16 (32 bytes per step inside the 128-byte swizzle atom) + the K-extension, which subtracts
                        // sigma^2 nrm_j / 2 and buries the padding; the query tiles of an item alternate (independent accumulators)
#pragma unroll
                        for (int ks = 0; ks < 5; ++ks) {
#pragma unroll
                            for (int mt = 0; mt < MT; ++mt) {
                                const uint64_t da = da0 + (uint64_t)(mt * (S::A_TILE >> 4));
                                const uint32_t d = tmem_base + ts * TCOLS + mt * K2_C;
                                if (ks < 4) tc_mma_f16_p(d, da + (uint64_t)(ks * 2), db + (uint64_t)(ks * 2), idesc, ks ? 1u : 0u, leader);
                                else tc_mma_f16_p(d, dax, dbx, idesc, 1u, leader);
                            }
                        }
                    }
                    tc_commit_p(&bempty[s], leader);
                    tc_commit_p(&tfull[ts], leader);
                    if (++s == K2_BSTAGES) { s = 0; ph ^= 1; }
                    if (++ts == K2_TSTAGES) { ts = 0; tph ^= 1; }
                }
                tc_commit_p(&aempty[ab], leader);   // all MMAs that read this query buffer have completed when this arrives
            }
        }
    } else {
        // ------------------------------ scan: one (stored query row, column half) per thread ------------------------------
        // all scores below are t = (sigma^2 / 2) a: the power-of-two factor commutes with every comparison
        const int quad = warp & 3, half = (warp >> 2) & 1, mt = warp >> 3;
        const int own = mt * 256 + half * 128 + quad * 32 + lane;
        const int partner = own ^ 128;
        // this thread's 64 columns: positions [32 half, 32 half + 32) of BOTH 64-blocks of a stage, so that group j of the thread
        // is "storage position 32 half + j of every block" (64 distinct groups per row for the 64 points of any one block)
        const uint32_t tm_lane = ((uint32_t)(quad * 32) << 16) + mt * K2_C + half * 32;
        uint32_t tcount = 0, icount = 0;
        // TS mode: the scan threads themselves put the query tile into tensor memory (each thread its own row: half 0 the
        // 32-bit columns 0..19, half 1 the columns 20..31 + the constant K-extension 32..39), one item ahead of the MMAs
        uint4 aw[5];
        auto load_a = [&](int it2) {
            const int b2 = it2 / P.qtiles, q02 = (it2 % P.qtiles) * 128;
            const long long grow = (long long)b2 * P.N + q02 + quad * 32 + lane;
            const bool inb = grow < (long long)P.B * P.N;
            const uint4* src = P.xh + grow * 8;
            const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
            if (half == 0) {
#pragma unroll
                for (int i = 0; i < 5; ++i) aw[i] = inb ? __ldg(src + i) : zero;
            } else {
#pragma unroll
                for (int i = 0; i < 3; ++i) aw[i] = inb ? __ldg(src + 5 + i) : zero;
                const __half2 h01 = __floats2half2_rn(64.f, 0.03125f), h23 = __floats2half2_rn(6.103515625e-05f, 32768.f);
                aw[3] = make_uint4(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23), 0u, 0u);
                aw[4] = zero;
            }
        };
        auto store_a = [&](uint32_t n) {                               // n = ordinal of the item inside this CTA
            const uint32_t buf = n & 1, use = n >> 1;
            mbar_wait(&aempty[buf], (use & 1) ^ 1);                    // the MMAs of item n - 2 have finished with this buffer
            const uint32_t ta = tmem_base + ((uint32_t)(quad * 32) << 16) + ACOL + buf * 64 + half * 20;
#pragma unroll
            for (int i = 0; i < 5; ++i) tc_st4(ta + 4 * i, aw[i]);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&afull[buf]);
        };
        if (TS && blockIdx.x < items) { load_a(blockIdx.x); store_a(0); }
        for (int item = blockIdx.x; item < items; item += gridDim.x, ++icount) {
            const int b = item / P.qtiles, q0 = (item % P.qtiles) * (128 * MT);
            const bool have_next = TS && item + (int)gridDim.x < items;
            if (have_next) load_a(item + gridDim.x);                   // in flight during pass 1
            const int srow = q0 + mt * 128 + quad * 32 + lane;        // storage position of this thread's query
            int row = srow;                                            // ... and the point it holds
            if ((srow >> 6) < full_blocks) {
                int a, bb;
                block_perm(srow >> 6, a, bb);
                row = (srow & ~63) | ((((srow & 63) - bb) * inv_mod64(a)) & 63);
            }
            const bool live = srow < P.N;                              // (srow < N  <=>  row < N)
            const float inv_cb = 1.f / __ldg(P.sc + 2 * b + 1);        // sigma^2 / 2, a power of two (NaN: unusable cloud)
            float ni = 0.f, cni = 0.f, gself = 0.f;
            if (live) {
                const float ni2 = __ldg(P.nrmpad + (size_t)b * P.Npad + srow);
                ni = sqrtf(ni2); cni = 2.5e-3f * ni * inv_cb;
                gself = ni2 * inv_cb;                                  // ~ the row's own score t_ii: normalises the skip table
            }
            const bool use_tbl = P.ctiles <= K2_TBL;
            int* wtbl = tbl + warp * K2_TBL;
            const float ub_extra = TIGHT ? cni * sqrtf(__ldg(P.r2c + b)) : 0.f;   // TIGHT: upper bound of cni * sn_j
            // ---------------- pass 1: running maximum of every column position (mod 32) ----------------
            float m[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) m[j] = -INFINITY;
            for (int cs = 0; cs < P.ctiles; ++cs, ++tcount) {
                const uint32_t ts = tcount % K2_TSTAGES, tph = (tcount / K2_TSTAGES) & 1;
                mbar_wait(&tfull[ts], tph);
                tc_fence_after();
                uint32_t r0[32], r1[32];
                tc_ld32x2(tmem_base + tm_lane + ts * TCOLS, r0, r1);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[ts]);
                float tm = -INFINITY;                                               // best raw score of the row in this block
                if (TIGHT) {                                                        // certified lower bounds
                    const float* xsj = xs + (tcount % K2_XSLOTS) * K2_C + half * 32;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 s0 = *reinterpret_cast<const float4*>(xsj + j), s1 = *reinterpret_cast<const float4*>(xsj + 64 + j);
                        m[j + 0] = fmax3(m[j + 0], fmaf(-cni, s0.x, __uint_as_float(r0[j + 0])), fmaf(-cni, s1.x, __uint_as_float(r1[j + 0])));
                        m[j + 1] = fmax3(m[j + 1], fmaf(-cni, s0.y, __uint_as_float(r0[j + 1])), fmaf(-cni, s1.y, __uint_as_float(r1[j + 1])));
                        m[j + 2] = fmax3(m[j + 2], fmaf(-cni, s0.z, __uint_as_float(r0[j + 2])), fmaf(-cni, s1.z, __uint_as_float(r1[j + 2])));
                        m[j + 3] = fmax3(m[j + 3], fmaf(-cni, s0.w, __uint_as_float(r0[j + 3])), fmaf(-cni, s1.w, __uint_as_float(r1[j + 3])));
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) m[j] = fmax3(m[j], __uint_as_float(r0[j]), __uint_as_float(r1[j]));
                }
                if (use_tbl) {
                    // skip table: D(warp, block) = min over the warp's rows of (t_ii - best score of the row in this block).  Pass 2
                    // reads the block only if D <= max over the rows of (t_ii - threshold): any per-row constant keeps the
                    // test exact-or-conservative, t_ii makes it tight (it removes the norm of the row from both sides).
#pragma unroll
                    for (int j = 0; j < 32; ++j) tm = fmax3(tm, __uint_as_float(r0[j]), __uint_as_float(r1[j]));
                    const float D = live ? gself - (tm + ub_extra) : INFINITY;
                    const int dk = __reduce_min_sync(kFull, fkey(D));
                    if (lane == 0) wtbl[cs] = dk;
                }
            }
            // ---------------- k-th largest of the row's 64 group maxima ----------------
            bitonic_sort32_desc(m);
#pragma unroll
            for (int j = 0; j < 32; ++j) ex[j * S::EXS + own] = m[j];
            named_bar(1, S::SCAN_THREADS);
#pragma unroll
            for (int j = 0; j < 32; ++j) m[j] = fmaxf(m[j], ex[(31 - j) * S::EXS + partner]);   // 32 largest of the union (bitonic)
            named_bar(2, S::SCAN_THREADS);                                                      // ex may be rewritten (next item)
            bitonic_merge32_desc(m);
            float tau0 = m[0];
#pragma unroll
            for (int j = 1; j < 32; ++j) tau0 = (j == P.k - 1) ? m[j] : tau0;
            float thr = INFINITY;
            if (live) {
                const float xxi = __ldg(P.xxpad + (size_t)b * P.Npad + row);
                const float r2 = __ldg(P.r2 + b), r2c = __ldg(P.r2c + b), sigma = __ldg(P.sc + 2 * b);
                const float rc = sqrtf(r2c);
                float eps = (1.9e-6f / sigma) * (ni + rc) + 7.62939453125e-6f * (xxi + r2) + 3.814697265625e-6f * r2c;
                if (!TIGHT) eps += 2.5e-3f * ni * rc;
                thr = fmaxf(tau0 - 2.f * eps * inv_cb, -1.0e9f);             // padded candidates sit near -2e9
                if (!(eps * inv_cb < INFINITY)) thr = __int_as_float(0x7fc00000);   // unusable bound: collect nothing, fall back
            }
            if (have_next) store_a(icount + 1);
            // ---------------- pass 2: collect everything at or above the threshold ----------------
            const int dthr = __reduce_max_sync(kFull, fkey(live ? gself - thr : -INFINITY));
            int cnt = 0;
            int* mine = P.cand + (((size_t)b * P.N + (live ? row : 0)) * 2 + half) * CAP;
            for (int cs = 0; cs < P.ctiles; ++cs, ++tcount) {
                const uint32_t ts = tcount % K2_TSTAGES, tph = (tcount / K2_TSTAGES) & 1;
                mbar_wait(&tfull[ts], tph);
                if (use_tbl && wtbl[cs] > dthr) {     // warp-uniform: no row of this warp has a candidate here
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tempty[ts]);           // (after tfull: the arrival must land in this use's phase)
                    continue;
                }
                tc_fence_after();
                uint32_t r0[32], r1[32];
                tc_ld32x2(tmem_base + tm_lane + ts * TCOLS, r0, r1);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[ts]);
                float u0[32], u1[32];
                if (TIGHT) {                                                       // upper bounds
                    const float* xsj = xs + (tcount % K2_XSLOTS) * K2_C + half * 32;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 s0 = *reinterpret_cast<const float4*>(xsj + j), s1 = *reinterpret_cast<const float4*>(xsj + 64 + j);
                        u0[j + 0] = fmaf(cni, s0.x, __uint_as_float(r0[j + 0])); u1[j + 0] = fmaf(cni, s1.x, __uint_as_float(r1[j + 0]));
                        u0[j + 1] = fmaf(cni, s0.y, __uint_as_float(r0[j + 1])); u1[j + 1] = fmaf(cni, s1.y, __uint_as_float(r1[j + 1]));
                        u0[j + 2] = fmaf(cni, s0.z, __uint_as_float(r0[j + 2])); u1[j + 2] = fmaf(cni, s1.z, __uint_as_float(r1[j + 2]));
                        u0[j + 3] = fmaf(cni, s0.w, __uint_as_float(r0[j + 3])); u1[j + 3] = fmaf(cni, s1.w, __uint_as_float(r1[j + 3]));
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) { u0[j] = __uint_as_float(r0[j]); u1[j] = __uint_as_float(r1[j]); }
                }
                // cheap test first: even among the blocks the table lets through, most rows have no candidate
                float mx = -INFINITY;
#pragma unroll
                for (int j = 0; j < 32; ++j) mx = fmax3(mx, u0[j], u1[j]);
                if (__any_sync(kFull, mx >= thr)) {
                    uint32_t mask0 = 0, mask1 = 0;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        mask0 |= (u0[j] >= thr) ? (1u << j) : 0u;
                        mask1 |= (u1[j] >= thr) ? (1u << j) : 0u;
                    }
                    // undo the scrambling of the two blocks of the stage: c = (pos - b) a^-1
                    int pa0 = 1, pb0 = 0, pa1 = 1, pb1 = 0;
                    if (2 * cs < full_blocks) { block_perm(2 * cs, pa0, pb0); pa0 = inv_mod64(pa0); }
                    if (2 * cs + 1 < full_blocks) { block_perm(2 * cs + 1, pa1, pb1); pa1 = inv_mod64(pa1); }
                    const int jbase = cs * K2_C, pos0 = half * 32;
                    while (mask0) {
                        const int j = __ffs(mask0) - 1;
                        mask0 &= mask0 - 1;
                        if (cnt < CAP) mine[cnt] = jbase + (((pos0 + j - pb0) * pa0) & 63);
                        ++cnt;
                    }
                    while (mask1) {
                        const int j = __ffs(mask1) - 1;
                        mask1 &= mask1 - 1;
                        if (cnt < CAP) mine[cnt] = jbase + 64 + (((pos0 + j - pb1) * pa1) & 63);
                        ++cnt;
                    }
                }
            }
            if (live) P.cnt[((size_t)b * P.N + row) * 2 + half] = cnt;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == SCAN_WARPS + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TS ? 512 : TCOLS * K2_TSTAGES) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// 2. one warp per query row: canonical re-score of the collected candidates, rank, write the first k
// The candidate rows are fetched COOPERATIVELY (coalesced: a quarter-warp reads 128 contiguous bytes of one candidate with
// LDG.128) into a padded shared-memory tile, half a row (32 channels) at a time, and each lane then continues the canonical
// fmaf chain of its own candidate out of shared memory (row stride 36 floats: the quarter-warp phases of LDS.128 / STS.128
// hit distinct banks).  A lane-per-candidate gather straight from global memory costs up to 32 L1 wavefronts per load
// instruction and ran at 90 % of the L1 wavefront peak.  The final order is a rank count over 64-bit keys
// (orderable(pd) << 32 | ~index: larger = better), two keys per LDS.128.
// a row that cannot be finished here flags its 64-row tile (once) and appends it to the work list of the exact kernel
__device__ __forceinline__ void knn2_flag_tile(int* __restrict__ flags, int* __restrict__ list, int tile) {
    if (atomicExch(flags + tile, 1) == 0) list[1 + atomicAdd(list, 1)] = tile;
}
constexpr int RF_STRIDE = 36;
constexpr int RF_WARPS = 8;
template <int CAP>
struct RefineSmem {
    static constexpr int KEYS = 2 * CAP + 2;      // + zero padding for the two-at-a-time rank loop
    static constexpr size_t rows = (size_t)RF_WARPS * 32 * RF_STRIDE * 4;
    static constexpr size_t off_xi = rows;
    static constexpr size_t off_key = off_xi + (size_t)RF_WARPS * 64 * 4;
    static constexpr size_t off_id = off_key + (size_t)RF_WARPS * KEYS * 8;
    static constexpr size_t total = off_id + (size_t)RF_WARPS * 2 * CAP * 4;
};

template <int CAP>
__global__ void __launch_bounds__(RF_WARPS * 32)
knn2_refine_kernel(const float* __restrict__ x, const float* __restrict__ xxpad, const int* __restrict__ cnt,
                   const int* __restrict__ cand, int B, int N, int Npad, int k, void* __restrict__ idx_out, int idx_i64,
                   int* __restrict__ flags, int* __restrict__ list) {
    using S = RefineSmem<CAP>;
    extern __shared__ __align__(16) uint8_t rsm[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float* s_rows = reinterpret_cast<float*>(rsm) + (size_t)w * 32 * RF_STRIDE;
    float* s_xi = reinterpret_cast<float*>(rsm + S::off_xi) + w * 64;
    unsigned long long* s_key = reinterpret_cast<unsigned long long*>(rsm + S::off_key) + w * S::KEYS;
    int* s_id = reinterpret_cast<int*>(rsm + S::off_id) + w * 2 * CAP;
    const long long grow = (long long)blockIdx.x * RF_WARPS + w;
    if (grow >= (long long)B * N) return;
    const int b = (int)(grow / N), qi = (int)(grow % N);
    const int c0 = __ldg(cnt + grow * 2), c1 = __ldg(cnt + grow * 2 + 1);
    const int total = c0 + c1;
    if (c0 > CAP || c1 > CAP || total < k) {      // overflow / unusable bound: the exact kernel recomputes the 64-row tile
        if (lane == 0) knn2_flag_tile(flags, list, b * ((N + 63) / 64) + qi / 64);
        return;
    }
    const float* xb = x + (size_t)b * N * 64;
    reinterpret_cast<float2*>(s_xi)[lane] = __ldg(reinterpret_cast<const float2*>(xb + (size_t)qi * 64) + lane);
    const float xxi = __ldg(xxpad + (size_t)b * Npad + qi);
    const int* l0 = cand + (size_t)grow * 2 * CAP;
    for (int s = lane; s < total; s += 32) s_id[s] = s < c0 ? __ldg(l0 + s) : __ldg(l0 + CAP + (s - c0));
    if (lane < 2) s_key[total + lane] = 0ull;     // padding keys: better than nothing
    __syncwarp();
    const int qw = lane >> 3, ql = lane & 7;      // quarter-warp and lane inside it: a quarter-warp moves 32 channels of one candidate
    for (int base = 0; base < total; base += 32) {
        const int nc = min(32, total - base);
        const int myid = lane < nc ? s_id[base + lane] : 0;
        float dot = 0.f;
#pragma unroll
        for (int ph = 0; ph < 2; ++ph) {
            __syncwarp();                         // the previous tile has been consumed
            for (int c = qw; c < nc; c += 4) {
                const int j = s_id[base + c];
                const float4 v = __ldg(reinterpret_cast<const float4*>(xb + (size_t)j * 64 + ph * 32) + ql);
                *reinterpret_cast<float4*>(s_rows + c * RF_STRIDE + ql * 4) = v;
            }
            __syncwarp();
            if (lane < nc) {
                const float4* rj = reinterpret_cast<const float4*>(s_rows + lane * RF_STRIDE);
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                    const float4 u = reinterpret_cast<const float4*>(s_xi)[ph * 8 + g], v = rj[g];
                    dot = __fmaf_rn(u.x, v.x, dot); dot = __fmaf_rn(u.y, v.y, dot);
                    dot = __fmaf_rn(u.z, v.z, dot); dot = __fmaf_rn(u.w, v.w, dot);
                }
            }
        }
        if (lane < nc) {
            const float xxj = __ldg(xxpad + (size_t)b * Npad + myid);
            const float t = -2.0f * dot;
            const float pd = __fadd_rn(__fsub_rn(__fsub_rn(-xxj, t), xxi), 0.0f);   // (+ 0: -0.0 and +0.0 must share one key)
            uint32_t u = __float_as_uint(pd);
            u ^= (u >> 31) ? 0xffffffffu : 0x80000000u;                  // monotone float -> uint
            s_key[base + lane] = ((unsigned long long)u << 32) | (uint32_t)(~myid);
        }
    }
    __syncwarp();
    const size_t o = (size_t)grow * k;
    const int npairs = (total + 1) >> 1;
    for (int base = 0; base < total; base += 32) {
        const int s = base + lane;
        const unsigned long long mine = s < total ? s_key[s] : ~0ull;
        int rank = 0;
        const ulonglong2* kp = reinterpret_cast<const ulonglong2*>(s_key);
#pragma unroll 4
        for (int t = 0; t < npairs; ++t) {
            const ulonglong2 kk = kp[t];                                 // warp broadcast
            rank += (kk.x > mine) + (kk.y > mine);
        }
        if (s < total && rank < k) {
            const int id = (int)~(uint32_t)mine;
            if (idx_i64) reinterpret_cast<long long*>(idx_out)[o + rank] = id;
            else reinterpret_cast<int*>(idx_out)[o + rank] = id;
        }
    }
}

// 2'. The same refine with the candidate rows fetched by the TMA unit (the default).  In the kernel above every candidate row
// crosses the LSU three times (LDG.128 into registers, STS.128 into the tile, LDS.128 back out): 290 L1 wavefronts per query
// row, 61 % of the L1 data-stage peak while 59 % of the warp stalls wait for those gathers.  Here one elected lane issues
// cp.async.bulk.tensor ... tile::gather4 (UTMALDG.2D.GATHER4): four arbitrary rows of the [B*N][64] fp32 feature map per
// instruction land in shared memory without touching the LSU, as two half-row tiles [32 candidates][128 B] in the 128-byte
// swizzle (16-byte chunk ^ (line & 7)), so that "lane = candidate" reads its row with conflict-free LDS.128.  The query row
// comes with a plain bulk copy on the same mbarrier.  Arithmetic, keys and ranking are those of knn2_refine_kernel: identical
// output.  Warps are persistent (row = warp + i * warps) and own one mbarrier each.
template <int CAP, int WARPS>
struct RefineTmaSmem {
    static constexpr int KEYS = 2 * CAP + 2;
    static constexpr size_t rows = (size_t)WARPS * 2 * 32 * 128;                     // per warp: two half-row tiles of 4 KB (1 KB aligned)
    static constexpr size_t off_xi = rows;                                           // [64] floats per warp
    static constexpr size_t off_key = off_xi + (size_t)WARPS * 256;
    static constexpr size_t key_bytes = (KEYS * 8 + 15) / 16 * 16;
    static constexpr size_t off_id = off_key + (size_t)WARPS * key_bytes;
    static constexpr size_t off_bar = off_id + (size_t)WARPS * (2 * CAP + 4) * 4;
    static constexpr size_t total = off_bar + WARPS * 8;
    static_assert(total <= 227 * 1024, "refine shared memory budget");
};

__device__ __forceinline__ void tma_gather4_e(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int col, const int4& r) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n\t}"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(col), "r"(r.x), "r"(r.y), "r"(r.z), "r"(r.w)
        : "memory");
}
__device__ __forceinline__ void bulk_load_e(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "elect.sync _|q, 0xffffffff;\n\t"
        "@q cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t}"
        ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

template <int CAP, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
knn2_refine_tma_kernel(const __grid_constant__ CUtensorMap tmap_x, const float* __restrict__ x, const float* __restrict__ xxpad,
                       const int* __restrict__ cnt, const int* __restrict__ cand, int B, int N, int Npad, int k,
                       void* __restrict__ idx_out, int idx_i64, int* __restrict__ flags, int* __restrict__ list) {
    using S = RefineTmaSmem<CAP, WARPS>;
    constexpr int IPL = (CAP + 31) / 32;               // list slots per lane and column half
    extern __shared__ __align__(1024) uint8_t rsm_t[];
    uint8_t* rsm = rsm_t;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint8_t* s_rows = rsm + (size_t)w * 2 * 32 * 128;
    const float4* s_xi = reinterpret_cast<const float4*>(rsm + S::off_xi + (size_t)w * 256);
    unsigned long long* s_key = reinterpret_cast<unsigned long long*>(rsm + S::off_key + (size_t)w * S::key_bytes);
    int* s_id = reinterpret_cast<int*>(rsm + S::off_id) + w * (2 * CAP + 4);
    uint64_t* bar = reinterpret_cast<uint64_t*>(rsm + S::off_bar) + w;
    if (lane == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const long long rows_total = (long long)B * N;
    const long long nw = (long long)gridDim.x * WARPS;
    uint32_t phase = 0;
    const int sw = lane & 7;
    // the list of the NEXT row travels in registers while the current row is processed (counts and both raw half lists: the
    // slots beyond the counts hold stale workspace bytes and are never used)
    int nc0 = 0, nc1 = 0, nl0[IPL], nl1[IPL];
    auto prefetch = [&](long long g) {
        if (g >= rows_total) return;
        nc0 = __ldg(cnt + g * 2); nc1 = __ldg(cnt + g * 2 + 1);
        const int* l0 = cand + (size_t)g * 2 * CAP;
#pragma unroll
        for (int i = 0; i < IPL; ++i) {
            const int s = lane + 32 * i;
            nl0[i] = s < CAP ? __ldg(l0 + s) : 0;
            nl1[i] = s < CAP ? __ldg(l0 + CAP + s) : 0;
        }
    };
    long long grow = (long long)blockIdx.x * WARPS + w;
    prefetch(grow);
    for (; grow < rows_total; grow += nw) {
        const int b = (int)(grow / N), qi = (int)(grow % N);
        const int c0 = nc0, c1 = nc1;
        const int total = c0 + c1;
        const bool bad = c0 > CAP || c1 > CAP || total < k;   // overflow / unusable bound: the exact kernel recomputes the 64-row tile
        const int rbase = b * N;                               // first row of the cloud in the [B*N][64] map
        if (!bad) {
#pragma unroll
            for (int i = 0; i < IPL; ++i) {
                const int s = lane + 32 * i;
                if (s < c0) s_id[s] = rbase + nl0[i];
                if (s < c1) s_id[c0 + s] = rbase + nl1[i];
            }
            if (lane < 4) s_id[total + lane] = rbase + qi;     // padding of the last gather4 (a row that is in L2 anyway)
            if (lane < 2) s_key[total + lane] = 0ull;          // padding keys: worse than anything
        }
        __syncwarp();
        if (bad) {
            if (lane == 0) knn2_flag_tile(flags, list, b * ((N + 63) / 64) + qi / 64);
            prefetch(grow + nw);
            continue;
        }
        const float xxi = __ldg(xxpad + (size_t)b * Npad + qi);
        for (int base = 0; base < total; base += 32) {
            const int nc = min(32, total - base);
            const int n4 = (nc + 3) >> 2;
            mbar_expect_tx_e(bar, (uint32_t)n4 * 1024u + (base == 0 ? 256u : 0u));
            if (base == 0) bulk_load_e(const_cast<float4*>(s_xi), x + (size_t)grow * 64, 256u, bar);
            for (int g = 0; g < n4; ++g) {
                const int4 r = *reinterpret_cast<const int4*>(s_id + base + 4 * g);       // warp broadcast
                tma_gather4_e(s_rows + g * 512, &tmap_x, bar, 0, r);
                tma_gather4_e(s_rows + 4096 + g * 512, &tmap_x, bar, 32, r);
            }
            const int myrow = lane < nc ? s_id[base + lane] : rbase;
            const float xxj = __ldg(xxpad + (size_t)b * Npad + (myrow - rbase));
            if (base == 0) prefetch(grow + nw);        // in flight behind the gathers
            mbar_wait(bar, phase);
            phase ^= 1u;
            float dot = 0.f;
#pragma unroll
            for (int ph = 0; ph < 2; ++ph) {
                const float4* rj = reinterpret_cast<const float4*>(s_rows + ph * 4096 + lane * 128);
#pragma unroll
                for (int g = 0; g < 8; ++g) {
                    const float4 u = s_xi[ph * 8 + g], v = rj[g ^ sw];
                    dot = __fmaf_rn(u.x, v.x, dot); dot = __fmaf_rn(u.y, v.y, dot);
                    dot = __fmaf_rn(u.z, v.z, dot); dot = __fmaf_rn(u.w, v.w, dot);
                }
            }
            if (lane < nc) {
                const float t = -2.0f * dot;
                const float pd = __fadd_rn(__fsub_rn(__fsub_rn(-xxj, t), xxi), 0.0f);   // (+ 0: -0.0 and +0.0 must share one key)
                uint32_t u = __float_as_uint(pd);
                u ^= (u >> 31) ? 0xffffffffu : 0x80000000u;                  // monotone float -> uint
                s_key[base + lane] = ((unsigned long long)u << 32) | (uint32_t)(~(myrow - rbase));
            }
            __syncwarp();                              // tile consumed (and keys visible) before the next gather overwrites it
        }
        const size_t o = (size_t)grow * k;
        const int npairs = (total + 1) >> 1;
        for (int base = 0; base < total; base += 32) {
            const int s = base + lane;
            const unsigned long long mine = s < total ? s_key[s] : ~0ull;
            int rank = 0;
            const ulonglong2* kp = reinterpret_cast<const ulonglong2*>(s_key);
#pragma unroll 4
            for (int t = 0; t < npairs; ++t) {
                const ulonglong2 kk = kp[t];                                 // warp broadcast
                rank += (kk.x > mine) + (kk.y > mine);
            }
            if (s < total && rank < k) {
                const int id = (int)~(uint32_t)mine;
                if (idx_i64) reinterpret_cast<long long*>(idx_out)[o + rank] = id;
                else reinterpret_cast<int*>(idx_out)[o + rank] = id;
            }
        }
        __syncwarp();                                  // keys / ids consumed before the next row rewrites them
    }
}

// 1 (default): TMA-gather refine; 0: LSU-gather refine (LPD_KNN_REFINE=0)
static int g_refine_tma = [] { const char* e = getenv("LPD_KNN_REFINE"); return (e && atoi(e) == 0) ? 0 : 1; }();
static int g_refine_warps = [] { const char* e = getenv("LPD_KNN_REFINE_WARPS"); return e ? atoi(e) : 22; }();

template <int CAP, int WARPS>
static int knn2_refine_tma_launch(const float* x, const float* xxpad, const int* cnt, const int* cand, int B, int N, int Npad, int k,
                                  void* idx, int idx_i64, int* flags, int* list, cudaStream_t st) {
    CUtensorMap tx;
    // box = one half row (32 floats = 128 B), 128B swizzle
    int rc = make_tmap(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, x, (long long)B * N, 64, 64, 1, 32);
    if (rc != LPD_OK) return rc;
    const size_t smem = RefineTmaSmem<CAP, WARPS>::total;
    static int sms = 0, per_sm = 0;                                   // per instantiation; one device model per process
    if (per_sm == 0) {
        LPD_CUDA_CHECK(allow_smem(knn2_refine_tma_kernel<CAP, WARPS>, smem));
        rc = sm_count(&sms);
        if (rc != LPD_OK) return rc;
        LPD_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, knn2_refine_tma_kernel<CAP, WARPS>, WARPS * 32, smem));
        if (per_sm < 1) per_sm = 1;
    }
    const long long want = ((long long)B * N + WARPS - 1) / WARPS;
    const long long blocks = want < (long long)sms * per_sm ? want : (long long)sms * per_sm;
    knn2_refine_tma_kernel<CAP, WARPS><<<(unsigned)blocks, WARPS * 32, smem, st>>>(tx, x, xxpad, cnt, cand, B, N, Npad, k, idx, idx_i64, flags, list);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

template <int CAP>
static int knn2_refine_launch(const float* x, const float* xxpad, const int* cnt, const int* cand, int B, int N, int Npad, int k,
                              void* idx, int idx_i64, int* flags, int* list, cudaStream_t st) {
    if (g_refine_tma) {
        if constexpr (CAP > 64) {                          // (the per-warp key / id buffers grow with CAP: 16 warps fit)
            return knn2_refine_tma_launch<CAP, 16>(x, xxpad, cnt, cand, B, N, Npad, k, idx, idx_i64, flags, list, st);
        } else {
            if (g_refine_warps == 4) return knn2_refine_tma_launch<CAP, 4>(x, xxpad, cnt, cand, B, N, Npad, k, idx, idx_i64, flags, list, st);
            if (g_refine_warps == 11) return knn2_refine_tma_launch<CAP, 11>(x, xxpad, cnt, cand, B, N, Npad, k, idx, idx_i64, flags, list, st);
            return knn2_refine_tma_launch<CAP, 22>(x, xxpad, cnt, cand, B, N, Npad, k, idx, idx_i64, flags, list, st);
        }
    }
    const size_t smem = RefineSmem<CAP>::total;
    LPD_CUDA_CHECK(allow_smem(knn2_refine_kernel<CAP>, smem));
    const unsigned rblocks = (unsigned)(((long long)B * N + RF_WARPS - 1) / RF_WARPS);
    knn2_refine_kernel<CAP><<<rblocks, RF_WARPS * 32, smem, st>>>(x, xxpad, cnt, cand, B, N, Npad, k, idx, idx_i64, flags, list);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

static inline size_t align_up2(size_t v, size_t a) { return (v + a - 1) / a * a; }

// candidate slots per (row, column half) for k <= 24.  40 is 1.5 x the ~27 candidates a row collects, but a row whose neighbours
// pile up in few strided groups gets a loose threshold and now and then (about one row in 3e5 on uniform clouds) collects more than
// 40 in one half: its 64-row tile then goes to the exact kernel, whose single CTA needs 0.86 ms for the 4096-candidate scan — a
// 30 % longer step for that batch.  64 slots make the overflow rare enough not to matter (LPD_KNN_CAP=40 restores the old value).
static int g_cap_small = [] { const char* e = getenv("LPD_KNN_CAP"); return (e && atoi(e) == 40) ? 40 : 64; }();

struct Knn2Ws {
    size_t off_xx, off_nrm, off_sn, off_ext, off_r2, off_r2c, off_mu, off_sc, off_flags, off_list, off_xh, off_cnt, off_cand, total;
    int npad, cap;
    Knn2Ws(int B, int N, int k) {
        npad = (N + 255) / 256 * 256;
        cap = k > 24 ? 128 : (g_cap_small == 40 ? 40 : 64);   // k > 24 (the per-candidate bound: ~45 candidates per row): 128 slots per half
        size_t o = 0;
        off_xx = o; o = align_up2(o + (size_t)B * npad * 4, 256);
        off_nrm = o; o = align_up2(o + (size_t)B * npad * 4, 256);
        off_sn = o; o = align_up2(o + (size_t)B * npad * 4, 256);
        off_ext = o; o = align_up2(o + (size_t)B * npad * 32, 256);
        off_r2 = o; o += (size_t)B * 4;
        off_r2c = o; o = align_up2(o + (size_t)B * 4, 256);
        off_mu = o; o = align_up2(o + (size_t)B * K2_CSPLIT * 196 * 4, 256);      // per-cloud partial sums / minima / maxima
        off_sc = o; o = align_up2(o + (size_t)B * 2 * 4, 256);
        off_flags = o; o = align_up2(o + (size_t)B * ((N + 63) / 64) * 4, 256);
        off_list = o; o = align_up2(o + ((size_t)B * ((N + 63) / 64) + 1) * 4, 256);     // work list of the exact kernel
        off_xh = o; o = align_up2(o + (size_t)B * N * 64 * 2, 256);
        off_cnt = o; o = align_up2(o + (size_t)B * N * 2 * 4, 256);
        off_cand = o; o = align_up2(o + (size_t)B * N * 2 * cap * 4, 256);
        total = o;
    }
};

size_t knn2_workspace_bytes(int B, int N, int k) { return Knn2Ws(B, N, k).total; }

template <int MT, int CAP, bool TIGHT, bool TS = false>
static int knn2_launch(const CUtensorMap& ta, const CUtensorMap& tb, const Knn2Params& P, cudaStream_t st) {
    const size_t smem = K2Smem<MT, TS>::total;
    LPD_CUDA_CHECK(allow_smem(knn2_tc_kernel<MT, CAP, TIGHT, TS>, smem));
    int sms = 0;
    const int rc = sm_count(&sms);
    if (rc != LPD_OK) return rc;
    const int items = P.B * P.qtiles;
    knn2_tc_kernel<MT, CAP, TIGHT, TS><<<items < sms ? items : sms, 256 * MT + 64, smem, st>>>(ta, tb, P);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

// mt = 1: 128 query rows per work item (8 scan warps); mt = 2: 256 rows (16 scan warps, every candidate tile feeds two MMAs)
int knn2_run(const float* x, int B, int N, int k, void* idx, int idx_i64, void* workspace, size_t workspace_bytes, int mt,
             cudaStream_t st) {
    const Knn2Ws W(B, N, k);
    if (workspace_bytes < W.total) return LPD_EWORKSPACE;
    uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
    float* xxpad = reinterpret_cast<float*>(ws + W.off_xx);
    float* nrmpad = reinterpret_cast<float*>(ws + W.off_nrm);
    float* snpad = reinterpret_cast<float*>(ws + W.off_sn);
    float* r2 = reinterpret_cast<float*>(ws + W.off_r2);
    float* r2c = reinterpret_cast<float*>(ws + W.off_r2c);
    float* mu = reinterpret_cast<float*>(ws + W.off_mu);
    float* sc = reinterpret_cast<float*>(ws + W.off_sc);
    int* flags = reinterpret_cast<int*>(ws + W.off_flags);
    int* list = reinterpret_cast<int*>(ws + W.off_list);
    __half* xh = reinterpret_cast<__half*>(ws + W.off_xh);
    LPD_CUDA_CHECK(cudaMemsetAsync(r2, 0, W.off_mu - W.off_r2, st));     // r2 and r2c
    LPD_CUDA_CHECK(cudaMemsetAsync(flags, 0, W.off_list - W.off_flags + sizeof(int), st));   // the flags and the list length
    knn2_center_kernel<<<dim3(K2_CSPLIT, B), 256, 0, st>>>(x, N, mu);
    LPD_LAUNCH_CHECK();
    static bool prep_smem_ok = false;
    if (!prep_smem_ok) { LPD_CUDA_CHECK(allow_smem(knn2_prep_kernel, K2_PREP_SMEM)); prep_smem_ok = true; }
    knn2_prep_kernel<<<dim3(ceil_div(W.npad, 256), B), 256, K2_PREP_SMEM, st>>>(x, mu, sc, N, W.npad, xh, reinterpret_cast<uint4*>(ws + W.off_ext), xxpad, nrmpad, snpad, r2, r2c);
    LPD_LAUNCH_CHECK();
    CUtensorMap ta, tb;   // xh fp16 [B*N][64]: boxes of 128 query rows / K2_C = 128 candidates per stage, 64 halves each
    int rc = make_tmap(&ta, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, xh, (long long)B * N, 64, 64, 128, 64);
    if (rc != LPD_OK) return rc;
    rc = make_tmap(&tb, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, xh, (long long)B * N, 64, 64, K2_C, 64);
    if (rc != LPD_OK) return rc;
    Knn2Params P;
    P.nrmpad = nrmpad; P.snpad = snpad; P.ext = reinterpret_cast<const uint4*>(ws + W.off_ext); P.xh = reinterpret_cast<const uint4*>(xh); P.xxpad = xxpad; P.r2 = r2; P.r2c = r2c; P.sc = sc;
    P.cnt = reinterpret_cast<int*>(ws + W.off_cnt);
    P.cand = reinterpret_cast<int*>(ws + W.off_cand);
    P.B = B; P.N = N; P.Npad = W.npad; P.k = k;
    P.qtiles = ceil_div(N, mt == 2 ? 256 : 128); P.ctiles = ceil_div(N, K2_C);
    // k <= 24: 64 (or 40) slots per (row, half), uniform error bound; k <= 32: 128 slots, per-candidate bound
    if (mt == 3) {          // 128 rows per item, query tile in tensor memory (TS-mode MMA)
        rc = (W.cap == 40) ? knn2_launch<1, 40, false, true>(ta, tb, P, st)
                           : (k <= 24 ? knn2_launch<1, 64, false, true>(ta, tb, P, st) : knn2_launch<1, 128, true, true>(ta, tb, P, st));
    } else if (W.cap == 40) rc = (mt == 2) ? knn2_launch<2, 40, false>(ta, tb, P, st) : knn2_launch<1, 40, false>(ta, tb, P, st);
    else if (k <= 24) rc = (mt == 2) ? knn2_launch<2, 64, false>(ta, tb, P, st) : knn2_launch<1, 64, false>(ta, tb, P, st);
    else             rc = (mt == 2) ? knn2_launch<2, 128, true>(ta, tb, P, st) : knn2_launch<1, 128, true>(ta, tb, P, st);
    if (rc != LPD_OK) return rc;
    rc = (W.cap == 40) ? knn2_refine_launch<40>(x, xxpad, P.cnt, P.cand, B, N, W.npad, k, idx, idx_i64, flags, list, st)
         : (W.cap == 64 ? knn2_refine_launch<64>(x, xxpad, P.cnt, P.cand, B, N, W.npad, k, idx, idx_i64, flags, list, st)
                        : knn2_refine_launch<128>(x, xxpad, P.cnt, P.cand, B, N, W.npad, k, idx, idx_i64, flags, list, st));
    if (rc != LPD_OK) return rc;
    return knn_simt64_list(x, B, N, k, idx, idx_i64, list, st);       // exact recompute of the flagged 64-row tiles only
}

// diagnostics for the tests / tools: where the tile flags of the last run live inside the workspace
size_t knn2_flags_offset(int B, int N, int k) { return Knn2Ws(B, N, k).off_flags; }
size_t knn2_cnt_offset(int B, int N, int k) { return Knn2Ws(B, N, k).off_cnt; }

}  // namespace tc
}  // namespace lpd
