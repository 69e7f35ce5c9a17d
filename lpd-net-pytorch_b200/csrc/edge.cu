// EdgeConv kernels.  The reference materialises the edge tensor [B, 2C, N, k] (40-80 MiB per cloud,
// get_graph_feature lpdnet_model.py:331-363) and runs Conv2d 1x1 + BatchNorm2d + LeakyReLU + max over it
// (lpdnet_model.py:246-258).  Here the edge tensor never exists in HBM:
//   * a 1x1 conv over cat(neighbour, centre) splits exactly into two per-point products
//     W.[f_j ; f_i] = P_j + Q_i (SURVEY App. A.3) which are computed once per POINT by lpd_gemm;
//   * edge_gather_ext_kernel gathers k rows of P per point and reduces them with max/min
//     (monotone BN+activation commute with the extremum);
//   * edgeconv_dg_kernel rebuilds the activated first-layer edge rows of one point in shared memory,
//     multiplies them by the second-layer weight (kept resident in shared memory by a persistent
//     CTA) and max-reduces over the k neighbours in registers.
#include "common.cuh"
#include <cuda_fp16.h>

namespace lpd {

template <int V> struct VecT;
template <> struct VecT<4> { using type = float4; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<1> { using type = float; };

template <int V>
__device__ __forceinline__ void vload(const float* __restrict__ p, float (&v)[V]) {
    using T = typename VecT<V>::type;
    const T t = *reinterpret_cast<const T*>(p);
    const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] = f[i];
}
template <int V>
__device__ __forceinline__ void vload_g(const float* __restrict__ p, float (&v)[V]) {
    using T = typename VecT<V>::type;
    const T t = __ldg(reinterpret_cast<const T*>(p));
    const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
    for (int i = 0; i < V; ++i) v[i] = f[i];
}
template <int V>
__device__ __forceinline__ void vstore(float* __restrict__ p, const float (&v)[V]) {
    using T = typename VecT<V>::type;
    T t;
    float* f = reinterpret_cast<float*>(&t);
#pragma unroll
    for (int i = 0; i < V; ++i) f[i] = v[i];
    *reinterpret_cast<T*>(p) = t;
}

__device__ __forceinline__ float act2(float v, int act, float slope) {
    // only the activations that occur on edge layers (LeakyReLU / ReLU / none)
    if (act == LPD_ACT_LEAKY) return v > 0.f ? v : v * slope;
    if (act == LPD_ACT_RELU) return fmaxf(v, 0.f);
    return v;
}

// ------------------------------------------------------------------------------------------------
// out[i][c] = act(s[c] * (q[i][c] + ext_m p[j(i,m)][c]) + t[c])
// One thread owns 4 channels of one point; C/4 threads per point, 256 threads per CTA.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
edge_gather_ext_kernel(const float* __restrict__ p, int ldp, const float* __restrict__ q, int ldq,
                       const int* __restrict__ idx, long long total_pts, int N, int k, int C,
                       const float* __restrict__ scale, const float* __restrict__ shift, int act, float slope,
                       float* __restrict__ out, int ldo) {
    const int tpp = C >> 2;                       // threads per point
    const int ppb = 256 / tpp;                    // points per block
    const int lp = threadIdx.x / tpp;
    const int c = (threadIdx.x % tpp) * 4;
    const long long pt = (long long)blockIdx.x * ppb + lp;
    if (lp >= ppb || pt >= total_pts) return;
    const long long cloud0 = (pt / N) * N;        // first row of this point's cloud
    const int* ip = idx + pt * k;

    float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    float mn[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
    int m = 0;
    if (tpp >= 32 && k <= 32) {
        // a warp works on ONE point: its lanes fetch the k neighbour indices once and hand them round with shuffles, and the
        // row address is one 32-bit multiply-add on a per-thread base (was: an index load + 64-bit address chain per row per thread)
        const int lane = threadIdx.x & 31;
        const int myj = lane < k ? __ldg(ip + lane) : 0;
        const float* base = p + cloud0 * ldp + c;
        for (; m + 5 <= k; m += 5) {
            float4 v[5];
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                const int j = __shfl_sync(0xffffffffu, myj, m + u);
                v[u] = __ldg(reinterpret_cast<const float4*>(base + (unsigned)(j * ldp)));
            }
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                mx[0] = fmaxf(mx[0], v[u].x); mx[1] = fmaxf(mx[1], v[u].y); mx[2] = fmaxf(mx[2], v[u].z); mx[3] = fmaxf(mx[3], v[u].w);
                mn[0] = fminf(mn[0], v[u].x); mn[1] = fminf(mn[1], v[u].y); mn[2] = fminf(mn[2], v[u].z); mn[3] = fminf(mn[3], v[u].w);
            }
        }
        for (; m < k; ++m) {
            const int j = __shfl_sync(0xffffffffu, myj, m);
            const float4 v = __ldg(reinterpret_cast<const float4*>(base + (unsigned)(j * ldp)));
            mx[0] = fmaxf(mx[0], v.x); mx[1] = fmaxf(mx[1], v.y); mx[2] = fmaxf(mx[2], v.z); mx[3] = fmaxf(mx[3], v.w);
            mn[0] = fminf(mn[0], v.x); mn[1] = fminf(mn[1], v.y); mn[2] = fminf(mn[2], v.z); mn[3] = fminf(mn[3], v.w);
        }
    }
    for (; m + 4 <= k; m += 4) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = __ldg(ip + m + u);
            v[u] = __ldg(reinterpret_cast<const float4*>(p + (cloud0 + j) * ldp + c));
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            mx[0] = fmaxf(mx[0], v[u].x); mx[1] = fmaxf(mx[1], v[u].y); mx[2] = fmaxf(mx[2], v[u].z); mx[3] = fmaxf(mx[3], v[u].w);
            mn[0] = fminf(mn[0], v[u].x); mn[1] = fminf(mn[1], v[u].y); mn[2] = fminf(mn[2], v[u].z); mn[3] = fminf(mn[3], v[u].w);
        }
    }
    for (; m < k; ++m) {
        const int j = __ldg(ip + m);
        const float4 v = __ldg(reinterpret_cast<const float4*>(p + (cloud0 + j) * ldp + c));
        mx[0] = fmaxf(mx[0], v.x); mx[1] = fmaxf(mx[1], v.y); mx[2] = fmaxf(mx[2], v.z); mx[3] = fmaxf(mx[3], v.w);
        mn[0] = fminf(mn[0], v.x); mn[1] = fminf(mn[1], v.y); mn[2] = fminf(mn[2], v.z); mn[3] = fminf(mn[3], v.w);
    }
    float qv[4] = {0.f, 0.f, 0.f, 0.f};
    if (q) vload_g<4>(q + pt * ldq + c, qv);
    float o[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const float s = scale ? __ldg(scale + c + u) : 1.f;
        const float t = shift ? __ldg(shift + c + u) : 0.f;
        const float e = (s >= 0.f) ? mx[u] : mn[u];
        o[u] = act2(fmaf(s, qv[u] + e, t), act, slope);
    }
    vstore<4>(out + pt * ldo + c, o);
}

// ------------------------------------------------------------------------------------------------
// Pre-scaled form (scale == shift == NULL: the caller folded the layer's BatchNorm into p and q, e.g. in the projection
// GEMM's epilogue), wide rows:   out[i][c] = act(q[i][c] + max_m p[j(i,m)][c]),   C = 128 * VPL.
// One WARP per point, VPL float4 per lane and row (lane l owns the 16-byte chunks l, l + 32, ...: every LDG.128 of the warp
// reads 512 contiguous bytes); per gathered row the warp spends one shuffle, one 32-bit multiply-add, VPL loads and 2 VPL
// three-input maxima (two rows per FMNMX3) — a fifth of the instructions of the generic kernel, which was 66 % issue-active.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float fmax3f(float a, float b, float c) {
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

template <int VPL>
__global__ void __launch_bounds__(256)
edge_gather_max_kernel(const float* __restrict__ p, int ldp, const float* __restrict__ q, int ldq,
                       const int* __restrict__ idx, long long total_pts, int N, int k, int act, float slope,
                       float* __restrict__ out, int ldo) {
    const int lane = threadIdx.x & 31;
    const long long pt = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (pt >= total_pts) return;
    const int myj = lane < k ? __ldg(idx + pt * k + lane) : 0;
    const float* base = p + (pt / N) * N * ldp + lane * 4;
    float4 qv[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v)
        qv[v] = q ? __ldg(reinterpret_cast<const float4*>(q + pt * ldq + lane * 4 + v * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 mx[VPL];
#pragma unroll
    for (int v = 0; v < VPL; ++v) mx[v] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    int m = 0;
    for (; m + 4 <= k; m += 4) {                     // 4 rows (4 VPL loads) in flight per lane
        float4 r[4][VPL];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = __shfl_sync(0xffffffffu, myj, m + u);
            const float* row = base + (unsigned)(j * ldp);
#pragma unroll
            for (int v = 0; v < VPL; ++v) r[u][v] = __ldg(reinterpret_cast<const float4*>(row + v * 128));
        }
#pragma unroll
        for (int u = 0; u < 4; u += 2)
#pragma unroll
            for (int v = 0; v < VPL; ++v) {
                mx[v].x = fmax3f(mx[v].x, r[u][v].x, r[u + 1][v].x); mx[v].y = fmax3f(mx[v].y, r[u][v].y, r[u + 1][v].y);
                mx[v].z = fmax3f(mx[v].z, r[u][v].z, r[u + 1][v].z); mx[v].w = fmax3f(mx[v].w, r[u][v].w, r[u + 1][v].w);
            }
    }
    for (; m < k; ++m) {
        const int j = __shfl_sync(0xffffffffu, myj, m);
        const float* row = base + (unsigned)(j * ldp);
#pragma unroll
        for (int v = 0; v < VPL; ++v) {
            const float4 r = __ldg(reinterpret_cast<const float4*>(row + v * 128));
            mx[v].x = fmaxf(mx[v].x, r.x); mx[v].y = fmaxf(mx[v].y, r.y); mx[v].z = fmaxf(mx[v].z, r.z); mx[v].w = fmaxf(mx[v].w, r.w);
        }
    }
#pragma unroll
    for (int v = 0; v < VPL; ++v) {
        float4 o;
        o.x = act2(qv[v].x + mx[v].x, act, slope); o.y = act2(qv[v].y + mx[v].y, act, slope);
        o.z = act2(qv[v].z + mx[v].z, act, slope); o.w = act2(qv[v].w + mx[v].w, act, slope);
        *reinterpret_cast<float4*>(out + pt * ldo + lane * 4 + v * 128) = o;
    }
}

// ------------------------------------------------------------------------------------------------
// The same with FP16 rows ("f16" precision mode): p, q, out are fp16 matrices with 256 channels (512 bytes per row: ONE LDG.128
// per lane and row — half the bytes of the fp32 form through the L1 / L2 data path, which is what bounds this kernel).  The max
// over the neighbours is taken on the fp16 values directly (exact), the centre term and the activation in fp32, one rounding
// to nearest on the way out.
// C = 64 (128-byte rows, LPDNetOrign's gather-only SN stage): 8 lanes cover a row, so the warp's four lane groups load four
// neighbour rows side by side (group g takes neighbours g, g + 4, ...) and combine their maxima with two shuffles.
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(256)
edge_gather_max_h_kernel(const __half* __restrict__ p, int ldp, const __half* __restrict__ q, int ldq,
                         const int* __restrict__ idx, long long total_pts, int N, int k, int act, float slope,
                         __half* __restrict__ out, int ldo) {
    constexpr int LPR = C / 8, G = 32 / LPR;         // lanes per row, rows per warp-wide load
    const int lane = threadIdx.x & 31, g = lane / LPR, col = (lane % LPR) * 8;
    const long long pt = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (pt >= total_pts) return;
    const int myj = lane < k ? __ldg(idx + pt * k + lane) : 0;
    const __half* base = p + (pt / N) * N * ldp + col;
    const uint4 qraw = q ? __ldg(reinterpret_cast<const uint4*>(q + pt * ldq + col)) : make_uint4(0u, 0u, 0u, 0u);
    const __half2 ninf = __float2half2_rn(-INFINITY);
    __half2 mx[4] = {ninf, ninf, ninf, ninf};
    int m = 0;
    for (; m + 5 * G <= k; m += 5 * G) {             // 5 rows in flight per lane
        uint4 r[5];
#pragma unroll
        for (int u = 0; u < 5; ++u) {
            const int j = __shfl_sync(0xffffffffu, myj, m + u * G + g);
            r[u] = __ldg(reinterpret_cast<const uint4*>(base + (unsigned)(j * ldp)));
        }
#pragma unroll
        for (int u = 0; u < 5; ++u) {
            const __half2* h = reinterpret_cast<const __half2*>(&r[u]);
#pragma unroll
            for (int v = 0; v < 4; ++v) mx[v] = __hmax2(mx[v], h[v]);
        }
    }
    for (; m < k; m += G) {
        const int mm = m + g;
        const int j = __shfl_sync(0xffffffffu, myj, mm < k ? mm : m);
        if (mm < k) {
            const uint4 r = __ldg(reinterpret_cast<const uint4*>(base + (unsigned)(j * ldp)));
            const __half2* h = reinterpret_cast<const __half2*>(&r);
#pragma unroll
            for (int v = 0; v < 4; ++v) mx[v] = __hmax2(mx[v], h[v]);
        }
    }
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const uint32_t o = __shfl_xor_sync(0xffffffffu, *reinterpret_cast<const uint32_t*>(&mx[v]), off);
            mx[v] = __hmax2(mx[v], *reinterpret_cast<const __half2*>(&o));
        }
    const __half2* qh = reinterpret_cast<const __half2*>(&qraw);
    uint4 o;
    __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        const float2 a = __half22float2(mx[v]), b = __half22float2(qh[v]);
        oh[v] = __floats2half2_rn(act2(a.x + b.x, act, slope), act2(a.y + b.y, act, slope));
    }
    if (g == 0) *reinterpret_cast<uint4*>(out + pt * ldo + col) = o;
}

// ------------------------------------------------------------------------------------------------
// Two chained edge layers, one warp per point, persistent CTAs with W2 resident in shared memory.
// ------------------------------------------------------------------------------------------------
struct DgParams {
    const float* p; const float* q; const int* idx;
    const float* s1; const float* t1; const float* w2; const float* s2; const float* t2;
    float* x1; float* x2;
    int ldp, ldq, ld1, ld2;
    long long total_pts; int N, k;
    int act; float slope;
};

template <int C1, int C2, int RP>
__global__ void __launch_bounds__(384, 1) edgeconv_dg_kernel(DgParams P) {
    constexpr int V1 = C1 / 32, V2 = C2 / 32;
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int passes = (P.k + RP - 1) / RP;
    const int KP = passes * RP;
    float* W2T = smem;                                   // [C1][C2]: W2T[c1][c2] = w2[c2][c1]
    float* Y = smem + C1 * C2 + (size_t)warp * KP * C1;  // this warp's first-layer rows [KP][C1]

    for (int e = threadIdx.x; e < C1 * C2; e += blockDim.x) {
        const int c1 = e / C2, c2 = e % C2;
        W2T[e] = __ldg(P.w2 + (size_t)c2 * C1 + c1);
    }
    float s1[V1], t1[V1], s2[V2], t2[V2];
#pragma unroll
    for (int u = 0; u < V1; ++u) { s1[u] = __ldg(P.s1 + lane * V1 + u); t1[u] = __ldg(P.t1 + lane * V1 + u); }
#pragma unroll
    for (int u = 0; u < V2; ++u) { s2[u] = __ldg(P.s2 + lane * V2 + u); t2[u] = __ldg(P.t2 + lane * V2 + u); }
    __syncthreads();

    for (long long pt = (long long)blockIdx.x * nwarps + warp; pt < P.total_pts; pt += (long long)gridDim.x * nwarps) {
        const long long cloud0 = (pt / P.N) * P.N;
        // ---- layer 1: y1[m][:] = act(s1 * (p[j] + q[i]) + t1) ----
        float qv[V1];
        vload_g<V1>(P.q + pt * P.ldq + lane * V1, qv);
        const int myj = (lane < P.k) ? __ldg(P.idx + pt * P.k + lane) : 0;
        float best1[V1];
#pragma unroll
        for (int u = 0; u < V1; ++u) best1[u] = -INFINITY;
        for (int m0 = 0; m0 < KP; m0 += 4) {
            float pv[4][V1];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int m = m0 + u;
                const int j = __shfl_sync(kFull, myj, m & 31);
                if (m < P.k) vload_g<V1>(P.p + (cloud0 + j) * P.ldp + lane * V1, pv[u]);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int m = m0 + u;
                if (m >= KP) break;
                float y[V1];
#pragma unroll
                for (int w = 0; w < V1; ++w) {
                    if (m < P.k) {
                        y[w] = act2(fmaf(s1[w], pv[u][w] + qv[w], t1[w]), P.act, P.slope);
                        best1[w] = fmaxf(best1[w], y[w]);
                    } else y[w] = 0.f;
                }
                vstore<V1>(Y + m * C1 + lane * V1, y);
            }
        }
        if (P.x1) vstore<V1>(P.x1 + pt * P.ld1 + lane * V1, best1);
        __syncwarp();

        // ---- layer 2: y2[m][:] = act(s2 * (W2 . y1[m]) + t2), x2 = max_m ----
        float best2[V2];
#pragma unroll
        for (int u = 0; u < V2; ++u) best2[u] = -INFINITY;
        for (int pass = 0; pass < passes; ++pass) {
            float acc[RP][V2];
#pragma unroll
            for (int r = 0; r < RP; ++r)
#pragma unroll
                for (int u = 0; u < V2; ++u) acc[r][u] = 0.f;
            const float* Yp = Y + pass * RP * C1;
#pragma unroll 2
            for (int kk = 0; kk < C1; kk += 4) {
                float w[4][V2];
#pragma unroll
                for (int u = 0; u < 4; ++u) vload<V2>(W2T + (kk + u) * C2 + lane * V2, w[u]);
#pragma unroll
                for (int r = 0; r < RP; ++r) {
                    const float4 a = *reinterpret_cast<const float4*>(Yp + r * C1 + kk);  // warp broadcast
#pragma unroll
                    for (int u = 0; u < V2; ++u) {
                        acc[r][u] = fmaf(a.x, w[0][u], acc[r][u]);
                        acc[r][u] = fmaf(a.y, w[1][u], acc[r][u]);
                        acc[r][u] = fmaf(a.z, w[2][u], acc[r][u]);
                        acc[r][u] = fmaf(a.w, w[3][u], acc[r][u]);
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < RP; ++r) {
                if (pass * RP + r < P.k) {
#pragma unroll
                    for (int u = 0; u < V2; ++u)
                        best2[u] = fmaxf(best2[u], act2(fmaf(s2[u], acc[r][u], t2[u]), P.act, P.slope));
                }
            }
        }
        vstore<V2>(P.x2 + pt * P.ld2 + lane * V2, best2);
        __syncwarp();  // Y is rebuilt by the next point
    }
}

template <int C1, int C2, int RP>
static int dg_launch(const DgParams& P, cudaStream_t st) {
    int dev = 0, sms = 0, smem_max = 0;
    LPD_CUDA_CHECK(cudaGetDevice(&dev));
    LPD_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    LPD_CUDA_CHECK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const int passes = (P.k + RP - 1) / RP;
    const size_t per_warp = (size_t)passes * RP * C1 * sizeof(float);
    const size_t wbytes = (size_t)C1 * C2 * sizeof(float);
    int warps = (int)(((size_t)smem_max - wbytes) / per_warp);
    if (warps > 12) warps = 12;
    warps &= ~3;
    LPD_REQUIRE(warps >= 4);
    const size_t smem = wbytes + per_warp * warps;
    LPD_CUDA_CHECK(allow_smem(edgeconv_dg_kernel<C1, C2, RP>, smem));
    long long need = (P.total_pts + warps - 1) / warps;
    int grid = (int)(need < sms ? need : sms);
    edgeconv_dg_kernel<C1, C2, RP><<<grid, warps * 32, smem, st>>>(P);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

}  // namespace lpd

extern "C" int lpd_edge_gather_ext(const float* p, int ldp, const float* q, int ldq,
                                   const int32_t* idx, int B, int N, int k, int C,
                                   const float* scale, const float* shift, int act, float slope,
                                   float* out, int ldo, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(p && idx && out);
    LPD_REQUIRE(B >= 1 && N >= 1 && k >= 1 && k <= N);
    LPD_REQUIRE(C >= 4 && C <= 1024 && (C % 4) == 0 && (256 % (C / 4)) == 0);
    LPD_REQUIRE(ldp % 4 == 0 && ldo % 4 == 0 && ldp >= C && ldo >= C && (!q || (ldq % 4 == 0 && ldq >= C)));
    LPD_REQUIRE(act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY);
    LPD_REQUIRE(((uintptr_t)p & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)q & 15) == 0);
    LPD_REQUIRE((long long)N * ldp < (1ll << 31));          // cloud-local row offsets are 32-bit
    const long long total = (long long)B * N;
    if (!scale && !shift && (C == 128 || C == 256) && k <= 32) {    // pre-scaled, wide rows: one warp per point
        const long long wblocks = (total + 7) / 8;
        LPD_REQUIRE(wblocks <= 0x7fffffffLL);
        if (C == 256) edge_gather_max_kernel<2><<<(unsigned)wblocks, 256, 0, as_stream(stream)>>>(p, ldp, q, ldq, idx, total, N, k, act, slope, out, ldo);
        else edge_gather_max_kernel<1><<<(unsigned)wblocks, 256, 0, as_stream(stream)>>>(p, ldp, q, ldq, idx, total, N, k, act, slope, out, ldo);
        LPD_LAUNCH_CHECK();
        return LPD_OK;
    }
    const int ppb = 256 / (C / 4);
    const long long blocks = (total + ppb - 1) / ppb;
    LPD_REQUIRE(blocks <= 0x7fffffffLL);
    edge_gather_ext_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(p, ldp, q, ldq, idx, total, N, k, C, scale, shift,
                                                                         act, slope, out, ldo);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_gather_max_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                                       int act, float slope, void* out, int ldo, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(p && idx && out && B >= 1 && N >= 1 && k >= 1 && k <= 32 && k <= N);
    LPD_REQUIRE(C == 256 || C == 64);
    LPD_REQUIRE(ldp % 8 == 0 && ldo % 8 == 0 && ldp >= C && ldo >= C && (!q || (ldq % 8 == 0 && ldq >= C)));
    LPD_REQUIRE(act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY);
    LPD_REQUIRE(((uintptr_t)p & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)q & 15) == 0);
    LPD_REQUIRE((long long)N * ldp < (1ll << 31));
    const long long total = (long long)B * N;
    const long long blocks = (total + 7) / 8;
    LPD_REQUIRE(blocks <= 0x7fffffffLL);
    auto kernel = C == 256 ? edge_gather_max_h_kernel<256> : edge_gather_max_h_kernel<64>;
    kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
        reinterpret_cast<const __half*>(p), ldp, reinterpret_cast<const __half*>(q), ldq, idx, total, N, k, act, slope,
        reinterpret_cast<__half*>(out), ldo);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edgeconv_dg(const float* p, int ldp, const float* q, int ldq,
                               const int32_t* idx, int B, int N, int k, int C1, int C2,
                               const float* s1, const float* t1, const float* w2,
                               const float* s2, const float* t2, int act, float slope,
                               float* x1, int ld1, float* x2, int ld2, void* stream) {
    using namespace lpd;
    LPD_REQUIRE(p && q && idx && s1 && t1 && w2 && s2 && t2 && x2);
    LPD_REQUIRE(B >= 1 && N >= 1 && k >= 1 && k <= 32 && k <= N);
    LPD_REQUIRE((C1 == 128 && C2 == 128) || (C1 == 64 && C2 == 64));
    LPD_REQUIRE(ldp % 4 == 0 && ldq % 4 == 0 && ld2 % 4 == 0 && (!x1 || ld1 % 4 == 0));
    LPD_REQUIRE(ldp >= C1 && ldq >= C1 && ld2 >= C2 && (!x1 || ld1 >= C1));
    LPD_REQUIRE(((uintptr_t)p & 15) == 0 && ((uintptr_t)q & 15) == 0 && ((uintptr_t)x2 & 15) == 0 && ((uintptr_t)x1 & 15) == 0);
    LPD_REQUIRE(act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY);
    DgParams P;
    P.p = p; P.q = q; P.idx = idx; P.s1 = s1; P.t1 = t1; P.w2 = w2; P.s2 = s2; P.t2 = t2;
    P.x1 = x1; P.x2 = x2; P.ldp = ldp; P.ldq = ldq; P.ld1 = ld1; P.ld2 = ld2;
    P.total_pts = (long long)B * N; P.N = N; P.k = k; P.act = act; P.slope = slope;
    cudaStream_t st = as_stream(stream);
    if (C1 == 128) {
        if (k <= 20) return dg_launch<128, 128, 20>(P, st);
        return dg_launch<128, 128, 16>(P, st);
    }
    if (k <= 20) return dg_launch<64, 64, 20>(P, st);
    return dg_launch<64, 64, 16>(P, st);
}
