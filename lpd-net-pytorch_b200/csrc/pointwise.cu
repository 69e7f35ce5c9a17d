// Fused input layers of the LPD-Net feature nets: conv1 (D -> 64) + BN + act and conv2 (64 -> 64) + BN + act per point in
// ONE pass (reference util/lpdnet_model.py:231-232 for LPDNet, :86-87 for LPDNetOrign).  Strict fp32: the result feeds the
// feature-space kNN.  The hidden map never leaves the SM (shared memory); the second-layer weights live in registers.
// (Two separate FFMA GEMMs moved the 64-wide hidden map through HBM and ran at 22 TFLOP/s: 0.16 ms per 64 clouds.)
#include "common.cuh"

namespace lpd {

constexpr int PW_THREADS = 128;
constexpr int PW_MAXD = 8;
constexpr int PW_STRIDE = 68;        // hidden-row stride in floats: 16-byte aligned rows, conflict-free STS.128

// Per warp, 32 points at a time:
//   phase 1  lane = point: the 64 hidden values h[c] = act(s1[c] * (w1[c] . x) + t1[c]) go to shared memory, row = point;
//   phase 2  lane = OUTPUT CHANNEL PAIR (o = lane, lane + 32), whose two rows of W2 (128 floats) live in registers for the whole
//            kernel: the hidden row of a point is read as 16 broadcast LDS.128 and multiplied into the lane's two accumulators, four
//            points in flight (eight independent fmaf chains).  Every output is the fmaf chain over c ascending, as before:
//            bit-identical features.
// The first version of this kernel kept the POINT in the lane and broadcast W2 out of shared memory: 1024 LDS.128 per point-warp, two
// wavefronts each, 87 % of the shared-memory pipe (ncu) and 0.104 ms per 64 clouds.  Here a point costs 16 LDS.128 + 128 FFMA per
// warp and its 64 outputs leave as two coalesced 128-byte stores, no staging.
__global__ void __launch_bounds__(PW_THREADS)
pointwise_mlp2_kernel(const float* __restrict__ x, int ldx, int D, long long M, const float* __restrict__ w1,
                      const float* __restrict__ s1, const float* __restrict__ t1, const float* __restrict__ w2,
                      const float* __restrict__ s2, const float* __restrict__ t2, float neg_slope, float* __restrict__ out, int ldo) {
    __shared__ __align__(16) float w1s[64 * PW_MAXD];
    __shared__ __align__(16) float s1s[64], t1s[64];
    __shared__ __align__(16) float hs_all[(PW_THREADS / 32) * 32 * PW_STRIDE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* hs = hs_all + warp * 32 * PW_STRIDE;
    for (int i = threadIdx.x; i < 64 * PW_MAXD; i += PW_THREADS) {
        const int c = i / PW_MAXD, d = i % PW_MAXD;
        w1s[i] = d < D ? __ldg(w1 + c * D + d) : 0.f;              // rows padded to PW_MAXD (the padding multiplies zeros)
    }
    if (threadIdx.x < 64) { s1s[threadIdx.x] = __ldg(s1 + threadIdx.x); t1s[threadIdx.x] = __ldg(t1 + threadIdx.x); }
    float wa[64], wb[64];                                          // rows lane and lane + 32 of W2 [o][c]
#pragma unroll
    for (int c4 = 0; c4 < 16; ++c4) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(w2 + lane * 64) + c4), b = __ldg(reinterpret_cast<const float4*>(w2 + (lane + 32) * 64) + c4);
        wa[4 * c4] = a.x; wa[4 * c4 + 1] = a.y; wa[4 * c4 + 2] = a.z; wa[4 * c4 + 3] = a.w;
        wb[4 * c4] = b.x; wb[4 * c4 + 1] = b.y; wb[4 * c4 + 2] = b.z; wb[4 * c4 + 3] = b.w;
    }
    const float sa = __ldg(s2 + lane), ta = __ldg(t2 + lane), sb = __ldg(s2 + lane + 32), tb = __ldg(t2 + lane + 32);
    __syncthreads();
    const long long nwarps = (long long)gridDim.x * (PW_THREADS / 32);
    for (long long p0 = ((long long)blockIdx.x * (PW_THREADS / 32) + warp) * 32; p0 < M; p0 += nwarps * 32) {
        // ---- phase 1: lane = point ----
        const long long pt = p0 + lane;
        __syncwarp();                                              // the previous tile's rows have been consumed
        if (pt < M) {
            float xin[PW_MAXD];
#pragma unroll
            for (int d = 0; d < PW_MAXD; ++d) xin[d] = d < D ? __ldg(x + pt * ldx + d) : 0.f;
            float4* hrow = reinterpret_cast<float4*>(hs + lane * PW_STRIDE);
#pragma unroll 4
            for (int c4 = 0; c4 < 16; ++c4) {
                float h[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int c = 4 * c4 + u;
                    float a = 0.f;
                    const float4 wl = *reinterpret_cast<const float4*>(w1s + c * PW_MAXD);
                    a = fmaf(xin[0], wl.x, a);
                    if (D > 1) a = fmaf(xin[1], wl.y, a);
                    if (D > 2) a = fmaf(xin[2], wl.z, a);
                    if (D > 3) a = fmaf(xin[3], wl.w, a);
                    if (D > 4) {
                        const float4 wh = *reinterpret_cast<const float4*>(w1s + c * PW_MAXD + 4);
                        a = fmaf(xin[4], wh.x, a);
                        if (D > 5) a = fmaf(xin[5], wh.y, a);
                        if (D > 6) a = fmaf(xin[6], wh.z, a);
                        if (D > 7) a = fmaf(xin[7], wh.w, a);
                    }
                    const float v = fmaf(s1s[c], a, t1s[c]);
                    h[u] = fmaxf(v, v * neg_slope);
                }
                hrow[c4] = make_float4(h[0], h[1], h[2], h[3]);
            }
        }
        __syncwarp();
        // ---- phase 2: lane = output channels lane and lane + 32, four points in flight ----
        const int npts = (int)((M - p0) < 32 ? (M - p0) : 32);
#pragma unroll 1
        for (int q0 = 0; q0 < npts; q0 += 4) {
            float a0[4] = {0.f, 0.f, 0.f, 0.f}, a1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c4 = 0; c4 < 16; ++c4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float4 h = *reinterpret_cast<const float4*>(hs + (q0 + u) * PW_STRIDE + 4 * c4);   // warp broadcast
                    a0[u] = fmaf(h.x, wa[4 * c4], a0[u]); a1[u] = fmaf(h.x, wb[4 * c4], a1[u]);
                    a0[u] = fmaf(h.y, wa[4 * c4 + 1], a0[u]); a1[u] = fmaf(h.y, wb[4 * c4 + 1], a1[u]);
                    a0[u] = fmaf(h.z, wa[4 * c4 + 2], a0[u]); a1[u] = fmaf(h.z, wb[4 * c4 + 2], a1[u]);
                    a0[u] = fmaf(h.w, wa[4 * c4 + 3], a0[u]); a1[u] = fmaf(h.w, wb[4 * c4 + 3], a1[u]);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (q0 + u < npts) {
                    float v0 = fmaf(sa, a0[u], ta), v1 = fmaf(sb, a1[u], tb);
                    v0 = fmaxf(v0, v0 * neg_slope); v1 = fmaxf(v1, v1 * neg_slope);
                    float* o = out + (p0 + q0 + u) * ldo;
                    o[lane] = v0;
                    o[lane + 32] = v1;
                }
            }
        }
    }
}

}  // namespace lpd

extern "C" int lpd_pointwise_mlp2(const float* x, int ldx, int D, long long M, const float* w1, const float* s1, const float* t1,
                                  const float* w2, const float* s2, const float* t2, int act, float slope, float* out, int ldo,
                                  void* stream) {
    using namespace lpd;
    LPD_REQUIRE(x && w1 && s1 && t1 && w2 && s2 && t2 && out && M >= 1);
    LPD_REQUIRE(D >= 1 && D <= PW_MAXD && ldx >= D && ldo >= 64);
    LPD_REQUIRE(act_is_slope(act, slope));
    const float neg_slope = act_neg_slope(act, slope);
    long long blocks = (M + PW_THREADS - 1) / PW_THREADS;
    if (blocks > 148 * 3) blocks = 148 * 3;                   // persistent: three resident blocks per SM (register-bound), W2 loaded once per thread
    pointwise_mlp2_kernel<<<(int)blocks, PW_THREADS, 0, as_stream(stream)>>>(x, ldx, D, M, w1, s1, t1, w2, s2, t2, neg_slope, out, ldo);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}
