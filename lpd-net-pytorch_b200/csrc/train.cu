// Train-mode kernels: batch-statistics BatchNorm (forward statistics, apply, backward), the train-mode EdgeConv
// pieces (edge statistics / arg-extremum, edge materialisation, backward with neighbour scatter), fused Adam.
// Replaces, in train() mode, nn.BatchNorm{1,2}d + activation (lpdnet_model.py:168-191,231-262; PointNetVlad.py:33,39,97),
// the autograd of get_graph_feature + conv + max (lpdnet_model.py:246-258) and torch.optim.Adam
// (train_pointnetvlad.py:57,129-130,158-159).
//
// Statistics are accumulated in fp64 (per-thread double accumulators, deterministic fixed-order tree: per-block partials
// [nparts][2][C] reduced by one thread per channel), because the naive fp32 E[z^2]-E[z]^2 cancels (SURVEY App. A.3).
//
// The kernels that touch the [B*N*k, C] edge tensors of a dense edge layer are templated on the storage type T of those
// tensors: fp32, or fp16 for the "f16" train precision mode (include/lpd_b200.h, "f16 storage of the edge tensors").  The
// fp16 forms compute in fp32 exactly as the fp32 forms do, on the values the fp16 storage holds; only loads and stores differ.
#include <cuda_fp16.h>

#include "common.cuh"

namespace lpd {

constexpr int TR_THREADS = 256;
constexpr int EDGE_U = 5;         // neighbour rows gathered per thread before any of them is consumed (k = 20: four rounds)
constexpr int GRAD_EXP_MAX = 100; // |E| bound of the gradient scale 2^E of the fp16 edge gradients (2^+-100 are normal fp32 numbers)

template <typename T> constexpr bool is_half_v = sizeof(T) == 2;

// V consecutive values (V = 4 or 8) of a row, to / from fp32 registers: fp32 as V/4 float4, fp16 as one 8- or 16-byte vector.
// ldg_vec reads through the read-only path, ld_vec with a plain load (buffers that the same kernel also writes).
template <int V> __device__ __forceinline__ void ldg_vec(const float* __restrict__ p, float (&v)[V]) {
#pragma unroll
    for (int i = 0; i < V / 4; ++i) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p) + i);
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
}
template <int V> __device__ __forceinline__ void ld_vec(const float* p, float (&v)[V]) {
#pragma unroll
    for (int i = 0; i < V / 4; ++i) {
        const float4 t = reinterpret_cast<const float4*>(p)[i];
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
    }
}
template <int V> __device__ __forceinline__ void st_vec(float* p, const float (&v)[V]) {
#pragma unroll
    for (int i = 0; i < V / 4; ++i) reinterpret_cast<float4*>(p)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
template <int V> __device__ __forceinline__ void h2f_vec(const uint32_t (&w)[V / 2], float (&v)[V]) {
#pragma unroll
    for (int i = 0; i < V / 2; ++i) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
        v[2 * i] = f.x; v[2 * i + 1] = f.y;
    }
}
template <int V> __device__ __forceinline__ void ldg_vec(const __half* __restrict__ p, float (&v)[V]) {
    uint32_t w[V / 2];
    if constexpr (V == 8) { const uint4 t = __ldg(reinterpret_cast<const uint4*>(p)); w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w; }
    else { const uint2 t = __ldg(reinterpret_cast<const uint2*>(p)); w[0] = t.x; w[1] = t.y; }
    h2f_vec<V>(w, v);
}
template <int V> __device__ __forceinline__ void ld_vec(const __half* p, float (&v)[V]) {
    uint32_t w[V / 2];
    if constexpr (V == 8) { const uint4 t = *reinterpret_cast<const uint4*>(p); w[0] = t.x; w[1] = t.y; w[2] = t.z; w[3] = t.w; }
    else { const uint2 t = *reinterpret_cast<const uint2*>(p); w[0] = t.x; w[1] = t.y; }
    h2f_vec<V>(w, v);
}
template <int V> __device__ __forceinline__ void st_vec(__half* p, const float (&v)[V]) {      // round to nearest
    uint32_t w[V / 2];
#pragma unroll
    for (int i = 0; i < V / 2; ++i) { const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]); w[i] = *reinterpret_cast<const uint32_t*>(&h); }
    if constexpr (V == 8) *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
    else *reinterpret_cast<uint2*>(p) = make_uint2(w[0], w[1]);
}
// V per-channel arg bytes (uchar4 or 8 bytes)
template <int V> __device__ __forceinline__ void st_arg(uint8_t* p, const int (&b)[V]) {
    if constexpr (V == 4) *reinterpret_cast<uchar4*>(p) = make_uchar4(b[0], b[1], b[2], b[3]);
    else *reinterpret_cast<uint2*>(p) = make_uint2((uint32_t)b[0] | (uint32_t)b[1] << 8 | (uint32_t)b[2] << 16 | (uint32_t)b[3] << 24,
                                                    (uint32_t)b[4] | (uint32_t)b[5] << 8 | (uint32_t)b[6] << 16 | (uint32_t)b[7] << 24);
}
template <int V> __device__ __forceinline__ void ld_arg(const uint8_t* p, int (&b)[V]) {
    if constexpr (V == 4) { const uchar4 a4 = *reinterpret_cast<const uchar4*>(p); b[0] = a4.x; b[1] = a4.y; b[2] = a4.z; b[3] = a4.w; }
    else {
        const uint2 t = *reinterpret_cast<const uint2*>(p);
#pragma unroll
        for (int u = 0; u < 4; ++u) { b[u] = (t.x >> (8 * u)) & 0xff; b[4 + u] = (t.y >> (8 * u)) & 0xff; }
    }
}

// order-preserving uint32 key of a float (unsigned compare of keys = float compare), for column min / max with integer atomics
__device__ __forceinline__ uint32_t f2key(float f) { const uint32_t b = __float_as_uint(f); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__device__ __forceinline__ float key2f(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// d act(v) / d v for the activations that follow a BatchNorm on the path.  GATE: out = aux * sigmoid(v).
__device__ __forceinline__ float act_grad(float v, int act, float slope, float aux) {
    switch (act) {
        case LPD_ACT_RELU: return v > 0.f ? 1.f : 0.f;
        case LPD_ACT_LEAKY: return v > 0.f ? 1.f : slope;
        case LPD_ACT_SIGMOID: { const float s = 1.f / (1.f + expf(-v)); return s * (1.f - s); }
        case LPD_ACT_GATE: { const float s = 1.f / (1.f + expf(-v)); return aux * s * (1.f - s); }
        default: return 1.f;
    }
}

// NONE / RELU / LEAKY are piecewise linear: act(v) = v > 0 ? v : v * gneg and act'(v) = v > 0 ? 1 : gneg with gneg = 1 / 0 / slope.
// The hot loops test this once per kernel (uniform branch) instead of switching per element.
__device__ __forceinline__ bool act_is_step(int act) { return act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY; }
__device__ __forceinline__ float act_gneg(int act, float slope) { return act == LPD_ACT_LEAKY ? slope : (act == LPD_ACT_RELU ? 0.f : 1.f); }

// Block-level reduction of per-thread column accumulators.  Threads are laid out as (lane, g): g = column group of
// V channels, `lanes` row lanes.  Writes partial[part][0][C] (s1) and partial[part][1][C] (s2).
template <int V = 4>
__device__ __forceinline__ void block_reduce_cols(double (&s1)[V], double (&s2)[V], int lane, int lanes, int g,
                                                  int C, bool active, double* __restrict__ partial, int part) {
    __shared__ double red[2][1024];               // one slot per column of the block's tile (<= 1024 columns)
    // serial fixed-order accumulation over the row lanes: lane 0 owns the result (deterministic)
    for (int l = 1; l < lanes; ++l) {
        __syncthreads();
        if (active && lane == l) {
#pragma unroll
            for (int u = 0; u < V; ++u) { red[0][g * V + u] = s1[u]; red[1][g * V + u] = s2[u]; }
        }
        __syncthreads();
        if (active && lane == 0) {
#pragma unroll
            for (int u = 0; u < V; ++u) { s1[u] += red[0][g * V + u]; s2[u] += red[1][g * V + u]; }
        }
    }
    if (active && lane == 0) {
        double* o = partial + (size_t)part * 2 * C;
#pragma unroll
        for (int u = 0; u < V; ++u) { o[g * V + u] = s1[u]; o[C + g * V + u] = s2[u]; }
    }
}

// ---- forward statistics: partial[b][0][c] = sum z, partial[b][1][c] = sum z^2 over the block's rows ------------
// grid (nparts, ceil(C/1024)); a block covers <= 1024 columns.  T = fp16 (V = 8): also the column min / max as order keys,
// minmax[0][c] (atomicMin, initialised to ~0) and minmax[1][c] (atomicMax, initialised to 0); and an entry at the fp16 limit
// (|z| >= 65504: where lpd_gemm_f16 saturates) counts as NaN, so an overflowing product makes the statistics non-finite.
template <typename T, int V>
__global__ void __launch_bounds__(TR_THREADS)
col_stats_kernel(const T* __restrict__ z, long long rows, int C, int ld, double* __restrict__ partial, uint32_t* __restrict__ minmax) {
    constexpr int VS = V == 4 ? 2 : 3;
    const int c0 = blockIdx.y * 1024;
    const int Cb = min(1024, C - c0);
    const int cg = Cb >> VS;
    const int lanes = max(1, TR_THREADS / cg);
    const int lane = threadIdx.x / cg, g = threadIdx.x % cg;
    const bool active = lane < lanes;
    double s1[V], s2[V];
    float mn[V], mx[V];
#pragma unroll
    for (int u = 0; u < V; ++u) { s1[u] = 0; s2[u] = 0; mn[u] = INFINITY; mx[u] = -INFINITY; }
    const long long rpb = (rows + gridDim.x - 1) / gridDim.x;
    const long long r0 = (long long)blockIdx.x * rpb, r1 = min(rows, r0 + rpb);
    if (active) {
        for (long long r = r0 + lane; r < r1; r += lanes) {
            float v[V];
            ldg_vec<V>(z + r * ld + c0 + g * V, v);
#pragma unroll
            for (int u = 0; u < V; ++u) {
                if constexpr (is_half_v<T>) {
                    mn[u] = fminf(mn[u], v[u]); mx[u] = fmaxf(mx[u], v[u]);
                    if (fabsf(v[u]) >= 65504.f) v[u] = __int_as_float(0x7fffffff);
                }
                s1[u] += v[u];
                s2[u] += (double)v[u] * v[u];
            }
        }
    }
    // partial layout is [nparts][2][C]; this block writes columns c0..c0+Cb
    block_reduce_cols<V>(s1, s2, lane, lanes, g, C, active, partial + c0, blockIdx.x);
    if constexpr (is_half_v<T>) {
        __shared__ uint32_t kmm[2][1024];
        for (int i = threadIdx.x; i < Cb; i += blockDim.x) { kmm[0][i] = ~0u; kmm[1][i] = 0u; }
        __syncthreads();
        if (active) {
#pragma unroll
            for (int u = 0; u < V; ++u) { atomicMin(&kmm[0][g * V + u], f2key(mn[u])); atomicMax(&kmm[1][g * V + u], f2key(mx[u])); }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < Cb; i += blockDim.x) {
            if (kmm[0][i] != ~0u) atomicMin(minmax + c0 + i, kmm[0][i]);
            if (kmm[1][i] != 0u) atomicMax(minmax + C + c0 + i, kmm[1][i]);
        }
    }
}

// warp-cooperative fixed-order sum of partial[p * stride + off] over p: lane l takes p = l, l+32, ... then a shuffle tree
// (the order is fixed by the launch geometry, so the result is deterministic)
__device__ __forceinline__ double warp_sum_parts(const double* __restrict__ partial, int nparts, size_t stride, size_t off) {
    const int lane = threadIdx.x & 31;
    double s = 0;
    for (int p = lane; p < nparts; p += 32) s += partial[(size_t)p * stride + off];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
    return s;
}

// ---- finalize: batch mean / biased var -> (scale, shift, mean, invstd), running-stat update.  One warp per channel. ------
__global__ void __launch_bounds__(256)
bn_finalize_kernel(const double* __restrict__ partial, int nparts, double count, int C,
                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float momentum,
                   float* __restrict__ running_mean, float* __restrict__ running_var,
                   float* __restrict__ out /* [4][C]: scale, shift, mean, invstd */) {
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (c >= C) return;
    const double s1 = warp_sum_parts(partial, nparts, (size_t)2 * C, c);
    const double s2 = warp_sum_parts(partial, nparts, (size_t)2 * C, (size_t)C + c);
    if ((threadIdx.x & 31) != 0) return;
    const double mean = s1 / count;
    double var = s2 / count - mean * mean;
    if (var < 0) var = 0;
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    const float sc = (gamma ? gamma[c] : 1.f) * invstd;
    out[c] = sc;
    out[C + c] = (beta ? beta[c] : 0.f) - (float)mean * sc;
    out[2 * C + c] = (float)mean;
    out[3 * C + c] = invstd;
    if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    if (running_var) {
        const double unb = count > 1 ? var * count / (count - 1) : var;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unb;
    }
}

// out[i] = sum over parts of partial[p][i]   (i < n), fp64 -> fp32.  One warp per output.
__global__ void __launch_bounds__(256)
colsum_finalize_kernel(const double* __restrict__ partial, int nparts, int n, float* __restrict__ out) {
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= n) return;
    const double s = warp_sum_parts(partial, nparts, (size_t)n, i);
    if ((threadIdx.x & 31) == 0) out[i] = (float)s;
}

// ---- elementwise affine + activation: out = act(scale * z + shift) (GATE: aux * sigmoid) ---------------------------
__global__ void __launch_bounds__(TR_THREADS)
affine_act_kernel(const float* __restrict__ z, long long rows, int C, int ldz, const float* __restrict__ scale,
                  const float* __restrict__ shift, int act, float slope, const float* __restrict__ aux, int ldaux,
                  float* __restrict__ out, int ldo) {
    const int cg = C >> 2;
    const long long total = rows * cg;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / cg;
        const int c = (int)(e % cg) * 4;
        const float4 v = *reinterpret_cast<const float4*>(z + r * ldz + c);
        const float4 s = scale ? __ldg(reinterpret_cast<const float4*>(scale + c)) : make_float4(1.f, 1.f, 1.f, 1.f);
        const float4 t = shift ? __ldg(reinterpret_cast<const float4*>(shift + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 o = make_float4(fmaf(s.x, v.x, t.x), fmaf(s.y, v.y, t.y), fmaf(s.z, v.z, t.z), fmaf(s.w, v.w, t.w));
        if (act == LPD_ACT_GATE) {
            const float4 a = *reinterpret_cast<const float4*>(aux + r * ldaux + c);
            o.x = a.x * (1.f / (1.f + expf(-o.x))); o.y = a.y * (1.f / (1.f + expf(-o.y)));
            o.z = a.z * (1.f / (1.f + expf(-o.z))); o.w = a.w * (1.f / (1.f + expf(-o.w)));
        } else {
            o.x = apply_act(o.x, act, slope); o.y = apply_act(o.y, act, slope);
            o.z = apply_act(o.z, act, slope); o.w = apply_act(o.w, act, slope);
        }
        *reinterpret_cast<float4*>(out + r * ldo + c) = o;
    }
}

// ---- BN backward, pass 1: S1 = sum dzbn, S2 = sum dzbn * xhat ; dzbn = dy * act'(scale z + shift) ------------------
__global__ void __launch_bounds__(TR_THREADS)
bn_bwd_reduce_kernel(const float* __restrict__ dy, int lddy, const float* __restrict__ z, int ldz, long long rows, int C,
                     const float* __restrict__ bn /* [4][C] */, int act, float slope, const float* __restrict__ aux, int ldaux,
                     double* __restrict__ partial) {
    const int c0 = blockIdx.y * 1024;
    const int Cb = min(1024, C - c0);
    const int cg = Cb >> 2;
    const int lanes = max(1, TR_THREADS / cg);
    const int lane = threadIdx.x / cg, g = threadIdx.x % cg;
    const bool active = lane < lanes;
    const int c = c0 + g * 4;
    double s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
    const long long rpb = (rows + gridDim.x - 1) / gridDim.x;
    const long long r0 = (long long)blockIdx.x * rpb, r1 = min(rows, r0 + rpb);
    const bool step = act_is_step(act);
    const float gneg = act_gneg(act, slope);
    if (active) {
        float sc[4], sh[4], mu[4], is[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { sc[u] = bn[c + u]; sh[u] = bn[C + c + u]; mu[u] = bn[2 * C + c + u]; is[u] = bn[3 * C + c + u]; }
        for (long long r = r0 + lane; r < r1; r += lanes) {
            const float4 zv4 = __ldg(reinterpret_cast<const float4*>(z + r * ldz + c));
            const float4 dv4 = __ldg(reinterpret_cast<const float4*>(dy + r * lddy + c));
            float4 av4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (act == LPD_ACT_GATE) av4 = __ldg(reinterpret_cast<const float4*>(aux + r * ldaux + c));
            const float zv[4] = {zv4.x, zv4.y, zv4.z, zv4.w}, dv[4] = {dv4.x, dv4.y, dv4.z, dv4.w}, av[4] = {av4.x, av4.y, av4.z, av4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float pre = fmaf(sc[u], zv[u], sh[u]);
                const float d = dv[u] * (step ? (pre > 0.f ? 1.f : gneg) : act_grad(pre, act, slope, av[u]));
                const float xh = (zv[u] - mu[u]) * is[u];
                s1[u] += d;
                s2[u] += (double)d * xh;
            }
        }
    }
    block_reduce_cols(s1, s2, lane, lanes, g, C, active, partial + c0, blockIdx.x);
}

// ---- BN backward, pass 2: dz = scale * (dzbn - S1/count - xhat * S2/count) ------------------------------------------
__global__ void __launch_bounds__(TR_THREADS)
bn_bwd_apply_kernel(const float* __restrict__ dy, int lddy, const float* __restrict__ z, int ldz, long long rows, int C,
                    const float* __restrict__ bn, const float* __restrict__ S /* [2][C] */, float inv_count, int act, float slope,
                    const float* __restrict__ aux, int ldaux, float* __restrict__ dz, int lddz) {
    // thread = (row lane, group of 4 channels): the per-channel constants are loaded once, rows are walked with a grid stride
    const int c0 = blockIdx.y * 1024;
    const int Cb = min(1024, C - c0);
    const int cg = Cb >> 2;
    const int lanes = max(1, TR_THREADS / cg);
    const int lane = threadIdx.x / cg, g = threadIdx.x % cg;
    if (lane >= lanes) return;
    const int c = c0 + g * 4;
    const bool step = act_is_step(act);
    const float gneg = act_gneg(act, slope);
    float sc[4], sh[4], mu[4], is[4], k1[4], k2[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        sc[u] = __ldg(bn + c + u); sh[u] = __ldg(bn + C + c + u); mu[u] = __ldg(bn + 2 * C + c + u); is[u] = __ldg(bn + 3 * C + c + u);
        k1[u] = __ldg(S + c + u) * inv_count; k2[u] = __ldg(S + C + c + u) * inv_count;
    }
    for (long long r = (long long)blockIdx.x * lanes + lane; r < rows; r += (long long)gridDim.x * lanes) {
        const float4 zv4 = *reinterpret_cast<const float4*>(z + r * ldz + c);
        const float4 dv4 = *reinterpret_cast<const float4*>(dy + r * lddy + c);
        float4 av4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (act == LPD_ACT_GATE) av4 = *reinterpret_cast<const float4*>(aux + r * ldaux + c);
        const float zv[4] = {zv4.x, zv4.y, zv4.z, zv4.w}, dv[4] = {dv4.x, dv4.y, dv4.z, dv4.w}, av[4] = {av4.x, av4.y, av4.z, av4.w};
        float o[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float pre = fmaf(sc[u], zv[u], sh[u]);
            const float d = dv[u] * (step ? (pre > 0.f ? 1.f : gneg) : act_grad(pre, act, slope, av[u]));
            const float xh = (zv[u] - mu[u]) * is[u];
            o[u] = sc[u] * (d - k1[u] - xh * k2[u]);
        }
        *reinterpret_cast<float4*>(dz + r * lddz + c) = make_float4(o[0], o[1], o[2], o[3]);
    }
}

// =====================================================================================================================
// Train-mode EdgeConv.  Edge pre-activation z[e=(i,m)][c] = p[j(i,m)][c] + q[i][c]  (exact decomposition, App. A.3).
// Thread (point, 4 channels); a block walks points with a grid stride so that statistics reduce per block.
// =====================================================================================================================
struct EdgeArgs {
    const float* p; int ldp; const float* q; int ldq; const int* idx;
    long long M; int N, k, C;
};

// per point: zsel = q + (gamma >= 0 ? max : min)_m p_j, arg = first m reaching it; block partials of sum z, sum z^2.
__global__ void __launch_bounds__(TR_THREADS)
edge_sel_stats_kernel(EdgeArgs a, const float* __restrict__ gamma, float* __restrict__ zsel, int ldz,
                      uint8_t* __restrict__ arg, double* __restrict__ partial) {
    const int cg = a.C >> 2;
    const int lanes = TR_THREADS / cg;
    const int lane = threadIdx.x / cg, g = threadIdx.x % cg;
    const bool active = lane < lanes;
    const int c = g * 4;
    double s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
    if (active) {
        // the extremum is a MAXIMUM of sg * v with sg = +-1 (sign of gamma): one compare + two selects per element, no branch
        float sg[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) sg[u] = (gamma ? __ldg(gamma + c + u) : 1.f) >= 0.f ? 1.f : -1.f;
        for (long long pt = (long long)blockIdx.x * lanes + lane; pt < a.M; pt += (long long)gridDim.x * lanes) {
            const long long cloud0 = (pt / a.N) * a.N;
            const int* ip = a.idx + pt * a.k;
            float best[4], sum[4] = {0, 0, 0, 0}, sq[4] = {0, 0, 0, 0};
            int bi[4] = {0, 0, 0, 0};
#pragma unroll
            for (int u = 0; u < 4; ++u) best[u] = -INFINITY;           // of sg * v
            // EDGE_U neighbour rows in flight per thread (the index -> row dependency chain was the whole cost of this loop);
            // the accumulation order stays m ascending
            for (int m0 = 0; m0 < a.k; m0 += EDGE_U) {
                int jj[EDGE_U];
                float4 vv[EDGE_U];
#pragma unroll
                for (int w = 0; w < EDGE_U; ++w) jj[w] = (m0 + w < a.k) ? __ldg(ip + m0 + w) : 0;
#pragma unroll
                for (int w = 0; w < EDGE_U; ++w) vv[w] = __ldg(reinterpret_cast<const float4*>(a.p + (cloud0 + jj[w]) * a.ldp + c));
#pragma unroll
                for (int w = 0; w < EDGE_U; ++w) {
                    const int m = m0 + w;
                    if (m < a.k) {
                        const float v[4] = {vv[w].x, vv[w].y, vv[w].z, vv[w].w};
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float wv = v[u] * sg[u];                      // exact
                            const bool better = wv > best[u];                   // strict: the first m reaching the extremum
                            best[u] = better ? wv : best[u];
                            bi[u] = better ? m : bi[u];
                            sum[u] += v[u];
                            sq[u] = fmaf(v[u], v[u], sq[u]);
                        }
                    }
                }
            }
            float qv[4] = {0.f, 0.f, 0.f, 0.f};
            if (a.q) { const float4 t = __ldg(reinterpret_cast<const float4*>(a.q + pt * a.ldq + c)); qv[0] = t.x; qv[1] = t.y; qv[2] = t.z; qv[3] = t.w; }
            float o[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                o[u] = best[u] * sg[u] + qv[u];
                const double qd = qv[u];
                s1[u] += (double)sum[u] + a.k * qd;
                s2[u] += (double)sq[u] + 2.0 * qd * (double)sum[u] + a.k * qd * qd;
            }
            *reinterpret_cast<float4*>(zsel + pt * ldz + c) = make_float4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<uchar4*>(arg + pt * a.C + c) = make_uchar4(bi[0], bi[1], bi[2], bi[3]);
        }
    }
    block_reduce_cols(s1, s2, lane, lanes, g, a.C, active, partial, blockIdx.x);
}

// y[(i,m)][c] = act(scale * (p_j + q_i) + shift), stored as T (fp16: rounded to nearest); a thread covers V channels
template <typename T, int V>
__global__ void __launch_bounds__(TR_THREADS)
edge_materialize_kernel(EdgeArgs a, const float* __restrict__ scale, const float* __restrict__ shift, int act, float slope,
                        T* __restrict__ y) {
    constexpr int VS = V == 4 ? 2 : 3;
    const int cg = a.C >> VS;
    const long long total = a.M * a.k * cg;
    const bool step = act_is_step(act);
    const float gneg = act_gneg(act, slope);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long edge = e / cg;
        const int c = (int)(e % cg) * V;
        const long long pt = edge / a.k;
        const long long cloud0 = (pt / a.N) * a.N;
        const int j = __ldg(a.idx + edge);
        float pv[V], qv[V], s[V], t[V], o[V];
        ldg_vec<V>(a.p + (cloud0 + j) * a.ldp + c, pv);
#pragma unroll
        for (int u = 0; u < V; ++u) qv[u] = 0.f;
        if (a.q) ldg_vec<V>(a.q + pt * a.ldq + c, qv);
        ldg_vec<V>(scale + c, s);
        ldg_vec<V>(shift + c, t);
#pragma unroll
        for (int u = 0; u < V; ++u) o[u] = fmaf(s[u], pv[u] + qv[u], t[u]);
        if (step) {
#pragma unroll
            for (int u = 0; u < V; ++u) o[u] = o[u] > 0.f ? o[u] : o[u] * gneg;
        } else {
#pragma unroll
            for (int u = 0; u < V; ++u) o[u] = apply_act(o[u], act, slope);
        }
        st_vec<V>(y + edge * a.C + c, o);
    }
}

// dense edge tensor z [M][k][C] (stored as T): zsel = (gamma >= 0 ? max : min)_m z, arg = first m reaching it
template <typename T, int V>
__global__ void __launch_bounds__(TR_THREADS)
edge_sel_dense_kernel(const T* __restrict__ z, long long M, int k, int C, const float* __restrict__ gamma,
                      float* __restrict__ zsel, int ldz, uint8_t* __restrict__ arg) {
    constexpr int VS = V == 4 ? 2 : 3;
    const int cg = C >> VS;
    const long long total = M * cg;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long pt = e / cg;
        const int c = (int)(e % cg) * V;
        float sg[V], best[V];                                 // maximum of sg * v, sg = sign of gamma (see edge_sel_stats_kernel)
        int bi[V];
#pragma unroll
        for (int u = 0; u < V; ++u) { sg[u] = (gamma ? __ldg(gamma + c + u) : 1.f) >= 0.f ? 1.f : -1.f; best[u] = -INFINITY; bi[u] = 0; }
        for (int m0 = 0; m0 < k; m0 += EDGE_U) {
            float vv[EDGE_U][V];
#pragma unroll
            for (int w = 0; w < EDGE_U; ++w) {
                if (m0 + w < k) ldg_vec<V>(z + (pt * k + m0 + w) * C + c, vv[w]);
                else {
#pragma unroll
                    for (int u = 0; u < V; ++u) vv[w][u] = 0.f;
                }
            }
#pragma unroll
            for (int w = 0; w < EDGE_U; ++w) {
                const int m = m0 + w;
                if (m < k) {
#pragma unroll
                    for (int u = 0; u < V; ++u) {
                        const float wv = vv[w][u] * sg[u];
                        const bool better = wv > best[u];
                        best[u] = better ? wv : best[u];
                        bi[u] = better ? m : bi[u];
                    }
                }
            }
        }
        float o[V];
#pragma unroll
        for (int u = 0; u < V; ++u) o[u] = best[u] * sg[u];
        st_vec<V>(zsel + pt * ldz + c, o);
        st_arg<V>(arg + pt * C + c, bi);
    }
}

// dense layer backward: dz[(i,m)][c] = scale * ([m == arg] * g[i][c] - S1/cnt - xhat(z) * S2/cnt), g = dx * act'(scale zsel + shift)
// (in place over z allowed).  T = fp16: z and dz are fp16 and dz is stored as fp16(gscale[0] * dz), gscale[0] = 2^E.
template <typename T, int V>
__global__ void __launch_bounds__(TR_THREADS)
edge_dense_bwd_apply_kernel(const T* z, long long M, int k, int C, const float* __restrict__ bn,
                            const float* __restrict__ S, float inv_count, int act, float slope,
                            const float* __restrict__ dx, int lddx, const float* __restrict__ zsel, int ldzs,
                            const uint8_t* __restrict__ arg, T* dz, const float* __restrict__ gscale) {
    constexpr int VS = V == 4 ? 2 : 3;
    const int cg = C >> VS;
    const long long total = M * cg;
    float g2 = 1.f;
    if constexpr (is_half_v<T>) g2 = __ldg(gscale);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long pt = e / cg;
        const int c = (int)(e % cg) * V;
        float sc[V], mu[V], is[V], gsel[V], k1[V], k2[V];
        int ar[V];
        ld_arg<V>(arg + pt * C + c, ar);
        float dxv[V], zsv[V];
        ldg_vec<V>(dx + pt * lddx + c, dxv);
        ldg_vec<V>(zsel + pt * ldzs + c, zsv);
#pragma unroll
        for (int u = 0; u < V; ++u) {
            sc[u] = __ldg(bn + c + u); mu[u] = __ldg(bn + 2 * C + c + u); is[u] = __ldg(bn + 3 * C + c + u);
            const float sh = __ldg(bn + C + c + u);
            gsel[u] = dxv[u] * act_grad(fmaf(sc[u], zsv[u], sh), act, slope, 0.f);
            k1[u] = __ldg(S + c + u) * inv_count;
            k2[u] = __ldg(S + C + c + u) * inv_count;
        }
        for (int m = 0; m < k; ++m) {
            float v[V];
            ld_vec<V>(z + (pt * k + m) * C + c, v);
            float o[V];
#pragma unroll
            for (int u = 0; u < V; ++u) {
                const float xh = (v[u] - mu[u]) * is[u];
                o[u] = sc[u] * ((m == ar[u] ? gsel[u] : 0.f) - k1[u] - xh * k2[u]);
                if constexpr (is_half_v<T>) o[u] *= g2;
            }
            st_vec<V>(dz + (pt * k + m) * C + c, o);
        }
    }
}

// 4 channels of a dy row: loaded raw (float4 / 4 halves), converted to fp32 where they are consumed, so that the loads of all
// EDGE_U rows are in flight first.  T = fp16 holds 2^E * dy, undone by the exact power-of-two multiply by dyscale = 2^-E.
__device__ __forceinline__ float4 ldg_dy4(const float* __restrict__ p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ uint2 ldg_dy4(const __half* __restrict__ p) { return __ldg(reinterpret_cast<const uint2*>(p)); }
__device__ __forceinline__ float4 dy4_f32(float4 v, float) { return v; }
__device__ __forceinline__ float4 dy4_f32(uint2 v, float s) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
    return make_float4(a.x * s, a.y * s, b.x * s, b.y * s);
}

// decomposed layer backward.  dzbn[(i,m)][c] = (dy[(i,m)][c] + [m == arg[i][c]] * dx[i][c]) * act'(scale (p_j + q_i) + shift)
//   REDUCE: block partials of S1 = sum dzbn, S2 = sum dzbn * xhat
//   APPLY : dz = scale * (dzbn - S1/cnt - xhat * S2/cnt) ; dq[i] = sum_m dz ; dp[j] += dz   (fp32 atomics)
// T: storage of dy (fp16: scaled by 2^E, dyscale[0] = 2^-E); p, q, dx, dp, dq stay fp32.
template <bool APPLY, typename T = float>
__global__ void __launch_bounds__(TR_THREADS)
edge_bwd_kernel(EdgeArgs a, const float* __restrict__ bn, int act, float slope,
                const float* __restrict__ dx, int lddx, const uint8_t* __restrict__ arg, const T* __restrict__ dy,
                const float* __restrict__ S, float inv_count, double* __restrict__ partial,
                float* __restrict__ dp, int lddp, float* __restrict__ dq, int lddq, const float* __restrict__ dyscale = nullptr) {
    const int cg = a.C >> 2;
    const int lanes = TR_THREADS / cg;
    const int lane = threadIdx.x / cg, g = threadIdx.x % cg;
    const bool active = lane < lanes;
    const int c = g * 4;
    const int C = a.C;
    double s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
    if (active) {
        float sc[4], sh[4], mu[4], is[4], k1[4] = {0, 0, 0, 0}, k2[4] = {0, 0, 0, 0};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            sc[u] = __ldg(bn + c + u); sh[u] = __ldg(bn + C + c + u); mu[u] = __ldg(bn + 2 * C + c + u); is[u] = __ldg(bn + 3 * C + c + u);
            if (APPLY) { k1[u] = __ldg(S + c + u) * inv_count; k2[u] = __ldg(S + C + c + u) * inv_count; }
        }
        // d act / d v of the edge layers' activations is a step function: 1 above zero, gneg below (NONE: 1, RELU: 0, LEAKY: slope)
        const float gneg = act == LPD_ACT_LEAKY ? slope : (act == LPD_ACT_RELU ? 0.f : 1.f);
        float sdy = 1.f;
        if constexpr (is_half_v<T>) sdy = __ldg(dyscale);
        for (long long pt = (long long)blockIdx.x * lanes + lane; pt < a.M; pt += (long long)gridDim.x * lanes) {
            const long long cloud0 = (pt / a.N) * a.N;
            const int* ip = a.idx + pt * a.k;
            float qv[4] = {0.f, 0.f, 0.f, 0.f}, dxv[4] = {0.f, 0.f, 0.f, 0.f};
            int ar[4] = {-1, -1, -1, -1};
            if (a.q) { const float4 t = __ldg(reinterpret_cast<const float4*>(a.q + pt * a.ldq + c)); qv[0] = t.x; qv[1] = t.y; qv[2] = t.z; qv[3] = t.w; }
            if (dx) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(dx + pt * lddx + c));
                dxv[0] = t.x; dxv[1] = t.y; dxv[2] = t.z; dxv[3] = t.w;
                const uchar4 a4 = *reinterpret_cast<const uchar4*>(arg + pt * C + c);
                ar[0] = a4.x; ar[1] = a4.y; ar[2] = a4.z; ar[3] = a4.w;
            }
            float dqa[4] = {0.f, 0.f, 0.f, 0.f};
            for (int m0 = 0; m0 < a.k; m0 += EDGE_U) {      // EDGE_U rows in flight, accumulation order unchanged (see above)
                int jj[EDGE_U];
                float4 pp[EDGE_U];
                decltype(ldg_dy4(dy)) dd[EDGE_U];
#pragma unroll
                for (int w = 0; w < EDGE_U; ++w) jj[w] = (m0 + w < a.k) ? __ldg(ip + m0 + w) : 0;
#pragma unroll
                for (int w = 0; w < EDGE_U; ++w) {
                    pp[w] = __ldg(reinterpret_cast<const float4*>(a.p + (cloud0 + jj[w]) * a.ldp + c));
                    dd[w] = {};
                    if (dy && m0 + w < a.k) dd[w] = ldg_dy4(dy + (pt * a.k + m0 + w) * C + c);
                }
#pragma unroll
                for (int w = 0; w < EDGE_U; ++w) {
                    const int m = m0 + w;
                    if (m < a.k) {
                        const float pv[4] = {pp[w].x, pp[w].y, pp[w].z, pp[w].w};
                        const float4 d4 = dy4_f32(dd[w], sdy);
                        const float dyv[4] = {d4.x, d4.y, d4.z, d4.w};
                        float o[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const float zz = pv[u] + qv[u];
                            const float d = (dyv[u] + (m == ar[u] ? dxv[u] : 0.f)) * (fmaf(sc[u], zz, sh[u]) > 0.f ? 1.f : gneg);
                            const float xh = (zz - mu[u]) * is[u];
                            if (APPLY) {
                                o[u] = sc[u] * (d - k1[u] - xh * k2[u]);
                                dqa[u] += o[u];
                            } else {
                                s1[u] += d;
                                s2[u] += (double)d * xh;
                            }
                        }
                        if (APPLY) atomicAdd(reinterpret_cast<float4*>(dp + (cloud0 + jj[w]) * lddp + c), make_float4(o[0], o[1], o[2], o[3]));
                    }
                }
            }
            if (APPLY && dq) *reinterpret_cast<float4*>(dq + pt * lddq + c) = make_float4(dqa[0], dqa[1], dqa[2], dqa[3]);
        }
    }
    if (!APPLY) block_reduce_cols(s1, s2, lane, lanes, g, C, active, partial, blockIdx.x);
}

// gather-only edges (get_graph_feature_Origin(cat=False), lpdnet_model.py:116-145): backward of e[(i,m)] = f[j(i,m)] is the
// scatter-add dp[j] += dy[(i,m)]  (the index_put_(accumulate=True) of torch's autograd)
__global__ void __launch_bounds__(TR_THREADS)
edge_scatter_add_kernel(const float* __restrict__ dy, const int* __restrict__ idx, long long M, int N, int k, int C,
                        float* __restrict__ dp, int lddp) {
    const int cg = C >> 2;
    const long long total = M * k * cg;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long edge = e / cg;
        const int c = (int)(e % cg) * 4;
        const long long pt = edge / k;
        const long long cloud0 = (pt / N) * N;
        const int j = __ldg(idx + edge);
        const float4 v = __ldg(reinterpret_cast<const float4*>(dy + edge * C + c));
        atomicAdd(reinterpret_cast<float4*>(dp + (cloud0 + j) * lddp + c), v);
    }
}

// ---- power-of-two scale of the fp16 edge gradients (lpd_edge_grad_scale_f16) --------------------------------------------
// pass 1: amax[c] = max_i |dx[i][c]| as float bits (non-negative floats order like their bits); amax zeroed first
__global__ void __launch_bounds__(TR_THREADS)
col_absmax_kernel(const float* __restrict__ dx, int lddx, long long M, int C, uint32_t* __restrict__ amax) {
    __shared__ uint32_t sm[1024];
    const int cg = C >> 2;
    const int lanes = TR_THREADS / cg;
    const int lane = threadIdx.x / cg, g = threadIdx.x % cg;
    for (int i = threadIdx.x; i < C; i += blockDim.x) sm[i] = 0u;
    __syncthreads();
    if (lane < lanes) {
        float m[4] = {0.f, 0.f, 0.f, 0.f};
        for (long long r = (long long)blockIdx.x * lanes + lane; r < M; r += (long long)gridDim.x * lanes) {
            float v[4];
            ldg_vec<4>(dx + r * lddx + g * 4, v);
#pragma unroll
            for (int u = 0; u < 4; ++u) m[u] = fabsf(v[u]) > m[u] || v[u] != v[u] ? fabsf(v[u]) : m[u];   // NaN wins
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) atomicMax(&sm[g * 4 + u], __float_as_uint(m[u]));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x)
        if (sm[i]) atomicMax(amax + i, sm[i]);
}

// pass 2 (one block): the bounds of include/lpd_b200.h -> E -> scale[0][:K] = 2^E, scale[1][:K] = 2^-E
__global__ void __launch_bounds__(256)
edge_grad_scale_kernel(const uint32_t* __restrict__ amax, int C, const float* __restrict__ bn, const float* __restrict__ S,
                       double inv_count, float gmax, const uint32_t* __restrict__ zminmax, const __half* __restrict__ w, int ldw,
                       int K, float* __restrict__ scale) {
    __shared__ double bz[1024];
    __shared__ double red[256];
    __shared__ int e_sh;
    double b = 0;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const double mean = bn[2 * C + c], is = bn[3 * C + c];
        const double X = fmax(fabs((double)key2f(zminmax[c]) - mean), fabs((double)key2f(zminmax[C + c]) - mean)) * is;
        const double v = fabs((double)bn[c]) * ((double)__uint_as_float(amax[c]) * gmax + fabs((double)S[c]) * inv_count
                                                + X * fabs((double)S[C + c]) * inv_count);
        bz[c] = v;
        b = (v > b || v != v) ? v : b;
    }
    __syncthreads();
    for (int kk = threadIdx.x; kk < K; kk += blockDim.x) {
        double s = 0;
        for (int c = 0; c < C; ++c) s += fabs((double)__half2float(w[(size_t)c * ldw + kk])) * bz[c];
        b = (s > b || s != s) ? s : b;
    }
    red[threadIdx.x] = b;
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = 0;
        for (int i = 0; i < (int)blockDim.x; ++i) m = (red[i] > m || red[i] != red[i]) ? red[i] : m;
        int E;
        if (!(m < INFINITY)) E = 0;                    // NaN / inf gradients: unscaled, they stay non-finite
        else if (m == 0) E = GRAD_EXP_MAX;
        else {
            int ex;
            frexp(m, &ex);                             // m < 2^ex  ->  2^E * m < 2^14
            E = min(GRAD_EXP_MAX, max(-GRAD_EXP_MAX, 14 - ex));
        }
        e_sh = E;
    }
    __syncthreads();
    const float up = ldexpf(1.f, e_sh), down = ldexpf(1.f, -e_sh);
    for (int i = threadIdx.x; i < K; i += blockDim.x) { scale[i] = up; scale[K + i] = down; }
}

// ---- Adam (torch.optim.Adam defaults: no amsgrad, L2 weight decay folded into the gradient) ------------------------
__global__ void __launch_bounds__(TR_THREADS)
adam_kernel(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
            float lr, float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt, float gscale) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float gi = g[i] * gscale;
        const float wi = w[i];
        if (wd != 0.f) gi = fmaf(wd, wi, gi);
        const float mi = b1 * m[i] + (1.f - b1) * gi;
        const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        w[i] = wi - (lr / bc1) * (mi / denom);
    }
}

// y += alpha * x   (strided rows)
__global__ void __launch_bounds__(TR_THREADS)
axpy_kernel(float* __restrict__ y, int ldy, const float* __restrict__ x, int ldx, long long rows, int C, float alpha) {
    const long long total = rows * C;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / C;
        const int c = (int)(e % C);
        y[r * ldy + c] += alpha * x[r * ldx + c];
    }
}

static inline int grid_for(long long work_items, int per_block = TR_THREADS, int max_blocks = 148 * 16) {
    long long b = (work_items + per_block - 1) / per_block;
    if (b < 1) b = 1;
    if (b > max_blocks) b = max_blocks;
    return (int)b;
}

static inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace lpd

using namespace lpd;

extern "C" int lpd_bn_stats(const float* z, long long rows, int C, int ld, double* partial, int nparts, void* stream) {
    LPD_REQUIRE(z && partial && rows >= 1 && C >= 4 && C % 4 == 0 && ld % 4 == 0 && ld >= C && nparts >= 1 && nparts <= 65535);
    LPD_REQUIRE(al16(z));
    LPD_REQUIRE(C <= 1024 || C % 1024 == 0);
    dim3 grid(nparts, ceil_div(C, 1024));
    col_stats_kernel<float, 4><<<grid, TR_THREADS, 0, as_stream(stream)>>>(z, rows, C, ld, partial, nullptr);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_bn_finalize(const double* partial, int nparts, double count, int C, const float* gamma, const float* beta,
                               float eps, float momentum, float* running_mean, float* running_var, float* bn_out, void* stream) {
    LPD_REQUIRE(partial && bn_out && nparts >= 1 && C >= 1 && count >= 1);
    bn_finalize_kernel<<<ceil_div(C, 8), 256, 0, as_stream(stream)>>>(partial, nparts, count, C, gamma, beta, eps, momentum,
                                                                      running_mean, running_var, bn_out);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_colsum_finalize(const double* partial, int nparts, int n, float* out, void* stream) {
    LPD_REQUIRE(partial && out && nparts >= 1 && n >= 1);
    colsum_finalize_kernel<<<ceil_div(n, 8), 256, 0, as_stream(stream)>>>(partial, nparts, n, out);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_affine_act(const float* z, long long rows, int C, int ldz, const float* scale, const float* shift, int act,
                              float slope, const float* aux, int ldaux, float* out, int ldo, void* stream) {
    LPD_REQUIRE(z && out && rows >= 1 && C >= 4 && C % 4 == 0 && ldz % 4 == 0 && ldo % 4 == 0 && al16(z) && al16(out));
    LPD_REQUIRE(act != LPD_ACT_GATE || (aux && ldaux % 4 == 0 && al16(aux)));
    affine_act_kernel<<<grid_for(rows * (C / 4)), TR_THREADS, 0, as_stream(stream)>>>(z, rows, C, ldz, scale, shift, act, slope,
                                                                                   aux, ldaux, out, ldo);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_bn_bwd_reduce(const float* dy, int lddy, const float* z, int ldz, long long rows, int C, const float* bn,
                                 int act, float slope, const float* aux, int ldaux, double* partial, int nparts, void* stream) {
    LPD_REQUIRE(dy && z && bn && partial && rows >= 1 && C >= 4 && C % 4 == 0 && lddy % 4 == 0 && ldz % 4 == 0);
    LPD_REQUIRE(al16(dy) && al16(z) && nparts >= 1 && nparts <= 65535);
    LPD_REQUIRE(C <= 1024 || C % 1024 == 0);
    LPD_REQUIRE(act != LPD_ACT_GATE || (aux && ldaux % 4 == 0 && al16(aux)));
    dim3 grid(nparts, ceil_div(C, 1024));
    bn_bwd_reduce_kernel<<<grid, TR_THREADS, 0, as_stream(stream)>>>(dy, lddy, z, ldz, rows, C, bn, act, slope, aux, ldaux, partial);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_bn_bwd_apply(const float* dy, int lddy, const float* z, int ldz, long long rows, int C, const float* bn,
                                const float* S, double count, int act, float slope, const float* aux, int ldaux,
                                float* dz, int lddz, void* stream) {
    LPD_REQUIRE(dy && z && bn && S && dz && rows >= 1 && C >= 4 && C % 4 == 0 && lddy % 4 == 0 && ldz % 4 == 0 && lddz % 4 == 0);
    LPD_REQUIRE(al16(dy) && al16(z) && al16(dz) && count >= 1);
    LPD_REQUIRE(act != LPD_ACT_GATE || (aux && ldaux % 4 == 0 && al16(aux)));
    LPD_REQUIRE(C <= 1024 || C % 1024 == 0);
    const int cgb = (C < 1024 ? C : 1024) / 4, lanes_b = TR_THREADS / cgb > 0 ? TR_THREADS / cgb : 1;
    LPD_REQUIRE(cgb <= TR_THREADS);
    dim3 grid_b(grid_for(rows, lanes_b), ceil_div(C, 1024));
    bn_bwd_apply_kernel<<<grid_b, TR_THREADS, 0, as_stream(stream)>>>(dy, lddy, z, ldz, rows, C, bn, S,
                                                                                     (float)(1.0 / count), act, slope, aux, ldaux, dz, lddz);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

static int edge_args(EdgeArgs& a, const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C) {
    LPD_REQUIRE(p && idx && B >= 1 && N >= 1 && k >= 1 && k <= 255 && C >= 4 && C % 4 == 0 && C <= 1024);
    LPD_REQUIRE(ldp % 4 == 0 && al16(p) && (!q || (ldq % 4 == 0 && al16(q))));
    a.p = p; a.ldp = ldp; a.q = q; a.ldq = ldq; a.idx = idx; a.M = (long long)B * N; a.N = N; a.k = k; a.C = C;
    return LPD_OK;
}

extern "C" int lpd_edge_sel_stats(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                                  const float* gamma, float* zsel, int ldz, uint8_t* arg, double* partial, int nparts, void* stream) {
    EdgeArgs a;
    int rc = edge_args(a, p, ldp, q, ldq, idx, B, N, k, C);
    if (rc != LPD_OK) return rc;
    LPD_REQUIRE(zsel && arg && partial && nparts >= 1 && ldz % 4 == 0 && al16(zsel) && (reinterpret_cast<uintptr_t>(arg) & 3u) == 0);
    edge_sel_stats_kernel<<<nparts, TR_THREADS, 0, as_stream(stream)>>>(a, gamma, zsel, ldz, arg, partial);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_materialize(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                                    const float* scale, const float* shift, int act, float slope, float* y, void* stream) {
    EdgeArgs a;
    int rc = edge_args(a, p, ldp, q, ldq, idx, B, N, k, C);
    if (rc != LPD_OK) return rc;
    LPD_REQUIRE(scale && shift && y && al16(y));
    edge_materialize_kernel<float, 4><<<grid_for(a.M * k * (C / 4)), TR_THREADS, 0, as_stream(stream)>>>(a, scale, shift, act, slope, y);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_sel_dense(const float* z, long long M, int k, int C, const float* gamma, float* zsel, int ldz,
                                  uint8_t* arg, void* stream) {
    LPD_REQUIRE(z && zsel && arg && M >= 1 && k >= 1 && k <= 255 && C >= 4 && C % 4 == 0 && ldz % 4 == 0 && al16(z) && al16(zsel));
    edge_sel_dense_kernel<float, 4><<<grid_for(M * (C / 4)), TR_THREADS, 0, as_stream(stream)>>>(z, M, k, C, gamma, zsel, ldz, arg);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_dense_bwd_apply(const float* z, long long M, int k, int C, const float* bn, const float* S, double count,
                                        int act, float slope, const float* dx, int lddx, const float* zsel, int ldzs,
                                        const uint8_t* arg, float* dz, void* stream) {
    LPD_REQUIRE(z && bn && S && dx && zsel && arg && dz && M >= 1 && k >= 1 && C >= 4 && C % 4 == 0 && lddx % 4 == 0 && ldzs % 4 == 0);
    LPD_REQUIRE(al16(z) && al16(dz) && al16(dx) && al16(zsel) && count >= 1);
    edge_dense_bwd_apply_kernel<float, 4><<<grid_for(M * (C / 4)), TR_THREADS, 0, as_stream(stream)>>>(z, M, k, C, bn, S, (float)(1.0 / count),
                                                                                                    act, slope, dx, lddx, zsel, ldzs, arg, dz, nullptr);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_bwd_reduce(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                                   const float* bn, int act, float slope, const float* dx, int lddx, const uint8_t* arg,
                                   const float* dy, double* partial, int nparts, void* stream) {
    EdgeArgs a;
    int rc = edge_args(a, p, ldp, q, ldq, idx, B, N, k, C);
    if (rc != LPD_OK) return rc;
    LPD_REQUIRE(bn && partial && nparts >= 1 && (dx || dy) && (!dx || (arg && lddx % 4 == 0 && al16(dx))) && (!dy || al16(dy)));
    LPD_REQUIRE(act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY);     // step-function gradients only
    edge_bwd_kernel<false><<<nparts, TR_THREADS, 0, as_stream(stream)>>>(a, bn, act, slope, dx, lddx, arg, dy, nullptr, 0.f, partial,
                                                                        nullptr, 0, nullptr, 0, nullptr);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_bwd_apply(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                                  const float* bn, int act, float slope, const float* dx, int lddx, const uint8_t* arg,
                                  const float* dy, const float* S, double count, float* dp, int lddp, float* dq, int lddq,
                                  void* stream) {
    EdgeArgs a;
    int rc = edge_args(a, p, ldp, q, ldq, idx, B, N, k, C);
    if (rc != LPD_OK) return rc;
    LPD_REQUIRE(bn && S && dp && count >= 1 && (dx || dy) && (!dx || (arg && lddx % 4 == 0 && al16(dx))) && (!dy || al16(dy)));
    LPD_REQUIRE(lddp % 4 == 0 && al16(dp) && (!dq || (lddq % 4 == 0 && al16(dq))));
    LPD_REQUIRE(act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY);     // step-function gradients only
    // dp accumulates with atomics: zero its C columns first
    LPD_CUDA_CHECK(cudaMemset2DAsync(dp, (size_t)lddp * 4, 0, (size_t)C * 4, (size_t)a.M, as_stream(stream)));
    edge_bwd_kernel<true><<<148 * 8, TR_THREADS, 0, as_stream(stream)>>>(a, bn, act, slope, dx, lddx, arg, dy, S, (float)(1.0 / count),
                                                                        nullptr, dp, lddp, dq, lddq, nullptr);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_adam(float* w, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2, float eps,
                        float weight_decay, int step, float grad_scale, void* stream) {
    LPD_REQUIRE(w && g && m && v && n >= 1 && step >= 1);
    const float bc1 = 1.f - powf(beta1, (float)step);
    const float bc2 = sqrtf(1.f - powf(beta2, (float)step));
    adam_kernel<<<grid_for(n), TR_THREADS, 0, as_stream(stream)>>>(w, g, m, v, n, lr, beta1, beta2, eps, weight_decay, bc1, bc2, grad_scale);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_axpy(float* y, int ldy, const float* x, int ldx, long long rows, int C, float alpha, void* stream) {
    LPD_REQUIRE(y && x && rows >= 1 && C >= 1 && ldy >= C && ldx >= C);
    axpy_kernel<<<grid_for(rows * C), TR_THREADS, 0, as_stream(stream)>>>(y, ldy, x, ldx, rows, C, alpha);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_scatter_add(const float* dy, const int32_t* idx, int B, int N, int k, int C, float* dp, int lddp, void* stream) {
    LPD_REQUIRE(dy && idx && dp && B >= 1 && N >= 1 && k >= 1 && C >= 4 && C % 4 == 0 && lddp % 4 == 0 && al16(dy) && al16(dp));
    const long long M = (long long)B * N;
    LPD_CUDA_CHECK(cudaMemset2DAsync(dp, (size_t)lddp * 4, 0, (size_t)C * 4, (size_t)M, as_stream(stream)));
    edge_scatter_add_kernel<<<grid_for(M * k * (C / 4)), TR_THREADS, 0, as_stream(stream)>>>(dy, idx, M, N, k, C, dp, lddp);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

// ---- "f16" train precision mode: fp16 storage of a dense edge layer's [M*k][C] tensors (include/lpd_b200.h) ---------------
static inline bool al8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

extern "C" int lpd_bn_stats_f16(const void* z, long long rows, int C, int ld, double* partial, int nparts, uint32_t* minmax,
                                void* stream) {
    LPD_REQUIRE(z && partial && minmax && rows >= 1 && C >= 8 && C % 8 == 0 && C <= 1024 && ld % 8 == 0 && ld >= C);
    LPD_REQUIRE(nparts >= 1 && nparts <= 65535 && al16(z) && al16(minmax));
    LPD_CUDA_CHECK(cudaMemsetAsync(minmax, 0xff, (size_t)C * 4, as_stream(stream)));
    LPD_CUDA_CHECK(cudaMemsetAsync(minmax + C, 0, (size_t)C * 4, as_stream(stream)));
    col_stats_kernel<__half, 8><<<dim3(nparts, 1), TR_THREADS, 0, as_stream(stream)>>>(reinterpret_cast<const __half*>(z), rows, C, ld,
                                                                                     partial, minmax);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_materialize_f16(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k,
                                        int C, const float* scale, const float* shift, int act, float slope, void* y, void* stream) {
    EdgeArgs a;
    int rc = edge_args(a, p, ldp, q, ldq, idx, B, N, k, C);
    if (rc != LPD_OK) return rc;
    LPD_REQUIRE(C % 8 == 0 && scale && shift && y && al16(y) && al16(scale) && al16(shift));
    edge_materialize_kernel<__half, 8><<<grid_for(a.M * k * (C / 8)), TR_THREADS, 0, as_stream(stream)>>>(a, scale, shift, act, slope,
                                                                                                         reinterpret_cast<__half*>(y));
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_sel_dense_f16(const void* z, long long M, int k, int C, const float* gamma, float* zsel, int ldz,
                                      uint8_t* arg, void* stream) {
    LPD_REQUIRE(z && zsel && arg && M >= 1 && k >= 1 && k <= 255 && C >= 8 && C % 8 == 0 && ldz % 4 == 0 && ldz >= C);
    LPD_REQUIRE(al16(z) && al16(zsel) && al8(arg));
    edge_sel_dense_kernel<__half, 8><<<grid_for(M * (C / 8)), TR_THREADS, 0, as_stream(stream)>>>(
        reinterpret_cast<const __half*>(z), M, k, C, gamma, zsel, ldz, arg);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_dense_bwd_apply_f16(const void* z, long long M, int k, int C, const float* bn, const float* S, double count,
                                            int act, float slope, const float* dx, int lddx, const float* zsel, int ldzs,
                                            const uint8_t* arg, void* dz, const float* gscale, void* stream) {
    LPD_REQUIRE(z && bn && S && dx && zsel && arg && dz && gscale && M >= 1 && k >= 1 && k <= 255 && C >= 8 && C % 8 == 0);
    LPD_REQUIRE(lddx % 4 == 0 && ldzs % 4 == 0 && al16(z) && al16(dz) && al16(dx) && al16(zsel) && al8(arg) && count >= 1);
    edge_dense_bwd_apply_kernel<__half, 8><<<grid_for(M * (C / 8)), TR_THREADS, 0, as_stream(stream)>>>(
        reinterpret_cast<const __half*>(z), M, k, C, bn, S, (float)(1.0 / count), act, slope, dx, lddx, zsel, ldzs, arg,
        reinterpret_cast<__half*>(dz), gscale);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_bwd_reduce_f16(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                                       const float* bn, int act, float slope, const float* dx, int lddx, const uint8_t* arg,
                                       const void* dy, const float* dyscale, double* partial, int nparts, void* stream) {
    EdgeArgs a;
    int rc = edge_args(a, p, ldp, q, ldq, idx, B, N, k, C);
    if (rc != LPD_OK) return rc;
    LPD_REQUIRE(C % 8 == 0 && bn && partial && nparts >= 1 && dy && dyscale && al16(dy) && (!dx || (arg && lddx % 4 == 0 && al16(dx))));
    LPD_REQUIRE(act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY);     // step-function gradients only
    edge_bwd_kernel<false, __half><<<nparts, TR_THREADS, 0, as_stream(stream)>>>(a, bn, act, slope, dx, lddx, arg,
                                                                                reinterpret_cast<const __half*>(dy), nullptr, 0.f,
                                                                                partial, nullptr, 0, nullptr, 0, dyscale);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_bwd_apply_f16(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                                      const float* bn, int act, float slope, const float* dx, int lddx, const uint8_t* arg,
                                      const void* dy, const float* dyscale, const float* S, double count, float* dp, int lddp,
                                      float* dq, int lddq, void* stream) {
    EdgeArgs a;
    int rc = edge_args(a, p, ldp, q, ldq, idx, B, N, k, C);
    if (rc != LPD_OK) return rc;
    LPD_REQUIRE(C % 8 == 0 && bn && S && dp && count >= 1 && dy && dyscale && al16(dy) && (!dx || (arg && lddx % 4 == 0 && al16(dx))));
    LPD_REQUIRE(lddp % 4 == 0 && al16(dp) && (!dq || (lddq % 4 == 0 && al16(dq))));
    LPD_REQUIRE(act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY);
    LPD_CUDA_CHECK(cudaMemset2DAsync(dp, (size_t)lddp * 4, 0, (size_t)C * 4, (size_t)a.M, as_stream(stream)));
    edge_bwd_kernel<true, __half><<<148 * 8, TR_THREADS, 0, as_stream(stream)>>>(a, bn, act, slope, dx, lddx, arg,
                                                                                reinterpret_cast<const __half*>(dy), S,
                                                                                (float)(1.0 / count), nullptr, dp, lddp, dq, lddq, dyscale);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}

extern "C" int lpd_edge_grad_scale_f16(const float* dx, int lddx, long long M, int C, const float* bn, const float* S, double count,
                                       int act, float slope, const uint32_t* zminmax, const void* w, int ldw, int K,
                                       uint32_t* work, float* scale, void* stream) {
    LPD_REQUIRE(dx && bn && S && zminmax && w && work && scale && M >= 1 && C >= 8 && C % 8 == 0 && C <= 1024 && count >= 1);
    LPD_REQUIRE(K >= 1 && K <= 1024 && ldw >= K && lddx % 4 == 0 && lddx >= C && al16(dx) && al16(work));
    LPD_REQUIRE(act == LPD_ACT_NONE || act == LPD_ACT_RELU || act == LPD_ACT_LEAKY);     // step-function gradients only
    const float gmax = act == LPD_ACT_LEAKY ? fmaxf(1.f, fabsf(slope)) : 1.f;       // max |act'| of a step activation
    LPD_CUDA_CHECK(cudaMemsetAsync(work, 0, (size_t)C * 4, as_stream(stream)));
    const int lanes = TR_THREADS / (C / 4);
    col_absmax_kernel<<<grid_for(M, lanes), TR_THREADS, 0, as_stream(stream)>>>(dx, lddx, M, C, work);
    LPD_LAUNCH_CHECK();
    edge_grad_scale_kernel<<<1, 256, 0, as_stream(stream)>>>(work, C, bn, S, 1.0 / count, gmax, zminmax,
                                                             reinterpret_cast<const __half*>(w), ldw, K, scale);
    LPD_LAUNCH_CHECK();
    return LPD_OK;
}
