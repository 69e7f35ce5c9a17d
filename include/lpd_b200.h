/*
 * lpd_b200.h — C ABI of the B200 (sm_100a) kernels behind the LPD-Net hot path.
 *
 * The reference (qiaozhijian/LPD-Net-Pytorch) has no FFI of its own: its hot path is a chain of
 * torch ops inside util/lpdnet_model.py, util/PointNetVlad.py, loss/pointnetvlad_loss.py and
 * evaluate.py.  Every entry point below names the reference call site (file:line, relative to the
 * reference root) whose arithmetic it replaces.  The Python host modules in
 * lpd-net-pytorch_b200/ bind these with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  All pointers are DEVICE pointers unless the
 *     name ends in _host.  The caller owns every buffer (inputs, outputs, workspaces).
 *   - fp32 storage everywhere, row-major, POINT-MAJOR: a feature map is X[rows][C] with
 *     rows = B*N points and C contiguous.  (The reference is channel-major [B,C,N]; the host
 *     modules transpose only at the public per-function boundary.)
 *   - kNN / retrieval indices are int32 and CLOUD-LOCAL (0..N-1) unless stated otherwise.
 *   - `stream` is a cudaStream_t passed as void*.  All launches are asynchronous on it;
 *     nothing synchronises, allocates or frees.
 *   - Return value: LPD_OK (0) or a negative lpd_status.  No exceptions cross the ABI.
 */
#ifndef LPD_B200_H
#define LPD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LPD_ABI_VERSION 2

typedef enum lpd_status {
    LPD_OK = 0,
    LPD_EINVAL = -1,     /* bad shape / alignment / unsupported parameter            */
    LPD_EWORKSPACE = -2, /* workspace too small                                       */
    LPD_ECUDA = -3,      /* a CUDA runtime call or launch failed (see lpd_last_cuda_error) */
    LPD_EUNSUPPORTED = -4 /* device is not sm_100 or feature not built                */
} lpd_status;

/* activation selector of the fused epilogues */
typedef enum lpd_act {
    LPD_ACT_NONE = 0,
    LPD_ACT_RELU = 1,      /* F.relu, PointNetVlad.py:156-167, lpdnet_model.py:297-303 */
    LPD_ACT_LEAKY = 2,     /* nn.LeakyReLU(slope), lpdnet_model.py:24,153             */
    LPD_ACT_SIGMOID = 3,   /* nn.Sigmoid, PointNetVlad.py:111                          */
    LPD_ACT_GATE = 4,      /* out = aux * sigmoid(v): GatingContext, PointNetVlad.py:111-113 */
    LPD_ACT_ADD = 5        /* lpd_gemm only: out = v + aux (aux may alias the output: gradient accumulation) */
} lpd_act;

/* operand layouts of lpd_gemm */
#define LPD_A_MK 0 /* A stored [M][K], K contiguous */
#define LPD_A_KM 1 /* A stored [K][M], M contiguous */
#define LPD_B_NK 0 /* B stored [N][K], K contiguous (a conv / linear weight [Cout][Cin]) */
#define LPD_B_KN 1 /* B stored [K][N], N contiguous (NetVLAD cluster / hidden weights)   */

int lpd_abi_version(void);
const char* lpd_status_str(int status);
/* text of the last CUDA error seen by this library on the calling thread ("" if none) */
const char* lpd_last_cuda_error(void);
/* properties of the current device: SM count, compute capability, opt-in shared memory bytes */
int lpd_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* smem_optin_bytes);

/* ---------------------------------------------------------------------------------------------
 * Folded BatchNorm (eval mode): scale = gamma / sqrt(var + eps), shift = beta - mean * scale.
 * Replaces the running-stat branch of every nn.BatchNorm{1,2}d on the path
 * (lpdnet_model.py:168-191, PointNetVlad.py:33,39,97,215-230).  `bias` (nullable) is the conv /
 * linear bias that precedes the BN: shift += bias * scale.
 * ------------------------------------------------------------------------------------------- */
int lpd_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var,
                const float* bias, float eps, int C, float* scale, float* shift, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Batched 2-D transpose  in[b][R][C] -> out[b][C][R]   (channel-major <-> point-major)
 * Replaces the transposes at lpdnet_model.py:212,348 and PointNetVlad.py:46.
 * ------------------------------------------------------------------------------------------- */
int lpd_transpose(const float* in, float* out, int batch, int rows, int cols, void* stream);

/* ---------------------------------------------------------------------------------------------
 * kNN: fused pairwise distance + top-k, the N x N matrix never leaves the SM.
 * Replaces knn(), lpdnet_model.py:317-326 (matmul, pow/sum, two subtractions, topk).
 *   x    [B][N][C] point-major, C in {3, 64} (any C <= 64 multiple of 1 is accepted)
 *   idx  [B][N][k]: k nearest by the CANONICAL order (SURVEY App. A.1):
 *          dot_ij = fmaf chain over c = 0..C-1 (acc starts at +0),  xx_j = same chain on (x_j,x_j)
 *          pd_ij  = ((-xx_j) - (-2*dot_ij)) - xx_i            (fp32, that operation order)
 *          sorted by pd descending, ties by j ascending.
 *   idx_i64 != 0 writes int64 (the dtype of the public knn() API), else int32.
 *   1 <= k <= 32, k <= N.
 * ------------------------------------------------------------------------------------------- */
int lpd_knn(const float* x, int B, int N, int C, int k, void* idx, int idx_i64, void* stream);

/* Same result as lpd_knn (bit-identical canonical order) for C == 64, with the distance GEMM on the tensor cores:
 * low-precision gram tiles (tcgen05) filter candidates, the survivors are re-scored in canonical fp32 arithmetic, and rows
 * whose candidate list cannot be proven complete fall back to the CUDA-core kernel.  `workspace`: device scratch of at least
 * lpd_knn_workspace_bytes(B, N, C, k) bytes, 16-byte aligned.  Requires sm_100. */
size_t lpd_knn_workspace_bytes(int B, int N, int C, int k);
int lpd_knn_tc(const float* x, int B, int N, int C, int k, void* idx, int idx_i64,
               void* workspace, size_t workspace_bytes, void* stream);
/* Filter formulation used by lpd_knn_tc (process-wide; returns the previous value, v outside 0..3 only queries):
 *   0  one pass, 3xTF32 gram, per-row replace-worst candidate lists (csrc/knn_tc.cu);
 *   1  two passes, fp16 gram of the centred features with the norm folded into the MMA, strided group maxima -> provable
 *      threshold -> collect, 128 query rows per work item (csrc/knn_tc2.cu; default);
 *   2  the same with 256 query rows per work item;
 *   3  variant 1 with the query tile held in tensor memory (TS-mode tcgen05.mma; measured on par with 1).
 * The indices are bit-identical to lpd_knn for every variant. */
int lpd_knn_tc_variant(int v);
/* Diagnostics: byte offset, inside the workspace of the LAST lpd_knn_tc call with these sizes and the current variant, of
 * the int32 [B][ceil(N/64)] array that marks the 64-row tiles recomputed by the exact CUDA-core kernel. */
size_t lpd_knn_tc_flags_offset(int B, int N, int C, int k);

/* Same result as lpd_knn (bit-identical canonical order) for C == 3 (Cartesian kNN, lpdnet_model.py:255): a uniform grid
 * over the cloud decides which candidates are scored (cells in growing shells around the query, pruned with a bound that
 * covers the fp32 rounding of the canonical score), every scored candidate uses the canonical arithmetic and order.
 * x [B][N][3]; workspace >= lpd_knn_xyz_workspace_bytes(B, N) bytes, 16-byte aligned. */
size_t lpd_knn_xyz_workspace_bytes(int B, int N);
int lpd_knn_xyz(const float* x, int B, int N, int k, void* idx, int idx_i64, void* workspace, size_t workspace_bytes,
                void* stream);

/* Spatial (grid-cell) order of every cloud: perm[b][t] = original index of the t-th point in cell order (stable inside a
 * cell, so it is a pure function of the cloud), inv (nullable) = the inverse permutation, xyz_sorted (nullable) = the
 * coordinates in that order.  Every per-point stage of the path is permutation-equivariant and NetVLAD sums over the
 * points (PointNetVlad.py:61-66), so the host modules run each cloud in this order for memory locality.
 * workspace >= lpd_knn_xyz_workspace_bytes(B, N). */
int lpd_cell_order(const float* x, int B, int N, int32_t* perm, int32_t* inv, float* xyz_sorted,
                   void* workspace, size_t workspace_bytes, void* stream);

/* lpd_cell_order that also leaves in `workspace` the search grid of the RE-ORDERED cloud xyz_sorted (required), and the kNN of that
 * cloud on that grid: lpd_knn_xyz(xyz_sorted, ...) without the second counting sort (a cloud in cell order is its own sort).
 * The workspace must stay untouched between the two calls.  Same result as lpd_knn_xyz, bit for bit. */
int lpd_cell_order_grid(const float* x, int B, int N, int32_t* perm, int32_t* inv, float* xyz_sorted,
                        void* workspace, size_t workspace_bytes, void* stream);
int lpd_knn_xyz_ordered(int B, int N, int k, void* idx, int idx_i64, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * General fp32 GEMM with fused per-column affine + activation epilogue (CUDA-core FFMA path,
 * "strict" fp32 arithmetic):
 *     C[b][m][n] = act( scale[n] * sum_k A[b][m][k] * B[b][k][n] + shift[n] )      (+ aux for GATE)
 * Replaces every nn.Conv1d / nn.Conv2d 1x1 (+BatchNorm +activation) and nn.Linear / matmul on the
 * path: lpdnet_model.py:231-232,262,297-305 ; PointNetVlad.py:48,76,104,155-170,209-230.
 *   scale / shift nullable (=> 1 / 0).  lda/ldb/ldc are leading dimensions in elements,
 *   stride* are per-batch element strides (0 => operand shared by all batches).
 *   aux (LPD_ACT_GATE only) has the layout of C.
 * ------------------------------------------------------------------------------------------- */
int lpd_gemm(const float* A, int a_layout, int lda, long long strideA,
             const float* B, int b_layout, int ldb, long long strideB,
             float* C, int ldc, long long strideC,
             int M, int N, int K, int batch,
             const float* scale, const float* shift, int act, float slope, const float* aux,
             void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core GEMM ("fast" arithmetic): same contract as lpd_gemm for the conv / linear case
 *     C[m][n] = act( scale[n] * sum_k A[m][k] * B[n][k] + shift[n] ),   A [M][K], B [N][K] K-contiguous,
 * executed with TMA-fed tcgen05.mma kind::tf32 (operands rounded to TF32 by the tensor core, fp32
 * accumulation in TMEM).  Requires sm_100, lda/ldb/ldc multiples of 4 and 16-byte aligned bases.
 * N % 4 == 0; act in {NONE, RELU, LEAKY with 0 <= slope <= 1}.  Replaces the same call sites as lpd_gemm where the stated
 * TF32 tolerance applies (DESIGN.md, "precision modes").
 * ------------------------------------------------------------------------------------------- */
int lpd_gemm_tf32(const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                  int M, int N, int K, const float* scale, const float* shift, int act, float slope,
                  void* stream);
/* The same kernel, batched and / or accumulating (training backward: the per-cloud NetVLAD products
 * da[b] = F[b] dvraw[b], dF[b] += a[b] dvraw[b]^T of PointNetVlad.py:64-68's backward, and input gradients that add into an
 * existing buffer):  C[z*M + m][n] (+)= act(scale[n] * sum_k A[z*M + m][k] * B[z*N + n][k] + shift[n]),  z < batch.
 * A [batch*M][lda], B [batch*N][ldb], C [batch*M][ldc] are the per-slice matrices stacked on their row axis. */
int lpd_gemm_tf32_ex(const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                     int M, int N, int K, int batch, int accumulate, const float* scale, const float* shift, int act,
                     float slope, void* stream);

/* Tensor-core GEMM contracting over the ROWS of two point-major maps (both operands "MN-major" for the tensor core):
 *     C[z][m][n] = sum_{k < K} A[z*K + k][m] * B[z*K + k][n]        A [batch*K][lda], B [batch*K][ldb]
 * TF32 operands, fp32 accumulation.  Used for the NetVLAD aggregate vraw[b] = F[b]^T a[b] (PointNetVlad.py:64-66), the
 * weight gradients dW = dZ^T A of every conv / linear layer (split over row slices z, reduced by lpd_splitk_reduce).
 * batch > 1 requires K % 32 == 0.  Requires sm_100, 16-byte aligned bases, leading dimensions multiples of 4. */
int lpd_gemm_tf32_tn(const float* A, int lda, const float* B, int ldb, float* C, int ldc, long long strideC,
                     int M, int N, int K, int batch, void* stream);

/* FP16-operand forms of the tensor-core GEMMs ("f16" precision mode of the eval path; csrc/gemm_tc.cu): operands are fp16
 * matrices (rounded to nearest by the producing kernel's epilogue or by lpd_f32_to_f16), products accumulate in fp32 on
 * tcgen05 kind::f16.  fp16 keeps 11 significant bits under round-to-nearest where kind::tf32 TRUNCATES fp32 operands to 10
 * (measured on the reference goldens: 1e-5 vs 5e-5 max-abs descriptor error), at twice the tensor rate and half the bytes.
 * Out-of-range results saturate to +-65504 (cvt.rn.satfinite) when the output is fp16.
 *   lpd_gemm_f16:     C[m][n] = act(scale[n] * sum_k A[m][k] W[n][k] + shift[n]);  A [M][lda], W [N][ldw] fp16 (lda, ldw % 8 == 0),
 *                     C fp32 (out_half == 0) or fp16 (out_half != 0) with leading dimension ldc (% 4 == 0) in elements.
 *   lpd_gemm_f16_tn:  C[z][m][n] = sum_{k<K} A[z*K+k][m] B[z*K+k][n]  (fp16 operands, fp32 C; batch > 1 needs K % 64 == 0).
 *   lpd_f32_to_f16:   y[r][c] = fp16(x[r][c]) for a [rows][cols] matrix (weights, once per parameter version). */
int lpd_gemm_f16(const void* A, int lda, const void* W, int ldw, void* C, int ldc, int out_half,
                 int M, int N, int K, const float* scale, const float* shift, int act, float slope, void* stream);
int lpd_gemm_f16_tn(const void* A, int lda, const void* B, int ldb, float* C, int ldc, long long strideC,
                    int M, int N, int K, int batch, void* stream);
int lpd_f32_to_f16(const float* x, long long ldx, void* y, long long ldy, long long rows, int cols, void* stream);
/* lpd_gemm_f16 followed by a max over each cloud's R rows, without writing the [M][N] product (PointNetVlad.py:164-169, the STN's
 * conv3 + bn3 + relu + mp1):
 *     out[b][n] = max_{r < R} act(scale[n] * sum_k A[b*R + r][k] W[n][k] + shift[n])        out fp32 [M/R][N]
 * A [M][lda], W [N][ldw] fp16; scale / shift may be NULL.  The GEMM epilogue writes the column maxima of every 32-row block to
 * part (fp32 [M/32][N], caller-provided, no initialisation needed), and lpd_colmax reduces those per cloud in the same call.
 * Each element goes through the same epilogue as lpd_gemm_f16 with fp32 output, so out equals lpd_colmax of that product exactly.
 * Requires R % 32 == 0, M % R == 0, M / R <= 65535, N % 256 == 0, lda, ldw % 8 == 0, 16-byte aligned pointers and act in
 * {NONE, RELU, LEAKY with 0 <= slope <= 1}; otherwise LPD_EINVAL with nothing launched. */
int lpd_gemm_f16_colmax(const void* A, int lda, const void* W, int ldw, int M, int N, int K, int R,
                        const float* scale, const float* shift, int act, float slope, float* part, float* out, void* stream);
/* "3xTF32" operand preparation: x (n contiguous floats) = hi + lo, hi = x truncated to TF32, lo = x - hi; out [3][n] holds
 * [hi; hi; lo] (role 0, the A side) or [hi; lo; hi] (role 1, the B side), so that one lpd_gemm_tf32_tn contraction over the stacked
 * rows accumulates hi.hi + hi.lo + lo.hi in fp32.  Used by the NetVLAD hidden projection (65536 x 256, PointNetVlad.py:76), which
 * stays at fp32 accuracy on the tensor cores in every precision mode but "fp32". */
int lpd_split3_tf32(const float* x, long long n, float* out, int role, void* stream);
/* the A side of that projection in one pass: v [B][R] row-major -> out [3][R][Bp] = v transposed, split [hi; hi; lo], Bp % 4 == 0. */
int lpd_transpose_split3(const float* v, int B, long long R, int Bp, float* out, void* stream);
/* lpd_gemm_tf32 with the result written as fp16 (C [M][ldc] halves): the projection in front of the f16-mode edge kernels, whose
 * input (the conv2 feature map that also feeds the exact feature-space kNN) stays fp32. */
int lpd_gemm_tf32_out16(const float* A, int lda, const float* B, int ldb, void* C, int ldc, int M, int N, int K,
                        const float* scale, const float* shift, int act, float slope, void* stream);
/* lpd_softmax64 that also writes the probabilities as fp16 (a_h [M][64]): the B operand of the f16-mode NetVLAD aggregate. */
int lpd_softmax64_f16(float* a, long long M, void* a_h, void* stream);
/* f16-mode forms of the pre-scaled edge kernels (fp16 rows in and out, see lpd_edge_gather_ext / lpd_edgeconv_dg_tf32):
 *   lpd_edge_gather_max_f16:  out[i][:] = act(q[i][:] + max_m p[j(i,m)][:]),  C == 256 or 64     (csrc/edge.cu)
 *                             (C == 64 with q == NULL, ACT_NONE: LPDNetOrign's gather-only SN stage, reference
 *                             lpdnet_model.py:104, :144)
 *   lpd_edgeconv_dg20_f16:    k == 20, 128 channels; y1 = act(p_j + q_i) and W2 in fp16, second layer on tcgen05 kind::f16,
 *                             x1 / x2 written as fp16                                             (csrc/edge_tc20.cu) */
int lpd_edge_gather_max_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                            int act, float slope, void* out, int ldo, void* stream);
int lpd_edgeconv_dg20_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N,
                          const void* w2, const float* s2, const float* t2, int act, float slope,
                          void* x1, int ld1, void* x2, int ld2, void* stream);
/* the same kernel for k == 32 (idx [B][N][32]; four points per 128-edge tile): the C5 stress shape of BASELINE.json */
int lpd_edgeconv_dg32_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N,
                          const void* w2, const float* s2, const float* t2, int act, float slope,
                          void* x1, int ld1, void* x2, int ld2, void* stream);
/* LPDNetOrign's convDG1 + convDG2 + max (reference lpdnet_model.py:98-107), f16 mode, 64 channels, k == 20 or 32 (any other k:
 * LPD_EINVAL, no launch).  The edge [f_i ; f_j - f_i] is decomposed as P = Wb f_j, Q = (Wa - Wb) f_i, and DG1's folded BatchNorm is
 * carried by p' = s1 P and q' = s1 Q + t1 (fp16 [B*N][ldp] / [B*N][ldq], ldp, ldq % 8 == 0, 16-byte aligned: lpd_gemm_tf32_out16
 * with epilogue vectors [s1 | s1], [0 | t1]).  Per edge y1 = act(p'_j + q'_i) in fp16, z = W2 y1 on tcgen05 kind::f16 with fp32
 * accumulation (W2 fp16 [64][64] row-major, 16-byte aligned), then
 *     x2[i][c] = max_m act(s2[c] z_m[c] + t2[c])            (the min over m is taken where s2[c] < 0)
 * written as fp16 to x2 [B*N][ld2] (ld2 >= 64 and even).  act in {NONE, RELU, LEAKY with 0 <= slope <= 1}.  No allocation, no host
 * synchronisation: capturable into a CUDA graph. */
int lpd_edgeconv_dg64_f16(const void* p, int ldp, const void* q, int ldq, const int32_t* idx, int B, int N, int k,
                          const void* w2, const float* s2, const float* t2, int act, float slope,
                          void* x2, int ld2, void* stream);

/* Fused input layers of the LPD-Net feature nets (lpdnet_model.py:231-232, :86-87), strict fp32, one pass:
 *     out[m][:] = act(s2 * (W2 . act(s1 * (W1 . x[m][0..D)) + t1)) + t2),   W1 [64][D], W2 [64][64], D <= 8
 * x [M][ldx], out [M][ldo]; act in {NONE, RELU, LEAKY with 0 <= slope <= 1}. */
int lpd_pointwise_mlp2(const float* x, int ldx, int D, long long M, const float* w1, const float* s1, const float* t1,
                       const float* w2, const float* s2, const float* t2, int act, float slope, float* out, int ldo,
                       void* stream);

/* column max over rows of each cloud: out[b][c] = max_n x[b][n][c]
 * (MaxPool2d((num_points,1)) PointNetVlad.py:137,169 ; torch.max(x,2) lpdnet_model.py:300) */
int lpd_colmax(const float* x, int B, int N, int C, int ldx, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * EdgeConv, neighbour-gather + extremum (exact decomposition of a 1x1 conv over
 * cat(neighbour, centre) followed by a monotone BN+activation and max over k, SURVEY App. A.3):
 *     out[i][c] = act( s[c] * (q[i][c] + ext_m p[j(i,m)][c]) + t[c] ),  ext = max if s[c] >= 0 else min
 * Replaces get_graph_feature + convDG1/convSN1 + max, lpdnet_model.py:246-250,255-258 (x1, x3),
 * and with q == NULL the gather-only edges of LPDNetOrign, lpdnet_model.py:104-107.
 *   p, q: [B*N][ldp / ldq] (C columns used), idx [B][N][k] cloud-local int32.
 * ------------------------------------------------------------------------------------------- */
int lpd_edge_gather_ext(const float* p, int ldp, const float* q, int ldq,
                        const int32_t* idx, int B, int N, int k, int C,
                        const float* scale, const float* shift, int act, float slope,
                        float* out, int ldo, void* stream);

/* ---------------------------------------------------------------------------------------------
 * EdgeConv, two chained edge layers fused; the N x k x C edge tensors never touch HBM:
 *     y1[i][m][:] = act(s1 * (p[j(i,m)][:] + q[i][:]) + t1)        C1 channels
 *     y2[i][m][:] = act(s2 * (W2 . y1[i][m][:]) + t2)              C2 channels, W2 [C2][C1]
 *     x1[i][:] = max_m y1[i][m][:]  (optional, x1 may be NULL)     x2[i][:] = max_m y2[i][m][:]
 * Replaces get_graph_feature + convDG1 + max + convDG2 + max, lpdnet_model.py:246-252 (C1=C2=128)
 * and get_graph_feature_Origin + convDG1 + convDG2 + max, lpdnet_model.py:98-101 (C1=C2=64).
 * ------------------------------------------------------------------------------------------- */
int lpd_edgeconv_dg(const float* p, int ldp, const float* q, int ldq,
                    const int32_t* idx, int B, int N, int k, int C1, int C2,
                    const float* s1, const float* t1, const float* w2,
                    const float* s2, const float* t2, int act, float slope,
                    float* x1, int ld1, float* x2, int ld2, void* stream);

/* Same contract as lpd_edgeconv_dg with the second edge layer on the tensor cores (tcgen05 kind::tf32, the
 * activated first-layer edge rows are written by the gathering warps straight into the UMMA shared-memory
 * layout; fp32 first layer, TF32 second layer, fp32 accumulation).  Requires sm_100.
 * s1 == t1 == NULL selects the PRE-SCALED form for the reference's own shape (k == 20, C1 == C2 == 128): the caller has folded the
 * first layer's BatchNorm into the projections (p = s1 * Wn f, q = s1 * Wc f + t1, e.g. in the projection GEMM's epilogue), so
 * y1 = act(p_j + q_i); csrc/edge_tc20.cu. */
int lpd_edgeconv_dg_tf32(const float* p, int ldp, const float* q, int ldq,
                         const int32_t* idx, int B, int N, int k, int C1, int C2,
                         const float* s1, const float* t1, const float* w2,
                         const float* s2, const float* t2, int act, float slope,
                         float* x1, int ld1, float* x2, int ld2, void* stream);

/* ---------------------------------------------------------------------------------------------
 * NetVLAD soft-assignment: a[m][:] = softmax_K( s * (x[m][:] . Wc) + t )
 * Replaces PointNetVlad.py:48-59 (matmul, BatchNorm1d(K) or cluster_biases, softmax).
 *   x [M][D], wc [D][K] (the reference's cluster_weights layout), a [M][K], K == 64.
 * ------------------------------------------------------------------------------------------- */
int lpd_netvlad_assign(const float* x, int M, int D, const float* wc, const float* scale,
                       const float* shift, int K, float* a, void* stream);

/* in-place row softmax over exactly 64 columns: a[m][:] = softmax(a[m][:])  (PointNetVlad.py:58, the
 * second half of lpd_netvlad_assign, exposed for the tensor-core assignment path) */
int lpd_softmax64(float* a, long long M, void* stream);

/* ---------------------------------------------------------------------------------------------
 * NetVLAD residual + normalisations, in place on the raw aggregate
 *     vraw[b][d][k] = sum_n a[b][n][k] * x[b][n][d]     (computed with lpd_gemm, A_KM x B_KN)
 *     v = vraw - (sum_n a[b][n][k]) * wc2[d][k] ; v /= max(||v[:,k]||,1e-12) ; v /= max(||v||,1e-12)
 * Replaces PointNetVlad.py:61-74.  `asum_ws` is a [B][8][K] float workspace (partial sums over N).
 * ------------------------------------------------------------------------------------------- */
int lpd_netvlad_finish(float* vlad, const float* a, const float* wc2, int B, int N, int D, int K,
                       float* asum_ws, void* stream);

/* The soft assignment in ONE launch (PointNetVlad.py:48-59): a = softmax_k(scale[k] * (x . Wc)[m][k] + shift[k]) as the epilogue
 * of the tensor-core GEMM (x [M][lda] fp16 when a_f16 else fp32 consumed as TF32, W = cluster_weights^T [64][ldw] of the same
 * type; fp32 accumulation).  Writes a32 [M][64] fp32 and / or a16 [M][64] fp16 (either may be NULL, not both) and, when apart is
 * not NULL, apart[m / 32][64] = the column sums of every block of 32 rows (fp32 values; apart holds ceil(M / 32) * 64 floats;
 * with max_samples % 32 == 0 these are per-cloud partial sums of a_sum, PointNetVlad.py:61).  Requires sm_100. */
int lpd_gemm_softmax64(const void* A, int a_f16, int lda, const void* W, int ldw, int M, int K, const float* scale,
                       const float* shift, float* a32, void* a16, float* apart, void* stream);

/* lpd_netvlad_finish on given partial sums: apart [B][nparts][K] (sum over nparts = a_sum).  One thread-block cluster of 8 CTAs
 * per cloud; requires D % 128 == 0 and D <= 1024.  Replaces PointNetVlad.py:61-74. */
int lpd_netvlad_finish_parts(float* vlad, const float* apart, int nparts, const float* wc2, int B, int D, int K, void* stream);

/* Tail of NetVLAD + context gating in one launch (PointNetVlad.py:76-81, 103-115):
 *     h[b][o] = s2[o] * sum_s part[s][b][o] + t2[o]                       (split-K partial sums of v . hidden1_weights, bn2 folded)
 *     out[b][o] = h[b][o] * sigmoid(sg[o] * sum_i h[b][i] wg[i][o] + tg[o])   (gating_weights [O][O] as stored; sg / tg = folded bn1 or
 *                                                                           NULL / gating_biases)
 * O <= 1024; s2, t2, sg, tg may be NULL. */
int lpd_hidden_gate(const float* part, int splits, int B, int O, const float* s2, const float* t2, const float* wg,
                    const float* sg, const float* tg, float* out, void* stream);

/* deterministic split-K reduce + affine: out[m][n] = scale[n]*sum_s part[s][m][n] + shift[n]
 * (second half of the 65536->256 hidden projection + bn2, PointNetVlad.py:76-78) */
int lpd_splitk_reduce(const float* part, int splits, int M, int N, const float* scale,
                      const float* shift, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Lazy / non-lazy triplet and quadruplet hinge losses, forward and backward in one launch each.
 * Replaces best_pos_distance / triplet_loss / quadruplet_loss, loss/pointnetvlad_loss.py:6-97.
 *   q [Bq][1][D], pos [Bq][P][D], neg [Bq][Nn][D], other [Bq][1][D] (other == NULL => triplet)
 *   flags: bit0 use_min, bit1 lazy, bit2 ignore_zero_loss.
 *   loss: 1 float.  Gradients (nullable as a group) have the input layouts and are the gradient
 *   of `loss` scaled by *grad_out (device scalar, nullable => 1).
 * ------------------------------------------------------------------------------------------- */
int lpd_quadruplet_loss(const float* q, const float* pos, const float* neg, const float* other,
                        int Bq, int P, int Nn, int D, float m1, float m2, int flags,
                        float* loss, float* gq, float* gpos, float* gneg, float* gother,
                        const float* grad_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Retrieval: exact brute-force k nearest database rows of every query, Euclidean, fp64
 * difference-form accumulation (the arithmetic of sklearn KDTree on float32 input), ties by
 * lower database index.  Replaces KDTree(database).query(q, k=25), evaluate.py:168,186-187.
 *   db [Ndb][D], q [Nq][D], idx [Nq][k] int32 (+ idx_offset added, for sharded databases),
 *   dist [Nq][k] double (squared distances; nullable).  1 <= k <= 32.  Entries beyond Ndb are -1.
 *   workspace: device scratch of at least lpd_retrieval_workspace_bytes(Ndb, Nq, k) bytes
 *   (per-database-split partial lists, merged deterministically).
 * ------------------------------------------------------------------------------------------- */
size_t lpd_retrieval_workspace_bytes(int Ndb, int Nq, int k);
int lpd_retrieval_topk(const float* db, int Ndb, const float* q, int Nq, int D, int k,
                       int idx_offset, int32_t* idx, double* dist,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Merge `lists` sorted top-k lists per query (part_dist / part_idx [lists][Nq][k], GLOBAL database indices, -1 = empty
 * slot) into one: ascending distance, ties to the lower index — the merge step of the database-sharded search (each
 * rank's lpd_retrieval_topk list, all-gathered over NCCL; SURVEY §8e). */
int lpd_topk_merge(const double* part_dist, const int32_t* part_idx, int lists, int Nq, int k,
                   int32_t* idx, double* dist, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Retrieval on the tensor cores, per database SEGMENT (csrc/retrieval_tc.cu).  Replaces the per-run-pair
 * KDTree(DATABASE_VECTORS[m]).query(q, k=25) loop of evaluate.py:59-70,168,186-187 for ALL runs in one call: the
 * databases of all runs are stacked row-wise, segment s = rows [seg_off[s], seg_off[s+1]), and every query is searched in
 * every segment.  Filter (3xTF32 split distance GEMM on tcgen05 -> approximate scores, k-th-score threshold with a proven
 * error margin) + refine (the fp64 difference-form arithmetic of lpd_retrieval_topk): results are BIT-IDENTICAL to
 * lpd_retrieval_topk run on each segment (ascending (distance, index); ties to the lower index).
 *   db [Ndb][D], q [Nq][D], D % 4 == 0, D <= 1024; seg_off int32 [S+1] (device), ascending, seg_off[0] >= 0, seg_off[S] <= Ndb
 *   idx  int32  [S][Nq][k]: segment-local row (global_idx == 0) or database row + idx_offset (global_idx != 0); -1 = empty
 *   dist double [S][Nq][k] squared distances (nullable)
 *   workspace: lpd_retrieval_tc_workspace_bytes(Ndb, Nq, D) bytes, 256-byte aligned (split operands + the [Nq][Ndb] scores)
 * A database sharded over ranks / cut into ~1000-row pseudo-segments is finished with lpd_topk_merge (the [S][Nq][k]
 * layout is that function's input layout).
 * ------------------------------------------------------------------------------------------- */
size_t lpd_retrieval_tc_workspace_bytes(int Ndb, int Nq, int D);
int lpd_retrieval_tc(const float* db, int Ndb, const float* q, int Nq, int D, int k,
                     const int32_t* seg_off, int S, int global_idx, int idx_offset,
                     int32_t* idx, double* dist, void* workspace, size_t workspace_bytes, void* stream);

/* get_recall's counting (evaluate.py:176-206) for all (query, database segment) units at once, on the device.
 *   idx [S][Nq][k] segment-local top-k (lpd_retrieval_tc), k <= 25.  There are R runs; segment s is the database of run
 *   seg_run[s] (nullable: s itself; a rank that holds a subset of the runs passes their numbers).  q_run int32 [Nq] = run of
 *   each query: a query is not searched in its own run's database (evaluate.py:61-62); q_run[i] < 0 = belongs to no run.
 *   Truth in CSR form: the true neighbours of query i in run m are truth_idx[truth_off[i*R+m] .. truth_off[i*R+m+1])
 *   (indices local to that run's database; empty = the query is skipped, :181-182).
 *   seg_thresh int32 [S] = max(int(round(len(db_s)/100)), 1) (:174).
 *   Outputs (caller zeroes the counters), row = max(q_run[i], 0) * S + s:  hist int32 [R*S][25] first-hit rank histogram
 *   (:189-193), n_eval [R*S] evaluated queries, n_onepct [R*S] queries with a true neighbour among the first seg_thresh ranks
 *   (:200-201), sim float [Nq][S] (nullable; needs db, seg_off, q, D) = dot(query, its top-1) where the top-1 is a true
 *   neighbour (:191), NaN elsewhere. */
int lpd_recall_count(const int32_t* idx, int S, int Nq, int k, const int32_t* q_run, int R, const int32_t* seg_run,
                     const int32_t* truth_off, const int32_t* truth_idx, const int32_t* seg_thresh,
                     const float* db, const int32_t* seg_off, const float* q, int D,
                     int32_t* hist, int32_t* n_eval, int32_t* n_onepct, float* sim, void* stream);

/* =============================================================================================
 * TRAIN MODE (reference: model.train() forward, loss.backward(), optimizer.step();
 * train_pointnetvlad.py:121-130,150-159).  Batch-statistics BatchNorm and the backward pass.
 * A "bn" block is 4 consecutive float rows of C: scale = gamma*invstd, shift = beta - mean*scale,
 * mean, invstd  (what lpd_bn_finalize writes and the backward kernels read).
 * "partial" buffers are double [nparts][2][C] per-block partial sums (deterministic two-stage reduce).
 * ============================================================================================= */

/* column sums of z and z^2 over rows -> partial.  nn.BatchNorm{1,2}d batch statistics (torch batch_norm, training=True)
 * of lpdnet_model.py:168-173,189-191,231-262 and PointNetVlad.py:33,39,97.  C % 4 == 0, ld % 4 == 0. */
int lpd_bn_stats(const float* z, long long rows, int C, int ld, double* partial, int nparts, void* stream);
/* partial -> bn block [4][C]; updates running_mean / running_var in place (nullable) with `momentum` and the unbiased
 * variance, as torch does.  `count` = number of values per channel. */
int lpd_bn_finalize(const double* partial, int nparts, double count, int C, const float* gamma, const float* beta,
                    float eps, float momentum, float* running_mean, float* running_var, float* bn_out, void* stream);
/* out[i] = (float) sum_p partial[p][i], i < n  (n = 2*C for a partial buffer: [S1 | S2]) */
int lpd_colsum_finalize(const double* partial, int nparts, int n, float* out, void* stream);
/* out = act(scale * z + shift) elementwise over [rows][C]; LPD_ACT_GATE: out = aux * sigmoid(scale*z+shift). */
int lpd_affine_act(const float* z, long long rows, int C, int ldz, const float* scale, const float* shift, int act,
                   float slope, const float* aux, int ldaux, float* out, int ldo, void* stream);
/* backward of  y = act(BN_batch(z)):  dzbn = dy * act'(scale*z+shift);
 *   reduce: partial of S1 = sum dzbn (= d beta), S2 = sum dzbn * xhat (= d gamma)
 *   apply : dz = scale * (dzbn - S1/count - xhat * S2/count)          (S = float [2][C]; dz may alias dy) */
int lpd_bn_bwd_reduce(const float* dy, int lddy, const float* z, int ldz, long long rows, int C, const float* bn,
                      int act, float slope, const float* aux, int ldaux, double* partial, int nparts, void* stream);
int lpd_bn_bwd_apply(const float* dy, int lddy, const float* z, int ldz, long long rows, int C, const float* bn,
                     const float* S, double count, int act, float slope, const float* aux, int ldaux,
                     float* dz, int lddz, void* stream);

/* Train-mode EdgeConv (get_graph_feature + Conv2d + BatchNorm2d(batch stats) + act + max, lpdnet_model.py:246-258).
 * Edge pre-activation z[(i,m)][c] = p[j(i,m)][c] + q[i][c] (q nullable).  BN and the activation are monotone per channel,
 * so max_m act(BN(z)) = act(BN(zsel)), zsel = q + (gamma >= 0 ? max : min)_m p_j:
 *   lpd_edge_sel_stats : zsel [M][ldz], arg uint8 [M][C] (first m reaching the extremum), partial of (sum z, sum z^2)
 *                        over all M*k edges (closed form per point, SURVEY App. A.3)
 *   lpd_edge_materialize: y[(i,m)][:] = act(scale*(p_j+q_i)+shift), dense [M*k][C] (input of a following edge layer)
 *   lpd_edge_sel_dense : the same selection over an already materialised z [M][k][C] */
int lpd_edge_sel_stats(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                       const float* gamma, float* zsel, int ldz, uint8_t* arg, double* partial, int nparts, void* stream);
int lpd_edge_materialize(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                         const float* scale, const float* shift, int act, float slope, float* y, void* stream);
int lpd_edge_sel_dense(const float* z, long long M, int k, int C, const float* gamma, float* zsel, int ldz,
                       uint8_t* arg, void* stream);
/* backward of a materialised edge layer whose only consumer is the max over m:
 *   dz[(i,m)][c] = scale * ([m == arg[i][c]] * dx[i][c] * act'(scale*zsel+shift) - S1/count - xhat(z) * S2/count)
 * (S from lpd_bn_bwd_reduce over the [M][C] arrays dx / zsel; dz may alias z) */
int lpd_edge_dense_bwd_apply(const float* z, long long M, int k, int C, const float* bn, const float* S, double count,
                             int act, float slope, const float* dx, int lddx, const float* zsel, int ldzs,
                             const uint8_t* arg, float* dz, void* stream);
/* backward of a decomposed edge layer: incoming gradient = dense dy [(i,m)][C] (nullable) + dx [M][lddx] routed to arg
 * (nullable).  reduce -> partial (S1, S2); apply -> dq[i] = sum_m dz, dp[j] += dz (fp32 atomics; dp's C columns are zeroed
 * first) — the index_put_(accumulate=True) of the reference's autograd. */
int lpd_edge_bwd_reduce(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                        const float* bn, int act, float slope, const float* dx, int lddx, const uint8_t* arg,
                        const float* dy, double* partial, int nparts, void* stream);
int lpd_edge_bwd_apply(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                       const float* bn, int act, float slope, const float* dx, int lddx, const uint8_t* arg,
                       const float* dy, const float* S, double count, float* dp, int lddp, float* dq, int lddq,
                       void* stream);

/* f16 storage of the edge tensors (the "f16" train precision mode of featnet="lpdnet", set_train_precision in ops.py).
 * The dense DG2 edge layer keeps its four [M*k][C] tensors in fp16: y1 (input rows), z2e (pre-activations), and their
 * gradients dz2e and dy1.  Every kernel below computes in fp32 exactly as its fp32 form above does, on the values the fp16
 * storage holds; fp16 results are rounded to nearest.  Requirements on top of the fp32 forms: C % 8 == 0, 1 <= k <= 255,
 * fp16 pointers 16-byte aligned, arg 8-byte aligned, non-null scale pointers; otherwise LPD_EINVAL with nothing launched.
 *   lpd_bn_stats_f16          : lpd_bn_stats over fp16 z (C <= 1024), plus the exact column min / max as order keys in
 *                               minmax uint32 [2][C] (read by lpd_edge_grad_scale_f16).  |z| >= 65504 (the fp16 limit, where
 *                               lpd_gemm_f16 saturates) counts as NaN: z must fit fp16's range, or the statistics and with them
 *                               the loss come out non-finite — never silently wrong.
 *   lpd_edge_materialize_f16  : lpd_edge_materialize with y stored as fp16 (p, q fp32).
 *   lpd_edge_sel_dense_f16    : lpd_edge_sel_dense over fp16 z (zsel fp32, arg uint8 as before).
 *   lpd_edge_dense_bwd_apply_f16: lpd_edge_dense_bwd_apply over fp16 z, writing fp16(2^E * dz) (in place over z allowed).
 *   lpd_edge_bwd_{reduce,apply}_f16: lpd_edge_bwd_{reduce,apply} with a required fp16 dy holding 2^E * dy; each value is
 *                               multiplied by dyscale[0] = 2^-E in fp32 (exact) before use.
 * Gradient scaling.  BN backward over count = M*k edges makes dz2e tiny (below fp16's subnormal floor 6e-8 for many entries
 * at training sizes), so dz2e and dy1 are stored as fp16(2^E * value) with ONE power-of-two exponent E per step, computed on
 * the device (no host synchronisation, no skipped steps) from a bound:
 *     max|dz_c|  <= |scale_c| * (max_i|dx_ic| * max(1, |gneg|) + |S1_c|/count + X_c * |S2_c|/count),
 *     X_c = max(|min_c - mean_c|, |max_c - mean_c|) * invstd_c   (the column range lpd_bn_stats_f16 recorded),
 *     max|dy1_k| <= sum_c |W2[c][k]| * max|dz_c|                  (dy1 = dz2e . W2, W2 [C][K] fp16, ldw),
 * and E is the largest integer with 2^E * (both bounds) <= 2^14 (|E| <= 100; E = 0 when a bound is not finite).
 *   lpd_edge_grad_scale_f16   : dx [M][lddx] (point-level gradient of the max), bn, S (lpd_bn_bwd_reduce over dx / zsel),
 *                               zminmax, W2 -> scale fp32 [2][K]: scale[0][:] = 2^E, scale[1][:] = 2^-E.  work: uint32 [C]
 *                               scratch.  Two launches (column max of |dx|, then one block for the bounds).
 * Consumers undo the scale exactly: lpd_edge_bwd_*_f16 take dyscale = scale[1]; dW2 = (2^E dz2e)^T y1 runs on lpd_gemm_f16_tn
 * and lpd_splitk_reduce with the vector scale[1]; dy1 = dz2e . W2 is linear and runs on lpd_gemm_f16 with fp16 output. */
int lpd_bn_stats_f16(const void* z, long long rows, int C, int ld, double* partial, int nparts, uint32_t* minmax, void* stream);
int lpd_edge_materialize_f16(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                             const float* scale, const float* shift, int act, float slope, void* y, void* stream);
int lpd_edge_sel_dense_f16(const void* z, long long M, int k, int C, const float* gamma, float* zsel, int ldz, uint8_t* arg,
                           void* stream);
int lpd_edge_dense_bwd_apply_f16(const void* z, long long M, int k, int C, const float* bn, const float* S, double count,
                                 int act, float slope, const float* dx, int lddx, const float* zsel, int ldzs,
                                 const uint8_t* arg, void* dz, const float* gscale, void* stream);
int lpd_edge_bwd_reduce_f16(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                            const float* bn, int act, float slope, const float* dx, int lddx, const uint8_t* arg,
                            const void* dy, const float* dyscale, double* partial, int nparts, void* stream);
int lpd_edge_bwd_apply_f16(const float* p, int ldp, const float* q, int ldq, const int32_t* idx, int B, int N, int k, int C,
                           const float* bn, int act, float slope, const float* dx, int lddx, const uint8_t* arg,
                           const void* dy, const float* dyscale, const float* S, double count, float* dp, int lddp,
                           float* dq, int lddq, void* stream);
int lpd_edge_grad_scale_f16(const float* dx, int lddx, long long M, int C, const float* bn, const float* S, double count,
                            int act, float slope, const uint32_t* zminmax, const void* w, int ldw, int K,
                            uint32_t* work, float* scale, void* stream);

/* backward of the gather-only edges e[(i,m)][:] = f[j(i,m)][:] (get_graph_feature_Origin(cat=False), lpdnet_model.py:116-145;
 * forward = lpd_edge_materialize with q = NULL, scale 1, shift 0, no activation): dp[j] += dy[(i,m)], dp zeroed first. */
int lpd_edge_scatter_add(const float* dy, const int32_t* idx, int B, int N, int k, int C, float* dp, int lddp, void* stream);

/* NetVLAD train mode: lpd_netvlad_finish that also saves asum [B][K], the clamped intra norms n1 [B][K] and the clamped
 * global norm n2 [B]; its backward (in place on dv [B][D][K] -> d vraw; dasum [B][K]; dwc2 [D][K]); softmax backward
 * with the a_sum gradient folded in (in place on da [M][64]).  PointNetVlad.py:58-74. */
int lpd_netvlad_finish_train(float* vlad, const float* a, const float* wc2, int B, int N, int D, int K,
                             float* asum, float* n1, float* n2, void* stream);
int lpd_netvlad_finish_bwd(float* dv, const float* v, const float* wc2, const float* asum, const float* n1,
                           const float* n2, int B, int D, int K, float* dasum, float* dwc2, void* stream);
int lpd_softmax64_bwd(float* da, const float* a, const float* dasum, long long M, int N, void* stream);

/* column max over the points of each cloud with argmax, and its backward (dx[b][arg][c] += dout[b][c]).
 * torch.max(x, 2) lpdnet_model.py:300 ; MaxPool2d((num_points,1)) PointNetVlad.py:137,169. */
int lpd_colmax_arg(const float* x, int B, int N, int C, int ldx, float* out, int32_t* arg, void* stream);
int lpd_colmax_bwd(const float* dout, const int32_t* arg, int B, int N, int C, float* dx, int lddx, void* stream);

/* torch.optim.Adam step (train_pointnetvlad.py:57,130,159) over a flat parameter buffer; g is multiplied by grad_scale
 * first (1/world_size after a gradient all-reduce-sum).  step >= 1. */
int lpd_adam(float* w, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2, float eps,
             float weight_decay, int step, float grad_scale, void* stream);
/* y[r][c] += alpha * x[r][c] */
int lpd_axpy(float* y, int ldy, const float* x, int ldx, long long rows, int C, float alpha, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LPD_B200_H */
