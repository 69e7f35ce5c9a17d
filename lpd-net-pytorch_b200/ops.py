"""Tensor-level wrappers over the C ABI: torch supplies device memory and the stream, nothing else.

Every function takes CUDA float32 (or int32) tensors, allocates its outputs with torch.empty and
launches on torch's current stream.  Feature maps are POINT-MAJOR [rows, C] (see include/lpd_b200.h).
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import (ACT_ADD, ACT_GATE, ACT_LEAKY, ACT_NONE, ACT_RELU, ACT_SIGMOID, A_KM, A_MK, B_KN, B_NK)

__all__ = ["bn_fold", "transpose", "knn", "knn_tc_variant", "pointwise_mlp2", "gemm", "colmax", "edge_gather_ext", "edgeconv_dg",
           "gemm_tf32", "linear", "set_precision", "get_precision", "set_train_precision", "get_train_precision", "netvlad_assign", "softmax64", "netvlad_finish", "splitk_reduce", "quadruplet_loss", "retrieval_topk", "retrieval_tc", "retrieval_search", "recall_count",
           "ACT_NONE", "ACT_RELU", "ACT_LEAKY", "ACT_SIGMOID", "ACT_GATE", "A_MK", "A_KM", "B_NK", "B_KN"]


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


# ---- weights epoch: kernels that update parameters / buffers through raw pointers (lpd_adam, lpd_bn_finalize's running
# statistics) do not bump torch's tensor._version, so every cache keyed on the parameters (folded BatchNorm, re-laid-out
# weights, captured CUDA graphs) also keys on this counter --------------------------------------------------------------
_weights_epoch = 0


def weights_epoch() -> int:
    return _weights_epoch


def bump_weights_epoch() -> None:
    global _weights_epoch
    _weights_epoch += 1


def dispatch_key() -> tuple:
    """everything outside the parameters that a captured forward bakes in (precision mode, kernel selection switches)"""
    return (_precision, SPATIAL_ORDER, KNN_TENSOR_CORES, KNN_GRID, knn_tc_variant(-1) if _lib._lib is not None else -1)


# ---- launch accounting / per-call device timing (used by bench.py; off by default) ----------------------------
_launches = 0          # kernels launched through this module since reset_launch_count()
_profile = None        # None, or a list receiving (label, start_event, end_event)


def reset_launch_count() -> None:
    global _launches
    _launches = 0


def launch_count() -> int:
    return _launches


def profile(enable: bool):
    """Start / stop recording one CUDA-event pair around every C-ABI call on the current stream."""
    global _profile
    rec, _profile = _profile, ([] if enable else None)
    return rec


def _call(label: str, nlaunch: int, fn, *args) -> None:
    global _launches
    if _profile is not None:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        rc = fn(*args)
        e.record()
        _profile.append((label, s, e))
    else:
        rc = fn(*args)
    _launches += nlaunch
    _lib.check(rc, label)


def _p(t):
    return None if t is None else t.data_ptr()


def _f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.LpdError(f"{name} must be a CUDA tensor: the lpd_b200 kernels have no CPU path")
    if t.dtype != torch.float32:
        raise _lib.LpdError(f"{name} must be float32, got {t.dtype}")
    if t.device.index != torch.cuda.current_device():
        # the C ABI launches on the calling thread's current device / stream: one process (or at least one
        # torch.cuda.device scope) per GPU; nn.DataParallel-style cross-device calls are rejected, not mis-launched
        raise _lib.LpdError(f"{name} lives on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                            f"call torch.cuda.set_device (one process per GPU) or wrap the call in torch.cuda.device(...)")
    return t


def bn_fold(gamma, beta, mean, var, eps: float, bias=None):
    """(scale, shift) of an eval-mode BatchNorm, optionally absorbing a preceding conv bias."""
    lib = _lib.load()
    _f32(mean, "running_mean")
    C = mean.numel()
    out = torch.empty(2, C, device=mean.device, dtype=torch.float32)
    _call("lpd_bn_fold", 1, lib.lpd_bn_fold, _p(gamma), _p(beta), _p(mean), _p(var), _p(bias), float(eps), C,
                               out[0].data_ptr(), out[1].data_ptr(), _stream())
    return out[0], out[1]


def transpose(x: torch.Tensor) -> torch.Tensor:
    """[b, R, C] -> [b, C, R] (contiguous)."""
    lib = _lib.load()
    x = _f32(x, "x").contiguous()
    b, R, Cc = x.shape
    out = torch.empty(b, Cc, R, device=x.device, dtype=torch.float32)
    _call("lpd_transpose", 1, lib.lpd_transpose, x.data_ptr(), out.data_ptr(), b, R, Cc, _stream())
    return out


# C == 64: exact filter-and-refine kNN with the gram tiles on tcgen05 (lpd_knn_tc: fp16 two-pass threshold filter, or the
# 3xTF32 single-pass filter, + canonical fp32 re-score).  Bit-identical to the CUDA-core kernel; rows whose candidate list
# cannot be proven complete are recomputed by it.
KNN_TENSOR_CORES = True
# C == 3: exact grid-accelerated kNN (lpd_knn_xyz); bit-identical to the brute-force scan of lpd_knn.
KNN_GRID = True


def knn_tc_variant(v: int = -1) -> int:
    """Select the filter formulation of the tensor-core kNN (see lpd_knn_tc_variant in include/lpd_b200.h); returns the
    previous one.  v = -1 only queries."""
    return int(_lib.load().lpd_knn_tc_variant(int(v)))


def knn(x_pm: torch.Tensor, k: int, int64: bool = False, diag: dict | None = None) -> torch.Tensor:
    """x_pm [B, N, C] point-major -> idx [B, N, k] (int32, or int64 for the public API), canonical order.
    The result is bit-identical whichever kernel computes it.  `diag` (tests / tools): receives "flagged_tiles", the number
    of 64-row tiles the tensor-core filter handed to the exact CUDA-core kernel (synchronises)."""
    lib = _lib.load()
    x_pm = _f32(x_pm, "x").contiguous()
    B, N, Cc = x_pm.shape
    idx = torch.empty(B, N, k, device=x_pm.device, dtype=torch.int64 if int64 else torch.int32)
    if KNN_TENSOR_CORES and Cc == 64 and N >= 128 and x_pm.data_ptr() % 16 == 0:
        nbytes = lib.lpd_knn_workspace_bytes(B, N, Cc, k)
        ws = torch.empty((nbytes + 3) // 4, device=x_pm.device, dtype=torch.float32)
        _call(f"lpd_knn_tc[C={Cc},k={k}]", 5, lib.lpd_knn_tc, x_pm.data_ptr(), B, N, Cc, k, idx.data_ptr(), int(int64),
              ws.data_ptr(), ws.numel() * 4, _stream())
        if diag is not None:
            off = lib.lpd_knn_tc_flags_offset(B, N, Cc, k) // 4
            diag["flagged_tiles"] = int((ws.view(torch.int32)[off: off + B * ((N + 63) // 64)] != 0).sum().item())
            diag["tiles"] = B * ((N + 63) // 64)
    elif KNN_GRID and Cc == 3 and N >= 64 and _grid_of(x_pm) is not None:
        # the cloud came out of cell_order(): its search grid is already in that call's workspace
        ws = _grid_of(x_pm)
        _call(f"lpd_knn_xyz[k={k}]", 2, lib.lpd_knn_xyz_ordered, B, N, k, idx.data_ptr(), int(int64), ws.data_ptr(), ws.numel() * 4, _stream())
    elif KNN_GRID and Cc == 3 and N >= 64:
        nbytes = lib.lpd_knn_xyz_workspace_bytes(B, N)
        ws = torch.empty((nbytes + 3) // 4, device=x_pm.device, dtype=torch.float32)
        _call(f"lpd_knn_xyz[k={k}]", 2, lib.lpd_knn_xyz, x_pm.data_ptr(), B, N, k, idx.data_ptr(), int(int64), ws.data_ptr(),
              ws.numel() * 4, _stream())
    else:
        _call(f"lpd_knn[C={Cc},k={k}]", 1, lib.lpd_knn, x_pm.data_ptr(), B, N, Cc, k, idx.data_ptr(), int(int64), _stream())
    return idx


# Run each cloud in spatial (grid-cell) order inside the models (see lpd_cell_order): same descriptors up to fp32 summation
# order, better gather locality and far fewer kNN list updates.
SPATIAL_ORDER = True


# one-entry cache: the re-ordered cloud of the last cell_order() call and the workspace holding its search grid.  The cache keeps
# both tensors alive, so the data pointer identifies the cloud; _version catches in-place edits.
_grid_cache = None


def _grid_of(x_pm: torch.Tensor):
    c = _grid_cache
    if (c is not None and x_pm.data_ptr() == c[0].data_ptr() and tuple(x_pm.shape) == tuple(c[0].shape) and c[0]._version == c[2]
            and x_pm.device == c[0].device):
        return c[1]
    return None


def cell_order(xyz: torch.Tensor, want_inv: bool = False):
    """xyz [B, N, 3] -> (perm int32 [B, N], inv int32 [B, N] or None, xyz_sorted [B, N, 3]).  knn(xyz_sorted, k) reuses the grid this
    call built (lpd_cell_order_grid / lpd_knn_xyz_ordered)."""
    lib = _lib.load()
    xyz = _f32(xyz, "xyz").contiguous()
    B, N, _ = xyz.shape
    perm = torch.empty(B, N, device=xyz.device, dtype=torch.int32)
    inv = torch.empty(B, N, device=xyz.device, dtype=torch.int32) if want_inv else None
    out = torch.empty_like(xyz)
    nbytes = lib.lpd_knn_xyz_workspace_bytes(B, N)
    ws = torch.empty((nbytes + 3) // 4, device=xyz.device, dtype=torch.float32)
    _call("lpd_cell_order", 1, lib.lpd_cell_order_grid, xyz.data_ptr(), B, N, perm.data_ptr(), _p(inv), out.data_ptr(), ws.data_ptr(),
          ws.numel() * 4, _stream())
    global _grid_cache
    _grid_cache = (out, ws, out._version)
    return perm, inv, out


def gemm(A, B, *, a_layout=A_MK, b_layout=B_NK, M, N, K, lda=None, ldb=None, out=None, ldc=None,
         batch=1, strideA=0, strideB=0, strideC=0, scale=None, shift=None, act=ACT_NONE, slope=0.0, aux=None):
    """out[b][m][n] = act(scale[n] * sum_k A[b][m][k] B[b][k][n] + shift[n]); see lpd_gemm."""
    lib = _lib.load()
    _f32(A, "A"), _f32(B, "B")
    if lda is None:
        lda = K if a_layout == A_MK else M
    if ldb is None:
        ldb = K if b_layout == B_NK else N
    if out is None:
        ldc = N
        out = torch.empty((batch, M, N) if batch > 1 else (M, N), device=A.device, dtype=torch.float32)
        if batch > 1:
            strideC = M * N
    elif ldc is None:
        ldc = out.stride(-2)
    _call(f"lpd_gemm[{M}x{N}x{K}x{batch}]", 1, lib.lpd_gemm, A.data_ptr(), a_layout, lda, strideA, B.data_ptr(), b_layout, ldb, strideB,
                            out.data_ptr(), ldc, strideC, M, N, K, batch, _p(scale), _p(shift), act, float(slope),
                            _p(aux), _stream())
    return out


# ---- precision mode of the dense conv / linear layers ----------------------------------------------------------
#   "fp32": every GEMM on the CUDA cores (lpd_gemm, plain FFMA)        — strict parity mode
#   "tf32": large K-contiguous GEMMs on the tensor cores (lpd_gemm_tf32) — fast mode, fp32 operands truncated to TF32 by the MMA
#   "f16":  the eval path of all three feature nets (featnet=lpdnet and lpdnetorigin at k = 20 or 32: downstream of the
#           feature-space kNN; featnet=pointnet at N % 64 == 0: after conv2, and the STNs' conv2 / conv3) keeps its activations in
#           FP16 (rounded to nearest, 11 significant bits) and multiplies on tcgen05 kind::f16 with fp32 accumulation: half the
#           bytes, twice the tensor rate, and a SMALLER error than "tf32" (measured 1e-5 vs 5e-5 max-abs on the lpdnet golden,
#           2e-5 / 4.5e-5 vs 7e-5 / 1.3e-4 on the two pointnet goldens).  Everything else (training, other k, other N) behaves as
#           in "tf32".
_precision = "fp32"


def set_precision(mode: str) -> str:
    """Select "fp32" (strict), "tf32" or "f16" (tensor cores); returns the previous mode."""
    global _precision
    if mode not in ("fp32", "tf32", "f16"):
        raise ValueError("precision must be 'fp32', 'tf32' or 'f16'")
    prev, _precision = _precision, mode
    return prev


def get_precision() -> str:
    return _precision


def gemm_tf32(A, W, *, M, N, K, lda=None, ldw=None, out=None, ldc=None, scale=None, shift=None, act=ACT_NONE, slope=0.0, batch=1,
              accumulate=False):
    """out[z*M + m][n] (+)= act(scale[n] * sum_k A[z*M + m][k] W[z*N + n][k] + shift[n]) on the tensor cores (TF32);
    batch > 1: the per-slice matrices are stacked on their row axis; accumulate: adds into `out`."""
    lib = _lib.load()
    _f32(A, "A"), _f32(W, "W")
    lda = K if lda is None else lda
    ldw = K if ldw is None else ldw
    if out is None:
        if accumulate:
            raise ValueError("gemm_tf32: accumulate needs an output buffer")
        out = torch.empty(batch * M, N, device=A.device, dtype=torch.float32)
        ldc = N
    elif ldc is None:
        ldc = out.stride(-2)
    label = f"lpd_gemm_tf32[{M}x{N}x{K}]" if batch == 1 else f"lpd_gemm_tf32[{M}x{N}x{K}x{batch}]"
    _call(label, 1, lib.lpd_gemm_tf32_ex, A.data_ptr(), lda, W.data_ptr(), ldw, out.data_ptr(), ldc,
          M, N, K, batch, int(bool(accumulate)), _p(scale), _p(shift), act, float(slope), _stream())
    return out


def gemm_tf32_tn(A, Bm, *, M, N, K, lda, ldb, batch=1, out=None):
    """out[z][m][n] = sum_{k<K} A[z*K+k][m] * Bm[z*K+k][n] on the tensor cores (TF32): contraction over the ROWS of two
    point-major maps (weight gradients, NetVLAD aggregate).  -> [batch, M, N]"""
    lib = _lib.load()
    _f32(A, "A"), _f32(Bm, "B")
    if out is None:
        out = torch.empty(batch, M, N, device=A.device, dtype=torch.float32)
    _call(f"lpd_gemm_tf32_tn[{M}x{N}x{K}x{batch}]", 1, lib.lpd_gemm_tf32_tn, A.data_ptr(), lda, Bm.data_ptr(), ldb, out.data_ptr(), N,
          M * N, M, N, K, batch, _stream())
    return out


def to_f16(x: torch.Tensor) -> torch.Tensor:
    """fp32 [rows, cols] (last dim contiguous) -> fp16 copy, rounded to nearest (lpd_f32_to_f16)"""
    lib = _lib.load()
    _f32(x, "x")
    rows, cols = x.shape
    y = torch.empty(rows, cols, device=x.device, dtype=torch.float16)
    _call("lpd_f32_to_f16", 1, lib.lpd_f32_to_f16, x.data_ptr(), x.stride(0), y.data_ptr(), cols, rows, cols, _stream())
    return y


def split3_tf32(x: torch.Tensor, role: int) -> torch.Tensor:
    """contiguous fp32 [rows, cols] -> [3 * rows, cols]: the TF32 hi / lo split stacked as [hi; hi; lo] (role 0) or [hi; lo; hi]
    (role 1), see lpd_split3_tf32"""
    lib = _lib.load()
    x = _f32(x, "x").contiguous()
    rows, cols = x.shape
    out = torch.empty(3 * rows, cols, device=x.device, dtype=torch.float32)
    _call("lpd_split3_tf32", 1, lib.lpd_split3_tf32, x.data_ptr(), x.numel(), out.data_ptr(), int(role), _stream())
    return out


def transpose_split3(v: torch.Tensor, Bp: int) -> torch.Tensor:
    """v [B, R] fp32 -> [3 * R, Bp]: v transposed and TF32-split as [hi; hi; lo] (lpd_transpose_split3)"""
    lib = _lib.load()
    v = _f32(v, "v").contiguous()
    B, R = v.shape
    out = torch.empty(3 * R, Bp, device=v.device, dtype=torch.float32)
    _call("lpd_transpose_split3", 1, lib.lpd_transpose_split3, v.data_ptr(), B, R, Bp, out.data_ptr(), _stream())
    return out


def _f16(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda or t.dtype != torch.float16:
        raise _lib.LpdError(f"{name} must be a CUDA float16 tensor, got {t.dtype} on {t.device}")
    if t.device.index != torch.cuda.current_device():
        raise _lib.LpdError(f"{name} lives on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}")
    return t


def gemm_f16(A, W, *, M, N, K, lda=None, ldw=None, out=None, ldc=None, out_half=False, scale=None, shift=None, act=ACT_NONE, slope=0.0):
    """out[m][n] = act(scale[n] * sum_k A[m][k] W[n][k] + shift[n]) with fp16 operands on the tensor cores (fp32 accumulate);
    the output is fp32, or fp16 when out_half (or `out` is an fp16 tensor)."""
    lib = _lib.load()
    _f16(A, "A"), _f16(W, "W")
    lda = K if lda is None else lda
    ldw = K if ldw is None else ldw
    if out is None:
        out = torch.empty(M, N, device=A.device, dtype=torch.float16 if out_half else torch.float32)
        ldc = N
    else:
        out_half = out.dtype == torch.float16
        if ldc is None:
            ldc = out.stride(-2)
    _call(f"lpd_gemm_f16[{M}x{N}x{K}]", 1, lib.lpd_gemm_f16, A.data_ptr(), lda, W.data_ptr(), ldw, out.data_ptr(), ldc, int(out_half),
          M, N, K, _p(scale), _p(shift), act, float(slope), _stream())
    return out


def gemm_f16_colmax(A, W, *, M, N, K, R, scale=None, shift=None, act, slope):
    """out[b][n] = max_{r<R} act(scale[n] * sum_k A[b*R + r][k] W[n][k] + shift[n]) -> fp32 [M/R, N], fp16 operands on the tensor
    cores; the [M, N] product is never written (lpd_gemm_f16_colmax: R % 32 == 0, N % 256 == 0).  Allocates, besides the output,
    an fp32 [M/32, N] scratch buffer for the column maxima of every 32-row block."""
    lib = _lib.load()
    _f16(A, "A"), _f16(W, "W")
    part = torch.empty(M // 32, N, device=A.device, dtype=torch.float32)
    out = torch.empty(M // R, N, device=A.device, dtype=torch.float32)
    _call(f"lpd_gemm_f16_colmax[{M}x{N}x{K}]", 2, lib.lpd_gemm_f16_colmax, A.data_ptr(), A.stride(0), W.data_ptr(), W.stride(0), M, N, K,
          R, _p(scale), _p(shift), act, float(slope), part.data_ptr(), out.data_ptr(), _stream())
    return out


def gemm_f16_tn(A, Bm, *, M, N, K, lda, ldb, batch=1, out=None):
    """out[z][m][n] = sum_{k<K} A[z*K+k][m] * Bm[z*K+k][n], fp16 operands (rows = the contraction axis), fp32 out [batch, M, N]"""
    lib = _lib.load()
    _f16(A, "A"), _f16(Bm, "B")
    if out is None:
        out = torch.empty(batch, M, N, device=A.device, dtype=torch.float32)
    _call(f"lpd_gemm_f16_tn[{M}x{N}x{K}x{batch}]", 1, lib.lpd_gemm_f16_tn, A.data_ptr(), lda, Bm.data_ptr(), ldb, out.data_ptr(), N,
          M * N, M, N, K, batch, _stream())
    return out


def gemm_tf32_out16(A, W, *, M, N, K, lda=None, ldw=None, scale=None, shift=None, act=ACT_NONE, slope=0.0):
    """fp32 operands (TF32 MMA), fp16 output [M, N]: the projection in front of the f16-mode edge kernels"""
    lib = _lib.load()
    _f32(A, "A"), _f32(W, "W")
    out = torch.empty(M, N, device=A.device, dtype=torch.float16)
    _call(f"lpd_gemm_tf32[{M}x{N}x{K}]", 1, lib.lpd_gemm_tf32_out16, A.data_ptr(), K if lda is None else lda, W.data_ptr(),
          K if ldw is None else ldw, out.data_ptr(), N, M, N, K, _p(scale), _p(shift), act, float(slope), _stream())
    return out


def softmax64_f16(a, M):
    """in place on a [M, 64] fp32; also returns the fp16 copy (the B operand of the f16-mode NetVLAD aggregate)"""
    lib = _lib.load()
    a_h = torch.empty(M, 64, device=a.device, dtype=torch.float16)
    _call("lpd_softmax64", 1, lib.lpd_softmax64_f16, a.data_ptr(), M, a_h.data_ptr(), _stream())
    return a, a_h


def edge_gather_max_f16(p, ldp, q, ldq, idx, B, N, k, C, act, slope, out, ldo):
    """out = act(q + max_m p[j(i,m)]) on fp16 rows (C == 256 or 64): lpd_edge_gather_max_f16"""
    lib = _lib.load()
    _f16(p, "p")
    _call(f"lpd_edge_gather_ext[C={C}]", 1, lib.lpd_edge_gather_max_f16, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C,
          act, float(slope), out.data_ptr(), ldo, _stream())
    return out


def edgeconv_dg20_f16(p, ldp, q, ldq, idx, B, N, w2_h, s2, t2, act, slope, x1, ld1, x2, ld2):
    """the 128-channel double edge layer with fp16 rows in and out, k = 20 or 32 taken from idx [B, N, k]
    (lpd_edgeconv_dg20_f16 / lpd_edgeconv_dg32_f16)"""
    lib = _lib.load()
    _f16(p, "p"), _f16(w2_h, "w2")
    k = idx.shape[-1]
    if k not in (20, 32):
        raise _lib.LpdError(f"edgeconv_dg20_f16: k must be 20 or 32, got {k}")
    _call("lpd_edgeconv_dg_f16[128x128]", 1, lib.lpd_edgeconv_dg20_f16 if k == 20 else lib.lpd_edgeconv_dg32_f16, p.data_ptr(), ldp, q.data_ptr(), ldq, idx.data_ptr(), B, N,
          w2_h.data_ptr(), s2.data_ptr(), t2.data_ptr(), act, float(slope), _p(x1), ld1, x2.data_ptr(), ld2, _stream())
    return x1, x2


def edgeconv_dg64_f16(p, ldp, q, ldq, idx, B, N, w2_h, s2, t2, act, slope, x2, ld2):
    """LPDNetOrign's 64-channel double edge layer with fp16 rows in and out (lpd_edgeconv_dg64_f16); k = idx.shape[-1], and any
    k but 20 or 32 is rejected by the library"""
    lib = _lib.load()
    _f16(p, "p"), _f16(q, "q"), _f16(w2_h, "w2"), _f16(x2, "x2")
    k = idx.shape[-1]
    _call("lpd_edgeconv_dg_f16[64x64]", 1, lib.lpd_edgeconv_dg64_f16, p.data_ptr(), ldp, q.data_ptr(), ldq, idx.data_ptr(), B, N,
          k, w2_h.data_ptr(), s2.data_ptr(), t2.data_ptr(), act, float(slope), x2.data_ptr(), ld2, _stream())
    return x2


def _tn_ok(A, Bm, M, N, K, lda, ldb, batch):
    return (_precision != "fp32" and M >= 64 and N >= 64 and N % 4 == 0 and lda % 4 == 0 and ldb % 4 == 0 and K >= 256
            and (batch == 1 or K % 32 == 0) and A.data_ptr() % 16 == 0 and Bm.data_ptr() % 16 == 0)


def linear(A, W, *, M, N, K, lda=None, out=None, ldc=None, scale=None, shift=None, act=ACT_NONE, slope=0.0):
    """conv1x1 / linear layer y = act(scale * (A . W^T) + shift) with W [N, K]; dispatches on the precision mode."""
    lda_ = K if lda is None else lda
    if (_precision != "fp32" and K >= 32 and K % 4 == 0 and lda_ % 4 == 0 and N >= 64 and N % 4 == 0 and M >= 128
            and (ldc is None or ldc % 4 == 0) and A.data_ptr() % 16 == 0 and (out is None or out.data_ptr() % 16 == 0)):
        return gemm_tf32(A, W, M=M, N=N, K=K, lda=lda, out=out, ldc=ldc, scale=scale, shift=shift, act=act, slope=slope)
    return gemm(A, W, M=M, N=N, K=K, lda=lda, out=out, ldc=ldc, scale=scale, shift=shift, act=act, slope=slope)


def pointwise_mlp2(x, D, M, w1, s1, t1, w2, s2, t2, act=ACT_NONE, slope=0.0, ldx=None):
    """out [M, 64] = act(s2 * (W2 . act(s1 * (W1 . x[:, :D]) + t1)) + t2): the two input 1x1 convs of the LPD-Net feature nets in
    one strict-fp32 pass (the 64-wide hidden map stays in registers)."""
    lib = _lib.load()
    _f32(x, "x")
    out = torch.empty(M, 64, device=x.device, dtype=torch.float32)
    _call("lpd_pointwise_mlp2", 1, lib.lpd_pointwise_mlp2, x.data_ptr(), x.stride(-2) if ldx is None else ldx, D, M, w1.data_ptr(),
          s1.data_ptr(), t1.data_ptr(), w2.data_ptr(), s2.data_ptr(), t2.data_ptr(), act, float(slope), out.data_ptr(), 64, _stream())
    return out


def colmax(x: torch.Tensor, B: int, N: int, C: int, ldx: int | None = None) -> torch.Tensor:
    lib = _lib.load()
    _f32(x, "x")
    out = torch.empty(B, C, device=x.device, dtype=torch.float32)
    _call("lpd_colmax", 1, lib.lpd_colmax, x.data_ptr(), B, N, C, C if ldx is None else ldx, out.data_ptr(), _stream())
    return out


def edge_gather_ext(p, ldp, q, ldq, idx, B, N, k, C, scale, shift, act, slope, out, ldo):
    lib = _lib.load()
    _call(f"lpd_edge_gather_ext[C={C}]", 1, lib.lpd_edge_gather_ext, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C, _p(scale), _p(shift),
                                       act, float(slope), out.data_ptr(), ldo, _stream())
    return out


def edgeconv_dg(p, ldp, q, ldq, idx, B, N, k, C1, C2, s1, t1, w2, s2, t2, act, slope, x1, ld1, x2, ld2):
    """Two fused edge layers (see lpd_edgeconv_dg); second layer on the tensor cores in "tf32" precision mode.
    s1 = t1 = None: p / q already carry the first layer's folded BatchNorm (tf32 mode, k == 20, C1 == C2 == 128)."""
    lib = _lib.load()
    tf32 = _precision != "fp32" and act != ACT_SIGMOID
    fn, label = (lib.lpd_edgeconv_dg_tf32, "lpd_edgeconv_dg_tf32") if tf32 else (lib.lpd_edgeconv_dg, "lpd_edgeconv_dg")
    if s1 is None and not (tf32 and k == 20 and C1 == 128 and C2 == 128):
        raise _lib.LpdError("edgeconv_dg: the pre-scaled form (s1 = t1 = None) exists for tf32 mode, k == 20, 128 channels only")
    _call(f"{label}[{C1}x{C2}]", 1, fn, p.data_ptr(), ldp, q.data_ptr(), ldq, idx.data_ptr(), B, N, k, C1, C2,
          _p(s1), _p(t1), w2.data_ptr(), s2.data_ptr(), t2.data_ptr(),
          act, float(slope), _p(x1), ld1, x2.data_ptr(), ld2, _stream())
    return x1, x2


def netvlad_assign(x, M, D, wc, scale, shift, K=64, out=None):
    lib = _lib.load()
    if out is None:
        out = torch.empty(M, K, device=x.device, dtype=torch.float32)
    _call("lpd_netvlad_assign", 2, lib.lpd_netvlad_assign, x.data_ptr(), M, D, wc.data_ptr(), _p(scale), _p(shift), K, out.data_ptr(),
                                      _stream())
    return out


def softmax64(a, M):
    lib = _lib.load()
    _call("lpd_softmax64", 1, lib.lpd_softmax64, a.data_ptr(), M, _stream())
    return a


def netvlad_finish(vlad, a, wc2, B, N, D, K=64):
    """in place on vlad [B, D, K]; returns it viewed as [B, D*K]."""
    lib = _lib.load()
    ws = torch.empty(B * 8 * K, device=vlad.device, dtype=torch.float32)
    _call("lpd_netvlad_finish", 2, lib.lpd_netvlad_finish, vlad.data_ptr(), a.data_ptr(), wc2.data_ptr(), B, N, D, K, ws.data_ptr(),
                                      _stream())
    return vlad.view(B, D * K)


def gemm_softmax64(x, wct, *, M, K, scale=None, shift=None, want32=True, want16=False, want_parts=False):
    """soft assignment in one launch: softmax over the 64 clusters as the epilogue of the tensor-core GEMM x [M, K] . wct [64, K]^T
    (both fp16, or both fp32 consumed as TF32).  Returns (a32 | None, a16 | None, apart [ceil(M/32), 64] | None)."""
    lib = _lib.load()
    f16 = x.dtype == torch.float16
    (_f16 if f16 else _f32)(x, "x"), (_f16 if f16 else _f32)(wct, "wct")
    a32 = torch.empty(M, 64, device=x.device, dtype=torch.float32) if want32 else None
    a16 = torch.empty(M, 64, device=x.device, dtype=torch.float16) if want16 else None
    apart = torch.empty((M + 31) // 32, 64, device=x.device, dtype=torch.float32) if want_parts else None
    _call(f"lpd_gemm_softmax64[{M}x64x{K}]", 1, lib.lpd_gemm_softmax64, x.data_ptr(), int(f16), K, wct.data_ptr(), K, M, K, _p(scale), _p(shift),
          _p(a32), _p(a16), _p(apart), _stream())
    return a32, a16, apart


def netvlad_finish_parts(vlad, apart, nparts, wc2, B, D, K=64):
    """netvlad_finish on given partial column sums of the assignment, apart [B, nparts, K]; in place on vlad [B, D, K]"""
    lib = _lib.load()
    _call("lpd_netvlad_finish", 1, lib.lpd_netvlad_finish_parts, vlad.data_ptr(), apart.data_ptr(), nparts, wc2.data_ptr(), B, D, K, _stream())
    return vlad.view(B, D * K)


def hidden_gate(part, splits, B, O, s2, t2, wg, sg, tg):
    """split-K reduce of the hidden projection + bn2 + context gating in one launch -> [B, O]"""
    lib = _lib.load()
    out = torch.empty(B, O, device=part.device, dtype=torch.float32)
    _call("lpd_hidden_gate", 1, lib.lpd_hidden_gate, part.data_ptr(), splits, B, O, _p(s2), _p(t2), wg.data_ptr(), _p(sg), _p(tg),
          out.data_ptr(), _stream())
    return out


def splitk_reduce(part, splits, M, N, scale=None, shift=None):
    lib = _lib.load()
    out = torch.empty(M, N, device=part.device, dtype=torch.float32)
    _call("lpd_splitk_reduce", 1, lib.lpd_splitk_reduce, part.data_ptr(), splits, M, N, _p(scale), _p(shift), out.data_ptr(), _stream())
    return out


def quadruplet_loss(q, pos, neg, other, m1, m2, use_min, lazy, ignore_zero_loss, need_grad=False, grad_out=None):
    """Returns loss [1] and, if need_grad, (gq, gpos, gneg, gother)."""
    lib = _lib.load()
    q, pos, neg = _f32(q, "q").contiguous(), _f32(pos, "pos").contiguous(), _f32(neg, "neg").contiguous()
    other = None if other is None else _f32(other, "other").contiguous()
    Bq, P, D = pos.shape
    Nn = neg.shape[1]
    flags = int(bool(use_min)) | (int(bool(lazy)) << 1) | (int(bool(ignore_zero_loss)) << 2)
    loss = torch.empty(1, device=q.device, dtype=torch.float32)
    grads = (None, None, None, None)
    if need_grad:
        grads = (torch.empty_like(q), torch.empty_like(pos), torch.empty_like(neg),
                 None if other is None else torch.empty_like(other))
    _call("lpd_quadruplet_loss", 1, lib.lpd_quadruplet_loss, q.data_ptr(), pos.data_ptr(), neg.data_ptr(), _p(other), Bq, P, Nn, D,
                                       float(m1), float(m2), flags, loss.data_ptr(), _p(grads[0]), _p(grads[1]),
                                       _p(grads[2]), _p(grads[3]), _p(grad_out), _stream())
    return (loss, grads) if need_grad else loss


def retrieval_topk(db: torch.Tensor, q: torch.Tensor, k: int, idx_offset: int = 0, want_dist: bool = True):
    """db [Ndb, D], q [Nq, D] -> (idx int32 [Nq, k], squared dist float64 [Nq, k] or None)."""
    lib = _lib.load()
    db, q = _f32(db, "db").contiguous(), _f32(q, "q").contiguous()
    Ndb, D = db.shape
    Nq = q.shape[0]
    idx = torch.empty(Nq, k, device=db.device, dtype=torch.int32)
    dist = torch.empty(Nq, k, device=db.device, dtype=torch.float64) if want_dist else None
    ws_bytes = lib.lpd_retrieval_workspace_bytes(Ndb, Nq, k)
    ws = torch.empty((ws_bytes + 7) // 8, device=db.device, dtype=torch.float64)
    _call("lpd_retrieval_topk", 2, lib.lpd_retrieval_topk, db.data_ptr(), Ndb, q.data_ptr(), Nq, D, k, idx_offset, idx.data_ptr(), _p(dist),
                                      ws.data_ptr(), ws.numel() * 8, _stream())
    return idx, dist


def topk_merge(part_dist: torch.Tensor, part_idx: torch.Tensor):
    """part_dist float64 / part_idx int32 [lists, Nq, k] (global indices, -1 = empty) -> (idx [Nq, k], dist [Nq, k])"""
    lib = _lib.load()
    lists, Nq, k = part_idx.shape
    part_dist, part_idx = part_dist.contiguous(), part_idx.contiguous()
    idx = torch.empty(Nq, k, device=part_idx.device, dtype=torch.int32)
    dist = torch.empty(Nq, k, device=part_idx.device, dtype=torch.float64)
    _call("lpd_topk_merge", 1, lib.lpd_topk_merge, part_dist.data_ptr(), part_idx.data_ptr(), lists, Nq, k, idx.data_ptr(),
          dist.data_ptr(), _stream())
    return idx, dist


def retrieval_tc(db: torch.Tensor, q: torch.Tensor, k: int, seg_off: torch.Tensor, global_idx: bool = False, idx_offset: int = 0,
                 want_dist: bool = True):
    """Tensor-core filter + exact fp64 refine, per database segment (lpd_retrieval_tc): db [Ndb, D], q [Nq, D], seg_off int32
    [S+1] on the device -> (idx int32 [S, Nq, k], squared dist float64 [S, Nq, k] or None); bit-identical to retrieval_topk
    run on each segment."""
    lib = _lib.load()
    db, q = _f32(db, "db").contiguous(), _f32(q, "q").contiguous()
    Ndb, D = db.shape
    Nq, S = q.shape[0], seg_off.numel() - 1
    idx = torch.empty(S, Nq, k, device=db.device, dtype=torch.int32)
    dist = torch.empty(S, Nq, k, device=db.device, dtype=torch.float64) if want_dist else None
    nbytes = lib.lpd_retrieval_tc_workspace_bytes(Ndb, Nq, D)
    ws = torch.empty(nbytes, device=db.device, dtype=torch.uint8)
    _call(f"lpd_retrieval_tc[{Nq}x{Ndb}x{D}]", 4, lib.lpd_retrieval_tc, db.data_ptr(), Ndb, q.data_ptr(), Nq, D, k, seg_off.data_ptr(), S,
          int(bool(global_idx)), int(idx_offset), idx.data_ptr(), _p(dist), ws.data_ptr(), nbytes, _stream())
    return idx, dist


RETRIEVAL_TC_MIN = 1 << 22      # Nq * Ndb from which the tensor-core filter beats the fp64 brute force (below: launch-bound)
RETRIEVAL_SEG = 1024            # pseudo-segment length of the single-database search (one warp pass per segment)


def retrieval_search(db: torch.Tensor, q: torch.Tensor, k: int, idx_offset: int = 0, want_dist: bool = True):
    """k nearest rows of ONE database for every query: (idx int32 [Nq, k] + idx_offset, squared dist float64 [Nq, k]).
    Large problems run the tensor-core filter over ~1000-row pseudo-segments and merge the per-segment lists
    (lpd_topk_merge); small ones the fp64 brute force.  Both give bit-identical results."""
    Ndb, D = db.shape
    Nq = q.shape[0]
    if Nq * Ndb < RETRIEVAL_TC_MIN or D % 4 or D > 1024 or k > Ndb:
        return retrieval_topk(db, q, k, idx_offset=idx_offset, want_dist=want_dist)
    seg = torch.arange(0, Ndb + RETRIEVAL_SEG, RETRIEVAL_SEG, device=db.device, dtype=torch.int32).clamp_(max=Ndb)
    idx, dist = retrieval_tc(db, q, k, seg, global_idx=True, idx_offset=idx_offset)
    if seg.numel() == 2:
        return idx[0], (dist[0] if want_dist else None)
    i, d = topk_merge(dist, idx)
    return i, (d if want_dist else None)


def recall_count(idx, q_run, R, truth_off, truth_idx, seg_thresh, seg_run=None, db=None, seg_off=None, q=None):
    """get_recall's counting for all (query, segment) units (lpd_recall_count) -> (hist int32 [R, S, 25], n_eval [R, S],
    n_onepct [R, S], sim float32 [Nq, S] or None)"""
    lib = _lib.load()
    S, Nq, k = idx.shape
    dev = idx.device
    counters = torch.zeros(R * S * 27, device=dev, dtype=torch.int32)
    hist, n_eval, n_one = counters[: R * S * 25], counters[R * S * 25: R * S * 26], counters[R * S * 26:]
    sim = torch.empty(Nq, S, device=dev, dtype=torch.float32) if db is not None else None
    D = 0 if db is None else db.shape[1]
    _call("lpd_recall_count", 1, lib.lpd_recall_count, idx.data_ptr(), S, Nq, k, q_run.data_ptr(), R, _p(seg_run),
          truth_off.data_ptr(), truth_idx.data_ptr(), seg_thresh.data_ptr(), _p(db), _p(seg_off), _p(q), D, hist.data_ptr(),
          n_eval.data_ptr(), n_one.data_ptr(), _p(sim), _stream())
    return hist.view(R, S, 25), n_eval.view(R, S), n_one.view(R, S), sim


# =====================================================================================================================
# train mode: batch-statistics BatchNorm, backward kernels, Adam (include/lpd_b200.h, "TRAIN MODE")
# =====================================================================================================================
SM_COUNT = 148


def _nparts(rows: int, per: int = 64) -> int:
    return int(max(1, min(SM_COUNT * 8, (rows + per - 1) // per)))


def _partial(nparts: int, C: int, dev) -> torch.Tensor:
    return torch.empty(nparts * 2 * C, device=dev, dtype=torch.float64)


def bn_finalize(partial, nparts, count, C, gamma, beta, eps, momentum, running_mean, running_var):
    """-> bn block [4, C] (scale, shift, mean, invstd); running stats updated in place."""
    lib = _lib.load()
    bn = torch.empty(4, C, device=partial.device, dtype=torch.float32)
    _call("lpd_bn_finalize", 1, lib.lpd_bn_finalize, partial.data_ptr(), nparts, float(count), C, _p(gamma), _p(beta), float(eps),
          float(momentum), _p(running_mean), _p(running_var), bn.data_ptr(), _stream())
    if running_mean is not None or running_var is not None:
        bump_weights_epoch()                                     # running statistics written through raw pointers
    return bn


def bn_stats(z, rows, C, ld):
    """column (sum, sum of squares) partials of z [rows, C] (ld) -> (partial, nparts)"""
    lib = _lib.load()
    nparts = _nparts(rows)
    part = _partial(nparts, C, z.device)
    _call(f"lpd_bn_stats[C={C}]", 1, lib.lpd_bn_stats, z.data_ptr(), rows, C, ld, part.data_ptr(), nparts, _stream())
    return part, nparts


def colsum_finalize(partial, nparts, n):
    lib = _lib.load()
    out = torch.empty(n, device=partial.device, dtype=torch.float32)
    _call("lpd_colsum_finalize", 1, lib.lpd_colsum_finalize, partial.data_ptr(), nparts, n, out.data_ptr(), _stream())
    return out


def affine_act(z, rows, C, ldz, scale, shift, act=ACT_NONE, slope=0.0, aux=None, ldaux=0, out=None, ldo=None):
    lib = _lib.load()
    if out is None:
        out = torch.empty(rows, C, device=z.device, dtype=torch.float32)
        ldo = C
    _call(f"lpd_affine_act[C={C}]", 1, lib.lpd_affine_act, z.data_ptr(), rows, C, ldz, _p(scale), _p(shift), act, float(slope),
          _p(aux), ldaux, out.data_ptr(), ldo, _stream())
    return out


def bn_bwd(dy, lddy, z, ldz, rows, C, bn, act, slope, count=None, aux=None, ldaux=0, dz=None, lddz=None):
    """backward of act(BN_batch(z)) -> (dz [rows, C], S [2, C] = (dbeta, dgamma)); dz may alias dy."""
    lib = _lib.load()
    nparts = _nparts(rows)
    part = _partial(nparts, C, z.device)
    _call(f"lpd_bn_bwd_reduce[C={C}]", 1, lib.lpd_bn_bwd_reduce, dy.data_ptr(), lddy, z.data_ptr(), ldz, rows, C, bn.data_ptr(),
          act, float(slope), _p(aux), ldaux, part.data_ptr(), nparts, _stream())
    S = colsum_finalize(part, nparts, 2 * C).view(2, C)
    if dz is None:
        dz = torch.empty(rows, C, device=z.device, dtype=torch.float32)
        lddz = C
    _call(f"lpd_bn_bwd_apply[C={C}]", 1, lib.lpd_bn_bwd_apply, dy.data_ptr(), lddy, z.data_ptr(), ldz, rows, C, bn.data_ptr(),
          S.data_ptr(), float(rows if count is None else count), act, float(slope), _p(aux), ldaux, dz.data_ptr(), lddz, _stream())
    return dz, S


def bn_bwd_sums(dy, lddy, z, ldz, rows, C, bn, act, slope):
    """only the (S1, S2) sums of the BN backward (used for arg-routed edge gradients)"""
    lib = _lib.load()
    nparts = _nparts(rows)
    part = _partial(nparts, C, z.device)
    _call(f"lpd_bn_bwd_reduce[C={C}]", 1, lib.lpd_bn_bwd_reduce, dy.data_ptr(), lddy, z.data_ptr(), ldz, rows, C, bn.data_ptr(),
          act, float(slope), None, 0, part.data_ptr(), nparts, _stream())
    return colsum_finalize(part, nparts, 2 * C).view(2, C)


def edge_sel_stats(p, ldp, q, ldq, idx, B, N, k, C, gamma):
    """-> (zsel [M, C], arg uint8 [M, C], partial, nparts) for z = p_j + q_i over all edges"""
    lib = _lib.load()
    M = B * N
    zsel = torch.empty(M, C, device=p.device, dtype=torch.float32)
    arg = torch.empty(M, C, device=p.device, dtype=torch.uint8)
    nparts = SM_COUNT * 8
    part = _partial(nparts, C, p.device)
    _call(f"lpd_edge_sel_stats[C={C}]", 1, lib.lpd_edge_sel_stats, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C,
          _p(gamma), zsel.data_ptr(), C, arg.data_ptr(), part.data_ptr(), nparts, _stream())
    return zsel, arg, part, nparts


def edge_materialize(p, ldp, q, ldq, idx, B, N, k, C, scale, shift, act, slope):
    lib = _lib.load()
    y = torch.empty(B * N * k, C, device=p.device, dtype=torch.float32)
    _call(f"lpd_edge_materialize[C={C}]", 1, lib.lpd_edge_materialize, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C,
          scale.data_ptr(), shift.data_ptr(), act, float(slope), y.data_ptr(), _stream())
    return y


def edge_sel_dense(z, M, k, C, gamma):
    lib = _lib.load()
    zsel = torch.empty(M, C, device=z.device, dtype=torch.float32)
    arg = torch.empty(M, C, device=z.device, dtype=torch.uint8)
    _call(f"lpd_edge_sel_dense[C={C}]", 1, lib.lpd_edge_sel_dense, z.data_ptr(), M, k, C, _p(gamma), zsel.data_ptr(), C,
          arg.data_ptr(), _stream())
    return zsel, arg


def edge_dense_bwd_apply(z, M, k, C, bn, S, count, act, slope, dx, lddx, zsel, arg):
    """in place on z: -> dz [M*k, C]"""
    lib = _lib.load()
    _call(f"lpd_edge_dense_bwd_apply[C={C}]", 1, lib.lpd_edge_dense_bwd_apply, z.data_ptr(), M, k, C, bn.data_ptr(), S.data_ptr(),
          float(count), act, float(slope), dx.data_ptr(), lddx, zsel.data_ptr(), C, arg.data_ptr(), z.data_ptr(), _stream())
    return z


def edge_bwd(p, ldp, q, ldq, idx, B, N, k, C, bn, act, slope, dx, lddx, arg, dy, dp, lddp, dq, lddq, S=None):
    """backward of a decomposed edge layer: fills dp (atomics, zeroed first) and dq; returns S [2, C] (dbeta, dgamma).
    If S is given (arg-routed gradient only: computed over the [M, C] arrays) the gather-reduce pass is skipped."""
    lib = _lib.load()
    count = B * N * k
    if S is None:
        nparts = SM_COUNT * 8
        part = _partial(nparts, C, p.device)
        _call(f"lpd_edge_bwd_reduce[C={C}]", 1, lib.lpd_edge_bwd_reduce, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C,
              bn.data_ptr(), act, float(slope), _p(dx), lddx, _p(arg), _p(dy), part.data_ptr(), nparts, _stream())
        S = colsum_finalize(part, nparts, 2 * C).view(2, C)
    _call(f"lpd_edge_bwd_apply[C={C}]", 2, lib.lpd_edge_bwd_apply, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C,
          bn.data_ptr(), act, float(slope), _p(dx), lddx, _p(arg), _p(dy), S.data_ptr(), float(count),
          dp.data_ptr(), lddp, _p(dq), lddq, _stream())
    return S


def edge_scatter_add(dy, idx, B, N, k, C, dp=None, lddp=None):
    """dp[j(i,m)] += dy[(i,m)] -> dp [B*N, C]"""
    lib = _lib.load()
    if dp is None:
        dp = torch.empty(B * N, C, device=dy.device, dtype=torch.float32)
        lddp = C
    _call(f"lpd_edge_scatter_add[C={C}]", 2, lib.lpd_edge_scatter_add, dy.data_ptr(), idx.data_ptr(), B, N, k, C, dp.data_ptr(), lddp, _stream())
    return dp


def act_bwd(dy, lddy, z, ldz, rows, C, act, slope, dz=None, lddz=None):
    """dz = dy * act'(z) for an activation that follows a plain (BatchNorm-free) layer: the BN backward with the identity
    statistics block (scale 1, shift 0, mean 0, invstd 1) and zero reduction terms."""
    lib = _lib.load()
    ident = torch.zeros(6, C, device=z.device, dtype=torch.float32)
    ident[0].fill_(1.0)
    ident[3].fill_(1.0)
    if dz is None:
        dz = torch.empty(rows, C, device=z.device, dtype=torch.float32)
        lddz = C
    _call(f"lpd_bn_bwd_apply[C={C}]", 1, lib.lpd_bn_bwd_apply, dy.data_ptr(), lddy, z.data_ptr(), ldz, rows, C, ident.data_ptr(),
          ident[4].data_ptr(), 1.0, act, float(slope), None, 0, dz.data_ptr(), lddz, _stream())
    return dz


def netvlad_finish_train(vlad, a, wc2, B, N, D, K=64):
    """in place on vlad [B, D, K] -> (v [B, D*K], asum [B, K], n1 [B, K], n2 [B])"""
    lib = _lib.load()
    dev = vlad.device
    asum = torch.empty(B, K, device=dev, dtype=torch.float32)
    n1 = torch.empty(B, K, device=dev, dtype=torch.float32)
    n2 = torch.empty(B, device=dev, dtype=torch.float32)
    _call("lpd_netvlad_finish_train", 1, lib.lpd_netvlad_finish_train, vlad.data_ptr(), a.data_ptr(), wc2.data_ptr(), B, N, D, K,
          asum.data_ptr(), n1.data_ptr(), n2.data_ptr(), _stream())
    return vlad.view(B, D * K), asum, n1, n2


def netvlad_finish_bwd(dv, v, wc2, asum, n1, n2, B, D, K=64):
    """in place on dv [B, D*K] -> (dvraw [B, D, K], dasum [B, K], dwc2 [D, K])"""
    lib = _lib.load()
    dasum = torch.empty(B, K, device=dv.device, dtype=torch.float32)
    dwc2 = torch.empty(D, K, device=dv.device, dtype=torch.float32)
    _call("lpd_netvlad_finish_bwd", 2, lib.lpd_netvlad_finish_bwd, dv.data_ptr(), v.data_ptr(), wc2.data_ptr(), asum.data_ptr(),
          n1.data_ptr(), n2.data_ptr(), B, D, K, dasum.data_ptr(), dwc2.data_ptr(), _stream())
    return dv.view(B, D, K), dasum, dwc2


def softmax64_bwd(da, a, dasum, M, N):
    lib = _lib.load()
    _call("lpd_softmax64_bwd", 1, lib.lpd_softmax64_bwd, da.data_ptr(), a.data_ptr(), _p(dasum), M, N, _stream())
    return da


def colmax_arg(x, B, N, C, ldx=None):
    lib = _lib.load()
    out = torch.empty(B, C, device=x.device, dtype=torch.float32)
    arg = torch.empty(B, C, device=x.device, dtype=torch.int32)
    _call("lpd_colmax_arg", 1, lib.lpd_colmax_arg, x.data_ptr(), B, N, C, C if ldx is None else ldx, out.data_ptr(), arg.data_ptr(), _stream())
    return out, arg


def colmax_bwd(dout, arg, B, N, C, dx, lddx):
    lib = _lib.load()
    _call("lpd_colmax_bwd", 1, lib.lpd_colmax_bwd, dout.data_ptr(), arg.data_ptr(), B, N, C, dx.data_ptr(), lddx, _stream())
    return dx


def adam(w, g, m, v, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0):
    lib = _lib.load()
    _call("lpd_adam", 1, lib.lpd_adam, w.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), w.numel(), float(lr), float(beta1),
          float(beta2), float(eps), float(weight_decay), int(step), float(grad_scale), _stream())
    bump_weights_epoch()                                         # parameters written through raw pointers


def axpy(y, ldy, x, ldx, rows, C, alpha=1.0):
    lib = _lib.load()
    _call("lpd_axpy", 1, lib.lpd_axpy, y.data_ptr(), ldy, x.data_ptr(), ldx, rows, C, float(alpha), _stream())
    return y


def wgrad(dz, lddz, a, lda, rows, Nout, Kin, out=None):
    """dW[n][k] = sum_r dz[r][n] * a[r][k]  (weight gradient of z = a . W^T), split over the rows and reduced in a fixed
    order (deterministic).  -> [Nout, Kin]"""
    bn = 256 if _precision != "fp32" else 128
    tiles = ((Nout + 127) // 128) * ((Kin + bn - 1) // bn)
    want = max(1, min(512, (2 * SM_COUNT + tiles - 1) // tiles, rows // 256 if rows >= 256 else 1))
    splits = 1
    while splits * 2 <= want and rows % (splits * 2) == 0:
        splits *= 2
    per = rows // splits
    part = torch.empty(splits, Nout, Kin, device=dz.device, dtype=torch.float32)
    if _tn_ok(dz, a, Nout, Kin, per, lddz, lda, splits):
        gemm_tf32_tn(dz, a, M=Nout, N=Kin, K=per, lda=lddz, ldb=lda, batch=splits, out=part)
    else:
        gemm(dz, a, a_layout=A_KM, b_layout=B_KN, M=Nout, N=Kin, K=per, lda=lddz, ldb=lda, out=part, ldc=Kin,
             batch=splits, strideA=per * lddz, strideB=per * lda, strideC=Nout * Kin)
    if splits == 1 and out is None:
        return part[0]
    res = splitk_reduce(part, splits, Nout, Kin)
    if out is not None:
        axpy(out, Kin, res, Kin, Nout, Kin, 1.0)
        return out
    return res


# ---- train precision mode -------------------------------------------------------------------------------------------
#   "default": training runs with the numerics of the precision mode above (fp32 storage of every activation and gradient)
#   "f16":     the train-mode forward and backward of featnet="lpdnet" keep the four [B*N*k, 128] tensors of the DG2 edge layer in
#              FP16: y1 (activated DG1 edge rows, rounded to nearest), z2e = y1 . W2^T (lpd_gemm_f16, fp32 accumulate), and their
#              gradients dz2e and dy1, stored as fp16(2^E * value) with one device-computed power-of-two exponent E per step
#              (include/lpd_b200.h, "f16 storage of the edge tensors").  Half the bytes of the step's largest tensors and 1.85 GB
#              less peak memory at 2 x 22 x 4096 points.  Needs get_precision() "tf32" or "f16"; z2e must fit fp16's range
#              (|z| < 65504), or the loss comes out non-finite.  lpdnetorigin and pointnet training ignore it.
_train_precision = "default"


def set_train_precision(mode: str) -> str:
    """Select "default" or "f16" storage of the LPD-Net DG2 edge tensors in training; returns the previous mode."""
    global _train_precision
    if mode not in ("default", "f16"):
        raise ValueError("train precision must be 'default' or 'f16'")
    prev, _train_precision = _train_precision, mode
    return prev


def get_train_precision() -> str:
    return _train_precision


def bn_stats_f16(z, rows, C, ld):
    """lpd_bn_stats over fp16 z -> (partial, nparts, minmax uint32 keys [2, C])"""
    lib = _lib.load()
    _f16(z, "z")
    nparts = _nparts(rows)
    part = _partial(nparts, C, z.device)
    minmax = torch.empty(2, C, device=z.device, dtype=torch.int32)
    _call(f"lpd_bn_stats_f16[C={C}]", 1, lib.lpd_bn_stats_f16, z.data_ptr(), rows, C, ld, part.data_ptr(), nparts, minmax.data_ptr(),
          _stream())
    return part, nparts, minmax


def edge_materialize_f16(p, ldp, q, ldq, idx, B, N, k, C, scale, shift, act, slope):
    lib = _lib.load()
    y = torch.empty(B * N * k, C, device=p.device, dtype=torch.float16)
    _call(f"lpd_edge_materialize_f16[C={C}]", 1, lib.lpd_edge_materialize_f16, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C,
          scale.data_ptr(), shift.data_ptr(), act, float(slope), y.data_ptr(), _stream())
    return y


def edge_sel_dense_f16(z, M, k, C, gamma):
    lib = _lib.load()
    _f16(z, "z")
    zsel = torch.empty(M, C, device=z.device, dtype=torch.float32)
    arg = torch.empty(M, C, device=z.device, dtype=torch.uint8)
    _call(f"lpd_edge_sel_dense_f16[C={C}]", 1, lib.lpd_edge_sel_dense_f16, z.data_ptr(), M, k, C, _p(gamma), zsel.data_ptr(), C,
          arg.data_ptr(), _stream())
    return zsel, arg


def edge_grad_scale_f16(dx, lddx, M, C, bn, S, count, act, slope, zminmax, w_h):
    """-> scale fp32 [2, K]: row 0 = 2^E, row 1 = 2^-E, E the exponent of the fp16 edge gradients (lpd_edge_grad_scale_f16);
    w_h: the layer's fp16 weight [C, K]"""
    lib = _lib.load()
    _f16(w_h, "w")
    K = w_h.shape[1]
    work = torch.empty(C, device=dx.device, dtype=torch.int32)
    scale = torch.empty(2, K, device=dx.device, dtype=torch.float32)
    _call(f"lpd_edge_grad_scale_f16[C={C}]", 2, lib.lpd_edge_grad_scale_f16, dx.data_ptr(), lddx, M, C, bn.data_ptr(), S.data_ptr(),
          float(count), act, float(slope), zminmax.data_ptr(), w_h.data_ptr(), w_h.stride(0), K, work.data_ptr(), scale.data_ptr(),
          _stream())
    return scale


def edge_dense_bwd_apply_f16(z, M, k, C, bn, S, count, act, slope, dx, lddx, zsel, arg, gscale):
    """in place on fp16 z: -> fp16 2^E * dz [M*k, C], gscale[0] = 2^E"""
    lib = _lib.load()
    _f16(z, "z")
    _call(f"lpd_edge_dense_bwd_apply_f16[C={C}]", 1, lib.lpd_edge_dense_bwd_apply_f16, z.data_ptr(), M, k, C, bn.data_ptr(),
          S.data_ptr(), float(count), act, float(slope), dx.data_ptr(), lddx, zsel.data_ptr(), C, arg.data_ptr(), z.data_ptr(),
          gscale.data_ptr(), _stream())
    return z


def edge_bwd_f16(p, ldp, q, ldq, idx, B, N, k, C, bn, act, slope, dx, lddx, arg, dy, dyscale, dp, lddp, dq, lddq):
    """edge_bwd with the dense incoming gradient given as fp16 dy = 2^E * gradient, dyscale[0] = 2^-E"""
    lib = _lib.load()
    _f16(dy, "dy")
    count = B * N * k
    nparts = SM_COUNT * 8
    part = _partial(nparts, C, p.device)
    _call(f"lpd_edge_bwd_reduce_f16[C={C}]", 1, lib.lpd_edge_bwd_reduce_f16, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C,
          bn.data_ptr(), act, float(slope), _p(dx), lddx, _p(arg), dy.data_ptr(), dyscale.data_ptr(), part.data_ptr(), nparts, _stream())
    S = colsum_finalize(part, nparts, 2 * C).view(2, C)
    _call(f"lpd_edge_bwd_apply_f16[C={C}]", 2, lib.lpd_edge_bwd_apply_f16, p.data_ptr(), ldp, _p(q), ldq, idx.data_ptr(), B, N, k, C,
          bn.data_ptr(), act, float(slope), _p(dx), lddx, _p(arg), dy.data_ptr(), dyscale.data_ptr(), S.data_ptr(), float(count),
          dp.data_ptr(), lddp, _p(dq), lddq, _stream())
    return S


def wgrad_f16(dz_h, lddz, a_h, lda, rows, Nout, Kin, scale):
    """dW[n][k] = scale[k] * sum_r dz_h[r][n] * a_h[r][k] for fp16 operands (the gradient dz_h stored scaled, scale = its inverse
    scale per output column): lpd_gemm_f16_tn over row slices that are multiples of 64 rows, then the fixed-order
    lpd_splitk_reduce.  -> fp32 [Nout, Kin]"""
    bn = 256
    tiles = ((Nout + 127) // 128) * ((Kin + bn - 1) // bn)
    want = max(1, min(512, (2 * SM_COUNT + tiles - 1) // tiles, rows // 256 if rows >= 256 else 1))
    splits = 1
    while splits * 2 <= want and rows % (splits * 2) == 0 and (rows // (splits * 2)) % 64 == 0:
        splits *= 2
    per = rows // splits
    part = torch.empty(splits, Nout, Kin, device=dz_h.device, dtype=torch.float32)
    gemm_f16_tn(dz_h, a_h, M=Nout, N=Kin, K=per, lda=lddz, ldb=lda, batch=splits, out=part)
    return splitk_reduce(part, splits, Nout, Kin, scale=scale)
