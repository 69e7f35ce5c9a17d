"""ctypes binding of liblpd_b200.so (the C ABI declared in include/lpd_b200.h).

The library is the product: there is no Python / torch fallback.  Importing this module without the
built shared object, or calling into it without a CUDA device, raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "liblpd_b200.so"

# status codes / enums mirrored from include/lpd_b200.h
LPD_OK = 0
ACT_NONE, ACT_RELU, ACT_LEAKY, ACT_SIGMOID, ACT_GATE, ACT_ADD = 0, 1, 2, 3, 4, 5
A_MK, A_KM = 0, 1
B_NK, B_KN = 0, 1
ABI_VERSION = 2

_vp, _i, _f, _ll, _sz, _d = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_size_t, C.c_double

# name -> (restype, argtypes); every symbol include/lpd_b200.h declares
SIGNATURES = {
    "lpd_abi_version": (_i, []),
    "lpd_status_str": (C.c_char_p, [_i]),
    "lpd_last_cuda_error": (C.c_char_p, []),
    "lpd_device_info": (_i, [C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_sz)]),
    "lpd_bn_fold": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp, _vp]),
    "lpd_transpose": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "lpd_knn": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "lpd_knn_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "lpd_knn_tc": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _sz, _vp]),
    "lpd_knn_tc_variant": (_i, [_i]),
    "lpd_knn_tc_flags_offset": (_sz, [_i, _i, _i, _i]),
    "lpd_knn_xyz_workspace_bytes": (_sz, [_i, _i]),
    "lpd_knn_xyz": (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _sz, _vp]),
    "lpd_cell_order": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "lpd_cell_order_grid": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "lpd_knn_xyz_ordered": (_i, [_i, _i, _i, _vp, _i, _vp, _sz, _vp]),
    "lpd_gemm": (_i, [_vp, _i, _i, _ll, _vp, _i, _i, _ll, _vp, _i, _ll, _i, _i, _i, _i,
                      _vp, _vp, _i, _f, _vp, _vp]),
    "lpd_gemm_tf32": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _f, _vp]),
    "lpd_gemm_tf32_ex": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _f, _vp]),
    "lpd_gemm_tf32_tn": (_i, [_vp, _i, _vp, _i, _vp, _i, _ll, _i, _i, _i, _i, _vp]),
    "lpd_gemm_f16": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _f, _vp]),
    "lpd_gemm_f16_tn": (_i, [_vp, _i, _vp, _i, _vp, _i, _ll, _i, _i, _i, _i, _vp]),
    "lpd_f32_to_f16": (_i, [_vp, _ll, _vp, _ll, _ll, _i, _vp]),
    "lpd_split3_tf32": (_i, [_vp, _ll, _vp, _i, _vp]),
    "lpd_transpose_split3": (_i, [_vp, _i, _ll, _i, _vp, _vp]),
    "lpd_gemm_tf32_out16": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _f, _vp]),
    "lpd_softmax64_f16": (_i, [_vp, _ll, _vp, _vp]),
    "lpd_edge_gather_max_f16": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _f, _vp, _i, _vp]),
    "lpd_edgeconv_dg20_f16": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _f, _vp, _i, _vp, _i, _vp]),
    "lpd_edgeconv_dg32_f16": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _f, _vp, _i, _vp, _i, _vp]),
    "lpd_edgeconv_dg64_f16": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _f, _vp, _i, _vp]),
    "lpd_pointwise_mlp2": (_i, [_vp, _i, _i, _ll, _vp, _vp, _vp, _vp, _vp, _vp, _i, _f, _vp, _i, _vp]),
    "lpd_colmax": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "lpd_edge_gather_ext": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _f, _vp, _i, _vp]),
    "lpd_edgeconv_dg": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _f,
                             _vp, _i, _vp, _i, _vp]),
    "lpd_edgeconv_dg_tf32": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _f,
                                  _vp, _i, _vp, _i, _vp]),
    "lpd_netvlad_assign": (_i, [_vp, _i, _i, _vp, _vp, _vp, _i, _vp, _vp]),
    "lpd_softmax64": (_i, [_vp, _ll, _vp]),
    "lpd_netvlad_finish": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "lpd_splitk_reduce": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "lpd_gemm_softmax64": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lpd_netvlad_finish_parts": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _vp]),
    "lpd_hidden_gate": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lpd_quadruplet_loss": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _f, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "lpd_retrieval_workspace_bytes": (_sz, [_i, _i, _i]),
    "lpd_retrieval_topk": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "lpd_topk_merge": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "lpd_retrieval_tc_workspace_bytes": (_sz, [_i, _i, _i]),
    "lpd_retrieval_tc": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "lpd_recall_count": (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    # ---- train mode ----
    "lpd_bn_stats": (_i, [_vp, _ll, _i, _i, _vp, _i, _vp]),
    "lpd_bn_finalize": (_i, [_vp, _i, _d, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp]),
    "lpd_colsum_finalize": (_i, [_vp, _i, _i, _vp, _vp]),
    "lpd_affine_act": (_i, [_vp, _ll, _i, _i, _vp, _vp, _i, _f, _vp, _i, _vp, _i, _vp]),
    "lpd_bn_bwd_reduce": (_i, [_vp, _i, _vp, _i, _ll, _i, _vp, _i, _f, _vp, _i, _vp, _i, _vp]),
    "lpd_bn_bwd_apply": (_i, [_vp, _i, _vp, _i, _ll, _i, _vp, _vp, _d, _i, _f, _vp, _i, _vp, _i, _vp]),
    "lpd_edge_sel_stats": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _i, _vp]),
    "lpd_edge_materialize": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _i, _f, _vp, _vp]),
    "lpd_edge_sel_dense": (_i, [_vp, _ll, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "lpd_edge_dense_bwd_apply": (_i, [_vp, _ll, _i, _i, _vp, _vp, _d, _i, _f, _vp, _i, _vp, _i, _vp, _vp, _vp]),
    "lpd_edge_bwd_reduce": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _f, _vp, _i, _vp, _vp, _vp, _i, _vp]),
    "lpd_edge_bwd_apply": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _f, _vp, _i, _vp, _vp, _vp, _d,
                                _vp, _i, _vp, _i, _vp]),
    "lpd_edge_scatter_add": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "lpd_netvlad_finish_train": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "lpd_netvlad_finish_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "lpd_softmax64_bwd": (_i, [_vp, _vp, _vp, _ll, _i, _vp]),
    "lpd_colmax_arg": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "lpd_colmax_bwd": (_i, [_vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "lpd_adam": (_i, [_vp, _vp, _vp, _vp, _ll, _f, _f, _f, _f, _f, _i, _f, _vp]),
    "lpd_axpy": (_i, [_vp, _i, _vp, _i, _ll, _i, _f, _vp]),
}

_lib = None


class LpdError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared object once; fail loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("LPD_B200_LIB", LIB_PATH))
    if not path.exists():
        raise LpdError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"or `make -C {_HERE / 'csrc'}`; there is no CPU or torch fallback.")
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.lpd_abi_version() != ABI_VERSION:
        raise LpdError(f"ABI version mismatch: library {lib.lpd_abi_version()} != binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != LPD_OK:
        lib = load()
        msg = lib.lpd_status_str(rc).decode()
        detail = lib.lpd_last_cuda_error().decode()
        raise LpdError(f"{what} failed: {msg}" + (f" [{detail}]" if detail else ""))


def device_info() -> dict:
    lib = load()
    sm, maj, mnr, smem = _i(), _i(), _i(), _sz()
    check(lib.lpd_device_info(C.byref(sm), C.byref(maj), C.byref(mnr), C.byref(smem)), "lpd_device_info")
    return {"sm_count": sm.value, "cc": (maj.value, mnr.value), "smem_optin": smem.value}
