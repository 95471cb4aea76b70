"""ctypes binding of ``libpegncde.so`` (the C-ABI declared in ``include/pegncde.h``).

There is NO fallback: if the shared library is missing the import of this module raises,
and every compute entry point raises :class:`PegError` on a non-zero status.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PEGNCDE_LIB") or os.path.join(_HERE, "libpegncde.so")   # PEGNCDE_LIB: A/B builds of the same ABI (tools/)

PEG_FLAG_TENSOR_CORES = 1
PEG_FLAG_TF32_FAST = 2
PEG_FLAG_DIRECTED = 4
PEG_FLAG_ADJ_LIGHT = 8
PEG_FLAG_NO_FUSED_SMALL = 64
PEG_FLAG_FUSED_SMALL = 128
PEG_FLAG_TF32X3 = 16
PEG_FLAG_BF16X2 = 32

PEG_WS_VF_FWD, PEG_WS_VF_VJP, PEG_WS_SOLVE_FWD, PEG_WS_SOLVE_BWD, PEG_WS_STEP = range(5)


class PegDims(Structure):
    _fields_ = [(k, c_int32) for k in ("B", "n", "ldn", "h", "e", "L", "T", "flags")]


class PegShard(Structure):
    """Row-sharded mode (include/pegncde.h): the pointer tables are HOST arrays of `world` device pointers."""
    _fields_ = [("rank", c_int32), ("world", c_int32), ("n_glob", c_int32), ("row0", c_int32), ("adj_coef_t", c_void_p),
                ("vt_hi", POINTER(c_void_p)), ("vt_lo", POINTER(c_void_p)), ("vexp", POINTER(c_void_p)), ("colsum", POINTER(c_void_p)),
                ("flags", POINTER(c_void_p)), ("epoch", POINTER(ctypes.c_uint32)), ("epoch_dev", c_void_p)]


class PegAdaptState(Structure):
    """Per-trajectory state of the device-side step-size controller (include/pegncde.h)."""
    _fields_ = [("tprev", c_float), ("tnext", c_float), ("done", c_int32), ("nacc", c_int32), ("attempts", c_int32), ("rejected", c_int32),
                ("mi", c_int32), ("mi0", c_int32), ("mi1", c_int32), ("keep", c_int32), ("h", c_float), ("overflow", c_int32)]


class PegSparse(Structure):
    """Sparse (CSR) adjacency path of one batch (include/pegncde.h): absolute row offsets, both orientations."""
    _fields_ = [("nnz", c_int64), ("nnz_stride", c_int64)] + [(k, c_void_p) for k in ("row_ptr", "col", "coef", "row_ptr_t", "col_t", "coef_t")]


class PegControl(Structure):
    _fields_ = [(k, c_void_p) for k in ("ts", "adj_coef", "adj_rowsum", "adj_diag", "adj_total", "tch_coef", "x_coef", "adj_colsum", "adj_absmax")] + [("shard", POINTER(PegShard)), ("sparse", POINTER(PegSparse)), ("adj_static", c_void_p)]


class PegError(RuntimeError):
    def __init__(self, code: int, where: str):
        self.code = code
        msg = lib().pegncde_strerror(code).decode()
        extra = ""
        if code == 4:
            extra = f" [cudaError {lib().pegncde_last_cuda_error()}]"
        super().__init__(f"{where}: pegncde error {code}: {msg}{extra}")


_lib = None

# name -> (restype, argtypes); mirrors include/pegncde.h one to one
_P = c_void_p
_DIMS = POINTER(PegDims)
_CTL = POINTER(PegControl)
SIGNATURES = {
    "pegncde_param_count": (c_size_t, [_DIMS]),
    "pegncde_param_offsets": (c_int, [_DIMS, POINTER(c_int64)]),
    "pegncde_pack_adj": (c_int, [_P, _DIMS, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pegncde_pack_adj_range": (c_int, [_P, _DIMS, c_int32, c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pegncde_adj_stats": (c_int, [_P, _DIMS, _P, _P, _P, _P, _P]),
    "pegncde_build_adj": (c_int, [_P, _DIMS, _P, _P, _P, _P, _P, _P, _P]),
    "pegncde_adj_colsums": (c_int, [_P, _DIMS, _P, _P]),
    "pegncde_build_adj_rect": (c_int, [_P, _DIMS, c_int32, c_int32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pegncde_shard_buffer_bytes": (c_int, [_DIMS, c_int32, POINTER(c_size_t)]),
    "pegncde_adj_absmax": (c_int, [_P, _DIMS, c_int32, c_int32, _P, _P]),
    "pegncde_build_adj_sparse": (c_int, [_P, _DIMS, POINTER(PegSparse), _P, _P, _P, _P, _P, _P, _P, _P]),
    "pegncde_pack_adj_sparse": (c_int, [_P, _DIMS, POINTER(PegSparse), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pegncde_build_adj_static": (c_int, [_P, _DIMS, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pegncde_pack_x": (c_int, [_P, _DIMS, _P, _P, _P, _P, _P]),
    "pegncde_workspace_bytes": (c_size_t, [_DIMS, c_int32, c_int32]),
    "pegncde_vf_fwd": (c_int, [_P, _DIMS, _CTL, _P, c_float, _P, _P, _P, c_size_t]),
    "pegncde_vf_vjp": (c_int, [_P, _DIMS, _CTL, _P, c_float, _P, _P, _P, _P, _P, _P, c_size_t]),
    "pegncde_vf_vjp_adj": (c_int, [_P, _DIMS, _CTL, _P, c_float, _P, _P, _P, _P, _P, _P, _P, c_size_t]),
    "pegncde_step_fwd": (c_int, [_P, _DIMS, _CTL, _P, c_float, c_float, _P, _P, c_int32, _P, _P, _P, _P, _P, c_size_t]),
    "pegncde_step_fwd_batched": (c_int, [_P, _DIMS, _CTL, _P, _P, _P, _P, _P, c_int32, _P, _P, _P, _P, _P, c_size_t]),
    "pegncde_adaptive_control": (c_int, [_P, _DIMS, _P, c_float, c_float, c_float, c_float, c_float, c_float, c_int32, _P, c_int32, c_int32,
                                         _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "pegncde_tsit5_dense": (c_int, [_P, _DIMS, c_float, c_float, _P, _P, _P, _P, _P]),
    "pegncde_tsit5_dense_weights": (None, [c_float, POINTER(c_float)]),
    "pegncde_scaled_sumsq": (c_int, [_P, _DIMS, _P, _P, _P, _P, c_float, c_float, _P]),
    "pegncde_solve_fwd": (c_int, [_P, _DIMS, _CTL, _P, POINTER(c_float), c_int32, _P, _P, _P, _P, _P, c_size_t]),
    "pegncde_stage_store_bytes": (c_size_t, [_DIMS, c_int32]),
    "pegncde_solve_bwd": (c_int, [_P, _DIMS, _CTL, _P, POINTER(c_float), c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t]),
    "pegncde_solve_bwd_adj": (c_int, [_P, _DIMS, _CTL, _P, POINTER(c_float), c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t]),
    "pegncde_strerror": (c_char_p, [c_int]),
    "pegncde_last_cuda_error": (c_int, []),
    "pegncde_version": (c_char_p, []),
    "pegncde_launch_count": (c_uint64, []),
    "pegncde_profile_enable": (c_int, [c_int32]),
    "pegncde_profile_read": (c_int, [c_int32, POINTER(c_uint64), POINTER(c_uint64), POINTER(c_double), POINTER(c_double), POINTER(c_double)]),
}


def lib() -> ctypes.CDLL:
    """Loads libpegncde.so (built by ``__graft_entry__.build()`` / ``csrc/Makefile``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA extension is mandatory (no CPU fallback). "
                "Build it with `python -c 'import __graft_entry__ as g; g.build()'` or `make -C "
                "perm_equiv_graph_neural_cdes_b200/csrc`."
            )
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(code: int, where: str) -> None:
    if code != 0:
        raise PegError(code, where)
