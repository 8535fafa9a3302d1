"""ctypes binding of the C ABI declared in ``include/bof_b200.h``.

This is test/bench plumbing only: the product is the CUDA library plus the C++ adapters that keep
the reference's ``flash_blas.h`` signatures.  There is no fallback of any kind -- if the shared
library is missing the import of :func:`load` raises, and every compute entry point needs a B200.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libbof_b200.so"

BOF_OK, BOF_EINVAL, BOF_ECUDA, BOF_ENOMEM, BOF_ENODEV, BOF_EIO = 0, -1, -2, -3, -4, -5


class BofConfig(C.Structure):
    _fields_ = [
        ("device", C.c_int32),
        ("n_copy_threads", C.c_int32),
        ("stage_bytes", C.c_uint64),
        ("n_stage_bufs", C.c_int32),
        ("csrmm_max_nnz", C.c_uint64),
        ("gemm_row_block", C.c_uint64),
        ("gemm_k_chunk", C.c_int32),
        ("gemm_force_path", C.c_int32),
        ("gemm_wave_sync", C.c_int32),
        ("gemm_split", C.c_int32),
        ("radix_max_bits", C.c_int32),
        ("spmv_t_atomic", C.c_int32),
    ]


class BofStats(C.Structure):
    _fields_ = [
        ("h2d_bytes", C.c_double),
        ("d2h_bytes", C.c_double),
        ("h2d_ms", C.c_double),
        ("d2h_ms", C.c_double),
        ("kernel_ms", C.c_double),
        ("stage_in_ms", C.c_double),
        ("stage_out_ms", C.c_double),
        ("total_ms", C.c_double),
        ("kernel_launches", C.c_int64),
    ]


_vp, _i64, _f32, _ch, _sz = C.c_void_p, C.c_int64, C.c_float, C.c_char, C.c_size_t

# name -> (restype, argtypes); must list every symbol of include/bof_b200.h (tests check this)
PROTOTYPES = {
    "bof_abi_version": (C.c_int, []),
    "bof_ctx_create": (C.c_int, [C.POINTER(BofConfig), C.POINTER(_vp)]),
    "bof_ctx_destroy": (C.c_int, [_vp]),
    "bof_last_error": (C.c_char_p, [_vp]),
    "bof_get_stats": (C.c_int, [_vp, C.POINTER(BofStats)]),
    "bof_launch_count": (_i64, [_vp]),
    "bof_register_mapping": (C.c_int, [_vp, _sz, C.c_int, C.c_uint64]),
    "bof_unregister_mapping": (C.c_int, [_vp]),
    "bof_spmm_csr_f32": (C.c_int, [_vp, _vp, _ch, _i64, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _i64, _f32,
                                   _vp, _i64, _vp, _sz]),
    "bof_spmm_workspace_bytes": (_sz, [_ch, _i64, _i64, _i64]),
    "bof_spmv_csr_f32": (C.c_int, [_vp, _vp, _ch, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "bof_idx_narrow": (C.c_int, [_vp, _vp, _vp, _vp, _i64]),
    "bof_idx_widen": (C.c_int, [_vp, _vp, _vp, _vp, _i64]),
    "bof_sgemm_f32": (C.c_int, [_vp, _vp, _ch, _ch, _ch, _i64, _i64, _i64, _f32, _vp, _i64, _vp, _i64, _f32,
                                _vp, _i64, _vp, _sz]),
    "bof_sgemm_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "bof_sgemv_f32": (C.c_int, [_vp, _vp, _ch, _ch, _i64, _i64, _f32, _vp, _i64, _vp, _f32, _vp, _vp, _sz]),
    "bof_sgemv_workspace_bytes": (_sz, [_ch, _ch, _i64, _i64]),
    "bof_tc_issue_rate": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "bof_csr2csc": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz]),
    "bof_csr2csc_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "bof_row_sqnorm_f32": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _vp]),
    "bof_kmeans_assign": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz]),
    "bof_kmeans_workspace_bytes": (_sz, [_i64, _i64, _i64, C.c_int]),
    "bof_kmeans_point_planes_bytes": (_sz, [_i64, _i64]),
    "bof_kmeans_prepare_points": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp]),
    "bof_kmeans_reduce": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _sz]),
    "bof_kmeans_reduce_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "bof_kmeans_finalize": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp]),
    "bof_host_csrmm": (C.c_int, [_vp, _ch, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _ch, _vp, _vp]),
    "bof_host_gemm": (C.c_int, [_vp, _ch, _ch, _ch, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _i64, _i64,
                                _i64]),
    "bof_host_gemm_devb": (C.c_int, [_vp, _ch, _ch, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _i64, _i64, _i64]),
    "bof_host_csrmm_devb": (C.c_int, [_vp, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _vp, _vp]),
    "bof_host_kmeans_dist": (C.c_int, [_vp, _ch, _ch, _ch, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _i64, _i64, _i64,
                                       _vp, _vp]),
    "bof_host_gemv": (C.c_int, [_vp, _ch, _ch, _i64, _i64, _f32, _f32, _vp, _i64, _vp, _vp]),
    "bof_host_csrgemv": (C.c_int, [_vp, _ch, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "bof_host_csrcsc": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "bof_csr_open": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, C.POINTER(_vp)]),
    "bof_csr_build_transpose": (C.c_int, [_vp]),
    "bof_csr_arrays": (C.c_int, [_vp, _ch, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i64)]),
    "bof_csr_mm": (C.c_int, [_vp, _ch, _i64, _f32, _f32, _ch, _vp, _vp]),
    "bof_csr_mv": (C.c_int, [_vp, _ch, _vp, _vp]),
    "bof_csr_close": (C.c_int, [_vp]),
    "bof_kmeans_open": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, C.POINTER(_vp)]),
    "bof_kmeans_local_step": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_sz)]),
    "bof_kmeans_update": (C.c_int, [_vp]),
    "bof_kmeans_get": (C.c_int, [_vp, _vp, _vp]),
    "bof_kmeans_allreduce": (C.c_int, [_vp]),
    "bof_kmeans_lloyd": (C.c_int, [_vp, _i64]),
    "bof_kmeans_stream": (_vp, [_vp]),
    "bof_comm_unique_id": (C.c_int, [_vp]),
    "bof_comm_init": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "bof_comm_finalize": (C.c_int, [_vp]),
    "bof_comm_world": (C.c_int, [_vp]),
    "bof_comm_rank": (C.c_int, [_vp]),
    "bof_dist_gemm": (C.c_int, [_vp, _ch, _ch, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _i64, _i64, _i64]),
    "bof_dist_csrmm": (C.c_int, [_vp, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _vp, _vp]),
    "bof_mgpu_create": (C.c_int, [C.POINTER(BofConfig), C.c_int, _vp, C.POINTER(_vp)]),
    "bof_mgpu_destroy": (C.c_int, [_vp]),
    "bof_mgpu_count": (C.c_int, [_vp]),
    "bof_mgpu_ctx": (_vp, [_vp, C.c_int]),
    "bof_mgpu_last_error": (C.c_char_p, [_vp]),
    "bof_mgpu_gemm": (C.c_int, [_vp, _ch, _ch, _ch, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _i64, _i64, _i64]),
    "bof_mgpu_csrmm": (C.c_int, [_vp, _ch, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _vp, _ch, _vp, _vp]),
    "bof_mgpu_csrgemv": (C.c_int, [_vp, _ch, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "bof_mgpu_gemv": (C.c_int, [_vp, _ch, _ch, _i64, _i64, _f32, _f32, _vp, _i64, _vp, _vp]),
    "bof_mgpu_kmeans_lloyd": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _i64, _vp]),
    "bof_kmeans_close": (C.c_int, [_vp]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library (built by ``__graft_entry__.build()``); never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` at the repo "
            "root (nvcc, sm_100a). There is no CPU or PyTorch fallback for this path.")
    lib = C.CDLL(os.fspath(LIB_PATH), mode=C.RTLD_GLOBAL)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here == ABI drift
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class BofError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"bof_b200 error {code}: {msg}")
        self.code = code


def ch(c: str) -> bytes:
    return c.encode("ascii")[:1]


def ptr(x) -> int | None:
    """Raw address of a numpy array / torch tensor / int / None."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    if hasattr(x, "ctypes"):
        return x.ctypes.data
    raise TypeError(type(x))
