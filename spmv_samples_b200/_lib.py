"""ctypes binding of libspmvb200.so (the C ABI in include/spmv_b200.h).

There is no fallback of any kind: if the shared library is missing or a call returns a
non-zero status, this module raises.  `build()` compiles the library in-tree with nvcc for
sm_100a (cross-compiles without a GPU).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPMVB200_LIB") or os.path.join(_PKG, "libspmvb200.so")  # env: ablation builds
CSRC = os.path.join(_PKG, "csrc")

OK = 0
KIND_MERGE, KIND_VECTOR, KIND_LIGHT, KIND_AUTO, KIND_CUSPARSE, KIND_STREAM = 0, 1, 2, 3, 4, 5
FLAG_STATIC_PATTERN = 1   # SPMVB200_FLAG_STATIC_PATTERN
CG_JACOBI = 1             # SPMVB200_CG_JACOBI
GMRES_MAX_RESTART = 64    # SPMVB200_GMRES_MAX_RESTART
SEMIRINGS = {"plus_times": 0, "min_plus": 1, "max_plus": 2, "or_and": 3}
MAX_PEERS = 8
IPC_HANDLE_BYTES = 64


class SpmvB200Error(RuntimeError):
    def __init__(self, status: int, where: str, detail: str = ""):
        self.status = status
        super().__init__(f"{where}: status {status} ({detail})")


class Args(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("offset_bits", C.c_int32), ("value_bits", C.c_int32),
        ("n_peers", C.c_int32),
        ("n_rows", C.c_int64), ("n_cols", C.c_int64), ("nnz", C.c_int64),
        ("Ap", C.c_void_p), ("Aj", C.c_void_p), ("Ax", C.c_void_p), ("x", C.c_void_p),
        ("y", C.c_void_p), ("alpha_dev", C.c_void_p), ("y_peers", C.POINTER(C.c_void_p)),
        ("stream", C.c_void_p),
        ("semiring", C.c_int32), ("flags", C.c_int32), ("beta_dev", C.c_void_p),
    ]


class SpmmArgs(C.Structure):
    _fields_ = [
        ("offset_bits", C.c_int32), ("value_bits", C.c_int32), ("k", C.c_int32), ("reserved", C.c_int32),
        ("n_rows", C.c_int64), ("n_cols", C.c_int64), ("nnz", C.c_int64),
        ("Ap", C.c_void_p), ("Aj", C.c_void_p), ("Ax", C.c_void_p), ("X", C.c_void_p),
        ("ldx", C.c_int64), ("Y", C.c_void_p), ("ldy", C.c_int64), ("alpha_dev", C.c_void_p),
        ("stream", C.c_void_p),
    ]


class CgArgs(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("offset_bits", C.c_int32), ("value_bits", C.c_int32), ("flags", C.c_int32),
        ("n", C.c_int64), ("nnz", C.c_int64),
        ("Ap", C.c_void_p), ("Aj", C.c_void_p), ("Ax", C.c_void_p), ("b", C.c_void_p), ("x", C.c_void_p),
        ("rtol", C.c_double), ("max_iter", C.c_int64), ("stream", C.c_void_p),
    ]


class CgOut(C.Structure):
    _fields_ = [
        ("iterations", C.c_int64), ("residual_norm", C.c_double), ("b_norm", C.c_double),
        ("converged", C.c_int32), ("breakdown", C.c_int32),
    ]


class RowStats(C.Structure):
    _fields_ = [
        ("n_rows", C.c_int64), ("nnz", C.c_int64), ("max_row_len", C.c_int64),
        ("empty_rows", C.c_int64), ("mean_row_len", C.c_double), ("std_row_len", C.c_double),
        ("chosen_kind", C.c_int32), ("chosen_width", C.c_int32),
    ]


_lib = None


def build(verbose: bool = False) -> str:
    """Compile libspmvb200.so in-tree (nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo)."""
    jobs = str(min(8, os.cpu_count() or 1))
    r = subprocess.run(["make", "-C", CSRC, "-j", jobs], capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libspmvb200.so failed:\n" + (r.stdout or "") + (r.stderr or ""))
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C spmv_samples_b200/csrc`. There is no CPU or PyTorch fallback.")
    L = C.CDLL(LIB_PATH)
    L.spmvb200_status_string.restype = C.c_char_p
    L.spmvb200_last_cuda_error.restype = C.c_char_p
    L.spmvb200_version.restype = C.c_char_p
    L.spmvb200_spmv.argtypes = [C.POINTER(Args)]
    L.spmvb200_spmv.restype = C.c_int
    L.spmvb200_spmm.argtypes = [C.POINTER(SpmmArgs)]
    L.spmvb200_spmm.restype = C.c_int
    L.spmvb200_cg.argtypes = [C.POINTER(CgArgs), C.POINTER(CgOut)]
    L.spmvb200_cg.restype = C.c_int
    L.spmvb200_bicgstab.argtypes = [C.POINTER(CgArgs), C.POINTER(CgOut)]
    L.spmvb200_bicgstab.restype = C.c_int
    L.spmvb200_gmres.argtypes = [C.POINTER(CgArgs), C.c_int32, C.POINTER(CgOut)]
    L.spmvb200_gmres.restype = C.c_int
    L.spmvb200_launch_count.restype = C.c_int64
    L.spmvb200_get_option.restype = C.c_int64
    L.spmvb200_get_option.argtypes = [C.c_char_p]
    L.spmvb200_set_option.argtypes = [C.c_char_p, C.c_int64]
    L.spmvb200_merge_tile_items.restype = C.c_int64
    L.spmvb200_merge_tile_items.argtypes = [C.c_int, C.c_int]
    L.spmvb200_row_stats.argtypes = [C.c_int, C.c_int64, C.c_int64, C.c_void_p,
                                     C.POINTER(RowStats), C.c_void_p]
    L.spmvb200_merge_path_partition_o32.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_int64,
                                                    C.c_int64, C.c_void_p, C.c_void_p]
    L.spmvb200_merge_path_partition_o64.argtypes = [C.c_int32, C.c_int64, C.c_void_p, C.c_int64,
                                                    C.c_int64, C.c_void_p, C.c_void_p]
    L.spmvb200_row_split_o32.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.c_int,
                                         C.POINTER(C.c_int64), C.c_void_p]
    L.spmvb200_row_split_o64.argtypes = [C.c_int32, C.c_int64, C.c_void_p, C.c_int,
                                         C.POINTER(C.c_int64), C.c_void_p]
    for tag in ("o32", "o64"):
        getattr(L, f"spmvb200_rows_at_cost_{tag}").argtypes = [
            C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.POINTER(C.c_int64),
            C.POINTER(C.c_int64), C.c_void_p]
    L.spmvb200_gen_uniform_pm1.argtypes = [C.c_int, C.c_uint64, C.c_uint32, C.c_uint64, C.c_int64,
                                           C.c_void_p, C.c_void_p]
    L.spmvb200_gen_lap2d.argtypes = [C.c_int, C.c_int, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]
    L.spmvb200_gen_uniform_rows.argtypes = [C.c_int, C.c_int, C.c_int32, C.c_int32, C.c_int32,
                                            C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p]
    L.spmvb200_gen_rmat_edges.argtypes = [C.c_int32, C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p,
                                          C.c_void_p, C.c_void_p]
    L.spmvb200_coo_to_csr.argtypes = [C.c_int, C.c_int, C.c_int32, C.c_int64, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p]
    L.spmvb200_matrix_create.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64,
                                         C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.POINTER(C.c_void_p)]
    L.spmvb200_matrix_create_from_device.argtypes = L.spmvb200_matrix_create.argtypes
    L.spmvb200_sum_squares.argtypes = [C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.spmvb200_inv_sqrt.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.spmvb200_power_create.argtypes = [C.c_int, C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int64, C.c_int64,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
    L.spmvb200_power_create_from_device.argtypes = L.spmvb200_power_create.argtypes
    L.spmvb200_power_reset.argtypes = [C.c_void_p]
    L.spmvb200_power_steps.argtypes = [C.c_void_p, C.c_int]
    L.spmvb200_power_run.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
    L.spmvb200_power_sync.argtypes = [C.c_void_p]
    L.spmvb200_power_get.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    L.spmvb200_power_destroy.argtypes = [C.c_void_p]
    L.spmvb200_power_exchange.argtypes = [C.c_void_p]
    L.spmvb200_power_destroy.restype = None
    L.spmvb200_norm_exchange.argtypes = [C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_uint64,
                                         C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
    L.spmvb200_main_kernel_time.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    L.spmvb200_device_malloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    L.spmvb200_device_free.argtypes = [C.c_void_p]
    L.spmvb200_matrix_spmv_host.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.spmvb200_matrix_submit_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.spmvb200_matrix_wait.argtypes = [C.c_void_p, C.c_int]
    L.spmvb200_matrix_destroy.argtypes = [C.c_void_p]
    L.spmvb200_matrix_destroy.restype = None
    L.spmvb200_ipc_export.argtypes = [C.c_void_p, C.c_char_p]
    L.spmvb200_ipc_open.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
    L.spmvb200_ipc_close.argtypes = [C.c_void_p]
    L.spmvb200_release_cache.restype = None
    L.spmvb200_gather_yardstick.argtypes = [C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.POINTER(C.c_double)]
    L.spmvb200_hot_x_table_info.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    L.spmvb200_hot_x_info.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_double),
                                      C.POINTER(C.c_double)]
    for kind in ("merge", "vector", "light", "stream", "auto", "cusparse"):
        for otag, otype in (("o32", C.c_int32), ("o64", C.c_int64)):
            for vtag in ("f32", "f64"):
                fn = getattr(L, f"spmvb200_{kind}_i32_{otag}_{vtag}")
                fn.argtypes = [C.c_int32, C.c_int32, otype, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p]
                fn.restype = C.c_int
    _lib = L
    return L


def check(status: int, where: str) -> None:
    if status != OK:
        L = lib()
        detail = L.spmvb200_status_string(status).decode()
        if status in (3, 5):
            detail += ": " + L.spmvb200_last_cuda_error().decode()
        raise SpmvB200Error(status, where, detail)


def exported_symbols():
    """Names declared in include/spmv_b200.h (parsed), for the load/export test."""
    import re

    hdr = os.path.join(os.path.dirname(_PKG), "include", "spmv_b200.h")
    text = open(hdr).read()
    names = set(re.findall(r"SPMVB200_API\s+[^;(]*?\b(spmvb200_\w+)\s*\(", text))
    for kind in re.findall(r"SPMVB200_DECLARE_KIND\((\w+)\)", text):
        if kind == "KIND":
            continue
        for otag in ("o32", "o64"):
            for vtag in ("f32", "f64"):
                names.add(f"spmvb200_{kind}_i32_{otag}_{vtag}")
    return sorted(names)
