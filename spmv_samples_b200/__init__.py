"""spmv_samples_b200 -- B200-native CSR SpMV behind the plugin surface of
peakcrosser7/spmv-samples.

The product is libspmvb200.so (hand-written sm_100a kernels, C ABI in include/spmv_b200.h)
plus the C++ host headers in include/ (spmv.h, load.hpp, timer.hpp) and main.cu.  This
Python package is the thin binding used by tests, bench.py and the multi-GPU driver:

    spmv      SpMV(kind_str, n_rows, n_cols, nnz, Ap, Aj, Ax, x, y) and SPMV_KINDS
    generate  device-side synthetic matrices (BASELINE.json configs c1..c5)
    matrix    CsrMatrix: host-buffer (end-to-end) front end
    solve     cg(): conjugate-gradient solve on the device (SPD matrices), bicgstab(): BiCGSTAB
              and gmres(): restarted GMRES for general square matrices; all optionally
              Jacobi-preconditioned

Importing the package does not need a GPU; calling into it does, and nothing falls back.
"""
from . import _lib  # noqa: F401

__all__ = ["_lib", "spmv", "generate", "matrix", "solve"]
