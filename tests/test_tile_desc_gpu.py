"""The persistent table kernel reads each tile's row ends and row starts from the tile descriptors
(csrc/merge.cu, tile_desc_kernel) instead of Ap.  On the tile edges that the descriptors encode
(tests/test_tile_desc_cpu.py), y must be bit-identical to the plain merge kernel's, which reads Ap;
and the descriptors must follow the partition: reused while it is, rebuilt whenever it is searched
again."""
import contextlib

import numpy as np
import pytest

import reference_model as model
import test_tile_desc_cpu as shapes
from oracle import generators as g

torch = pytest.importorskip("torch")

N_COLS = 4096


@contextlib.contextmanager
def options(**kv):
    from spmv_samples_b200 import spmv
    old = {k: spmv.get_option(k) for k in kv}
    try:
        for k, v in kv.items():
            spmv.set_option(k, v)
        yield
    finally:
        for k, v in old.items():
            spmv.set_option(k, v)


@pytest.fixture(scope="module")
def cuda(built_lib):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    assert int(built_lib.spmvb200_merge_tile_items(32, 32)) == shapes.TILE
    assert int(built_lib.spmvb200_merge_tile_items(64, 32)) == shapes.TILE


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def case(name, off):
    if name == "rmat_s17":      # several tiles per group of the persistent grid
        Ap, Aj, Ax = g.rmat(17, 16, 9, offset_dtype=off)
        return Ap, Aj, Ax, g.gen_x(4, 1 << 17)
    # int32 offsets: the table kernel's own flag path, which the descriptors replace for int64
    Ap = shapes.matrices()[name].astype(off)
    rng = np.random.default_rng(len(name))
    nnz = int(Ap[-1])
    # half of the nonzeros in 32 columns: hot columns, table entries and plain gathers all occur
    Aj = np.where(rng.random(nnz) < 0.5, rng.integers(0, 32, nnz), rng.integers(0, N_COLS, nnz)).astype(np.int32)
    Ax = rng.uniform(-1, 1, nnz).astype(np.float32)
    return Ap, Aj, Ax, g.gen_x(3, N_COLS)


# 64 hot columns: some gathers from the table, some from x_hot, the rest from x
TABLE = dict(hot_x=1, hot_x_table=1, hot_x_max_bytes=64 * 4)


def run(d, n_rows, n_cols, **kw):
    from spmv_samples_b200 import spmv
    y = torch.full((n_rows,), float("nan"), device="cuda")
    spmv.spmv_ex("merge", *d, y, n_cols=n_cols, **kw)
    torch.cuda.synchronize()
    return y


@pytest.mark.gpu
@pytest.mark.parametrize("off", [np.int32, np.int64])
@pytest.mark.parametrize("name", sorted(shapes.matrices()) + ["rmat_s17"])
def test_table_kernel_on_tile_edges_is_bit_identical(cuda, name, off):
    from spmv_samples_b200 import spmv
    Ap, Aj, Ax, x = case(name, off)
    n_rows, n_cols = len(Ap) - 1, len(x)
    d = [dev(a) for a in (Ap, Aj, Ax, x)]
    try:
        spmv.release_cache()
        with options(hot_x=0):
            y0 = run(d, n_rows, n_cols)
        # R-MAT's 64 most frequent columns take too few gathers for a plan: the default x_hot size
        with options(**dict(TABLE, hot_x_max_bytes=32 << 20) if name == "rmat_s17" else TABLE):
            y1 = run(d, n_rows, n_cols)
            assert spmv.hot_x_info(d[1])["table_columns"] > 0
            # peer replicas: only rows with nonzeros are sent to them
            rep = torch.zeros(n_rows + 4, device="cuda")
            y2 = run(d, n_rows, n_cols, y_peers=[rep.data_ptr() + 4 * 4])
    finally:
        spmv.release_cache()
    assert torch.equal(y0, y1), name
    assert torch.equal(y0, y2), name
    nonempty = torch.from_numpy(np.diff(Ap.astype(np.int64)) > 0).cuda()
    assert torch.equal(rep[4:][nonempty], y0[nonempty])
    ref = model.spmv_fp64(Ap, Aj, Ax, x)
    scale = model.abs_scale(Ap, Aj, Ax, x)
    assert np.all(np.abs(y0.cpu().numpy() - ref) <= 1e-5 * scale + 1e-30)


@pytest.mark.gpu
def test_descriptors_follow_the_partition(cuda):
    """Flagged, flagged, Ap changed in place, unflagged, flagged: every call equals a fresh plain call
    on the Ap of the moment.  A flagged call reuses the coordinates and the descriptors; a call that
    searches again also builds the descriptors again (one launch more than the search alone).  The
    descriptors are built for 64-bit offsets and fp32 only (csrc/merge.cu, tile_desc_used)."""
    from spmv_samples_b200 import spmv
    off = np.int64
    Ap, Aj, Ax, x = case("empty_runs", off)
    n_rows = len(Ap) - 1
    d = [dev(a) for a in (Ap, Aj, Ax, x)]
    lens = np.diff(Ap.astype(np.int64))
    np.random.default_rng(5).shuffle(lens)                      # same n_rows, same nnz
    Ap2 = np.zeros_like(Ap)
    np.cumsum(lens, out=Ap2[1:])

    def plain():
        with options(hot_x=0):
            return run(d, n_rows, N_COLS)

    def counted(flag):
        before = spmv.launch_count()
        y = run(d, n_rows, N_COLS, static_pattern=flag)
        return y, spmv.launch_count() - before

    launches, ok = {}, []
    try:
        spmv.release_cache()
        y_ref = plain()
        with options(**TABLE):
            y, launches["first"] = counted(True)
            ok.append(torch.equal(y, y_ref))
            y, launches["reused"] = counted(True)
            ok.append(torch.equal(y, y_ref))
        d[0].copy_(torch.from_numpy(Ap2).cuda())
        y_ref2 = plain()
        with options(**TABLE):
            y, launches["searched"] = counted(False)
            ok.append(torch.equal(y, y_ref2))
            y, launches["reused_again"] = counted(True)
            ok.append(torch.equal(y, y_ref2))
        # the same sequence through the hot-x kernel without the table: no descriptors
        with options(hot_x=1, hot_x_table=0, hot_x_max_bytes=64 * 4):
            counted(True)
            _, launches["hot_reused"] = counted(True)
            d[0].copy_(torch.from_numpy(Ap.astype(off)).cuda())
            y, launches["hot_searched"] = counted(False)
            ok.append(torch.equal(y, plain()))
    finally:
        spmv.release_cache()
    assert all(ok), ok
    assert launches["reused"] == launches["reused_again"]
    assert launches["hot_searched"] == launches["hot_reused"] + 1                 # the search
    assert launches["searched"] == launches["reused"] + 2                         # search + descriptors
    assert launches["first"] > launches["reused"]                                 # plan + descriptors
