"""Bit-exact plus-times parity for every SpMV / SpMM kernel variant, through integer-valued inputs.

The tolerance suites accept |y - y_ref| <= 1e-5 * sum_j |a_ij x_j|; in a row of 10^5 nonzeros one
product is below that bar, so a dropped or doubled nonzero can pass them.  Here Ax and x are
nonzero integers small enough that every partial sum of every row is an exactly representable
integer (fp32: max_row_len * max|a| * max|x| < 2^24; fp64: < 2^53).  Every summation order then
gives the same exact result, the expected y is computed on the host in int64, and the kernels
must match it bit for bit: a dropped, duplicated or misplaced product changes y.

The matrix shapes are derived from the kernels' own tile sizes, and a CPU test checks that every
edge class they are meant to hit (row ends on tile boundaries, every 16-byte alignment shift at a
tile start, rows spanning 1 / 2 / many tiles, tiles made only of empty rows, ...) is really hit.
"""
import contextlib

import numpy as np
import pytest

from oracle import cpu

torch = pytest.importorskip("torch")

# ---------------------------------------------------------------------------------- constants
# Tile sizes of the merge-path kernels, in path items (rows + nonzeros).  The register-staged tile
# kernels (and the shared-memory table kernel) and the TMA-staged variant are read through
# spmvb200_merge_tile_items; the generalised (semiring / beta) kernel uses the TMA variant's
# kMergeTile = 256 * 8 - 4 (csrc/merge.cu:46), which the ABI reports with "merge_staging" = 1.
# The SpMM tile kernel's ms_tile (csrc/spmm.cu:221) is not exposed: 128 threads x 8 items - 4 when
# k * sizeof(value) <= 8 bytes, 128 x 4 - 4 otherwise.
SPMM_TILES = (1020, 508)
VECTOR_WIDTHS = (1, 2, 4, 8, 16, 32)
K_HUGE_ROW = 16384          # csrc/row_dot.cuh:122, rows the CSR-vector kernel hands to a whole CTA
K_LONG_STEPS = 64           # csrc/row_dot.cuh:91, a row is "long" for T lanes beyond 64 * T
K_LIGHT_HEAVY_NNZ = 16384   # csrc/light.cu:33, a claim with more nonzeros than this is heavy
K_LIGHT_MEGA_ROW = 8192     # csrc/light.cu:34, a row of a heavy claim longer than this goes to a CTA
LIGHT_CLAIM = 256           # "light_rows_per_claim" used on the tier shapes
STREAM_ROWS = 256           # csrc/stream.cu:31, rows per tile of the CSR-stream kernel
STREAM_CAP = 2048           # csrc/stream.cu:34, nonzeros per stage
EXACT_LIMIT = {np.dtype(np.float32): 1 << 24, np.dtype(np.float64): 1 << 53}
X_CAP = 1 << 20             # widest |x| used: a column read from the wrong place changes y
A_CAP = 8
N_COLS = 4096
HOT_COLS = 32               # columns that take about half of the nonzeros (hot-x plan, table)


def merge_tiles():
    """(register tile, TMA / generalised tile) as the library reports them."""
    from spmv_samples_b200 import _lib
    L = _lib.lib()
    # the reported size follows "merge_staging", which a caller may have set: ask for each form
    with options(merge_staging=0):
        reg = int(L.spmvb200_merge_tile_items(32, 32))
        assert int(L.spmvb200_merge_tile_items(64, 32)) == reg
    with options(merge_staging=1):
        tma = int(L.spmvb200_merge_tile_items(32, 32))
    return reg, tma


@contextlib.contextmanager
def options(**kv):
    """Set library options for the duration of a block and restore the values found before."""
    from spmv_samples_b200 import spmv
    old = {k: spmv.get_option(k) for k in kv}
    try:
        for k, v in kv.items():
            spmv.set_option(k, v)
        yield
    finally:
        for k, v in old.items():
            spmv.set_option(k, v)


# ---------------------------------------------------------------------------------- inputs
def exact_inputs(Ap, Aj, n_cols, dtype, seed, spare_bits=0):
    """Nonzero integer Ax and x for the pattern (Ap, Aj), as wide as the exactness bound allows:
    max_row_len * max|a| * max|x| < 2^(mantissa + 1 - spare_bits).  Returns (Ax, x, amax, xmax)."""
    dtype = np.dtype(dtype)
    lens = np.diff(np.asarray(Ap, dtype=np.int64))
    longest = max(int(lens.max()) if lens.size else 0, 1)
    budget = ((EXACT_LIMIT[dtype] >> spare_bits) - 1) // longest    # largest allowed |a| * |x|
    assert budget >= 1, f"a row of {longest} nonzeros cannot be summed exactly in {dtype}"
    amax = max(1, min(A_CAP, budget // 8))
    xmax = max(1, min(X_CAP, budget // amax))
    rng = np.random.default_rng(seed)

    def nonzero_ints(n, m):
        v = rng.integers(1, m + 1, n)
        return np.where(rng.random(n) < 0.5, -v, v).astype(dtype)

    return nonzero_ints(Aj.size, amax), nonzero_ints(n_cols, xmax), amax, xmax


def exact_reference(Ap, Aj, Ax, x):
    """y = A x in int64, no floating point: the row sums of exact integer products."""
    prod = Ax.astype(np.int64) * x.astype(np.int64)[Aj]
    cs = np.zeros(prod.size + 1, dtype=np.int64)
    np.cumsum(prod, out=cs[1:])
    Ap = np.asarray(Ap, dtype=np.int64)
    return cs[Ap[1:]] - cs[Ap[:-1]]


def pattern(lens, seed, n_cols=N_COLS, off=np.int32):
    """CSR pattern with the given row lengths.  Half the nonzeros fall on HOT_COLS columns (so a
    hot-x plan and its shared-memory table have something to hold), the rest anywhere."""
    lens = np.asarray(lens, dtype=np.int64)
    Ap = np.zeros(lens.size + 1, dtype=np.int64)
    np.cumsum(lens, out=Ap[1:])
    rng = np.random.default_rng(seed)
    nnz = int(Ap[-1])
    Aj = rng.integers(0, n_cols, nnz)
    hot = rng.random(nnz) < 0.5
    Aj[hot] = rng.integers(0, HOT_COLS, int(hot.sum())) * (n_cols // HOT_COLS)
    return Ap.astype(off), Aj.astype(np.int32)


def lens_from_row_ends(ends):
    """Row lengths such that row r's end is path item ends[r] (row r ends at Ap[r+1] + r)."""
    ends = np.asarray(ends, dtype=np.int64)
    prev = np.concatenate([[-1], ends[:-1]])
    lens = ends - prev - 1
    assert np.all(lens >= 0)
    return lens.tolist()


# ---------------------------------------------------------------------------------- shapes
def merge_shapes(T):
    """Row-length lists at the edges of a merge-path tile of T path items."""
    s = {}
    for k in (-1, 0, 1):
        # row ends on the first three tile boundaries, each shifted by k
        s[f"T{T}_row_end_at_T{k:+d}"] = lens_from_row_ends([T + k, 2 * T + k, 3 * T + k, 3 * T + k + 37])
    # a row inside one tile, one across one boundary, one across many (the carry fixup runs)
    s[f"T{T}_rows_span_1_2_many"] = [T // 2, T, 5 * T + 3, 1]
    # a whole tile of empty rows (R = T, Z = 0: the 16-bit markers and s_y indexing of the marker
    # form at their largest) in a run of empty rows that crosses two tile boundaries, between
    # non-empty rows
    s[f"T{T}_empty_rows_fill_tiles"] = [3, T - 10] + [0] * (2 * T + 5) + [2 * T + 1, 0, 0, 5]
    # nnz % 8 = 0..7 with the last row long: the element-wise tail of the last vectors
    for r in range(8):
        head = [5, 0, 17, 1]
        last = 3 * T + 1
        last += (r - (sum(head) + last)) % 8
        s[f"T{T}_nnz_mod8_{r}_last_long"] = head + [last]
    # many short rows and some long ones: every alignment shift sy & 3 at many tile starts
    rng = np.random.default_rng(T)
    lens = rng.integers(0, 24, 3 * T)
    lens[rng.random(lens.size) < 0.1] = 0
    lens[[7, T, 2 * T + 1]] = [T + 3, 2 * T - 1, 4 * T + 2]
    s[f"T{T}_mixed_many_tiles"] = lens.tolist()
    return s


def vector_shapes():
    lens = [0, 1, 2, 3]
    for t in VECTOR_WIDTHS:
        for base in (4 * t, K_LONG_STEPS * t):
            lens += [base - 1, 0, base, 3, base + 1]
    return {
        "vector_width_edges": lens,
        "vector_huge_rows": [5, K_HUGE_ROW - 1, 0, K_HUGE_ROW, 1, K_HUGE_ROW + 1, 7],
        # more huge rows in one CTA than its queue holds (csrc/row_dot.cuh:123): the rest stay on
        # the warp-level path
        "vector_huge_queue_overflow": [K_HUGE_ROW + 1 + (i % 5) for i in range(11)],
    }


def light_shapes():
    C = LIGHT_CLAIM
    at_limit = [K_LIGHT_HEAVY_NNZ // C] * C                      # exactly kLightHeavyNnz: light
    over = at_limit[:-1] + [K_LIGHT_HEAVY_NNZ // C + 1]         # one more: heavy
    mega = [K_LIGHT_MEGA_ROW - 1, K_LIGHT_MEGA_ROW, K_LIGHT_MEGA_ROW + 1] + [3] * (C - 3)
    short = [4] * C
    return {
        "light_heavy_claim_edges": at_limit + over + short + mega + short + over + [9] * 17,
        "light_mega_rows_last_claim": short * 3 + [0] * 100 + mega[:3] + [2] * 20,
    }


def stream_shapes():
    R, S = STREAM_ROWS, STREAM_CAP
    per = S // R

    def tile(total):     # R rows holding `total` nonzeros
        lens = [per] * R
        lens[-1] += total - per * R
        return lens
    return {
        "stream_stage_edges": tile(S - 1) + tile(S) + tile(S + 1) + tile(2 * S) + tile(2 * S + 1) + [3],
        "stream_rows_edges": [1] * (R - 1) + [S + 1] + [2] * R + [0] * (R + 1) + [S - 1, S, S + 1],
    }


def all_merge_shapes():
    reg, tma = merge_tiles()
    return {**merge_shapes(reg), **merge_shapes(tma)}


# ---------------------------------------------------------------------------------- CPU checks
def _row_end_items(Ap):
    Ap = np.asarray(Ap, dtype=np.int64)
    return Ap[1:] + np.arange(Ap.size - 1, dtype=np.int64)


def tile_edge_classes(Ap, T):
    """Which edge classes of a merge-path tile of T items the pattern hits."""
    Ap = np.asarray(Ap, dtype=np.int64)
    n_rows, nnz = Ap.size - 1, int(Ap[-1])
    cx, cy = cpu.merge_tile_coords(Ap, T)
    tiles = cx.size - 1
    got = set()
    ends = _row_end_items(Ap)
    for t in range(1, tiles):
        for k in (-1, 0, 1):
            if np.any(ends == t * T + k):
                got.add(f"row_end_at_T{k:+d}")
    for t in range(tiles):
        d1 = min((t + 1) * T, n_rows + nnz)
        R = int(cx[t + 1] - cx[t])
        Z = int((d1 - cx[t + 1]) - cy[t])
        if Z > 0:
            got.add(f"shift_{int(cy[t]) & 3}")
        if Z == 0 and R == T:
            got.add("tile_of_empty_rows")
    lens = np.diff(Ap)
    first_item = Ap[:-1] + np.arange(n_rows)           # path item of the row's first nonzero
    for r in np.nonzero(lens > 0)[0]:
        span = int((first_item[r] + lens[r] - 1) // T - first_item[r] // T) + 1
        got.add("row_spans_1_tile" if span == 1 else "row_spans_2_tiles" if span == 2 else "row_spans_many_tiles")
    empty = lens == 0
    for t in range(1, tiles):
        b = t * T
        r = int(np.searchsorted(ends, b))               # first row ending at or after b
        if 0 < r < n_rows and empty[r - 1] and empty[r]:
            got.add("empty_run_crosses_tile")
    if n_rows and lens[-1] >= 64:
        got.add(f"nnz_mod8_{nnz % 8}_last_long")
    return got


TILE_CLASSES = ({f"row_end_at_T{k:+d}" for k in (-1, 0, 1)} | {f"shift_{s}" for s in range(4)}
                | {"tile_of_empty_rows", "row_spans_1_tile", "row_spans_2_tiles", "row_spans_many_tiles",
                   "empty_run_crosses_tile"} | {f"nnz_mod8_{r}_last_long" for r in range(8)})


def check_exact_bound(Ap, Aj, Ax, x):
    """Every partial sum of every row is an exactly representable integer, no product is 0."""
    limit = EXACT_LIMIT[np.dtype(Ax.dtype)]
    lens = np.diff(np.asarray(Ap, dtype=np.int64))
    assert np.all(Ax == np.round(Ax)) and np.all(x == np.round(x))
    assert np.all(Ax != 0) and np.all(x != 0)
    longest = int(lens.max()) if lens.size else 0
    assert longest * int(np.abs(Ax).max(initial=0)) * int(np.abs(x).max()) < limit


def test_shapes_hit_every_tile_edge_and_inputs_are_exact(built_lib):
    """CPU only: the shape lists hit every edge class at the kernels' current tile sizes (read from
    the library), and every generated case satisfies the exactness bound."""
    reg, tma = merge_tiles()
    assert reg % 4 == 0 and tma % 4 == 0 and reg != tma
    for T, shapes in ((reg, merge_shapes(reg)), (tma, merge_shapes(tma)),
                      *((T, merge_shapes(T)) for T in SPMM_TILES)):
        seen = set()
        for name, lens in shapes.items():
            Ap, _ = pattern(lens, 1)
            seen |= tile_edge_classes(Ap, T)
        assert TILE_CLASSES <= seen, (T, sorted(TILE_CLASSES - seen))
    # beyond the merge path
    v = {int(n) for lens in vector_shapes().values() for n in lens}
    for t in VECTOR_WIDTHS:
        for base in (4 * t, K_LONG_STEPS * t):
            assert {base - 1, base, base + 1} <= v, (t, base)
    assert {K_HUGE_ROW - 1, K_HUGE_ROW, K_HUGE_ROW + 1} <= v
    claims, rows = set(), set()
    for lens in light_shapes().values():
        lens = np.asarray(lens)
        for c in range(0, lens.size, LIGHT_CLAIM):
            blk = lens[c:c + LIGHT_CLAIM]
            claims.add(int(blk.sum()))
            if blk.sum() > K_LIGHT_HEAVY_NNZ:
                rows |= {int(n) for n in blk}
    assert {K_LIGHT_HEAVY_NNZ, K_LIGHT_HEAVY_NNZ + 1} <= claims
    assert {K_LIGHT_MEGA_ROW - 1, K_LIGHT_MEGA_ROW, K_LIGHT_MEGA_ROW + 1} <= rows
    tiles = set()
    for lens in stream_shapes().values():
        lens = np.asarray(lens)
        tiles |= {int(lens[c:c + STREAM_ROWS].sum()) for c in range(0, lens.size, STREAM_ROWS)}
        assert lens.size % STREAM_ROWS != 0                     # a partial last tile
    assert {STREAM_CAP - 1, STREAM_CAP, STREAM_CAP + 1, 2 * STREAM_CAP, 2 * STREAM_CAP + 1} <= tiles
    # the exactness bound and nonzero products, for every case at every type
    every = {**merge_shapes(reg), **merge_shapes(tma), **vector_shapes(), **light_shapes(), **stream_shapes()}
    for T in SPMM_TILES:
        every.update(merge_shapes(T))
    for i, (name, lens) in enumerate(sorted(every.items())):
        Ap, Aj = pattern(lens, i)
        for dt in (np.float32, np.float64):
            Ax, x, amax, xmax = exact_inputs(Ap, Aj, N_COLS, dt, i)
            check_exact_bound(Ap, Aj, Ax, x)
            if dt == np.float64:
                assert xmax == X_CAP, name
            assert np.all(np.abs(exact_reference(Ap, Aj, Ax, x)) < EXACT_LIMIT[np.dtype(dt)])
    # the reference is the plain row sum
    Ap, Aj = pattern([3, 0, 5], 0, n_cols=8)
    Ax = np.array([1, -2, 3, 4, 5, -6, 7, 8], dtype=np.float32)
    x = np.arange(1, 9, dtype=np.float32)
    assert exact_reference(Ap, Aj, Ax, x).tolist() == [
        sum(int(Ax[k]) * int(x[Aj[k]]) for k in range(0, 3)), 0,
        sum(int(Ax[k]) * int(x[Aj[k]]) for k in range(3, 8))]


def test_options_context_restores_what_it_found(built_lib):
    from spmv_samples_b200 import spmv
    before = {k: spmv.get_option(k) for k in ("stream_ctas_per_sm", "hot_x_max_bytes", "merge_algo")}
    assert before["stream_ctas_per_sm"] == 3 and before["hot_x_max_bytes"] == 32 << 20
    with pytest.raises(RuntimeError):
        with options(stream_ctas_per_sm=1, hot_x_max_bytes=64, merge_algo=0):
            assert spmv.get_option("stream_ctas_per_sm") == 1
            raise RuntimeError("leave the block early")
    assert {k: spmv.get_option(k) for k in before} == before


# ---------------------------------------------------------------------------------- GPU helpers
OFF_VAL = [(np.int32, np.float32), (np.int32, np.float64), (np.int64, np.float32), (np.int64, np.float64)]
OV_IDS = ["o32f32", "o32f64", "o64f32", "o64f64"]


@pytest.fixture(scope="module")
def cuda(built_lib):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from spmv_samples_b200 import spmv
    names = ("merge_algo", "merge_staging", "merge_carveout", "hot_x", "hot_x_max_bytes", "hot_x_table",
             "hot_x_table_bytes", "vector_width", "vector_rows_per_subwarp", "light_width",
             "light_rows_per_claim", "stream_ctas_per_sm", "cusparse_alg", "side_stream",
             "assume_static_pattern", "spmm_force_merge", "spmm_force_vector", "spmm_by_columns")
    before = {k: spmv.get_option(k) for k in names}
    yield
    torch.cuda.synchronize()
    spmv.release_cache()
    assert {k: spmv.get_option(k) for k in names} == before, "an option was not restored"


class Case:
    """One exact test case on the device: pattern, integer values, int64 expectation."""

    def __init__(self, name, lens, off, val, seed, spare_bits=0):
        self.name = name
        self.Ap, self.Aj = pattern(lens, seed, off=off)
        self.Ax, self.x, _, _ = exact_inputs(self.Ap, self.Aj, N_COLS, val, seed, spare_bits)
        self.y_ref = exact_reference(self.Ap, self.Aj, self.Ax, self.x)
        self.n_rows = self.Ap.size - 1
        self.d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (self.Ap, self.Aj, self.Ax, self.x)]

    def y(self, fill=float("nan")):
        return torch.full((self.n_rows,), fill, dtype=self.d[2].dtype, device="cuda")

    def check(self, y, what, scale=1.0, y0=None):
        """y == scale * (A x) [+ beta-term y0], compared exactly (all values are exact in fp64)."""
        got = y.cpu().numpy().astype(np.float64)
        want = self.y_ref.astype(np.float64) * scale
        if y0 is not None:
            want = want + y0
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, (f"{what} / {self.name}: {bad.size} of {self.n_rows} rows differ, first rows "
                               f"{bad[:5].tolist()}: got {got[bad[:5]].tolist()}, want {want[bad[:5]].tolist()}")


def cases(shapes, off, val, spare_bits=0):
    return [Case(n, lens, off, val, i, spare_bits) for i, (n, lens) in enumerate(sorted(shapes.items()))]


def run(kind, c, **kw):
    from spmv_samples_b200 import spmv
    y = c.y()
    if kw:
        spmv.spmv_ex(kind, *c.d, y, n_cols=N_COLS, **kw)
    else:
        spmv.SpMV(kind, c.n_rows, N_COLS, c.Aj.size, *c.d, y)
    torch.cuda.synchronize()
    return y


# ---------------------------------------------------------------------------------- merge path
MERGE_PATHS = {
    "plain": {"hot_x": 0},
    "hot_x": {"hot_x": 1, "hot_x_table": 0},
    "table": {"hot_x": 1, "hot_x_table": 1},
    "staging": {"merge_staging": 1, "hot_x": 0},
}


def _merge_opts(path, algo, isz):
    o = dict(MERGE_PATHS[path], merge_algo=algo)
    if path in ("hot_x", "table"):
        o["hot_x_max_bytes"] = 64 * isz                         # 64 hot columns in x_hot
    if path == "table":
        # 8 tiles in flight (scan values, flags, warp totals) + 16 table entries: ranks 0..15 come
        # from shared memory, 16..63 from x_hot, the other columns from x
        o["hot_x_table_bytes"] = 8 * (1024 * isz + 1024 + 4 * 2 * isz) + 16 * isz
    return o


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [0, 1])
@pytest.mark.parametrize("path", sorted(MERGE_PATHS))
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_merge_exact(cuda, off, val, path, algo):
    """Every tile body (markers / flags, with and without the register cap), each with and without
    peer replicas and a device alpha, through the plain, hot-x, table and TMA-staged kernels."""
    from spmv_samples_b200 import spmv
    if path in ("table", "staging") and algo == 0:
        pytest.skip("the table and TMA-staged kernels have one tile body (merge_algo does not apply)")
    isz = np.dtype(val).itemsize
    alpha = torch.tensor([0.5], dtype=torch.float32 if val == np.float32 else torch.float64, device="cuda")
    try:
        with options(**_merge_opts(path, algo, isz)):
            for c in cases(all_merge_shapes(), off, val):
                spmv.release_cache()
                c.check(run("merge", c), f"merge {path} algo {algo}")
                if path in ("hot_x", "table"):
                    info = spmv.hot_x_info(c.d[1])
                    assert info["hot_columns"] > 0, c.name
                    assert (info["table_columns"] > 0) == (path == "table"), (c.name, info)
                # peer replicas (at an offset, as a peer's slice is) and alpha
                reps = [torch.zeros(c.n_rows + 8, dtype=c.d[2].dtype, device="cuda") for _ in range(2)]
                peers = [reps[0].data_ptr(), reps[1].data_ptr() + 4 * isz]
                y = c.y()
                spmv.spmv_ex("merge", *c.d, y, n_cols=N_COLS, alpha_dev=alpha, y_peers=peers)
                torch.cuda.synchronize()
                c.check(y, f"merge {path} algo {algo} alpha + peers", scale=0.5)
                nonempty = np.diff(c.Ap.astype(np.int64)) > 0
                yh = y.cpu().numpy()
                for i, r in enumerate(reps):
                    rv = r[4 * i:4 * i + c.n_rows].cpu().numpy()
                    assert np.array_equal(rv[nonempty], yh[nonempty]), (c.name, "peer", i)
                y = c.y()
                spmv.spmv_ex("merge", *c.d, y, n_cols=N_COLS, alpha_dev=alpha)
                torch.cuda.synchronize()
                c.check(y, f"merge {path} algo {algo} alpha", scale=0.5)
    finally:
        spmv.release_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_merge_call_sequence_options_exact(cuda, off, val):
    """Options that change how a call is sequenced, not what it computes: the side stream for the
    partition and x_hot refill, vouching for the pattern (option and flag), the carveout."""
    from spmv_samples_b200 import spmv
    shapes = all_merge_shapes()
    cs = cases(shapes, off, val)
    try:
        for carve in (-1, 28, 100):
            with options(merge_carveout=carve):
                for c in cs:
                    c.check(run("merge", c), f"merge carveout {carve}")
        with options(side_stream=1, assume_static_pattern=1, hot_x=1, hot_x_max_bytes=64 * np.dtype(val).itemsize):
            for c in cs:
                spmv.release_cache()
                for rep in range(3):
                    c.check(run("merge", c), f"side stream + assumed static pattern, call {rep}")
        with options(side_stream=1):
            for c in cs:
                for rep in range(2):
                    c.check(run("merge", c, static_pattern=rep > 0), f"side stream, flag {rep > 0}")
    finally:
        spmv.release_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("table", [0, 1])
@pytest.mark.parametrize("off", [np.int32, np.int64])
def test_static_pattern_flag_exact_across_a_changed_pattern(cuda, off, table):
    """The sequence of test_static_pattern_flag_reuses_and_never_goes_stale, compared exactly:
    unflagged, flagged twice, then a new pattern in the same buffers (one unflagged call), then
    flagged again."""
    from spmv_samples_b200 import spmv
    reg, _ = merge_tiles()
    c = Case("static", merge_shapes(reg)[f"T{reg}_mixed_many_tiles"], off, np.float32, 7)
    try:
        with options(hot_x=1 if table else 0, hot_x_table=table, hot_x_max_bytes=256):
            for flag in (False, True, True):
                c.check(run("merge", c, static_pattern=flag), f"static_pattern={flag}")
            lens = np.diff(c.Ap.astype(np.int64))
            np.random.default_rng(3).shuffle(lens)              # same n_rows, same nnz
            Ap2 = np.zeros_like(c.Ap)
            np.cumsum(lens, out=Ap2[1:])
            c.Ap = Ap2
            c.d[0].copy_(torch.from_numpy(Ap2).cuda())
            c.y_ref = exact_reference(c.Ap, c.Aj, c.Ax, c.x)
            c.check(run("merge", c, static_pattern=False), "new pattern, unflagged")
            for _ in range(2):
                c.check(run("merge", c, static_pattern=True), "new pattern, flagged")
    finally:
        spmv.release_cache()


# ---------------------------------------------------------------------------------- other kinds
@pytest.mark.gpu
@pytest.mark.parametrize("rps", [1, 4])
@pytest.mark.parametrize("width", VECTOR_WIDTHS)
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_vector_exact(cuda, off, val, width, rps):
    from spmv_samples_b200 import spmv
    shapes = {**vector_shapes(), **{k: v for k, v in all_merge_shapes().items() if "mixed" in k or "mod8" in k}}
    alpha = torch.tensor([0.5], dtype=torch.float32 if val == np.float32 else torch.float64, device="cuda")
    with options(vector_width=width, vector_rows_per_subwarp=rps):
        for c in cases(shapes, off, val):
            c.check(run("vector", c), f"vector width {width} rps {rps}")
            y = c.y()
            spmv.spmv_ex("vector", *c.d, y, n_cols=N_COLS, alpha_dev=alpha)
            torch.cuda.synchronize()
            c.check(y, f"vector width {width} rps {rps} alpha", scale=0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("width", [0] + list(VECTOR_WIDTHS))
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_light_exact(cuda, off, val, width):
    shapes = {**light_shapes(), **vector_shapes()}
    for rpc in (LIGHT_CLAIM, 0):
        with options(light_width=width, light_rows_per_claim=rpc):
            for c in cases(shapes, off, val):
                c.check(run("light", c), f"light width {width} claim {rpc}")


@pytest.mark.gpu
@pytest.mark.parametrize("ctas", [1, 3])
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_stream_exact(cuda, off, val, ctas):
    shapes = {**stream_shapes(), **{k: v for k, v in all_merge_shapes().items() if "mod8" in k}}
    with options(stream_ctas_per_sm=ctas):
        for c in cases(shapes, off, val):
            c.check(run("stream", c), f"stream ctas/SM {ctas}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["auto", "cusp", "cusp1", "cusp2", "light_vec", "light_warp", "cub_merge"])
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_auto_and_reference_labels_exact(cuda, off, val, kind):
    shapes = {**all_merge_shapes(), **vector_shapes(), **light_shapes(), **stream_shapes()}
    for c in cases(shapes, off, val):
        c.check(run(kind, c), kind)


@pytest.mark.gpu
@pytest.mark.parametrize("alg", [0, 1, 2])
@pytest.mark.parametrize("val", [np.float32, np.float64])
def test_cusparse_baseline_exact(cuda, val, alg):
    """The cuSPARSE baseline on the same integer inputs (32-bit offsets: it does not take 64-bit
    offsets with 32-bit indices).  A mismatch is recorded, not hidden behind a looser bar."""
    shapes = {**all_merge_shapes(), **vector_shapes()}
    bad = []
    with options(cusparse_alg=alg):
        for c in cases(shapes, np.int32, val):
            if c.Aj.size > c.n_rows * N_COLS:
                continue
            y = run("cusparse", c).cpu().numpy().astype(np.float64)
            if not np.array_equal(y, c.y_ref.astype(np.float64)):
                bad.append(c.name)
    if bad:
        pytest.xfail(f"cuSPARSE (alg {alg}) is not bit-exact on integer inputs for {bad}")


# ---------------------------------------------------------------------------------- SpMM
@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 4, 8])
@pytest.mark.parametrize("route", ["auto", "vector", "merge", "columns"])
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_spmm_exact(cuda, off, val, route, k):
    """Y = alpha A X with leading dimensions larger than k, each column exact."""
    from spmv_samples_b200 import spmv
    route_opts = {"auto": {}, "vector": {"spmm_force_vector": 1}, "merge": {"spmm_force_merge": 1},
                  "columns": {"spmm_by_columns": 1}}[route]
    T = 1020 if k * np.dtype(val).itemsize <= 8 else 508
    shapes = {**merge_shapes(T), "vector_huge_rows": vector_shapes()["vector_huge_rows"]}
    tdt = torch.float32 if val == np.float32 else torch.float64
    with options(**route_opts):
        for i, c in enumerate(cases(shapes, off, val)):
            xs = [c.x] + [exact_inputs(c.Ap, c.Aj, N_COLS, val, 1000 * i + j)[1] for j in range(1, k)]
            for alpha in (None, 0.5):
                # leading dimensions 16 and 24 (> k, rows 16-byte aligned as the kernel requires)
                Xb = torch.full((N_COLS, 16), float("nan"), dtype=tdt, device="cuda")
                X = Xb[:, :k]
                X.copy_(torch.from_numpy(np.stack(xs, axis=1)).cuda())
                Yb = torch.full((c.n_rows, 24), float("nan"), dtype=tdt, device="cuda")
                Y = Yb[:, :k]
                a = torch.tensor([alpha], dtype=tdt, device="cuda") if alpha else None
                spmv.spmm(c.d[0], c.d[1], c.d[2], X, Y, alpha_dev=a)
                torch.cuda.synchronize()
                got = Y.cpu().numpy().astype(np.float64)
                for j in range(k):
                    want = exact_reference(c.Ap, c.Aj, c.Ax, xs[j]).astype(np.float64) * (alpha or 1.0)
                    bad = np.nonzero(got[:, j] != want)[0]
                    assert bad.size == 0, (route, k, c.name, j, alpha, bad[:5].tolist())
                assert bool(torch.isnan(Yb[:, k:]).all()), "SpMM wrote past k in a row of Y"


# ---------------------------------------------------------------------------------- generalised kernel
@pytest.mark.gpu
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_generalised_kernel_exact_on_its_tile_edges(cuda, off, val):
    """y = alpha A x + beta y through the generalised merge kernel (alpha, beta powers of two), and
    the min-plus / max-plus / or-and semirings, on the shapes of its 2044-item tile."""
    from spmv_samples_b200 import spmv
    _, tma = merge_tiles()
    tdt = torch.float32 if val == np.float32 else torch.float64
    alpha = torch.tensor([0.5], dtype=tdt, device="cuda")
    beta = torch.tensor([-2.0], dtype=tdt, device="cuda")
    for c in cases(merge_shapes(tma), off, val, spare_bits=2):
        y0 = np.random.default_rng(5).integers(-64, 65, c.n_rows).astype(val)
        y = torch.from_numpy(y0.copy()).cuda()
        spmv.spmv_ex("merge", *c.d, y, n_cols=N_COLS, alpha_dev=alpha, beta_dev=beta)
        torch.cuda.synchronize()
        c.check(y, "alpha A x + beta y", scale=0.5, y0=-2.0 * y0.astype(np.float64))
        y = torch.from_numpy(y0.copy()).cuda()
        spmv.spmv_ex("merge", *c.d, y, n_cols=N_COLS, beta_dev=beta)
        torch.cuda.synchronize()
        c.check(y, "A x + beta y", y0=-2.0 * y0.astype(np.float64))
        x = c.x.copy()
        x[::7] = 0                                          # or-and sees zeros
        dx = torch.from_numpy(x).cuda()
        for sr in ("min_plus", "max_plus", "or_and"):
            y = c.y()
            spmv.spmv_ex("merge", c.d[0], c.d[1], c.d[2], dx, y, n_cols=N_COLS, semiring=sr)
            torch.cuda.synchronize()
            want = cpu.spmv_semiring(c.Ap, c.Aj, c.Ax, x, sr)
            assert np.array_equal(y.cpu().numpy(), want), (sr, c.name)


# ---------------------------------------------------------------------------------- past 2^31 nonzeros
@pytest.mark.gpu
def test_full_size_rmat27_every_row_exact(cuda):
    """R-MAT scale 27 (c5: 2^31 nonzeros, int64 offsets) with integer values: every row of merge,
    vector, light and auto, and of merge on the second call with the static-pattern flag (hot-x plan
    + shared-memory table, the benchmark's path), against an int64 y built on the device."""
    import time
    from spmv_samples_b200 import generate as gen, spmv
    free, _ = torch.cuda.mem_get_info()
    if free < 90e9:
        pytest.skip("c5 needs ~80 GB of device memory while it is being built")
    t0 = time.perf_counter()
    m = gen.make_config("c5")
    n, nnz = m.n_rows, m.nnz
    Ap = m.Ap
    longest = int((Ap[1:] - Ap[:-1]).max())
    limit = EXACT_LIMIT[np.dtype(np.float32)]
    budget = (limit - 1) // longest
    amax = max(1, min(A_CAP, budget // 8))
    xmax = max(1, min(X_CAP, budget // amax))
    assert longest * amax * xmax < limit
    g = torch.Generator(device="cuda").manual_seed(27)

    def nonzero_ints(out, mx):
        v = torch.randint(1, mx + 1, out.shape, generator=g, device="cuda", dtype=torch.int32)
        sgn = torch.randint(0, 2, out.shape, generator=g, device="cuda", dtype=torch.int32) * 2 - 1
        out.copy_(v * sgn)

    chunk = 1 << 26
    for s in range(0, nnz, chunk):
        nonzero_ints(m.Ax[s:s + chunk], amax)
    x = torch.empty(m.n_cols, dtype=torch.float32, device="cuda")
    nonzero_ints(x, xmax)
    # int64 y: row of each nonzero by a search in Ap, products summed with index_add_
    y_ref = torch.zeros(n, dtype=torch.int64, device="cuda")
    xi = x.to(torch.int64)
    for s in range(0, nnz, chunk):
        e = min(s + chunk, nnz)
        pos = torch.arange(s, e, device="cuda", dtype=torch.int64)
        rows = torch.searchsorted(Ap, pos, right=True) - 1
        del pos
        prod = m.Ax[s:e].to(torch.int64) * xi[m.Aj[s:e].long()]
        y_ref.index_add_(0, rows, prod)
        del rows, prod
    del xi
    assert int(y_ref.abs().max()) < limit
    want = y_ref.to(torch.float32)                          # exact: |y| < 2^24
    del y_ref
    # rows with nonzeros on both sides of offset 2^31 and 2^32 (what exists at this size)
    straddle = []
    for B in (1 << 31, 1 << 32):
        if B < nnz:
            r = int(torch.searchsorted(Ap, torch.tensor([B], dtype=torch.int64, device="cuda"), right=True)) - 1
            if int(Ap[r]) < B:
                straddle.append(r)
    last_row = int(torch.searchsorted(Ap, torch.tensor([nnz - 1], dtype=torch.int64, device="cuda"), right=True)) - 1
    straddle.append(last_row)                               # holds nonzero 2^31 - 1 when nnz = 2^31
    assert nnz >= (1 << 31) and Ap.dtype == torch.int64
    rows = torch.tensor(sorted(set(straddle)), device="cuda")

    def check(y, what):
        torch.cuda.synchronize()
        assert bool(torch.equal(y[rows], want[rows])), (what, "rows at the 2^31 / 2^32 offsets")
        diff = int((y != want).sum())
        assert diff == 0, (what, f"{diff} of {n} rows differ")

    y = torch.empty(n, dtype=torch.float32, device="cuda")
    for kind in ("merge", "vector", "light", "auto"):
        y.fill_(float("nan"))
        spmv.SpMV(kind, n, m.n_cols, nnz, Ap, m.Aj, m.Ax, x, y)
        check(y, kind)
    spmv.release_cache()
    try:
        for call in range(2):
            y.fill_(float("nan"))
            spmv.spmv_ex("merge", Ap, m.Aj, m.Ax, x, y, n_cols=m.n_cols, static_pattern=True)
            torch.cuda.synchronize()
            if call == 1:
                info = spmv.hot_x_info(m.Aj)
                assert info["hot_columns"] > 0 and info["table_columns"] > 0, info
                check(y, "merge, static pattern, second call")
    finally:
        spmv.release_cache()
    print(f"c5 exact: {n} rows, {nnz} nonzeros, longest row {longest}, |a| <= {amax}, |x| <= {xmax}, "
          f"rows at the 2^31 / 2^32 offsets {sorted(set(straddle))}, {time.perf_counter() - t0:.1f} s")
    del y, want, x, m, Ap
    torch.cuda.empty_cache()
