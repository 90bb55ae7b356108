"""Inf, NaN and stored zeros through every SpMV / SpMM kernel variant, each row checked exactly
against IEEE semantics.

test_exact_gpu.py proves that every kernel adds the right products, with nonzero integer values.
With finite values, a product that a kernel must mask out (a neighbouring row's nonzero in the same
16-byte load, the slots of a tile before its first or after its last nonzero) is a * 0 or 0 * x,
which is exactly 0, so a kernel that drops the select on the product passes there.  Here the same
integer inputs carry +inf, -inf and NaN where the kernels mask (tile edges, shared vectors, long
rows, the element-wise tail, hot and cold columns of x), and about 1 % of Ax are stored zeros.

For each row the IEEE result does not depend on the summation order, and FMA contraction does not
change it either:
  NaN if a product is NaN (NaN in Ax or x, or a stored 0 times +-inf), or the row has both a +inf
  and a -inf product; else +-inf if it has a product of that sign; else the exact int64 sum.
So the kernels are compared exactly (NaN-aware; the sign of zero and NaN payloads are not checked).
"""
import itertools

import numpy as np
import pytest

from oracle import cpu
from test_exact_gpu import (HOT_COLS, LIGHT_CLAIM, MERGE_PATHS, N_COLS, OFF_VAL, OV_IDS, VECTOR_WIDTHS, _merge_opts, exact_inputs, light_shapes,
                            merge_shapes, merge_tiles, options, pattern, stream_shapes, vector_shapes)

torch = pytest.importorskip("torch")

SPECIALS = (np.inf, -np.inf, np.nan)
# short rows put before the last row of every shape: room for one row of each class, and most rows
# stay finite, so the exact check keeps its weight
TAIL = [1 + i % 8 for i in range(48)]
PER_RULE = 8                # poisoned places per rule (and per tile size for P1)
LONG_ROW = 64               # longer rows are reduced by more than a sub-warp / cross tiles
HOT = np.arange(HOT_COLS) * (N_COLS // HOT_COLS)


# ---------------------------------------------------------------------------------- expectation
def row_classes(Ap, Aj, Ax, x):
    """Per row: (y under IEEE in float64, dict of boolean class arrays)."""
    Ap = np.asarray(Ap, dtype=np.int64)
    n = Ap.size - 1
    a = Ax.astype(np.float64)
    v = x.astype(np.float64)[Aj]
    with np.errstate(invalid="ignore"):
        prod = a * v
    rows = np.repeat(np.arange(n), np.diff(Ap))

    def any_of(mask):
        return np.bincount(rows, mask, n) > 0

    fin = np.isfinite(prod)
    ip = np.where(fin, a, 0).astype(np.int64) * np.where(fin, v, 0).astype(np.int64)
    cs = np.zeros(ip.size + 1, dtype=np.int64)
    np.cumsum(ip, out=cs[1:])
    y = (cs[Ap[1:]] - cs[Ap[:-1]]).astype(np.float64)
    nan_prod = np.isnan(prod)
    zero_inf = nan_prod & (a == 0) & np.isinf(v)
    pinf, ninf = any_of(prod == np.inf), any_of(prod == -np.inf)
    nan = any_of(nan_prod) | (pinf & ninf)
    y[pinf] = np.inf
    y[ninf] = -np.inf
    y[nan] = np.nan
    only_zero_inf = any_of(zero_inf) & ~any_of(nan_prod & ~zero_inf) & ~(pinf & ninf)
    classes = {"finite": ~nan & ~pinf & ~ninf, "+inf": pinf & ~nan, "-inf": ninf & ~nan, "nan": nan,
               "nan_only_from_0*inf": only_zero_inf}
    return y, classes


def ieee_spmv(Ap, Aj, Ax, x):
    return row_classes(Ap, Aj, Ax, x)[0]


def check(got, want, what):
    got = got.cpu().numpy().astype(np.float64) if hasattr(got, "cpu") else np.asarray(got, np.float64)
    if np.array_equal(got, want, equal_nan=True):
        return
    bad = np.nonzero(~((got == want) | (np.isnan(got) & np.isnan(want))))[0]
    raise AssertionError(f"{what}: {bad.size} of {want.size} rows differ, first rows {bad[:5].tolist()}: "
                         f"got {got[bad[:5]].tolist()}, want {want[bad[:5]].tolist()}")


# ---------------------------------------------------------------------------------- placements
def with_tail(lens):
    """TAIL inserted before the last row; the last row grows so that nnz % 8 is unchanged."""
    lens = list(lens)
    out = lens[:-1] + TAIL + lens[-1:]
    out[-1] += (sum(lens) - sum(out)) % 8
    return out


def place_specials(Ap, Aj, Ax, x, tiles, seed, spare_rows, hot=HOT):
    """Ax, x and Aj with special values placed by rule (P1..P6 below); returns (Aj, Ax, x, at) where
    `at` records what was placed where."""
    Ap64 = np.asarray(Ap, dtype=np.int64)
    nnz, n_rows = Aj.size, Ap64.size - 1
    lens = np.diff(Ap64)
    Aj, Ax, x = Aj.copy(), Ax.copy(), x.copy()
    rng = np.random.default_rng(seed)
    cycle = itertools.cycle(SPECIALS)
    at = {"P1": {}, "P2": [], "P3": [], "P4": [], "P5_cols": [], "P6": []}
    poisoned = set()

    def put(k):
        Ax[k] = next(cycle)
        poisoned.add(int(k))

    def some(items):
        items = list(items)
        return items if len(items) <= PER_RULE else [items[i] for i in sorted(rng.choice(len(items), PER_RULE, replace=False))]

    # P2: a nonzero in the aligned 4-element vector of the next row's first nonzero or of the previous
    # row's last one -- what the CSR-vector, light and SpMM vector kernels mask.  First, so that
    # the neighbour rows are still finite when they are picked.
    ne = np.nonzero(lens > 0)[0]
    a, b = ne[:-1], ne[1:]
    last, first = Ap64[a + 1] - 1, Ap64[b]
    same = last // 4 == first // 4
    cand = list(zip(np.concatenate([last[same], first[same]]).tolist(),
                    np.concatenate([b[same], a[same]]).tolist()))
    rows_used = set()
    for i in rng.permutation(len(cand)).tolist():
        k, nb = cand[i]
        r = int(np.searchsorted(Ap64, k, side="right") - 1)
        if len(at["P2"]) >= PER_RULE:
            break
        if r in rows_used or nb in rows_used:
            continue
        rows_used |= {r, nb}
        put(k)
        at["P2"].append((k, nb))
    # P1: the last nonzero before and the first nonzero after a tile boundary
    for T in tiles:
        _, cy = cpu.merge_tile_coords(Ap, T)
        bounds = sorted({int(v) for v in cy[1:-1] if 0 < v < nnz})
        at["P1"][T] = some(bounds)
        for v in at["P1"][T]:
            put(v - 1)
            put(v)
    # P3: the middle of every other long row (the carry fix-up, warp- and CTA-wide rows)
    long_rows = np.nonzero(lens > LONG_ROW)[0][::2]
    for r in some(long_rows.tolist()):
        k = int(Ap64[r] + lens[r] // 2 + rng.integers(-2, 3))
        put(k)
        at["P3"].append(k)
    # P4: the matrix's last nonzero, read element-wise
    if nnz % 8:
        put(nnz - 1)
        at["P4"].append(nnz - 1)
    # P5: three cold columns, each used by a few rows, hold +inf, -inf and NaN
    count = np.bincount(Aj, minlength=x.size)
    cold = np.setdiff1d(np.nonzero((count >= 1) & (count <= 4))[0], hot)
    if cold.size < 3:
        cold = np.setdiff1d(np.arange(x.size), hot)
    cols = rng.choice(cold, 3, replace=False)
    x[cols] = SPECIALS
    at["P5_cols"] = cols.tolist()
    # one spare short row for each class, its first nonzero moved to a special column
    _, cl = row_classes(Ap64, Aj, Ax, x)
    spare = [int(r) for r in spare_rows if cl["finite"][r] and lens[r] > 0]
    pinf, ninf, nanc = (int(c) for c in cols)
    for (col, value), r in zip(((pinf, 1.0), (pinf, -1.0), (nanc, 1.0), (pinf, 0.0), (ninf, 0.0)), spare):
        k = int(Ap64[r])
        Aj[k] = col
        Ax[k] = value * abs(Ax[k]) if value else 0.0
        poisoned.add(k)
    # P6: about 1 % of Ax become +-0.0 (a finite product of 0, or NaN with an infinite x)
    free = np.setdiff1d(np.arange(nnz), np.fromiter(poisoned, dtype=np.int64, count=len(poisoned)))
    z = rng.choice(free, max(1, nnz // 100), replace=False) if free.size else free
    Ax[z] = np.where(rng.random(z.size) < 0.5, -0.0, 0.0)
    at["P6"] = z.tolist()
    return Aj, Ax, x, at


class Case:
    """One case on the device: the exact inputs of test_exact_gpu with special values placed."""

    def __init__(self, name, lens, off, val, seed, tiles):
        self.name = name
        lens = with_tail(lens)
        Ap, Aj = pattern(lens, seed, off=off)
        Ax, x, _, _ = exact_inputs(Ap, Aj, N_COLS, val, seed)
        tail = len(lens) - 1 - len(TAIL) + np.arange(len(TAIL))
        self.Ap = Ap
        self.Aj, self.Ax, self.x, self.at = place_specials(Ap, Aj, Ax, x, tiles, seed, tail)
        self.n_rows = Ap.size - 1
        self.want = ieee_spmv(self.Ap, self.Aj, self.Ax, self.x)
        self._d = None

    @property
    def d(self):
        if self._d is None:
            self._d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (self.Ap, self.Aj, self.Ax, self.x)]
        return self._d

    def y(self, fill=float("nan")):
        return torch.full((self.n_rows,), fill, dtype=self.d[2].dtype, device="cuda")


def cases(shapes, off, val, tiles):
    return [Case(n, lens, off, val, i, tiles) for i, (n, lens) in enumerate(sorted(shapes.items()))]


def all_merge_shapes():
    reg, tma = merge_tiles()
    return {**merge_shapes(reg), **merge_shapes(tma)}


# ---------------------------------------------------------------------------------- CPU check
def test_construction_places_every_class(built_lib):
    """CPU only: every case holds each class (finite, +inf, -inf, NaN, and NaN only from 0 * inf),
    at least half of the non-empty rows stay finite, P1 poisons both sides of a boundary in different
    rows, a P2 poison has a finite neighbour row, and the finite products are exact."""
    reg, tma = merge_tiles()
    families = [(all_merge_shapes(), (reg, tma))]
    families += [({**vector_shapes(), **light_shapes(), **stream_shapes()}, (reg,))]
    families += [(merge_shapes(T), (T,)) for T in (1020, 508)]
    both_sides, p2_finite_nb, total = {}, 0, {"finite": 0, "nonempty": 0}
    for shapes, tiles in families:
        for i, (name, lens) in enumerate(sorted(shapes.items())):
            for val in (np.float32, np.float64):
                c = Case(name, lens, np.int32, val, i, tiles)
                y, cl = row_classes(c.Ap, c.Aj, c.Ax, c.x)
                for k, rows in cl.items():
                    assert rows.any(), (name, val, k)
                nonempty = np.diff(c.Ap.astype(np.int64)) > 0
                total["finite"] += int(cl["finite"][nonempty].sum())
                total["nonempty"] += int(nonempty.sum())
                if nonempty.sum() >= 100:
                    assert cl["finite"][nonempty].mean() >= 0.5, (name, val)
                row_of = np.repeat(np.arange(c.n_rows), np.diff(c.Ap.astype(np.int64)))
                for T, bounds in c.at["P1"].items():
                    for b in bounds:
                        assert not np.isfinite(c.Ax[b - 1]) and not np.isfinite(c.Ax[b])
                        if row_of[b - 1] != row_of[b]:
                            both_sides[T] = both_sides.get(T, 0) + 1
                p2_finite_nb += sum(bool(cl["finite"][nb]) for _, nb in c.at["P2"])
                # exactness of the finite products: every partial sum of finite terms is exact
                fin = np.isfinite(c.Ax)
                xf = np.isfinite(c.x)
                lim = 1 << (24 if val == np.float32 else 53)
                longest = int(np.diff(c.Ap.astype(np.int64)).max())
                assert longest * np.abs(c.Ax[fin]).max() * np.abs(c.x[xf]).max() < lim, name
                assert np.all(c.Ax[fin] == np.round(c.Ax[fin])) and np.all(c.x[xf] == np.round(c.x[xf]))
                assert np.all(np.abs(y[cl["finite"]]) < lim)
                assert set(c.at["P5_cols"]).isdisjoint(HOT.tolist())
    assert total["finite"] >= total["nonempty"] / 2, total
    assert set(both_sides) == {reg, tma, 1020, 508}, both_sides
    assert p2_finite_nb > 0
    # the classifier on a hand-made row set
    Ap = np.array([0, 2, 4, 6, 8, 10, 10], dtype=np.int32)
    Aj = np.arange(10, dtype=np.int32)
    Ax = np.array([1, 2, 1, np.inf, np.inf, np.inf, -1, np.inf, 0, 3], dtype=np.float32)
    x = np.array([3, -1, 1, 1, 1, -1, 1, np.nan, np.inf, 1], dtype=np.float32)
    y, cl = row_classes(Ap, Aj, Ax, x)
    assert np.array_equal(y, [1, np.inf, np.nan, np.nan, np.nan, 0], equal_nan=True)
    assert cl["nan_only_from_0*inf"].tolist() == [False, False, False, False, True, False]
    assert cl["nan"][2] and not cl["+inf"][2] and not cl["-inf"][2]   # +inf and -inf in one row


# ---------------------------------------------------------------------------------- GPU
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


def run(kind, c, x=None, **kw):
    from spmv_samples_b200 import spmv
    y = c.y()
    d = c.d if x is None else c.d[:3] + [x]
    spmv.spmv_ex(kind, *d, y, n_cols=N_COLS, **kw)
    torch.cuda.synchronize()
    return y


def _dev_scalar(v, val):
    return torch.tensor([v], dtype=torch.float32 if val == np.float32 else torch.float64, device="cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [0, 1])
@pytest.mark.parametrize("path", sorted(MERGE_PATHS))
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_merge_special_values(cuda, off, val, path, algo):
    """The plain, hot-x, table and TMA-staged kernels (both tile bodies where both apply), device
    alpha 0.5 and -2 (a negative alpha flips infinities), two peer replicas; on the hot-x and table
    paths also one pass per hot column set to NaN, read from the shared-memory table or x_hot."""
    from spmv_samples_b200 import spmv
    if path in ("table", "staging") and algo == 0:
        pytest.skip("the table and TMA-staged kernels have one tile body (merge_algo does not apply)")
    isz = np.dtype(val).itemsize
    reg, tma = merge_tiles()
    what = f"merge {path} algo {algo}"
    try:
        with options(**_merge_opts(path, algo, isz)):
            for c in cases(all_merge_shapes(), off, val, (reg, tma)):
                spmv.release_cache()
                check(run("merge", c), c.want, f"{what} / {c.name}")
                for a in (0.5, -2.0):
                    alpha = _dev_scalar(a, val)
                    reps = [torch.zeros(c.n_rows + 8, dtype=c.d[2].dtype, device="cuda") for _ in range(2)]
                    peers = [reps[0].data_ptr(), reps[1].data_ptr() + 4 * isz]
                    y = run("merge", c, alpha_dev=alpha, y_peers=peers)
                    check(y, a * c.want, f"{what} alpha {a} + peers / {c.name}")
                    nonempty = np.diff(c.Ap.astype(np.int64)) > 0
                    yh = y.cpu().numpy()
                    for i, r in enumerate(reps):
                        rv = r[4 * i:4 * i + c.n_rows].cpu().numpy()
                        assert np.array_equal(rv[nonempty], yh[nonempty], equal_nan=True), (c.name, "peer", i, a)
                if path in ("hot_x", "table") and "mixed" in c.name:
                    info = spmv.hot_x_info(c.d[1])
                    assert info["hot_columns"] >= HOT_COLS, (c.name, info)
                    if path == "table":   # some hot columns come from the table, the others from x_hot
                        assert 0 < info["table_columns"] < HOT_COLS, (c.name, info)
                    for col in HOT:
                        x = c.x.copy()
                        x[col] = np.nan
                        y = run("merge", c, x=torch.from_numpy(x).cuda())
                        check(y, ieee_spmv(c.Ap, c.Aj, c.Ax, x), f"{what} / {c.name}, x[{col}] = NaN")
    finally:
        spmv.release_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("rps", [1, 4])
@pytest.mark.parametrize("width", VECTOR_WIDTHS)
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_vector_special_values(cuda, off, val, width, rps):
    reg, _ = merge_tiles()
    shapes = {**vector_shapes(), **{k: v for k, v in merge_shapes(reg).items() if "mixed" in k or "mod8" in k}}
    with options(vector_width=width, vector_rows_per_subwarp=rps):
        for c in cases(shapes, off, val, (reg,)):
            check(run("vector", c), c.want, f"vector width {width} rps {rps} / {c.name}")


@pytest.mark.gpu
@pytest.mark.parametrize("width", [0] + list(VECTOR_WIDTHS))
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_light_special_values(cuda, off, val, width):
    reg, _ = merge_tiles()
    cs = cases({**light_shapes(), **vector_shapes()}, off, val, (reg,))
    for rpc in (LIGHT_CLAIM, 0):
        with options(light_width=width, light_rows_per_claim=rpc):
            for c in cs:
                check(run("light", c), c.want, f"light width {width} claim {rpc} / {c.name}")


@pytest.mark.gpu
@pytest.mark.parametrize("ctas", [1, 3])
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_stream_special_values(cuda, off, val, ctas):
    reg, _ = merge_tiles()
    shapes = {**stream_shapes(), **{k: v for k, v in merge_shapes(reg).items() if "mod8" in k}}
    with options(stream_ctas_per_sm=ctas):
        for c in cases(shapes, off, val, (reg,)):
            check(run("stream", c), c.want, f"stream ctas/SM {ctas} / {c.name}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["auto", "cusp", "cusp1", "cusp2", "light_vec", "light_warp", "cub_merge"])
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_auto_and_reference_labels_special_values(cuda, off, val, kind):
    from spmv_samples_b200 import spmv
    reg, tma = merge_tiles()
    shapes = {**all_merge_shapes(), **vector_shapes(), **light_shapes(), **stream_shapes()}
    for c in cases(shapes, off, val, (reg, tma)):
        y = c.y()
        spmv.SpMV(kind, c.n_rows, N_COLS, c.Aj.size, *c.d, y)
        torch.cuda.synchronize()
        check(y, c.want, f"{kind} / {c.name}")


@pytest.mark.gpu
def test_host_buffer_spmv_special_values(cuda):
    """CsrMatrix.spmv: host x in, host y out."""
    from spmv_samples_b200.matrix import CsrMatrix
    reg, _ = merge_tiles()
    c = Case("mixed", merge_shapes(reg)[f"T{reg}_mixed_many_tiles"], np.int64, np.float32, 3, (reg,))
    m = CsrMatrix(c.n_rows, N_COLS, c.Ap, c.Aj, c.Ax)
    try:
        check(m.spmv(c.x), c.want, "CsrMatrix.spmv")
    finally:
        m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("alg", [0, 1, 2])
@pytest.mark.parametrize("val", [np.float32, np.float64])
def test_cusparse_baseline_special_values(cuda, val, alg):
    """The cuSPARSE baseline (32-bit offsets); a mismatch is recorded as an xfail."""
    reg, tma = merge_tiles()
    bad = []
    with options(cusparse_alg=alg):
        for c in cases({**all_merge_shapes(), **vector_shapes()}, np.int32, val, (reg, tma)):
            y = run("cusparse", c).cpu().numpy().astype(np.float64)
            if not np.array_equal(y, c.want, equal_nan=True):
                bad.append(c.name)
    if bad:
        pytest.xfail(f"cuSPARSE (alg {alg}) does not follow IEEE row by row for {bad}")


@pytest.mark.gpu
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_table_kernel_special_values_rmat17(cuda, off, val):
    """The persistent table kernel on R-MAT scale 17 with the table forced: with int64 offsets and
    fp32 values it reads the tile descriptors, the path of the scale-27 power step."""
    from oracle import generators as g
    from spmv_samples_b200 import spmv
    reg, _ = merge_tiles()
    Ap, Aj, _ = g.rmat(17, 16, 9, offset_dtype=off)
    n = Ap.size - 1
    Ax, x, _, _ = exact_inputs(Ap, Aj, n, val, 17)
    lens = np.diff(Ap.astype(np.int64))
    spare = np.nonzero((lens >= 1) & (lens <= 8))[0][::1000]
    Aj, Ax, x, _ = place_specials(Ap, Aj, Ax, x, (reg,), 17, spare, hot=np.zeros(0, dtype=np.int64))
    want = ieee_spmv(Ap, Aj, Ax, x)
    d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (Ap, Aj, Ax, x)]
    try:
        spmv.release_cache()
        with options(hot_x=1, hot_x_table=1, hot_x_max_bytes=32 << 20):
            for flag in (False, True):
                y = torch.full((n,), float("nan"), dtype=d[2].dtype, device="cuda")
                spmv.spmv_ex("merge", *d, y, n_cols=n, static_pattern=flag)
                torch.cuda.synchronize()
                assert spmv.hot_x_info(d[1])["table_columns"] > 0
                check(y, want, f"table kernel, R-MAT 17, static_pattern={flag}")
    finally:
        spmv.release_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 4, 8])
@pytest.mark.parametrize("route", ["auto", "vector", "merge", "columns"])
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_spmm_special_values(cuda, off, val, route, k):
    """Special values in one column j of X reach column j of Y only; those in Ax reach every column
    of their row; Y past k stays untouched."""
    from spmv_samples_b200 import spmv
    route_opts = {"auto": {}, "vector": {"spmm_force_vector": 1}, "merge": {"spmm_force_merge": 1},
                  "columns": {"spmm_by_columns": 1}}[route]
    T = 1020 if k * np.dtype(val).itemsize <= 8 else 508
    shapes = {**merge_shapes(T), "vector_huge_rows": vector_shapes()["vector_huge_rows"]}
    tdt = torch.float32 if val == np.float32 else torch.float64
    with options(**route_opts):
        for i, c in enumerate(cases(shapes, off, val, (T,))):
            j0 = i % k
            xs = [exact_inputs(c.Ap, c.Aj, N_COLS, val, 1000 * i + j)[1] for j in range(k)]
            xs[j0] = c.x
            Xb = torch.full((N_COLS, 16), float("nan"), dtype=tdt, device="cuda")
            Xb[:, :k].copy_(torch.from_numpy(np.stack(xs, axis=1)).cuda())
            Yb = torch.full((c.n_rows, 24), float("nan"), dtype=tdt, device="cuda")
            spmv.spmm(c.d[0], c.d[1], c.d[2], Xb[:, :k], Yb[:, :k])
            torch.cuda.synchronize()
            got = Yb[:, :k].cpu().numpy().astype(np.float64)
            for j in range(k):
                check(got[:, j], ieee_spmv(c.Ap, c.Aj, c.Ax, xs[j]), f"spmm {route} k {k} column {j} / {c.name}")
            assert bool(torch.isnan(Yb[:, k:]).all()), "SpMM wrote past k in a row of Y"


@pytest.mark.gpu
@pytest.mark.parametrize("off,val", OFF_VAL, ids=OV_IDS)
def test_generalised_kernel_special_values(cuda, off, val):
    """y = A x + beta y with beta = -2 and +-inf in y; min-plus / max-plus with +-inf in x (an
    unreached vertex) and finite Ax; or-and with NaN, +-inf and +-0 in Ax and x."""
    from spmv_samples_b200 import spmv
    _, tma = merge_tiles()
    beta = _dev_scalar(-2.0, val)
    for c in cases(merge_shapes(tma), off, val, (tma,)):
        rng = np.random.default_rng(len(c.name))
        y0 = rng.integers(-64, 65, c.n_rows).astype(val)
        y0[rng.choice(c.n_rows, 6, replace=False)] = [np.inf, -np.inf] * 3
        y = torch.from_numpy(y0.copy()).cuda()
        spmv.spmv_ex("merge", *c.d, y, n_cols=N_COLS, beta_dev=beta)
        torch.cuda.synchronize()
        with np.errstate(invalid="ignore"):                # inf - inf: NaN
            want = c.want + -2.0 * y0.astype(np.float64)
        check(y, want, f"A x + beta y / {c.name}")
        # min-plus / max-plus: Ax finite, x holds +inf and -inf, no combine gives NaN
        Ax = np.where(np.isfinite(c.Ax), c.Ax, 1).astype(val)
        x = np.where(np.isfinite(c.x), c.x, np.inf).astype(val)
        x[rng.choice(N_COLS, 200, replace=False)] = np.inf
        x[rng.choice(N_COLS, 50, replace=False)] = -np.inf
        dAx, dx = torch.from_numpy(Ax).cuda(), torch.from_numpy(x).cuda()
        empty = np.diff(c.Ap.astype(np.int64)) == 0
        for sr, ident in (("min_plus", np.inf), ("max_plus", -np.inf)):
            y = c.y()
            spmv.spmv_ex("merge", c.d[0], c.d[1], dAx, dx, y, n_cols=N_COLS, semiring=sr)
            torch.cuda.synchronize()
            got = y.cpu().numpy()
            assert np.array_equal(got, cpu.spmv_semiring(c.Ap, c.Aj, Ax, x, sr)), (sr, c.name)
            assert np.all(got[empty] == ident), (sr, c.name)
            assert np.isinf(got[~empty]).any() and np.isfinite(got).any(), (sr, c.name)
        # or-and: NaN counts as non-zero, +-0 as zero
        Ax = c.Ax.copy()
        x = c.x.copy()
        x[rng.choice(N_COLS, 400, replace=False)] = -0.0
        x[::9] = 0.0
        y = c.y()
        spmv.spmv_ex("merge", c.d[0], c.d[1], c.d[2], torch.from_numpy(x).cuda(), y, n_cols=N_COLS,
                     semiring="or_and")
        torch.cuda.synchronize()
        assert np.array_equal(y.cpu().numpy(), cpu.spmv_semiring(c.Ap, c.Aj, Ax, x, "or_and")), ("or_and", c.name)
