"""Gather-bound kernel paths on wide matrices, against an extended-precision row sum.

The engine picks kernels from statistics it measures at conversion: the band max |col - row| (primitives.cu
gathers_need_l2) selects the load-fed entry streams of CRS and COO and keeps SS off its short-row kernels; the size of x
and the spread of the rows over column blocks (ss.cu make_col_block_engine) select the column-block engines of ELL, JDS
and SS; CSS with several blocks switches to sliced-ELL blocks or the tile-stream per block.  Small test matrices never
meet these conditions, so this file builds matrices whose x is 50 MB (band above the limit, no column blocks) and
128 MB (three column blocks), with the row shapes where the kernels' units meet: 4-entry lanes, 128-entry warp passes,
2048-entry tiles, empty rows, single-entry rows, rows through several tiles.

Accuracy.  p = val * x[col] are the fp64 products every kernel forms (unfused).  Summed in any order in fp64, a row of
n products lies within n * 2^-53 * sum|p| of their exact sum (Jeannerod & Rump, 2013), and the reference below is the
exact sum rounded once (math.fsum) or an extended-precision sum whose own error is far inside that bound.  Kernels that
keep the ascending column order must match the sequential CRS result bit for bit.
"""
import math

import numpy as np
import pytest

U = 2.0 ** -53
# decision constants of the engine, in columns of fp64 x
BAND_COLS = (32 << 20) // 8          # primitives.cu gathers_need_l2: a wider band makes the gathers depend on L2
X_L2_COLS = (64 << 20) // 8          # ss.cu make_col_block_engine: a larger x is column-blocked
SLICE_COLS = (45 << 20) // 8         # colblocks.cuh COLBLOCK_SLICE_BYTES: widest column block
SPREAD_MIN = 1.5                     # ... when the rows touch this many column blocks on average (also CSS)
PAD_MAX = 2.0                        # sliced ELL per column block while it needs at most this many slots per entry
TS_LONG = 64                         # tile-stream: longer rows (per column block) are reduced by a warp
JDS_LONG = 2048                      # JDS: longer rows are reduced by a warp
TILE = 2048

NCOL = {"A": (BAND_COLS + X_L2_COLS) // 2,   # band 1.5x the limit, x 0.75x the column-block limit: no column blocks
        "B": 1 << 24}                         # x = 128 MB: column-blocked
N_COLBLOCKS = -(-NCOL["B"] // SLICE_COLS)
assert N_COLBLOCKS == 3 and NCOL["B"] > 1.5 * X_L2_COLS

# the boundary row-length lists of test_crs_entry_stream and test_coo_entry_stream_chunk_boundaries
BOUNDARY_LENS = ([4] * 64 + [128] * 3 + [256, 256, 1, 255, 2048, 2047, 1, 1, 4096 + 256, 3],
                 [1] * 5000,
                 [0, 0, 3, 0, 125, 0, 0, 128, 1, 0, 255, 257, 0, 0, 0, 6000, 0, 2, 0, 0],
                 [27] * 700 + [0] * 9,
                 [7] * 3000 + [0] * 9,
                 [300] * 40 + [5] * 13,
                 [1, 2047, 2048 * 5, 1])

FORMATS = [("crs", {}), ("coo", {}), ("ell", {}), ("jds", {}), ("ss", {}), ("css", {"n_block": 3}), ("csr5", {}),
           ("hyb", {})]
ROW_FORMATS = ("crs", "ss", "css", "ell", "dia")      # formats with multiply_rows
G = 4096                                              # guard band, entries
CANARY = -12345.0


# ------------------------------------------------------------------------------------------ reference and bound
def row_reference(nRow, row, p, extended=None):
    """(ref, bound): ref = sum of the products of each row, exact up to far less than the bound; bound = n * 2^-53 *
    sum|p| per row.  extended: use np.longdouble (None = when it has more than 52 mantissa bits), else math.fsum."""
    lens = np.bincount(row, minlength=nRow)[:nRow]
    ptr = np.concatenate([[0], np.cumsum(lens)])
    if extended is None:
        extended = np.finfo(np.longdouble).nmant > 52
    ref = np.zeros(nRow, np.longdouble)
    mag = np.zeros(nRow, np.longdouble)
    nz = np.flatnonzero(lens)
    if extended and len(nz):
        pl = p.astype(np.longdouble)
        ref[nz] = np.add.reduceat(pl, ptr[nz])
        mag[nz] = np.add.reduceat(np.abs(pl), ptr[nz])
        # an extended sum of n terms is off by up to (n-1) 2^-64 sum|p|: inside the margin of the bound up to n = 2049
        nz = np.flatnonzero(lens > 2048)
    for r in nz:
        q = p[ptr[r]:ptr[r + 1]]
        ref[r] = math.fsum(q)
        mag[r] = math.fsum(np.abs(q))
    return ref, lens * U * mag


def within_bound(y, ref, bound):
    return np.abs(y.astype(np.longdouble) - ref) <= bound


def assert_rows(y, c, tag, exact=None):
    """y within the bound on every row, empty rows exactly +0.0, rows in `exact` bit-identical to the CRS result."""
    ok = within_bound(y, c.ref, c.bound)
    assert np.all(ok), (tag, "rows off: %d, first %d" % ((~ok).sum(), int(np.flatnonzero(~ok)[0])))
    e = c.lens == 0
    assert np.all(y[e] == 0.0) and not np.any(np.signbit(y[e])), (tag, "empty rows must be +0.0")
    if exact is not None:
        assert np.array_equal(y[exact], c.y_crs[exact]), (tag, "rows off the sequential CRS bits: %d" % (y[exact] != c.y_crs[exact]).sum())


def test_row_bound_checker():
    """The checker itself: it accepts fp64 sums of the same products in 100 random orders (sequential and pairwise) and
    rejects a sum with one product dropped or duplicated; the extended-precision and the fsum reference agree."""
    rng = np.random.default_rng(1)
    lens = np.array([0, 1, 2, 7, 0, 33, 128, 2049, 3000, 5, 0])
    nRow = len(lens)
    row = np.repeat(np.arange(nRow), lens)
    p = rng.choice([-1.0, 1.0], len(row)) * 10.0 ** rng.uniform(-6, 6, len(row)) * rng.uniform(-1, 1, len(row))
    ptr = np.concatenate([[0], np.cumsum(lens)])
    for extended in (True, False):
        if extended and np.finfo(np.longdouble).nmant <= 52:
            continue
        ref, bound = row_reference(nRow, row, p, extended=extended)
        ref2, bound2 = row_reference(nRow, row, p, extended=not extended)
        assert np.all(np.abs(ref - ref2) <= bound) and np.allclose(bound.astype(float), bound2.astype(float), rtol=1e-12, atol=0)
        for trial in range(100):
            y = np.zeros(nRow)
            for r in range(nRow):
                q = p[ptr[r]:ptr[r + 1]][rng.permutation(lens[r])]
                y[r] = np.cumsum(q)[-1] if len(q) and trial % 2 else np.sum(q)   # sequential / pairwise
            assert np.all(within_bound(y, ref, bound)), trial
        for r in np.flatnonzero(lens):
            q = p[ptr[r]:ptr[r + 1]]
            big = int(np.argmax(np.abs(q)))
            for bad in (np.delete(q, big), np.append(q, q[big])):
                y = np.array([math.fsum(p[ptr[i]:ptr[i + 1]]) for i in range(nRow)])
                y[r] = math.fsum(bad)
                assert not within_bound(y, ref, bound)[r], (r, lens[r])


# ------------------------------------------------------------------------------------------ wide matrices
class Case:
    pass


def wide_case(name, lens, nCol, seed):
    """Sorted duplicate-free COO: row i takes lens[i] distinct columns drawn uniformly from [0, nCol); values of random
    sign with magnitudes 10^U(-6,6).  Also the per-block statistics the engine decides on."""
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, np.int64)
    nRow = len(lens)
    row = np.repeat(np.arange(nRow, dtype=np.int64), lens)
    col = rng.integers(0, nCol, len(row))
    while True:
        key = row * nCol + col
        key.sort()
        col = key - row * nCol
        dup = np.flatnonzero(key[1:] == key[:-1]) + 1
        if not len(dup):
            break
        col[dup] = rng.integers(0, nCol, len(dup))
    c = Case()
    c.name, c.nRow, c.nCol, c.lens = name, nRow, nCol, lens
    c.row, c.col = row.astype(np.int32), col.astype(np.int32)
    c.val = rng.choice([-1.0, 1.0], len(row)) * 10.0 ** rng.uniform(-6, 6, len(row))
    c.x = rng.uniform(-1.0, 1.0, nCol)
    c.x2 = rng.uniform(-1.0, 1.0, nCol)
    c.ptr = np.concatenate([[0], np.cumsum(lens)])
    if len(row):
        assert np.max(np.abs(col - row)) > 1.2 * BAND_COLS, name           # the band is what selects the load-fed paths
    # three column blocks of ceil(nCol / 3) columns: the engine's blocks on width B, CSS's (n_block = 3) on both widths
    Bw = -(-nCol // 3)
    cnt = np.bincount(row * 3 + col // Bw, minlength=3 * nRow).reshape(nRow, 3)
    c.piece_max = cnt.max(axis=1)
    nonempty = lens > 0
    spread = (cnt > 0).sum() / max(1, nonempty.sum())
    nSl = -(-nRow // 32)
    pad = np.zeros((nSl * 32, 3), np.int64)
    pad[:nRow] = cnt
    slots = 64 * (-(-pad.reshape(nSl, 32, 3).max(axis=1) // 2)).sum()      # V = 2 slots per group, 32 lanes
    ratio = slots / max(1, len(row))
    # keep clear of the thresholds (the padding is an average over thousands of slices: K = 11 gives 2.05 +- 0.003)
    assert not 0.9 * SPREAD_MIN < spread < 1.1 * SPREAD_MIN, (name, spread)
    assert not 0.99 * PAD_MAX < ratio < 1.01 * PAD_MAX, (name, ratio)
    c.blocked_engine = 0 if spread < SPREAD_MIN else 1 if ratio <= PAD_MAX else 2
    return c


def with_reference(c, oracle):
    p = c.val * c.x[c.col]
    c.ref, c.bound = row_reference(c.nRow, c.row, p)
    c.y_crs = oracle.crs_result(c.nRow, c.row, c.col, c.val, c.x)
    return c


def bulk_lens(kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "k11":
        return [11] * (1 << 19)
    if kind == "k32":
        return [32] * (1 << 18)
    lens = np.minimum(rng.zipf(1.5, 1 << 16), 4096)             # power law, R-MAT-like
    lens[rng.random(len(lens)) < 0.1] = 0
    return lens


def cases_for(width, oracle):
    nCol = NCOL[width]
    out = [wide_case("lens%d" % i, l, nCol, 100 + i) for i, l in enumerate(BOUNDARY_LENS)]
    out += [wide_case(k, bulk_lens(k, 7), nCol, 200 + i) for i, k in enumerate(("k11", "k32", "powerlaw"))]
    return [with_reference(c, oracle) for c in out]


@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


@pytest.fixture(scope="module")
def wide(oracle):
    memo = {}

    def get(width):
        if width not in memo:
            memo[width] = cases_for(width, oracle)
        return memo[width]
    return get


# ------------------------------------------------------------------------------------------ device helpers
class Guarded:
    """x between NaN bands and y between canary bands: a gather outside x poisons y, a store outside y breaks a canary."""

    def __init__(self, x, nRow):
        import torch
        self.nRow = nRow
        self.xb = torch.full((len(x) + 2 * G,), float("nan"), dtype=torch.float64, device="cuda")
        self.xb[G:G + len(x)] = torch.from_numpy(x).cuda()
        self.yb = torch.full((nRow + 2 * G,), CANARY, dtype=torch.float64, device="cuda")
        self.xp, self.yp = self.xb.data_ptr() + 8 * G, self.yb.data_ptr() + 8 * G

    def reset(self):
        self.yb.fill_(CANARY)

    def y(self, lo=0, hi=None, tag=""):
        """y after a multiply of rows [lo, hi): everything outside them still holds the canary."""
        import torch
        hi = self.nRow if hi is None else hi
        torch.cuda.synchronize()
        yb = self.yb.cpu().numpy()
        assert np.all(yb[:G + lo] == CANARY) and np.all(yb[G + hi:] == CANARY), (tag, "store outside rows [%d,%d)" % (lo, hi))
        return yb[G:G + self.nRow]


def convert(sp, fmt, opt, c):
    return sp.SpMatOpt(fmt, **opt).convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))


def exact_rows(fmt, A, c):
    """Rows the format sums in ascending column order with one thread: bit-identical to the sequential CRS result."""
    eng = A.scalar("col_block_engine") if fmt in ("ell", "jds", "ss") else None
    if eng == 1 or (fmt == "ell" and eng == 0):
        return np.ones(c.nRow, bool)
    if eng == 2:
        return c.piece_max <= TS_LONG
    if fmt == "ss":
        return c.lens <= TS_LONG
    if fmt == "jds":
        return c.lens <= JDS_LONG
    return None


def assert_path(fmt, A, c, width, reached):
    """The kernel each case is meant to reach: a moved threshold fails here instead of quietly testing another path."""
    if fmt == "crs":
        assert A.scalar("crs_kernel") == 3, c.name                 # load-fed entry stream
    if fmt == "coo":
        assert A.scalar("coo_path") == 2, c.name                   # load-fed entry stream
    if fmt == "ss":
        assert A.scalar("short_row_path") == 0, c.name             # gather-bound: not the row-chunk stream
    if fmt in ("ell", "jds", "ss"):
        want = c.blocked_engine if width == "B" else 0
        got = (A.scalar("col_blocks"), A.scalar("col_block_engine"))
        assert got == ((N_COLBLOCKS if want else 0), want), (fmt, c.name, got)
        reached.add((fmt, want))
    if fmt == "css":
        assert A.scalar("nBlock") == 3 and A.scalar("col_block_engine") == c.blocked_engine, (c.name, A.scalar("col_block_engine"))
        reached.add((fmt, c.blocked_engine))


# ------------------------------------------------------------------------------------------ tests
@pytest.mark.gpu
@pytest.mark.parametrize("width", ["A", "B"])
def test_wide_paths_and_accuracy(sp, wide, width):
    """Every format on every wide case: the intended kernel, no access outside x and y, every row within the bound of the
    extended-precision sum, empty rows +0.0, order-keeping kernels bit-identical to the CRS result."""
    reached = set()
    for c in wide(width):
        g = Guarded(c.x, c.nRow)
        for fmt, opt in FORMATS:
            A = convert(sp, fmt, opt, c)
            assert_path(fmt, A, c, width, reached)
            g.reset()
            A.multiply(g.xp, g.yp)
            y = g.y(tag=(fmt, c.name))
            assert_rows(y, c, (fmt, c.name), exact_rows(fmt, A, c))
            A.destroy()
    if width == "B":      # both column-block engines were reached at this size, for every format that has them
        assert reached >= {(f, e) for f in ("ell", "jds", "ss", "css") for e in (1, 2)}, sorted(reached)
    else:
        assert reached >= {("ell", 0), ("jds", 0), ("ss", 0), ("css", 1), ("css", 2)}, sorted(reached)


def range_cuts(c):
    """Row cuts: rows whose entries start off each of the entry stream's units, the two sides of every row that runs
    through several tiles (so neighbouring ranges start or end inside its tiles), a run of empty rows."""
    cuts = {0, c.nRow}
    start = c.ptr[:-1]
    for unit in (4, 128, 256, TILE):
        off = np.flatnonzero((start % unit != 0) & (c.lens > 0))
        if len(off):
            cuts.add(int(off[len(off) // 2]))
    multi = np.flatnonzero((c.lens > 0) & ((c.ptr[1:] - 1) // TILE > start // TILE))
    for r in multi[:3]:
        cuts |= {int(r), int(r) + 1}
    empty = np.flatnonzero(c.lens == 0)
    if len(empty):
        r = int(empty[len(empty) // 2])
        e = r
        while e < c.nRow and c.lens[e] == 0:
            e += 1
        cuts |= {r, e}
    cuts = sorted(cuts)
    return list(zip(cuts[:-1], cuts[1:]))


@pytest.mark.gpu
@pytest.mark.parametrize("width", ["A", "B"])
def test_wide_row_ranges(sp, wide, width):
    """multiply_rows on cuts off every unit, around multi-tile rows and over empty rows only: each range writes exactly
    its rows, and the pieces give the bits of the whole multiply."""
    for c in wide(width):
        if c.name == "k32":
            continue                              # same kernels as k11 at the uniform shape, only more entries
        g = Guarded(c.x, c.nRow)
        pieces = range_cuts(c)
        for fmt, opt in FORMATS:
            if fmt not in ROW_FORMATS:
                continue
            A = convert(sp, fmt, opt, c)
            g.reset()
            A.multiply(g.xp, g.yp)
            whole = g.y(tag=(fmt, c.name)).copy()
            for a, b in pieces:
                g.reset()
                A.multiply_rows(a, b, g.xp, g.yp)
                y = g.y(a, b, tag=(fmt, c.name, a, b))
                assert np.array_equal(y[a:b], whole[a:b]), (fmt, c.name, a, b)
            A.destroy()


def capture_check(sp, A, fmt, nRow, x1, x2, cuts, tag):
    """One eager multiply, prepare_rows for the cuts, then multiply and the prepared multiply_rows captured on a
    non-default stream; x is overwritten in place before the replay: same bits as the eager multiply with that x."""
    import torch
    xd = torch.from_numpy(x2).cuda()
    y_eager = torch.full((nRow,), float("nan"), dtype=torch.float64, device="cuda")
    A.multiply(xd.data_ptr(), y_eager.data_ptr())
    rows = fmt in ROW_FORMATS
    pieces = list(zip(cuts[:-1], cuts[1:]))
    if rows:
        for a, b in pieces:
            A.prepare_rows(a, b)
    xd.copy_(torch.from_numpy(x1))
    y_full = torch.full((nRow,), float("nan"), dtype=torch.float64, device="cuda")
    y_rows = torch.full((nRow,), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    graph, stream = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=stream):
        h = stream.cuda_stream
        A.multiply(xd.data_ptr(), y_full.data_ptr(), h)
        if rows:
            for a, b in pieces:
                A.multiply_rows(a, b, xd.data_ptr(), y_rows.data_ptr(), h)
    xd.copy_(torch.from_numpy(x2))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(y_full, y_eager), tag
    if rows:
        assert torch.equal(y_rows, y_eager), tag


@pytest.mark.gpu
@pytest.mark.parametrize("width", ["A", "B"])
def test_wide_capture_prepared_rows(sp, wide, width):
    """CUDA-graph capture of every format and path reached on the wide matrices, including the tile-streams that the
    column-block engines and gather-bound CSS blocks run: prepare_rows must cover them (b200spmv.h)."""
    for c in wide(width):
        if not c.name.startswith(("k11", "k32", "powerlaw")):
            continue
        n = c.nRow
        cuts = [0, n // 3, n // 3 + 1, 2 * n // 3 + 5, n]
        for fmt, opt in FORMATS:
            A = convert(sp, fmt, opt, c)
            capture_check(sp, A, fmt, n, c.x, c.x2, cuts, (fmt, c.name, width))
            A.destroy()


@pytest.mark.gpu
def test_banded_capture_prepared_rows(sp, oracle):
    """The same capture on a banded matrix for the paths of test_guard_bands_around_x_and_y."""
    from test_gpu_parity import GUARD_FORMATS
    nr, nc, row, col, val = oracle.stencil("lap3d7", 13)
    rng = np.random.default_rng(9)
    x1, x2 = rng.random(nc), rng.random(nc)
    for fmt, opt in GUARD_FORMATS:
        if opt.get("profile"):
            continue                              # profiled multiplies synchronise by design
        A = sp.SpMatOpt(fmt, **opt).convert_host(sp.SpMat(nr, nc, row, col, val))
        capture_check(sp, A, fmt, nr, x1, x2, [0, 129, 130, nr - 77, nr], (fmt, opt))
        A.destroy()


@pytest.mark.gpu
def test_wide_host_pipeline(sp, oracle):
    """multiply_host with page-locked vectors at 2^20 rows on width B: row chunks with x uploaded in pieces (CRS, load-fed
    entry stream) and per-column-slice multiplies of CSS's sliced-ELL blocks.  A new x each call; same bits as the device
    multiply.  One slice of 32 rows in four has 32 entries, the others are empty (about 8 M entries)."""
    import torch
    n, K = 1 << 20, 32
    lens = np.zeros(n, np.int64)
    lens.reshape(-1, 4, 32)[:, 0, :] = K
    c = with_reference(wide_case("pipeline", lens, NCOL["B"], 300), oracle)
    xs = np.empty(c.nCol)
    y = np.empty(n)
    assert sp.host_register(xs) and sp.host_register(y)
    try:
        for fmt, opt in (("crs", {}), ("css", {"n_block": 3})):
            A = convert(sp, fmt, opt, c)
            if fmt == "crs":
                assert A.scalar("crs_kernel") == 3 and A.scalar("has_rows") == 1
            else:
                assert A.scalar("col_block_engine") == 1 and c.blocked_engine == 1
            for i, x in enumerate((c.x, c.x2, c.x[::-1].copy())):
                xs[:] = x
                y[:] = np.nan
                A.multiply_host(xs, y)
                xd = torch.from_numpy(x).cuda()
                yd = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
                A.multiply(xd.data_ptr(), yd.data_ptr())
                torch.cuda.synchronize()
                assert np.array_equal(y, yd.cpu().numpy()), (fmt, i)
                if i == 0:
                    assert_rows(y, c, fmt)
            A.destroy()
    finally:
        sp.host_unregister(xs)
        sp.host_unregister(y)


@pytest.mark.gpu
def test_wide_row_blocks(sp, oracle, monkeypatch):
    """Row blocks (blocked.cu, forced small with B200SPMV_BLOCK_NNZ) on width A: each block is an ordinary matrix that
    measures its own band and stays on the load-fed entry stream; y within the bound, a row range across blocks."""
    c = with_reference(wide_case("powerlaw", bulk_lens("powerlaw", 7), NCOL["A"], 202), oracle)
    g = Guarded(c.x, c.nRow)
    for fmt in ("crs", "coo"):
        monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(c.row) // 5))
        A = convert(sp, fmt, {}, c)
        monkeypatch.delenv("B200SPMV_BLOCK_NNZ")
        assert A.scalar("row_blocks") >= 4 and A.scalar("nNnz") == len(c.row)
        assert A.scalar("crs_kernel" if fmt == "crs" else "coo_path") == (3 if fmt == "crs" else 2)
        g.reset()
        A.multiply(g.xp, g.yp)
        whole = g.y(tag=fmt).copy()
        assert_rows(whole, c, fmt)
        if fmt == "crs":
            lo, hi = c.nRow // 7, c.nRow - c.nRow // 5
            A.prepare_rows(lo, hi)
            g.reset()
            A.multiply_rows(lo, hi, g.xp, g.yp)
            assert np.array_equal(g.y(lo, hi, tag=fmt)[lo:hi], whole[lo:hi])
        A.destroy()
