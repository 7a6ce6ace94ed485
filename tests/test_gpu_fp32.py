"""The fp32 variants (options.precision) against exact fp32 and fp64 row sums.

precision = 1: fp32 values, x and y, products and sums in fp32.  precision = 2: the same vectors, sums in fp64, rounded to
fp32 once.  a32 and x32 are the inputs as the conversion rounds them (val.astype(np.float32)); p = a32 * x32 are the
exact products (exact in fp64) and s their exact sum per row.

seq(1) sums the fp32 products in ascending column order in fp32 (numpy neither fuses nor flushes subnormals).  seq(2)
sums the exact products in the same order in fp64 and rounds once.  The kernels that keep that order (the CRS row-chunk
stream, tile-stream rows of at most 64 entries, ELL, DIA, and row blocks of any of them) must give the bits of seq; CSR5
and longer tile-stream rows must lie within
    precision 2: |y - s| <= 2^-24 |s| + n 2^-53 sum|p| + 2^-149     (an fp64 sum in any order, rounded once)
    precision 1: |y - s| <= (n+1) 2^-24 sum|p| + (n+1) 2^-149        (fp32 products and sums in any order)
A precision-2 row rounded to fp32 partway (a tile's partial, then the carries) breaks the first bound on a cancelling row.
"""
import numpy as np
import pytest

from test_gpu_gather_bound import BOUNDARY_LENS, row_reference
from test_gpu_parity import _short_row_matrix

E24, U, TINY = 2.0 ** -24, 2.0 ** -53, 2.0 ** -149
TS_LONG = 64                        # tile-stream: longer rows are not summed in column order
G = 4096                            # guard band, entries
CANARY = np.float32(-12345.0)
PATHS = [("crs", {}), ("crs", {"crs_path": 1}), ("ell", {}), ("dia", {}), ("csr5", {"csr5_sigma": 4}),
         ("csr5", {"csr5_sigma": 16})]


# ------------------------------------------------------------------------------------------ references
def row_ptr(nRow, row):
    lens = np.bincount(row, minlength=nRow)[:nRow]
    return lens, np.concatenate([[0], np.cumsum(lens)])


def seq(prec, nRow, row, col, a32, x32):
    """Row sums in ascending column order: fp32 products and sums (1), exact products summed in fp64 and rounded once (2).
    Vectorised over the rows: step k adds the k-th entry of every row that has one."""
    lens, ptr = row_ptr(nRow, row)
    with np.errstate(all="ignore"):
        if prec == 1:
            p, acc = a32 * x32[col], np.zeros(nRow, np.float32)
        else:
            p, acc = a32.astype(np.float64) * x32[col].astype(np.float64), np.zeros(nRow)
        order = np.argsort(-lens, kind="stable")
        n_longer = len(order) - np.searchsorted(lens[order][::-1], np.arange(int(lens.max(initial=0))), side="right")
        for k, m in enumerate(n_longer):
            r = order[:m]
            acc[r] = acc[r] + p[ptr[r] + k]
        return acc if prec == 1 else acc.astype(np.float32)


def bound(prec, nRow, row, col, a32, x32):
    """(s, limit): the exact row sums (row_reference: extended precision or fsum) and the bound of the module docstring."""
    p = a32.astype(np.float64) * x32[col].astype(np.float64)
    s, _ = row_reference(nRow, row, p)
    lens, _ = row_ptr(nRow, row)
    mag = np.zeros(nRow, np.longdouble)
    np.add.at(mag, row, np.abs(p).astype(np.longdouble))
    n = lens.astype(np.longdouble)
    if prec == 2:
        return s, E24 * np.abs(s) + n * U * mag + TINY
    return s, (n + 1) * E24 * mag + (n + 1) * TINY


def same_bits(a, b):
    """Per row: the same fp32 bits (the sign of zero included), or NaN in both."""
    na, nb = np.isnan(a), np.isnan(b)
    return (na & nb) | (~na & ~nb & (a.view(np.uint32) == b.view(np.uint32)))


def within(y, s, lim):
    with np.errstate(invalid="ignore"):
        return np.abs(y.astype(np.longdouble) - s) <= lim


class Case:
    def __init__(self, name, nRow, nCol, row, col, val, x):
        self.name, self.nRow, self.nCol = name, nRow, nCol
        self.row, self.col, self.val, self.x = row.astype(np.int32), col.astype(np.int32), np.asarray(val, np.float64), x
        self.a32, self.x32 = self.val.astype(np.float32), x.astype(np.float32)
        self.lens, self.ptr = row_ptr(nRow, self.row)
        self.seq = {q: seq(q, nRow, self.row, self.col, self.a32, self.x32) for q in (1, 2)}
        self.lim = {q: bound(q, nRow, self.row, self.col, self.a32, self.x32) for q in (1, 2)}


def check(y, c, prec, exact, tag):
    """exact: rows that must carry the bits of seq(prec) (None = all).  Every row whose seq(prec) is finite lies within
    the bound; empty rows are +0.0."""
    ref = c.seq[prec]
    rows = np.ones(c.nRow, bool) if exact is None else exact
    ok = same_bits(y, ref) | ~rows
    assert np.all(ok), (tag, "rows off seq(%d): %d, first %d" % (prec, (~ok).sum(), int(np.flatnonzero(~ok)[0])))
    s, lim = c.lim[prec]
    fin = np.isfinite(ref)
    ok = within(y, s, lim) | ~fin
    assert np.all(ok), (tag, "rows off the bound: %d, first %d" % ((~ok).sum(), int(np.flatnonzero(~ok)[0])))
    e = c.lens == 0
    assert np.all(y[e].view(np.uint32) == 0), (tag, "empty rows must be +0.0")


# ------------------------------------------------------------------------------------------ the checker itself (CPU)
def test_fp32_row_checker():
    """seq(1) and seq(2) differ on designed rows; the precision-2 bound accepts fp64 sums of the same exact products in
    random orders, rounded once, and rejects one intermediate fp32 rounding on a cancelling row and a dropped product."""
    rows = [[2.0 ** 24, 1.0, 1.0], [1.0, 2.0 ** 24, 1.0, 1.0, 1.0], [2.0 ** 25, 1.0, 1.0, 1.0]]
    for v in rows:
        n = len(v)
        row, col = np.zeros(n, np.int32), np.arange(n, dtype=np.int32)
        a32, x32 = np.array(v, np.float32), np.ones(n, np.float32)
        s1, s2 = seq(1, 1, row, col, a32, x32), seq(2, 1, row, col, a32, x32)
        assert s2[0] == np.float32(sum(v)) and s1[0] != s2[0], v
        s, lim = bound(2, 1, row, col, a32, x32)
        assert within(s2, s, lim)[0] and not within(s1, s, lim)[0], v
        assert within(s1, *bound(1, 1, row, col, a32, x32))[0], v
    rng = np.random.default_rng(3)
    lens = np.array([0, 1, 2, 5, 65, 200, 0, 2049, 6000, 3])
    nRow = len(lens)
    row = np.repeat(np.arange(nRow), lens).astype(np.int32)
    ptr = np.concatenate([[0], np.cumsum(lens)])
    nCol = 8000
    col = np.concatenate([np.sort(rng.choice(nCol, k, replace=False)) for k in lens]).astype(np.int32)
    a32 = (rng.choice([-1, 1], len(row)) * 10.0 ** rng.uniform(-2, 0, len(row))).astype(np.float32)
    x32 = rng.uniform(-1, 1, nCol).astype(np.float32)
    x32[[0, nCol - 1]] = 1.0
    pair = lens >= 65                              # a +-2^20 pair at the first and last entries: cancelling rows
    col[ptr[:-1][pair]], col[ptr[1:][pair] - 1] = 0, nCol - 1
    a32[ptr[:-1][pair]], a32[ptr[1:][pair] - 1] = 2.0 ** 20, -2.0 ** 20
    p = a32.astype(np.float64) * x32[col].astype(np.float64)
    s, lim = bound(2, nRow, row, col, a32, x32)
    assert np.all(within(seq(2, nRow, row, col, a32, x32), s, lim))
    assert np.all(within(seq(1, nRow, row, col, a32, x32), *bound(1, nRow, row, col, a32, x32)))
    for trial in range(50):
        y = np.zeros(nRow, np.float32)
        for r in range(nRow):
            q = p[ptr[r]:ptr[r + 1]][rng.permutation(lens[r])]
            y[r] = np.float32(np.cumsum(q)[-1] if len(q) and trial % 2 else np.sum(q))
        assert np.all(within(y, s, lim)), trial
    for r in np.flatnonzero(lens):
        q = p[ptr[r]:ptr[r + 1]]
        y = seq(2, nRow, row, col, a32, x32)
        y[r] = np.float32(np.sum(np.delete(q, int(np.argmax(np.abs(q))))))       # one product dropped
        assert not within(y, s, lim)[r], (r, lens[r])
        if pair[r]:                                 # the partial up to a cut rounded to fp32, then the rest in fp64
            for cut in (2, lens[r] // 2, lens[r] - 1):
                y[r] = np.float32(float(np.float32(np.sum(q[:cut]))) + np.sum(q[cut:]))
                assert not within(y, s, lim)[r], (r, lens[r], cut)


# ------------------------------------------------------------------------------------------ device helpers
@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


def convert(sp, fmt, opt, prec, c):
    A = sp.SpMatOpt(fmt, precision=prec, **opt).convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))
    assert A.scalar("precision") == prec
    return A


def device_multiply(A, c, x32=None):
    """multiply_f32 with x between NaN bands and y between canary bands (twice: the second over the first's y)."""
    import torch
    x32 = c.x32 if x32 is None else x32
    xb = torch.full((c.nCol + 2 * G,), float("nan"), dtype=torch.float32, device="cuda")
    xb[G:G + c.nCol] = torch.from_numpy(x32).cuda()
    yb = torch.full((c.nRow + 2 * G,), float(CANARY), dtype=torch.float32, device="cuda")
    for _ in range(2):
        A.multiply_f32(xb.data_ptr() + 4 * G, yb.data_ptr() + 4 * G)
    torch.cuda.synchronize()
    yb = yb.cpu().numpy()
    assert np.all(yb[:G] == CANARY) and np.all(yb[G + c.nRow:] == CANARY), "store outside y"
    return yb[G:G + c.nRow]


def run(sp, fmt, opt, prec, c):
    """y of the device entry; the host entry must give the same bits."""
    A = convert(sp, fmt, opt, prec, c)
    y = device_multiply(A, c)
    yh = np.full(c.nRow, np.nan, np.float32)
    A.multiply_host_f32(c.x32, yh)
    assert np.array_equal(y.view(np.uint32), yh.view(np.uint32)), (fmt, opt, prec, c.name, "host entry")
    return A, y


def exact_rows(fmt, A, c):
    """Rows summed in ascending column order by one thread (None = all), else the bound only."""
    if fmt == "csr5":
        return np.zeros(c.nRow, bool)
    if fmt == "crs" and A.scalar("crs_kernel") == 0:
        return c.lens <= TS_LONG                    # tile-stream; crs_kernel 1 = row-chunk stream, every row
    return None


def check_paths(sp, c, paths=PATHS):
    for fmt, opt in paths:
        if fmt == "dia" and len(np.unique(c.col.astype(np.int64) - c.row)) * c.nRow > 3e7:
            continue
        if fmt == "ell" and c.lens.max(initial=0) > c.nCol:
            continue
        for prec in (1, 2):
            A, y = run(sp, fmt, opt, prec, c)
            if fmt == "crs":
                want = 0 if opt.get("crs_path") == 1 or c.lens.max(initial=0) > 16 else 1
                assert A.scalar("crs_kernel") == want, (c.name, opt, A.scalar("crs_kernel"))
            check(y, c, prec, exact_rows(fmt, A, c), (fmt, opt, prec, c.name))
            A.destroy()


def sorted_case(name, lens, nCol, seed, lo=-2, hi=0):
    """Row i takes lens[i] distinct sorted columns in [0, nCol); values of random sign, magnitudes 10^U(lo,hi)."""
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, np.int64)
    row = np.repeat(np.arange(len(lens)), lens)
    col = np.concatenate([np.sort(rng.choice(nCol, int(k), replace=False)) for k in lens]) if len(row) else row
    val = rng.choice([-1.0, 1.0], len(row)) * 10.0 ** rng.uniform(lo, hi, len(row))
    return Case(name, len(lens), nCol, row, col, val, rng.uniform(-1.0, 1.0, nCol))


# ------------------------------------------------------------------------------------------ tests
@pytest.mark.gpu
@pytest.mark.parametrize("max_len", [1, 5, 8, 9, 16])
def test_fp32_chunk_stream_boundaries(sp, max_len):
    """Short rows (the MAXL 8 and 16 instantiations of the row-chunk stream, ELL V = 2 and 4) with empty rows and an empty
    tail, through every fp32 path at both precisions."""
    rng = np.random.default_rng(500 + max_len)
    nRow, nCol = 5003, 4097
    row, col, val = _short_row_matrix(rng, nRow, nCol, max_len)
    keep = row < nRow - 37
    c = Case("short%d" % max_len, nRow, nCol, row[keep], col[keep], val[keep], rng.uniform(-1.0, 1.0, nCol))
    A = convert(sp, "ell", {}, 2, c)
    assert A.scalar("slice_vec") == (4 if max_len % 4 == 0 else 2)
    A.destroy()
    check_paths(sp, c, [p for p in PATHS if p[0] != "dia"])


@pytest.mark.gpu
@pytest.mark.parametrize("K", [3, 31, 32, 33])
def test_fp32_ell_slice_groups(sp, K):
    """ELL slices whose longest row varies from slice to slice: odd and even group counts (the kernel takes groups in
    pairs), V = 2 (K = 3, 31) and V = 4 (K = 32, 33), fully empty slices."""
    rng = np.random.default_rng(600 + K)
    nSl = 97
    lens = np.zeros(nSl * 32, np.int64)
    for s in range(nSl):
        m = 0 if s % 11 == 5 else 1 + (7 * s) % K
        if m:
            lens[32 * s:32 * s + 32] = rng.integers(0, m + 1, 32)
            lens[32 * s + int(rng.integers(32))] = m
    lens[-40:] = 0
    c = sorted_case("ellK%d" % K, lens, 700, 610 + K)
    V = 4 if K % 4 == 0 or K >= 32 else 2
    groups = {-(-int(c.lens[32 * s:32 * s + 32].max()) // V) for s in range(nSl)}
    assert {g % 2 for g in groups if g} == {0, 1}
    A = convert(sp, "ell", {}, 1, c)
    assert A.scalar("slice_vec") == V and A.scalar("K") == K
    A.destroy()
    check_paths(sp, c, [p for p in PATHS if p[0] != "dia"])


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(BOUNDARY_LENS)))
def test_fp32_tile_boundaries(sp, i):
    """The boundary row-length lists of the entry-stream tests at a narrow width: rows that start a few entries before a
    2048-entry tile edge, rows of more than 64 entries across it, a row through five tiles."""
    c = sorted_case("lens%d" % i, BOUNDARY_LENS[i], 12007, 700 + i)
    check_paths(sp, c, [p for p in PATHS if p[0] != "dia"])


def cancelling_case(tile, seed):
    """Rows of 65 ... 6000 entries with a +-2^20 pair at their first and last entries, each starting a few entries before
    an edge of `tile`-entry tiles so that the pair lands in different tiles; short filler rows in between."""
    rng = np.random.default_rng(seed)
    nCol = 8192
    long_lens = [65, 66, 100, 127, 200, 513, 2047, 2100, 6000]
    lead = [1, 2, 17, 63, 64, 65, 100, 127, 1000]
    lens, pos, pair_rows = [], 0, []
    for L, d in zip(long_lens, lead):
        d = min(d, L - 1, tile - 1)
        start = -(-(pos + d) // tile) * tile - d       # the first such start at or after pos
        while pos < start:
            k = min(int(rng.integers(0, 9)), start - pos)
            lens.append(k)
            pos += k
        pair_rows.append(len(lens))
        lens.append(L)
        pos += L
        lens += [0, 3]
        pos += 3
    c = sorted_case("cancel%d" % tile, lens, nCol, seed)
    ptr = np.concatenate([[0], np.cumsum(lens)])
    col, val, x = c.col.copy(), c.val.copy(), c.x.copy()
    for r in pair_rows:                             # first and last entries: columns 0 and nCol-1, x = 1, values +-2^20
        col[ptr[r] + 1:ptr[r + 1] - 1] = np.sort(rng.choice(np.arange(1, nCol - 1), lens[r] - 2, replace=False))
        col[ptr[r]], col[ptr[r + 1] - 1] = 0, nCol - 1
        val[ptr[r]], val[ptr[r + 1] - 1] = 2.0 ** 20, -2.0 ** 20
    x[[0, nCol - 1]] = 1.0
    c = Case(c.name, c.nRow, nCol, c.row, col, val, x)
    c.pair_rows = np.array(pair_rows)
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("tile", [2048, 512, 128])
def test_fp32_cancelling_rows_across_tiles(sp, tile):
    """Cancelling long rows across the edges of the CRS tile-stream (2048 entries) and CSR5 tiles (sigma 16: 512, sigma 4:
    128).  Precision 2 must round once: a partial rounded to fp32 at the tile edge is off the bound by orders of
    magnitude on these rows."""
    c = cancelling_case(tile, 800 + tile)
    s, lim = c.lim[2]
    assert np.all(lim[c.pair_rows] < 1e-4)           # the bound on those rows, against ~2^-4 for an early rounding
    check_paths(sp, c, [p for p in PATHS if p[0] != "dia"])


def banded(nRow, nCol, offsets, seed):
    rng = np.random.default_rng(seed)
    r = np.repeat(np.arange(nRow), len(offsets))
    cc = r + np.tile(offsets, nRow)
    keep = (cc >= 0) & (cc < nCol)
    row, col = r[keep], cc[keep]
    val = rng.choice([-1.0, 1.0], len(row)) * rng.uniform(0.5, 2.0, len(row))
    return Case("banded%dx%d" % (nRow, nCol), nRow, nCol, row, col, val, rng.uniform(-1.0, 1.0, nCol))


@pytest.mark.gpu
def test_fp32_stencils_and_bands(sp, oracle):
    """lap2d5, lap3d7, box3d27 (5, 7, 27 diagonals: remainders 1, 3, 3 of DIA's unroll by 4) with random values, and
    rectangular banded matrices whose diagonals leave the matrix at both ends, through DIA, ELL and CRS."""
    rng = np.random.default_rng(11)
    cases = []
    for kind, n in (("lap2d5", 61), ("lap3d7", 17), ("box3d27", 11)):
        nr, nc, row, col, val = oracle.stencil(kind, n)
        val = rng.choice([-1.0, 1.0], len(val)) * rng.uniform(0.5, 2.0, len(val))
        cases.append(Case(kind, nr, nc, row, col, val, rng.uniform(-1.0, 1.0, nc)))
    offsets = np.array([-300, -17, -1, 0, 2, 5, 64, 1000])
    cases += [banded(2000, 1403, offsets, 12), banded(1201, 2500, offsets, 13)]
    for c in cases:
        check_paths(sp, c, [p for p in PATHS if p[0] in ("crs", "ell", "dia")])


def dynamic_case(seed):
    """Rows of products below 2^-126 (fp32 subnormals), rows like [2^24, 1, 1] whose fp32 and fp64 sums differ, rows of
    products that overflow fp32 while their sum fits, and ordinary rows.  Columns 0-15: x ~ 2^-70; 16-31: x = 1;
    32-47: x = 2^64; 48-63: x ~ U(-1, 1)."""
    rng = np.random.default_rng(seed)
    nCol = 64
    x = np.concatenate([rng.choice([-1.0, 1.0], 16) * rng.uniform(1, 2, 16) * 2.0 ** -70, np.ones(16),
                        np.full(16, 2.0 ** 64), rng.uniform(-1.0, 1.0, 16)])
    rows = []                                        # (columns, values, kind)
    for i in range(40):                              # subnormal products, and sums of them that become normal
        k = int(rng.integers(1, 13))
        rows.append((np.sort(rng.choice(16, k, replace=False)),
                     rng.choice([-1.0, 1.0], k) * rng.uniform(1, 2, k) * 2.0 ** (-70 + (i % 3) * 6), "sub"))
    designed = [[2.0 ** 24, 1.0, 1.0], [1.0, 2.0 ** 24, 1.0, 1.0, 1.0], [2.0 ** 25, 1.0, 1.0, 1.0], [-2.0 ** 24, -1.0, -1.0],
                [2.0 ** 24, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0, 1.0]]
    for v in designed:
        rows.append((16 + np.arange(len(v)), np.array(v), "diff"))
    big = 2.0 ** 64
    over = [[1.5 * big, -(1.5 * big - 2.0 ** 50)], [1.5 * big, -1.25 * big], [1.75 * big, 0.5, -1.5 * big, 1.0],
            [-1.5 * big, 1.5 * big - 2.0 ** 40, 3.0]]
    for v in over:
        rows.append((32 + np.arange(len(v)), np.array(v), "diff"))
    rows.append((np.array([32]), np.array([1.5 * big]), "over"))                 # overflows in both precisions
    for i in range(20):
        k = int(rng.integers(0, 9))
        rows.append((48 + np.sort(rng.choice(16, k, replace=False)), rng.uniform(-1.0, 1.0, k), "plain"))
    order = rng.permutation(len(rows))
    rows = [rows[i] for i in order]
    row = np.concatenate([np.full(len(cl), r) for r, (cl, _, _) in enumerate(rows)])
    col = np.concatenate([cl for cl, _, _ in rows])
    val = np.concatenate([v for _, v, _ in rows])
    c = Case("dynamic", len(rows), nCol, row, col, val, x)
    c.kind = np.array([k for _, _, k in rows])
    return c


@pytest.mark.gpu
def test_fp32_dynamic_range(sp):
    """Subnormal products come out as the reference's subnormals (an -ftz build flushes them); products that overflow fp32
    give the reference's inf / NaN at precision 1 and a finite, bit-exact sum at precision 2; on these rows and the
    [2^24, 1, 1] kind the two precisions differ, each matching its own reference."""
    c = dynamic_case(21)
    sub = c.kind == "sub"
    y1 = c.seq[1]
    assert np.any((y1[sub] != 0) & (np.abs(y1[sub]) < 2.0 ** -126)) and np.any(np.abs(y1[sub]) >= 2.0 ** -126)
    diff = c.kind == "diff"
    assert np.all(~same_bits(c.seq[1], c.seq[2])[diff])
    assert np.all(np.isfinite(c.seq[2][diff])) and np.any(np.isnan(c.seq[1][diff]))
    for fmt, opt in PATHS:
        ys = {}
        for prec in (1, 2):
            A, ys[prec] = run(sp, fmt, opt, prec, c)
            check(ys[prec], c, prec, exact_rows(fmt, A, c), (fmt, opt, prec))
            A.destroy()
        if fmt != "csr5":                            # precision 1 on overflowing products: order-dependent elsewhere
            assert np.all(~same_bits(ys[1], ys[2])[diff]), (fmt, opt)


@pytest.mark.gpu
def test_fp32_input_rounding(sp):
    """A diagonal matrix with x = 1: values halfway between fp32 neighbours (ties to even), in the fp32 subnormal range,
    halfway between subnormals, and below half the smallest subnormal.  Every path returns val.astype(np.float32)."""
    rng = np.random.default_rng(31)
    f = (rng.choice([-1.0, 1.0], 3000) * 10.0 ** rng.uniform(-30, 30, 3000)).astype(np.float32)
    mid = (f.astype(np.float64) + np.nextafter(f, np.float32(np.inf)).astype(np.float64)) / 2
    sub = rng.choice([-1.0, 1.0], 1000) * rng.uniform(2.0 ** -149, 2.0 ** -126, 1000)
    submid = (rng.integers(1, 1 << 23, 1000) + 0.5) * 2.0 ** -149
    tiny = rng.uniform(0.1, 0.49, 200) * 2.0 ** -149
    val = np.concatenate([mid, -mid[:500], sub, submid, tiny, [2.0 ** -150, 3 * 2.0 ** -150, 2.0 ** -126 * (1 - 2.0 ** -25)]])
    n = len(val)
    idx = np.arange(n)
    c = Case("diag", n, n, idx, idx, val, np.ones(n))
    a32 = val.astype(np.float32)
    assert np.any(a32[:3000] == f) and np.any(a32[:3000] != f)       # ties to even: both neighbours occur
    assert np.any((a32 != 0) & (np.abs(a32) < 2.0 ** -126)) and np.any(a32 == 0)
    for fmt, opt in PATHS:
        for prec in (1, 2):
            A, y = run(sp, fmt, opt, prec, c)
            assert np.array_equal(y, a32), (fmt, opt, prec, int((y != a32).sum()))
            check(y, c, prec, None, (fmt, opt, prec))
            A.destroy()


@pytest.mark.gpu
def test_fp32_guard_bands(sp, oracle):
    """x between NaN bands, y between canary bands (device_multiply) for every path and precision on the matrices of
    test_guard_bands_around_x_and_y."""
    rng = np.random.default_rng(41)
    mats = [("lap3d7", oracle.stencil("lap3d7", 13)), ("lap2d5", oracle.stencil("lap2d5", 37)),
            ("rmat", oracle.rmat(7, 10, 30000)), ("uniform", oracle.uniform(3, 3001, 2777, 9))]
    for name, (nr, nc, row, col, val) in mats:
        c = Case(name, nr, nc, row, col, val, rng.uniform(-1.0, 1.0, nc))
        check_paths(sp, c)


def capture_check(sp, A, c, x2, tag):
    """multiply_f32 of a fresh handle captured in a CUDA graph (its first launch inside the capture) on a side stream; x
    overwritten before the replay: the bits of an eager multiply with that x."""
    import torch
    xd = torch.from_numpy(c.x32).cuda()
    yg = torch.full((c.nRow,), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    graph, stream = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.graph(graph, stream=stream):
        A.multiply_f32(xd.data_ptr(), yg.data_ptr(), stream.cuda_stream)
    xd.copy_(torch.from_numpy(x2))
    graph.replay()
    torch.cuda.synchronize()
    ye = torch.full((c.nRow,), float("nan"), dtype=torch.float32, device="cuda")
    A.multiply_f32(xd.data_ptr(), ye.data_ptr())
    torch.cuda.synchronize()
    assert torch.equal(yg.view(torch.int32), ye.view(torch.int32)), tag


@pytest.mark.gpu
def test_fp32_graph_capture(sp, oracle, monkeypatch):
    """Every path, both precisions, and a row-blocked handle, captured before its first multiply."""
    rng = np.random.default_rng(51)
    nr, nc, row, col, val = oracle.rmat(7, 10, 30000)
    rm = Case("rmat", nr, nc, row, col, val, rng.uniform(-1.0, 1.0, nc))
    nr, nc, row, col, val = oracle.stencil("lap3d7", 13)
    st = Case("lap3d7", nr, nc, row, col, val, rng.uniform(-1.0, 1.0, nc))
    for fmt, opt in PATHS:
        for prec in (1, 2):
            for c in ((st,) if fmt == "dia" else (st, rm)):
                x2 = rng.uniform(-1.0, 1.0, c.nCol).astype(np.float32)
                A = convert(sp, fmt, opt, prec, c)
                capture_check(sp, A, c, x2, (fmt, opt, prec, c.name))
                A.destroy()
    monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(rm.row) // 5))
    A = convert(sp, "crs", {}, 2, rm)
    monkeypatch.delenv("B200SPMV_BLOCK_NNZ")
    assert A.scalar("row_blocks") >= 4
    capture_check(sp, A, rm, rng.uniform(-1.0, 1.0, rm.nCol).astype(np.float32), "blocked")
    A.destroy()


@pytest.mark.gpu
def test_fp32_row_blocks(sp, oracle, monkeypatch):
    """Row blocks (B200SPMV_BLOCK_NNZ) of every path at both precisions: the order-keeping rows carry the bits of the
    unblocked handle and of seq, the others lie within the bound."""
    rng = np.random.default_rng(61)
    cases = []
    for nr, nc, row, col, val in (oracle.stencil("lap3d7", 20), oracle.rmat(42, 11, 60000)):
        cases.append(Case("m%d" % nr, nr, nc, row, col, val, rng.uniform(-1.0, 1.0, nc)))
    for fmt, opt in PATHS:
        for c in cases[:1] if fmt == "dia" else cases:
            for prec in (1, 2):
                A, whole = run(sp, fmt, opt, prec, c)
                exact = exact_rows(fmt, A, c)
                A.destroy()
                monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(max(1000, len(c.row) // 5)))
                A, cut = run(sp, fmt, opt, prec, c)
                monkeypatch.delenv("B200SPMV_BLOCK_NNZ")
                assert A.scalar("row_blocks") >= 4, (fmt, opt)
                check(cut, c, prec, exact, (fmt, opt, prec, c.name, "blocked"))
                rows = np.ones(c.nRow, bool) if exact is None else exact
                assert np.all(same_bits(cut, whole)[rows]), (fmt, opt, prec, c.name)
                A.destroy()


@pytest.mark.gpu
def test_fp32_handles_have_no_row_ranges(sp, monkeypatch):
    """multiply_rows has no fp32-vector variant: every precision handle reports has_rows = 0, and multiply_rows on it is
    refused (-4, a call the handle's precision rules out; CSR5 has no row ranges at all, -3)."""
    import torch
    c = sorted_case("rows", [3, 0, 5, 70, 1] * 300, 500, 71)
    xd = torch.zeros(c.nCol, dtype=torch.float64, device="cuda")
    yd = torch.zeros(c.nRow, dtype=torch.float64, device="cuda")
    for blocked in (False, True):
        for fmt, opt in PATHS:
            for prec in (1, 2):
                if blocked:
                    monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(c.row) // 4))
                A = convert(sp, fmt, opt, prec, c)
                monkeypatch.delenv("B200SPMV_BLOCK_NNZ", raising=False)
                assert A.scalar("has_rows") == 0, (fmt, opt, prec, blocked)
                with pytest.raises(sp.B200SpmvError) as e:
                    A.multiply_rows(0, 10, xd.data_ptr(), yd.data_ptr())
                assert e.value.status == (-3 if fmt == "csr5" else -4), (fmt, opt, prec, blocked)
                A.destroy()
