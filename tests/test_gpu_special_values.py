"""Signed zeros, infinities and NaN through every kernel (include/b200spmv.h, Conventions; DESIGN.md 5b).

Stored-entry semantics (every format and path but those below): y_i depends only on the stored entries of row i and on
x at their columns.  Its IEEE class follows from the exact products p = a * x[c] of those entries: NaN if any p is NaN (a
NaN in x or A, a stored 0 times +-Inf) or if the row has both +Inf and -Inf products; else +-Inf if it has infinite
products of one sign; else finite, within n 2^-53 sum|p| of the exact sum (test_gpu_gather_bound.row_reference; fp32:
the bounds of test_gpu_fp32).  The class does not depend on the summation order while the finite part cannot overflow
(finite magnitudes here stay far below 1e300 / n), so it holds for the re-associating kernels too.  A row whose products
are all +-0 is +0.0, as the reference's sum from +0.0 gives: a -0.0 only comes out of a sum whose every term is -0.0.

Reference-padding semantics (DIA, SS and CSS with ss_faithful = 1): the reference's own operations, 0 * x over its
padding included; y equals the oracle bit for bit.  DIA's padding is every position of its diagonals inside the matrix,
so its class and its bits are those of the matrix with every such position stored (dia_expanded).

Bit claims compare uint64 / uint32 views, every NaN equal to every other NaN (payloads are not compared).

The special values sit where the kernels' units meet: x[0] (ragged ends of the entry streams, ELL's V rounding),
x[1..7] (ELL's K padding), x[nCol-1], the first column of every column block, columns no row stores; NaN / +-Inf / 0 in
A at the first and last entries of 128-, 512-, 1024- and 2048-entry tiles and in the pieces of rows that tiles carry;
stored zeros against x[0] = Inf; rows of -0.0 products (zero values, and -0.0 in x against positive values).  The last
row of a matrix keeps finite values, so that an x read by a ragged end shows there.
"""
import numpy as np
import pytest

from test_gpu_fp32 import bound as f32_bound, same_bits as same_bits32, seq as f32_seq, within as f32_within
from test_gpu_gather_bound import (BOUNDARY_LENS, FORMATS as WIDE_FORMATS, NCOL, assert_path, bulk_lens, exact_rows as
                                   wide_exact_rows, row_reference, wide_case)

G = 4096                                    # guard band, entries
CANARY = -12345.0
SPECIALS = (np.nan, np.inf, -np.inf)
TS_LONG, JDS_LONG = 64, 2048
FIN, PINF, NINF, NAN = 0, 1, 2, 3

# formats and options on the small matrices; faithful SS / CSS and DIA are compared with the oracle
NARROW = [("crs", {}), ("crs", {"crs_path": 1}), ("crs", {"crs_path": 4}), ("coo", {}), ("coo", {"coo_path": 1}),
          ("ell", {}), ("jds", {}), ("ss", {}), ("ss", {"segment_width": 4, "ss_faithful": 1}), ("css", {"n_block": 3}),
          ("css", {"segment_width": 4, "n_block": 3, "ss_faithful": 1}), ("csr5", {"csr5_sigma": 4}),
          ("csr5", {"csr5_sigma": 16}), ("csr5", {"csr5_sigma": 32}), ("hyb", {}), ("dia", {})]
ROW_FORMATS = ("crs", "ss", "css", "ell", "dia")
F32_FORMATS = ("crs", "ell", "dia", "csr5")


# ------------------------------------------------------------------------------------------ reference
def products(val, x, col):
    with np.errstate(all="ignore"):
        return val * x[col]


def classes(nRow, row, p):
    """IEEE class of each row's stored-entry sum: FIN, PINF, NINF or NAN."""
    cnt = lambda m: np.bincount(row, weights=m.astype(np.float64), minlength=nRow)[:nRow] > 0
    nan, pinf, ninf = cnt(np.isnan(p)), cnt(p == np.inf), cnt(p == -np.inf)
    cls = np.full(nRow, FIN)
    cls[ninf] = NINF
    cls[pinf] = PINF
    cls[nan | (pinf & ninf)] = NAN
    return cls


class Expect:
    """What y must be for one matrix and x: the class of every row, and the extended-precision sum and its bound for the
    finite rows.  prec = 1 / 2: fp32 values and vectors (a32, x32), the bounds of test_gpu_fp32."""

    def __init__(self, nRow, row, col, val, x, prec=0):
        self.nRow, self.prec = nRow, prec
        if prec:
            a, xv = val.astype(np.float32), x.astype(np.float32)
            p = products(a.astype(np.float64), xv.astype(np.float64), col)
        else:
            p = products(val, x, col)
        self.cls = classes(nRow, row, p)
        fin = np.isfinite(p)                        # the finite rows have finite products only
        if prec:
            a0 = np.where(fin, a, np.float32(0))
            x0 = np.where(np.isfinite(xv), xv, np.float32(0))
            self.ref, self.bound = f32_bound(prec, nRow, row, col, a0, x0)
        else:
            self.ref, self.bound = row_reference(nRow, row, np.where(fin, p, 0.0))


def class_errors(y, e):
    """Rows of y that break stored-entry semantics (boolean mask)."""
    with np.errstate(invalid="ignore"):
        ok = np.where(e.cls == NAN, np.isnan(y), False)
        ok |= (e.cls == PINF) & (y == np.inf)
        ok |= (e.cls == NINF) & (y == -np.inf)
        fin = (e.cls == FIN) & np.isfinite(y)
        val = np.abs(y.astype(np.longdouble) - e.ref) <= e.bound if not e.prec else f32_within(y, e.ref, e.bound)
        ok |= fin & val & ~((y == 0) & np.signbit(y))
    return ~ok


def assert_classes(y, e, tag, rows=None):
    bad = class_errors(y, e)
    if rows is not None:
        bad &= rows
    if np.any(bad):
        r = int(np.flatnonzero(bad)[0])
        raise AssertionError((tag, "rows off stored-entry semantics: %d, first %d: y %r, class %d" % (bad.sum(), r, y[r], e.cls[r])))


def same_bits(a, b):
    """Per row: the same bits (the sign of zero included), or NaN in both."""
    if a.dtype == np.float32:
        return same_bits32(a, b)
    na, nb = np.isnan(a), np.isnan(b)
    return (na & nb) | (~na & ~nb & (a.view(np.uint64) == b.view(np.uint64)))


def assert_bits(y, ref, tag, rows=None):
    ok = same_bits(y, ref)
    if rows is not None:
        ok |= ~rows
    assert np.all(ok), (tag, "rows off the claimed bits: %d, first %d" % ((~ok).sum(), int(np.flatnonzero(~ok)[0])))


def dia_expanded(nRow, nCol, row, col, val):
    """DIA's stored entries: every position of its diagonals inside the matrix, zeros where A has none (sorted)."""
    offs = np.unique(col.astype(np.int64) - row)
    r = np.concatenate([np.arange(max(0, -o), min(nRow, nCol - o)) for o in offs]) if len(offs) else np.zeros(0, np.int64)
    c = np.concatenate([np.arange(max(0, -o), min(nRow, nCol - o)) + o for o in offs]) if len(offs) else r
    o = np.lexsort((c, r))
    r, c = r[o], c[o]
    v = np.zeros(len(r))
    at = np.searchsorted(r * nCol + c, row.astype(np.int64) * nCol + col)
    v[at] = val
    return r.astype(np.int32), c.astype(np.int32), v


# ------------------------------------------------------------------------------------------ the checker itself (CPU)
def test_special_value_checker():
    """The class checker accepts every summation order of the same products and rejects: NaN in a row that stores no
    non-finite column, +Inf where the row holds both +-Inf products, -0.0 on a row of zero products, a finite value on
    a row with a NaN product, a dropped or duplicated finite product."""
    rng = np.random.default_rng(5)
    nCol = 40
    x = rng.uniform(-1, 1, nCol)
    x[[0, 1, 2, 3]] = [np.nan, np.inf, -np.inf, -0.0]
    rows = [[5, 6, 7], [1, 5, 9], [2, 9], [1, 2, 8], [0, 4], [3, 11, 12], [], [13, 14, 15, 16, 17], [1, 18], [19]]
    vals = [[1.0, -2.0, 3.0], [2.0, 1.0, 1.0], [1.0, 4.0], [1.0, 1.0, 1.0], [1.0, 1.0], [2.0, 0.0, 0.0], [],
            [1e3, -1e-3, 7.0, 1.0, -5.0], [0.0, 1.0], [np.nan]]
    x[11], x[12] = 0.5, -0.5
    vals[5] = [2.0, -0.0, 0.0]                               # 2 * -0.0, -0.0 * 0.5, 0.0 * -0.5: all -0.0
    row = np.concatenate([np.full(len(r), i) for i, r in enumerate(rows)]).astype(np.int32)
    col = np.concatenate([np.array(r, int) for r in rows]).astype(np.int32)
    val = np.concatenate([np.array(v, float) for v in vals])
    nRow = len(rows)
    e = Expect(nRow, row, col, val, x)
    assert e.cls.tolist() == [FIN, PINF, NINF, NAN, NAN, FIN, FIN, FIN, NAN, NAN]
    p = products(val, x, col)
    ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])])
    with np.errstate(all="ignore"):
        for trial in range(200):
            y = np.zeros(nRow)
            for r in range(nRow):
                q = p[ptr[r]:ptr[r + 1]][rng.permutation(ptr[r + 1] - ptr[r])]
                s = 0.0                                        # sequential from +0.0, or pairwise
                for v in q:
                    s = s + v
                y[r] = s if trial % 2 else (np.sum(q) if len(q) else 0.0)
            assert not np.any(class_errors(y, e)), trial
        good = np.array([np.sum(p[ptr[r]:ptr[r + 1]]) for r in range(nRow)]) + 0.0
    assert not np.any(class_errors(good, e))
    for r, bad in ((0, np.nan), (6, np.nan), (1, -np.inf), (3, np.inf), (3, 1.0), (5, -0.0), (6, -0.0), (4, 0.0),
                   (9, 0.0), (1, 1.0), (0, good[0] + p[0]), (0, good[0] - p[1]), (7, good[7] - 1e3)):
        y = good.copy()
        y[r] = bad
        assert class_errors(y, e)[r], (r, bad)
    # fp32: the same classes through a32, x32
    e32 = Expect(nRow, row, col, val, x, prec=2)
    assert e32.cls.tolist() == e.cls.tolist()
    y32 = f32_seq(2, nRow, row, col, val.astype(np.float32), x.astype(np.float32))
    assert not np.any(class_errors(y32, e32))
    y32[5] = np.float32(-0.0)
    assert class_errors(y32, e32)[5]
    # bits: NaN equals NaN whatever its payload, -0.0 is not +0.0
    a = np.array([np.nan, -0.0, 1.0])
    b = np.array([-np.nan, 0.0, 1.0])
    assert same_bits(a, b).tolist() == [True, False, True]
    assert same_bits(a.astype(np.float32), b.astype(np.float32)).tolist() == [True, False, True]
    # DIA's expansion stores every in-range position of its diagonals
    r2, c2, v2 = dia_expanded(3, 4, np.array([0, 2]), np.array([1, 1]), np.array([5.0, 6.0]))
    assert list(zip(r2.tolist(), c2.tolist(), v2.tolist())) == [(0, 1, 5.0), (1, 0, 0.0), (1, 2, 0.0), (2, 1, 6.0), (2, 3, 0.0)]


# ------------------------------------------------------------------------------------------ matrices and poison
class Case:
    """A sorted duplicate-free COO with poisoned values and two poisoned x: "edge" (x[0] = +Inf and nothing else) and
    "spread" (NaN / +-Inf at the columns listed in the module docstring)."""

    def __init__(self, name, nRow, nCol, row, col, val, seed, poison=True):
        rng = np.random.default_rng(seed)
        self.name, self.nRow, self.nCol = name, int(nRow), int(nCol)
        self.row, self.col = np.asarray(row, np.int32), np.asarray(col, np.int32)
        self.lens = np.bincount(self.row, minlength=self.nRow)[:self.nRow]
        self.ptr = np.concatenate([[0], np.cumsum(self.lens)])
        x = rng.uniform(-1.0, 1.0, self.nCol)
        x[rng.random(self.nCol) < 0.01] = -0.0
        self.val = np.array(val, np.float64)
        if poison:
            self.val = poison_values(self, rng, x)
        self.xs = {"edge": x.copy(), "spread": x.copy()}
        if self.nCol:
            self.xs["edge"][0] = np.inf
            self.xs["spread"][:] = spread_x(self, x, rng)

    def expect(self, kind, prec=0):
        key = (kind, prec)
        if not hasattr(self, "_e"):
            self._e = {}
        if key not in self._e:
            self._e[key] = Expect(self.nRow, self.row, self.col, self.val, self.xs[kind], prec)
        return self._e[key]

    def crs(self, oracle, kind):
        return oracle.crs_result(self.nRow, self.row, self.col, self.val, self.xs[kind])


def poison_values(c, rng, x):
    val = c.val.copy()
    nnz = len(val)
    if nnz == 0:
        return val
    stop = c.ptr[c.row[-1]]                          # the last row keeps finite values
    at = {0}
    for u in (128, 512, 1024, 2048):
        ks = list(range(1, min(nnz // u, 4) + 1)) + [nnz // u]
        at |= {k * u + d for k in ks for d in (-1, 0)}
    at = sorted(a for a in at if 0 <= a < stop)
    val[at] = np.resize(np.array(SPECIALS + (0.0,)), len(at))
    # rows through a 2048-entry tile edge: a special value only in the piece the next tile carries
    start, end = c.ptr[:-1], c.ptr[1:]
    multi = np.flatnonzero((c.lens > 0) & ((end - 1) // 2048 > start // 2048) & (end <= stop))
    for i, r in enumerate(multi[:3]):
        e = (start[r] // 2048 + 1) * 2048 + 3
        if e < end[r]:
            val[e] = SPECIALS[i % 3]
    # explicit zeros against x[0] (= +Inf in the "edge" x): 0 * Inf = NaN
    z = np.flatnonzero(c.col[:stop] == 0)
    val[z[::2]] = 0.0
    # rows of -0.0 products: zero values of the opposite sign to x, positive values against x = -0.0
    for r in np.flatnonzero(c.lens[:-1] > 0)[3::11]:
        b, e = c.ptr[r], c.ptr[r + 1]
        if not np.all(np.isfinite(val[b:e])):
            continue
        xc = x[c.col[b:e]]
        val[b:e] = np.where(xc == 0, np.abs(val[b:e]) + 1.0, np.copysign(0.0, -xc))
    return val


def spread_x(c, x, rng):
    x = x.copy()
    n = c.nCol
    hit = [0, n - 1] + list(range(1, min(8, n)))
    for nb in (2, 3):                                # column-block starts: the engine's and CSS's blocks
        B = -(-n // nb)
        hit += list(range(B, n, B))
    unused = np.setdiff1d(np.arange(n), c.col)
    if len(unused):
        hit += [int(unused[0]), int(unused[len(unused) // 2]), int(unused[-1])]
    if len(c.col):                                   # the column of the matrix's last entry
        hit.append(int(c.col[-1]))
    hit = sorted(set(h for h in hit if 0 <= h < n))
    x[hit] = np.resize(np.array(SPECIALS), len(hit))
    return x


def lens_case(name, lens, seed, nCol=None):
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, np.int64)
    nCol = nCol or max(4096, 2 * int(lens.max(initial=0)))
    row = np.repeat(np.arange(len(lens)), lens)
    col = np.concatenate([np.sort(rng.choice(nCol, int(k), replace=False)) for k in lens]) if len(row) else row
    val = rng.choice([-1.0, 1.0], len(row)) * 10.0 ** rng.uniform(-6, 6, len(row))
    return Case(name, len(lens), nCol, row, col, val, seed)


# ------------------------------------------------------------------------------------------ device helpers
@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


def handle(sp, fmt, opt, c, row=None, col=None, val=None):
    row = c.row if row is None else row
    col = c.col if col is None else col
    val = c.val if val is None else val
    return sp.SpMatOpt(fmt, **opt).convert_host(sp.SpMat(c.nRow, c.nCol, row, col, val))


def call(fn, x, ny, dtype=np.float64, lo=0, hi=None, misalign=False, tag=""):
    """fn(x_ptr, y_ptr) twice, x between NaN bands, y NaN-poisoned between canary bands: the second call runs over the
    first's y and must give its bits; rows outside [lo, hi) keep the poison.  misalign: x 8 bytes off 16-byte alignment."""
    import torch
    hi = ny if hi is None else hi
    td = torch.float64 if dtype == np.float64 else torch.float32
    isz = np.dtype(dtype).itemsize
    sh = 1 if misalign else 0
    xb = torch.full((len(x) + 2 * G + sh,), float("nan"), dtype=td, device="cuda")
    xb[G + sh:G + sh + len(x)] = torch.from_numpy(np.asarray(x, dtype)).cuda()
    yb = torch.full((ny + 2 * G,), CANARY, dtype=td, device="cuda")
    yb[G:G + ny] = float("nan")
    out = []
    for _ in range(2):
        fn(xb.data_ptr() + isz * (G + sh), yb.data_ptr() + isz * G)
        torch.cuda.synchronize()
        y = yb.cpu().numpy()
        assert np.all(y[:G] == CANARY) and np.all(y[G + ny:] == CANARY), (tag, "store outside y")
        out.append(y[G:G + ny].copy())
    assert_bits(out[1], out[0], (tag, "second call over the first's y"))
    assert np.all(np.isnan(out[0][:lo])) and np.all(np.isnan(out[0][hi:])), (tag, "store outside rows [%d,%d)" % (lo, hi))
    return out[0]


def host_calls(sp, A, x, ny, f32=False):
    """multiply_host{,_f32} with pageable and with page-locked vectors: both must give the same bits."""
    dt = np.float32 if f32 else np.float64
    xs, ys = [], []
    for pinned in (False, True):
        xh = np.asarray(x, dt).copy()
        yh = np.full(ny, np.nan, dt)
        if pinned and not (sp.host_register(xh) and (ny == 0 or sp.host_register(yh))):
            continue
        try:
            (A.multiply_host_f32 if f32 else A.multiply_host)(xh, yh)
        finally:
            if pinned:
                sp.host_unregister(xh)
                if ny:
                    sp.host_unregister(yh)
        ys.append(yh)
    assert len(ys) == 2
    assert_bits(ys[1], ys[0], "pinned and pageable")
    return ys[0]


def claimed_rows(fmt, opt, A, c):
    """Rows whose fp64 y the format claims bit-identical to the sequential CRS result (None = none)."""
    if fmt == "crs":
        k = A.scalar("crs_kernel")
        return np.ones(c.nRow, bool) if k == 1 else (c.lens <= TS_LONG) if k == 0 else None
    if fmt == "coo":
        return c.lens <= TS_LONG if A.scalar("coo_path") == 1 else None
    if fmt == "ell":
        return np.ones(c.nRow, bool)
    if fmt == "jds":
        return c.lens <= JDS_LONG
    if fmt == "hyb":
        return c.lens - A.scalar("K") <= TS_LONG
    return None


def faithful_reference(oracle, fmt, opt, c, x):
    if fmt == "dia":
        return oracle.dia_spmv(oracle.dia_convert(c.nRow, c.nCol, c.row, c.col, c.val), x)
    if fmt == "ss":
        return oracle.ss_spmv(oracle.ss_convert(c.nRow, c.row, c.col, c.val, opt["segment_width"]), x)
    return oracle.css_spmv(oracle.css_convert(c.nRow, c.nCol, c.row, c.col, c.val, opt["segment_width"], opt["n_block"]), x)


def dia_ok(c):
    return len(np.unique(c.col.astype(np.int64) - c.row)) * max(c.nRow, 1) <= 3e7


def check_y(oracle, fmt, opt, A, c, kind, y, tag, rows=None):
    """y of the fp64 multiply on rows (None = all): rule 1 or rule 2, and the bits the format claims."""
    x = c.xs[kind]
    if fmt == "dia" or opt.get("ss_faithful"):
        assert_bits(y, faithful_reference(oracle, fmt, opt, c, x), tag, rows)
        if fmt == "dia":
            r2, c2, v2 = dia_expanded(c.nRow, c.nCol, c.row, c.col, c.val)
            assert_classes(y, Expect(c.nRow, r2, c2, v2, x), tag, rows)
        return
    assert_classes(y, c.expect(kind), tag, rows)
    claim = claimed_rows(fmt, opt, A, c)
    if claim is not None:
        assert_bits(y, c.crs(oracle, kind), tag, claim if rows is None else claim & rows)


def cut_rows(c, kind):
    """Row-range cuts at a NaN row and the row after it, at a row of -0.0 products, and in the middle."""
    e = c.expect(kind)
    cuts = {0, c.nRow, c.nRow // 2}
    nan = np.flatnonzero(e.cls == NAN)
    if len(nan):
        r = int(nan[len(nan) // 2])
        cuts |= {r, r + 1}
    return sorted(cuts)


def run_f32(sp, oracle, fmt, opt, c, tag):
    """multiply_f32 and multiply_host_f32 at precision 1 and 2."""
    for prec in (1, 2):
        A = handle(sp, fmt, dict(opt, precision=prec), c)
        for kind in c.xs:
            x32 = c.xs[kind].astype(np.float32)
            y = call(A.multiply_f32, x32, c.nRow, np.float32, tag=(tag, prec, kind))
            assert_bits(host_calls(sp, A, x32, c.nRow, f32=True), y, (tag, prec, kind, "host"))
            if fmt == "dia":
                r2, c2, v2 = dia_expanded(c.nRow, c.nCol, c.row, c.col, c.val)
                e = Expect(c.nRow, r2, c2, v2, c.xs[kind], prec)
                seq = f32_seq(prec, c.nRow, r2, c2, v2.astype(np.float32), x32)
            else:
                e = c.expect(kind, prec)
                seq = f32_seq(prec, c.nRow, c.row, c.col, c.val.astype(np.float32), x32)
            assert_classes(y, e, (tag, prec, kind))
            exact = None
            if fmt in ("ell", "dia") or (fmt == "crs" and A.scalar("crs_kernel") == 1):
                exact = np.ones(c.nRow, bool)
            elif fmt == "crs":
                exact = c.lens <= TS_LONG
            if exact is not None:
                assert_bits(y, seq, (tag, prec, kind, "seq"), exact)
        A.destroy()


def multi_x(c, k, dtype=np.float64):
    """X[:, j] = the "edge" x scaled, with one more non-finite value per vector at a different stored column."""
    X = np.stack([c.xs["edge"] * (1.0 + 0.25 * j) for j in range(k)], 1)
    used = np.unique(c.col)
    for j in range(k):
        if len(used):
            X[int(used[(j * 7919 + len(used) // 3) % len(used)]), j] = SPECIALS[j % 3]
    return np.ascontiguousarray(X.astype(dtype))


def run_multi(sp, A, c, f32, tag, same_kernel):
    """multiply_multi{,_f32} at k = 3 and 8: column j has the classes of A X[:, j] (a NaN of X[:, j] reaches only Y[:, j])
    and, where the multi-vector kernel is the single multiply's, its bits."""
    import torch
    dt = np.float32 if f32 else np.float64
    td = torch.float32 if f32 else torch.float64
    for k in (3, 8):
        X = multi_x(c, k, dt)
        Xd = torch.from_numpy(X).cuda()
        Yd = torch.full((c.nRow, k), float("nan"), dtype=td, device="cuda")
        (A.multiply_multi_f32 if f32 else A.multiply_multi)(k, Xd.data_ptr(), k, Yd.data_ptr(), k)
        torch.cuda.synchronize()
        Y = Yd.cpu().numpy()
        for j in range(k):
            xj = np.ascontiguousarray(X[:, j])
            e = Expect(c.nRow, c.row, c.col, c.val, xj.astype(np.float64), A.scalar("precision") if f32 else 0)
            assert_classes(Y[:, j], e, (tag, k, j))
            if same_kernel:
                y1 = call(A.multiply_f32 if f32 else A.multiply, xj, c.nRow, dt, tag=(tag, k, j))
                assert_bits(Y[:, j], y1, (tag, k, j, "single multiply"))


def run_all(sp, oracle, fmt, opt, c, tag):
    """Every entry point of one handle on both poisoned x; returns the handle."""
    A = handle(sp, fmt, opt, c)
    for kind in c.xs:
        x = c.xs[kind]
        y = call(A.multiply, x, c.nRow, tag=(tag, kind), misalign=False)
        check_y(oracle, fmt, opt, A, c, kind, y, (tag, kind))
        assert_bits(host_calls(sp, A, x, c.nRow), y, (tag, kind, "host"))
        if fmt in ROW_FORMATS and A.scalar("has_rows"):
            cuts = cut_rows(c, kind)
            for a, b in zip(cuts[:-1], cuts[1:]):
                yr = call(lambda xp, yp: A.multiply_rows(a, b, xp, yp), x, c.nRow, lo=a, hi=b, tag=(tag, kind, a, b))
                assert_bits(yr[a:b], y[a:b], (tag, kind, a, b, "rows"))
    return A


# ------------------------------------------------------------------------------------------ tests
@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(BOUNDARY_LENS)))
def test_special_boundary_lens(sp, oracle, i):
    """The boundary row lengths at a narrow width (TMA-fed entry streams, tile-stream, CSR5, COO tile kernel, ELL, JDS,
    SS, CSS, HYB, faithful SS / CSS): every entry point on both poisoned x."""
    c = lens_case("lens%d" % i, BOUNDARY_LENS[i], 40 + i)
    for fmt, opt in NARROW:
        if fmt == "dia" and not dia_ok(c):
            continue
        tag = (c.name, fmt, opt)
        A = run_all(sp, oracle, fmt, opt, c, tag)
        if fmt == "crs":
            want = {1: 0, 4: 2}.get(opt.get("crs_path"), 1 if c.lens.max() <= 16 else 0)
            assert A.scalar("crs_kernel") == want, (tag, A.scalar("crs_kernel"))
            run_multi(sp, A, c, False, tag, same_kernel=want in (1, 2))
        if fmt == "coo":
            assert A.scalar("coo_path") == opt.get("coo_path", 0), tag
        A.destroy()
        if fmt in F32_FORMATS and not opt.get("crs_path") == 4:
            run_f32(sp, oracle, fmt, opt, c, tag)
    # the fp32 multi-vector forms: row-chunk stream or entry stream on val32
    for prec in (1, 2):
        A = handle(sp, "crs", {"precision": prec}, c)
        run_multi(sp, A, c, True, (c.name, "crs f32", prec), same_kernel=A.scalar("crs_kernel") == 1)
        A.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("lap2d5", 90), ("lap3d7", 22), ("box3d27", 13)])
def test_special_stencils(sp, oracle, monkeypatch, kind, n):
    """Stencils: the row-chunk stream under both feeds, DIA TMA-fed and direct (misaligned x), CSS blocks on the
    row-chunk stream, ELL, SS; multiply_rows, fp32 and the multi-vector row-chunk stream."""
    nr, nc, row, col, val = oracle.stencil(kind, n)
    c = Case(kind, nr, nc, row, col, val, seed=n)
    for feed in ("dict", "idx"):
        if feed == "idx":
            monkeypatch.setenv("B200SPMV_CS_FEED", "idx")
        A = run_all(sp, oracle, "crs", {}, c, (kind, feed))
        monkeypatch.delenv("B200SPMV_CS_FEED", raising=False)
        assert A.scalar("crs_kernel") == (1 if kind != "box3d27" else 0), (kind, A.scalar("crs_kernel"))
        if kind != "box3d27":
            assert A.scalar("chunk_feed") == (1 if feed == "dict" else 0), (kind, feed)
        run_multi(sp, A, c, False, (kind, feed), same_kernel=A.scalar("crs_kernel") == 1)
        A.destroy()
    for fmt, opt in (("dia", {}), ("css", {}), ("ss", {}), ("ell", {}), ("jds", {}), ("coo", {}), ("csr5", {}),
                     ("hyb", {}), ("ss", {"segment_width": 4, "ss_faithful": 1})):
        A = run_all(sp, oracle, fmt, opt, c, (kind, fmt, opt))
        if fmt == "dia":
            assert A.scalar("tma") == 1, kind
            for k in c.xs:                                        # misaligned x: the direct kernel
                y = call(A.multiply, c.xs[k], c.nRow, misalign=True, tag=(kind, "dia direct", k))
                check_y(oracle, fmt, opt, A, c, k, y, (kind, "dia direct", k))
        if fmt == "css" and kind != "box3d27":
            assert A.scalar("chunk_feed") == 1, kind              # blocks on the row-chunk stream
        A.destroy()
    for fmt in ("crs", "ell", "dia"):
        run_f32(sp, oracle, fmt, {}, c, (kind, fmt))


@pytest.mark.gpu
@pytest.mark.parametrize("width", ["A", "B"])
def test_special_wide(sp, oracle, width):
    """The gather-bound paths of test_gpu_gather_bound (load-fed entry streams, both column-block engines, CSS sliced-ELL
    and tile-stream blocks): one poisoned x per format, the kernel each case is meant to reach asserted."""
    reached = set()
    for name, lens, seed in (("lens0", BOUNDARY_LENS[0], 100), ("lens3", BOUNDARY_LENS[3], 103),     # engine 2, 1
                             ("k11", bulk_lens("k11", 7), 200), ("powerlaw", bulk_lens("powerlaw", 7), 202)):
        w = wide_case(name, lens, NCOL[width], seed)
        c = Case(name, w.nRow, w.nCol, w.row, w.col, w.val, seed)
        c.xs = {"spread": c.xs["spread"]}
        w.lens = c.lens
        for fmt, opt in WIDE_FORMATS:
            A = handle(sp, fmt, opt, c)
            assert_path(fmt, A, w, width, reached)
            y = call(A.multiply, c.xs["spread"], c.nRow, tag=(width, name, fmt))
            assert_classes(y, c.expect("spread"), (width, name, fmt))
            exact = wide_exact_rows(fmt, A, w)
            if exact is None:
                exact = claimed_rows(fmt, opt, A, c) if fmt in ("coo", "hyb") else None
            if exact is not None:
                assert_bits(y, c.crs(oracle, "spread"), (width, name, fmt), exact)
            A.destroy()
    if width == "B":
        assert reached >= {(f, e) for f in ("ell", "jds", "ss", "css") for e in (1, 2)}, sorted(reached)


@pytest.mark.gpu
@pytest.mark.parametrize("K,ragged", [(3, False), (3, True)])
def test_special_hyb_tails(sp, oracle, K, ragged):
    """HYB's COO tail at every kind of tile edge (test_gpu_hyb.EDGE_RUNS), poisoned."""
    from test_gpu_hyb import EDGE_RUNS, rows_to_coo, tail_layout
    rng = np.random.default_rng(300 + K + ragged)
    lens, _ = tail_layout(rng, K, EDGE_RUNS, ragged)
    row, col, val = rows_to_coo(rng, lens, 6000)
    c = Case("hyb K%d %s" % (K, ragged), len(lens), 6000, row, col, val, seed=K + 2 * ragged)
    A = handle(sp, "hyb", {"hyb_k": K}, c)
    assert A.scalar("K") == K
    for kind in c.xs:
        y = call(A.multiply, c.xs[kind], c.nRow, tag=(c.name, kind))
        check_y(oracle, "hyb", {}, A, c, kind, y, (c.name, kind))
    A.destroy()


@pytest.mark.gpu
def test_special_empty(sp, oracle):
    """An empty matrix and one whose last rows are empty: those rows are +0.0 whatever x holds."""
    e = Case("empty", 77, 50, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0), seed=1)
    t = lens_case("trailing empty", [3, 0, 5, 1, 2] + [0] * 40, 2, nCol=64)
    for c in (e, t):
        c.xs["nan"] = np.full(c.nCol, np.nan)
        for fmt, opt in NARROW:
            A = run_all(sp, oracle, fmt, opt, c, (c.name, fmt, opt))
            A.destroy()
            if fmt in F32_FORMATS:
                run_f32(sp, oracle, fmt, opt, c, (c.name, fmt, opt))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,opt", __import__("test_gpu_transpose").OPTION_SETS)
def test_special_transpose(sp, oracle, fmt, opt):
    """multiply_transpose{,_f32}: A^T x has the classes of A^T's stored entries and the bits of a handle converted from
    the transposed triplets."""
    prec = opt.get("precision", 0)
    dt = np.float32 if prec else np.float64
    # the second: 5000 single entries over 20 columns, so that A^T has 20 rows of about 250 entries
    for c in (lens_case("lens0", BOUNDARY_LENS[0], 60, nCol=8000), lens_case("lens1", BOUNDARY_LENS[1], 61, nCol=20)):
        o = np.lexsort((c.row, c.col))
        cT = Case(c.name + "^T", c.nCol, c.nRow, c.col[o], c.row[o], c.val[o], seed=62, poison=False)
        if fmt == "dia" and not dia_ok(cT):
            continue
        if fmt == "ell" and cT.lens.max(initial=0) > cT.nCol:
            continue
        T = handle(sp, fmt, dict(opt, transpose=1), c)
        B = handle(sp, fmt, opt, cT)
        for kind in cT.xs:
            u = cT.xs[kind].astype(dt)
            yT = call(T.multiply_transpose_f32 if prec else T.multiply_transpose, u, cT.nRow, dt, tag=(fmt, opt, kind))
            yB = call(B.multiply_f32 if prec else B.multiply, u, cT.nRow, dt, tag=(fmt, opt, kind))
            assert_bits(yT, yB, (fmt, opt, c.name, kind, "A^T x"))
            if fmt == "dia":
                r2, c2, v2 = dia_expanded(cT.nRow, cT.nCol, cT.row, cT.col, cT.val)
                e = Expect(cT.nRow, r2, c2, v2, cT.xs[kind], prec)
            elif opt.get("ss_faithful"):
                continue
            else:
                v = cT.val.astype(np.float32).astype(np.float64) if opt.get("value_f32") else cT.val
                e = Expect(cT.nRow, cT.row, cT.col, v, cT.xs[kind], prec)
            assert_classes(yT, e, (fmt, opt, c.name, kind))
        T.destroy()
        B.destroy()


@pytest.mark.gpu
def test_special_row_blocks(sp, oracle, monkeypatch):
    """Row blocks (B200SPMV_BLOCK_NNZ) at every precision: each block is an ordinary matrix with its own ragged end."""
    c = lens_case("lens0", BOUNDARY_LENS[0], 70)
    for fmt, opt in (("crs", {}), ("coo", {}), ("crs", {"precision": 1}), ("crs", {"precision": 2})):
        monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(c.row) // 5 + 3))
        A = handle(sp, fmt, opt, c)
        monkeypatch.delenv("B200SPMV_BLOCK_NNZ")
        assert A.scalar("row_blocks") >= 4, (fmt, opt)
        prec = opt.get("precision", 0)
        for kind in c.xs:
            if prec:
                y = call(A.multiply_f32, c.xs[kind].astype(np.float32), c.nRow, np.float32, tag=(fmt, opt, kind))
            else:
                y = call(A.multiply, c.xs[kind], c.nRow, tag=(fmt, opt, kind))
            assert_classes(y, c.expect(kind, prec), (fmt, opt, kind))
        A.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["crs", "ell", "jds"])
def test_special_multi_gpu(sp, oracle, fmt):
    """b200spmv_mg_*: NaN / +-Inf at halo columns (the first and last columns of every GPU's row range) reach only the
    rows that store them, on as many GPUs as the box has (up to 8)."""
    from singlespmv_b200.mg import MgSpMat
    from test_gpu_parity import _mg_counts
    nr, nc, row, col, val = oracle.stencil("lap3d7", 30)
    c = Case("lap3d7", nr, nc, row, col, val, seed=9)
    for g in _mg_counts(sp):
        M = MgSpMat(g, fmt).convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))
        b = M.bounds()
        x = c.xs["edge"].copy()
        for i, r in enumerate(b[1:-1]):                          # the columns just across every split
            x[[r - 1, min(r + 900, c.nCol - 1)]] = SPECIALS[i % 3]
        y = np.full(c.nRow, np.nan)
        M.multiply_host(x, y)
        assert_classes(y, Expect(c.nRow, c.row, c.col, c.val, x), (fmt, g))
        assert_bits(y, oracle.crs_result(c.nRow, c.row, c.col, c.val, x), (fmt, g))
        M.destroy()
