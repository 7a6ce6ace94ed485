"""HYB (hyb.cu): an ELL part of width K plus a COO tail, against a host oracle of the same split.

Conversion.  K is the largest width k that at least need = min(nRow, max(4096, nRow / 3)) rows fill, counted in a
histogram of row lengths capped at 4096; K = 1 when no width qualifies; options.hyb_k > 0 is taken as the width, clamped
to the longest row.  The first K entries of every row go into an ELL part (exported as [nRow][K] with the reference's
padding rule, so oracle.ell_convert of the head triplets gives the expected arrays), the rest into a COO tail sorted by
(row, col).

Multiply.  The ELL kernel writes y, then the COO tile kernel in its accumulate mode (coo.cu coo_accumulate) continues
every row's sum with its tail entries.  The tail stream is cut into tiles of 2048 entries.  A run of one row's tail
entries that crosses a tile edge is either left entirely to the fix-up kernel, which recomputes it from the untouched
y[r] (at most 64 entries in all), or added piece by piece, the fix-up adding the carries of the later tiles (longer
runs).  The tile kernel decides by a look-ahead 64 entries past the run start, the fix-up by walking 64 entries either
way from the tile start: the two must agree for every split, or a piece is lost or added twice.

y is checked against the extended-precision row sum and its bound n 2^-53 sum|p| of test_gpu_gather_bound: every row
within the bound, rows whose tail has at most 64 entries (a row of at most K + 64 entries) bit-identical to the
sequential CRS result, empty rows +0.0, nothing stored outside y, the same bits when y already holds the result.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import skewed_matrix
from test_gpu_gather_bound import G, Guarded, assert_rows, capture_check, row_reference

HIST_CAP = 4096           # hyb.cu: the row-length histogram is capped here, and so is K
TILE = 2048               # coo.cu COO_TILE: entries of the tail per tile
LONG = 64                 # coo.cu COO_LONG: longer runs are reduced by a warp; shorter ones crossing an edge are recomputed


# ------------------------------------------------------------------------------------------ host oracle
def hyb_width(lens, k_opt):
    """K as HybFormat::convert chooses it from the row lengths."""
    lens = np.asarray(lens, np.int64)
    nRow = len(lens)
    max_len = int(lens.max()) if nRow else 0
    if k_opt > 0:
        return min(k_opt, max_len)
    if nRow == 0 or max_len == 0:
        return 0
    cap = min(max_len, HIST_CAP)
    hist = np.bincount(np.minimum(lens, cap), minlength=cap + 1)
    rows_with = np.cumsum(hist[::-1])[::-1]                     # rows_with[k] = rows of at least k entries (capped)
    need = min(nRow, max(HIST_CAP, nRow // 3))
    fill = np.flatnonzero(rows_with[1:] >= need)
    return int(fill[-1]) + 1 if len(fill) else 1


def hyb_split(nRow, row, col, val, k_opt):
    """(K, head, tail): head = the first K entries of every row, tail = the rest, both as (row, col, val) in (row, col)
    order."""
    row, col, val = np.asarray(row, np.int32), np.asarray(col, np.int32), np.asarray(val, np.float64)
    lens = np.bincount(row, minlength=nRow)[:nRow]
    K = hyb_width(lens, k_opt)
    ptr = np.concatenate([[0], np.cumsum(lens)])
    in_head = np.arange(len(row)) - ptr[row] < K
    return K, (row[in_head], col[in_head], val[in_head]), (row[~in_head], col[~in_head], val[~in_head])


def ell_slots(nRow, head_lens, K):
    """Stored slots of the sliced ELL part (ell.cu): slices of 32 rows, slice-local width rounded up to V slots."""
    V = 4 if K % 4 == 0 or K >= 32 else 2
    nsl = -(-nRow // 32)
    pad = np.zeros(nsl * 32, np.int64)
    pad[:nRow] = head_lens
    return int((-(-pad.reshape(nsl, 32).max(axis=1) // V)).sum()) * 32 * V


class Case:
    def __init__(self, name, nRow, nCol, row, col, val, x, oracle):
        self.name, self.nRow, self.nCol = name, int(nRow), int(nCol)
        self.row, self.col = np.ascontiguousarray(row, np.int32), np.ascontiguousarray(col, np.int32)
        self.val, self.x = np.ascontiguousarray(val, np.float64), np.ascontiguousarray(x, np.float64)
        self.lens = np.bincount(self.row, minlength=self.nRow)[:self.nRow]
        self.ref, self.bound = row_reference(self.nRow, self.row, self.val * self.x[self.col])
        self.y_crs = oracle.crs_result(self.nRow, self.row, self.col, self.val, self.x)


def random_values(rng, n):
    return rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-6, 6, n)


def rows_to_coo(rng, lens, nCol):
    """Sorted duplicate-free COO: row i takes lens[i] distinct columns drawn uniformly from [0, nCol).  Values of random
    sign with magnitudes 10^U(-6,6)."""
    lens = np.asarray(lens, np.int64)
    ptr = np.concatenate([[0], np.cumsum(lens)])
    row = np.repeat(np.arange(len(lens), dtype=np.int64), lens)
    col = rng.integers(0, nCol, len(row))
    for r in np.flatnonzero(lens > nCol // 8):                          # dense rows: a permutation each
        col[ptr[r]:ptr[r + 1]] = rng.permutation(nCol)[:lens[r]]
    while True:                                                         # sparse rows: redraw duplicates
        key = np.sort(row * nCol + col)
        col = key - row * nCol
        dup = np.flatnonzero(key[1:] == key[:-1]) + 1
        if not len(dup):
            break
        col[dup] = rng.integers(0, nCol, len(dup))
    return row.astype(np.int32), col.astype(np.int32), random_values(rng, len(row))


# ------------------------------------------------------------------------------------------ CPU: the oracle and the options
def test_hyb_split_by_hand():
    """The width rule on hand-worked row lengths, and one split written out."""
    # nRow < 4096: need = nRow, so K = the shortest row, or 1 when a row is empty
    assert hyb_width([3, 5, 2, 7], 0) == 2
    assert hyb_width([3, 0, 5, 2], 0) == 1
    assert hyb_width([9, 9, 0], 0) == 1
    # nRow >= 4096: need = max(4096, nRow / 3)
    assert hyb_width([5] * 4096 + [1] * 4904, 0) == 5                  # 9000 rows: 4096 binds
    assert hyb_width([5] * 4095 + [1] * 4905, 0) == 1
    assert hyb_width([8] * 4999 + [6] + [2] * 10000, 0) == 6           # 15000 rows: nRow / 3 = 5000 binds (4096 would give 8)
    assert hyb_width([8] * 5000 + [2] * 10001, 0) == 8                 # 15001 rows: need 5000
    assert hyb_width([8] * 5000 + [2] * 10003, 0) == 2                 # 15003 rows: need 5001
    # rows longer than 4096 count as 4096 long: K stops at the cap
    assert hyb_width([5000] * 4100, 0) == 4096
    assert hyb_width([4097] * 4096 + [0] * 4, 0) == 4096
    assert hyb_width([4095] * 4096 + [9000] * 4, 0) == 4095
    # hyb_k > 0: that width, clamped to the longest row
    assert hyb_width([3, 5, 2], 3) == 3 and hyb_width([3, 5, 2], 9) == 5 and hyb_width([3, 5, 2], 1) == 1
    assert hyb_width([0, 0], 4) == 0 and hyb_width([0, 0], 0) == 0 and hyb_width([], 0) == 0
    # a split with K = 2 (four rows, one empty)
    row = [0, 0, 0, 1, 3, 3, 3, 3]
    col = [1, 4, 6, 2, 0, 1, 2, 5]
    val = [1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0, 8.0]
    K, head, tail = hyb_split(4, row, col, val, 0)
    assert K == 1                                                       # row 2 is empty: no width fills all four rows
    K, head, tail = hyb_split(4, row, col, val, 2)
    assert K == 2
    assert [list(a) for a in head] == [[0, 0, 1, 3, 3], [1, 4, 2, 0, 1], [1.0, 2.0, 4.0, 5.0, 6.0]]
    assert [list(a) for a in tail] == [[0, 3, 3], [6, 2, 5], [3.0, 7.0, 8.0]]


def test_recommend_hyb_branch_edges():
    """b200spmv_recommend_format at the edges of its HYB branch (0.5 < ELL fill < 0.9 and CV <= 0.5), from hand-made
    statistics that keep clear of the DIA, CSR5 and CSS rules (many diagonals, x of 8 KB)."""
    import singlespmv_b200 as sp
    from singlespmv_b200._lib import Options, Stats, lib

    def rec(nnz, rowMax, rowMean, rowVar, nRow=1000):
        st = Stats()
        st.nRow, st.nCol, st.nnz, st.rowMax, st.rowMin = nRow, 1000, nnz, rowMax, 1
        st.rowMean, st.rowVar, st.nDiag = rowMean, rowVar, 1999
        f = lib.b200spmv_recommend_format(C.byref(st), C.byref(Options()))
        return [k for k, v in sp.FORMATS.items() if v == f][0]
    assert rec(9000, 10, 9.0, 0.25) == "ell"                           # ELL fill exactly 0.9
    assert rec(8999, 10, 8.999, 0.25) == "hyb"                         # just below 0.9
    assert rec(5001, 10, 5.001, 0.25) == "hyb"                         # just above 0.5
    assert rec(5000, 10, 5.0, 0.25) == "crs"                           # exactly 0.5
    assert rec(8000, 12, 8.0, 16.0) == "hyb"                           # CV = sqrt(16) / 8 = 0.5 exactly
    assert rec(8000, 12, 8.0, 16.0001) == "crs"                        # CV just above 0.5
    assert rec(8000, 12, 8.0, 4.0) == "hyb"


def test_create_rejects_negative_hyb_k():
    """A negative hyb_k is refused at create instead of being taken as the width rule."""
    import singlespmv_b200 as sp
    for k in (-1, -4096):
        with pytest.raises(sp.B200SpmvError) as e:
            sp.SpMatOpt("hyb", hyb_k=k)
        assert e.value.status == -1 and "hyb_k" in str(e.value)
    for k in (0, 1, 1 << 20):
        sp.SpMatOpt("hyb", hyb_k=k).destroy()


# ------------------------------------------------------------------------------------------ device helpers
@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


def convert(sp, c, k_opt):
    return sp.SpMatOpt("hyb", hyb_k=k_opt).convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))


def multiply_checked(A, c, tag):
    """y over a NaN-poisoned y between canary bands, then a second multiply over that result: the same bits."""
    g = Guarded(c.x, c.nRow)
    g.yb[G:G + c.nRow] = float("nan")
    A.multiply(g.xp, g.yp)
    y = g.y(tag=tag).copy()
    A.multiply(g.xp, g.yp)
    assert np.array_equal(g.y(tag=tag), y), (tag, "a second multiply changed y")
    return y


def check_hyb(sp, oracle, A, c, k_opt, tag, arrays=True):
    """Structure and exports against hyb_split, y against the row reference; returns y."""
    K, head, tail = hyb_split(c.nRow, c.row, c.col, c.val, k_opt)
    assert A.scalar("K") == K and A.scalar("tail_nnz") == len(tail[0]), (tag, A.scalar("K"), K)
    head_lens = np.bincount(head[0], minlength=c.nRow)[:c.nRow]
    slots = ell_slots(c.nRow, head_lens, K)
    alg = 12 * slots + 8 * (-(-c.nRow // 32) + 1) + 16 * len(tail[0]) + 8 * c.nCol + 8 * c.nRow
    assert A.scalar("alg_bytes") == alg, tag
    if arrays:
        m = oracle.ell_convert(c.nRow, *head)
        assert m["K"] == K, tag                                          # the longest head is K long
        assert np.array_equal(A.array("ell_col_idx", np.int32), m["col_idx"].ravel()), tag
        assert np.array_equal(A.array("ell_val", np.float64), m["val"].ravel()), tag
        for name, want, dt in (("coo_row_idx", tail[0], np.int32), ("coo_col_idx", tail[1], np.int32),
                               ("coo_val", tail[2], np.float64)):
            assert np.array_equal(A.array(name, dt), want), (tag, name)
    y = multiply_checked(A, c, tag)
    assert_rows(y, c, tag, exact=c.lens <= K + LONG)
    return y


def shared_cases(oracle):
    from test_gpu_parity import cases
    out = [Case(*t, oracle=oracle) for t in cases(oracle)]
    rng = np.random.default_rng(23)
    for kind, n in (("lap3d7", 13), ("box3d27", 9)):
        nr, nc, row, col, val = oracle.stencil(kind, n)
        out.append(Case("%s_%d" % (kind, n), nr, nc, row, col, val, rng.uniform(-1, 1, nc), oracle))
    # 13000 rows: nRow / 3 binds the width rule; 5 % of the rows 1350 long, 20 % empty
    row, col, val = skewed_matrix(rng, 13000, 1500, 10)
    out.append(Case("skew13000", 13000, 1500, row, col, val, rng.uniform(-1, 1, 1500), oracle))
    # uniform rows of 8 with a 10 % minority of 30
    lens = np.where(rng.random(6000) < 0.1, 30, 8)
    row, col, val = rows_to_coo(rng, lens, 5000)
    out.append(Case("uniform8_10pc30", 6000, 5000, row, col, val, rng.uniform(-1, 1, 5000), oracle))
    return out


# ------------------------------------------------------------------------------------------ tests
@pytest.mark.gpu
def test_hyb(sp, oracle):
    """Every shared case with hyb_k in {0 (the width rule), 1, 3, the longest row, above it}: K, tail_nnz, the five
    exported arrays and alg_bytes as the oracle splits, y within the bound, rows of at most K + 64 entries bit-identical
    to the CRS result, empty rows +0.0, idempotent on a poisoned y."""
    reached = set()
    for c in shared_cases(oracle):
        longest = int(c.lens.max()) if c.nRow else 0
        for k in sorted({0, 1, 3, longest, longest + 5}):
            A = convert(sp, c, k)
            check_hyb(sp, oracle, A, c, k, (c.name, k))
            if k == 0:                                                  # (K = 1 fallback, nRow / 3 binds)
                reached.add((A.scalar("K") == 1 and c.lens.min() == 0, c.nRow // 3 > HIST_CAP))
            A.destroy()
    # the width rule met the K = 1 fallback, a shortest-row K, and a case where nRow / 3 binds
    assert {(True, False), (False, False), (False, True)} <= reached, sorted(reached)


def tail_layout(rng, K, runs, ragged):
    """Row lengths for hyb_k = K whose tails meet the tile edges as asked.  runs: (L, a) = one row with a tail of L
    entries, a of them in front of a tile edge (a = 0: the tail starts on an edge; a = L: it ends on one).  Filler rows
    with tails of 1..40 entries move each run into place; an empty row and a row without a tail sit in front of every
    run.  ragged: the tail ends inside a tile, else on a tile edge.  Returns (lens, run_rows)."""
    lens, run_rows, pos = [], [], 0

    def fill(gap):
        nonlocal pos
        while gap > 0:
            t = min(gap, int(rng.integers(1, 41)))
            lens.append(K + t)
            gap -= t
            pos += t
    for L, a in runs:
        start = -(-(pos + a) // TILE) * TILE - a                      # first start at or after pos with a entries before an edge
        fill(start - pos)
        lens += [0, int(rng.integers(1, K + 1))]
        run_rows.append(len(lens))
        lens.append(K + L)
        pos += L
    if ragged:
        fill((TILE // 2 + 17 - pos) % TILE)
        assert pos % TILE != 0
    else:
        fill(-pos % TILE)
        assert pos % TILE == 0
    lens += [0, K]
    return np.array(lens, np.int64), run_rows


EDGE_RUNS = [(64, 1), (64, 63), (64, 32), (2, 1), (40, 40), (11, 1), (11, 10),          # at most 64 in all: fix-up recomputes
             (65, 1), (65, 64), (65, 33),                                                # exactly 65: pieces and carries
             (200, 10), (500, 64), (500, 65), (300, 100),                               # short piece (probe) / long piece before the edge
             (100, 0), (30, 0), (2048, 0), (4096, 0),                                    # starting on a tile start
             (2048 + 500, 300), (2 * 2048 + 400, 100), (2048 + 100, 0), (2 * 2048 + 50, 0)]   # through one / two whole tiles
CANCEL = (2048 + 1000, 500)                                                              # 500 | 2048 | 452: across two edges


@pytest.mark.parametrize("K,ragged", [(3, False), (3, True), (1, True)])
@pytest.mark.gpu
def test_hyb_tail_tile_edges(sp, oracle, K, ragged):
    """The accumulate mode of the COO tile kernel at every kind of tile edge (EDGE_RUNS), with rows without a tail and
    empty rows between the runs, a tail that fills its last tile or ends inside it, and one row whose tail cancels across
    two edges (a piece lost or added twice leaves the bound by far)."""
    rng = np.random.default_rng(100 + 10 * K + ragged)
    lens, run_rows = tail_layout(rng, K, EDGE_RUNS + [CANCEL], ragged)
    nRow, nCol = len(lens), 6000
    row, col, val = rows_to_coo(rng, lens, nCol)
    x = rng.uniform(-1.0, 1.0, nCol)
    # the cancelling row: its products are q, then -q in reverse (rounded through x), and 1 if the row is odd, so the
    # row sums to almost nothing while each of its pieces does not
    r = run_rows[-1]
    b, n = int(np.searchsorted(row, r)), int(lens[r])
    q = 10.0 ** rng.uniform(0, 3, n // 2)
    val[b:b + n] = np.concatenate([q, -q[::-1], np.ones(n % 2)]) / x[col[b:b + n]]
    c = Case("edges_K%d_%s" % (K, "ragged" if ragged else "full"), nRow, nCol, row, col, val, x, oracle)
    assert abs(float(c.ref[r])) < 1e-3 * float(q.sum())
    # the layout is what the runs ask for
    Kh, _, tail = hyb_split(nRow, row, col, val, K)
    assert Kh == K
    tptr = np.concatenate([[0], np.cumsum(np.maximum(lens - K, 0))])
    for rr, (L, a) in zip(run_rows, EDGE_RUNS + [CANCEL]):
        assert lens[rr] - K == L and (tptr[rr] + a) % TILE == 0, (rr, L, a)
    assert (len(tail[0]) % TILE != 0) == ragged
    A = convert(sp, c, K)
    check_hyb(sp, oracle, A, c, K, c.name)
    A.destroy()


@pytest.mark.gpu
def test_hyb_width_rule_and_recommendation(sp, oracle):
    """2e5 rows of 8 uniform random columns, 10 % of them 14 long, uploaded as a device COO: analyze + recommend pick
    HYB, its width rule picks K = 8 (every row fills 8, only 10 % fill 9), y has the CRS bits on every row.  Then the
    4096 cap on the device: 4100 rows of 4100 columns give K = 4096 and a tail of 4 entries per row."""
    rng = np.random.default_rng(5)
    nRow = 200000
    lens = np.where(rng.random(nRow) < 0.1, 14, 8)
    row, col, val = rows_to_coo(rng, lens, nRow)
    c = Case("uniform8_14", nRow, nRow, row, col, val, rng.uniform(-1, 1, nRow), oracle)
    d = sp.DeviceCoo.from_host_rows(sp.SpMat(nRow, nRow, row, col, val), 0, nRow)
    fmt, opts = d.recommend()
    assert fmt == "hyb", (fmt, opts, d.analyze()[0])
    A = sp.SpMatOpt(fmt, **opts).convert_device(d)
    assert A.scalar("K") == 8
    y = check_hyb(sp, oracle, A, c, 0, c.name, arrays=False)
    assert np.array_equal(y, c.y_crs)
    A.destroy()
    d.free()
    n, nCol = 4100, 8192
    row, col, val = rows_to_coo(rng, [n] * n, nCol)
    c = Case("cap", n, nCol, row, col, val, rng.uniform(-1, 1, nCol), oracle)
    A = convert(sp, c, 0)
    assert A.scalar("K") == HIST_CAP and A.scalar("tail_nnz") == 4 * n
    y = check_hyb(sp, oracle, A, c, 0, c.name, arrays=False)
    assert np.array_equal(y, c.y_crs)
    A.destroy()


def multi_tile_case(oracle, seed, nRow, long_tail):
    """Rows of 8 with a 10 % minority of 8 + 300 and one row of 8 + long_tail: the width rule keeps K = 8, and the
    tail runs through many tiles."""
    rng = np.random.default_rng(seed)
    lens = np.where(rng.random(nRow) < 0.1, 308, 8)
    lens[nRow // 2] = 8 + long_tail
    nCol = max(4000, 8 + long_tail)
    row, col, val = rows_to_coo(rng, lens, nCol)
    return Case("multi_tile_%d" % seed, nRow, nCol, row, col, val, rng.uniform(-1, 1, nCol), oracle)


@pytest.mark.gpu
def test_hyb_graph_capture(sp, oracle):
    """multiply captured in a CUDA graph on a side stream, x overwritten before the replay: the bits of an eager multiply
    with the new x.  The tail spans dozens of tiles."""
    c = multi_tile_case(oracle, 31, 5000, 5000)
    A = convert(sp, c, 0)
    assert A.scalar("K") == 8 and A.scalar("tail_nnz") > 20 * TILE
    x2 = np.random.default_rng(32).uniform(-1, 1, c.nCol)
    capture_check(sp, A, "hyb", c.nRow, c.x, x2, [0, c.nRow], "hyb capture")
    A.destroy()


@pytest.mark.gpu
def test_hyb_reconversion(sp, oracle):
    """One handle converted twice: a tail of many tiles then one inside a single tile, and the other way round.  K, the
    tail, its export and y are those of a fresh handle of the second matrix."""
    big = multi_tile_case(oracle, 41, 5000, 7000)
    rng = np.random.default_rng(42)
    lens = np.where(rng.random(700) < 0.05, 20, 4)
    row, col, val = rows_to_coo(rng, lens, 900)
    small = Case("one_tile", 700, 900, row, col, val, rng.uniform(-1, 1, 900), oracle)
    assert len(hyb_split(small.nRow, small.row, small.col, small.val, 0)[2][0]) < TILE
    for first, second in ((big, small), (small, big)):
        A = convert(sp, first, 0)
        multiply_checked(A, first, first.name)
        A.convert_host(sp.SpMat(second.nRow, second.nCol, second.row, second.col, second.val))
        fresh = convert(sp, second, 0)
        tag = (first.name, second.name)
        for s in ("K", "tail_nnz", "alg_bytes", "nRow", "nCol", "nNnz"):
            assert A.scalar(s) == fresh.scalar(s), (tag, s)
        for name, dt in (("coo_row_idx", np.int32), ("coo_col_idx", np.int32), ("coo_val", np.float64),
                         ("ell_col_idx", np.int32), ("ell_val", np.float64)):
            assert np.array_equal(A.array(name, dt), fresh.array(name, dt)), (tag, name)
        y = check_hyb(sp, oracle, A, second, 0, tag, arrays=False)
        assert np.array_equal(y, multiply_checked(fresh, second, tag)), tag
        A.destroy()
        fresh.destroy()


@pytest.mark.gpu
def test_hyb_rmat_scale(sp, oracle):
    """R-MAT of scale 20 with 2^24 draws from the device generator: the tail holds rows that run through many tiles.
    K and tail_nnz as the oracle splits, every row within the bound, rows of at most K + 64 entries bit-exact."""
    d = sp.DeviceCoo("rmat", 20, 1 << 24, 42)
    nRow, nCol, row, col, val = d.to_host()
    x = np.random.default_rng(43).uniform(-1, 1, nCol)
    c = Case("rmat_s20", nRow, nCol, row, col, val, x, oracle)
    K, _, tail = hyb_split(nRow, row, col, val, 0)
    assert int(np.bincount(tail[0]).max()) > 4 * TILE                   # a row whose tail runs through several tiles
    A = sp.SpMatOpt("hyb").convert_device(d)
    assert A.scalar("K") == K and A.scalar("tail_nnz") == len(tail[0])
    y = multiply_checked(A, c, c.name)
    assert_rows(y, c, c.name, exact=c.lens <= K + LONG)
    A.destroy()
    d.free()
