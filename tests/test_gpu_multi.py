"""b200spmv_multiply_multi: Y[:, :k] := A X[:, :k] for k = 1..8 row-major vectors on CRS handles.

Row-chunk stream and entry stream handles must give, in every column of Y, the bits of b200spmv_multiply on that column
of X; tile-stream handles run the entry stream and must stay within the extended-precision row bound.  X's columns >= k
hold NaN and Y's hold a canary, both sit between guard bands: a read of anything but X[:, :k] poisons Y, a store outside
Y[:, :k] breaks a canary."""
import numpy as np
import pytest

from test_gpu_gather_bound import BOUNDARY_LENS, NCOL, row_reference, wide_case, within_bound

G = 4096                      # guard band, doubles
CANARY = -12345.0
KS = (1, 2, 3, 5, 8)
ROW_CHUNK, ES_TMA, ES_LOAD = 1, 2, 3


@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


class Case:
    def __init__(self, name, nRow, nCol, row, col, val, seed=1):
        self.name, self.nRow, self.nCol = name, nRow, nCol
        self.row, self.col, self.val = np.asarray(row, np.int32), np.asarray(col, np.int32), np.asarray(val, np.float64)
        self.X = np.random.default_rng(seed).uniform(-1.0, 1.0, (nCol, 8))


def banded_case(name, lens, seed, nCol=16384):
    """Row i takes lens[i] distinct columns of [0, nCol): a band far below the 32 MB that makes gathers depend on L2."""
    rng = np.random.default_rng(seed)
    rows, cols = [], []
    for i, n in enumerate(lens):
        rows.append(np.full(n, i))
        cols.append(np.sort(rng.choice(nCol, n, replace=False)))
    row = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    col = np.concatenate(cols) if cols else np.zeros(0, np.int64)
    val = rng.choice([-1.0, 1.0], len(row)) * 10.0 ** rng.uniform(-6, 6, len(row))
    return Case(name, len(lens), nCol, row, col, val, seed)


def convert(sp, c, **opt):
    return sp.SpMatOpt("crs", **opt).convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))


class Guarded:
    """X (nCol x ldx) between NaN bands, columns >= k NaN; Y (nRow x ldy) between canary bands, columns >= k canaries."""

    def __init__(self, c, k, ldx, ldy):
        import torch
        self.c, self.k, self.ldx, self.ldy = c, k, ldx, ldy
        xb = np.full(c.nCol * ldx + 2 * G, np.nan)
        xb[G:G + c.nCol * ldx].reshape(c.nCol, ldx)[:, :k] = c.X[:, :k]
        self.xb = torch.from_numpy(xb).cuda()
        self.yb = torch.full((c.nRow * ldy + 2 * G,), CANARY, dtype=torch.float64, device="cuda")
        self.xp, self.yp = self.xb.data_ptr() + 8 * G, self.yb.data_ptr() + 8 * G

    def poison(self):
        self.yb[G:G + self.c.nRow * self.ldy].view(self.c.nRow, self.ldy)[:, :self.k] = float("nan")

    def y(self, tag):
        import torch
        torch.cuda.synchronize()
        yb = self.yb.cpu().numpy()
        n = self.c.nRow * self.ldy
        assert np.all(yb[:G] == CANARY) and np.all(yb[G + n:] == CANARY), (tag, "store outside Y")
        Y = yb[G:G + n].reshape(self.c.nRow, self.ldy)
        assert np.all(Y[:, self.k:] == CANARY), (tag, "store into a column >= k")
        return Y[:, :self.k].copy()


def multi(A, g, tag, stream=None):
    g.poison()
    A.multiply_multi(g.k, g.xp, g.ldx, g.yp, g.ldy, stream)
    return g.y(tag)


def singles(A, c, k):
    """column j of the single-vector multiply of X[:, j]"""
    import torch
    out = np.empty((c.nRow, k))
    for j in range(k):
        x = torch.from_numpy(np.ascontiguousarray(c.X[:, j])).cuda()
        y = torch.full((max(c.nRow, 1),), float("nan"), dtype=torch.float64, device="cuda")
        A.multiply(x.data_ptr(), y.data_ptr())
        torch.cuda.synchronize()
        out[:, j] = y.cpu().numpy()[:c.nRow]
    return out


def check(sp, A, c, k, tag, bits):
    """Two calls (Y poisoned before each): bit-identical to each other, +0.0 on empty rows, and either the bits of the
    single multiplies (bits) or within the extended-precision row bound of every column."""
    g = Guarded(c, k, k + 3, k + 1)
    Y1 = multi(A, g, tag)
    Y2 = multi(A, g, tag)
    assert np.array_equal(Y1.view(np.int64), Y2.view(np.int64)), (tag, "not deterministic")
    lens = np.bincount(c.row, minlength=c.nRow)[:c.nRow]
    empty = lens == 0
    assert np.all(Y1[empty].view(np.int64) == 0), (tag, "empty rows must be +0.0")
    if bits:
        S = singles(A, c, k)
        assert np.array_equal(Y1.view(np.int64), S.view(np.int64)), (tag, "not the bits of the single multiplies")
    for j in range(k):
        ref, bound = row_reference(c.nRow, c.row, c.val * c.X[c.col, j])
        assert np.all(within_bound(Y1[:, j], ref, bound)), (tag, j)


def multi_kernel(A):
    return A.scalar("multi_kernel")


# ------------------------------------------------------------------------------------------ every path x k
def path_cases(sp, oracle, monkeypatch):
    """(tag, handle factory, case, expected multi_kernel, bits of the single multiply)"""
    st = Case("lap3d7", *oracle.stencil("lap3d7", 13), seed=3)
    st2 = Case("lap2d5", *oracle.stencil("lap2d5", 37), seed=4)
    box = Case("box3d27", *oracle.stencil("box3d27", 11), seed=5)
    wide = wide_case("k11", [11] * (1 << 15), NCOL["A"], 9)
    wide = Case("wide", wide.nRow, wide.nCol, wide.row, wide.col, wide.val, seed=6)

    def idx_feed():
        monkeypatch.setenv("B200SPMV_CS_FEED", "idx")
        A = convert(sp, st)
        monkeypatch.delenv("B200SPMV_CS_FEED")
        assert A.scalar("chunk_feed") == 0
        return A

    def dict_feed():
        A = convert(sp, st)
        assert A.scalar("chunk_feed") == 1
        return A
    return [("dict", dict_feed, st, ROW_CHUNK, True),
            ("idx", idx_feed, st, ROW_CHUNK, True),
            ("crs_path=3", lambda: convert(sp, st2, crs_path=3), st2, ROW_CHUNK, True),
            ("tile-stream crs_path=1", lambda: convert(sp, st, crs_path=1), st, ES_TMA, False),
            ("tile-stream 27-entry rows", lambda: convert(sp, box), box, ES_TMA, False),
            ("entry stream load-fed", lambda: convert(sp, wide), wide, ES_LOAD, True),
            ("entry stream TMA-fed", lambda: convert(sp, st, crs_path=4), st, ES_TMA, True)]


@pytest.mark.gpu
def test_multi_every_path(sp, oracle, monkeypatch):
    for tag, make, c, kern, bits in path_cases(sp, oracle, monkeypatch):
        A = make()
        assert multi_kernel(A) == kern, tag
        for k in KS:
            check(sp, A, c, k, (tag, k), bits)
        A.destroy()


# ------------------------------------------------------------------------------------------ boundaries
@pytest.mark.gpu
def test_multi_boundaries(sp):
    """Row lengths at the row-chunk stream's limit and chunk size, rows that cross entry-stream tiles and 128-entry groups,
    a row longer than a tile, empty leading and trailing rows; banded (row-chunk stream, tile-stream, entry stream
    TMA-fed) and wide (entry stream load-fed)."""
    lens_sets = [list(l) for l in BOUNDARY_LENS]
    lens_sets += [[0] * 5 + [16] * 600 + [0] * 7, [16] * 256 + [1] * 255 + [0], [0] * 300 + [3]]
    for i, lens in enumerate(lens_sets):
        c = banded_case("lens%d" % i, lens, 300 + i)
        short = max(lens) <= 16
        for opt in ({}, {"crs_path": 1}, {"crs_path": 4}):
            A = convert(sp, c, **opt)
            mk = multi_kernel(A)
            assert mk == (ROW_CHUNK if short and not opt else ES_TMA), (i, opt, mk)
            for k in (1, 3, 8):
                check(sp, A, c, k, (i, opt, k), bits=mk == ROW_CHUNK or opt.get("crs_path") == 4)
            A.destroy()
    for i in (0, 2, 6):
        w = wide_case("w%d" % i, BOUNDARY_LENS[i], NCOL["A"], 400 + i)
        c = Case(w.name, w.nRow, w.nCol, w.row, w.col, w.val, seed=i)
        A = convert(sp, c)
        assert multi_kernel(A) == ES_LOAD
        for k in (2, 5):
            check(sp, A, c, k, ("wide", i, k), bits=True)
        A.destroy()


@pytest.mark.gpu
def test_multi_empty_matrices(sp):
    """No entries: every Y[r, j], j < k, becomes +0.0; no rows: nothing is written."""
    for nRow, nCol in ((10, 7), (0, 5), (6, 0)):
        c = Case("empty", nRow, nCol, [], [], [])
        for opt in ({}, {"crs_path": 1}, {"crs_path": 4}):
            A = convert(sp, c, **opt)
            for k in (1, 4, 8):
                g = Guarded(c, k, k + 3, k + 1)
                Y = multi(A, g, (nRow, opt, k))
                assert np.all(Y.view(np.int64) == 0), (nRow, opt, k)
            A.destroy()


# ------------------------------------------------------------------------------------------ guard bands on other matrices
@pytest.mark.gpu
def test_multi_guard_bands(sp, oracle):
    """The matrices of test_fp32_guard_bands, every reachable path, X and Y with ldx = ldy = k (no gaps)."""
    mats = [("lap3d7", oracle.stencil("lap3d7", 13)), ("lap2d5", oracle.stencil("lap2d5", 37)),
            ("rmat", oracle.rmat(7, 10, 30000)), ("uniform", oracle.uniform(3, 3001, 2777, 9))]
    for name, (nr, nc, row, col, val) in mats:
        c = Case(name, nr, nc, row, col, val, seed=11)
        for opt in ({}, {"crs_path": 1}, {"crs_path": 3}, {"crs_path": 4}):
            A = convert(sp, c, **opt)
            for k in (1, 4, 7):
                g = Guarded(c, k, k, k)
                Y = multi(A, g, (name, opt, k))
                for j in range(k):
                    ref, bound = row_reference(c.nRow, c.row, c.val * c.X[c.col, j])
                    assert np.all(within_bound(Y[:, j], ref, bound)), (name, opt, k, j)
            A.destroy()


# ------------------------------------------------------------------------------------------ graph capture
@pytest.mark.gpu
def test_multi_graph_capture(sp, oracle):
    """A capture after the first call replays to the same bits (X changed in between); the first call on a tile-stream
    handle inside a capture is refused with B200SPMV_ERR_STATE."""
    import torch
    st = Case("lap3d7", *oracle.stencil("lap3d7", 13), seed=21)
    rm = Case("rmat", *oracle.rmat(7, 10, 30000), seed=22)
    for c, opt in ((st, {}), (st, {"crs_path": 1}), (st, {"crs_path": 4}), (rm, {})):
        A = convert(sp, c, **opt)
        k = 5
        g = Guarded(c, k, k + 3, k + 1)
        multi(A, g, "warm-up")
        g.poison()
        graph, stream = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        with torch.cuda.graph(graph, stream=stream):
            A.multiply_multi(k, g.xp, g.ldx, g.yp, g.ldy, stream.cuda_stream)
        X2 = np.random.default_rng(23).uniform(-1.0, 1.0, (c.nCol, k))
        g.xb[G:G + c.nCol * g.ldx].view(c.nCol, g.ldx)[:, :k] = torch.from_numpy(X2).cuda()
        graph.replay()
        Yg = g.y(("graph", opt))
        Ye = multi(A, g, ("eager", opt))
        assert np.array_equal(Yg.view(np.int64), Ye.view(np.int64)), opt
        A.destroy()
    A = convert(sp, st, crs_path=1)
    g = Guarded(st, 2, 2, 2)
    stream = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    from singlespmv_b200._lib import lib
    with torch.cuda.graph(graph, stream=stream):
        st_ = lib.b200spmv_multiply_multi(A.h, 2, g.xp, g.ldx, g.yp, g.ldy, stream.cuda_stream)
    assert st_ == -4
    torch.cuda.synchronize()
    multi(A, g, "after the refused capture")
    A.destroy()


# ------------------------------------------------------------------------------------------ row blocks
@pytest.mark.gpu
def test_multi_row_blocks(sp, oracle, monkeypatch):
    """Row-blocked handles (B200SPMV_BLOCK_NNZ): the bits of the unblocked handle on order-keeping rows."""
    st = Case("lap3d7", *oracle.stencil("lap3d7", 17), seed=31)
    w = wide_case("k11", [11] * (1 << 14), NCOL["A"], 32)
    wide = Case("wide", w.nRow, w.nCol, w.row, w.col, w.val, seed=33)
    for c in (st, wide):
        for k in (1, 3, 8):
            A = convert(sp, c)
            Y0 = multi(A, Guarded(c, k, k + 3, k + 1), "unblocked")
            A.destroy()
            monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(c.row) // 5))
            B = convert(sp, c)
            monkeypatch.delenv("B200SPMV_BLOCK_NNZ")
            assert B.scalar("row_blocks") > 1
            Y1 = multi(B, Guarded(c, k, k + 3, k + 1), "blocked")
            B.destroy()
            if c is st:
                assert np.array_equal(Y0.view(np.int64), Y1.view(np.int64)), (c.name, k)
            for j in range(k):
                ref, bound = row_reference(c.nRow, c.row, c.val * c.X[c.col, j])
                assert np.all(within_bound(Y1[:, j], ref, bound)), (c.name, k, j)


# ------------------------------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_multi_refusals(sp, oracle):
    import torch
    from singlespmv_b200._lib import lib
    c = Case("lap2d5", *oracle.stencil("lap2d5", 9), seed=41)
    X = torch.zeros(c.nCol * 8, dtype=torch.float64, device="cuda")
    Y = torch.zeros(c.nRow * 8, dtype=torch.float64, device="cuda")
    xp, yp = X.data_ptr(), Y.data_ptr()

    def status(A, k=2, ldx=2, ldy=2, x=None, y=None):
        return lib.b200spmv_multiply_multi(A.h if A is not None else None, k, xp if x is None else x, ldx,
                                           yp if y is None else y, ldy, None)
    A = convert(sp, c)
    for k, ldx, ldy in ((0, 2, 2), (9, 9, 9), (-1, 2, 2), (3, 2, 3), (3, 3, 2)):
        assert status(A, k, ldx, ldy) == -1, (k, ldx, ldy)
    assert status(None) == -1
    assert lib.b200spmv_multiply_multi(A.h, 2, None, 2, yp, 2, None) == -1
    assert lib.b200spmv_multiply_multi(A.h, 2, xp, 2, None, 2, None) == -1
    assert status(A) == 0
    keep = [convert(sp, c, value_f32=1)]
    assert status(keep[-1]) == -3
    for prec in (1, 2):
        keep.append(convert(sp, c, precision=prec))
        assert status(keep[-1]) == -4, prec
    for fmt in sp.FORMATS:
        if fmt == "crs":
            continue
        B = sp.SpMatOpt(fmt, **({"n_block": 2} if fmt == "css" else {}))
        B.convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))
        assert status(B) == -3, fmt
    fresh = sp.SpMatOpt("crs")
    assert status(fresh) == -4
    with pytest.raises(sp.B200SpmvError) as e:
        sp.SpMatOpt("ell").convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val)).multiply_multi(2, xp, 2, yp, 2)
    assert e.value.status == -3


# ------------------------------------------------------------------------------------------ full size
@pytest.mark.gpu
def test_multi_full_size_c5(sp):
    """lap3d7 256^3, k = 4, X[:, j] = j + 1: row r of A X[:, j] is (j + 1) times the boundary faces of grid point r,
    a small integer, so Y equals the closed form exactly."""
    import torch
    n, k = 256, 4
    d = sp.DeviceCoo("lap3d7", n)
    A = sp.SpMatOpt("crs").convert_device(d)
    d.free()
    assert multi_kernel(A) == ROW_CHUNK
    N = n ** 3
    X = (torch.arange(k, dtype=torch.float64, device="cuda") + 1).repeat(N, 1).contiguous()
    Y = torch.full((N, k), float("nan"), dtype=torch.float64, device="cuda")
    A.multiply_multi(k, X.data_ptr(), k, Y.data_ptr(), k)
    torch.cuda.synchronize()
    r = torch.arange(N, device="cuda")
    faces = torch.zeros(N, dtype=torch.float64, device="cuda")
    for q in (r % n, (r // n) % n, r // (n * n)):
        faces += (q == 0).double() + (q == n - 1).double()
    ref = faces[:, None] * (torch.arange(k, dtype=torch.float64, device="cuda") + 1)[None, :]
    assert torch.equal(Y, ref)
    A.destroy()


# ------------------------------------------------------------------------------------------ without a device
def test_multi_argument_validation_without_gpu():
    """Status codes that need no device: NULL handle and bad k / ld are ERR_INVALID, an unconverted CRS handle is
    ERR_STATE, a non-CRS handle ERR_UNSUPPORTED -- all decided before any CUDA call."""
    import singlespmv_b200 as sp
    from singlespmv_b200._lib import lib
    m = sp.SpMatOpt("crs")
    assert lib.b200spmv_multiply_multi(None, 2, None, 2, None, 2, None) == -1
    for k, ldx, ldy in ((0, 1, 1), (9, 9, 9), (4, 3, 4), (4, 4, 3)):
        assert lib.b200spmv_multiply_multi(m.h, k, None, ldx, None, ldy, None) == -1, (k, ldx, ldy)
    assert lib.b200spmv_multiply_multi(m.h, 2, None, 2, None, 2, None) == -4
    with pytest.raises(sp.B200SpmvError) as e:
        m.multiply_multi(1, 0, 1, 0, 1)
    assert e.value.status == -4
    coo, f32 = sp.SpMatOpt("coo"), sp.SpMatOpt("crs", precision=1)
    assert lib.b200spmv_multiply_multi(coo.h, 2, None, 2, None, 2, None) == -3
    assert lib.b200spmv_multiply_multi(f32.h, 2, None, 2, None, 2, None) == -4
