"""b200spmv_multiply_multi_f32: Y[:, :k] := A X[:, :k] for k = 1..8 row-major fp32 vectors on CRS handles created with
precision = 1 or 2.

Row-chunk stream handles must give, in every column of Y, the bits of b200spmv_multiply_f32 on that column of X and of
seq(prec) (test_gpu_fp32.py); entry-stream handles (tile-stream, gather-bound and crs_path = 4 handles) must lie within
bound(prec).  X's columns >= k hold NaN and Y's hold a canary, both between guard bands: a read of anything but X[:, :k]
poisons Y, a store outside Y[:, :k] breaks a canary."""
import numpy as np
import pytest

from test_gpu_fp32 import CANARY, G, Case, cancelling_case, check, sorted_case
from test_gpu_gather_bound import BOUNDARY_LENS, NCOL, wide_case

KS = (1, 2, 3, 5, 8)
ROW_CHUNK, ES_TMA, ES_LOAD = 1, 2, 3


@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


class MCase:
    """A matrix and eight fp32 columns of X; col(j) is the test_gpu_fp32 Case of column j (its seq and bound)."""

    def __init__(self, name, nRow, nCol, row, col, val, seed=1, X=None):
        self.name, self.nRow, self.nCol = name, nRow, nCol
        self.row, self.col, self.val = np.asarray(row, np.int32), np.asarray(col, np.int32), np.asarray(val, np.float64)
        X = np.random.default_rng(seed).uniform(-1.0, 1.0, (nCol, 8)) if X is None else X
        self.X = np.ascontiguousarray(X.astype(np.float32))
        self.lens = np.bincount(self.row, minlength=nRow)[:nRow]
        self._cols = {}

    def col_case(self, j):
        if j not in self._cols:
            self._cols[j] = Case("%s[%d]" % (self.name, j), self.nRow, self.nCol, self.row, self.col, self.val,
                                 self.X[:, j].astype(np.float64))
        return self._cols[j]


def from_case(c, seed, X=None):
    return MCase(c.name, c.nRow, c.nCol, c.row, c.col, c.val, seed, X)


def stencil(oracle, kind, n, seed):
    """A stencil's pattern with random values (more rounding than its small integers)."""
    rng = np.random.default_rng(seed)
    nr, nc, row, col, val = oracle.stencil(kind, n)
    val = rng.choice([-1.0, 1.0], len(val)) * rng.uniform(0.5, 2.0, len(val))
    return MCase(kind, nr, nc, row, col, val, seed)


def convert(sp, c, prec, **opt):
    A = sp.SpMatOpt("crs", precision=prec, **opt).convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))
    assert A.scalar("precision") == prec
    return A


class Guarded:
    """X (nCol x ldx floats, starting `shift` floats into its buffer) between NaN bands, columns >= k NaN; Y (nRow x ldy)
    between canary bands, columns >= k canaries."""

    def __init__(self, c, k, ldx, ldy, shift=0):
        import torch
        self.c, self.k, self.ldx, self.ldy = c, k, ldx, ldy
        xb = np.full(c.nCol * ldx + 2 * G + shift, np.nan, np.float32)
        xb[G + shift:G + shift + c.nCol * ldx].reshape(c.nCol, ldx)[:, :k] = c.X[:, :k]
        self.xb = torch.from_numpy(xb).cuda()
        self.yb = torch.full((c.nRow * ldy + 2 * G,), float(CANARY), dtype=torch.float32, device="cuda")
        self.xp, self.yp = self.xb.data_ptr() + 4 * (G + shift), self.yb.data_ptr() + 4 * G
        self.shift = shift

    def set_x(self, X):
        import torch
        n = self.c.nCol * self.ldx
        self.xb[G + self.shift:G + self.shift + n].view(self.c.nCol, self.ldx)[:, :self.k] = torch.from_numpy(X).cuda()

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
    A.multiply_multi_f32(g.k, g.xp, g.ldx, g.yp, g.ldy, stream)
    return g.y(tag)


def singles(A, c, k):
    """column j of multiply_f32 on X[:, j]"""
    import torch
    out = np.empty((c.nRow, k), np.float32)
    for j in range(k):
        x = torch.from_numpy(np.ascontiguousarray(c.X[:, j])).cuda()
        y = torch.full((max(c.nRow, 1),), float("nan"), dtype=torch.float32, device="cuda")
        A.multiply_f32(x.data_ptr(), y.data_ptr())
        torch.cuda.synchronize()
        out[:, j] = y.cpu().numpy()[:c.nRow]
    return out


def check_multi(A, c, k, prec, tag, bits):
    """Two calls (Y poisoned before each): the same bits, and per column either the bits of multiply_f32 and of seq(prec)
    (bits) or bound(prec); empty rows +0.0 (check)."""
    g = Guarded(c, k, k + 3, k + 1)
    Y1 = multi(A, g, tag)
    Y2 = multi(A, g, tag)
    assert np.array_equal(Y1.view(np.uint32), Y2.view(np.uint32)), (tag, "not deterministic")
    if bits:
        S = singles(A, c, k)
        assert np.array_equal(Y1.view(np.uint32), S.view(np.uint32)), (tag, "not the bits of multiply_f32")
    for j in range(k):
        check(Y1[:, j], c.col_case(j), prec, None if bits else np.zeros(c.nRow, bool), (tag, j))
    return Y1


def multi_kernel(A):
    return A.scalar("multi_kernel_f32")


# ------------------------------------------------------------------------------------------ every path x k x precision
def path_cases(sp, oracle, monkeypatch):
    """(tag, handle factory (precision -> handle), case, expected multi_kernel_f32, bits of multiply_f32)"""
    st = stencil(oracle, "lap3d7", 13, 3)
    st2 = stencil(oracle, "lap2d5", 37, 4)
    box = stencil(oracle, "box3d27", 11, 5)
    wide = from_case(wide_case("k11", [11] * (1 << 15), NCOL["A"], 9), 6)

    def idx_feed(prec):
        monkeypatch.setenv("B200SPMV_CS_FEED", "idx")
        A = convert(sp, st, prec)
        monkeypatch.delenv("B200SPMV_CS_FEED")
        assert A.scalar("chunk_feed") == 0
        return A

    def dict_feed(prec):
        A = convert(sp, st, prec)
        assert A.scalar("chunk_feed") == 1
        return A
    return [("dict", dict_feed, st, ROW_CHUNK, True),
            ("idx", idx_feed, st, ROW_CHUNK, True),
            ("crs_path=3", lambda p: convert(sp, st2, p, crs_path=3), st2, ROW_CHUNK, True),
            ("tile-stream crs_path=1", lambda p: convert(sp, st, p, crs_path=1), st, ES_TMA, False),
            ("tile-stream 27-entry rows", lambda p: convert(sp, box, p), box, ES_TMA, False),
            ("entry stream load-fed", lambda p: convert(sp, wide, p), wide, ES_LOAD, False),
            ("entry stream TMA-fed", lambda p: convert(sp, st, p, crs_path=4), st, ES_TMA, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [1, 2])
def test_multi_f32_every_path(sp, oracle, monkeypatch, prec):
    for tag, make, c, kern, bits in path_cases(sp, oracle, monkeypatch):
        A = make(prec)
        assert multi_kernel(A) == kern, (tag, multi_kernel(A))
        for k in KS:
            check_multi(A, c, k, prec, (tag, prec, k), bits)
        A.destroy()


# ------------------------------------------------------------------------------------------ gather widths
@pytest.mark.gpu
def test_multi_f32_gather_widths(sp, oracle):
    """X aligned with ldx = k (vector gathers), X 4 bytes off and odd ldx (scalar gathers): the same bits."""
    st = stencil(oracle, "lap3d7", 13, 7)
    for opt in ({}, {"crs_path": 4}):
        for prec in (1, 2):
            A = convert(sp, st, prec, **opt)
            for k in (2, 3, 4, 6, 8):
                ref = multi(A, Guarded(st, k, k, k), (opt, prec, k, "aligned"))
                for ldx, shift in ((k, 1), (k + 1, 0), (2 * k + 1, 3)):
                    Y = multi(A, Guarded(st, k, ldx, k, shift), (opt, prec, k, ldx, shift))
                    assert np.array_equal(Y.view(np.uint32), ref.view(np.uint32)), (opt, prec, k, ldx, shift)
            A.destroy()


# ------------------------------------------------------------------------------------------ boundaries
def banded_case(name, lens, seed, nCol=16384):
    """Row i takes lens[i] distinct sorted columns of [0, nCol): a band far below the gather-bound limit."""
    c = sorted_case(name, lens, nCol, seed)
    return from_case(c, seed)


@pytest.mark.gpu
def test_multi_f32_boundaries(sp):
    """Row lengths at the row-chunk stream's 8 / 16-entry limits and chunk size, rows across entry-stream tiles and
    128-entry groups, a row through several tiles, empty leading and trailing rows; banded (row-chunk stream, tile-stream,
    entry stream TMA-fed) and wide (entry stream load-fed)."""
    lens_sets = [list(l) for l in BOUNDARY_LENS]
    lens_sets += [[0] * 5 + [16] * 600 + [0] * 7, [8] * 300 + [9] * 300, [16] * 256 + [1] * 255 + [0], [0] * 300 + [3]]
    for i, lens in enumerate(lens_sets):
        c = banded_case("lens%d" % i, lens, 300 + i)
        short = max(lens) <= 16
        for opt in ({}, {"crs_path": 1}, {"crs_path": 4}):
            for prec in (1, 2):
                A = convert(sp, c, prec, **opt)
                mk = multi_kernel(A)
                assert mk == (ROW_CHUNK if short and not opt else ES_TMA), (i, opt, mk)
                for k in (1, 3, 8):
                    check_multi(A, c, k, prec, (i, opt, prec, k), bits=mk == ROW_CHUNK)
                A.destroy()
    for i in (0, 2, 6):
        c = from_case(wide_case("w%d" % i, BOUNDARY_LENS[i], NCOL["A"], 400 + i), i)
        for prec in (1, 2):
            A = convert(sp, c, prec)
            assert multi_kernel(A) == ES_LOAD
            for k in (2, 5):
                check_multi(A, c, k, prec, ("wide", i, prec, k), bits=False)
            A.destroy()


# ------------------------------------------------------------------------------------------ precision-2 rounding
@pytest.mark.gpu
def test_multi_f32_cancelling_rows_across_tiles(sp):
    """Cancelling long rows across 2048-entry tiles through the entry stream (TMA- and load-fed): precision 2 must round
    once, so its pair rows stay within the precision-2 bound (a partial rounded to fp32 at a tile edge is far off)."""
    c0 = cancelling_case(2048, 900)
    rng = np.random.default_rng(901)
    X = rng.uniform(-1.0, 1.0, (c0.nCol, 8))
    X[[0, c0.nCol - 1]] = 1.0                       # the +-2^20 pair meets x = 1 in every column
    c = from_case(c0, 902, X)
    for j in range(8):
        s, lim = c.col_case(j).lim[2]
        assert np.all(lim[c0.pair_rows] < 1e-4), j
    for opt in ({}, {"crs_path": 4}):
        for prec in (1, 2):
            A = convert(sp, c, prec, **opt)
            assert multi_kernel(A) == ES_TMA
            for k in (1, 4, 8):
                check_multi(A, c, k, prec, ("cancel", opt, prec, k), bits=False)
            A.destroy()
    # the same rows on a gather-bound column range: load-fed
    Xw = np.random.default_rng(903).uniform(-1.0, 1.0, (NCOL["A"], 8))
    Xw[[0, NCOL["A"] - 1]] = 1.0
    col = np.where(c0.col == c0.nCol - 1, NCOL["A"] - 1, c0.col)
    cw = MCase("cancel-wide", c0.nRow, NCOL["A"], c0.row, col, c0.val, X=Xw)
    A = convert(sp, cw, 2)
    assert multi_kernel(A) == ES_LOAD
    for k in (1, 4, 8):
        check_multi(A, cw, k, 2, ("cancel-wide", k), bits=False)
    A.destroy()


# ------------------------------------------------------------------------------------------ empty matrices
@pytest.mark.gpu
def test_multi_f32_empty_matrices(sp):
    """No entries: every Y[r, j], j < k, becomes +0.0; no rows or no columns."""
    for nRow, nCol in ((10, 7), (0, 5), (6, 0)):
        c = MCase("empty", nRow, nCol, [], [], [])
        for opt in ({}, {"crs_path": 1}, {"crs_path": 4}):
            for prec in (1, 2):
                A = convert(sp, c, prec, **opt)
                assert multi_kernel(A) == 0, (nRow, nCol, opt, prec)          # no kernel: Y is only zero-filled
                for k in (1, 4, 8):
                    Y = multi(A, Guarded(c, k, k + 3, k + 1), (nRow, opt, prec, k))
                    assert np.all(Y.view(np.uint32) == 0), (nRow, opt, prec, k)
                A.destroy()


# ------------------------------------------------------------------------------------------ graph capture
@pytest.mark.gpu
def test_multi_f32_graph_capture(sp, oracle):
    """A capture after the first call replays to the eager bits with X changed in between; the first call on a
    tile-stream handle inside a capture is refused with B200SPMV_ERR_STATE, and the handle works afterwards."""
    import torch
    from singlespmv_b200._lib import lib
    st = stencil(oracle, "lap3d7", 13, 21)
    nr, nc, row, col, val = oracle.rmat(7, 10, 30000)
    rm = MCase("rmat", nr, nc, row, col, val, 22)
    for c, opt in ((st, {}), (st, {"crs_path": 1}), (st, {"crs_path": 4}), (rm, {})):
        for prec in (1, 2):
            A = convert(sp, c, prec, **opt)
            k = 5
            g = Guarded(c, k, k + 3, k + 1)
            multi(A, g, "warm-up")
            g.poison()
            graph, stream = torch.cuda.CUDAGraph(), torch.cuda.Stream()
            with torch.cuda.graph(graph, stream=stream):
                A.multiply_multi_f32(k, g.xp, g.ldx, g.yp, g.ldy, stream.cuda_stream)
            g.set_x(np.random.default_rng(23).uniform(-1.0, 1.0, (c.nCol, k)).astype(np.float32))
            graph.replay()
            Yg = g.y(("graph", opt, prec))
            Ye = multi(A, g, ("eager", opt, prec))
            assert np.array_equal(Yg.view(np.uint32), Ye.view(np.uint32)), (opt, prec)
            A.destroy()
    for prec in (1, 2):
        A = convert(sp, st, prec, crs_path=1)
        g = Guarded(st, 2, 2, 2)
        stream, graph = torch.cuda.Stream(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            status = lib.b200spmv_multiply_multi_f32(A.h, 2, g.xp, g.ldx, g.yp, g.ldy, stream.cuda_stream)
        assert status == -4, prec
        torch.cuda.synchronize()
        check_multi(A, st, 2, prec, ("after the refused capture", prec), bits=False)
        A.destroy()


# ------------------------------------------------------------------------------------------ row blocks
@pytest.mark.gpu
def test_multi_f32_row_blocks(sp, oracle, monkeypatch):
    """Row-blocked handles (B200SPMV_BLOCK_NNZ): the bits of the unblocked handle on the row-chunk stream, the bound on
    the entry stream (whose tiles the blocks cut differently)."""
    st = stencil(oracle, "lap3d7", 17, 31)
    wide = from_case(wide_case("k11", [11] * (1 << 14), NCOL["A"], 32), 33)
    for c in (st, wide):
        for prec in (1, 2):
            for k in (1, 3, 8):
                A = convert(sp, c, prec)
                Y0 = multi(A, Guarded(c, k, k + 3, k + 1), "unblocked")
                A.destroy()
                monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(c.row) // 5))
                B = convert(sp, c, prec)
                monkeypatch.delenv("B200SPMV_BLOCK_NNZ")
                assert B.scalar("row_blocks") > 1
                Y1 = check_multi(B, c, k, prec, ("blocked", c.name, prec, k), bits=c is st)
                B.destroy()
                if c is st:
                    assert np.array_equal(Y0.view(np.uint32), Y1.view(np.uint32)), (c.name, prec, k)


# ------------------------------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_multi_f32_refusals(sp, oracle):
    import torch
    from singlespmv_b200._lib import lib
    nr, nc, row, col, val = oracle.stencil("lap2d5", 9)
    c = MCase("lap2d5", nr, nc, row, col, val, 41)
    X = torch.zeros(c.nCol * 8, dtype=torch.float32, device="cuda")
    Y = torch.zeros(c.nRow * 8, dtype=torch.float32, device="cuda")
    xp, yp = X.data_ptr(), Y.data_ptr()

    def status(A, k=2, ldx=2, ldy=2, x=None, y=None):
        return lib.b200spmv_multiply_multi_f32(A.h if A is not None else None, k, xp if x is None else x, ldx,
                                               yp if y is None else y, ldy, None)
    for prec in (1, 2):
        A = convert(sp, c, prec)
        for k, ldx, ldy in ((0, 2, 2), (9, 9, 9), (-1, 2, 2), (3, 2, 3), (3, 3, 2)):
            assert status(A, k, ldx, ldy) == -1, (prec, k, ldx, ldy)
        assert lib.b200spmv_multiply_multi_f32(A.h, 2, None, 2, yp, 2, None) == -1
        assert lib.b200spmv_multiply_multi_f32(A.h, 2, xp, 2, None, 2, None) == -1
        assert status(A) == 0
        A.destroy()
    assert status(None) == -1
    keep = [convert(sp, c, 0), sp.SpMatOpt("crs", value_f32=1).convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))]
    for A in keep:
        assert status(A) == -4
        assert b"use b200spmv_multiply_multi" in lib.b200spmv_last_error()
    for fmt in sp.FORMATS:
        if fmt == "crs":
            continue
        opt = {"n_block": 2} if fmt == "css" else {}
        if fmt in ("ell", "dia", "csr5"):
            opt["precision"] = 1
        B = sp.SpMatOpt(fmt, **opt)
        B.convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))
        assert status(B) == -3, fmt
    assert status(sp.SpMatOpt("crs", precision=1)) == -4      # not converted
    # the fp64 entry keeps refusing precision handles, and reports no multi kernel for them
    A = convert(sp, c, 1)
    assert lib.b200spmv_multiply_multi(A.h, 2, xp, 2, yp, 2, None) == -4
    assert A.scalar("multi_kernel") == 0 and A.scalar("multi_kernel_f32") == ROW_CHUNK
    assert keep[0].scalar("multi_kernel_f32") == 0
    with pytest.raises(sp.B200SpmvError) as e:
        keep[0].multiply_multi_f32(2, xp, 2, yp, 2)
    assert e.value.status == -4


# ------------------------------------------------------------------------------------------ full size
@pytest.mark.gpu
@pytest.mark.parametrize("prec", [1, 2])
def test_multi_f32_full_size_c5(sp, prec):
    """lap3d7 256^3, k = 4, X[:, j] = j + 1: row r of A X[:, j] is (j + 1) times the boundary faces of grid point r, a
    small integer, so Y equals the closed form exactly."""
    import torch
    n, k = 256, 4
    d = sp.DeviceCoo("lap3d7", n)
    A = sp.SpMatOpt("crs", precision=prec).convert_device(d)
    d.free()
    assert multi_kernel(A) == ROW_CHUNK
    N = n ** 3
    X = (torch.arange(k, dtype=torch.float32, device="cuda") + 1).repeat(N, 1).contiguous()
    Y = torch.full((N, k), float("nan"), dtype=torch.float32, device="cuda")
    A.multiply_multi_f32(k, X.data_ptr(), k, Y.data_ptr(), k)
    torch.cuda.synchronize()
    r = torch.arange(N, device="cuda")
    faces = torch.zeros(N, dtype=torch.float32, device="cuda")
    for q in (r % n, (r // n) % n, r // (n * n)):
        faces += (q == 0).float() + (q == n - 1).float()
    ref = faces[:, None] * (torch.arange(k, dtype=torch.float32, device="cuda") + 1)[None, :]
    assert torch.equal(Y, ref)
    A.destroy()


# ------------------------------------------------------------------------------------------ without a device
def test_multi_f32_argument_validation_without_gpu():
    """Status codes that need no device, in the order of the header: NULL handle and bad k / ld are ERR_INVALID, a
    non-CRS handle ERR_UNSUPPORTED, a precision-0 handle (value_f32 too) and an unconverted one ERR_STATE -- all decided
    before any CUDA call."""
    import singlespmv_b200 as sp
    from singlespmv_b200._lib import lib
    m = sp.SpMatOpt("crs", precision=2)
    f = lib.b200spmv_multiply_multi_f32
    assert f(None, 2, None, 2, None, 2, None) == -1
    for k, ldx, ldy in ((0, 1, 1), (9, 9, 9), (4, 3, 4), (4, 4, 3)):
        assert f(m.h, k, None, ldx, None, ldy, None) == -1, (k, ldx, ldy)
        assert f(sp.SpMatOpt("ell").h, k, None, ldx, None, ldy, None) == -1, (k, ldx, ldy)
    assert f(m.h, 2, None, 2, None, 2, None) == -4
    with pytest.raises(sp.B200SpmvError) as e:
        m.multiply_multi_f32(1, 0, 1, 0, 1)
    assert e.value.status == -4
    assert f(sp.SpMatOpt("ell", precision=1).h, 2, None, 2, None, 2, None) == -3
    assert f(sp.SpMatOpt("coo").h, 2, None, 2, None, 2, None) == -3
    for opt in ({}, {"value_f32": 1}):
        assert f(sp.SpMatOpt("crs", **opt).h, 2, None, 2, None, 2, None) == -4, opt
        assert b"use b200spmv_multiply_multi" in lib.b200spmv_last_error(), opt
