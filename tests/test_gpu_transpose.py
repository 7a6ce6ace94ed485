"""y := A^T x: handles created with options.transpose = 1 (b200spmv_multiply_transpose{,_f32}).

Conversion transposes A's sorted COO on the device and converts the result as a second matrix of the handle's format and
options.  So for every format and option set:
  1. multiply_transpose has the bits of multiply on a handle B of the same format and options converted from the
     host-transposed COO (nCol x nRow, np.lexsort((row, col))), _f32 those of multiply_f32, and every "t." array and
     scalar equals B's;
  2. the forward entries, arrays and scalars are those of a transpose = 0 handle;
  3. A^T x lies within the bound the format meets for A x: the extended-precision row bound of test_gpu_gather_bound in
     fp64, the fp32 bounds of test_gpu_fp32 at precision 1 / 2.
x (nRow entries) sits between NaN bands and y (nCol entries) between canary bands; y is poisoned before every call.
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_fp32 import bound as f32_bound
from test_gpu_fp32 import within
from test_gpu_gather_bound import BOUNDARY_LENS, NCOL, row_reference, wide_case, within_bound

G = 4096                      # guard band, entries
CANARY = -12345.0
TILE = 2048                   # entry-stream tile (entries)

OPTION_SETS = [("crs", {}), ("crs", {"crs_path": 1}), ("crs", {"crs_path": 3}), ("crs", {"crs_path": 4}),
               ("crs", {"value_f32": 1}),
               ("coo", {"coo_path": 0}), ("coo", {"coo_path": 1}), ("coo", {"coo_path": 2}), ("coo", {"coo_path": 3}),
               ("ell", {"col_blocks": 2}), ("ell", {"col_blocks": -1}), ("jds", {"col_blocks": 2}),
               ("jds", {"col_blocks": -1}), ("ss", {"col_blocks": 2}), ("ss", {"col_blocks": -1}),
               ("ss", {"ss_faithful": 1}), ("css", {"ss_faithful": 1}), ("css", {"n_block": 2}),
               ("dia", {}), ("csr5", {}), ("hyb", {})]
OPTION_SETS += [(f, {"precision": p}) for f in ("crs", "ell", "dia", "csr5") for p in (1, 2)]

ARRAYS = ("ptr", "idx", "val", "row_idx", "col_idx", "length", "perm", "diag", "ioff", "H", "nStep", "row_ptr",
          "segment_index", "sum_segs", "sum_segs_count", "tile_desc", "tile_desc_offset", "tile_desc_offset_ptr",
          "tile_ptr", "coo_col_idx", "coo_row_idx", "coo_val", "ell_col_idx", "ell_val")
SCALARS = ("nRow", "nCol", "nNnz", "format", "has_rows", "B", "H", "K", "W", "alg_bytes", "bit_scansum_offset",
           "bit_y_offset", "chunk_feed", "col_block_engine", "col_blocks", "coo_path", "crs_kernel", "launches",
           "maxLength", "multi_kernel", "multi_kernel_f32", "nBlock", "nDiag", "nLong", "nRuns", "nStep", "nTiles",
           "num_offsets", "num_packet", "p", "precision", "row_blocks", "short_row_path", "sigma", "slice_vec", "slots",
           "tail_nnz", "tma", "totalH", "value_f32")


@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


# ------------------------------------------------------------------------------------------ matrices
class Case:
    def __init__(self, name, nRow, nCol, row, col, val, seed=1):
        self.name, self.nRow, self.nCol = name, int(nRow), int(nCol)
        self.row, self.col = np.asarray(row, np.int32), np.asarray(col, np.int32)
        self.val = np.asarray(val, np.float64)
        rng = np.random.default_rng(seed)
        self.x, self.xf = rng.uniform(-1.0, 1.0, self.nCol), rng.uniform(-1.0, 1.0, self.nCol)   # A x
        self.u = rng.uniform(-1.0, 1.0, self.nRow)                                                # A^T u

    def transposed(self):
        """A^T as the host sees it: the triplets swapped and sorted by (col, row)."""
        o = np.lexsort((self.row, self.col))
        return Case(self.name + "^T", self.nCol, self.nRow, self.col[o], self.row[o], self.val[o])


def random_case(name, nRow, nCol, seed, max_len):
    """Rows of 0..max_len distinct columns (a quarter empty), columns >= nCol // 2 + 7 never used (empty columns)."""
    rng = np.random.default_rng(seed)
    use = max(1, nCol // 2 + 7) if nCol > 16 else nCol
    rows, cols = [], []
    for r in range(nRow):
        n = 0 if rng.random() < 0.25 else int(rng.integers(1, min(max_len, use) + 1))
        rows.append(np.full(n, r))
        cols.append(np.sort(rng.choice(use, n, replace=False)))
    row, col = np.concatenate(rows), np.concatenate(cols)
    val = rng.choice([-1.0, 1.0], len(row)) * 10.0 ** rng.uniform(-3, 3, len(row))
    return Case(name, nRow, nCol, row, col, val, seed)


def lens_case(name, lens, seed):
    """Row i takes lens[i] distinct columns of [0, nCol)."""
    rng = np.random.default_rng(seed)
    nCol = max(4096, 2 * max(lens))
    row = np.repeat(np.arange(len(lens)), lens)
    col = np.concatenate([np.sort(rng.choice(nCol, n, replace=False)) for n in lens]) if len(lens) else []
    val = rng.choice([-1.0, 1.0], len(row)) * 10.0 ** rng.uniform(-6, 6, len(row))
    return Case(name, len(lens), nCol, row, col, val, seed)


def arrow_case(n, seed):
    """Every row references column 0 (and its diagonal): A^T's row 0 has n entries, longer than a tile."""
    rng = np.random.default_rng(seed)
    row = np.concatenate([[0], np.repeat(np.arange(1, n), 2)])
    col = np.concatenate([[0], np.stack([np.zeros(n - 1, int), np.arange(1, n)], 1).ravel()])
    return Case("arrow", n, n, row, col, rng.uniform(-1.0, 1.0, len(row)), seed)


def cases(oracle):
    out = [random_case("rect nRow<nCol", 300, 1000, 1, 40), random_case("rect nRow>nCol", 1000, 300, 2, 40),
           Case("lap2d5", *oracle.stencil("lap2d5", 20), seed=3), Case("lap3d7", *oracle.stencil("lap3d7", 9), seed=4),
           Case("box3d27", *oracle.stencil("box3d27", 6), seed=5), Case("rmat", *oracle.rmat(7, 10, 30000), seed=6),
           arrow_case(3000, 7)]
    assert out[-1].transposed().row.tolist().count(0) == 3000 > TILE
    w = wide_case("wide", [11] * (1 << 12), NCOL["A"], 8)
    out.append(Case("wide", w.nRow, w.nCol, w.row, w.col, w.val, seed=8))
    out += [lens_case("lens%d" % i, l, 20 + i) for i, l in enumerate(BOUNDARY_LENS)]
    return out


def skip(fmt, c):
    """DIA holds one column of x per diagonal: the wide and R-MAT matrices have tens of thousands."""
    return fmt == "dia" and len(np.unique(c.col.astype(np.int64) - c.row)) * max(c.nRow, c.nCol) > 3e7


# ------------------------------------------------------------------------------------------ handles and calls
def handle(sp, fmt, opt, c, transpose=0):
    return sp.SpMatOpt(fmt, transpose=transpose, **opt).convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))


def call(A, entry, x, ny, dtype=np.float64):
    """entry(x, y) with x between NaN bands and y (poisoned) between canary bands; returns y."""
    import torch
    td = torch.float64 if dtype == np.float64 else torch.float32
    isz = np.dtype(dtype).itemsize
    xb = torch.full((len(x) + 2 * G,), float("nan"), dtype=td, device="cuda")
    xb[G:G + len(x)] = torch.from_numpy(np.asarray(x, dtype)).cuda()
    yb = torch.full((ny + 2 * G,), CANARY, dtype=td, device="cuda")
    yb[G:G + ny] = float("nan")
    getattr(A, entry)(xb.data_ptr() + isz * G, yb.data_ptr() + isz * G)
    torch.cuda.synchronize()
    y = yb.cpu().numpy()
    assert np.all(y[:G] == CANARY) and np.all(y[G + ny:] == CANARY), (entry, "store outside y")
    return y[G:G + ny].copy()


def bits(a):
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


def arrays(A, prefix=""):
    """{name: (status or size, bytes)} for every array name any format exports"""
    from singlespmv_b200._lib import lib
    out = {}
    for n in ARRAYS:
        key = (prefix + n).encode()
        size = lib.b200spmv_get_array(A.h, key, None, 0)
        data = b""
        if size > 0:
            buf = C.create_string_buffer(size)
            assert lib.b200spmv_get_array(A.h, key, buf, size) == size
            data = buf.raw
        out[n] = (size, data)
    return out


def scalars(A, prefix=""):
    from singlespmv_b200._lib import lib
    out = {}
    for n in SCALARS:
        v = C.c_longlong(-7)
        st = lib.b200spmv_get_scalar(A.h, (prefix + n).encode(), C.byref(v))
        out[n] = (st, v.value if st == 0 else None)
    return out


def prec_of(opt):
    return opt.get("precision", 0)


def within_format_bound(y, M, x, opt, tag):
    """Rule 3 on y = M x (M a Case)."""
    prec = prec_of(opt)
    if prec:
        s, lim = f32_bound(prec, M.nRow, M.row, M.col, M.val.astype(np.float32), x.astype(np.float32))
        fin = np.isfinite(s.astype(np.float64))
        ok = within(y, s, lim) | ~fin
    else:
        v = M.val.astype(np.float32).astype(np.float64) if opt.get("value_f32") else M.val
        ref, bnd = row_reference(M.nRow, M.row, v * x[M.col])
        ok = within_bound(y, ref, bnd)
    assert np.all(ok), (tag, "rows off the bound: %d" % (~ok).sum())
    empty = np.bincount(M.row, minlength=M.nRow)[:M.nRow] == 0
    assert np.all(bits(y[empty]) == 0), (tag, "empty rows must be +0.0")


def check_rules(sp, fmt, opt, c):
    """Rules 1-3 for one format, option set and matrix."""
    tag = (fmt, opt, c.name)
    prec = prec_of(opt)
    dt = np.float32 if prec else np.float64
    fwd, bwd = ("multiply_f32", "multiply_transpose_f32") if prec else ("multiply", "multiply_transpose")
    cT = c.transposed()
    T = handle(sp, fmt, opt, c, transpose=1)
    P = handle(sp, fmt, opt, c)
    B = handle(sp, fmt, opt, cT)
    assert T.scalar("transpose") == 1 and P.scalar("transpose") == 0, tag
    assert T.scalar("t.nRow") == c.nCol and T.scalar("t.nCol") == c.nRow and T.scalar("t.nNnz") == len(c.row), tag
    # rule 1: A^T is B
    assert arrays(T, "t.") == arrays(B), tag
    assert scalars(T, "t.") == scalars(B), tag
    yT = call(T, bwd, c.u, c.nCol, dt)
    yB = call(B, fwd, c.u, c.nCol, dt)
    assert np.array_equal(bits(yT), bits(yB)), (tag, "A^T x is not B x")
    # rule 2: the forward direction is untouched
    assert arrays(T) == arrays(P), tag
    assert scalars(T) == scalars(P), tag
    y1 = call(T, fwd, c.x, c.nRow, dt)
    y0 = call(P, fwd, c.x, c.nRow, dt)
    assert np.array_equal(bits(y1), bits(y0)), (tag, "forward multiply changed")
    if prec:
        h1, h0 = np.full(c.nRow, np.nan, np.float32), np.full(c.nRow, np.nan, np.float32)
        T.multiply_host_f32(c.x.astype(np.float32), h1)
        P.multiply_host_f32(c.x.astype(np.float32), h0)
    else:
        h1, h0 = np.full(c.nRow, np.nan), np.full(c.nRow, np.nan)
        T.multiply_host(c.x, h1)
        P.multiply_host(c.x, h0)
    assert np.array_equal(bits(h1), bits(h0)), (tag, "forward host multiply changed")
    if not prec and c.nRow > 2:
        import torch
        from singlespmv_b200._lib import lib
        r0, r1 = c.nRow // 3, 2 * c.nRow // 3
        out = []
        for A in (T, P):
            xd = torch.from_numpy(c.x).cuda()
            yd = torch.full((c.nRow,), CANARY, dtype=torch.float64, device="cuda")
            st = lib.b200spmv_multiply_rows(A.h, r0, r1, xd.data_ptr(), yd.data_ptr(), None)
            torch.cuda.synchronize()
            out.append((st, bits(yd.cpu().numpy()).tolist()))
        assert out[0] == out[1], (tag, "multiply_rows changed")
    if fmt == "crs" and not prec and not opt.get("value_f32") and c.nRow:
        import torch
        k = 3
        X = torch.from_numpy(np.stack([c.x, c.xf, -c.x], 1).copy()).cuda()
        Ys = []
        for A in (T, P):
            Y = torch.full((c.nRow, k), float("nan"), dtype=torch.float64, device="cuda")
            A.multiply_multi(k, X.data_ptr(), k, Y.data_ptr(), k)
            torch.cuda.synchronize()
            Ys.append(Y.cpu().numpy())
        assert np.array_equal(bits(Ys[0]), bits(Ys[1])), (tag, "multiply_multi changed")
    if fmt == "crs" and prec and c.nRow:
        import torch
        k = 2
        X = torch.from_numpy(np.stack([c.x, c.xf], 1).astype(np.float32)).cuda()
        Ys = []
        for A in (T, P):
            Y = torch.full((c.nRow, k), float("nan"), dtype=torch.float32, device="cuda")
            A.multiply_multi_f32(k, X.data_ptr(), k, Y.data_ptr(), k)
            torch.cuda.synchronize()
            Ys.append(Y.cpu().numpy())
        assert np.array_equal(bits(Ys[0]), bits(Ys[1])), (tag, "multiply_multi_f32 changed")
    # rule 3
    within_format_bound(yT, cT, c.u, opt, tag)
    for A in (T, P, B):
        A.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,opt", OPTION_SETS, ids=["%s-%s" % (f, "-".join("%s%s" % kv for kv in o.items()) or "default")
                                                     for f, o in OPTION_SETS])
def test_transpose_every_format(sp, oracle, fmt, opt):
    for c in cases(oracle):
        if not skip(fmt, c):
            check_rules(sp, fmt, opt, c)


# ------------------------------------------------------------------------------------------ the transpose itself
@pytest.mark.gpu
def test_transpose_coo_is_the_host_lexsort(sp, oracle):
    """On COO handles the t. triplets are the host lexsort bit for bit, empty rows and empty columns included."""
    for c in (random_case("rect", 700, 2000, 31, 60), random_case("tall", 2000, 150, 32, 60),
              Case("rmat", *oracle.rmat(11, 12, 60000), seed=33), arrow_case(3000, 34)):
        cT = c.transposed()
        assert np.any(np.bincount(c.col, minlength=c.nCol) == 0) or c.name == "arrow"
        T = handle(sp, "coo", {}, c, transpose=1)
        assert np.array_equal(T.array("t.row_idx", np.int32), cT.row), c.name
        assert np.array_equal(T.array("t.col_idx", np.int32), cT.col), c.name
        assert np.array_equal(T.array("t.val", np.float64).view(np.int64), cT.val.view(np.int64)), c.name
        T.destroy()


# ------------------------------------------------------------------------------------------ empty matrices
@pytest.mark.gpu
def test_transpose_empty_matrices(sp):
    """No entries: y of nCol becomes +0.0; with nCol = 0 nothing is written."""
    for nRow, nCol in ((10, 7), (0, 5), (6, 0)):
        c = Case("empty", nRow, nCol, [], [], [])
        for fmt, opt in OPTION_SETS:
            prec = prec_of(opt)
            dt = np.float32 if prec else np.float64
            try:
                B = handle(sp, fmt, opt, c.transposed())
                P = handle(sp, fmt, opt, c)
            except sp.B200SpmvError as e:           # a shape the format does not hold: A^T's conversion refuses it too
                with pytest.raises(sp.B200SpmvError) as e2:
                    handle(sp, fmt, opt, c, transpose=1)
                assert e2.value.status == e.value.status, (fmt, opt, nRow, nCol)
                continue
            T = handle(sp, fmt, opt, c, transpose=1)
            y = call(T, "multiply_transpose_f32" if prec else "multiply_transpose", c.u, nCol, dt)
            assert np.all(bits(y) == 0), (fmt, opt, nRow, nCol)
            for A in (T, P, B):
                A.destroy()


# ------------------------------------------------------------------------------------------ row blocks
@pytest.mark.gpu
def test_transpose_row_blocks(sp, oracle, monkeypatch):
    """B200SPMV_BLOCK_NNZ small: both A and A^T are row-blocked.  Order-keeping paths give the bits of the unblocked
    handle, the others stay within the bound."""
    st = Case("lap3d7", *oracle.stencil("lap3d7", 17), seed=41)
    rm = Case("rmat", *oracle.rmat(7, 12, 80000), seed=42)
    for fmt, opt, c, exact in (("crs", {}, st, True), ("ell", {}, st, True), ("dia", {}, st, True),
                               ("crs", {"precision": 2}, st, True), ("crs", {}, rm, False), ("coo", {}, rm, False),
                               ("csr5", {}, rm, False)):
        tag = (fmt, opt, c.name)
        prec = prec_of(opt)
        dt = np.float32 if prec else np.float64
        fwd, bwd = ("multiply_f32", "multiply_transpose_f32") if prec else ("multiply", "multiply_transpose")
        U = handle(sp, fmt, opt, c, transpose=1)
        monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(c.row) // 5))
        T = handle(sp, fmt, opt, c, transpose=1)
        monkeypatch.delenv("B200SPMV_BLOCK_NNZ")
        assert T.scalar("row_blocks") > 1 and T.scalar("t.row_blocks") > 1, tag
        yT, yU = call(T, bwd, c.u, c.nCol, dt), call(U, bwd, c.u, c.nCol, dt)
        fT, fU = call(T, fwd, c.x, c.nRow, dt), call(U, fwd, c.x, c.nRow, dt)
        if exact:
            assert np.array_equal(bits(yT), bits(yU)) and np.array_equal(bits(fT), bits(fU)), tag
        within_format_bound(yT, c.transposed(), c.u, opt, tag)
        within_format_bound(fT, c, c.x, opt, tag)
        T.destroy()
        U.destroy()


# ------------------------------------------------------------------------------------------ reconversion
@pytest.mark.gpu
def test_transpose_reconversion(sp, oracle, monkeypatch):
    """One handle converted again and again: other shapes, and across the row-block limit both ways; A^T follows."""
    from singlespmv_b200._lib import lib
    seq = [(random_case("r1", 400, 900, 51, 30), None), (random_case("r2", 1200, 250, 52, 30), None),
           (Case("lap3d7", *oracle.stencil("lap3d7", 11), seed=53), 2000), (random_case("r3", 500, 500, 54, 30), None),
           (Case("lap2d5", *oracle.stencil("lap2d5", 40), seed=55), 1500)]
    for fmt in ("crs", "ell", "coo"):
        T = sp.SpMatOpt(fmt, transpose=1)
        for c, limit in seq:
            if limit:
                monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(limit))
            T.convert_host(sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val))
            B = handle(sp, fmt, {}, c.transposed())          # the same row-block limit: B is A^T converted alike
            monkeypatch.delenv("B200SPMV_BLOCK_NNZ", raising=False)
            v = C.c_longlong()
            st = lib.b200spmv_get_scalar(T.h, b"t.row_blocks", C.byref(v))
            assert (st == 0 and v.value > 1) if limit else st != 0, (fmt, c.name)
            assert T.scalar("t.nRow") == c.nCol and T.scalar("t.nCol") == c.nRow, (fmt, c.name)
            yT, yB = call(T, "multiply_transpose", c.u, c.nCol), call(B, "multiply", c.u, c.nCol)
            assert np.array_equal(bits(yT), bits(yB)), (fmt, c.name)
            B.destroy()
        T.destroy()


# ------------------------------------------------------------------------------------------ graph capture
@pytest.mark.gpu
def test_transpose_graph_capture(sp, oracle):
    """After an eager call, a captured multiply_transpose{,_f32} replays to the eager bits after x changed."""
    import torch
    rng = np.random.default_rng(61)
    st = Case("lap3d7", *oracle.stencil("lap3d7", 13), seed=62)
    rm = Case("rmat", *oracle.rmat(7, 10, 30000), seed=63)
    for fmt, opt in (("crs", {}), ("crs", {"crs_path": 1}), ("crs", {"crs_path": 4}), ("ell", {}), ("dia", {}),
                     ("csr5", {}), ("crs", {"precision": 1}), ("crs", {"precision": 2}), ("ell", {"precision": 2}),
                     ("dia", {"precision": 1}), ("csr5", {"precision": 2})):
        prec = prec_of(opt)
        td = torch.float32 if prec else torch.float64
        entry = "multiply_transpose_f32" if prec else "multiply_transpose"
        for c in ((st,) if fmt == "dia" else (st, rm)):
            T = handle(sp, fmt, opt, c, transpose=1)
            xd = torch.from_numpy(c.u).to(td).cuda()
            yg = torch.full((c.nCol,), float("nan"), dtype=td, device="cuda")
            getattr(T, entry)(xd.data_ptr(), yg.data_ptr())
            yg.fill_(float("nan"))
            torch.cuda.synchronize()
            graph, stream = torch.cuda.CUDAGraph(), torch.cuda.Stream()
            with torch.cuda.graph(graph, stream=stream):
                getattr(T, entry)(xd.data_ptr(), yg.data_ptr(), stream.cuda_stream)
            xd.copy_(torch.from_numpy(rng.uniform(-1.0, 1.0, c.nRow)).to(td))
            graph.replay()
            torch.cuda.synchronize()
            ye = torch.full((c.nCol,), float("nan"), dtype=td, device="cuda")
            getattr(T, entry)(xd.data_ptr(), ye.data_ptr())
            torch.cuda.synchronize()
            iv = torch.int32 if prec else torch.int64
            assert torch.equal(yg.view(iv), ye.view(iv)), (fmt, opt, c.name)
            T.destroy()


# ------------------------------------------------------------------------------------------ full size
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["crs", "dia"])
def test_transpose_full_size_lap3d7(sp, fmt):
    """lap3d7 256^3 is symmetric: A^T's arrays are A's, A^T x has the bits of A x, and with x = 1 every y[r] is the number
    of boundary faces of grid point r, exactly."""
    import torch
    n = 256
    d = sp.DeviceCoo("lap3d7", n)
    T = sp.SpMatOpt(fmt, transpose=1).convert_device(d)
    d.free()
    for name in (("ptr", "idx", "val") if fmt == "crs" else ("ioff", "diag")):
        dt = np.float64 if name in ("val", "diag") else np.int32
        assert np.array_equal(T.array("t." + name, dt), T.array(name, dt)), name
    for s in ("crs_kernel", "alg_bytes", "tma", "nDiag"):
        try:
            assert T.scalar("t." + s) == T.scalar(s), s
        except sp.B200SpmvError:
            pass
    N = n ** 3
    x = torch.ones(N, dtype=torch.float64, device="cuda")
    yf = torch.full((N,), float("nan"), dtype=torch.float64, device="cuda")
    yt = torch.full((N,), float("nan"), dtype=torch.float64, device="cuda")
    T.multiply(x.data_ptr(), yf.data_ptr())
    T.multiply_transpose(x.data_ptr(), yt.data_ptr())
    torch.cuda.synchronize()
    r = torch.arange(N, device="cuda")
    faces = torch.zeros(N, dtype=torch.float64, device="cuda")
    for q in (r % n, (r // n) % n, r // (n * n)):
        faces += (q == 0).double() + (q == n - 1).double()
    assert torch.equal(yt, faces) and torch.equal(yf, faces)
    x = torch.rand(N, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    T.multiply(x.data_ptr(), yf.data_ptr())
    T.multiply_transpose(x.data_ptr(), yt.data_ptr())
    torch.cuda.synchronize()
    assert torch.equal(yt.view(torch.int64), yf.view(torch.int64))
    T.destroy()


# ------------------------------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_transpose_refusals(sp, oracle):
    """Every status of b200spmv_multiply_transpose{,_f32} in its order, the precision mismatches, the t. names of a
    handle without A^T, and the multi-GPU handle."""
    import torch
    from singlespmv_b200._lib import Options, lib
    c = random_case("rect", 50, 80, 71, 10)
    x = torch.zeros(c.nRow, dtype=torch.float64, device="cuda")
    y = torch.zeros(c.nCol, dtype=torch.float64, device="cuda")
    xp, yp = x.data_ptr(), y.data_ptr()
    for fn in (lib.b200spmv_multiply_transpose, lib.b200spmv_multiply_transpose_f32):
        assert fn(None, xp, yp, None) == -1
        fresh = sp.SpMatOpt("crs", transpose=1)
        assert fn(fresh.h, xp, yp, None) == -4                    # before convert
        assert fn(fresh.h, None, None, None) == -4                # ... decided before the NULL vectors
        plain = handle(sp, "crs", {}, c)
        assert fn(plain.h, xp, yp, None) == -4                    # transpose = 0
        assert fn(plain.h, None, None, None) == -4
    T = handle(sp, "crs", {}, c, transpose=1)
    assert lib.b200spmv_multiply_transpose(T.h, None, yp, None) == -1
    assert lib.b200spmv_multiply_transpose(T.h, xp, None, None) == -1
    assert lib.b200spmv_multiply_transpose(T.h, xp, yp, None) == 0
    assert lib.b200spmv_multiply_transpose_f32(T.h, xp, yp, None) == -4      # precision 0: fp32 vectors refused
    T32 = handle(sp, "crs", {"precision": 1}, c, transpose=1)
    assert lib.b200spmv_multiply_transpose(T32.h, xp, yp, None) == -4        # precision 1: fp64 vectors refused
    assert lib.b200spmv_multiply_transpose_f32(T32.h, xp, yp, None) == 0
    # shapes the other way round: x of nRow, y of nCol; an empty side takes NULL
    e = Case("no rows", 0, 9, [], [], [])
    E = handle(sp, "crs", {}, e, transpose=1)
    assert lib.b200spmv_multiply_transpose(E.h, None, yp, None) == 0
    assert lib.b200spmv_multiply_transpose(E.h, xp, None, None) == -1
    torch.cuda.synchronize()
    plain = handle(sp, "crs", {}, c)
    v = C.c_longlong()
    assert lib.b200spmv_get_scalar(plain.h, b"t.nRow", C.byref(v)) == -4
    assert lib.b200spmv_get_array(plain.h, b"t.ptr", None, 0) == -4
    assert lib.b200spmv_get_scalar(plain.h, b"transpose", C.byref(v)) == 0 and v.value == 0
    o = Options()
    o.transpose = 1
    m = C.c_void_p()
    assert lib.b200spmv_mg_create(1, 0, C.byref(o), C.byref(m)) == -3 and not m.value
    for h in (T, T32, E, plain):
        h.destroy()


# ------------------------------------------------------------------------------------------ without a device
def test_transpose_without_gpu():
    """create validates transpose; multiply_transpose{,_f32} decide NULL handle / unconverted before any CUDA call; the
    option takes the first reserved slot and leaves the struct's size alone."""
    import os
    import re

    import singlespmv_b200 as sp
    from singlespmv_b200._lib import Options, lib
    for bad in (2, -1):
        with pytest.raises(sp.B200SpmvError) as e:
            sp.SpMatOpt("crs", transpose=bad)
        assert e.value.status == -1
    m = sp.SpMatOpt("ell", transpose=1)
    for fn in (lib.b200spmv_multiply_transpose, lib.b200spmv_multiply_transpose_f32):
        assert fn(None, None, None, None) == -1
        assert fn(m.h, None, None, None) == -4
    names = [n for n, _ in Options._fields_]
    assert names[-2:] == ["transpose", "reserved"] and Options._fields_[-1][1]._length_ == 4
    assert C.sizeof(Options) == 16 * C.sizeof(C.c_int)
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "b200spmv.h")).read()
    body = hdr.split("typedef struct {", 1)[1].split("} b200spmv_options;", 1)[0]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"int\s+(\w+(?:\[\d+\])?)\s*;", body)
    assert fields[-2:] == ["transpose", "reserved[4]"] and len(fields) == 13
