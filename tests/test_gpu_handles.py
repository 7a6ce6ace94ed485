"""Handles after their first conversion: converted again, and living side by side with other handles.

b200spmv_convert_coo_* on a converted handle converts the new matrix into the format object that already exists, so
every format's conversion has to drop what an earlier matrix or an earlier call left behind: the row-range caches of
prepare_rows, the entry-stream metadata and carries that the first multiply_multi{,_f32} builds, column-block engines,
the host pipeline's plan.  And converting one handle must not change what another live handle computes (a multigrid
hierarchy holds several operators at once).  So:
  A. one handle R converted through matrices that flip each format's internal choices equals, after every conversion,
     a fresh handle F of the same options and matrix: scalars, arrays ("t." ones too) and the bits or refusal of every
     entry point; every entry point that builds state lazily has run on R before it is converted again; y lies within
     the format's bound (test_gpu_transpose.within_format_bound), so "equal to fresh" is anchored to the reference;
  B. the same across the row-block limit, both ways;
  C. a live handle multiplies to the same bits while another handle is converted, converted again, used and destroyed;
     DIA's shared-memory windows, and the edges of its TMA variant;
  D. a conversion refused for bad input leaves the handle unconverted: every entry point answers B200SPMV_ERR_STATE,
     never the old matrix's results, and a good conversion after it equals F;
  E. the multi-GPU handle converted again from host COOs and from the device generator equals a fresh one.
x lies between NaN bands; y and Y are poisoned and lie between canary bands sized for the current matrix, and the
columns k..ld-1 of Y are canaries too.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import skewed_matrix
from test_gpu_gather_bound import NCOL, Guarded, range_cuts, wide_case
from test_gpu_transpose import (CANARY, OPTION_SETS, Case, G, arrays, bits, call, handle, random_case, scalars, skip,
                                within_format_bound)

pytestmark = pytest.mark.gpu

INVALID, UNSUPPORTED, STATE = -1, -3, -4
IDS = ["%s-%s" % (f, "-".join("%s%s" % kv for kv in o.items()) or "default") for f, o in OPTION_SETS]
MULTI_K = ((1, 2), (3, 4), (8, 9))             # (k, ld): ld > k, row-vector loads possible for k = 3 only
COL_BLOCK_SETS = ("ell", "jds", "ss", "css")   # formats with column-block engines


@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


# ------------------------------------------------------------------------------------------ matrices
def with_rows(c):
    """c with the row lengths and pointers range_cuts needs."""
    c.lens = np.bincount(c.row, minlength=c.nRow)[:c.nRow]
    c.ptr = np.concatenate([[0], np.cumsum(c.lens)])
    return c


def case(name, nRow, nCol, row, col, val, seed):
    return with_rows(Case(name, nRow, nCol, row, col, val, seed))


def wide(width, lens, seed):
    w = wide_case("wide" + width, lens, NCOL[width], seed)
    return case(w.name, w.nRow, w.nCol, w.row, w.col, w.val, seed)


def stencil(oracle, kind, n, seed):
    return case("%s n=%d" % (kind, n), *oracle.stencil(kind, n), seed=seed)


def skewed(name, nRow, nCol, seed):
    """Empty rows, rows of 0.9 nCol entries (longer than a 2048-entry tile) and short rows."""
    row, col, val = skewed_matrix(np.random.default_rng(seed), nRow, nCol, 9)
    return case(name, nRow, nCol, row, col, val, seed)


def spmat(sp, c):
    return sp.SpMat(c.nRow, c.nCol, c.row, c.col, c.val)


def sequence(oracle, fmt):
    """Matrices that flip each format's internal choices, ending with the first one again (buffers grow after they
    shrank).  The column-block formats also see an x of 128 MB, which switches column blocks on and off."""
    seq = [wide("A", [11] * (1 << 12), 8),                            # CRS: load-fed entry stream
           stencil(oracle, "box3d27", 14, 2),                        # CRS: tile-stream; DIA: TMA, 9 runs
           skewed("skewed 900x2600", 900, 2600, 3),
           stencil(oracle, "lap3d7", 13, 4),                         # CRS: row-chunk stream
           case("empty 10x7", 10, 7, [], [], [], 5),
           with_rows(random_case("tall 3000x40", 3000, 40, 6, 30))]
    if fmt in COL_BLOCK_SETS:
        seq.insert(3, wide("B", [1, 2047, 2048 * 5, 1], 106))
    seq = [c for c in seq if not skip(fmt, c)]
    return seq + [seq[0]]


# ------------------------------------------------------------------------------------------ entry points
def attempt(sp, f):
    """(0, f()), or (status, None) when the library refuses the call."""
    try:
        return 0, f()
    except sp.B200SpmvError as e:
        return e.status, None


def guarded_X(nCol, k, ld, dtype, seed):
    """X (nCol x ld, row-major) between NaN bands; its columns k..ld-1 are NaN as well."""
    import torch
    td = torch.float64 if dtype == np.float64 else torch.float32
    xb = torch.full((nCol * ld + 2 * G,), float("nan"), dtype=td, device="cuda")
    gen = torch.Generator("cuda").manual_seed(seed)
    xb[G:G + nCol * ld].view(nCol, ld)[:, :k] = torch.rand((nCol, k), generator=gen, dtype=td, device="cuda") * 2 - 1
    return xb


def call_multi(A, entry, k, ld, xb, nRow):
    """entry(k, X, ld, Y, ld) with Y[:, :k] poisoned, Y[:, k:] and the bands around Y canaries; returns Y[:, :k]."""
    import torch
    Yb = torch.full((nRow * ld + 2 * G,), CANARY, dtype=xb.dtype, device="cuda")
    Yb[G:G + nRow * ld].view(nRow, ld)[:, :k] = float("nan")
    esz = xb.element_size()
    getattr(A, entry)(k, xb.data_ptr() + esz * G, ld, Yb.data_ptr() + esz * G, ld)
    torch.cuda.synchronize()
    Y = Yb.cpu().numpy()
    Yv = Y[G:G + nRow * ld].reshape(nRow, ld)
    assert np.all(Y[:G] == CANARY) and np.all(Y[G + nRow * ld:] == CANARY), (entry, k, "store outside Y")
    assert np.all(Yv[:, k:] == CANARY), (entry, k, "store into the columns k..ld-1 of Y")
    return Yv[:, :k].copy()


class Inputs:
    """The vectors every handle of one matrix is multiplied with: x for multiply_rows between NaN bands, X of every k."""

    def __init__(self, c):
        self.g = Guarded(c.x, c.nRow)
        self.X = {(dt, k): guarded_X(c.nCol, k, ld, dt, 10 * k + (dt == np.float32))
                  for dt in (np.float64, np.float32) for k, ld in MULTI_K}


def observe(sp, A, c, inp, tag):
    """Everything the handle shows for matrix c: scalars and arrays (A's and A^T's), and the (status, bits) of every
    entry point.  Calling them builds whatever the handle builds lazily."""
    from singlespmv_b200._lib import lib
    out = {"scalars": scalars(A), "t.scalars": scalars(A, "t."), "arrays": arrays(A), "t.arrays": arrays(A, "t.")}
    for entry, v, ny, dt in (("multiply", c.x, c.nRow, np.float64), ("multiply_f32", c.x, c.nRow, np.float32),
                             ("multiply_transpose", c.u, c.nCol, np.float64),
                             ("multiply_transpose_f32", c.u, c.nCol, np.float32)):
        out[entry] = attempt(sp, lambda: bits(call(A, entry, v, ny, dt)).tobytes())
    h = np.full(c.nRow, np.nan)
    out["multiply_host"] = attempt(sp, lambda: A.multiply_host(c.x, h) or bits(h).tobytes())
    h32 = np.full(c.nRow, np.nan, np.float32)
    out["multiply_host_f32"] = attempt(sp, lambda: A.multiply_host_f32(c.x.astype(np.float32), h32) or bits(h32).tobytes())
    for entry, dt in (("multiply_multi", np.float64), ("multiply_multi_f32", np.float32)):
        for k, ld in MULTI_K:
            out[entry, k] = attempt(sp, lambda: bits(call_multi(A, entry, k, ld, inp.X[dt, k], c.nRow)).tobytes())
    g = inp.g
    for a, b in range_cuts(c):
        st_prep = lib.b200spmv_prepare_rows(A.h, a, b)
        lo, hi = C.c_int(-7), C.c_int(-7)
        st_ext = lib.b200spmv_rows_col_extent(A.h, a, b, C.byref(lo), C.byref(hi))
        g.reset()
        g.yb[G + a:G + b] = float("nan")
        st = lib.b200spmv_multiply_rows(A.h, a, b, g.xp, g.yp, None)
        y = g.y(a, b, tag=(tag, "rows", a, b))                     # rows outside [a, b) keep their canary
        out["rows", a, b] = (st_prep, st_ext, lo.value, hi.value, st, bits(y[a:b]).tobytes() if st == 0 else None)
    return out


def assert_same(oR, oF, tag):
    assert oR.keys() == oF.keys(), tag
    for key in oF:
        assert oR[key] == oF[key], (tag, key, "differs from a fresh handle")


def anchor(oF, c, opt, transpose, tag):
    """y = A x (and A^T u) of the fresh handle within the format's bound."""
    dt = np.float32 if opt.get("precision") else np.float64
    fwd, bwd = ("multiply_f32", "multiply_transpose_f32") if opt.get("precision") else ("multiply", "multiply_transpose")
    st, y = oF[fwd]
    assert st == 0, (tag, fwd, st)
    within_format_bound(np.frombuffer(y, dt), c, c.x, opt, (tag, fwd))
    if transpose:
        st, y = oF[bwd]
        assert st == 0, (tag, bwd, st)
        within_format_bound(np.frombuffer(y, dt), c.transposed(), c.u, opt, (tag, bwd))


def check_fresh(sp, R, fmt, opt, c, transpose, tag, inp=None):
    """R (just converted from c) against a fresh handle of c: the same everything.  Returns what R showed."""
    F = handle(sp, fmt, opt, c, transpose)
    inp = inp or Inputs(c)
    oF = observe(sp, F, c, inp, tag)
    oR = observe(sp, R, c, inp, tag)
    assert_same(oR, oF, tag)
    anchor(oF, c, opt, transpose, tag)
    F.destroy()
    return oR


# ------------------------------------------------------------------------------------------ A. one handle, many matrices
@pytest.mark.parametrize("transpose", [0, 1])
@pytest.mark.parametrize("fmt,opt", OPTION_SETS, ids=IDS)
def test_reconversion_equals_fresh(sp, oracle, fmt, opt, transpose):
    """One handle converted through the whole sequence: after every conversion it is a fresh handle of that matrix."""
    R = sp.SpMatOpt(fmt, transpose=transpose, **opt)
    kernels = set()
    for c in sequence(oracle, fmt):
        tag = (fmt, opt, transpose, c.name)
        st, _ = attempt(sp, lambda: R.convert_host(spmat(sp, c)))
        if st:                                   # a shape the format does not hold: a fresh handle refuses it alike
            assert attempt(sp, lambda: handle(sp, fmt, opt, c, transpose))[0] == st, tag
            continue
        oR = check_fresh(sp, R, fmt, opt, c, transpose, tag)
        kernels.add(oR["scalars"]["crs_kernel"])
        if fmt == "dia" and c.name == "box3d27 n=14":
            assert oR["scalars"]["tma"] == (0, 1) and oR["scalars"]["nRuns"] == (0, 9), tag
    if fmt == "crs" and not opt:
        # the default CRS handle went through the tile-stream, the row-chunk stream and the load-fed entry stream
        assert {(0, 0), (0, 1), (0, 3)} <= kernels, sorted(kernels)
    R.destroy()


# ------------------------------------------------------------------------------------------ B. row-block limit
@pytest.mark.parametrize("opt", [{}, {"precision": 2}], ids=["crs-default", "crs-precision2"])
def test_reconversion_across_row_blocks(sp, oracle, monkeypatch, opt):
    """Row blocks (B200SPMV_BLOCK_NNZ small) on and off and on again on one handle: each conversion equals a fresh
    handle converted under the same limit, the multi-vector multiplies included."""
    from singlespmv_b200._lib import lib
    st = stencil(oracle, "lap3d7", 13, 21)
    rm = case("rmat", *oracle.rmat(7, 12, 80000), seed=22)
    sk = skewed("skewed 900x2600", 900, 2600, 23)
    R = sp.SpMatOpt("crs", **opt)
    for c, parts in ((st, None), (rm, 5), (sk, None), (st, 4), (rm, None)):
        tag = (opt, c.name, parts)
        if parts:
            monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(c.row) // parts))
        R.convert_host(spmat(sp, c))
        F = handle(sp, "crs", opt, c)
        monkeypatch.delenv("B200SPMV_BLOCK_NNZ", raising=False)
        v = C.c_longlong()
        status = lib.b200spmv_get_scalar(R.h, b"row_blocks", C.byref(v))
        assert (status == 0 and v.value > 1) if parts else status != 0, tag
        inp = Inputs(c)
        oF = observe(sp, F, c, inp, tag)
        assert_same(observe(sp, R, c, inp, tag), oF, tag)
        anchor(oF, c, opt, 0, tag)
        F.destroy()
    R.destroy()


# ------------------------------------------------------------------------------------------ C. coexisting handles
@pytest.mark.parametrize("fmt,opt", OPTION_SETS, ids=IDS)
def test_live_handle_untouched(sp, oracle, fmt, opt):
    """H1 keeps multiplying to its first bits while H2 is converted, converted again, used and destroyed."""
    a = stencil(oracle, "lap3d7", 13, 31)
    b = with_rows(random_case("rect 700x400", 700, 400, 32, 40))
    c = skewed("skewed 900x2600", 900, 2600, 33)
    inp = Inputs(a)
    H1 = handle(sp, fmt, opt, a)
    first = observe(sp, H1, a, inp, (fmt, "H1"))
    anchor(first, a, opt, 0, (fmt, "H1"))
    H2 = handle(sp, fmt, opt, b)
    assert_same(observe(sp, H1, a, inp, "H1"), first, (fmt, opt, "after H2 converted"))
    H2.convert_host(spmat(sp, c))
    assert_same(observe(sp, H1, a, inp, "H1"), first, (fmt, opt, "after H2 converted again"))
    observe(sp, H2, c, Inputs(c), (fmt, "H2"))                    # multi-vector multiplies and row ranges on H2
    assert_same(observe(sp, H1, a, inp, "H1"), first, (fmt, opt, "after H2 multiplied"))
    H2.destroy()
    assert_same(observe(sp, H1, a, inp, "H1"), first, (fmt, opt, "after H2 destroyed"))
    H1.destroy()


def diagonals_case(offsets, n, seed):
    """n x n, every entry of the diagonals col - row = offsets."""
    rows = [np.arange(max(0, -d), min(n, n - d)) for d in offsets]
    row = np.concatenate(rows)
    col = np.concatenate([r + d for r, d in zip(rows, offsets)])
    o = np.lexsort((col, row))
    val = np.random.default_rng(seed).uniform(-1.0, 1.0, len(row))
    return Case("diagonals %d" % len(offsets), n, n, row[o], col[o], val, seed)


def runs_offsets(sizes, gap=2):
    """Offsets of consecutive diagonal runs of the given sizes, runs separated by gap - 1 empty diagonals, centred."""
    offs, d = [], 0
    for s in sizes:
        offs += list(range(d, d + s))
        d += s + gap
    return [o - offs[len(offs) // 2] for o in offs]


def dia_reference(oracle, c):
    return oracle.dia_spmv(oracle.dia_convert(c.nRow, c.nCol, c.row, c.col, c.val), c.x)


def call_x_offset(A, x, ny):
    """multiply with x 8 bytes off a 16-byte boundary (between NaN bands): no TMA copy can take it."""
    import torch
    xb = torch.full((len(x) + 2 * G + 1,), float("nan"), dtype=torch.float64, device="cuda")
    xb[G + 1:G + 1 + len(x)] = torch.from_numpy(x).cuda()
    xp = xb.data_ptr() + 8 * (G + 1)
    assert xp % 16 == 8
    yb = torch.full((ny + 2 * G,), CANARY, dtype=torch.float64, device="cuda")
    yb[G:G + ny] = float("nan")
    A.multiply(xp, yb.data_ptr() + 8 * G)
    torch.cuda.synchronize()
    y = yb.cpu().numpy()
    assert np.all(y[:G] == CANARY) and np.all(y[G + ny:] == CANARY), "store outside y"
    return y[G:G + ny].copy()


def test_dia_live_handles_keep_their_windows(sp, oracle):
    """Two TMA handles whose x windows exceed 48 KB of shared memory: 16 runs (65,792 B) and 12 runs (49,344 B).
    Converting the smaller one after the larger must leave the larger one multiplying, to its earlier bits."""
    c16 = diagonals_case(runs_offsets([1] * 16), 3000, 41)
    c12 = diagonals_case(runs_offsets([1] * 12), 2500, 42)
    H1 = handle(sp, "dia", {}, c16)
    assert (H1.scalar("nDiag"), H1.scalar("nRuns"), H1.scalar("tma")) == (16, 16, 1)
    y1 = call(H1, "multiply", c16.x, c16.nRow)
    assert np.array_equal(bits(y1), bits(dia_reference(oracle, c16)))
    H2 = handle(sp, "dia", {}, c12)
    assert (H2.scalar("nDiag"), H2.scalar("nRuns"), H2.scalar("tma")) == (12, 12, 1)
    assert np.array_equal(bits(call(H1, "multiply", c16.x, c16.nRow)), bits(y1)), "H1 after H2's conversion"
    assert np.array_equal(bits(call(H2, "multiply", c12.x, c12.nRow)), bits(dia_reference(oracle, c12)))
    H2.convert_host(spmat(sp, c16))                               # and back: both at 16 runs
    assert np.array_equal(bits(call(H2, "multiply", c16.x, c16.nRow)), bits(y1))
    H2.destroy()
    assert np.array_equal(bits(call(H1, "multiply", c16.x, c16.nRow)), bits(y1)), "H1 after H2's destruction"
    H1.destroy()


@pytest.mark.parametrize("sizes,tma", [([4] * 16, 1), ([4] * 15 + [5], 0), ([1] * 17, 0), ([2] * 8 + [1] * 8, 1)],
                         ids=["64diag-16runs", "65diag", "17runs", "24diag-16runs"])
def test_dia_tma_edges(sp, oracle, sizes, tma):
    """The TMA variant takes up to 64 diagonals in up to 16 runs.  On each side of both limits y has the bits of the
    reference order; on a TMA handle an x 8 bytes off a 16-byte boundary takes the direct kernel, with the same bits."""
    c = diagonals_case(runs_offsets(sizes), 3000, 50 + len(sizes))
    A = handle(sp, "dia", {}, c)
    assert A.scalar("nDiag") == sum(sizes) and A.scalar("tma") == tma, (sizes, A.scalar("tma"))
    ref = bits(dia_reference(oracle, c))
    assert np.array_equal(bits(call(A, "multiply", c.x, c.nRow)), ref)
    assert np.array_equal(bits(call_x_offset(A, c.x, c.nRow)), ref)
    A.destroy()


# ------------------------------------------------------------------------------------------ D. a refused conversion
def bad_inputs(c):
    """(what is wrong, row, col, val) of c broken in one place each."""
    ends = np.flatnonzero(np.diff(c.row) > 0)
    j = int(ends[len(ends) // 2])                                             # c.row[j] < c.row[j + 1]
    swap = np.arange(len(c.row))
    swap[[j, j + 1]] = [j + 1, j]
    dup = np.insert(np.arange(len(c.row)), j, j)
    col = c.col.copy()
    col[-1] = c.nCol
    return [("unsorted", c.row[swap], c.col[swap], c.val[swap]), ("duplicate", c.row[dup], c.col[dup], c.val[dup]),
            ("column >= nCol", c.row, col, c.val)]


def assert_unconverted(sp, A, U, c, tag):
    """Every entry point of A refuses as on the never-converted handle U: B200SPMV_ERR_STATE, except the multi-vector
    forms that U refuses for its format or options first.  Nothing is written."""
    import torch
    from singlespmv_b200._lib import lib
    n = max(c.nRow, c.nCol) * 9 + 16
    xd = torch.zeros(n, dtype=torch.float64, device="cuda")
    yd = torch.full((n,), CANARY, dtype=torch.float64, device="cuda")
    xh, yh = np.zeros(n), np.full(n, CANARY)
    xp, yp = xd.data_ptr(), yd.data_ptr()
    lo, hi, v = C.c_int(), C.c_int(), C.c_longlong()

    def statuses(H):
        h = H.h
        return {"multiply": lib.b200spmv_multiply(h, xp, yp, None),
                "multiply_f32": lib.b200spmv_multiply_f32(h, xp, yp, None),
                "multiply_transpose": lib.b200spmv_multiply_transpose(h, xp, yp, None),
                "multiply_transpose_f32": lib.b200spmv_multiply_transpose_f32(h, xp, yp, None),
                "multiply_host": lib.b200spmv_multiply_host(h, xh.ctypes.data, yh.ctypes.data),
                "multiply_host_f32": lib.b200spmv_multiply_host_f32(h, xh.ctypes.data, yh.ctypes.data),
                "multiply_rows": lib.b200spmv_multiply_rows(h, 0, 1, xp, yp, None),
                "prepare_rows": lib.b200spmv_prepare_rows(h, 0, 1),
                "col_extent": lib.b200spmv_rows_col_extent(h, 0, 1, C.byref(lo), C.byref(hi)),
                "multiply_multi": lib.b200spmv_multiply_multi(h, 3, xp, 3, yp, 3, None),
                "multiply_multi_f32": lib.b200spmv_multiply_multi_f32(h, 3, xp, 3, yp, 3, None),
                "get_scalar": lib.b200spmv_get_scalar(h, b"nRow", C.byref(v)),
                "get_scalar t.": lib.b200spmv_get_scalar(h, b"t.nRow", C.byref(v)),
                "get_array": lib.b200spmv_get_array(h, b"t.val", None, 0)}

    got, want = statuses(A), statuses(U)
    torch.cuda.synchronize()
    assert got == want, (tag, got, want)
    for entry, st in got.items():
        assert st == (want[entry] if entry.startswith("multiply_multi") else STATE), (tag, entry, st)
        assert st in (STATE, UNSUPPORTED), (tag, entry, st)
    assert all(st == STATE for st, _ in scalars(A).values()), tag
    assert all(s == (STATE, b"") for s in arrays(A).values()), tag
    assert torch.all(yd == CANARY) and np.all(yh == CANARY), (tag, "a refused call wrote y")


@pytest.mark.parametrize("fmt,opt", OPTION_SETS, ids=IDS)
def test_refused_reconversion(sp, oracle, fmt, opt):
    """A converted handle (A^T too) given a COO that breaks the input contract: B200SPMV_ERR_INVALID, then it is
    unconverted; the next good conversion equals a fresh handle.  JDS also refuses an imposed permutation of the
    wrong length."""
    first = with_rows(random_case("first 300x200", 300, 200, 61, 20))
    nxt = with_rows(random_case("next 260x330", 260, 330, 62, 25))
    U = sp.SpMatOpt(fmt, transpose=1, **opt)
    breaks = [(what, sp.SpMat(first.nRow, first.nCol, r, c, v)) for what, r, c, v in bad_inputs(first)]
    if fmt == "jds":
        breaks.append(("permutation of nRow + 1 entries", spmat(sp, first)))
    inp = Inputs(nxt)
    for what, bad in breaks:
        tag = (fmt, opt, what)
        R = handle(sp, fmt, opt, first, transpose=1)
        observe(sp, R, first, Inputs(first), tag)                 # lazily built state of the first matrix
        if what.startswith("permutation"):
            R.set_jds_perm(np.arange(first.nRow + 1))
        with pytest.raises(sp.B200SpmvError) as e:
            R.convert_host(bad)
        assert e.value.status == INVALID, (tag, e.value.status)
        assert_unconverted(sp, R, U, first, tag)
        F = handle(sp, fmt, opt, nxt, transpose=1)
        if what.startswith("permutation"):
            R.set_jds_perm(F.array("perm", np.int32))             # the fresh handle's own order: the same arrays
        R.convert_host(spmat(sp, nxt))
        assert_same(observe(sp, R, nxt, inp, tag), observe(sp, F, nxt, inp, tag), tag)
        F.destroy()
        R.destroy()
    U.destroy()


# ------------------------------------------------------------------------------------------ E. multi-GPU handle
def test_mg_reconversion(sp, oracle):
    """One MgSpMat converted from a host COO, another host COO, then the device generator: y has the bits of a fresh
    MgSpMat of the same matrix every time."""
    from singlespmv_b200.mg import MgSpMat
    from test_gpu_parity import _mg_counts
    a = stencil(oracle, "lap3d7", 12, 71)
    b = skewed("skewed 2500", 2500, 2500, 72)
    nr, nc, _, _, _ = oracle.stencil("box3d27", 10)
    rng = np.random.default_rng(73)
    for g in _mg_counts(sp):
        M = MgSpMat(g, "crs")
        for what in (a, b, "box3d27"):
            if what == "box3d27":
                M.convert_synth("box3d27", 10)
                F = MgSpMat(g, "crs").convert_synth("box3d27", 10)
                nRow = nr
            else:
                M.convert_host(spmat(sp, what))
                F = MgSpMat(g, "crs").convert_host(spmat(sp, what))
                nRow = what.nRow
            tag = (g, getattr(what, "name", what))
            assert M.scalar("nNnz") == F.scalar("nNnz") and np.array_equal(M.bounds(), F.bounds()), tag
            x = rng.uniform(-1.0, 1.0, nRow)
            yM, yF = np.full(nRow, np.nan), np.full(nRow, np.nan)
            M.multiply_host(x, yM)
            F.multiply_host(x, yF)
            assert np.array_equal(bits(yM), bits(yF)) and np.all(np.isfinite(yM)), tag
            F.destroy()
        M.destroy()
