"""GPU parity tests proper: the CUDA path, called through the C-ABI (ctypes), against the oracle.

Index arrays: bit-exact against oracle/spmv_oracle.c (pinned to the reference, tests/test_oracle.py)
and against the committed golden vectors produced by the reference itself.
y: against the reference's CRS result (SURVEY.md 8c/8d).  Tolerance 1e-12 per row, relative to
|y_ref| OR -- the reference's own "abs OR rel" precedent, src/util.cpp:77 -- to sum_j |a_ij x_j|
(a reordered sum of a cancelling row cannot do better).  Kernels that keep the reference's
sequential ascending-column order must be bit-identical, and the tests say which.
"""
import numpy as np
import pytest

from conftest import golden_names, load_golden, skewed_matrix

pytestmark = pytest.mark.gpu

TOL = 1e-12
GOLD = golden_names()


@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


def assert_y(y, y_ref, row, col, val, x, nRow, exact=False, tol=TOL):
    assert y.shape == y_ref.shape and np.all(np.isfinite(y))
    if exact:
        assert np.array_equal(y, y_ref), "expected bit-identical y, max diff %g" % np.max(np.abs(y - y_ref))
        return
    mag = np.zeros(nRow)
    np.add.at(mag, row, np.abs(val * x[col]))
    err = np.abs(y - y_ref)
    ok = (err <= tol * np.abs(y_ref)) | (err <= tol * mag)
    assert np.all(ok), "rows off: %d, worst err/mag %g" % ((~ok).sum(), np.max(err / np.maximum(mag, 1e-300)))


def cases(oracle):
    """(name, nRow, nCol, row, col, val, x) -- goldens + randomized skew/empty/ragged inputs."""
    out = []
    for name in GOLD:
        g = load_golden(name)
        out.append((name, int(g["nRow"]), int(g["nCol"]), g["in_row"], g["in_col"], g["in_val"], g["x"]))
    rng = np.random.default_rng(7)
    for i, (nRow, nCol, d) in enumerate([(257, 301, 12), (1000, 777, 40), (5000, 5000, 6), (33, 4000, 3)]):
        row, col, val = skewed_matrix(rng, nRow, nCol, d)
        out.append(("skew%d" % i, nRow, nCol, row, col, val, rng.random(nCol)))
    # edge cases: empty matrix, single entry, one dense row, all-empty tail
    out.append(("empty", 7, 5, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0), rng.random(5)))
    out.append(("single", 4, 4, np.array([2], np.int32), np.array([3], np.int32), np.array([2.5]), rng.random(4)))
    n = 9000
    out.append(("onelong", 3, n, np.full(n, 1, np.int32), np.arange(n, dtype=np.int32), rng.standard_normal(n),
                rng.random(n)))
    nr, nc, r_, c_, v_ = oracle.stencil("lap2d5", 40)
    out.append(("lap2d5_40", nr, nc, r_, c_, v_, oracle.reference_vectors(nc, nr)[0]))
    nr, nc, r_, c_, v_ = oracle.rmat(42, 11, 60000)
    out.append(("rmat_s11", nr, nc, r_, c_, v_, oracle.reference_vectors(nc, nr)[0]))
    return out


@pytest.fixture(scope="module")
def all_cases(oracle):
    return cases(oracle)


def run_host(sp, fmt, nRow, nCol, row, col, val, x, **opt):
    A = sp.SpMat(nRow, nCol, row, col, val)
    A_opt, x_opt = sp.OptimizeProblem(A, sp.Vec(x), fmt, **opt)
    y = sp.Vec(np.full(nRow, np.nan))          # garbage the multiply must fully overwrite
    sp.SpMV(A_opt, x_opt, y)
    y1 = y.val.copy()
    y.val[:] = -7.0
    sp.SpMV(A_opt, x_opt, y)                   # the reference verifies twice (src/main.cpp:40-56)
    assert np.array_equal(y1, y.val), "%s multiply is not idempotent" % fmt
    return A_opt, y1


# ------------------------------------------------------------------------------------------ CRS
def test_crs(sp, oracle, all_cases):
    for name, nRow, nCol, row, col, val, x in all_cases:
        m = oracle.crs_convert(nRow, row, col, val)
        y_ref = oracle.crs_spmv(m, x)
        A_opt, y = run_host(sp, "crs", nRow, nCol, row, col, val, x)
        for k, dt in (("ptr", np.int32), ("idx", np.int32), ("val", np.float64)):
            assert np.array_equal(A_opt.array(k, dt), m[k]), (name, k)
        assert A_opt.scalar("alg_bytes") == 12 * len(row) + 4 * (nRow + 1) + 8 * nCol + 8 * nRow
        assert_y(y, y_ref, row, col, val, x, nRow)
        # rows of <= 64 entries are summed in the reference's own order -> bit-identical
        short = np.diff(m["ptr"]) <= 64
        assert np.array_equal(y[short], y_ref[short]), name


@pytest.mark.parametrize("name", GOLD)
def test_crs_golden_arrays(sp, name):
    g = load_golden(name)
    A_opt, y = run_host(sp, "crs", int(g["nRow"]), int(g["nCol"]), g["in_row"], g["in_col"], g["in_val"], g["x"])
    for k, dt in (("ptr", np.int32), ("idx", np.int32), ("val", np.float64)):
        assert np.array_equal(A_opt.array(k, dt), g["crs." + k])
    short = np.diff(g["crs.ptr"]) <= 64        # one thread per row, reference order -> exact
    assert np.array_equal(y[short], g["crs.y"][short])
    assert_y(y, g["crs.y"], g["in_row"], g["in_col"], g["in_val"], g["x"], int(g["nRow"]))


@pytest.mark.parametrize("fmt,opt", [("crs", {}), ("ss", {"segment_width": 8}), ("css", {"segment_width": 4, "n_block": 3}),
                                     ("ell", {}), ("dia", {})])
def test_multiply_rows(sp, oracle, fmt, opt):
    import torch
    nr, nc, row, col, val = oracle.stencil("lap3d7", 20)
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    A_opt, _ = run_host(sp, fmt, nr, nc, row, col, val, x, **opt)
    xd = torch.from_numpy(x).cuda()
    yd = torch.full((nr,), float("nan"), dtype=torch.float64, device="cuda")
    cuts = [0, 1, 399, 400, 4001, 7600, nr]
    for a, b in zip(cuts[:-1], cuts[1:]):
        A_opt.multiply_rows(a, b, xd.data_ptr(), yd.data_ptr())
    torch.cuda.synchronize()
    y = yd.cpu().numpy()
    if fmt == "css":
        assert_y(y, y_ref, row, col, val, x, nr)        # block partial sums are re-associated
    else:
        assert np.array_equal(y, y_ref)
    # rows outside the requested range are left alone
    yd.fill_(-3.0)
    A_opt.multiply_rows(1000, 2000, xd.data_ptr(), yd.data_ptr())
    torch.cuda.synchronize()
    y = yd.cpu().numpy()
    assert np.all(y[:1000] == -3.0) and np.all(y[2000:] == -3.0) and np.array_equal(y[1000:2000], y_ref[1000:2000]) or fmt == "css"
    for bad in ("coo", "jds", "csr5"):
        B_opt, _ = run_host(sp, bad, 3, 3, [0, 1], [0, 1], [1.0, 2.0], np.ones(3))
        with pytest.raises(sp.B200SpmvError) as e:
            B_opt.multiply_rows(0, 1, xd.data_ptr(), yd.data_ptr())
        assert e.value.status == -3


@pytest.mark.parametrize("fmt,opt", [("crs", {}), ("css", {"n_block": 3}), ("ell", {}), ("dia", {}), ("jds", {})])
def test_host_multiply_pipeline_large(sp, oracle, fmt, opt):
    """>= 2^20 rows: b200spmv_multiply_host runs row chunks with the D2H of y overlapped (formats with row ranges)."""
    nr, nc, row, col, val = oracle.stencil("lap2d5", 1100)
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    A_opt, y = run_host(sp, fmt, nr, nc, row, col, val, x, **opt)
    if fmt == "css":
        assert_y(y, y_ref, row, col, val, x, nr)
    else:
        assert np.array_equal(y, y_ref)
    # a DIFFERENT x on the same handle: a multiply that starts before its slice of x has landed would still
    # see the previous vector in the staging buffer
    for x2 in (x[::-1].copy(), np.full(nc, 0.25), x * 3.0 + 1.0):
        y2 = np.full(nr, np.nan)
        A_opt.multiply_host(x2, y2)
        y2_ref = oracle.crs_result(nr, row, col, val, x2)
        if fmt == "css":
            assert_y(y2, y2_ref, row, col, val, x2, nr)
        else:
            assert np.array_equal(y2, y2_ref)


def test_crs_entry_stream(sp, oracle, all_cases):
    """crs_path = 4: the entry stream (entry_stream.cuh; the default on gather-bound matrices such as config 3) -- row starts as a
    bit per entry instead of row_ptr, segmented warp scans; within the tolerance for every case incl. empty rows, one long row,
    rows ending on every lane / group / chunk / tile boundary; row ranges leave the other rows alone."""
    import torch
    rng = np.random.default_rng(17)
    extra = []
    for lens in ([4] * 64 + [128] * 3 + [256, 256, 1, 255, 2048, 2047, 1, 1, 4096 + 256, 3], [1] * 5000,
                 [0, 0, 3, 0, 125, 0, 0, 128, 1, 0, 255, 257, 0, 0, 0, 6000, 0, 2, 0, 0], [27] * 700 + [0] * 9, [1, 2047, 2048 * 5, 1]):
        nRow, nCol = len(lens), 12000
        row = np.repeat(np.arange(nRow), lens).astype(np.int32)
        col = np.concatenate([np.sort(rng.choice(nCol, size=l, replace=False)) for l in lens] + [np.zeros(0, int)]).astype(np.int32)
        extra.append(("lens", nRow, nCol, row, col, rng.standard_normal(len(row)), rng.random(nCol)))
    for name, nRow, nCol, row, col, val, x in list(all_cases) + extra:
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        A_opt, y = run_host(sp, "crs", nRow, nCol, row, col, val, x, crs_path=4)
        if len(row):
            assert A_opt.scalar("crs_kernel") == 2, name                  # small matrices are banded enough: TMA-fed
        assert_y(y, y_ref, row, col, val, x, nRow)
        if nRow > 40:
            xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
            yd = torch.full((nRow,), -3.0, dtype=torch.float64, device="cuda")
            lo, hi = nRow // 5, nRow - nRow // 3
            A_opt.prepare_rows(lo, hi)
            A_opt.multiply_rows(lo, hi, xd.data_ptr(), yd.data_ptr())
            torch.cuda.synchronize()
            yy = yd.cpu().numpy()
            assert np.all(yy[:lo] == -3.0) and np.all(yy[hi:] == -3.0), name
            assert np.array_equal(yy[lo:hi], y[lo:hi]), name               # deterministic: same bits as the whole multiply


def test_crs_paths_agree(sp, oracle):
    """Short-row matrices take the row-block stream by default; crs_path=1 forces the tile-stream.  Both sum every
    row in the reference's order -> identical y, and both equal the reference CRS result bit for bit."""
    for kind, n in (("lap3d7", 21), ("lap2d5", 130)):
        nr, nc, row, col, val = oracle.stencil(kind, n)
        x = oracle.reference_vectors(nc, nr)[0]
        y_ref = oracle.crs_result(nr, row, col, val, x)
        for fmt in ("crs", "ss"):
            A_auto, y_auto = run_host(sp, fmt, nr, nc, row, col, val, x)
            A_tile, y_tile = run_host(sp, fmt, nr, nc, row, col, val, x, crs_path=1)
            assert A_auto.scalar("short_row_path") == 1 and A_tile.scalar("short_row_path") == 0
            if fmt == "crs":
                assert A_auto.scalar("launches") == 1 and A_tile.scalar("launches") == 2
            assert np.array_equal(y_auto, y_ref) and np.array_equal(y_tile, y_ref)
    # longer rows: the short-row kernels do not apply
    nr, nc, row, col, val = oracle.stencil("box3d27", 9)
    A_opt, _ = run_host(sp, "crs", nr, nc, row, col, val, np.ones(nc))
    assert A_opt.scalar("short_row_path") == 0 and A_opt.scalar("maxLength") == 27


def test_crs_f32_storage(sp, oracle, all_cases):
    """options.value_f32: values rounded to fp32 once, arithmetic in fp64.  Two checks: (1) bit-identical to the
    fp64 path run on the rounded matrix (fp32 -> fp64 widening is exact), (2) within the north star's 1e-5 of the
    reference CRS result on the unrounded matrix."""
    for name, nRow, nCol, row, col, val, x in all_cases:
        val32 = val.astype(np.float32).astype(np.float64)
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        A_opt, y = run_host(sp, "crs", nRow, nCol, row, col, val, x, value_f32=1)
        assert A_opt.scalar("value_f32") == 1
        assert A_opt.scalar("alg_bytes") == 8 * len(row) + 4 * (nRow + 1) + 8 * nCol + 8 * nRow
        assert np.array_equal(A_opt.array("val", np.float64), val32), name
        _, y64 = run_host(sp, "crs", nRow, nCol, row, col, val32, x)
        assert np.array_equal(y, y64), name
        assert_y(y, y_ref, row, col, val, x, nRow, tol=1e-5)
    with pytest.raises(sp.B200SpmvError) as e:
        sp.SpMatOpt("ell", value_f32=1)
    assert e.value.status == -3


# ------------------------------------------------------------------------------------------ ELL
def test_ell(sp, oracle, all_cases):
    for name, nRow, nCol, row, col, val, x in all_cases:
        if name == "onelong" or name.startswith("rmat"):
            K = int(np.max(np.bincount(row, minlength=nRow))) if len(row) else 0
            if K * nRow > 5e7:
                continue
        m = oracle.ell_convert(nRow, row, col, val)
        if m["K"] > nCol:
            continue
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        A_opt, y = run_host(sp, "ell", nRow, nCol, row, col, val, x)
        assert A_opt.scalar("K") == m["K"], name
        assert np.array_equal(A_opt.array("col_idx", np.int32), m["col_idx"].ravel()), name
        assert np.array_equal(A_opt.array("val", np.float64), m["val"].ravel()), name
        # one lane per row, ascending slots, unfused mul/add; padding adds +0.0 -> same bits except -0.0
        assert np.array_equal(y, oracle.ell_spmv(m, x)), name
        assert_y(y, y_ref, row, col, val, x, nRow)


@pytest.mark.parametrize("name", GOLD)
def test_ell_golden(sp, name):
    g = load_golden(name)
    A_opt, y = run_host(sp, "ell", int(g["nRow"]), int(g["nCol"]), g["in_row"], g["in_col"], g["in_val"], g["x"])
    assert A_opt.scalar("K") == int(g["ell.K"])
    assert np.array_equal(A_opt.array("col_idx", np.int32), g["ell.col_idx"])
    assert np.array_equal(A_opt.array("val", np.float64), g["ell.val"])
    assert np.array_equal(y, g["ell.y"])


# ------------------------------------------------------------------------------------------ COO
def test_coo(sp, oracle, all_cases):
    for name, nRow, nCol, row, col, val, x in all_cases:
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        # default: the entry stream (segmented warp scans re-associate the sums: tolerance, deterministic)
        A_opt, y = run_host(sp, "coo", nRow, nCol, row, col, val, x)
        assert np.array_equal(A_opt.array("row_idx", np.int32), row), name      # opt_coo.cpp:14-19 aliases the input
        assert np.array_equal(A_opt.array("col_idx", np.int32), col), name
        assert np.array_equal(A_opt.array("val", np.float64), val), name
        assert A_opt.scalar("alg_bytes") == 16 * len(row) + 8 * nCol + 8 * nRow
        assert A_opt.scalar("coo_path") in (0, 2)                                # entry stream, TMA- or load-fed
        assert_y(y, y_ref, row, col, val, x, nRow)
        for forced in (2, 3):
            A_f, y_f = run_host(sp, "coo", nRow, nCol, row, col, val, x, coo_path=forced)
            assert A_f.scalar("coo_path") == (2 if forced == 2 else 0)
            assert_y(y_f, y_ref, row, col, val, x, nRow)
        # coo_path = 1: the order-preserving tile kernel
        A_opt, y = run_host(sp, "coo", nRow, nCol, row, col, val, x, coo_path=1)
        assert A_opt.scalar("coo_path") == 1
        assert_y(y, y_ref, row, col, val, x, nRow)
        short = np.bincount(row, minlength=nRow) <= 64
        assert np.array_equal(y[short], y_ref[short]), name                     # serial order == the verifier's (util.cpp:67-72)
        assert np.array_equal(y[short], oracle.coo_spmv(nRow, row, col, val, x)[short]), name


def test_coo_tile_boundaries(sp, oracle):
    """Runs that start/end exactly on the 2048-entry tile edges, cross one or several tiles, empty-row gaps."""
    rng = np.random.default_rng(3)
    for lens in ([2048, 2048, 1], [2047, 2, 2047, 5000, 0, 0, 3], [1, 0, 4095, 64, 65, 0, 2048 * 3, 7], [10] * 700 + [0] * 50):
        nRow, nCol = len(lens), 9000
        row = np.repeat(np.arange(nRow), lens).astype(np.int32)
        col = np.concatenate([np.sort(rng.choice(nCol, size=l, replace=False)) for l in lens] + [np.zeros(0, int)]).astype(np.int32)
        val = rng.standard_normal(len(row))
        x = rng.random(nCol)
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        for fmt, opt in (("coo", {"coo_path": 1}), ("crs", {}), ("ss", {})):
            _, y = run_host(sp, fmt, nRow, nCol, row, col, val, x, **opt)
            assert_y(y, y_ref, row, col, val, x, nRow)
            short = np.array(lens) <= 64
            assert np.array_equal(y[short], y_ref[short]), (fmt, lens[:4])
        _, y = run_host(sp, "coo", nRow, nCol, row, col, val, x)
        assert_y(y, y_ref, row, col, val, x, nRow)


def test_coo_entry_stream_chunk_boundaries(sp, oracle):
    """The entry stream's units: 4 entries per lane, 128 per warp pass, 256 per warp chunk, 2048 per tile.  Runs that start or
    end exactly on each of them, runs that pass through whole chunks and tiles, single-entry rows, empty-row gaps, ragged ends."""
    rng = np.random.default_rng(11)
    shapes = ([4] * 64 + [128] * 3 + [256, 256, 1, 255, 2048, 2047, 1, 1, 4096 + 256, 3],
              [1] * 5000,
              [0, 0, 3, 0, 125, 0, 0, 128, 1, 0, 255, 257, 0, 0, 0, 6000, 0, 2, 0, 0],
              [7] * 3000 + [0] * 9,
              [300] * 40 + [5] * 13,
              [1, 2047, 2048 * 5, 1])
    for lens in shapes:
        nRow, nCol = len(lens), 12000
        row = np.repeat(np.arange(nRow), lens).astype(np.int32)
        col = np.concatenate([np.sort(rng.choice(nCol, size=l, replace=False)) for l in lens] + [np.zeros(0, int)]).astype(np.int32)
        val = rng.standard_normal(len(row))
        x = rng.random(nCol)
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        for path in (2, 3):                                  # load-fed and TMA-fed entry stream
            _, y = run_host(sp, "coo", nRow, nCol, row, col, val, x, coo_path=path)
            assert_y(y, y_ref, row, col, val, x, nRow)
            empty = np.array(lens) == 0
            assert np.all(y[empty] == 0.0)


# ------------------------------------------------------------------------------------------ JDS
def test_jds(sp, oracle, all_cases):
    for name, nRow, nCol, row, col, val, x in all_cases:
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        m = oracle.jds_convert(nRow, row, col, val)               # stable convention: ties by ascending row
        A_opt, y = run_host(sp, "jds", nRow, nCol, row, col, val, x)
        assert A_opt.scalar("maxLength") == m["maxLength"], name
        for k in ("perm", "length", "ptr", "col_idx"):
            assert np.array_equal(A_opt.array(k, np.int32), m[k]), (name, k)
        assert np.array_equal(A_opt.array("val", np.float64), m["val"]), name
        assert_y(y, y_ref, row, col, val, x, nRow)
        short = np.diff(oracle.crs_convert(nRow, row, col, val)["ptr"]) <= 2048
        assert np.array_equal(y[short], y_ref[short]), name       # thread-per-row: the reference's own order


@pytest.mark.parametrize("name", GOLD)
def test_jds_golden_reference_tie_order(sp, name):
    """With the reference's own perm imposed (its std::sort is unstable), every array is bit-exact."""
    g = load_golden(name)
    nRow, nCol = int(g["nRow"]), int(g["nCol"])
    A_opt = sp.SpMatOpt("jds")
    A_opt.set_jds_perm(g["jds.perm"])
    A_opt.convert_host(sp.SpMat(nRow, nCol, g["in_row"], g["in_col"], g["in_val"]))
    assert A_opt.scalar("maxLength") == int(g["jds.maxLength"])
    for k in ("perm", "length", "ptr", "col_idx"):
        assert np.array_equal(A_opt.array(k, np.int32), g["jds." + k]), k
    assert np.array_equal(A_opt.array("val", np.float64), g["jds.val"])
    y = np.full(nRow, np.nan)
    A_opt.multiply_host(g["x"], y)
    assert np.array_equal(y, g["jds.y"])
    # default (stable) order: same length/ptr, perm equal up to ties
    B_opt, yb = run_host(sp, "jds", nRow, nCol, g["in_row"], g["in_col"], g["in_val"], g["x"])
    assert np.array_equal(B_opt.array("ptr", np.int32), g["jds.ptr"])
    pb = B_opt.array("perm", np.int32)
    assert np.array_equal(g["jds.length"][pb], g["jds.length"][g["jds.perm"]])
    assert np.array_equal(yb, g["jds.y"])


def test_jds_rejects_bad_perm(sp):
    A = sp.SpMat(3, 3, [0, 0, 1], [0, 1, 1], [1.0, 2.0, 3.0])
    for perm in ([1, 0, 2], [0, 0, 1], [0, 1, 5]):
        m = sp.SpMatOpt("jds")
        m.set_jds_perm(perm)
        with pytest.raises(sp.B200SpmvError):
            m.convert_host(A)


# ------------------------------------------------------------------------------------------ DIA
def banded_cases(oracle):
    rng = np.random.default_rng(11)
    out = []
    for kind, n in (("lap2d5", 33), ("lap3d7", 9), ("box3d27", 10), ("box3d27", 17)):
        nr, nc, r, c, v = oracle.stencil(kind, n)
        out.append(("%s_%d" % (kind, n), nr, nc, r, c, v, oracle.reference_vectors(nc, nr)[0]))
    # rectangular band with random values, odd sizes (exercises unaligned window edges), 70 diagonals (direct kernel)
    for nr, nc, offs in ((1031, 1100, [-40, -3, -2, 0, 1, 2, 7, 60, 61]), (777, 600, list(range(-35, 35)))):
        rows, cols = [], []
        for i in range(nr):
            cs = [i + o for o in offs if 0 <= i + o < nc and rng.random() < 0.8]
            rows += [i] * len(cs)
            cols += cs
        r, c = np.array(rows, np.int32), np.array(cols, np.int32)
        out.append(("band_%dx%d" % (nr, nc), nr, nc, r, c, rng.standard_normal(len(r)), rng.random(nc)))
    return out


def test_dia(sp, oracle, all_cases):
    small = [c for c in all_cases if c[1] * (c[1] + c[2]) < 3e7 and not c[0].startswith(("rmat", "onelong"))]
    for name, nRow, nCol, row, col, val, x in small + banded_cases(oracle):
        m = oracle.dia_convert(nRow, nCol, row, col, val)
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        A_opt, y = run_host(sp, "dia", nRow, nCol, row, col, val, x)
        assert A_opt.scalar("nDiag") == m["nDiag"], name
        assert np.array_equal(A_opt.array("ioff", np.int32), m["ioff"]), name
        assert np.array_equal(A_opt.array("diag", np.float64), m["diag"].ravel()), name
        assert np.array_equal(y, oracle.dia_spmv(m, x)), name     # ascending diagonals per row, unfused
        assert np.array_equal(y, y_ref), name                     # ... which is also the CRS order
    assert A_opt.scalar("tma") == 0                               # 70 diagonals -> direct kernel was covered


@pytest.mark.parametrize("name", GOLD)
def test_dia_golden(sp, name):
    g = load_golden(name)
    A_opt, y = run_host(sp, "dia", int(g["nRow"]), int(g["nCol"]), g["in_row"], g["in_col"], g["in_val"], g["x"])
    assert A_opt.scalar("nDiag") == int(g["dia.nDiag"])
    assert np.array_equal(A_opt.array("ioff", np.int32), g["dia.ioff"])
    assert np.array_equal(A_opt.array("diag", np.float64), g["dia.diag"])
    assert np.array_equal(y, g["dia.y"])


def test_dia_tma_path_used(sp, oracle):
    nr, nc, r, c, v = oracle.stencil("box3d27", 12)
    A_opt, _ = run_host(sp, "dia", nr, nc, r, c, v, np.ones(nc))
    assert A_opt.scalar("nDiag") == 27 and A_opt.scalar("nRuns") == 9 and A_opt.scalar("tma") == 1


# ------------------------------------------------------------------------------------------ SS / CSS
SS_ARRAYS = ("row_ptr", "row_idx", "col_idx", "segment_index", "sum_segs_count", "sum_segs")


def test_ss(sp, oracle, all_cases):
    for name, nRow, nCol, row, col, val, x in all_cases:
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        for W in (1, 4, 32, 1024):
            if W > 32 and len(row) < 5000:
                continue
            m = oracle.ss_convert(nRow, row, col, val, W)
            A_opt, y = run_host(sp, "ss", nRow, nCol, row, col, val, x, segment_width=W)
            assert (A_opt.scalar("H"), A_opt.scalar("nStep"), A_opt.scalar("W")) == (m["H"], m["nStep"], W), (name, W)
            for k in SS_ARRAYS:
                assert np.array_equal(A_opt.array(k, np.int32), m[k]), (name, W, k)
            assert np.array_equal(A_opt.array("val", np.float64), m["val"]), (name, W)
            assert_y(y, y_ref, row, col, val, x, nRow)                 # fused one-pass multiply
            short = np.diff(m["row_ptr"]) <= 64
            assert np.array_equal(y[short], y_ref[short]), (name, W)
            # three-phase schedule in the reference's operation order: bit-identical to the reference's SS result
            F_opt, yf = run_host(sp, "ss", nRow, nCol, row, col, val, x, segment_width=W, ss_faithful=1)
            assert np.array_equal(yf, oracle.ss_spmv(m, x)), (name, W)
            assert_y(yf, y_ref, row, col, val, x, nRow)


@pytest.mark.parametrize("name", GOLD)
@pytest.mark.parametrize("variant,W", [("ss_opt_w2", 2), ("ss_opt_w4", 4), ("ss_opt_w32", 32)])
def test_ss_golden(sp, name, variant, W):
    g = load_golden(name)
    F_opt, yf = run_host(sp, "ss", int(g["nRow"]), int(g["nCol"]), g["in_row"], g["in_col"], g["in_val"], g["x"],
                         segment_width=W, ss_faithful=1)
    assert F_opt.scalar("H") == int(g[variant + ".H"]) and F_opt.scalar("nStep") == int(g[variant + ".nStep"])
    for k in SS_ARRAYS:
        assert np.array_equal(F_opt.array(k, np.int32), g["%s.%s" % (variant, k)]), k
    assert np.array_equal(F_opt.array("val", np.float64), g[variant + ".val"])
    assert np.array_equal(yf, g[variant + ".y"])                       # the reference's own SS result, bit for bit


def test_css(sp, oracle, all_cases):
    for name, nRow, nCol, row, col, val, x in all_cases:
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        for W, N in ((4, 2), (32, 4), (8, 7)):
            m = oracle.css_convert(nRow, nCol, row, col, val, W, N)
            A_opt, y = run_host(sp, "css", nRow, nCol, row, col, val, x, segment_width=W, n_block=N)
            for k in ("B", "nBlock", "totalH"):
                assert A_opt.scalar(k) == m[k], (name, W, N, k)
            for k in ("H", "nStep", "row_ptr", "row_idx", "col_idx", "segment_index", "sum_segs_count", "sum_segs"):
                assert np.array_equal(A_opt.array(k, np.int32), m[k]), (name, W, N, k)
            assert np.array_equal(A_opt.array("val", np.float64), m["val"]), (name, W, N)
            assert_y(y, y_ref, row, col, val, x, nRow)
            F_opt, yf = run_host(sp, "css", nRow, nCol, row, col, val, x, segment_width=W, n_block=N, ss_faithful=1)
            assert np.array_equal(yf, oracle.css_spmv(m, x)), (name, W, N)


@pytest.mark.parametrize("name", GOLD)
@pytest.mark.parametrize("variant,W,N", [("css_opt_w2_n2", 2, 2), ("css_opt_w4_n3", 4, 3), ("css_opt_w32_n4", 32, 4)])
def test_css_golden(sp, name, variant, W, N):
    g = load_golden(name)
    F_opt, yf = run_host(sp, "css", int(g["nRow"]), int(g["nCol"]), g["in_row"], g["in_col"], g["in_val"], g["x"],
                         segment_width=W, n_block=N, ss_faithful=1)
    for k in ("B", "nBlock", "totalH"):
        assert F_opt.scalar(k) == int(g["%s.%s" % (variant, k)]), k
    for k in ("H", "nStep", "row_ptr", "col_idx", "sum_segs_count", "sum_segs"):
        assert np.array_equal(F_opt.array(k, np.int32), g["%s.%s" % (variant, k)]), k
    assert np.array_equal(F_opt.array("val", np.float64), g[variant + ".val"])
    assert np.array_equal(yf, g[variant + ".y"])


# ------------------------------------------------------------------------------------------ CSR5
CSR5_ARRAYS = (("tile_desc", np.uint32), ("tile_desc_offset_ptr", np.int32), ("tile_desc_offset", np.int32),
               ("col_idx", np.int32), ("val", np.float64))


def check_csr5_arrays(A_opt, m, tag):
    for k in ("sigma", "p", "bit_y_offset", "bit_scansum_offset", "num_packet", "num_offsets"):
        assert A_opt.scalar(k) == int(m[k]), (tag, k)
    p = int(m["p"])
    ta, tb = A_opt.array("tile_ptr", np.uint32), np.array(m["tile_ptr"], np.uint32)
    if p > 0:     # the tail tile's dirty bit comes from an out-of-bounds read upstream (format_avx2.h:48-55)
        ta[p - 1:] &= 0x7FFFFFFF
        tb[p - 1:] &= 0x7FFFFFFF
    assert np.array_equal(ta, tb), (tag, "tile_ptr")
    for k, dt in CSR5_ARRAYS:
        assert np.array_equal(A_opt.array(k, dt), m[k]), (tag, k)


def test_csr5(sp, oracle, all_cases):
    for name, nRow, nCol, row, col, val, x in all_cases:
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        for sigma in (-1, 0, 4, 7, 32):
            A_opt, y = run_host(sp, "csr5", nRow, nCol, row, col, val, x, csr5_sigma=sigma)
            ref_rule = oracle.csr5_auto_sigma(nRow, len(row))      # anonymouslib_cuda.h:293-317
            want = {-1: ref_rule, 0: max(ref_rule, 16)}.get(sigma, sigma)
            assert A_opt.scalar("sigma") == want, (name, sigma)
            m = oracle.csr5_convert(nRow, row, col, val, want)
            check_csr5_arrays(A_opt, m, (name, sigma))
            assert_y(y, y_ref, row, col, val, x, nRow)
            assert_y(y, oracle.csr5_spmv(m, x), row, col, val, x, nRow)


@pytest.mark.parametrize("name", GOLD)
@pytest.mark.parametrize("sigma", [4, 16])
def test_csr5_golden(sp, name, sigma):
    """Arrays produced by the reference's own conversion routines (omega = 32), committed as fixtures."""
    g = load_golden(name)
    nRow, nCol = int(g["nRow"]), int(g["nCol"])
    A_opt, y = run_host(sp, "csr5", nRow, nCol, g["in_row"], g["in_col"], g["in_val"], g["x"], csr5_sigma=sigma)
    ref = {k[len("csr5_s%d." % sigma):]: g[k] for k in g if k.startswith("csr5_s%d." % sigma)}
    check_csr5_arrays(A_opt, ref, (name, sigma))
    assert_y(y, g["crs.y"], g["in_row"], g["in_col"], g["in_val"], g["x"], nRow)


def test_csr5_empty_row_patterns(sp, oracle):
    """Leading / trailing / interior runs of empty rows, rows starting exactly on tile boundaries (sigma 4: tile = 128)."""
    rng = np.random.default_rng(5)
    for lens in ([0, 0, 0, 128, 0, 128, 256, 0, 0, 1, 0], [127, 1, 0, 0, 128, 3, 0, 125, 600, 0], [0] * 40 + [5] * 200 + [0] * 300,
                 [1000, 0, 0, 24, 0], [128] * 9, [3, 0] * 400):
        nRow, nCol = len(lens), 1500
        row = np.repeat(np.arange(nRow), lens).astype(np.int32)
        col = np.concatenate([np.sort(rng.choice(nCol, size=l, replace=False)) for l in lens] + [np.zeros(0, int)]).astype(np.int32)
        val = rng.standard_normal(len(row))
        x = rng.random(nCol)
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        for sigma in (4, 5):
            m = oracle.csr5_convert(nRow, row, col, val, sigma)
            A_opt, y = run_host(sp, "csr5", nRow, nCol, row, col, val, x, csr5_sigma=sigma)
            check_csr5_arrays(A_opt, m, (lens[:5], sigma))
            assert_y(y, y_ref, row, col, val, x, nRow)


# ------------------------------------------------------------------------------------------ inputs
def test_rejects_unsorted_and_duplicates(sp):
    x = np.ones(4)
    for row, col in (([1, 0], [0, 0]), ([0, 0], [1, 1]), ([0, 5], [0, 0]), ([0, 0], [2, 1])):
        A = sp.SpMat(4, 4, row, col, [1.0, 2.0])
        with pytest.raises(sp.B200SpmvError) as e:
            sp.OptimizeProblem(A, sp.Vec(x), "crs")
        assert e.value.status == -1


@pytest.mark.parametrize("kind,p0,p1", [("lap2d5", 37, 0), ("lap3d7", 13, 0), ("box3d27", 11, 0),
                                        ("uniform", 3000, 32), ("rmat", 10, 30000)])
def test_synth_matches_oracle(sp, oracle, kind, p0, p1):
    seed = 42 if kind == "rmat" else 1
    d = sp.DeviceCoo(kind, p0, p1, seed)
    nRow, nCol, row, col, val = d.to_host()
    if kind == "uniform":
        ref = oracle.uniform(seed, p0, p0, p1)
    elif kind == "rmat":
        ref = oracle.rmat(seed, p0, p1)
    else:
        ref = oracle.stencil(kind, p0)
    assert (nRow, nCol) == (ref[0], ref[1])
    assert np.array_equal(row, ref[2]) and np.array_equal(col, ref[3]) and np.array_equal(val, ref[4])


def test_synth_row_range(sp, oracle):
    full = sp.DeviceCoo("lap3d7", 12).to_host()
    part = sp.DeviceCoo("lap3d7", 12, row_begin=500, row_end=1100).to_host()
    sel = (full[2] >= 500) & (full[2] < 1100)
    assert np.array_equal(part[2], full[2][sel]) and np.array_equal(part[3], full[3][sel])
    u = sp.DeviceCoo("uniform", 4096, 16, 1, row_begin=100, row_end=900).to_host()
    ref = oracle.uniform(1, 4096, 4096, 16, 100, 900)
    assert np.array_equal(u[3], ref[3]) and np.array_equal(u[4], ref[4])


# ------------------------------------------------------------------------------------------ full-size properties
def test_full_size_linearity_crs_ell(sp):
    """At a BASELINE-scale shape the oracle is too slow; use size-independent properties:
    A(ax + bz) == a Ax + b Az (to rounding), formats agree with each other, y(ones) == row sums."""
    import torch
    d = sp.DeviceCoo("uniform", 1 << 20, 32, 1)
    n = d.nRow
    crs = sp.SpMatOpt("crs").convert_device(d)
    ell = sp.SpMatOpt("ell").convert_device(d)
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    z = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    out = {}
    for name, m in (("crs", crs), ("ell", ell)):
        ys = []
        for v in (x, z, 2.0 * x + 0.5 * z):
            y = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
            m.multiply(v.data_ptr(), y.data_ptr())
            torch.cuda.synchronize()
            ys.append(y)
        lin = 2.0 * ys[0] + 0.5 * ys[1]
        assert torch.allclose(ys[2], lin, rtol=1e-12, atol=1e-12)
        out[name] = ys[0]
    assert torch.equal(out["crs"], out["ell"])          # both sum each row in ascending-column order


# ------------------------------------------------------------------------------------------ row-partitioned path
@pytest.mark.parametrize("kind,n,parts", [("lap3d7", 24, 2), ("lap3d7", 24, 5), ("box3d27", 14, 3), ("lap2d5", 90, 4)])
def test_partitioned_blocks_match_single_gpu(sp, oracle, kind, n, parts):
    """All blocks of the multi-GPU path on one device (device-to-device copies stand in for NCCL):
    same device code (halo plan, renumbering, pack, multiply_rows) -> y bit-identical to the reference CRS."""
    import torch
    from singlespmv_b200 import dist as spd
    nr, nc, row, col, val = oracle.stencil(kind, n)
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    bounds, blocks = spd.build_local_group(kind, n, 0, 1, parts)
    ptr = oracle.crs_convert(nr, row, col, val)["ptr"]
    targets = [len(row) * g // parts for g in range(parts + 1)]
    assert [int(b) for b in bounds] == [int(np.searchsorted(ptr, t, side="left")) for t in targets[:-1]] + [nr]
    xd = torch.from_numpy(x).cuda()
    for b in blocks:
        lo, hi = int(bounds[b.rank]), int(bounds[b.rank + 1])
        b.x_owned.copy_(xd[lo:hi])
        assert b.interiorBegin <= b.interiorEnd
    for _ in range(2):
        spd.local_group_multiply(blocks)
    torch.cuda.synchronize()
    y = torch.cat([b.y for b in blocks]).cpu().numpy()
    assert np.array_equal(y, y_ref)
    # interior rows really are the bulk and really touch no halo
    if kind == "lap3d7" and parts == 2:
        assert blocks[0].nLeft == 0 and blocks[0].nRight == n * n and blocks[1].nLeft == n * n
        assert blocks[0].interiorEnd - blocks[0].interiorBegin == blocks[0].nRows - n * n
    for b in blocks:
        b.free()


@pytest.mark.parametrize("kind,n,parts", [("lap3d7", 24, 2), ("lap3d7", 24, 5), ("box3d27", 14, 3), ("uniform", 4096, 4)])
def test_x_window_exchange_kernel(sp, oracle, kind, n, parts):
    """The peer-memory exchange of the torchrun path (csrc/xwin.cu) with every rank's window in one process on one GPU:
    flags, pull and acknowledgement over several steps with a NEW x each step; y bit-identical to the reference CRS."""
    import ctypes as C
    import torch
    from singlespmv_b200 import dist as spd
    from singlespmv_b200._lib import lib
    if kind == "uniform":
        nr, nc, row, col, val = oracle.uniform(1, n, n, 8)
        p1 = 8
    else:
        nr, nc, row, col, val = oracle.stencil(kind, n)
        p1 = 0
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    bounds, blocks = spd.build_local_group(kind, n, p1, 1, parts, windows=True)
    streams = [torch.cuda.Stream() for _ in blocks]
    xd = torch.from_numpy(x).cuda()
    for step, scale in enumerate((1.0, 2.0, 0.5, 1.0)):
        for b in blocks:
            lo, hi = int(bounds[b.rank]), int(bounds[b.rank + 1])
            b.x_owned.copy_(xd[lo:hi] * scale)
        spd.local_group_multiply_windows(blocks, streams)
        torch.cuda.synchronize()
        y = torch.cat([b.y for b in blocks]).cpu().numpy()
        assert np.array_equal(y, y_ref * scale), "step %d" % step
    for b in blocks:
        steps, bad = C.c_longlong(), C.c_int()
        assert lib.b200spmv_xwin_status(b.win, C.byref(steps), C.byref(bad)) == 0
        assert steps.value == 4 and bad.value == 0
        b.free()


def test_partition_rows_from_coo(sp, oracle):
    import ctypes as C
    from singlespmv_b200._lib import lib, check
    d = sp.DeviceCoo("rmat", 12, 100000, 42)
    _, _, row, col, val = d.to_host()
    ptr = oracle.crs_convert(d.nRow, row, col, val)["ptr"]
    for parts in (2, 8):
        b = np.empty(parts + 1, np.int32)
        check(lib.b200spmv_partition_rows(d.c.row_d, d.nNnz, d.nRow, parts, b.ctypes.data_as(C.c_void_p)))
        assert b[0] == 0 and b[-1] == d.nRow and np.all(np.diff(b) >= 0)
        per = np.diff(ptr[b])
        assert per.max() - per.min() <= 2 * np.diff(ptr).max()        # balanced up to one row


# ------------------------------------------------------------------------------------------ statistics + recommendation
@pytest.mark.parametrize("kind,p0,p1,expect", [("lap2d5", 300, 0, "dia"), ("box3d27", 40, 0, "dia"), ("lap3d7", 50, 0, "dia"),
                                                ("uniform", 1 << 16, 32, "ell"), ("rmat", 15, 1 << 20, "csr5")])
def test_analyze_and_recommend(sp, oracle, kind, p0, p1, expect):
    d = sp.DeviceCoo(kind, p0, p1, 42 if kind == "rmat" else 1)
    nRow, nCol, row, col, val = d.to_host()
    st, _ = d.analyze()
    ref = oracle.counter(nRow, nCol, row, col)            # matrix/script/counter.cpp restated
    for k in ("rowMax", "rowMin", "colMax", "colMin", "nDiag"):
        assert st[k] == ref[k], k
    assert st["nnz"] == len(row) and st["nEmptyRows"] == int((np.bincount(row, minlength=nRow) == 0).sum())
    assert abs(st["rowVar"] - ref["rowVar"]) <= 1e-9 * max(1.0, ref["rowVar"])
    fmt, opts = d.recommend()
    assert fmt == expect, (fmt, opts, st)


def test_recommend_rules_at_baseline_scale(sp):
    """The rule table on the BASELINE.json shapes, from their closed-form statistics (no 500 M-entry matrix needed)."""
    import ctypes as C
    from singlespmv_b200._lib import Options, Stats, lib
    def rec(**kw):
        st = Stats()
        for k, v in kw.items():
            setattr(st, k, v)
        o = Options()
        f = lib.b200spmv_recommend_format(C.byref(st), C.byref(o))
        return [k for k, v in sp.FORMATS.items() if v == f][0], o.n_block
    n2 = 1 << 24
    assert rec(nRow=n2, nCol=n2, nnz=n2 * 32, rowMax=32, rowMin=32, rowMean=32.0, rowVar=0.0, nDiag=2 * n2 - 1) == ("css", 3)   # c2
    assert rec(nRow=1 << 23, nCol=1 << 23, nnz=258673573, rowMax=400000, rowMean=30.8, rowVar=1e5, nDiag=1 << 24)[0] == "csr5"  # c3
    assert rec(nRow=256 ** 3, nCol=256 ** 3, nnz=766 ** 3, rowMax=27, rowMean=26.8, rowVar=0.5, nDiag=27)[0] == "dia"           # c4
    assert rec(nRow=512 ** 3, nCol=512 ** 3, nnz=937951232, rowMax=7, rowMean=6.99, rowVar=0.01, nDiag=7)[0] == "dia"           # c5
    assert rec(nRow=1000, nCol=1000, nnz=9000, rowMax=40, rowMean=9.0, rowVar=20.0, nDiag=900)[0] == "crs"


# ------------------------------------------------------------------------------------------ BASELINE.json full sizes
def _mult(m, x, n):
    import torch
    y = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
    m.multiply(x.data_ptr(), y.data_ptr())
    torch.cuda.synchronize()
    return y


@pytest.mark.parametrize("kind,p0,fmts", [("box3d27", 256, ("dia", "ell", "jds", "crs")),      # config 4
                                          ("lap3d7", 512, ("crs", "dia", "ell")),               # config 5
                                          ("lap2d5", 1024, ("crs", "dia", "ell", "jds", "ss", "coo"))])   # config 1
def test_full_size_stencils(sp, kind, p0, fmts):
    """At BASELINE.json's full sizes the oracle is too slow; size-independent properties instead:
    * A.1 has a closed form for the stencils (diagonal = points-1, off-diagonals = -1): y_i = points - count_i,
      an exact small integer -> checks every row of every format;
    * every format that sums a row in ascending column order must agree bit for bit on a random x;
    * linearity A(2x + z/2) = 2Ax + Az/2."""
    import torch
    d = sp.DeviceCoo(kind, p0)
    n = d.nRow
    stats, _ = d.analyze()
    points = {"lap2d5": 5, "lap3d7": 7, "box3d27": 27}[kind]
    assert stats["rowMax"] == points and stats["nDiag"] == points and stats["nEmptyRows"] == 0
    mats = {f: sp.SpMatOpt(f).convert_device(d) for f in fmts}
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    z = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    ones = torch.ones(n, dtype=torch.float64, device="cuda")
    # count_i = entries of row i, closed form of the generator (no wrap-around at the grid border)
    idx = torch.arange(n, device="cuda")
    span = lambda a: 1 + (a > 0).long() + (a < p0 - 1).long()
    if kind == "lap2d5":
        counts = span(idx // p0) + span(idx % p0) - 1
    else:
        si, sj, sk = span(idx // (p0 * p0)), span((idx // p0) % p0), span(idx % p0)
        counts = si + sj + sk - 2 if kind == "lap3d7" else si * sj * sk
    assert int(counts.sum().item()) == d.nNnz
    counts = counts.double()
    del idx
    ys = {}
    for f, m in mats.items():
        y1 = _mult(m, ones, n)
        assert torch.equal(y1, points - counts), f
        ys[f] = _mult(m, x, n)
        lin = _mult(m, 2.0 * x + 0.5 * z, n)
        assert torch.allclose(lin, 2.0 * ys[f] + 0.5 * _mult(m, z, n), rtol=1e-12, atol=1e-12), f
    first = fmts[0]
    for f in fmts[1:]:
        if f == "coo":                 # the entry stream re-associates the sums across lanes
            assert torch.allclose(ys[f], ys[first], rtol=1e-12, atol=1e-13), (f, first)
        else:
            assert torch.equal(ys[f], ys[first]), (f, first)


def test_full_size_uniform_and_rmat(sp, oracle):
    """Configs 2 and 3 at full size, against the ORACLE (VERDICT r1: not only format against format): the first 2^21 rows
    of config 2 / the whole of config 3 are downloaded and multiplied by the C restatement of the reference's CRS loop
    (src/opt_crs.cpp:44-70); every format of the config must match it -- bit for bit where one thread sums a row of at most
    64 entries in column order (all of config 2), within 1e-12 otherwise."""
    import torch
    for kind, p0, p1, seed, fmts, opts, rows in (("uniform", 1 << 24, 32, 1, ("ell", "jds", "ss", "css"), {"css": {"n_block": 3}}, 1 << 21),
                                                 ("rmat", 23, 1 << 28, 42, ("crs", "csr5", "coo"), {}, None)):
        d = sp.DeviceCoo(kind, p0, p1, seed)
        n = d.nRow
        x_h = sp.reference_vectors(n, 0, 3)[0]
        x = torch.from_numpy(x_h).cuda()
        if rows is None:
            _, _, row, col, val = d.to_host()
            rows = n
        else:
            part = sp.DeviceCoo(kind, p0, p1, seed, 0, rows)
            _, _, row, col, val = part.to_host()
            part.free()
        y_ref = oracle.crs_result(rows, row, col, val, x_h)
        mag = np.bincount(row, weights=np.abs(val * x_h[col]), minlength=rows)[:rows]
        lens = np.bincount(row, minlength=rows)[:rows]
        del row, col, val
        for f in fmts:
            m = sp.SpMatOpt(f, **opts.get(f, {})).convert_device(d)
            if kind == "uniform" and f in ("ell", "jds", "ss"):
                assert m.scalar("col_blocks") == 3 and m.scalar("col_block_engine") == 1, f   # the gather-bound layout is what runs
            y = _mult(m, x, n)[:rows].cpu().numpy()
            m.destroy()
            err = np.abs(y - y_ref)
            assert np.all((err <= 1e-12 * np.abs(y_ref)) | (err <= 1e-12 * mag)), (kind, f, float(err.max()))
            if f in ("ell", "jds", "ss"):                                   # (crs on R-MAT: the entry stream, sums re-associated)
                short = lens <= 64
                assert np.array_equal(y[short], y_ref[short]), (kind, f)
        d.free()


# ------------------------------------------------------------------------------------------ beyond 2^31-1 entries on one GPU
@pytest.mark.parametrize("fmt", ["crs", "coo", "ell", "jds", "dia", "ss", "css", "csr5", "hyb"])
def test_row_blocked_matches_unblocked(sp, oracle, fmt, monkeypatch):
    """csrc/blocked.cu with the block size forced down (B200SPMV_BLOCK_NNZ): the row blocks a matrix of more than 2^31-1
    entries is cut into give the same y as the single matrix -- bit for bit, since rows are never split."""
    import torch
    cases_ = [oracle.stencil("lap3d7", 20), oracle.rmat(42, 11, 60000)] if fmt != "dia" else [oracle.stencil("lap3d7", 20)]
    for nr, nc, row, col, val in cases_:
        x = oracle.reference_vectors(nc, nr)[0]
        A = sp.SpMat(nr, nc, row, col, val)
        monkeypatch.delenv("B200SPMV_BLOCK_NNZ", raising=False)
        whole = sp.SpMatOpt(fmt).convert_host(A)
        monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(max(1000, len(row) // 5)))
        cut = sp.SpMatOpt(fmt).convert_host(A)
        monkeypatch.delenv("B200SPMV_BLOCK_NNZ", raising=False)
        assert cut.scalar("row_blocks") >= 4 and cut.scalar("nNnz") == len(row) and cut.scalar("nRow") == nr
        xd = torch.from_numpy(x).cuda()
        ys = []
        for m in (whole, cut):
            y = torch.full((nr,), float("nan"), dtype=torch.float64, device="cuda")
            m.multiply(xd.data_ptr(), y.data_ptr())
            torch.cuda.synchronize()
            ys.append(y.cpu().numpy())
        y_ref = oracle.crs_result(nr, row, col, val, x)
        assert_y(ys[1], y_ref, row, col, val, x, nr)
        if fmt in ("crs", "ell", "jds", "dia", "ss"):          # one thread per row of at most 64 entries either way
            short = np.bincount(row, minlength=nr) <= 64
            assert np.array_equal(ys[0][short], ys[1][short]), fmt
        if cut.scalar("has_rows"):
            y = torch.full((nr,), float("nan"), dtype=torch.float64, device="cuda")
            lo, hi = nr // 3, nr - nr // 7
            cut.multiply_rows(lo, hi, xd.data_ptr(), y.data_ptr())
            torch.cuda.synchronize()
            assert np.array_equal(y.cpu().numpy()[lo:hi], ys[1][lo:hi]) and bool(torch.isnan(y[:lo]).all()) and bool(torch.isnan(y[hi:]).all())
        whole.destroy()
        cut.destroy()


def test_more_than_int32_entries_on_one_gpu(sp):
    """2.6 G entries (uniform, 2^26 rows x 40): beyond the reference's int nNnz (src/util.h:8).  Checked through the
    closed form of A.1 (every row sums its own 40 values: compared with a block-wise recomputation from the COO
    arrays) and linearity."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 150 * (1 << 30):
        pytest.skip("needs ~120 GB of device memory")
    d = sp.DeviceCoo("uniform", 1 << 26, 40, 1)
    assert d.nNnz == (1 << 26) * 40 > 2 ** 31
    m = sp.SpMatOpt("crs").convert_device(d)
    assert m.scalar("nNnz") == d.nNnz and m.scalar("row_blocks") >= 2
    n = d.nRow
    ones = torch.ones(n, dtype=torch.float64, device="cuda")
    y1 = _mult(m, ones, n)
    # row sums straight from the COO values: rows have exactly 40 consecutive entries
    from singlespmv_b200.dist import _DevArray
    vals = torch.as_tensor(_DevArray(d.c.val_d, d.nNnz), device="cuda").view(n, 40)
    acc = torch.zeros(n, dtype=torch.float64, device="cuda")
    for k in range(40):                                        # ascending column order
        acc += vals[:, k]
    assert m.scalar("crs_kernel") == 3                         # gather-bound: the load-fed entry stream (sums re-associated)
    assert torch.allclose(y1, acc, rtol=1e-13, atol=0.0)
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    y = _mult(m, x, n)
    y2 = _mult(m, 2.0 * x, n)
    assert torch.equal(y2, 2.0 * y) and bool(torch.isfinite(y).all())
    m.destroy()
    d.free()


# ------------------------------------------------------------------------------------------ round 2 additions
def _short_row_matrix(rng, nRow, nCol, max_len):
    """Rows of 0..max_len entries (many empty, many full), sorted, duplicate-free."""
    rows, cols = [], []
    for r in range(nRow):
        k = rng.random()
        n = 0 if k < 0.15 else max_len if k < 0.4 else int(rng.integers(1, max_len + 1))
        c = np.sort(rng.choice(nCol, size=n, replace=False))
        rows.append(np.full(n, r))
        cols.append(c)
    row = np.concatenate(rows).astype(np.int32)
    col = np.concatenate(cols).astype(np.int32)
    return row, col, rng.standard_normal(len(row))


@pytest.mark.parametrize("max_len", [1, 5, 8, 9, 16])
def test_crs_short_row_kernels_bit_exact(sp, oracle, max_len):
    """The three CRS kernels that can take a short-row matrix -- tile-stream (crs_path=1), row-block stream (2), TMA-fed
    row-chunk stream (3, the default) -- all sum every row in the reference's order: bit-identical y, also on row
    ranges that start and end off the kernels' chunk / 16-byte boundaries, with empty rows and an empty tail."""
    import torch
    rng = np.random.default_rng(100 + max_len)
    nRow, nCol = 5003, 4097
    row, col, val = _short_row_matrix(rng, nRow, nCol, max_len)
    keep = row < nRow - 37                                   # trailing empty rows
    row, col, val = row[keep], col[keep], val[keep]
    x = rng.random(nCol)
    y_ref = oracle.crs_result(nRow, row, col, val, x)
    xd = torch.from_numpy(x).cuda()
    for path in (1, 2, 3, 0):
        for fmt in ("crs", "ss"):
            A_opt, y = run_host(sp, fmt, nRow, nCol, row, col, val, x, crs_path=path)
            assert np.array_equal(y, y_ref), (fmt, path)
            yd = torch.full((nRow,), float("nan"), dtype=torch.float64, device="cuda")
            cuts = [0, 3, 517, 518, 1031, 4000, nRow - 1, nRow]
            for a, b in zip(cuts[:-1], cuts[1:]):
                A_opt.multiply_rows(a, b, xd.data_ptr(), yd.data_ptr())
            torch.cuda.synchronize()
            assert np.array_equal(yd.cpu().numpy(), y_ref), (fmt, path, "ranges")
    A32, y32 = run_host(sp, "crs", nRow, nCol, row, col, val, x, value_f32=1, crs_path=3)
    _, y32_tile = run_host(sp, "crs", nRow, nCol, row, col, val, x, value_f32=1, crs_path=1)
    assert np.array_equal(y32, y32_tile)


def test_ell_dense_row_never_reads_past_x(sp):
    """ADVICE r1: the slots that round a slice up to the vector width used to carry col = k >= nCol when a row was
    (nearly) dense.  x lives in a buffer followed by NaNs: any gather past x[nCol-1] would poison y (0 * NaN)."""
    import torch
    for nRow, nCol in ((6, 5), (40, 7), (3, 1), (65, 33)):
        rows, cols = [np.full(nCol, 1)], [np.arange(nCol)]                # one dense row
        rows.append(np.array([0]))
        cols.append(np.array([nCol - 1]))
        order = np.lexsort((np.concatenate(cols), np.concatenate(rows)))
        row = np.concatenate(rows)[order].astype(np.int32)
        col = np.concatenate(cols)[order].astype(np.int32)
        val = np.arange(1, len(row) + 1, dtype=np.float64)
        A_opt = sp.SpMatOpt("ell").convert_host(sp.SpMat(nRow, nCol, row, col, val))
        assert A_opt.scalar("K") == nCol
        buf = torch.full((nCol + 64,), float("nan"), dtype=torch.float64, device="cuda")
        buf[:nCol] = torch.arange(1, nCol + 1, dtype=torch.float64)
        yd = torch.full((nRow,), float("nan"), dtype=torch.float64, device="cuda")
        A_opt.multiply(buf.data_ptr(), yd.data_ptr())
        torch.cuda.synchronize()
        y = yd.cpu().numpy()
        x = np.arange(1, nCol + 1, dtype=np.float64)
        y_ref = np.zeros(nRow)
        np.add.at(y_ref, row, val * x[col])
        assert np.all(np.isfinite(y)) and np.allclose(y, y_ref, rtol=1e-14), (nRow, nCol, y)
        lcol = A_opt.array("col_idx", np.int32).reshape(nRow, nCol)
        assert np.array_equal(lcol[2], np.arange(nCol))                   # empty row: padding col = k (opt_ell.cpp:48)


GUARD_FORMATS = [("crs", {}), ("crs", {"crs_path": 1}), ("crs", {"crs_path": 4}), ("coo", {"coo_path": 3}), ("coo", {"coo_path": 2}), ("coo", {"coo_path": 1}), ("ell", {}), ("jds", {}), ("dia", {}),
                 ("ss", {}), ("css", {"n_block": 3}), ("csr5", {}), ("hyb", {}), ("ell", {"col_blocks": 3}), ("jds", {"col_blocks": 2})]


@pytest.mark.parametrize("fmt,opt", GUARD_FORMATS)
def test_guard_bands_around_x_and_y(sp, oracle, fmt, opt):
    """Stand-in for compute-sanitizer memcheck (closed on this pool, profiles/r2_sanitizer.md): x lies between NaN bands and y
    between canary bands inside larger buffers.  A gather outside x poisons y, a store outside y breaks a canary."""
    import torch
    G = 4096
    mats = [oracle.stencil("lap3d7", 13), oracle.stencil("lap2d5", 37)]
    if fmt != "dia":
        mats += [oracle.rmat(7, 10, 30000), oracle.uniform(3, 3001, 2777, 9)]
    for nr, nc, row, col, val in mats:
        x = np.random.default_rng(nr).random(nc)
        y_ref = oracle.crs_result(nr, row, col, val, x)
        A = sp.SpMatOpt(fmt, **opt).convert_host(sp.SpMat(nr, nc, row, col, val))
        xb = torch.full((nc + 2 * G,), float("nan"), dtype=torch.float64, device="cuda")
        xb[G:G + nc] = torch.from_numpy(x).cuda()
        yb = torch.full((nr + 2 * G,), -12345.0, dtype=torch.float64, device="cuda")
        xp, yp = xb.data_ptr() + 8 * G, yb.data_ptr() + 8 * G
        for _ in range(2):
            A.multiply(xp, yp)
        torch.cuda.synchronize()
        assert bool((yb[:G] == -12345.0).all()) and bool((yb[G + nr:] == -12345.0).all()), (fmt, nr, "store outside y")
        y = yb[G:G + nr].cpu().numpy()
        assert np.all(np.isfinite(y)), (fmt, nr, "gather outside x")
        assert_y(y, y_ref, row, col, val, x, nr)
        if A.scalar("has_rows") and nr > 300:
            lo, hi = 129, nr - 77
            yb.fill_(-12345.0)
            A.multiply_rows(lo, hi, xp, yp)
            torch.cuda.synchronize()
            assert bool((yb[:G + lo] == -12345.0).all()) and bool((yb[G + hi:] == -12345.0).all()), (fmt, nr, "row range")
            assert np.array_equal(yb[G + lo:G + hi].cpu().numpy(), y[lo:hi])
        A.destroy()


@pytest.mark.parametrize("fmt,opt", [("crs", {}), ("crs", {"crs_path": 1}), ("css", {"n_block": 3}), ("ell", {}), ("dia", {}),
                                     ("ss", {})])
def test_host_multiply_pipeline_pinned(sp, oracle, fmt, opt):
    """Page-locked host vectors (b200spmv_host_register, what plugin/opt_b200.cpp does): x goes up in pieces, a row
    chunk starts when the pieces up to its largest column have landed, y comes back chunk by chunk.  Same bits as the
    device-resident multiply, also when x changes between calls."""
    nr, nc, row, col, val = oracle.stencil("lap2d5", 1100)
    x = oracle.reference_vectors(nc, nr)[0]
    A_opt = sp.SpMatOpt(fmt, **opt).convert_host(sp.SpMat(nr, nc, row, col, val))
    xs = x.copy()
    y = np.full(nr, np.nan)
    assert sp.host_register(xs) and sp.host_register(y)
    try:
        for x2 in (x, x[::-1].copy(), np.full(nc, 0.25), x * 3.0 + 1.0):
            xs[:] = x2
            y[:] = np.nan
            A_opt.multiply_host(xs, y)
            y_ref = oracle.crs_result(nr, row, col, val, x2)
            if fmt == "css":
                assert_y(y, y_ref, row, col, val, x2, nr)
            else:
                assert np.array_equal(y, y_ref)
    finally:
        sp.host_unregister(xs)
        sp.host_unregister(y)
    lo, hi = A_opt.col_extent(0, 32 * 1100)
    if fmt != "css":
        assert lo == 0 and 33 * 1100 - 1 <= hi <= 33 * 1100 + 31        # 5-point stencil: rows < 32 n reach column < 33 n
    else:
        assert (lo, hi) == (0, nc - 1)


def test_col_extent_random(sp, oracle):
    rng = np.random.default_rng(5)
    nRow, nCol = 700, 900
    row, col, val = skewed_matrix(rng, nRow, nCol, 9)
    for fmt in ("crs", "ss", "ell", "dia"):
        A_opt = sp.SpMatOpt(fmt).convert_host(sp.SpMat(nRow, nCol, row, col, val))
        for a, b in ((0, nRow), (10, 11), (100, 400), (699, 700), (5, 5)):
            sel = (row >= a) & (row < b)
            lo, hi = A_opt.col_extent(a, b)
            if sel.any():
                assert lo <= col[sel].min() and hi >= col[sel].max(), (fmt, a, b)
                if fmt in ("crs", "ss"):
                    assert (lo, hi) == (col[sel].min(), col[sel].max())
            elif fmt in ("crs", "ss"):
                assert hi < lo


def test_multiply_rows_in_cuda_graph_after_prepare(sp, oracle):
    """Tile-stream row ranges read two row pointers back on first use; prepare_rows does that ahead of time so the
    range can be captured, and an unprepared range inside a capture is refused instead of breaking the capture."""
    import torch
    nr, nc, row, col, val = oracle.stencil("box3d27", 14)
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    A_opt = sp.SpMatOpt("crs", crs_path=1).convert_host(sp.SpMat(nr, nc, row, col, val))
    assert A_opt.scalar("short_row_path") == 0
    xd = torch.from_numpy(x).cuda()
    yd = torch.full((nr,), float("nan"), dtype=torch.float64, device="cuda")
    cuts = [0, 700, 701, 2000, nr]
    for a, b in zip(cuts[:-1], cuts[1:]):
        A_opt.prepare_rows(a, b)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        s = torch.cuda.current_stream().cuda_stream
        for a, b in zip(cuts[:-1], cuts[1:]):
            A_opt.multiply_rows(a, b, xd.data_ptr(), yd.data_ptr(), s)
        with pytest.raises(sp.B200SpmvError) as e:
            A_opt.multiply_rows(5, 9, xd.data_ptr(), yd.data_ptr(), s)
        assert e.value.status == -4
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(yd.cpu().numpy(), y_ref)


def test_ss_css_profile_phases(sp, oracle):
    """options.profile with ss_faithful: the reference's PROF_BEGIN/END pairs (src/opt_ss.cpp:225-304) as CUDA events."""
    nr, nc, row, col, val = oracle.stencil("lap2d5", 300)
    x = oracle.reference_vectors(nc, nr)[0]
    for fmt, opt in (("ss", {"segment_width": 4}), ("css", {"segment_width": 4, "n_block": 2})):
        A_opt, y = run_host(sp, fmt, nr, nc, row, col, val, x, ss_faithful=1, profile=1, **opt)
        assert A_opt.scalar("MulTime_ns") > 0 and A_opt.scalar("SumTime_ns") > 0
        B_opt, y2 = run_host(sp, fmt, nr, nc, row, col, val, x, ss_faithful=1, **opt)
        assert np.array_equal(y, y2) and B_opt.scalar("MulTime_ns") == 0


@pytest.mark.parametrize("fmt", ["ell", "jds", "ss"])
def test_column_blocked_layout_bit_exact(sp, oracle, fmt):
    """options.col_blocks: the row-wise formats multiplied column block by column block (colblocks.cuh), each row's
    running sum continued from block to block -> same bits as the reference CRS result for any block count, empty rows
    included; the reference arrays the format exports are untouched."""
    rng = np.random.default_rng(31)
    mats = []
    nRow, nCol = 3001, 2500
    row, col, val = _short_row_matrix(rng, nRow, nCol, 24)
    mats.append((nRow, nCol, row, col, val, rng.random(nCol)))
    nr, nc, r_, c_, v_ = oracle.uniform(1, 4096, 4096, 32)
    mats.append((nr, nc, r_, c_, v_, oracle.reference_vectors(nc, nr)[0]))
    nr, nc, r_, c_, v_ = oracle.stencil("lap2d5", 50)
    mats.append((nr, nc, r_, c_, v_, oracle.reference_vectors(nc, nr)[0]))
    for nRow, nCol, row, col, val, x in mats:
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        base_opt, y0 = run_host(sp, fmt, nRow, nCol, row, col, val, x, col_blocks=-1)
        assert base_opt.scalar("col_blocks") == 0 and np.array_equal(y0, y_ref)
        for nb in (1, 2, 3, 7):
            A_opt, y = run_host(sp, fmt, nRow, nCol, row, col, val, x, col_blocks=nb)
            assert A_opt.scalar("col_blocks") >= 1 and A_opt.scalar("launches") >= A_opt.scalar("col_blocks")
            assert np.array_equal(y, y_ref), (fmt, nb)
            assert A_opt.scalar("alg_bytes") == base_opt.scalar("alg_bytes")
        auto_opt, _ = run_host(sp, fmt, nRow, nCol, row, col, val, x)
        assert auto_opt.scalar("col_blocks") == 0             # x fits in L2: the decision leaves small matrices alone


@pytest.mark.parametrize("fmt", ["ell", "jds", "ss"])
def test_column_block_engines(sp, oracle, fmt, monkeypatch):
    """The two column-block engines (colblocks.cuh): one sliced ELL per column block (default while the padding stays below
    two slots per entry) and the tile-stream per block.  Both continue every row's sum from block to block: same bits."""
    nr, nc, row, col, val = oracle.uniform(5, 6000, 6000, 32)
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    monkeypatch.delenv("B200SPMV_COL_BLOCK_ENGINE", raising=False)
    A1, y1 = run_host(sp, fmt, nr, nc, row, col, val, x, col_blocks=3)
    assert A1.scalar("col_block_engine") == 1 and A1.scalar("col_blocks") == 3
    monkeypatch.setenv("B200SPMV_COL_BLOCK_ENGINE", "crs")
    A2, y2 = run_host(sp, fmt, nr, nc, row, col, val, x, col_blocks=3)
    monkeypatch.delenv("B200SPMV_COL_BLOCK_ENGINE", raising=False)
    assert A2.scalar("col_block_engine") == 2
    assert np.array_equal(y1, y_ref) and np.array_equal(y2, y_ref)
    if fmt == "ss":
        # CSS itself on a gather-bound matrix: the same ELL blocks with the block sums ADDED (src/opt_css.cpp:298): same
        # association as its tile-stream path, within the tolerance of the CRS order
        C1, z1 = run_host(sp, "css", nr, nc, row, col, val, x, n_block=3, segment_width=4)
        assert C1.scalar("col_block_engine") == 1
        monkeypatch.setenv("B200SPMV_COL_BLOCK_ENGINE", "crs")
        C2, z2 = run_host(sp, "css", nr, nc, row, col, val, x, n_block=3, segment_width=4)
        monkeypatch.delenv("B200SPMV_COL_BLOCK_ENGINE", raising=False)
        assert C2.scalar("col_block_engine") == 2 and np.array_equal(z1, z2)
        assert_y(z1, y_ref, row, col, val, x, nr)
    # a skewed matrix would need far more than two slots per entry: the tile-stream engine takes it
    nr, nc, row, col, val = oracle.rmat(42, 12, 120000)
    x = oracle.reference_vectors(nc, nr)[0]
    A3, y3 = run_host(sp, fmt, nr, nc, row, col, val, x, col_blocks=2)
    assert A3.scalar("col_block_engine") == 2
    assert_y(y3, oracle.crs_result(nr, row, col, val, x), row, col, val, x, nr)


def test_column_blocked_long_rows_within_tolerance(sp, oracle, all_cases):
    """Rows with more than 64 entries in one column block are reduced by a warp: within the 1e-12 tolerance; every
    other row stays bit-identical."""
    for name, nRow, nCol, row, col, val, x in all_cases:
        if nCol < 4:
            continue
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        A_opt, y = run_host(sp, "jds", nRow, nCol, row, col, val, x, col_blocks=2)
        assert_y(y, y_ref, row, col, val, x, nRow)
        short = np.diff(np.searchsorted(row, np.arange(nRow + 1))) <= 64
        assert np.array_equal(y[short], y_ref[short]), name


@pytest.mark.parametrize("kind,n,maxlen", [("box3d27", 14, 27), ("lap3d7", 20, 7)])
def test_css_blocks_on_row_chunk_stream(sp, oracle, kind, n, maxlen):
    """CSS column blocks with short rows go through the row-chunk stream (block sums ADDED to y, src/opt_css.cpp:298);
    result within the tolerance of the reference CRS result and equal to the tile-stream path's association."""
    nr, nc, row, col, val = oracle.stencil(kind, n)
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    for nb in (1, 2, 4):
        A_opt, y = run_host(sp, "css", nr, nc, row, col, val, x, n_block=nb, segment_width=4)
        assert_y(y, y_ref, row, col, val, x, nr)
        if nb == 1:
            assert np.array_equal(y, y_ref)


# ------------------------------------------------------------------------------------------ fp32 variant (SURVEY.md 8f-3)
@pytest.mark.parametrize("fmt", ["crs", "ell", "dia", "csr5"])
@pytest.mark.parametrize("precision", [1, 2])
def test_fp32_variant(sp, oracle, all_cases, fmt, precision):
    """options.precision: fp32 matrix values, fp32 x and y; sums in fp32 (1) or fp64 (2).  BASELINE.json's bar: within 1e-5
    of the reference's (fp64) CRS result per row, relative to |y_ref| or to sum_j |a_ij x_j|.  With fp64 sums only the
    rounding of the inputs remains (<= 1.2e-7); with fp32 sums a row of n entries may drift by n * 2^-24, so rows of
    more than 64 entries get the bound their length implies."""
    import torch
    for name, nRow, nCol, row, col, val, x in all_cases:
        lens = np.bincount(row, minlength=nRow) if len(row) else np.zeros(nRow, np.int64)
        K = int(lens.max()) if nRow else 0
        if fmt == "ell" and (K > nCol or K * nRow > 5e7):
            continue
        if fmt == "dia" and len(row) and len(np.unique(col.astype(np.int64) - row)) * nCol > 3e7:
            continue
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        mag = np.zeros(nRow)
        np.add.at(mag, row, np.abs(val * x[col]))
        A_opt = sp.SpMatOpt(fmt, precision=precision).convert_host(sp.SpMat(nRow, nCol, row, col, val))
        assert A_opt.scalar("precision") == precision
        if fmt == "crs":
            assert A_opt.scalar("alg_bytes") == 8 * len(row) + 4 * (nRow + 1) + 4 * nCol + 4 * nRow
            assert np.array_equal(A_opt.array("val", np.float64), val.astype(np.float32).astype(np.float64))
        x32 = x.astype(np.float32)
        y32 = np.full(nRow, np.nan, np.float32)
        A_opt.multiply_host_f32(x32, y32)
        xd = torch.from_numpy(x32).cuda()
        yd = torch.full((max(nRow, 1),), float("nan"), dtype=torch.float32, device="cuda")
        A_opt.multiply_f32(xd.data_ptr(), yd.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(yd.cpu().numpy()[:nRow], y32), name        # host-semantics = device-resident
        assert np.all(np.isfinite(y32)), name
        err = np.abs(y32.astype(np.float64) - y_ref)
        tol = np.full(nRow, 1e-5)
        if precision == 1:
            tol = np.maximum(tol, lens * 2.0 ** -23)
        if fmt == "csr5" and precision == 1:
            tol = np.maximum(tol, 3e-7 * np.sqrt(np.maximum(lens, 1)))      # fp32 segment sums; precision 2 rounds once
        ok = (err <= tol * np.abs(y_ref)) | (err <= tol * mag)
        assert np.all(ok), (name, int((~ok).sum()), float(np.max(err / np.maximum(mag, 1e-300))))
        with pytest.raises(sp.B200SpmvError) as e:                        # fp64 entry on an fp32 handle
            A_opt.multiply_host(x, np.empty(nRow))
        assert e.value.status == -4 or nRow == 0
    plain = sp.SpMatOpt(fmt).convert_host(sp.SpMat(3, 3, np.array([0], np.int32), np.array([1], np.int32), np.array([1.0])))
    with pytest.raises(sp.B200SpmvError) as e:
        plain.multiply_host_f32(np.ones(3, np.float32), np.ones(3, np.float32))
    assert e.value.status == -4
    with pytest.raises(sp.B200SpmvError) as e:
        sp.SpMatOpt("jds", precision=1)
    assert e.value.status == -3


def test_fp32_full_size_c5(sp):
    """Config 5 at full size in fp32: A.1 row sums are small integers (exact in fp32), so the result must be exact."""
    import torch
    d = sp.DeviceCoo("lap3d7", 256)
    n = d.nRow
    for fmt in ("crs", "ell", "dia"):
        A = sp.SpMatOpt(fmt, precision=1).convert_device(d)
        x = torch.ones(n, dtype=torch.float32, device="cuda")
        y = torch.full((n,), float("nan"), dtype=torch.float32, device="cuda")
        A.multiply_f32(x.data_ptr(), y.data_ptr())
        torch.cuda.synchronize()
        B = sp.SpMatOpt(fmt).convert_device(d)
        x64 = torch.ones(n, dtype=torch.float64, device="cuda")
        y64 = torch.empty(n, dtype=torch.float64, device="cuda")
        B.multiply(x64.data_ptr(), y64.data_ptr())
        torch.cuda.synchronize()
        assert torch.equal(y.double(), y64), fmt
        A.destroy()
        B.destroy()
    d.free()


# ------------------------------------------------------------------------------------------ one process, several GPUs (b200spmv_mg_*)
def _mg_counts(sp):
    n = sp.device_count()
    return [g for g in (1, 2, 3, 4, 8) if g <= n]


@pytest.mark.parametrize("fmt", ["crs", "ell", "jds"])
def test_mg_matches_single_gpu(sp, oracle, fmt):
    """b200spmv_mg_*: any host COO is split by non-zero balance over the GPUs of the box (as many as are visible; one
    on the driver's box, where the path degenerates to a single block without halo), columns renumbered monotonically
    -> y bit-identical to the single-GPU result of the same format and to the reference CRS result, through the host
    entry, the device-resident entries and repeated (graph-launched) steps."""
    from singlespmv_b200.mg import MgSpMat
    mats = []
    nr, nc, row, col, val = oracle.stencil("lap3d7", 30)
    mats.append(("lap3d7", nr, nc, row, col, val))
    nr, nc, row, col, val = oracle.rmat(42, 12, 90000)                   # halo = most of x: the all-gather-like case
    mats.append(("rmat", nr, nc, row, col, val))
    rng = np.random.default_rng(3)
    row, col, val = skewed_matrix(rng, 3000, 3000, 9)                    # empty rows, long rows
    mats.append(("skew", 3000, 3000, row, col, val))
    for name, nRow, nCol, row, col, val in mats:
        x = oracle.reference_vectors(nCol, nRow)[0]
        y_ref = oracle.crs_result(nRow, row, col, val, x)
        if fmt == "ell" and name != "lap3d7":
            continue
        _, y1 = run_host(sp, fmt, nRow, nCol, row, col, val, x)
        for g in _mg_counts(sp):
            M = MgSpMat(g, fmt).convert_host(sp.SpMat(nRow, nCol, row, col, val))
            b = M.bounds()
            assert b[0] == 0 and b[-1] == nRow and np.all(np.diff(b) >= 0)
            assert M.scalar("nNnz") == len(row) and M.scalar("nGPU") == g
            y = np.full(nRow, np.nan)
            M.multiply_host(x, y)
            short = np.diff(np.searchsorted(row, np.arange(nRow + 1))) <= 64
            assert np.array_equal(y[short], y_ref[short]), (name, g)
            assert_y(y, y_ref, row, col, val, x, nRow)
            if name == "lap3d7":                                     # rows of one thread each: partitioning cannot change a bit
                assert np.array_equal(y, y1), (name, g)
            x2 = x[::-1].copy()
            M.upload_x(x2)
            for _ in range(3):
                M.multiply()
            y2 = np.full(nRow, np.nan)
            M.download_y(y2)
            assert_y(y2, oracle.crs_result(nRow, row, col, val, x2), row, col, val, x2, nRow)
            if g > 1:
                assert M.scalar("halo_total") > 0
            M.destroy()


def test_mg_synthetic_blocks(sp, oracle):
    from singlespmv_b200.mg import MgSpMat
    nr, nc, row, col, val = oracle.stencil("box3d27", 20)
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    for g in _mg_counts(sp):
        M = MgSpMat(g, "crs").convert_synth("box3d27", 20)
        y = np.full(nr, np.nan)
        M.multiply_host(x, y)
        assert np.array_equal(y, y_ref), g
        assert M.scalar("alg_bytes") == 12 * len(row) + 4 * (nr + g) + 16 * nr
        M.destroy()
    with pytest.raises(sp.B200SpmvError):
        MgSpMat(64, "crs")                                               # more GPUs than the box has
