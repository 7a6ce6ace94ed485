"""CPU tests of the test infrastructure itself: the C restatement (oracle/spmv_oracle.c) must
reproduce, bit for bit, what the reference's own plugins produced on the committed golden
vectors (tests/golden/, made by make_golden.py from the unmodified reference)."""
import numpy as np
import pytest

from conftest import golden_names, load_golden

GOLD = golden_names()


def _inputs(g):
    return int(g["nRow"]), int(g["nCol"]), g["in_row"], g["in_col"], g["in_val"], g["x"]


def test_golden_present():
    assert len(GOLD) >= 9


def test_appendix_b_known_answers():
    """SURVEY.md Appendix B: values printed by the reference for matrix/test/10x10.mtx and 5x5.mtx."""
    g = load_golden("fixture_10x10")
    assert g["crs.ptr"].tolist() == [0, 6, 8, 14, 16, 17, 19, 27, 27, 27, 27]
    assert g["jds.ptr"].tolist() == [0, 7, 13, 16, 19, 22, 25, 26, 27]
    assert g["jds.length"].tolist() == [6, 2, 6, 2, 1, 2, 8, 0, 0, 0]
    assert g["ss_opt_w2.segment_index"].tolist() == [0, 1, 2, 0, 0, 1, 2, 0, 0, 0, 0, 1, 2, 0]
    assert g["ss_opt_w2.sum_segs"].tolist() == [2, 6, 12, 1, 5, 11]
    np.testing.assert_allclose(g["crs.y"][:3], [2.0532159628594369, 1.572726975927468, 6.159647888578311],
                               rtol=0, atol=0)
    np.testing.assert_allclose(g["x"][:3], [0.56138017520372763, 0.22498331276000633, 0.39309177938527046],
                               rtol=0, atol=0)
    g5 = load_golden("fixture_5x5")
    assert g5["dia.ioff"].tolist() == [4, 5, 6]
    assert g5["dia.diag"].reshape(3, 5).tolist() == [[0, 0, 0, 1, 0], [0, 1, 0, 0, 0], [0, 0, 1, 1, 1]]


@pytest.mark.parametrize("name", GOLD)
def test_reference_vectors(oracle, name):
    g = load_golden(name)
    x, _ = oracle.reference_vectors(int(g["nCol"]), int(g["nRow"]), 3)
    assert np.array_equal(x, g["x"])


@pytest.mark.parametrize("name", GOLD)
def test_crs_coo(oracle, name):
    g = load_golden(name)
    nRow, nCol, row, col, val, x = _inputs(g)
    m = oracle.crs_convert(nRow, row, col, val)
    for k in ("ptr", "idx", "val"):
        assert np.array_equal(m[k], g["crs." + k]), k
    assert np.array_equal(oracle.crs_spmv(m, x), g["crs.y"])
    # COO: the reference scatters with omp atomic (order free); serial order == CRS order
    assert np.array_equal(oracle.coo_spmv(nRow, row, col, val, x), g["crs.y"])
    np.testing.assert_allclose(g["coo.y"], g["crs.y"], rtol=1e-13, atol=1e-300)


@pytest.mark.parametrize("name", GOLD)
def test_ell(oracle, name):
    g = load_golden(name)
    nRow, nCol, row, col, val, x = _inputs(g)
    m = oracle.ell_convert(nRow, row, col, val)
    assert m["K"] == int(g["ell.K"])
    assert np.array_equal(m["col_idx"].ravel(), g["ell.col_idx"])
    assert np.array_equal(m["val"].ravel(), g["ell.val"])
    assert np.array_equal(oracle.ell_spmv(m, x), g["ell.y"])


@pytest.mark.parametrize("name", GOLD)
def test_jds(oracle, name):
    g = load_golden(name)
    nRow, nCol, row, col, val, x = _inputs(g)
    # reference tie order (its std::sort is unstable): take perm from the reference run
    m = oracle.jds_convert(nRow, row, col, val, perm_in=g["jds.perm"])
    assert m["maxLength"] == int(g["jds.maxLength"])
    for k in ("perm", "length", "ptr", "col_idx", "val"):
        assert np.array_equal(m[k], g["jds." + k]), k
    assert np.array_equal(oracle.jds_spmv(m, x), g["jds.y"])
    # documented stable convention: same lengths/ptr, perm equal up to ties, same y
    s = oracle.jds_convert(nRow, row, col, val)
    assert np.array_equal(s["ptr"], g["jds.ptr"]) and np.array_equal(s["length"], g["jds.length"])
    assert np.array_equal(s["length"][s["perm"]], g["jds.length"][g["jds.perm"]])
    assert sorted(s["perm"].tolist()) == list(range(nRow))
    assert np.array_equal(oracle.jds_spmv(s, x), g["jds.y"])


@pytest.mark.parametrize("name", GOLD)
def test_dia(oracle, name):
    g = load_golden(name)
    nRow, nCol, row, col, val, x = _inputs(g)
    m = oracle.dia_convert(nRow, nCol, row, col, val)
    assert m["nDiag"] == int(g["dia.nDiag"])
    assert np.array_equal(m["ioff"], g["dia.ioff"])
    assert np.array_equal(m["diag"].ravel(), g["dia.diag"])
    assert np.array_equal(oracle.dia_spmv(m, x), g["dia.y"])


@pytest.mark.parametrize("name", GOLD)
@pytest.mark.parametrize("variant,W,mode", [("ss_simple_w4", 4, "simple"), ("ss_opt_w2", 2, "optimized"),
                                            ("ss_opt_w4", 4, "optimized"), ("ss_opt_w32", 32, "optimized")])
def test_ss(oracle, name, variant, W, mode):
    g = load_golden(name)
    nRow, nCol, row, col, val, x = _inputs(g)
    m = oracle.ss_convert(nRow, row, col, val, W)
    assert m["H"] == int(g[variant + ".H"]) and m["nStep"] == int(g[variant + ".nStep"])
    for k in ("row_ptr", "row_idx", "col_idx", "val", "segment_index", "sum_segs_count", "sum_segs"):
        assert np.array_equal(m[k], g["%s.%s" % (variant, k)]), k
    assert np.array_equal(oracle.ss_spmv(m, x, mode), g[variant + ".y"])


@pytest.mark.parametrize("name", GOLD)
@pytest.mark.parametrize("variant,W,N", [("css_opt_w2_n2", 2, 2), ("css_opt_w4_n3", 4, 3),
                                         ("css_opt_w32_n4", 32, 4)])
def test_css(oracle, name, variant, W, N):
    g = load_golden(name)
    nRow, nCol, row, col, val, x = _inputs(g)
    m = oracle.css_convert(nRow, nCol, row, col, val, W, N)
    for k in ("B", "nBlock", "totalH"):
        assert m[k] == int(g["%s.%s" % (variant, k)]), k
    for k in ("H", "nStep", "row_ptr", "col_idx", "val", "sum_segs_count", "sum_segs"):
        assert np.array_equal(m[k], g["%s.%s" % (variant, k)]), k
    assert np.array_equal(oracle.css_spmv(m, x), g[variant + ".y"])


CSR5_KEYS = ("tile_desc", "tile_desc_offset_ptr", "tile_desc_offset", "col_idx", "val")


def _csr5_same(a, b):
    p = a["p"]
    for k in ("p", "bit_y_offset", "bit_scansum_offset", "num_packet", "num_offsets"):
        assert int(a[k]) == int(b[k]), k
    ta, tb = np.array(a["tile_ptr"], np.uint32), np.array(b["tile_ptr"], np.uint32)
    if p > 0:        # the dirty bit of the tail tile depends on an out-of-bounds read upstream (format_avx2.h:48-55)
        ta[p - 1:] &= 0x7FFFFFFF
        tb[p - 1:] &= 0x7FFFFFFF
    assert np.array_equal(ta, tb), "tile_ptr"
    for k in CSR5_KEYS:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("name", GOLD)
@pytest.mark.parametrize("sigma", [4, 16])
def test_csr5(oracle, name, sigma):
    g = load_golden(name)
    nRow, nCol, row, col, val, x = _inputs(g)
    m = oracle.csr5_convert(nRow, row, col, val, sigma)
    ref = {k[len("csr5_s%d." % sigma):]: g[k] for k in g if k.startswith("csr5_s%d." % sigma)}
    _csr5_same(m, ref)
    y = oracle.csr5_spmv(m, x)
    np.testing.assert_allclose(y, g["crs.y"], rtol=1e-12, atol=1e-14)


def test_csr5_auto_sigma(oracle):
    # CSR5_cuda/anonymouslib_cuda.h:293-317
    assert [oracle.csr5_auto_sigma(10, n) for n in (0, 40, 50, 320, 330, 2560, 2570)] == [4, 4, 5, 32, 32, 32, 6]
