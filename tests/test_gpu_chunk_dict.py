"""The row-chunk stream's offset-dictionary feed (chunk_stream.cuh): every chunk of th rows stores its distinct col - row
offsets once (at most 16) and each row a bitmask of them.  A handle takes that feed (chunk_feed = 1) when every chunk fits
16 offsets, else the idx / ptr feed (chunk_feed = 0).  Either way every row is summed in ascending column order, so y must
carry the bits of the sequential CRS result, on whole multiplies and on row ranges.  B200SPMV_CS_FEED=idx forces the
old feed; B200SPMV_TMA_R=512 makes chunks of 512 rows."""
import numpy as np
import pytest

from test_gpu_fp32 import Case, same_bits

pytestmark = pytest.mark.gpu

G = 4096                                   # guard band, entries
CANARY = -12345.0
OFFS = np.array([-90, -77, -64, -41, -30, -17, -5, -1, 0, 1, 6, 19, 33, 52, 70, 90])    # 16 offsets


@pytest.fixture(scope="module")
def sp():
    import singlespmv_b200 as m
    assert m.device_count() > 0, "GPU tests need a CUDA device"
    return m


@pytest.fixture(params=[256, 512], ids=["th256", "th512"])
def th(request, monkeypatch):
    monkeypatch.setenv("B200SPMV_TMA_R", str(request.param))
    return request.param


def convert(sp, fmt, nr, nc, row, col, val, **opt):
    return sp.SpMatOpt(fmt, **opt).convert_host(sp.SpMat(nr, nc, row.astype(np.int32), col.astype(np.int32), val))


def guarded(A, nr, nc, x, rows=None):
    """multiply (or multiply_rows over rows) with x between NaN bands and y between canary bands; y outside the rows
    stays NaN."""
    import torch
    xb = torch.full((nc + 2 * G,), float("nan"), dtype=torch.float64, device="cuda")
    xb[G:G + nc] = torch.from_numpy(x).cuda()
    yb = torch.full((nr + 2 * G,), CANARY, dtype=torch.float64, device="cuda")
    yb[G:G + nr] = float("nan")
    xp, yp = xb.data_ptr() + 8 * G, yb.data_ptr() + 8 * G
    for _ in range(2):
        if rows is None:
            A.multiply(xp, yp)
        else:
            for a, b in rows:
                A.multiply_rows(a, b, xp, yp)
    torch.cuda.synchronize()
    yb = yb.cpu().numpy()
    assert np.all(yb[:G] == CANARY) and np.all(yb[G + nr:] == CANARY), "store outside y"
    return yb[G:G + nr]


def check_feed(sp, oracle, fmt, nr, nc, row, col, val, feed, cuts=None, **opt):
    """fmt's y (whole multiply, and row ranges between consecutive cuts) against the sequential CRS result, bit for bit,
    and the feed the handle took."""
    x = np.random.default_rng(nr).uniform(-1.0, 1.0, nc)
    y_ref = oracle.crs_result(nr, row, col, val, x)
    A = convert(sp, fmt, nr, nc, row, col, val, **opt)
    assert A.scalar("short_row_path") == 1 and A.scalar("chunk_feed") == feed, (fmt, opt, A.scalar("chunk_feed"))
    if fmt == "crs":
        assert A.scalar("crs_kernel") == 1 and A.scalar("launches") == 1
    assert np.array_equal(guarded(A, nr, nc, x), y_ref), (fmt, opt, "multiply")
    cuts = cuts if cuts is not None else [0, 3, 255, 256, 257, 517, 518, 1031, nr - 1, nr]
    cuts = sorted({min(c, nr) for c in cuts})
    y = guarded(A, nr, nc, x, list(zip(cuts[:-1], cuts[1:])))
    assert np.array_equal(y, y_ref), (fmt, opt, "ranges")
    a, b = min(129, nr), max(min(129, nr), nr - 77)                    # one range: NaN before and after it
    y = guarded(A, nr, nc, x, [(a, b)])
    assert np.all(np.isnan(y[:a])) and np.all(np.isnan(y[b:])) and np.array_equal(y[a:b], y_ref[a:b]), (fmt, opt, "range")
    A.destroy()
    return y_ref


def dict_matrix(nr, seed, extra=(), empty_chunks=(), tail=37, th=256):
    """Rows r with columns r + OFFS[j] for a random subset of j (clipped to [0, nr)): every chunk of th rows uses all 16
    offsets (rows 100 + j of a chunk take offset j), rows of 16 and of 1 entry, empty rows, empty chunks and an empty tail.
    extra: (row, offset) entries added on top (a 17th offset where wanted)."""
    rng = np.random.default_rng(seed)
    pick = rng.random((nr, 16)) < 0.45
    pick[rng.random(nr) < 0.1] = False                                  # empty rows
    full = rng.random(nr) < 0.1
    pick[full] = True                                                   # rows of 16 entries
    one = rng.random(nr) < 0.1
    pick[one] = False
    pick[one, rng.integers(0, 16, one.sum())] = True                    # rows of 1 entry
    r = np.arange(nr)
    for j in range(16):
        pick[(r % th) == 100 + j, j] = True
    for c in empty_chunks:
        pick[c * th:(c + 1) * th] = False
    pick[nr - tail:] = False
    pick[90, 0] = pick[nr - 91, 15] = True                              # columns 0 and nr - 1
    rows, cols = np.nonzero(pick)
    cols = rows + OFFS[cols]
    for rr, off in extra:
        rows, cols = np.append(rows, rr), np.append(cols, rr + off)
    keep = (cols >= 0) & (cols < nr)
    rows, cols = rows[keep], cols[keep]
    order = np.lexsort((cols, rows))
    rows, cols = rows[order], cols[order]
    assert cols.min() == 0 and cols.max() == nr - 1                      # offsets reach both ends of x
    return rows.astype(np.int32), cols.astype(np.int32), rng.standard_normal(len(rows))


# ------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("kind,n", [("lap2d5", 37), ("lap3d7", 13), ("lap3d7", 19)])
def test_stencils_take_the_dictionary(sp, oracle, th, kind, n):
    """Stencils whose row count is no multiple of 256 or 512: CRS and SS on the dictionary feed, bit-identical."""
    nr, nc, row, col, val = oracle.stencil(kind, n)
    assert nr % 256
    for fmt in ("crs", "ss"):
        check_feed(sp, oracle, fmt, nr, nc, row, col, val, 1)


def test_forced_idx_feed(sp, oracle, monkeypatch):
    """B200SPMV_CS_FEED=idx: the same stencil on the idx feed, the same bits."""
    nr, nc, row, col, val = oracle.stencil("lap3d7", 13)
    monkeypatch.setenv("B200SPMV_CS_FEED", "idx")
    for fmt in ("crs", "ss"):
        check_feed(sp, oracle, fmt, nr, nc, row, col, val, 0)


def test_sixteen_offsets_and_overflow(sp, oracle, th):
    """16 distinct offsets per chunk, empty rows and chunks, rows of 1 and 16 entries: the dictionary.  A 17th offset in
    one chunk, or only in the last chunk: the whole handle keeps the idx feed, with the same bits."""
    nr = 3 * th + 201
    row, col, val = dict_matrix(nr, 7, empty_chunks=(1,), th=th)
    lens = np.bincount(row, minlength=nr)
    assert lens.max() == 16 and (lens == 1).any() and (lens[th:2 * th] == 0).all()
    for fmt in ("crs", "ss"):
        check_feed(sp, oracle, fmt, nr, nr, row, col, val, 1)
    for extra in ([(5, 3)], [(nr - 40, -2)]):                           # the first chunk, the last chunk
        row, col, val = dict_matrix(nr, 7, extra=extra, empty_chunks=(1,), th=th)
        for fmt in ("crs", "ss"):
            check_feed(sp, oracle, fmt, nr, nr, row, col, val, 0)
    row, col, val = dict_matrix(nr, 8, extra=[(2 * th + 130, 2)], th=th)
    check_feed(sp, oracle, "crs", nr, nr, row, col, val, 0)


def test_short_random_rows_keep_the_idx_feed(sp, oracle):
    """Random short rows (those of test_crs_short_row_kernels_bit_exact) overflow the dictionary."""
    from test_gpu_parity import _short_row_matrix
    rng = np.random.default_rng(5)
    row, col, val = _short_row_matrix(rng, 3001, 4097, 9)
    check_feed(sp, oracle, "crs", 3001, 4097, row, col, val, 0)


@pytest.mark.parametrize("prec", [1, 2])
def test_fp32_precisions(sp, oracle, prec):
    """precision 1 and 2 on the dictionary feed: the bits of the exact fp32 / fp64 sequential sums (test_gpu_fp32.seq)."""
    import torch
    for name, (nr, nc, row, col, val) in (("lap3d7", oracle.stencil("lap3d7", 17)), ("dict", (1001, 1001) + dict_matrix(1001, 9))):
        c = Case(name, nr, nc, row, col, val, np.random.default_rng(nr).uniform(-1.0, 1.0, nc))
        A = convert(sp, "crs", nr, nc, c.row, c.col, c.val, precision=prec)
        assert A.scalar("chunk_feed") == 1 and A.scalar("crs_kernel") == 1, name
        xb = torch.full((nc + 2 * G,), float("nan"), dtype=torch.float32, device="cuda")
        xb[G:G + nc] = torch.from_numpy(c.x32).cuda()
        yb = torch.full((nr + 2 * G,), CANARY, dtype=torch.float32, device="cuda")
        A.multiply_f32(xb.data_ptr() + 4 * G, yb.data_ptr() + 4 * G)
        torch.cuda.synchronize()
        yb = yb.cpu().numpy()
        assert np.all(yb[:G] == np.float32(CANARY)) and np.all(yb[G + nr:] == np.float32(CANARY)), name
        assert np.all(same_bits(yb[G:G + nr], c.seq[prec])), (name, prec)
        A.destroy()


def test_value_f32(sp, oracle):
    """fp32 value storage: the fp64 result of the rounded matrix, bit for bit."""
    for nr, nc, row, col, val in (oracle.stencil("lap2d5", 41), (1001, 1001) + dict_matrix(1001, 10)):
        v32 = val.astype(np.float32).astype(np.float64)
        y_ref = check_feed(sp, oracle, "crs", nr, nc, row, col, v32, 1, value_f32=1)
        x = np.random.default_rng(nr).uniform(-1.0, 1.0, nc)
        A = convert(sp, "crs", nr, nc, row, col, val, value_f32=1)
        assert A.scalar("chunk_feed") == 1 and np.array_equal(guarded(A, nr, nc, x), y_ref)
        A.destroy()


def test_css_and_ss_blocks(sp, oracle, monkeypatch):
    """CSS on a stencil: its column blocks run the row-chunk stream (the first overwrites y, the others add), on the
    dictionary feed: the same bits as with the idx feed forced, and the host pipeline gives them too."""
    nr, nc, row, col, val = oracle.stencil("lap3d7", 17)
    x = np.random.default_rng(3).uniform(-1.0, 1.0, nc)
    y_ref = oracle.crs_result(nr, row, col, val, x)
    ys = {}
    for feed in ("dict", "idx"):
        if feed == "idx":
            monkeypatch.setenv("B200SPMV_CS_FEED", "idx")
        A = convert(sp, "css", nr, nc, row, col, val, n_block=3)
        assert A.scalar("nBlock") == 3 and A.scalar("col_block_engine") == 0
        assert A.scalar("chunk_feed") == (1 if feed == "dict" else 0)
        ys[feed] = guarded(A, nr, nc, x)
        yr = guarded(A, nr, nc, x, [(0, 300), (300, 1031), (1031, nr)])
        assert np.array_equal(yr, ys[feed])
        yh = np.full(nr, np.nan)
        A.multiply_host(x, yh)
        assert np.array_equal(yh, ys[feed])
        A.destroy()
    monkeypatch.delenv("B200SPMV_CS_FEED")
    assert np.array_equal(ys["dict"], ys["idx"])
    assert np.allclose(ys["dict"], y_ref, rtol=1e-13, atol=1e-13)


def test_host_pipeline(sp, oracle):
    """multiply_host (x up in pieces, row chunks as their columns land) on the dictionary feed: the sequential bits."""
    nr, nc, row, col, val = oracle.stencil("lap2d5", 1100)
    x = oracle.reference_vectors(nc, nr)[0]
    y_ref = oracle.crs_result(nr, row, col, val, x)
    for fmt in ("crs", "ss"):
        A = convert(sp, fmt, nr, nc, row, col, val)
        assert A.scalar("chunk_feed") == 1
        y = np.full(nr, np.nan)
        A.multiply_host(x, y)
        assert np.array_equal(y, y_ref), fmt
        A.destroy()


def test_row_blocks(sp, oracle, monkeypatch):
    """Forced row blocks (B200SPMV_BLOCK_NNZ): every block an ordinary handle on the dictionary feed."""
    nr, nc, row, col, val = oracle.stencil("lap3d7", 21)
    monkeypatch.setenv("B200SPMV_BLOCK_NNZ", str(len(row) // 5))
    for fmt in ("crs", "ss"):
        x = np.random.default_rng(nr).uniform(-1.0, 1.0, nc)
        A = convert(sp, fmt, nr, nc, row, col, val)
        assert A.scalar("row_blocks") >= 5 and A.scalar("chunk_feed") == 1
        assert np.array_equal(guarded(A, nr, nc, x), oracle.crs_result(nr, row, col, val, x)), fmt
        cuts = [0, 1, 700, 2049, nr // 2, nr - 300, nr]
        assert np.array_equal(guarded(A, nr, nc, x, list(zip(cuts[:-1], cuts[1:]))), oracle.crs_result(nr, row, col, val, x))
        A.destroy()


@pytest.mark.parametrize("parts", [2, 3])
def test_partitioned_blocks(sp, oracle, parts):
    """The row-partitioned blocks of the multi-GPU path (halo-renumbered columns), all on one GPU: every block on the
    dictionary feed, y the sequential bits."""
    import torch
    import singlespmv_b200.dist as spd
    n = 24
    d = sp.DeviceCoo("lap3d7", n)
    nr, nc, row, col, val = d.to_host()
    d.free()
    x = np.random.default_rng(4).uniform(-1.0, 1.0, nc)
    y_ref = oracle.crs_result(nr, row, col, val, x)
    bounds, blocks = spd.build_local_group("lap3d7", n, 0, 1, parts)
    xd = torch.from_numpy(x).cuda()
    for b in blocks:
        assert b.A.scalar("chunk_feed") == 1 and b.A.scalar("crs_kernel") == 1, b.rank
        b.x_owned.copy_(xd[int(bounds[b.rank]):int(bounds[b.rank + 1])])
    spd.local_group_multiply(blocks)
    torch.cuda.synchronize()
    assert np.array_equal(torch.cat([b.y for b in blocks]).cpu().numpy(), y_ref)
    for b in blocks:
        b.free()


def test_graph_capture_of_prepared_range(sp, oracle):
    """multiply_rows on a prepared range captured in a CUDA graph (first launch of the handle inside the capture), x
    overwritten before the replay: the bits of an eager multiply with that x."""
    import torch
    nr, nc, row, col, val = oracle.stencil("lap3d7", 15)
    rng = np.random.default_rng(6)
    for fmt in ("crs", "ss"):
        A = convert(sp, fmt, nr, nc, row, col, val)
        assert A.scalar("chunk_feed") == 1
        a, b = 300, nr - 211
        A.prepare_rows(a, b)
        xd = torch.from_numpy(rng.uniform(-1.0, 1.0, nc)).cuda()
        yg = torch.full((nr,), float("nan"), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        graph, stream = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        with torch.cuda.graph(graph, stream=stream):
            A.multiply_rows(a, b, xd.data_ptr(), yg.data_ptr(), stream.cuda_stream)
        x2 = rng.uniform(-1.0, 1.0, nc)
        xd.copy_(torch.from_numpy(x2))
        graph.replay()
        torch.cuda.synchronize()
        y = yg.cpu().numpy()
        assert np.all(np.isnan(y[:a])) and np.all(np.isnan(y[b:]))
        assert np.array_equal(y[a:b], oracle.crs_result(nr, row, col, val, x2)[a:b]), fmt
        A.destroy()
