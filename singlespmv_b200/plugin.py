"""Host-side mirror of the reference's plugin interface, over the C-ABI (no torch types cross it).

Reference interface (one format per binary, /root/reference/src/opt.h:1-28):

    void OptimizeProblem(const SpMat &A, const Vec &x, SpMatOpt &A_opt, VecOpt &x_opt);   // opt_crs.h:15
    extern "C" void SpMV(const SpMatOpt &A, const VecOpt &x, Vec &y);                      // opt_crs.h:16-18

Here the format is a run-time argument instead of a -DOPT_* macro; names, argument meaning and the
"y is fully overwritten, call it as often as you like" contract (src/main.cpp:41-88) are kept.
The C++ twin of this file is singlespmv_b200/plugin/opt_b200.{h,cpp}.
"""
import ctypes as C

import numpy as np

from ._lib import FORMATS, SYNTH, B200SpmvError, Coo, Options, Stats, check, lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class SpMat:
    """COO container sorted by (row, col) -- reference src/util.h:7-19.  Host arrays."""

    def __init__(self, nRow, nCol, row_idx, col_idx, val):
        self.nRow, self.nCol = int(nRow), int(nCol)
        self.row_idx = np.ascontiguousarray(row_idx, np.int32)
        self.col_idx = np.ascontiguousarray(col_idx, np.int32)
        self.val = np.ascontiguousarray(val, np.float64)
        self.nNnz = len(self.row_idx)


class Vec:
    """reference src/util.h:20-28"""

    def __init__(self, val):
        self.val = np.ascontiguousarray(val, np.float64)
        self.size = len(self.val)


class DeviceCoo:
    """Synthetic COO generated in HBM (b200spmv_synth); rows [rowBegin,rowEnd) of the matrix."""

    def __init__(self, kind, p0, p1=0, seed=1, row_begin=0, row_end=0, stream=None):
        self.c = Coo()
        if kind is not None:
            check(lib.b200spmv_synth(SYNTH[kind], int(p0), int(p1), int(seed), int(row_begin), int(row_end),
                                     C.byref(self.c), stream))
            self._dims()

    def _dims(self):
        self.nRow, self.nCol, self.nNnz = self.c.nRow, self.c.nCol, int(self.c.nnz)
        self.rowBegin, self.rowEnd = self.c.rowBegin, self.c.rowEnd

    @classmethod
    def from_mtx(cls, path, reference_semantics=False, stream=None):
        """Matrix-Market file -> device COO (b200spmv_load_mtx).  reference_semantics: src/util.cpp:30-66 exactly."""
        self = cls(None, 0)
        check(lib.b200spmv_load_mtx(str(path).encode(), 1 if reference_semantics else 0, C.byref(self.c), stream))
        self._dims()
        return self

    @classmethod
    def from_host_rows(cls, A, row_begin, row_end):
        """Rows [row_begin, row_end) of a host SpMat (sorted COO) as a device COO with global row ids."""
        self = cls(None, 0)
        e0, e1 = np.searchsorted(A.row_idx, [row_begin, row_end], side="left")
        check(lib.b200spmv_coo_upload(A.nRow, A.nCol, int(row_begin), int(row_end), int(e1 - e0), _ptr(A.row_idx[e0:e1]),
                                      _ptr(A.col_idx[e0:e1]), _ptr(A.val[e0:e1]), C.byref(self.c)))
        self._dims()
        return self

    def to_host(self):
        n = self.nNnz
        row, col, val = np.empty(n, np.int32), np.empty(n, np.int32), np.empty(n, np.float64)
        check(lib.b200spmv_coo_download(C.byref(self.c), _ptr(row), _ptr(col), _ptr(val)))
        return self.nRow, self.nCol, row, col, val

    def analyze(self):
        """Row/column statistics (reference matrix/script/counter.cpp) + diagonals, computed on the device."""
        st = Stats()
        check(lib.b200spmv_analyze(C.byref(self.c), C.byref(st), None))
        return {k: getattr(st, k) for k, _ in Stats._fields_}, st

    def recommend(self):
        """(format name, options dict) the engine would pick for this matrix."""
        _, st = self.analyze()
        o = Options()
        f = check(lib.b200spmv_recommend_format(C.byref(st), C.byref(o)))
        name = [k for k, v in FORMATS.items() if v == f][0]
        return name, {k: getattr(o, k) for k in ("segment_width", "n_block", "csr5_sigma") if getattr(o, k)}

    def free(self):
        if self.c is not None:
            lib.b200spmv_coo_free(C.byref(self.c))
            self.c = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class SpMatOpt:
    """Converted matrix = opaque b200spmv_matrix handle (the reference's per-format SpMatOpt struct).

    ``scalar(name)`` / ``array(name, dtype)`` read the fields back under the reference's names, in the
    reference's logical layout, for parity checks."""

    def __init__(self, fmt, segment_width=0, n_block=0, csr5_sigma=0, ss_faithful=0, value_f32=0, crs_path=0, profile=0, col_blocks=0, hyb_k=0, precision=0, coo_path=0,
                 transpose=0):
        self.fmt = fmt
        o = Options()
        o.segment_width, o.n_block, o.csr5_sigma, o.ss_faithful = segment_width, n_block, csr5_sigma, ss_faithful
        o.value_f32, o.crs_path, o.profile, o.col_blocks = value_f32, crs_path, profile, col_blocks
        o.hyb_k, o.precision, o.coo_path, o.transpose = hyb_k, precision, coo_path, transpose
        self.h = C.c_void_p()
        check(lib.b200spmv_create(FORMATS[fmt], C.byref(o), C.byref(self.h)))
        self.nRow = self.nCol = self.nNnz = 0

    def _dims(self):
        self.nRow, self.nCol, self.nNnz = self.scalar("nRow"), self.scalar("nCol"), self.scalar("nNnz")

    def convert_host(self, A):
        check(lib.b200spmv_convert_coo_host(self.h, A.nRow, A.nCol, A.nNnz, _ptr(A.row_idx), _ptr(A.col_idx),
                                            _ptr(A.val)))
        self._dims()
        return self

    def convert_device(self, coo, nRow=None, stream=None):
        """coo: DeviceCoo (or anything with .c Coo).  Row ids must be 0-based for this handle."""
        c = coo.c
        check(lib.b200spmv_convert_coo_device(self.h, c.nRow if nRow is None else nRow, c.nCol, c.nnz, c.row_d,
                                              c.col_d, c.val_d, stream))
        self._dims()
        return self

    def set_jds_perm(self, perm):
        perm = np.ascontiguousarray(perm, np.int32)
        check(lib.b200spmv_jds_set_perm_host(self.h, _ptr(perm), len(perm)))

    def scalar(self, name):
        v = C.c_longlong()
        check(lib.b200spmv_get_scalar(self.h, name.encode(), C.byref(v)))
        return int(v.value)

    def array(self, name, dtype):
        n = lib.b200spmv_get_array(self.h, name.encode(), None, 0)
        check(n)
        a = np.empty(n // np.dtype(dtype).itemsize, dtype)
        if n:
            check(lib.b200spmv_get_array(self.h, name.encode(), _ptr(a), a.nbytes))
        return a

    # device-resident multiply: x_ptr / y_ptr are raw device addresses (e.g. torch .data_ptr())
    def multiply(self, x_ptr, y_ptr, stream=None):
        check(lib.b200spmv_multiply(self.h, C.c_void_p(x_ptr), C.c_void_p(y_ptr), stream))

    def multiply_multi(self, k, X_ptr, ldx, Y_ptr, ldy, stream=None):
        """Y[:, :k] := A X[:, :k] for k = 1..8 device-resident row-major vectors (X[c*ldx + j], Y[r*ldy + j]): the matrix is
        streamed once for all k.  CRS handles with fp64 values and vectors (b200spmv_multiply_multi)."""
        check(lib.b200spmv_multiply_multi(self.h, k, C.c_void_p(X_ptr), ldx, C.c_void_p(Y_ptr), ldy, stream))

    def multiply_transpose(self, x_ptr, y_ptr, stream=None):
        """y := A^T x for device-resident vectors, x of nRow and y of nCol entries (b200spmv_multiply_transpose).  Handles
        created with transpose=1, which convert A^T as a second matrix of the same format; its scalars and arrays are read
        with the prefix "t." (scalar("t.nRow"), array("t.ptr", ...))."""
        check(lib.b200spmv_multiply_transpose(self.h, C.c_void_p(x_ptr), C.c_void_p(y_ptr), stream))

    def multiply_transpose_f32(self, x_ptr, y_ptr, stream=None):
        """y := A^T x with fp32 vectors: multiply_transpose for handles created with transpose=1 and precision=1 or 2
        (b200spmv_multiply_transpose_f32)."""
        check(lib.b200spmv_multiply_transpose_f32(self.h, C.c_void_p(x_ptr), C.c_void_p(y_ptr), stream))

    def multiply_rows(self, row_begin, row_end, x_ptr, y_ptr, stream=None):
        check(lib.b200spmv_multiply_rows(self.h, row_begin, row_end, C.c_void_p(x_ptr), C.c_void_p(y_ptr), stream))

    def prepare_rows(self, row_begin, row_end):
        """Host bookkeeping of a row range ahead of time, so that multiply_rows on it never synchronises
        (needed before capturing it in a CUDA graph)."""
        check(lib.b200spmv_prepare_rows(self.h, row_begin, row_end))

    def col_extent(self, row_begin, row_end):
        """(smallest, largest) column referenced by rows [row_begin, row_end); largest < smallest = empty rows."""
        lo, hi = C.c_int(), C.c_int()
        check(lib.b200spmv_rows_col_extent(self.h, row_begin, row_end, C.byref(lo), C.byref(hi)))
        return lo.value, hi.value

    def multiply_f32(self, x_ptr, y_ptr, stream=None):
        """fp32 vectors (handle created with precision=1 or 2); raw device addresses of float arrays."""
        check(lib.b200spmv_multiply_f32(self.h, C.c_void_p(x_ptr), C.c_void_p(y_ptr), stream))

    def multiply_multi_f32(self, k, X_ptr, ldx, Y_ptr, ldy, stream=None):
        """Y[:, :k] := A X[:, :k] for k = 1..8 device-resident row-major fp32 vectors (X[c*ldx + j], Y[r*ldy + j]): the
        matrix is streamed once for all k.  CRS handles created with precision=1 or 2 (b200spmv_multiply_multi_f32)."""
        check(lib.b200spmv_multiply_multi_f32(self.h, k, C.c_void_p(X_ptr), ldx, C.c_void_p(Y_ptr), ldy, stream))

    def multiply_host_f32(self, x, y):
        assert x.dtype == np.float32 and y.dtype == np.float32
        check(lib.b200spmv_multiply_host_f32(self.h, _ptr(x), _ptr(y)))

    def multiply_host(self, x, y):
        check(lib.b200spmv_multiply_host(self.h, _ptr(x), _ptr(y)))

    def destroy(self):
        if self.h:
            lib.b200spmv_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class VecOpt:
    """reference e.g. src/opt_crs.h:11-14: aliases the caller's x (src/opt_crs.cpp:11-12)."""

    def __init__(self, x):
        self.size, self.val = x.size, x.val


def OptimizeProblem(A, x, fmt="crs", **options):
    """Conversion (reference src/opt_<fmt>.cpp OptimizeProblem).  Returns (A_opt, x_opt)."""
    A_opt = SpMatOpt(fmt, **options)
    A_opt.convert_host(A)
    return A_opt, VecOpt(x)


def SpMV(A_opt, x_opt, y):
    """y := A x with host vectors: H2D x, multiply on the B200, D2H y (every y[i] overwritten)."""
    if x_opt.size != A_opt.nCol or y.size != A_opt.nRow:
        raise B200SpmvError(-1, "SpMV: vector sizes %d/%d do not match the %dx%d matrix"
                            % (x_opt.size, y.size, A_opt.nRow, A_opt.nCol))
    A_opt.multiply_host(x_opt.val, y.val)


def host_register(a):
    """Page-lock a numpy array in place (what plugin/opt_b200.cpp does with the driver's x and y).  Returns False
    when the driver refuses; the caller must keep `a` alive until host_unregister(a)."""
    if a.nbytes == 0:
        return False
    return lib.b200spmv_host_register(_ptr(a), a.nbytes) == 0


def host_unregister(a):
    lib.b200spmv_host_unregister(_ptr(a))


def reference_vectors(nCol, nRow, seed=3):
    """x (and y) exactly as the reference's driver draws them: src/main.cpp:18,31-32."""
    x = np.empty(nCol, np.float64)
    y = np.empty(nRow, np.float64)
    check(lib.b200spmv_reference_vectors(seed, nCol, nRow, _ptr(x), _ptr(y)))
    return x, y


def device_count():
    n = C.c_int()
    lib.b200spmv_device_count(C.byref(n))
    return n.value
