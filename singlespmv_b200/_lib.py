"""ctypes binding of libb200spmv.so -- the C-ABI declared in include/b200spmv.h.

The library is built in-tree by ``make -C singlespmv_b200/csrc`` (``__graft_entry__.build()``).
There is no fallback of any kind: a missing library raises at import of this module, and every
compute entry point fails with ``B200SpmvError`` when no CUDA device is present.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200spmv.so")

FORMATS = {"crs": 0, "coo": 1, "ell": 2, "jds": 3, "dia": 4, "ss": 5, "css": 6, "csr5": 7, "hyb": 8}
SYNTH = {"lap2d5": 0, "lap3d7": 1, "box3d27": 2, "uniform": 3, "rmat": 4}

class B200SpmvError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("libb200spmv status %d: %s" % (status, message))
        self.status = status


class Options(C.Structure):
    _fields_ = [("segment_width", C.c_int), ("n_block", C.c_int), ("csr5_sigma", C.c_int),
                ("ss_faithful", C.c_int), ("value_f32", C.c_int), ("crs_path", C.c_int), ("profile", C.c_int), ("col_blocks", C.c_int), ("precision", C.c_int), ("hyb_k", C.c_int), ("coo_path", C.c_int),
                ("transpose", C.c_int), ("reserved", C.c_int * 4)]


class Stats(C.Structure):
    _fields_ = [("nRow", C.c_int), ("nCol", C.c_int), ("nnz", C.c_longlong), ("rowMax", C.c_int), ("rowMin", C.c_int),
                ("colMax", C.c_int), ("colMin", C.c_int), ("rowMean", C.c_double), ("rowVar", C.c_double),
                ("nEmptyRows", C.c_longlong), ("nDiag", C.c_longlong)]


class Coo(C.Structure):
    _fields_ = [("nRow", C.c_int), ("nCol", C.c_int), ("rowBegin", C.c_int), ("rowEnd", C.c_int),
                ("nnz", C.c_longlong), ("row_d", C.c_void_p), ("col_d", C.c_void_p),
                ("val_d", C.c_void_p)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C singlespmv_b200/csrc).  singlespmv_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, ip, ll = C.c_void_p, C.c_int, C.c_longlong
    lib.b200spmv_version.restype = ip
    lib.b200spmv_last_error.restype = C.c_char_p
    lib.b200spmv_device_count.argtypes = [C.POINTER(ip)]
    lib.b200spmv_create.argtypes = [ip, C.POINTER(Options), C.POINTER(vp)]
    lib.b200spmv_destroy.argtypes = [vp]
    lib.b200spmv_convert_coo_host.argtypes = [vp, ip, ip, ll, vp, vp, vp]
    lib.b200spmv_convert_coo_device.argtypes = [vp, ip, ip, ll, vp, vp, vp, vp]
    lib.b200spmv_jds_set_perm_host.argtypes = [vp, vp, ip]
    lib.b200spmv_multiply.argtypes = [vp, vp, vp, vp]
    lib.b200spmv_multiply_host.argtypes = [vp, vp, vp]
    lib.b200spmv_multiply_multi.argtypes = [vp, ip, vp, ll, vp, ll, vp]
    lib.b200spmv_multiply_multi_f32.argtypes = [vp, ip, vp, ll, vp, ll, vp]
    lib.b200spmv_multiply_f32.argtypes = [vp, vp, vp, vp]
    lib.b200spmv_multiply_transpose.argtypes = [vp, vp, vp, vp]
    lib.b200spmv_multiply_transpose_f32.argtypes = [vp, vp, vp, vp]
    lib.b200spmv_multiply_host_f32.argtypes = [vp, vp, vp]
    lib.b200spmv_multiply_rows.argtypes = [vp, ip, ip, vp, vp, vp]
    lib.b200spmv_prepare_rows.argtypes = [vp, ip, ip]
    lib.b200spmv_rows_col_extent.argtypes = [vp, ip, ip, C.POINTER(ip), C.POINTER(ip)]
    lib.b200spmv_host_register.argtypes = [vp, C.c_ulonglong]
    lib.b200spmv_host_unregister.argtypes = [vp]
    lib.b200spmv_get_scalar.argtypes = [vp, C.c_char_p, C.POINTER(ll)]
    lib.b200spmv_get_array.argtypes = [vp, C.c_char_p, vp, ll]
    lib.b200spmv_get_array.restype = ll
    lib.b200spmv_synth.argtypes = [ip, ll, ll, C.c_ulonglong, ip, ip, C.POINTER(Coo), vp]
    lib.b200spmv_coo_free.argtypes = [C.POINTER(Coo)]
    lib.b200spmv_coo_upload.argtypes = [ip, ip, ip, ip, ll, vp, vp, vp, C.POINTER(Coo)]
    lib.b200spmv_coo_download.argtypes = [C.POINTER(Coo), vp, vp, vp]
    lib.b200spmv_reference_vectors.argtypes = [C.c_uint, ip, ip, vp, vp]
    lib.b200spmv_load_mtx.argtypes = [C.c_char_p, ip, C.POINTER(Coo), vp]
    lib.b200spmv_analyze.argtypes = [C.POINTER(Coo), C.POINTER(Stats), vp]
    lib.b200spmv_recommend_format.argtypes = [C.POINTER(Stats), C.POINTER(Options)]
    lib.b200spmv_partition_rows.argtypes = [vp, ll, ip, ip, vp]
    lib.b200spmv_partition_synth.argtypes = [ip, ll, ll, ip, vp]
    lib.b200spmv_mg_create.argtypes = [ip, ip, C.POINTER(Options), C.POINTER(vp)]
    lib.b200spmv_mg_destroy.argtypes = [vp]
    lib.b200spmv_mg_convert_coo_host.argtypes = [vp, ip, ip, ll, vp, vp, vp]
    lib.b200spmv_mg_convert_synth.argtypes = [vp, ip, ll, ll, C.c_ulonglong]
    lib.b200spmv_mg_multiply_host.argtypes = [vp, vp, vp]
    lib.b200spmv_mg_upload_x.argtypes = [vp, vp]
    lib.b200spmv_mg_multiply.argtypes = [vp]
    lib.b200spmv_mg_synchronize.argtypes = [vp]
    lib.b200spmv_mg_download_y.argtypes = [vp, vp]
    lib.b200spmv_mg_get_scalar.argtypes = [vp, C.c_char_p, C.POINTER(ll)]
    lib.b200spmv_mg_get_bounds.argtypes = [vp, vp]
    lib.b200spmv_halo_plan.argtypes = [C.POINTER(Coo), ip, ip, C.POINTER(vp), vp]
    lib.b200spmv_halo_info.argtypes = [vp, vp]
    lib.b200spmv_halo_cols.argtypes = [vp, vp, ll]
    lib.b200spmv_halo_cols.restype = ll
    lib.b200spmv_halo_set_send.argtypes = [vp, vp, ll]
    lib.b200spmv_halo_pack.argtypes = [vp, vp, vp, vp]
    lib.b200spmv_halo_free.argtypes = [vp]
    lib.b200spmv_xwin_create.argtypes = [ip, ip, ll, ll, C.POINTER(vp)]
    lib.b200spmv_xwin_x_ext.argtypes = [vp]
    lib.b200spmv_xwin_x_ext.restype = vp
    lib.b200spmv_xwin_export.argtypes = [vp, vp]
    lib.b200spmv_xwin_import.argtypes = [vp, ip, vp]
    lib.b200spmv_xwin_attach.argtypes = [vp, ip, vp]
    lib.b200spmv_xwin_plan.argtypes = [vp, vp, ip, ip, ip, vp, vp, ip]
    lib.b200spmv_xwin_exchange.argtypes = [vp, vp]
    lib.b200spmv_xwin_status.argtypes = [vp, C.POINTER(ll), C.POINTER(ip)]
    lib.b200spmv_xwin_free.argtypes = [vp]
    return lib


lib = _load()


def check(status):
    if status < 0:
        raise B200SpmvError(status, lib.b200spmv_last_error().decode("utf-8", "replace"))
    return status
