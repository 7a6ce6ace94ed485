"""CPU checks of the drop-in boundary: libb200spmv.so loads, exports every symbol include/b200spmv.h
declares, validates arguments, and refuses to compute without a CUDA device (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    out = []
    for fn in sorted(os.listdir(os.path.join(ROOT, "include"))):
        if fn.endswith(".h"):
            src = open(os.path.join(ROOT, "include", fn)).read()
            out += re.findall(r"B200SPMV_API[^;(]*?\b(b200spmv_\w+)\s*\(", src)
    return out


def test_header_declares_the_boundary():
    syms = declared_symbols()
    for must in ("b200spmv_create", "b200spmv_convert_coo_host", "b200spmv_convert_coo_device",
                 "b200spmv_multiply", "b200spmv_multiply_host", "b200spmv_get_array", "b200spmv_destroy"):
        assert must in syms


def test_library_exports_every_declared_symbol():
    import singlespmv_b200 as sp
    lib = C.CDLL(sp.LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.b200spmv_version() == 100


def test_no_torch_types_in_signatures():
    src = open(os.path.join(ROOT, "include", "b200spmv.h")).read()
    assert "torch" not in src.lower() and "at::" not in src


def test_argument_validation_without_gpu():
    import singlespmv_b200 as sp
    with pytest.raises(sp.B200SpmvError):
        sp.SpMatOpt("ss", segment_width=3)            # W must be a power of two (opt_ss.cpp:272)
    with pytest.raises(KeyError):
        sp.SpMatOpt("nonsense")
    m = sp.SpMatOpt("crs")
    with pytest.raises(sp.B200SpmvError) as e:        # multiply before convert
        m.multiply(0, 0)
    assert e.value.status == -4 or e.value.status == -1


def test_create_rejects_unknown_kernel_paths():
    """crs_path = 2 selected round 1's row-block stream, which was removed; it and every other value outside the documented
    crs_path / coo_path sets are refused at create instead of silently running some other kernel."""
    import singlespmv_b200 as sp
    for fmt, opt in (("crs", {"crs_path": 2}), ("ss", {"crs_path": 2}), ("crs", {"crs_path": 5}), ("crs", {"crs_path": -1}),
                     ("coo", {"coo_path": 4}), ("coo", {"coo_path": -1})):
        with pytest.raises(sp.B200SpmvError) as e:
            sp.SpMatOpt(fmt, **opt)
        assert e.value.status == -1, (fmt, opt)
        if opt.get("crs_path") == 2:
            assert "row-block stream" in str(e.value)
    for fmt, opt in (("crs", {"crs_path": 1}), ("crs", {"crs_path": 3}), ("crs", {"crs_path": 4}), ("ss", {"crs_path": 3}),
                     ("coo", {"coo_path": 1}), ("coo", {"coo_path": 3})):
        sp.SpMatOpt(fmt, **opt)


def test_environment_hooks_match_design_table():
    """The B200SPMV_* variables the library reads are exactly the ones DESIGN.md section 5c documents."""
    read = set()
    for dp, dns, fns in os.walk(os.path.join(ROOT, "singlespmv_b200")):
        dns[:] = [d for d in dns if d not in ("build", "__pycache__")]
        for fn in fns:
            if fn.endswith((".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dp, fn), errors="replace").read()
                read |= set(re.findall(r'getenv\(\s*"(B200SPMV_\w+)"', src))
            elif fn.endswith(".py"):
                src = open(os.path.join(dp, fn), errors="replace").read()
                read |= set(re.findall(r'(?:os\.environ\.get\(|os\.environ\[|os\.getenv\()\s*["\'](B200SPMV_\w+)', src))
    design = open(os.path.join(ROOT, "DESIGN.md")).read()
    section = design.split("\n## 5c.", 1)[1].split("\n## ", 1)[0]
    documented = set(re.findall(r"B200SPMV_\w+", section))
    assert "B200SPMV_DIST_EXCHANGE" in read and "B200SPMV_TMA_R" in read
    assert read == documented, {"read, not documented": sorted(read - documented), "documented, not read": sorted(documented - read)}


def test_no_cpu_fallback():
    """Without a device, conversion and multiply must fail loudly -- never compute on the host."""
    import singlespmv_b200 as sp
    if sp.device_count() > 0:
        pytest.skip("a CUDA device is present")
    A = sp.SpMat(3, 3, [0, 1, 2], [0, 1, 2], [1.0, 2.0, 3.0])
    with pytest.raises(sp.B200SpmvError) as e:
        sp.OptimizeProblem(A, sp.Vec(np.ones(3)), "crs")
    assert e.value.status == -2 and "no CPU fallback" in str(e.value)
    with pytest.raises(sp.B200SpmvError):
        sp.DeviceCoo("lap2d5", 8)


def test_multi_gpu_entry_points_need_a_device():
    """The multi-GPU entry points (single-process handle, x windows) refuse to work without CUDA devices and validate their
    arguments on the host."""
    import singlespmv_b200 as sp
    from singlespmv_b200._lib import lib
    h = C.c_void_p()
    assert lib.b200spmv_xwin_create(0, 0, 10, 0, C.byref(h)) == -1            # world < 1
    assert lib.b200spmv_xwin_create(3, 2, 10, 0, C.byref(h)) == -1            # rank outside the world
    assert lib.b200spmv_xwin_create(0, 2, 10, 11, C.byref(h)) == -1           # owned slice outside x_ext
    assert lib.b200spmv_xwin_exchange(None, None) < 0 and lib.b200spmv_xwin_free(None) == 0
    if sp.device_count() > 0:
        pytest.skip("a CUDA device is present")
    assert lib.b200spmv_xwin_create(0, 2, 10, 0, C.byref(h)) == -2 and not h.value
    m = C.c_void_p()
    assert lib.b200spmv_mg_create(2, 0, None, C.byref(m)) == -2 and b"no CPU fallback" in lib.b200spmv_last_error()


def test_product_does_not_touch_the_oracle():
    """oracle/ is test infrastructure: nothing under singlespmv_b200/ or include/ may reference it."""
    bad = []
    for base in ("singlespmv_b200", "include"):
        for dp, _, fns in os.walk(os.path.join(ROOT, base)):
            if "build" in dp.split(os.sep) or "__pycache__" in dp:
                continue
            for fn in fns:
                if fn.endswith((".py", ".cu", ".cuh", ".h", ".cpp", ".c")) or fn == "Makefile":
                    txt = open(os.path.join(dp, fn), errors="replace").read()
                    if re.search(r"liboracle|oracle_lib|orc_|libref_|oracle/_ref", txt):
                        bad.append(os.path.join(dp, fn))
    assert not bad, bad


def test_reference_vectors_match_the_oracle(oracle):
    import singlespmv_b200 as sp
    x, y = sp.reference_vectors(17, 9, 3)
    xo, yo = oracle.reference_vectors(17, 9, 3)
    assert np.array_equal(x, xo) and np.array_equal(y, yo)
    assert x[0] == 0.56138017520372763      # SURVEY.md Appendix B


def test_recommend_format_rules_on_cpu():
    """b200spmv_recommend_format is pure host logic: the rule table on the BASELINE.json shapes from their closed-form
    statistics (the device side, b200spmv_analyze, is checked in tests/test_gpu_parity.py)."""
    import singlespmv_b200 as sp
    from singlespmv_b200._lib import Options, Stats, lib

    def rec(**kw):
        st = Stats()
        for k, v in kw.items():
            setattr(st, k, v)
        o = Options()
        f = lib.b200spmv_recommend_format(C.byref(st), C.byref(o))
        return [k for k, v in sp.FORMATS.items() if v == f][0], o.n_block
    n2 = 1 << 24
    assert rec(nRow=1 << 20, nCol=1 << 20, nnz=5238784, rowMax=5, rowMean=4.996, rowVar=0.004, nDiag=5)[0] == "dia"              # c1
    assert rec(nRow=n2, nCol=n2, nnz=n2 * 32, rowMax=32, rowMin=32, rowMean=32.0, rowVar=0.0, nDiag=2 * n2 - 1) == ("css", 3)   # c2
    assert rec(nRow=1 << 23, nCol=1 << 23, nnz=258673573, rowMax=400000, rowMean=30.8, rowVar=1e5, nDiag=1 << 24)[0] == "csr5"  # c3
    assert rec(nRow=256 ** 3, nCol=256 ** 3, nnz=766 ** 3, rowMax=27, rowMean=26.8, rowVar=0.5, nDiag=27)[0] == "dia"           # c4
    assert rec(nRow=512 ** 3, nCol=512 ** 3, nnz=937951232, rowMax=7, rowMean=6.99, rowVar=0.01, nDiag=7)[0] == "dia"           # c5
    assert rec(nRow=1 << 16, nCol=1 << 16, nnz=32 << 16, rowMax=32, rowMean=32.0, rowVar=0.0, nDiag=100000)[0] == "ell"
    assert rec(nRow=1000, nCol=1000, nnz=9000, rowMax=40, rowMean=9.0, rowVar=20.0, nDiag=900)[0] == "crs"
    assert rec(nRow=10, nCol=10, nnz=0)[0] == "crs"


def test_baseline_shapes_closed_form(oracle):
    """The synthetic generators' sizes are the ones BASELINE.json / SURVEY.md 8 quote."""
    L = oracle.lib
    assert (L.synth_stencil_rows(0, 1024), L.synth_stencil_nnz(0, 1024)) == (1048576, 5238784)          # c1
    assert (L.synth_stencil_rows(2, 256), L.synth_stencil_nnz(2, 256)) == (16777216, 766 ** 3)          # c4
    assert (L.synth_stencil_rows(1, 512), L.synth_stencil_nnz(1, 512)) == (134217728, 937951232)        # c5
    for kind, n in ((0, 7), (1, 5), (2, 4)):                                                            # closed form == generator
        assert L.synth_stencil_nnz(kind, n) == len(oracle.stencil({0: "lap2d5", 1: "lap3d7", 2: "box3d27"}[kind], n)[2])
