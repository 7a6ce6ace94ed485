#!/usr/bin/env python
"""bench.py -- the reference's load -> convert -> repeat-multiply loop (src/main.cpp:58-102) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1..c5] [--format FMT] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one SpMV (y := A x) over the whole synthetic matrix of the workload.  Inputs are seeded, so two builds
run with the same arguments can be compared on the y that --dump-outputs writes.
Metric: SpMV GFLOP/s = 2 nnz / t (src/main.cpp:196), with effective HBM GB/s (compulsory bytes / t)
in `roofline`.  Workloads are BASELINE.json's configs (SURVEY.md 8d):

    c1  2-D 5-point Laplacian 1024^2          CRS (+ DIA, ELL; cold / warm / CUDA-graph figures)
    c2  uniform random 2^24 rows x 32/row     sliced-ELL, SS, JDS (+ CSS)
    c3  R-MAT scale 23, 2^28 draws            CSR5-style, adaptive CRS (vs cuSPARSE CSR)
    c4  3-D 27-point 256^3                    DIA (+ ELL, CRS)
    c5  3-D 7-point 512^3                     CRS, row-partitioned at N > 1 (all eight formats + cuSPARSE at N = 1)

The HEADLINE workload is c5 / CRS at every N (the config BASELINE.json's metric is quoted on at 1/2/4/8 GPUs; it
fits one GPU), so the N = 1, 2, 4, 8 lines are one strong-scaling curve.  At N = 1 the same run also measures
every other config x named format and reports them under `configs` (each with its own roofline fraction, ncu DRAM
traffic where a capture is committed, a sampled full-size parity check against the reference's CRS result, and
cuSPARSE CSR where BASELINE.json names the comparison).  --workload / --format restrict the run to one case.

--impl reference times the reference's own OpenMP CRS plugin (oracle/_ref/libref_crs.so, compiled
unmodified from /root/reference/src/opt_crs.cpp; else the C restatement in oracle/) on the host
cores: on the WHOLE workload matrix when the host has the memory for it, else on a bounded row sample.  That
leg, `cpu_baseline` and the `parity` checks are the only places this file touches oracle/.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree it runs from as it found it

L2_BYTES = 126 * 1024 * 1024
DUMP_ROWS = 1 << 21                     # --dump-outputs: rows of y kept from a larger result (<= 32 MiB with their indices)

WORKLOADS = {
    "c1": dict(kind="lap2d5", p0=1024, p1=0, seed=1, fmt="crs", formats=["crs", "dia", "ell"], f32=["crs"],
               name="CRS fp64, 2-D 5-point Laplacian 1024x1024 (1,048,576 rows, 5,238,784 nnz)"),
    "c2": dict(kind="uniform", p0=1 << 24, p1=32, seed=1, fmt="ell", formats=["ell", "ss", "jds", "css"], f32=["ell", "crs"],
               fmt_opts={"css": dict(n_block=3)},
               name="sliced-ELL / SS / JDS fp64, uniform random 16,777,216 rows x 32 nnz/row (536,870,912 nnz)"),
    "c3": dict(kind="rmat", p0=23, p1=1 << 28, seed=42, fmt="csr5", formats=["csr5", "crs"], cusparse=True, f32=["csr5", "crs"],
               name="CSR5-style and adaptive CRS fp64, R-MAT scale 23, 2^28 edge draws (duplicates removed)"),
    "c4": dict(kind="box3d27", p0=256, p1=0, seed=1, fmt="dia", formats=["dia", "ell", "crs"], f32=["dia", "ell"],
               name="DIA fp64, 3-D 27-point stencil 256^3 (16,777,216 rows, 449,455,096 nnz)"),
    "c5": dict(kind="lap3d7", p0=512, p1=0, seed=1, fmt="crs", cusparse=True, f32=["crs", "ell", "dia"],
               formats=["crs", "dia", "ell", "jds", "ss", "css", "csr5", "coo"],
               name="row-partitioned CRS fp64, 3-D 7-point Laplacian 512^3 (134,217,728 rows, 937,951,232 nnz)"),
}
MINI = {"c1": dict(p0=128), "c2": dict(p0=1 << 16), "c3": dict(p0=14, p1=1 << 18), "c4": dict(p0=32),
        "c5": dict(p0=64)}
HEADLINE = "c5"

# dram__bytes_read.sum + dram__bytes_write.sum of ONE multiply's launches of the dominant kernel, from the committed
# ncu --set full captures (profiles/r1_ncu_kernels.md, profiles/r2_ncu_kernels.md).  Keyed by (workload, format); else null.
NCU_TRAFFIC = {("c3", "csr5"): 3383375304,
               ("c4", "dia"): 3870562096, ("c4", "ell"): 5853024560, ("c5", "dia"): 9634725000,
               ("c5", "csr5"): 13638726000}
try:                                    # captures of this round's kernels, written by scripts/ncu_traffic.py
    with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as _f:
        for _k, _v in json.load(_f).items():
            NCU_TRAFFIC[tuple(_k.split("/"))] = _v
except Exception:
    pass
DOMINANT = {"crs": "chunk_stream_kernel (longest row <= 16, banded) / entry_stream_kernel (gather-bound) / tile_stream_kernel", "ss": "chunk_stream_kernel / tile_stream_kernel / ell_spmv_kernel per column block",
            "css": "tile_stream_kernel (one launch per column block)", "ell": "ell_spmv_kernel (gather-bound matrices: one launch per column block)",
            "jds": "jds_spmv_kernel / ell_spmv_kernel per column block (gather-bound matrices)", "dia": "dia_spmv_tma_kernel", "coo": "coo_stream_kernel",
            "csr5": "c5_compute_kernel", "hyb": "ell_spmv_kernel + coo_tile_kernel"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------ CPU legs (oracle/)
def cpu_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def host_memory_available():
    """Bytes this process may still allocate: /proc/meminfo MemAvailable capped by the cgroup limit."""
    avail = None
    try:
        with open("/proc/meminfo") as f:
            for ln in f:
                if ln.startswith("MemAvailable:"):
                    avail = int(ln.split()[1]) * 1024
    except Exception:
        pass
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            with open(lim) as f:
                v = f.read().strip()
            if v != "max":
                with open(cur) as f:
                    used = int(f.read().strip())
                left = int(v) - used
                avail = left if avail is None else min(avail, left)
        except Exception:
            pass
    return avail if avail is not None else 0


class CpuReferenceCrs:
    """The reference's OpenMP CRS SpMV (src/opt_crs.cpp:44-70) on the host: oracle/_ref when present (kind
    "reference"), else the C restatement (kind "port").  One object = one converted matrix."""

    def __init__(self, nRow, nCol, row, col, val, x):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import numpy as np
        import oracle_lib
        # all host threads, whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1 for its workers)
        try:
            C.CDLL("libgomp.so.1").omp_set_num_threads(C.c_int(cpu_threads()))
        except OSError:
            pass
        self.y = np.empty(nRow)
        self.nnz = len(row)
        if oracle_lib.ref_available("crs"):
            self.kind = "reference"
            lib = oracle_lib.RefPlugin("crs").lib
            lib.ref_convert(C.c_int(nRow), C.c_int(nCol), C.c_int(len(row)), row.ctypes, col.ctypes, val.ctypes, x.ctypes)
            self._keep = (row, col, val, x, lib)
            self.call = lambda: lib.ref_spmv(self.y.ctypes)
        else:
            self.kind = "port"
            orc = oracle_lib.Oracle()
            m = orc.crs_convert(nRow, row, col, val)
            lib = orc.lib
            self._keep = (m, x, lib)
            self.call = lambda: lib.orc_crs_spmv(C.c_int(nRow), m["ptr"].ctypes, m["idx"].ctypes, m["val"].ctypes,
                                                 x.ctypes, self.y.ctypes)

    def time(self, min_seconds, max_calls, warmup=1, exact_calls=None):
        times = []
        for _ in range(warmup):
            self.call()
        t_begin = time.perf_counter()
        while True:
            t0 = time.perf_counter()
            self.call()
            times.append(time.perf_counter() - t0)
            if exact_calls is not None:
                if len(times) >= exact_calls:
                    break
            elif (time.perf_counter() - t_begin >= min_seconds and len(times) >= 3) or len(times) >= max_calls:
                break
        return times


def per_row(wl):
    return {"lap2d5": 5, "lap3d7": 7, "box3d27": 27, "uniform": wl["p1"], "rmat": 32}[wl["kind"]]


def n_rows(wl):
    p0 = wl["p0"]
    return {"lap2d5": p0 * p0, "lap3d7": p0 ** 3, "box3d27": p0 ** 3, "uniform": p0, "rmat": 1 << p0}[wl["kind"]]


def sample_rows_for(wl):
    """Row count of the bounded CPU sample: ~64 M non-zeros (a few 10 ms per call on a server CPU)."""
    return min(n_rows(wl), max(1, (1 << 26) // per_row(wl)))


def stencil_row_counts(kind, n, r0, r1):
    """Entries of rows [r0, r1) of a stencil matrix, closed form (oracle/synth_oracle.c definitions)."""
    import numpy as np
    r = np.arange(r0, r1, dtype=np.int64)

    def span(i):
        return 1 + (i > 0).astype(np.int64) + (i < n - 1).astype(np.int64)
    if kind == "lap2d5":
        return span(r // n) + span(r % n) - 1
    k, j, i = r % n, (r // n) % n, r // (n * n)
    if kind == "lap3d7":
        return span(i) + span(j) + span(k) - 2
    return span(i) * span(j) * span(k)


def host_matrix(wl, rows):
    """Rows [0, rows) of the workload's matrix generated on the HOST by oracle/synth_oracle.c (bit-identical to the
    device generator, tests/test_gpu_parity.py::test_synth_matches_oracle), in parallel row slabs written straight
    into the final arrays."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import oracle_lib
    from concurrent.futures import ThreadPoolExecutor
    orc = oracle_lib.Oracle()
    kind, p0, p1, seed = wl["kind"], wl["p0"], wl["p1"], wl["seed"]
    if kind == "rmat":                  # global sort + dedupe: whole matrix only
        nRow, nCol, row, col, val = orc.rmat(seed, p0, p1)
        x, _ = orc.reference_vectors(nCol, 0, 3)
        return nRow, nCol, row, col, val, x
    nFull = n_rows(wl)
    slab = 1 << 20
    starts = list(range(0, rows, slab))
    if kind == "uniform":
        counts = [(min(rows, s + slab) - s) * p1 for s in starts]
    else:
        counts = [int(stencil_row_counts(kind, p0, s, min(rows, s + slab)).sum()) for s in starts]
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    nnz = int(offs[-1])
    row, col, val = np.empty(nnz, np.int32), np.empty(nnz, np.int32), np.empty(nnz, np.float64)
    kid = {"lap2d5": 0, "lap3d7": 1, "box3d27": 2}.get(kind)

    def fill(i):
        s, e, o, c = starts[i], min(rows, starts[i] + slab), int(offs[i]), counts[i]
        r_, c_, v_ = row[o:o + c], col[o:o + c], val[o:o + c]
        if kind == "uniform":
            orc.lib.synth_uniform(C.c_uint64(seed), C.c_int(nFull), C.c_int(p1), C.c_int(s), C.c_int(e),
                                  r_.ctypes, c_.ctypes, v_.ctypes)
        else:
            got = orc.lib.synth_stencil_range(C.c_int(kid), C.c_int(p0), C.c_int(s), C.c_int(e),
                                              r_.ctypes, c_.ctypes, v_.ctypes)
            assert got == c, (got, c)
    with ThreadPoolExecutor(max_workers=max(1, min(32, cpu_threads()))) as ex:
        list(ex.map(fill, range(len(starts))))
    x, _ = orc.reference_vectors(nFull, 0, 3)
    return rows, nFull, row, col, val, x


# ------------------------------------------------------------------------------------------ reference arm
def run_reference_arm(args, wl, wl_key):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["OMP_NUM_THREADS"] = str(cpu_threads())        # before libgomp initialises
    nFull = n_rows(wl)
    # whole matrix when the host can hold COO (16 B/nnz) + the plugin's CRS copy (12 B/nnz) + vectors with room to
    # spare; otherwise the bounded row sample (R-MAT: always its own generator's whole matrix)
    need = nFull * per_row(wl) * 30 + nFull * 24
    full = wl["kind"] != "rmat" and not args.sample and host_memory_available() > need + (8 << 30)
    rows = nFull if full else sample_rows_for(wl)
    nRow, nCol, row, col, val, x = host_matrix(wl, rows)
    ref = CpuReferenceCrs(nRow, nCol, row, col, val, x)
    times = ref.time(0, 0, warmup=args.warmup, exact_calls=args.steps)
    t = sum(times) / len(times)
    gflops = 2.0 * len(row) / t / 1e9
    what = "the whole workload matrix" if nRow == nFull else "first %d rows of the workload matrix" % nRow
    sample = "%s (%d rows, %d nnz), full-length x; reference CRS OpenMP SpMV, mean of %d calls" % (what, nRow, len(row), len(times))
    line = {"impl": "reference", "metric": "SpMV GFLOP/s", "value": gflops, "unit": "GFLOP/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": wl_key + ": " + wl["name"], "format": "crs (reference src/opt_crs.cpp)",
                                            "sample": sample, "whole_matrix": nRow == nFull},
            "cpu_baseline": {"value": gflops, "unit": "GFLOP/s", "cores": cpu_threads(), "kind": ref.kind, "sample": sample},
            "e2e": {"value": gflops, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ref.y)


def dump_outputs(out_dir, y):
    """--dump-outputs: the y of the timed path's last step as out_dir/y.npy, every row, or for more than DUMP_ROWS rows a
    fixed seeded sample of rows whose indices go to out_dir/y_rows.npy.  y is a numpy array or a CUDA tensor."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rows_path = os.path.join(out_dir, "y_rows.npy")
    rows = None
    if len(y) > DUMP_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(len(y), size=DUMP_ROWS, replace=False))
        np.save(rows_path, rows.astype(np.float64))
    elif os.path.exists(rows_path):
        os.remove(rows_path)
    if not isinstance(y, np.ndarray):                        # gather the sample on the device, copy only that
        import torch
        y = (y if rows is None else y[torch.from_numpy(rows).to(y.device)]).cpu().numpy()
    elif rows is not None:
        y = y[rows]
    np.save(os.path.join(out_dir, "y.npy"), y)


# ------------------------------------------------------------------------------------------ GPU arm, N = 1
class Timer:
    """CUDA-event timing on the launching stream.  L2-resident matrices are timed cold (512 MiB write between steps)."""

    def __init__(self, torch, stream):
        self.torch, self.stream, self.flush = torch, stream, None

    def run(self, fn, steps, warmup, cold):
        torch = self.torch
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if cold:
            if self.flush is None:
                self.flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.int32, device="cuda")
            evs = []
            for _ in range(steps):
                self.flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(self.stream)
                fn()
                b.record(self.stream)
                evs.append((a, b))
            torch.cuda.synchronize()
            return sum(a.elapsed_time(b) for a, b in evs) / steps
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(self.stream)
        for _ in range(steps):
            fn()
        b.record(self.stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    def graphed(self, fn, steps, reps=20):
        """`reps` back-to-back multiplies captured in ONE CUDA graph (SURVEY.md 8d: the CUDA-graph variant for c1):
        launch gaps between the ~15 us kernels disappear.  Returns ms per multiply, or None if capture fails."""
        torch = self.torch
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                sp = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                for _ in range(reps):
                    fn(sp)
            torch.cuda.synchronize()
            g.replay()
            torch.cuda.synchronize()
            n = max(3, steps // reps)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                g.replay()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / (n * reps)
            del g
            return ms
        except Exception as e:                               # noqa: BLE001
            sys.stderr.write("graph variant failed: %r\n" % (e,))
            try:
                torch.cuda.synchronize()
            except Exception:                                # noqa: BLE001
                pass
            return None


def parity_of(y, y_ref, mag, tol=1e-12):
    """Per-row comparison with the reference CRS result (SURVEY.md 8d tolerance: rel <= tol OR |dy| <= tol * sum |a x|;
    tol = 1e-12 for fp64, 1e-5 for the fp32 variant)."""
    import numpy as np
    y = y.astype(np.float64)
    err = np.abs(y - y_ref)
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = np.where(y_ref != 0, err / np.abs(y_ref), np.where(err == 0, 0.0, np.inf))
        relmag = np.where(mag != 0, err / mag, np.where(err == 0, 0.0, np.inf))
    ok = (rel <= tol) | (relmag <= tol)
    return {"rows": int(len(y)), "max_rel": float(rel.max()) if len(y) else 0.0,
            "max_rel_to_mag": float(relmag.max()) if len(y) else 0.0,
            "bit_identical": bool(np.array_equal(y, y_ref)), "within_%g" % tol: bool(ok.all())}


def cpu_sample(sp, wl, x_h):
    """First rows of the matrix on the host (device generator, downloaded) + the reference CRS object on them."""
    import numpy as np
    rows = sample_rows_for(wl)
    if wl["kind"] == "rmat":
        c = sp.DeviceCoo(wl["kind"], wl["p0"], wl["p1"], wl["seed"])
        rows = c.nRow
    else:
        c = sp.DeviceCoo(wl["kind"], wl["p0"], wl["p1"], wl["seed"], 0, rows)
    _, nCol, row, col, val = c.to_host()
    c.free()
    ref = CpuReferenceCrs(rows, nCol, row, col, val, x_h)
    ref.call()
    y_ref = ref.y.copy()
    mag = np.bincount(row, weights=np.abs(val * x_h[col]), minlength=rows)[:rows]
    return ref, rows, y_ref, mag


def run_case(sp, torch, timer, wl_key, wl, fmt, options, coo, x_d, y_d, sptr, steps, warmup, peak, mini, sample,
             after_timed=None):
    """Convert + time one format on one config.  Returns (entry dict, handle).  after_timed(y) is called with the result
    of the last timed step, before anything else writes y."""
    t0 = time.perf_counter()
    A = sp.SpMatOpt(fmt, **options).convert_device(coo)
    torch.cuda.synchronize()
    t_conv = time.perf_counter() - t0
    alg_bytes = A.scalar("alg_bytes")
    cold = alg_bytes < 2 * L2_BYTES
    f32 = bool(options.get("precision"))
    if f32:                                  # fp32 variant: float x and y (options.precision)
        x_d = x_d.float()
        y_d = torch.empty(y_d.shape, dtype=torch.float32, device="cuda")

    def step(s=None):
        if f32:
            A.multiply_f32(x_d.data_ptr(), y_d.data_ptr(), sptr if s is None else s)
        else:
            A.multiply(x_d.data_ptr(), y_d.data_ptr(), sptr if s is None else s)
    y_d.fill_(float("nan"))
    ms = timer.run(step, steps, warmup, cold)
    if after_timed is not None:
        after_timed(y_d)
    nnz = A.nNnz
    e = {"format": fmt, "options": {k: v for k, v in options.items() if v}, "gflops": 2.0 * nnz / (ms * 1e-3) / 1e9,
         "ms_per_step": ms, "alg_bytes": alg_bytes, "alg_gbs": alg_bytes / (ms * 1e-3) / 1e9,
         "frac": alg_bytes / (ms * 1e-3) / 1e9 / peak, "frac_of_8000": alg_bytes / (ms * 1e-3) / 1e9 / 8000.0,
         "traffic": None if mini else NCU_TRAFFIC.get((wl_key, fmt + ("_f32" if options.get("precision") else ""))),
         "launches_per_step": A.scalar("launches"),
         "convert_ms": t_conv * 1e3, "l2": "flushed between steps" if cold else "streams more than L2"}
    if cold:
        e["warm_l2_ms_per_step"] = timer.run(step, steps, 1, False)
        g = timer.graphed(step, steps)
        if g is not None:
            e["graph_ms_per_step"] = g
            e["graph_gflops"] = 2.0 * nnz / (g * 1e-3) / 1e9
    if sample is not None:
        _, rows, y_ref, mag = sample
        step()
        torch.cuda.synchronize()
        e["parity"] = parity_of(y_d[:rows].cpu().numpy(), y_ref, mag, 1e-5 if f32 else 1e-12)
    if f32:
        e["dtype"] = "f32 values and vectors, %s sums" % ("f32" if options["precision"] == 1 else "f64")
    return e, A


def index64_case(sp, torch, timer, sptr, peak, mini):
    """A matrix with more than 2^31-1 entries on ONE GPU (the reference's nNnz is an int, src/util.h:8; SURVEY.md 8f index
    variant): 3-D 7-point Laplacian 700^3 = 343,000,000 rows, 2,398,060,000 nnz, CRS.  The library cuts it into row blocks with
    32-bit offsets each (csrc/blocked.cu).  Checked on every row through the closed form of A.1."""
    p0 = 40 if mini else 700
    if mini:
        os.environ["B200SPMV_BLOCK_NNZ"] = "100000"
    try:
        coo = sp.DeviceCoo("lap3d7", p0)
        t0 = time.perf_counter()
        A = sp.SpMatOpt("crs").convert_device(coo)
        torch.cuda.synchronize()
        t_conv = time.perf_counter() - t0
        coo.free()
    finally:
        os.environ.pop("B200SPMV_BLOCK_NNZ", None)
    n, nnz = A.nRow, A.nNnz
    x_d = torch.ones(n, dtype=torch.float64, device="cuda")
    y_d = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")

    def step():
        A.multiply(x_d.data_ptr(), y_d.data_ptr(), sptr)
    ms = timer.run(step, 5, 3, False)
    idx = torch.arange(n, device="cuda")

    def span(a):
        return 1 + (a > 0).to(torch.int8) + (a < p0 - 1).to(torch.int8)
    cnt = span(idx // (p0 * p0)) + span((idx // p0) % p0) + span(idx % p0) - 2
    del idx
    ok = bool(torch.equal(y_d, (7 - cnt).double())) and int(cnt.sum(dtype=torch.int64).item()) == nnz
    alg = A.scalar("alg_bytes")
    e = {"workload": "CRS fp64, 3-D 7-point Laplacian %d^3 on one GPU" % p0, "nRow": n, "nnz": nnz, "beyond_int32": nnz > 2 ** 31 - 1,
         "row_blocks": A.scalar("row_blocks"), "ms_per_step": ms, "gflops": 2.0 * nnz / (ms * 1e-3) / 1e9, "alg_bytes": alg,
         "alg_gbs": alg / (ms * 1e-3) / 1e9, "frac": alg / (ms * 1e-3) / 1e9 / peak, "convert_ms": t_conv * 1e3,
         "check": "A.1 against the closed form on every row (exact small integers)", "ok": ok}
    A.destroy()
    return e


def cusparse_compare(torch, coo, x_d, y_d, sptr, warmup, steps):
    """Comparison point only (libb200cmp.so, singlespmv_b200/compare/): cusparseSpMV CSR on the same device arrays
    (the reference's src/opt_cusparse.cpp:57-83 re-expressed for cuSPARSE 12)."""
    cmp = C.CDLL(os.path.join(ROOT, "singlespmv_b200", "libb200cmp.so"))
    cmp.b200cmp_last_error.restype = C.c_char_p
    res = {}
    y_c = torch.empty_like(y_d)
    nnz = int(coo.c.nnz)
    for alg, name in ((1, "csr_alg1"), (2, "csr_alg2")):
        ms_c = C.c_float()
        st = cmp.b200cmp_cusparse_csr(C.c_int(coo.nRow), C.c_int(coo.nCol), C.c_longlong(nnz), C.c_void_p(coo.c.row_d),
                                      C.c_void_p(coo.c.col_d), C.c_void_p(coo.c.val_d), C.c_void_p(x_d.data_ptr()),
                                      C.c_void_p(y_c.data_ptr()), alg, warmup, steps, C.byref(ms_c), sptr)
        if st != 0:
            res[name] = {"error": cmp.b200cmp_last_error().decode()}
            continue
        torch.cuda.synchronize()
        rel = float(((y_c - y_d).abs().max() / y_d.abs().max()).item())
        res[name] = {"ms_per_step": ms_c.value, "gflops": 2.0 * nnz / (ms_c.value * 1e-3) / 1e9, "max_diff_rel_to_max_y": rel}
    del y_c
    return res


def gather_ceiling(torch):
    """Random 8-byte gathers, nothing else (singlespmv_b200/compare/gather_bench.cu): what L2 / DRAM sustain for the
    access pattern of config 2's x[col].  G gathers/s; x32 B = the L2 sector bandwidth it corresponds to."""
    try:
        cmp = C.CDLL(os.path.join(ROOT, "singlespmv_b200", "libb200cmp.so"))
        out = {}
        for name, tb in (("table_45MB", 45 << 20), ("table_134MB", 134217728), ("table_1GB", 1 << 30)):
            ms = C.c_float()
            mg = cmp.b200cmp_gather(C.c_longlong(tb), C.c_longlong(1 << 29), 2, 5, C.byref(ms))
            if mg > 0:
                out[name] = {"ggathers_per_s": mg * 1e6 / (ms.value * 1e-3) / 1e9, "ms_per_536M": ms.value * 536.870912 / mg}
        # the same gathers with a coalesced 12 B/gather stream through the threads' 128-bit loads beside them
        ms = C.c_float()
        mg = cmp.b200cmp_gather_stream(C.c_longlong(45 << 20), C.c_longlong(1 << 29), 2, 5, C.byref(ms))
        if mg > 0:
            out["table_45MB_plus_12B_stream"] = {"ggathers_per_s": mg * 1e6 / (ms.value * 1e-3) / 1e9, "ms_per_536M": ms.value * 536.870912 / mg}
        return out
    except Exception as e:                                   # noqa: BLE001
        return {"error": repr(e)}


def run_single(args, wl_key, only_format):
    import numpy as np
    import torch
    import singlespmv_b200 as sp

    torch.cuda.set_device(0)
    stream = torch.cuda.current_stream()
    sptr = C.c_void_p(stream.cuda_stream)
    timer = Timer(torch, stream)
    peak, peak_src = peaks()
    user_opts = {k: v for k, v in args.options.items() if v}

    def workload(key):
        wl = dict(WORKLOADS[key])
        if args.mini:
            wl.update(MINI[key])
            wl["name"] += " [MINI]"
        return wl

    # ---------------------------------------------------------------- headline: c5 / CRS unless told otherwise
    wl = workload(wl_key)
    t0 = time.perf_counter()
    coo = sp.DeviceCoo(wl["kind"], wl["p0"], wl["p1"], wl["seed"])
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    fmt = only_format or wl["fmt"]
    options = dict(wl.get("fmt_opts", {}).get(fmt, {}))
    options.update(user_opts)
    if fmt == "auto":                        # the engine's own pick from the matrix statistics (b200spmv_recommend_format)
        fmt, rec_opts = coo.recommend()
        for k, v in rec_opts.items():
            options.setdefault(k, v)
    nRow, nCol = coo.nRow, coo.nCol
    x_h, _ = sp.reference_vectors(nCol, 0, 3)                       # src/main.cpp:18,31
    x_d = torch.from_numpy(x_h).cuda()
    y_d = torch.full((nRow,), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    sample = None if args.no_cpu else cpu_sample(sp, wl, x_h)

    sampler = ClockSampler(0)
    sampler.start()
    dump = (lambda y: dump_outputs(args.dump_outputs, y)) if args.dump_outputs else None
    head, A = run_case(sp, torch, timer, wl_key, wl, fmt, options, coo, x_d, y_d, sptr, args.steps, args.warmup, peak,
                       args.mini, sample, dump)
    nnz, ms, alg_bytes = A.nNnz, head["ms_per_step"], head["alg_bytes"]

    # e2e: the reference-facing call SpMV(A_opt, x_opt, y) with HOST vectors, exactly as the C++ plugin issues it
    # (singlespmv_b200/plugin/opt_b200.cpp): x and y are ordinary (pageable) host arrays that the plugin page-locks once
    # -- x in OptimizeProblem, y on the first SpMV -- then every step is H2D x, multiply, D2H y inside the timed region
    f32 = bool(options.get("precision"))
    xh = x_h.astype(np.float32) if f32 else x_h.copy()
    yh = np.empty(nRow, np.float32 if f32 else np.float64)
    host_call = A.multiply_host_f32 if f32 else A.multiply_host
    pinned = sp.host_register(xh) and sp.host_register(yh)
    for _ in range(min(args.warmup, 3)):
        host_call(xh, yh)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        host_call(xh, yh)
    e2e_s = (time.perf_counter() - t0) / args.steps
    clocks = sampler.stop()
    if f32:
        x32, y32 = x_d.float(), torch.empty(nRow, dtype=torch.float32, device="cuda")
        A.multiply_f32(x32.data_ptr(), y32.data_ptr(), sptr)
        torch.cuda.synchronize()
        assert torch.equal(torch.from_numpy(yh), y32.cpu()), "host-semantics and device-resident results differ"
        del x32, y32
    else:
        A.multiply(x_d.data_ptr(), y_d.data_ptr(), sptr)
        torch.cuda.synchronize()
        assert torch.equal(torch.from_numpy(yh), y_d.cpu()), "host-semantics and device-resident results differ"
    sp.host_unregister(xh)
    sp.host_unregister(yh)

    dom_launches = A.scalar("nBlock") if fmt == "css" else 1
    if fmt in ("ell", "jds", "ss"):
        dom_launches = max(1, A.scalar("col_blocks"))        # column-block engine: one tile-stream launch per block
    line = {"metric": "SpMV GFLOP/s", "value": head["gflops"], "unit": "GFLOP/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if f32 else "f64", "data": "synthetic",
            "config": {"workload": wl_key + ": " + wl["name"], "format": fmt, "options": head["options"], "nRow": nRow,
                       "nCol": nCol, "nnz": nnz, "x": "srand(3) rand()/RAND_MAX (src/main.cpp:18,31)",
                       "l2": "flushed between steps (512 MiB write)" if head["l2"].startswith("flushed")
                             else "inputs larger than L2 (%.2f GB streamed per step)" % (alg_bytes / 1e9),
                       "parallelism": "1 GPU (the N = 2/4/8 lines row-partition the same matrix: strong scaling)",
                       "convert_ms": head["convert_ms"], "generate_ms": t_gen * 1e3},
            "roofline": {"bound": "hbm", "achieved": head["alg_gbs"], "peak": peak, "unit": "GB/s", "frac": head["frac"],
                         "frac_of_8000_nominal": head["frac_of_8000"],
                         "traffic": head["traffic"] // dom_launches if head["traffic"] else None, "peak_source": peak_src,
                         "kernel": DOMINANT.get(fmt, fmt), "alg_bytes_per_launch": alg_bytes // dom_launches,
                         "dominant_launches_per_step": dom_launches, "avg_launch_ms": ms / dom_launches,
                         "note": "achieved = alg_bytes_per_launch / avg_launch_ms (CUDA events over the timed region); "
                                 "traffic = ncu dram read+write per launch (profiles/r2_ncu_kernels.md); `configs` entries carry "
                                 "alg_bytes and traffic per multiply"},
            "e2e": {"value": 2.0 * nnz / e2e_s / 1e9, "unit": "GFLOP/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": (4 if f32 else 8) * nCol, "d2h_bytes_per_step": (4 if f32 else 8) * nRow,
                    "host_buffers": "numpy arrays page-locked once by the plugin layer (cudaHostRegister), as "
                                    "plugin/opt_b200.cpp does for the driver's x and y" if pinned else "pageable numpy arrays"},
            "gpu_launches": head["launches_per_step"] * args.steps, "clocks": clocks}
    if "parity" in head:
        line["parity"] = dict(head["parity"], against="reference CRS (src/opt_crs.cpp:44-70) on the first rows of the same matrix")
    for k in ("warm_l2_ms_per_step", "graph_ms_per_step", "graph_gflops"):
        if k in head:
            line["config"][k] = head[k]

    if sample is not None:
        ref = sample[0]
        times = ref.time(args.cpu_seconds, 2000)
        line["cpu_baseline"] = {"value": 2.0 * ref.nnz / min(times) / 1e9, "unit": "GFLOP/s", "cores": cpu_threads(), "kind": ref.kind,
                                "mean_value": 2.0 * ref.nnz / (sum(times) / len(times)) / 1e9,
                                "sample": "first %d rows (%d nnz) of the same matrix, full-length x; reference OpenMP CRS "
                                          "SpMV (src/opt_crs.cpp:44-70), min of %d calls over %.1f s (src/main.cpp:79-102 keeps the min; "
                                          "mean_value is the mean, the convention of --impl reference)"
                                          % (sample[1], ref.nnz, len(times), sum(times))}

    # ---------------------------------------------------------------- every other config x named format
    if args.configs != "none" and not only_format:
        want = sorted(WORKLOADS) if args.configs == "all" else [c for c in args.configs.split(",") if c in WORKLOADS]
        want = [c for c in want if c == wl_key] + [c for c in want if c != wl_key]     # the headline's matrix is loaded now
        steps2, warm2 = max(5, args.steps // 5), 3
        configs = {}
        for key in want:
            w = wl if key == wl_key else workload(key)
            entry = {"workload": w["name"], "formats": {}}
            try:
                if key != wl_key:
                    A.destroy()
                    coo.free()
                    del x_d, y_d
                    coo = sp.DeviceCoo(w["kind"], w["p0"], w["p1"], w["seed"])
                    x_h, _ = sp.reference_vectors(coo.nCol, 0, 3)
                    x_d = torch.from_numpy(x_h).cuda()
                    y_d = torch.full((coo.nRow,), float("nan"), dtype=torch.float64, device="cuda")
                    sample = None if args.no_cpu else cpu_sample(sp, w, x_h)
                entry.update(nRow=coo.nRow, nCol=coo.nCol, nnz=coo.nNnz)
                if sample is not None:
                    entry["parity_against"] = ("reference CRS result (oracle/_ref, src/opt_crs.cpp:44-70) on the first %d rows"
                                               % sample[1])
                for f2 in w["formats"]:
                    if key == wl_key and f2 == fmt:
                        e2 = dict(head)
                    else:
                        A.destroy()
                        o2 = dict(w.get("fmt_opts", {}).get(f2, {}))
                        try:
                            e2, A = run_case(sp, torch, timer, key, w, f2, o2, coo, x_d, y_d, sptr, steps2, warm2, peak,
                                             args.mini, sample)
                        except sp.B200SpmvError as err:
                            e2 = {"format": f2, "error": str(err)}
                    e2.pop("format", None)
                    entry["formats"][f2] = e2
                for f2 in w.get("f32", []):                # the fp32 variant (options.precision = 1), tolerance 1e-5
                    A.destroy()
                    try:
                        e2, A = run_case(sp, torch, timer, key, w, f2, dict(precision=1), coo, x_d, y_d, sptr, steps2, warm2,
                                         peak, args.mini, sample)
                    except sp.B200SpmvError as err:
                        e2 = {"format": f2, "error": str(err)}
                    e2.pop("format", None)
                    entry["formats"][f2 + "_f32"] = e2
                if w.get("cusparse"):
                    A.destroy()
                    A = sp.SpMatOpt("crs").convert_device(coo)      # y_d must hold a full result for the difference check
                    A.multiply(x_d.data_ptr(), y_d.data_ptr(), sptr)
                    torch.cuda.synchronize()
                    entry["cusparse"] = cusparse_compare(torch, coo, x_d, y_d, sptr, warm2, steps2)
            except Exception as err:                         # noqa: BLE001  (one config must not sink the line)
                entry["error"] = repr(err)
            configs[key] = entry
        line["configs"] = configs
        if args.configs == "all":
            try:
                A.destroy()
                coo.free()
                del x_d, y_d
                torch.cuda.empty_cache()
                line["index64"] = index64_case(sp, torch, timer, sptr, peak, args.mini)
            except Exception as err:                         # noqa: BLE001
                line["index64"] = {"error": repr(err)}
        if not args.mini or args.gather:
            line["gather_ceiling"] = gather_ceiling(torch)
    elif args.compare_cusparse:
        line["cusparse"] = cusparse_compare(torch, coo, x_d, y_d, sptr, args.warmup, args.steps)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--format", default=None)
    ap.add_argument("--configs", default=None, help="N = 1: which configs go into `configs`: all | none | c1,c3 "
                                                    "(default: all for the default headline run, none with --workload/--format)")
    ap.add_argument("--mini", action="store_true", help="shrunken shapes (debugging only; not a bench number)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and parity legs")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--sample", action="store_true", help="--impl reference: bounded row sample even if the whole matrix fits")
    ap.add_argument("--gather", action="store_true", help="run the gather-ceiling microbenchmark even with --mini")
    ap.add_argument("--no-graph", action="store_true", help="multi-GPU: launch each step eagerly instead of one CUDA graph")
    ap.add_argument("--compare-cusparse", action="store_true", help="also time cusparseSpMV CSR (comparison point)")
    ap.add_argument("--segment-width", type=int, default=0)
    ap.add_argument("--n-block", type=int, default=0)
    ap.add_argument("--sigma", type=int, default=0)
    ap.add_argument("--value-f32", action="store_true", help="CRS: fp32 storage of the matrix values, fp64 arithmetic")
    ap.add_argument("--precision", type=int, default=0, help="CRS / ELL: 1 = fp32 values, vectors and sums, 2 = fp32 with fp64 sums")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write y of the last timed step of the headline case to DIR/y.npy (a seeded sample of rows, "
                         "listed in DIR/y_rows.npy, when y is large); one process only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "b200" and (args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs needs a single-GPU run (--gpus 1) or --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    args.options = dict(segment_width=args.segment_width, n_block=args.n_block, csr5_sigma=args.sigma,
                        value_f32=1 if args.value_f32 else 0, precision=args.precision)
    wl_key = args.workload or HEADLINE
    if args.configs is None:
        args.configs = "none" if (args.workload or args.format) else "all"
    wl = dict(WORKLOADS[wl_key])
    if args.mini:
        wl.update(MINI[wl_key])
        wl["name"] += " [MINI]"
    if args.impl == "reference":
        return run_reference_arm(args, wl, wl_key)
    if args.gpus == 1 and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        return run_single(args, wl_key, args.format)
    from singlespmv_b200.dist import run_partitioned_bench
    return run_partitioned_bench(args, wl, wl_key)


if __name__ == "__main__":
    main()
