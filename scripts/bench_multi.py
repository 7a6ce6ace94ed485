"""Multi-vector CRS multiply (b200spmv_multiply_multi / _multi_f32) against k single multiplies, on one GPU.

    python scripts/bench_multi.py [--out DIR] [--configs c5,c4,c3,c2] [--ks 1,2,4,8] [--seconds 1.0] [--precision 0,1,2]

For every config (generated on the device, CRS) and k: CUDA-event time of multiply_multi on row-major X / Y (ldx = ldy =
k) and of k back-to-back b200spmv_multiply calls on the k columns (each a contiguous vector), each over at least
--seconds after warm-ups.  Reports time per vector, GFLOP/s = 2 nnz k / t and bytes / t with bytes = the CRS arrays once
(12 nnz + 4 (nRow + 1)) + 8 k (nCol + nRow).  Parity at the timed size: Y[:, j] against the single multiply of column j,
bit for bit, or else within 2 n 2^-53 sum|a x| per row (both results lie within half of that of the exact row sum).
Writes DIR/bench_multi.json with the card's name and power limit read in the same run.

--precision 1 / 2 (handles created with options.precision; default 0 only): multiply_multi_f32 on fp32 X / Y against k
multiply_f32 calls, bytes = 8 nnz + 4 (nRow + 1) + 4 k (nCol + nRow).  Parity: bits against the singles (required of row-chunk stream handles), or else both
results within the bound of tests/test_gpu_fp32.py for the precision (exact products, s = their row sum):
    precision 2: |y - s| <= 2^-24 |s| + n 2^-53 sum|p| + 2^-149,   precision 1: |y - s| <= (n+1) 2^-24 sum|p| + (n+1) 2^-149
evaluated on the device against an fp64 row sum, whose own error n 2^-53 sum|p| is added to the bound."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {   # the matrices of bench.py
    "c5": ("lap3d7", 512, 0, 1, "3-D 7-point 512^3"),
    "c4": ("box3d27", 256, 0, 1, "3-D 27-point 256^3"),
    "c3": ("rmat", 23, 1 << 28, 42, "R-MAT scale 23, 2^28 draws"),
    "c2": ("uniform", 1 << 24, 32, 1, "uniform random 2^24 rows x 32"),
}
KERNELS = {1: "row-chunk stream", 2: "entry stream (TMA-fed)", 3: "entry stream (load-fed)"}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, seconds, torch):
    """mean ms per call of fn over >= seconds, after warm-ups (CUDA events around the whole window)"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    e.record()
    torch.cuda.synchronize()
    n = max(5, int(seconds * 1000.0 / max(s.elapsed_time(e), 1e-3)) + 1)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n, n


def row_bound(A, X, k, torch):
    """2 n 2^-53 sum_j |a_rj x_jc| per row r and column c, on the device from the exported CRS arrays"""
    nRow = A.scalar("nRow")
    ptr = torch.from_numpy(A.array("ptr", np.int32).astype(np.int64)).cuda()
    idx = torch.from_numpy(A.array("idx", np.int32).astype(np.int64)).cuda()
    val = torch.from_numpy(A.array("val", np.float64)).cuda().abs_()
    lens = ptr[1:] - ptr[:-1]
    rows = torch.repeat_interleave(torch.arange(nRow, device="cuda"), lens)
    out = torch.zeros(nRow, k, dtype=torch.float64, device="cuda")
    for j in range(k):
        out[:, j].index_add_(0, rows, val * X[idx, j].abs())
    return out * (2.0 * lens.double() * 2.0 ** -53)[:, None] * 1.01


def fp32_within(A, X, Y, prec, torch):
    """Every Y[r, c] within the precision's bound of the fp64 row sum of the exact products (see the module docstring)."""
    nRow = A.scalar("nRow")
    ptr = torch.from_numpy(A.array("ptr", np.int32).astype(np.int64)).cuda()
    idx = torch.from_numpy(A.array("idx", np.int32).astype(np.int64)).cuda()
    val = torch.from_numpy(A.array("val", np.float64)).cuda()          # the fp32 values, widened exactly
    lens = ptr[1:] - ptr[:-1]
    rows = torch.repeat_interleave(torch.arange(nRow, device="cuda"), lens)
    n = lens.double()
    for j in range(X.shape[1]):
        p = val * X[idx, j].double()
        s = torch.zeros(nRow, dtype=torch.float64, device="cuda").index_add_(0, rows, p)
        mag = torch.zeros(nRow, dtype=torch.float64, device="cuda").index_add_(0, rows, p.abs())
        lim = n * 2.0 ** -53 * mag
        if prec == 2:
            lim += 2.0 ** -24 * s.abs() + n * 2.0 ** -53 * mag + 2.0 ** -149
        else:
            lim += (n + 1) * 2.0 ** -24 * mag + (n + 1) * 2.0 ** -149
        if not bool(((Y[:, j].double() - s).abs() <= lim).all()):
            return False
    return True


def run_config_f32(sp, torch, name, ks, seconds, prec):
    kind, p0, p1, seed, desc = CONFIGS[name]
    d = sp.DeviceCoo(kind, p0, p1, seed)
    A = sp.SpMatOpt("crs", precision=prec).convert_device(d)
    d.free()
    nRow, nCol, nnz = A.scalar("nRow"), A.scalar("nCol"), A.scalar("nNnz")
    mk = A.scalar("multi_kernel_f32")
    res = {"config": name, "precision": prec, "matrix": desc, "nRow": nRow, "nCol": nCol, "nnz": nnz, "multi_kernel": mk,
           "multi_kernel_name": KERNELS.get(mk, "?"), "single_kernel": A.scalar("crs_kernel"), "k": []}
    g = torch.Generator(device="cuda").manual_seed(7)
    for k in ks:
        X = torch.rand(nCol, k, dtype=torch.float32, device="cuda", generator=g) * 2 - 1
        Y = torch.full((nRow, k), float("nan"), dtype=torch.float32, device="cuda")
        xs = [X[:, j].contiguous() for j in range(k)]
        ys = [torch.full((nRow,), float("nan"), dtype=torch.float32, device="cuda") for _ in range(k)]

        def multi():
            A.multiply_multi_f32(k, X.data_ptr(), k, Y.data_ptr(), k, torch.cuda.current_stream().cuda_stream)

        def singles():
            for j in range(k):
                A.multiply_f32(xs[j].data_ptr(), ys[j].data_ptr(), torch.cuda.current_stream().cuda_stream)
        t_multi, n_multi = timed(multi, seconds, torch)
        t_single, n_single = timed(singles, seconds, torch)
        Ys = torch.stack(ys, dim=1)
        bits = bool(torch.equal(Y.view(torch.int32), Ys.view(torch.int32)))
        # the row-chunk stream keeps the single multiply's order: anything but its bits is a failure
        within = bits or (mk != 1 and fp32_within(A, X, Y, prec, torch) and fp32_within(A, X, Ys, prec, torch))
        nbytes = 8 * nnz + 4 * (nRow + 1) + 4 * k * (nCol + nRow)
        row = {"k": k, "multi_ms": t_multi, "multi_calls": n_multi, "singles_ms": t_single, "singles_calls": n_single,
               "multi_ms_per_vector": t_multi / k, "singles_ms_per_vector": t_single / k,
               "speedup": t_single / t_multi,
               "multi_gflops": 2.0 * nnz * k / (t_multi * 1e6), "singles_gflops": 2.0 * nnz * k / (t_single * 1e6),
               "bytes": nbytes, "multi_gbs": nbytes / (t_multi * 1e6),
               "parity": "bits" if bits else ("both within the fp32 bound" if within else
                                              "NOT the bits of multiply_f32" if mk == 1 else "OUTSIDE the fp32 bound")}
        print("%s p%d k=%d  multi %.3f ms (%.3f/vector, %.0f GFLOP/s, %.0f GB/s)  %d singles %.3f ms  x%.2f  %s" % (
            name, prec, k, t_multi, t_multi / k, row["multi_gflops"], row["multi_gbs"], k, t_single, row["speedup"],
            row["parity"]), flush=True)
        res["k"].append(row)
        del X, Y, xs, ys, Ys
    A.destroy()
    torch.cuda.empty_cache()
    return res


def run_config(sp, torch, name, ks, seconds):
    kind, p0, p1, seed, desc = CONFIGS[name]
    d = sp.DeviceCoo(kind, p0, p1, seed)
    A = sp.SpMatOpt("crs").convert_device(d)
    d.free()
    nRow, nCol, nnz = A.scalar("nRow"), A.scalar("nCol"), A.scalar("nNnz")
    mk = A.scalar("multi_kernel")
    res = {"config": name, "matrix": desc, "nRow": nRow, "nCol": nCol, "nnz": nnz, "multi_kernel": mk,
           "multi_kernel_name": KERNELS.get(mk, "?"), "single_kernel": A.scalar("crs_kernel"), "k": []}
    g = torch.Generator(device="cuda").manual_seed(7)
    bound = None
    for k in ks:
        X = torch.rand(nCol, k, dtype=torch.float64, device="cuda", generator=g) * 2 - 1
        Y = torch.full((nRow, k), float("nan"), dtype=torch.float64, device="cuda")
        xs = [X[:, j].contiguous() for j in range(k)]
        ys = [torch.full((nRow,), float("nan"), dtype=torch.float64, device="cuda") for _ in range(k)]

        def multi():
            A.multiply_multi(k, X.data_ptr(), k, Y.data_ptr(), k, torch.cuda.current_stream().cuda_stream)

        def singles():
            for j in range(k):
                A.multiply(xs[j].data_ptr(), ys[j].data_ptr(), torch.cuda.current_stream().cuda_stream)
        t_multi, n_multi = timed(multi, seconds, torch)
        t_single, n_single = timed(singles, seconds, torch)
        Ys = torch.stack(ys, dim=1)
        bits = bool(torch.equal(Y.view(torch.int64), Ys.view(torch.int64)))
        within = bits
        if not bits:
            bound = row_bound(A, X, k, torch)
            within = bool(((Y - Ys).abs() <= bound).all())
        nbytes = 12 * nnz + 4 * (nRow + 1) + 8 * k * (nCol + nRow)
        row = {"k": k, "multi_ms": t_multi, "multi_calls": n_multi, "singles_ms": t_single, "singles_calls": n_single,
               "multi_ms_per_vector": t_multi / k, "singles_ms_per_vector": t_single / k,
               "speedup": t_single / t_multi,
               "multi_gflops": 2.0 * nnz * k / (t_multi * 1e6), "singles_gflops": 2.0 * nnz * k / (t_single * 1e6),
               "bytes": nbytes, "multi_gbs": nbytes / (t_multi * 1e6),
               "parity": "bits" if bits else ("within row bound" if within else "OUTSIDE row bound")}
        print("%s k=%d  multi %.3f ms (%.3f/vector, %.0f GFLOP/s, %.0f GB/s)  %d singles %.3f ms  x%.2f  %s" % (
            name, k, t_multi, t_multi / k, row["multi_gflops"], row["multi_gbs"], k, t_single, row["speedup"],
            row["parity"]), flush=True)
        res["k"].append(row)
        del X, Y, xs, ys, Ys
    A.destroy()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_multi.json")
    ap.add_argument("--configs", default="c5,c4,c3,c2")
    ap.add_argument("--ks", default="1,2,4,8")
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--precision", default="0", help="comma list of 0 (fp64 multiply_multi), 1, 2 (multiply_multi_f32)")
    a = ap.parse_args()
    import torch
    import singlespmv_b200 as sp
    assert sp.device_count() > 0, "bench_multi.py needs a CUDA device"
    ks = [int(k) for k in a.ks.split(",")]
    out = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "date": time.strftime("%Y-%m-%d"),
           "seconds_per_window": a.seconds, "configs": []}
    print("card:", out["card"], flush=True)
    for prec in [int(p) for p in a.precision.split(",")]:
        for name in a.configs.split(","):
            if prec:
                out["configs"].append(run_config_f32(sp, torch, name, ks, a.seconds, prec))
            else:
                out["configs"].append(run_config(sp, torch, name, ks, a.seconds))
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_multi.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
