"""y := A^T x (b200spmv_multiply_transpose) against y := A x on the same handle, on one GPU.

    python scripts/bench_transpose.py --out DIR [--configs c5,c4,c3,c2] [--seconds 1.0] [--rounds 2]

For every config (generated on the device) the script runs CRS and the format profiles/r2_all_formats.md names best
(DIA for c5 / c4, CSR5 for c3, ELL for c2), and reports per format:
  - conversion wall time with transpose = 0 and 1 (host clock around convert + synchronise) and the device memory the
    handle holds in each case (torch.cuda.mem_get_info before and after; the generated COO is allocated before both);
  - CUDA-event time of multiply and of multiply_transpose on the transpose = 1 handle, each over at least --seconds
    after warm-ups, alternated --rounds times (the spread between rounds is the run-to-run spread);
  - GFLOP/s = 2 nnz / t and alg_bytes / t (t.alg_bytes for A^T), and the kernel each direction runs (crs_kernel,
    col_blocks, tma, ... with and without the t. prefix);
  - parity at the timed size.  c5 / c4 are symmetric: every t. array must equal A's and A^T x must have the bits of A x.
    c3 / c2: A^T x within 2 n 2^-53 sum|a x| per row of an fp64 row sum computed on the device from the t. CRS arrays
    (bench_multi.row_bound; both lie within half of that of the exact row sum).
Writes DIR/bench_transpose.json with the card's name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_multi import CONFIGS, ROOT, card, row_bound, timed  # noqa: E402

sys.path.insert(0, ROOT)

BEST = {"c5": "dia", "c4": "dia", "c3": "csr5", "c2": "ell"}
SYMMETRIC = ("c5", "c4")
ARRAYS = {"crs": ("ptr", "idx", "val"), "dia": ("ioff", "diag"), "csr5": ("row_ptr", "col_idx", "val"),
          "ell": ("col_idx", "val")}
KERNEL_SCALARS = ("crs_kernel", "col_blocks", "col_block_engine", "tma", "K", "nDiag", "sigma", "row_blocks")


class Prefixed:
    """A^T of a handle seen through the t. names (for bench_multi.row_bound)"""

    def __init__(self, A, prefix):
        self.A, self.prefix = A, prefix

    def scalar(self, n):
        return self.A.scalar(self.prefix + n)

    def array(self, n, dt):
        return self.A.array(self.prefix + n, dt)


def scalar_or_none(sp, A, n):
    try:
        return A.scalar(n)
    except sp.B200SpmvError:
        return None


def convert(sp, torch, d, fmt, transpose):
    """(handle, seconds, bytes held)"""
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    t0 = time.perf_counter()
    A = sp.SpMatOpt(fmt, transpose=transpose).convert_device(d)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    return A, sec, free0 - torch.cuda.mem_get_info()[0]


def run_format(sp, torch, name, d, fmt, seconds, rounds, crs_t):
    A0, conv0, mem0 = convert(sp, torch, d, fmt, 0)
    A0.destroy()
    T, conv1, mem1 = convert(sp, torch, d, fmt, 1)
    nRow, nCol, nnz = T.scalar("nRow"), T.scalar("nCol"), T.scalar("nNnz")
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.rand(nCol, dtype=torch.float64, device="cuda", generator=g) * 2 - 1      # A x
    u = torch.rand(nRow, dtype=torch.float64, device="cuda", generator=g) * 2 - 1      # A^T u
    y = torch.full((nRow,), float("nan"), dtype=torch.float64, device="cuda")
    yt = torch.full((nCol,), float("nan"), dtype=torch.float64, device="cuda")

    def fwd():
        T.multiply(x.data_ptr(), y.data_ptr(), torch.cuda.current_stream().cuda_stream)

    def bwd():
        T.multiply_transpose(u.data_ptr(), yt.data_ptr(), torch.cuda.current_stream().cuda_stream)
    t_fwd, t_bwd = [], []
    for _ in range(rounds):
        t_fwd.append(timed(fwd, seconds, torch)[0])
        t_bwd.append(timed(bwd, seconds, torch)[0])
    ab, abt = T.scalar("alg_bytes"), T.scalar("t.alg_bytes")
    res = {"format": fmt, "nRow": nRow, "nCol": nCol, "nnz": nnz,
           "convert_s": conv0, "convert_transpose_s": conv1, "held_bytes": mem0, "held_bytes_transpose": mem1,
           "multiply_ms": t_fwd, "multiply_transpose_ms": t_bwd,
           "multiply_gflops": 2.0 * nnz / (min(t_fwd) * 1e6), "multiply_transpose_gflops": 2.0 * nnz / (min(t_bwd) * 1e6),
           "alg_bytes": ab, "t_alg_bytes": abt,
           "multiply_gbs": ab / (min(t_fwd) * 1e6), "multiply_transpose_gbs": abt / (min(t_bwd) * 1e6),
           "kernel": {s: scalar_or_none(sp, T, s) for s in KERNEL_SCALARS},
           "t_kernel": {s: scalar_or_none(sp, T, "t." + s) for s in KERNEL_SCALARS}}
    # parity at the timed size
    if name in SYMMETRIC:
        same = all(np.array_equal(T.array("t." + a, np.uint8), T.array(a, np.uint8)) for a in ARRAYS[fmt])
        u.copy_(x)
        bwd()
        fwd()
        torch.cuda.synchronize()
        bits = bool(torch.equal(yt.view(torch.int64), y.view(torch.int64)))
        res["parity"] = "t. arrays = A's, A^T x = A x bit for bit" if same and bits else \
            "MISMATCH (arrays %s, bits %s)" % (same, bits)
    else:
        bwd()
        torch.cuda.synchronize()
        src = Prefixed(crs_t or T, "t.")                  # A^T's CRS arrays (of this config's CRS handle)
        ptr = torch.from_numpy(src.array("ptr", np.int32).astype(np.int64)).cuda()
        idx = torch.from_numpy(src.array("idx", np.int32).astype(np.int64)).cuda()
        val = torch.from_numpy(src.array("val", np.float64)).cuda()
        rows = torch.repeat_interleave(torch.arange(nCol, device="cuda"), ptr[1:] - ptr[:-1])
        s = torch.zeros(nCol, dtype=torch.float64, device="cuda").index_add_(0, rows, val * u[idx])
        del ptr, idx, val, rows
        ok = bool(((yt - s).abs() <= row_bound(src, u[:, None], 1, torch)[:, 0]).all())
        res["parity"] = "A^T x within the row bound" if ok else "A^T x OUTSIDE the row bound"
    print("%s %-4s  A x %.3f ms (%.0f GFLOP/s, %.0f GB/s)  A^T x %.3f ms (%.0f GFLOP/s, %.0f GB/s)  convert %.2f / %.2f s"
          "  held %.2f / %.2f GB  kernel %s / %s  %s" % (
              name, fmt, min(t_fwd), res["multiply_gflops"], res["multiply_gbs"], min(t_bwd),
              res["multiply_transpose_gflops"], res["multiply_transpose_gbs"], conv0, conv1, mem0 / 1e9, mem1 / 1e9,
              {k: v for k, v in res["kernel"].items() if v is not None},
              {k: v for k, v in res["t_kernel"].items() if v is not None}, res["parity"]), flush=True)
    del x, u, y, yt
    return T, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_transpose.json")
    ap.add_argument("--configs", default="c5,c4,c3,c2")
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    import torch
    import singlespmv_b200 as sp
    assert sp.device_count() > 0, "bench_transpose.py needs a CUDA device"
    out = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "date": time.strftime("%Y-%m-%d"),
           "seconds_per_window": a.seconds, "configs": []}
    print("card:", out["card"], flush=True)
    for name in a.configs.split(","):
        kind, p0, p1, seed, desc = CONFIGS[name]
        d = sp.DeviceCoo(kind, p0, p1, seed)
        rec = {"config": name, "matrix": desc, "formats": []}
        crs, r = run_format(sp, torch, name, d, "crs", a.seconds, a.rounds, None)
        rec["formats"].append(r)
        other, r = run_format(sp, torch, name, d, BEST[name], a.seconds, a.rounds, crs)
        rec["formats"].append(r)
        other.destroy()
        crs.destroy()
        d.free()
        torch.cuda.empty_cache()
        out["configs"].append(rec)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_transpose.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
