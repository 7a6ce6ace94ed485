"""The reference's sweep workflow for the gpu architecture (script/eval_sbatch.sh, script/gen_todo.sh, log/format.cpp)."""
import os
import subprocess

import pytest

from conftest import load_golden
from singlespmv_b200.sweep import log_format, sweep

BLOCK = """++++++++++++++++++++++++++++++++++++++++
             Architecture\tGPU
             MatrixFormat\tCRS
                   Matrix\t%s
      Performance(GFLOPS)\t%s
                     nRow\t10
                     nCol\t10
                     nNnz\t%s
        EffectiveBW(GB/s)\t123.5
----------------------------------------
"""


def test_log_format_matches_reference_semantics():
    text = BLOCK % ("b.mtx", "2.5", "300") + BLOCK % ("a.mtx", "1.5", "300") + BLOCK % ("c.mtx", "4.0", "27")
    data = log_format.parse(text.splitlines(True))
    rows = log_format.table(data)
    assert [r.split("\t")[0] for r in rows] == ["c.mtx", "a.mtx", "b.mtx"]          # by nNnz, then Matrix (format.cpp:44)
    assert rows[0] == "c.mtx\tGPU\tCRS\t4.0\t10\t10\t27"
    assert log_format.table(data, roofline=True)[0].endswith("\t123.5\t\t")
    assert log_format.total_gflops(data) == 8.0                                        # log/sum.sh


def test_todo_roundtrip(tmp_path):
    rows = sweep.gen_todo()
    assert ("gpu", "b200-crs", "-DOPT_B200 -DB200_DEVICE_RESIDENT -DB200_FORMAT=CRS") in rows
    assert any(p == "b200-css-w4-n3" for _, p, _ in rows) and any(p == "b200-csr5-s16" for _, p, _ in rows)
    f = tmp_path / "todo.csv"
    f.write_text("# CRS\n\n" + "\n".join(",".join(r) for r in rows[:3]) + "\n#gpu,skipped,-DX\n")
    assert sweep.read_todo(str(f)) == rows[:3]


def test_sweep_builds_one_binary_per_row(tmp_path):
    exe = sweep.build("b200-ss-w8", "-DOPT_B200 -DB200_FORMAT=SS -DSEGMENT_WIDTH=8", str(tmp_path))
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage" in r.stdout


@pytest.mark.gpu
def test_sweep_end_to_end(tmp_path):
    from test_plugin_driver import write_mtx
    mtx = str(tmp_path / "fixture_10x10.mtx")
    write_mtx(mtx, load_golden("fixture_10x10"))
    rows = [("gpu", "b200-css-w4-n2", "-DOPT_B200 -DB200_FORMAT=CSS -DSEGMENT_WIDTH=4 -DN_BLOCK=2 -DB200_DEVICE_RESIDENT"),
            ("gpu", "b200-dia", "-DOPT_B200 -DB200_FORMAT=DIA")]
    env = dict(os.environ, SPMV_MIN_SECONDS="0.02", SPMV_NTRY="2")
    logs = sweep.run(rows, [mtx, "synth:lap2d5:40"], str(tmp_path / "log"), str(tmp_path / "bin"), env=env)
    assert len(logs) == 2
    assert sweep.run(rows, [mtx], str(tmp_path / "log"), str(tmp_path / "bin"), env=env) == []       # .lock -> skipped
    data = log_format.parse(open(logs[0]))
    assert [d["MatrixFormat"] for d in data] == ["CSS", "CSS"] and data[0]["N_BLOCK"] == "2"
    assert [r.split("\t")[0] for r in log_format.table(data)] == ["fixture_10x10.mtx", "synth:lap2d5:40"]
