#!/bin/bash
# A/B of the row-chunk stream's column feed on one GPU, in one run of this script: the parent commit's tree against this one,
# alternating run by run, on the legs that run the row-chunk stream (c5 CRS, c5 SS, c5 CRS fp32, c1 CRS); then each leg
# once more on this tree with B200SPMV_CS_FEED=idx (the old feed in the new build), and the c5 CRS leg with 5 CTAs per
# SM and with 3 stages.  The dumped y of every run must equal the parent's bit for bit.
#
# Before the call, export the parent into an untracked directory of the working tree (ignored by git):
#   git archive --prefix=ab_parent/ <parent> | tar -x
# Usage: bash scripts/ab_chunk_feed.sh [reps (3)] [output directory (ab_out)]
#   -> the output directory: one bench line per run, summary.txt (the y dumps are compared, then deleted)
set -u
REPS=${1:-3}
mkdir -p "${2:-ab_out}"
OUT=$(cd "${2:-ab_out}" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.txt"
[ -f ab_parent/bench.py ] || { echo "ab_parent/ is missing: export the parent tree first"; exit 2; }
for t in . ab_parent; do
    (cd "$t" && python -c "import __graft_entry__ as g; g.build()") > "$OUT/build_$(basename "$(cd "$t" && pwd)").log" 2>&1 \
        || { echo "build of $t failed"; tail -20 "$OUT"/build_*.log; exit 1; }
done

LEGS=("c5crs|--workload c5" "c5ss|--workload c5 --format ss" "c5f32|--workload c5 --precision 1" "c1crs|--workload c1")
bench() {   # tree tag leg-args [env...]
    local dir=$1 tag=$2 args=$3
    shift 3
    mkdir -p "$OUT/y_$tag"
    (cd "$dir" && env "$@" timeout 600 python bench.py $args --no-cpu --dump-outputs "$OUT/y_$tag") > "$OUT/$tag.json" 2> "$OUT/$tag.err" \
        || { echo "run $tag failed"; tail -5 "$OUT/$tag.err"; }
}
for leg in "${LEGS[@]}"; do
    name=${leg%%|*}
    args=${leg#*|}
    for i in $(seq 1 "$REPS"); do
        bench ab_parent "${name}_parent_$i" "$args"
        bench . "${name}_branch_$i" "$args"
    done
    bench . "${name}_idxfeed_1" "$args" B200SPMV_CS_FEED=idx
done
bench . c5crs_ctas5_1 "--workload c5" B200SPMV_TMA_CTAS=5
bench . c5crs_stages3_1 "--workload c5" B200SPMV_TMA_S=3

python - "$OUT" "$REPS" <<'PY' | tee "$OUT/summary.txt"
import glob, json, os, sys
import numpy as np
out, reps = sys.argv[1], int(sys.argv[2])

def line(tag):
    try:
        return json.loads(open(os.path.join(out, tag + ".json")).read().strip().splitlines()[-1])
    except Exception:
        return None

def streamed(d, feed):
    """bytes one multiply streams, from the shapes: values, the column feed, x and y"""
    c = d["config"]
    nr, nc, nnz = c["nRow"], c["nCol"], c["nnz"]
    f32 = bool(c.get("options", {}).get("precision"))          # fp32 values and vectors
    vb = xb = 4 if f32 else 8
    cols = 4 * nnz + 4 * (nr + 1) if feed == "idx" else -(-nr // 256) * (16 + 256 // 32 + 256 // 2) * 4
    return vb * nnz + cols + xb * (nc + nr)

def same_y(a, b):
    ya, yb = (np.load(os.path.join(out, "y_" + t, "y.npy")) for t in (a, b))
    ra, rb = (os.path.join(out, "y_" + t, "y_rows.npy") for t in (a, b))
    rows_ok = (not os.path.exists(ra) and not os.path.exists(rb)) or np.array_equal(np.load(ra), np.load(rb))
    return rows_ok and ya.dtype == yb.dtype and np.array_equal(ya.view(np.uint8), yb.view(np.uint8))

print(open(os.path.join(out, "gpu.txt")).read().strip())
for name in ("c5crs", "c5ss", "c5f32", "c1crs"):
    runs = {}
    for tree in ("parent", "branch", "idxfeed"):
        for i in range(1, reps + 1):
            d = line("%s_%s_%d" % (name, tree, i))
            if d:
                runs.setdefault(tree, []).append((i, d))
    if "parent" not in runs or "branch" not in runs:
        print(name, "missing runs")
        continue
    d0 = runs["parent"][0][1]
    print("%s  dtype %s  alg_bytes %.3f GB  streamed: idx feed %.3f GB, dictionary feed %.3f GB"
          % (name, d0.get("dtype"), d0["roofline"]["alg_bytes_per_launch"] / 1e9, streamed(d0, "idx") / 1e9,
             streamed(d0, "dict") / 1e9))
    for tree, rs in runs.items():
        v = [d["value"] for _, d in rs]
        ms = [d["ms_per_step"] for _, d in rs]
        cv = [d["config"]["convert_ms"] for _, d in rs]
        print("  %-8s GFLOP/s %s  ms %s  convert_ms %s" % (tree, " ".join("%.1f" % x for x in v), " ".join("%.4f" % x for x in ms),
                                                         " ".join("%.1f" % x for x in cv)))
    pmax = max(d["value"] for _, d in runs["parent"])
    bmin = min(d["value"] for _, d in runs["branch"])
    print("  slowest branch / fastest parent = %.3f" % (bmin / pmax))
    ref = "%s_parent_1" % name
    diff = ["%s_%s_%d" % (name, tree, i) for tree, rs in runs.items() for i, _ in rs
            if "%s_%s_%d" % (name, tree, i) != ref and not same_y(ref, "%s_%s_%d" % (name, tree, i))]
    print("  y DIFFERS from %s: %s" % (ref, " ".join(diff)) if diff else "  y of every run equals that of " + ref)
for t in ("c5crs_ctas5_1", "c5crs_stages3_1"):
    d = line(t)
    print(t, "%.1f GFLOP/s" % d["value"] if d else "missing", "y same" if d and same_y("c5crs_parent_1", t) else "")
PY
rm -rf "$OUT"/y_*          # compared above; the dumps of c5 are 16 MiB each
