#!/bin/bash
# A/B of the padding and ragged-end changes (ELL padding slots read no x; the entry streams' ragged ends read no x; row
# sums stored with + 0.0) on one GPU, in one run of this script: the parent commit's tree against this one, alternating
# run by run, on the legs that run the changed kernels.  Then one short run per tree of further config / format pairs
# whose kernels changed, for the y dumps only.  The dumped y of every run must equal the parent's bit for bit.
#
# Before the call, export the parent into an untracked directory of the working tree (ignored by git):
#   git archive --prefix=ab_parent/ <parent> | tar -x
# Usage: bash scripts/ab_special_values.sh [reps (3)] [output directory (ab_out)] [legs to run, e.g. c4ell,c2css,dumps (all)]
#   -> the output directory: one bench line per run, summary.txt (the y dumps are compared, then deleted)
set -u
REPS=${1:-3}
ONLY=${3:-}
wanted() { [ -z "$ONLY" ] || [[ ",$ONLY," == *",$1,"* ]]; }
mkdir -p "${2:-ab_out}"
OUT=$(cd "${2:-ab_out}" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.txt"
[ -f ab_parent/bench.py ] || { echo "ab_parent/ is missing: export the parent tree first"; exit 2; }
for t in . ab_parent; do
    (cd "$t" && python -c "import __graft_entry__ as g; g.build()") > "$OUT/build_$(basename "$(cd "$t" && pwd)").log" 2>&1 \
        || { echo "build of $t failed"; tail -20 "$OUT"/build_*.log; exit 1; }
done

LEGS=("c4ell|--workload c4 --format ell" "c4hyb|--workload c4 --format hyb"
      "c2ell|--workload c2 --format ell" "c2jds|--workload c2 --format jds" "c2ss|--workload c2 --format ss"
      "c2css|--workload c2 --format css" "c2ellf32|--workload c2 --format ell --precision 1" "c3crs|--workload c3 --format crs" "c3coo|--workload c3 --format coo"
      "c5crs|--workload c5" "c5coo|--workload c5 --format coo")
DUMPS=("c1crs|--workload c1 --format crs" "c1coo|--workload c1 --format coo" "c1ell|--workload c1 --format ell"
       "c1hyb|--workload c1 --format hyb" "c2crs|--workload c2 --format crs" "c2coo|--workload c2 --format coo"
       "c2hyb|--workload c2 --format hyb" "c4crs|--workload c4 --format crs" "c4coo|--workload c4 --format coo"
       "c5ell|--workload c5 --format ell" "c5hyb|--workload c5 --format hyb" "c5ellf32|--workload c5 --format ell --precision 1")
bench() {   # tree tag leg-args
    local dir=$1 tag=$2 args=$3
    mkdir -p "$OUT/y_$tag"
    (cd "$dir" && timeout 900 python bench.py $args --no-cpu --dump-outputs "$OUT/y_$tag") > "$OUT/$tag.json" 2> "$OUT/$tag.err" \
        || { echo "run $tag failed"; tail -5 "$OUT/$tag.err"; }
}
for leg in "${LEGS[@]}"; do
    name=${leg%%|*}
    wanted "$name" || continue
    for i in $(seq 1 "$REPS"); do
        bench ab_parent "${name}_parent_$i" "${leg#*|}"
        bench . "${name}_branch_$i" "${leg#*|}"
    done
done
for leg in "${DUMPS[@]}"; do
    name=${leg%%|*}
    wanted dumps || continue
    bench ab_parent "${name}_parent_1" "${leg#*|} --steps 2 --warmup 3"
    bench . "${name}_branch_1" "${leg#*|} --steps 2 --warmup 3"
done

names=()
for leg in "${LEGS[@]}"; do wanted "${leg%%|*}" && names+=("${leg%%|*}"); done
for leg in "${DUMPS[@]}"; do wanted dumps && names+=("${leg%%|*}"); done
python - "$OUT" "$REPS" "${names[@]}" <<'PY' | tee "$OUT/summary.txt"
import json, os, sys
import numpy as np
out, reps, names = sys.argv[1], int(sys.argv[2]), sys.argv[3:]

def line(tag):
    try:
        return json.loads(open(os.path.join(out, tag + ".json")).read().strip().splitlines()[-1])
    except Exception:
        return None

def same_y(a, b):
    ya, yb = (np.load(os.path.join(out, "y_" + t, "y.npy")) for t in (a, b))
    ra, rb = (os.path.join(out, "y_" + t, "y_rows.npy") for t in (a, b))
    rows_ok = (not os.path.exists(ra) and not os.path.exists(rb)) or np.array_equal(np.load(ra), np.load(rb))
    return rows_ok and ya.dtype == yb.dtype and np.array_equal(ya.view(np.uint8), yb.view(np.uint8))

print(open(os.path.join(out, "gpu.txt")).read().strip())
for name in names:
    runs = {}
    for tree in ("parent", "branch"):
        for i in range(1, reps + 1):
            d = line("%s_%s_%d" % (name, tree, i))
            if d:
                runs.setdefault(tree, []).append((i, d))
    if "parent" not in runs or "branch" not in runs:
        print(name, "missing runs")
        continue
    print("%s  dtype %s" % (name, runs["parent"][0][1].get("dtype")))
    for tree, rs in runs.items():
        print("  %-8s GFLOP/s %s  ms %s" % (tree, " ".join("%.1f" % d["value"] for _, d in rs),
                                            " ".join("%.4f" % d["ms_per_step"] for _, d in rs)))
    pmax = max(d["value"] for _, d in runs["parent"])
    bmin = min(d["value"] for _, d in runs["branch"])
    print("  slowest branch / fastest parent = %.3f" % (bmin / pmax))
    ref = "%s_parent_1" % name
    try:
        diff = ["%s_%s_%d" % (name, tree, i) for tree, rs in runs.items() for i, _ in rs
                if "%s_%s_%d" % (name, tree, i) != ref and not same_y(ref, "%s_%s_%d" % (name, tree, i))]
        print("  y DIFFERS from %s: %s" % (ref, " ".join(diff)) if diff else "  y of every run equals that of " + ref)
    except OSError as err:
        print("  y not dumped:", err)
PY
rm -rf "$OUT"/y_*          # compared above; the dumps of c5 are 16 MiB each
