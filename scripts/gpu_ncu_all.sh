# ncu --set full, one launch of each format's multiply kernel on a BASELINE config (1 GPU).
# Each capture only after the same command exited 0 without ncu (B200_PROFILING.md).  Usage: bash scripts/gpu_ncu_all.sh [set]
mkdir -p gpurun_out
cap() { # name kernel-regex skip args...
  n=$1; k=$2; sk=$3; shift 3
  timeout 300 python bench.py "$@" --steps 2 --warmup 3 --no-cpu --no-also > gpurun_out/plain_$n.log 2>&1 && \
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:$k -s $sk -c 1 -f -o gpurun_out/prof_$n \
      python bench.py "$@" --steps 2 --warmup 3 --no-cpu --no-also > gpurun_out/ncu_$n.log 2>&1
  echo "$n rc=$?"
}
if [ "${1:-all}" = "late" ]; then   # kernels changed after the first capture round
cap dia7_c4    dia_spmv_tma       3 --workload c4 --format dia
cap dia3_c5    dia_spmv_tma       3 --workload c5 --format dia
cap csr5s16_c5 c5_compute_kernel  3 --workload c5 --format csr5
cap coo2_c5    coo_tile_kernel    3 --workload c5 --format coo
exit 0
fi
cap css_c2   tile_stream_kernel 9 --workload c2 --format css --n-block 3
cap jds_c2   jds_spmv_kernel    3 --workload c2 --format jds
cap csr5_c3  c5_compute_kernel  3 --workload c3 --format csr5
cap crs_c3   tile_stream_kernel 3 --workload c3 --format crs
cap coo_c5   coo_tile_kernel    3 --workload c5 --format coo
cap dia_c4   dia_spmv_tma       3 --workload c4 --format dia
cap ell_c4   ell_spmv_kernel    3 --workload c4 --format ell
cap crs_c1   tile_stream_kernel 3 --workload c1 --format crs
# launch list of the default bench command (shares per step)
timeout 300 python bench.py --steps 2 --warmup 3 --no-cpu --no-also > gpurun_out/plain_default.log 2>&1 && \
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/launches_default.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu --no-also > gpurun_out/ncu_default.log 2>&1
echo "launch list rc=$?"
