#!/usr/bin/env bash
# Round-2 ncu evidence (run under gpurun on one GPU): each command first runs plain, then under ncu.
set -u
mkdir -p gpurun_out
run() {  # name, kernel regex, skip, command...
  local name=$1 regex=$2 skip=$3; shift 3
  "$@" > "gpurun_out/${name}_plain.log" 2>&1 &&
  ncu --set full --clock-control none --import-source on -k "regex:${regex}" -s "${skip}" -c 1 -o "gpurun_out/r2_${name}" "$@" > "gpurun_out/${name}_ncu.log" 2>&1
  echo "${name}: rc=$? $(tail -n 1 gpurun_out/${name}_plain.log | head -c 300)"
}
run knn_final knn_search_kernel 2 python tools/run_case.py knn --k 10 --iters 1 --warm 2
run knn_k100 knn_search_kernel 2 python tools/run_case.py knn --k 100 --iters 1 --warm 2
run knn_d256 knn_search_kernel 2 python tools/run_case.py knn --k 10 --d 256 --iters 1 --warm 2
run l2norm l2norm_cells 2 python tools/run_case.py l2norm --batch 2048 --iters 1 --warm 2
run syrk cov_syrk_kernel 2 python tools/run_case.py pcafit --n 65536 --d 1280 --iters 1 --warm 1
run project_staged l2norm_project_kernel 2 python tools/run_case.py project --batch 2048 --iters 1 --warm 2
# launch list of the bench command (cold-cache, serialised: compare shares)
python bench.py --steps 2 --warmup 3 --no-extra --no-verify --preheat 0.2 > gpurun_out/launch_plain.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file gpurun_out/r2_launches.csv python bench.py --steps 2 --warmup 3 --no-extra --no-verify --preheat 0.2 > gpurun_out/launch_ncu.log 2>&1
echo "launch list rc=$?"
