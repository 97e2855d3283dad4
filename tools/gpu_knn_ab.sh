#!/bin/bash
# A/B of the shipped library against prebuilt variant libraries: $1 is the path of a variant library,
# or several separated by ';' (named variant0, variant1, ...).  The source has no tuning macros, so a
# variant is a library built from another tree, e.g. the parent commit checked out in a git worktree
# and built there with `python -m imagescry_b200._build`.  Every case alternates shipped / variant /
# shipped / variant in fresh processes, so that the GPU's thermal state (which moves these timings by
# several per cent) hits both alike.  The shipped library is restored afterwards.  $2 = "notest" skips
# the knn tests on the shipped library.
mkdir -p gpurun_out
LIB=imagescry_b200/lib/libimagescry_b200.so
cases=("knn --d 256 --k 10" "knn --d 64 --k 10" "knn --d 128 --k 16" "knn --d 1280 --k 10" "knn --d 256 --k 100" "graph --n 500000 --d 256 --k 10 --iters 3 --warm 1" "graph --n 131072 --d 256 --k 10")
# ISX_AB_CASES="preprocess --case nhwc_f32 --batch 4096;preprocess --case nhwc_bf16 --batch 4096" overrides the list
if [ -n "$ISX_AB_CASES" ]; then IFS=';' read -r -a cases <<< "$ISX_AB_CASES"; fi
IFS=';' read -r -a variants <<< "$1"
for v in "${variants[@]}"; do [ -f "$v" ] || { echo "no such library: $v"; exit 1; }; done
cp $LIB /tmp/lib_shipped.so
{
  if [ "$2" != "notest" ]; then timeout 900 python -m pytest tests/test_gpu_knn.py tests/test_gpu_guard_bands.py -x -q -m gpu 2>&1 | tail -2; fi
  names=(shipped)
  for i in "${!variants[@]}"; do cp "${variants[$i]}" /tmp/lib_variant$i.so; names+=(variant$i); echo "variant$i = ${variants[$i]}"; done
  for args in "${cases[@]}"; do
    for rep in 1 2; do
      for which in "${names[@]}"; do
        cp /tmp/lib_$which.so $LIB
        echo -n "$which "; timeout 300 python tools/run_case.py $args --iters 5 --warm 3 2>&1 | tail -1
      done
    done
  done
} 2>&1 | tee gpurun_out/knn_ab.log
cp /tmp/lib_shipped.so $LIB
