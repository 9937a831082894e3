#!/bin/bash
# The GPU measurements of r03f, in three calls (each under ten minutes):
#   run_r03f.sh sweep   build, smoke(), the join tests, and a sweep of the point tree's bucket size over prebuilt
#                       libraries (build/lib_b<B>.so: c2b_join.cuh with JN_BUCKET = B, the build's nvcc flags; B = 4 is
#                       this change) with profiles/join_probe.py --resident-only
#   run_r03f.sh probe   build, profiles/join_probe.py (profiles/r03f_join_probe.json), the default bench line
#   run_r03f.sh suite   build, the whole GPU suite
cd "$(dirname "$0")/.." || exit 1
OUT=build/r03f_out
SO=city2ba_b200/libcity2ba_cuda.so
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/gpu.txt 2>&1
cat $OUT/gpu.txt
timeout 400 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $OUT/smoke.txt 2>&1
echo "build+smoke rc $?"; tail -1 $OUT/smoke.txt
case "$1" in
  sweep)
    cp -p $SO build/lib_b4.so
    timeout 300 python -m pytest tests/test_gpu_join.py tests/test_oracle_join.py -q -rs > $OUT/pytest_join.txt 2>&1
    echo "pytest join rc $?"; tail -3 $OUT/pytest_join.txt
    for b in 1 2 4 8 16; do
      cp -p build/lib_b$b.so $SO
      timeout 100 python profiles/join_probe.py --resident-only --repeats 3 --out $OUT/sweep_b$b.json \
        > $OUT/sweep_b$b.txt 2>&1
      echo "B=$b rc $? $(grep -o '"median": [0-9.]*' $OUT/sweep_b$b.json | tr '\n' ' ')"
    done
    cp -p build/lib_b4.so $SO ;;
  probe)
    timeout 300 python profiles/join_probe.py --out $OUT/r03f_join_probe.json > $OUT/probe.txt 2>&1
    echo "probe rc $?"; tail -c 600 $OUT/probe.txt
    timeout 200 python bench.py --gpus 1 --steps 10 --warmup 3 > $OUT/bench_cfg4.json 2> $OUT/bench.err
    echo "bench rc $?"; cut -c1-300 $OUT/bench_cfg4.json ;;
  suite)
    timeout 500 python -m pytest tests -m gpu -q -rs > $OUT/pytest_gpu.txt 2>&1
    echo "pytest rc $?"; tail -3 $OUT/pytest_gpu.txt ;;
esac
