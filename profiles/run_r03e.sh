#!/bin/bash
# The GPU measurements of r03e (profiles/r03e_ab_same_box.txt): same-box A/B of prebuilt libraries, a sweep of the
# hook grid_x_split, then the GPU suite, smoke() and the default bench line of this change.
#
# build/lib_<v>.so (nvcc flags of __graft_entry__.build()):
#   parent  af312d4: cells of max_dist/4 in x, y and z
#   new     this change: cells max_dist/4 in y and z, 1/grid_x_split of that in x (default 8)
#   packed  new + the fused pass's 32-point chunks packed across rows (measured and dropped)
cd "$(dirname "$0")/.." || exit 1
mkdir -p build/r03e_out
OUT=build/r03e_out
SO=city2ba_b200/libcity2ba_cuda.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $OUT/gpu.txt 2>&1
cat $OUT/gpu.txt
cp build/lib_new.so $SO
timeout 400 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > $OUT/smoke.txt 2>&1
echo "build+smoke rc $?"; tail -1 $OUT/smoke.txt
cp build/lib_new.so $SO

# the default bench line's resident pass (cfg4, grid rebuilt every step) and its secondary cfg3 / cfg5 lines
i=0
for v in parent new parent new; do
  i=$((i+1))
  cp build/lib_$v.so $SO
  timeout 300 python bench.py --gpus 1 --steps 10 --warmup 3 --no-cpu-baseline --no-exhaustive --no-noise --no-extras \
    > $OUT/ab_${i}_$v.json 2> $OUT/ab_${i}_$v.err
  echo "ab $i $v rc $?"
done

# the split, and the packed chunks at k = 1 and at the default k
cp build/lib_new.so $SO
for k in 1 2 4 8 16 8 1; do
  C2B_GRID_X_SPLIT=$k timeout 150 python profiles/shard_probe.py --workload cfg4 --shard 0/1 --steps 10 --drop-grid \
    > $OUT/sweep_k$k.txt 2>&1
  echo "k=$k $(tail -1 $OUT/sweep_k$k.txt)"
done
for k in 1 8; do
  for v in parent packed new packed new; do
    cp build/lib_$v.so $SO
    C2B_GRID_X_SPLIT=$k timeout 150 python profiles/shard_probe.py --workload cfg4 --shard 0/1 --steps 10 --drop-grid \
      > $OUT/pack_k${k}_$v.txt 2>&1
    echo "k=$k $v $(tail -1 $OUT/pack_k${k}_$v.txt)"
  done
done

cp build/lib_new.so $SO
timeout 900 python -m pytest tests -m gpu -q -rs > $OUT/pytest_gpu.txt 2>&1
echo "pytest rc $?"; tail -2 $OUT/pytest_gpu.txt
timeout 500 python bench.py --gpus 1 --steps 10 --warmup 3 > $OUT/bench_cfg4.json 2> $OUT/bench.err
echo "bench rc $?"; cut -c1-300 $OUT/bench_cfg4.json
