#!/bin/bash
# One gpurun call: the round-2 measurement set (bench lines of every config, randomised S, large batch, K4 roofline, ncu traffic captures).
OUT=gpurun_out/${1:-r02m}
mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw,memory.total --format=csv > $OUT/gpu.txt 2>&1
for cfg in cfg1 cfg2 cfg3 cfg5; do
  echo "== bench $cfg"; timeout 900 python bench.py --config $cfg --no-cpu-baseline 2>&1 | tail -1 | tee $OUT/bench_$cfg.json | cut -c1-160
done
echo "== bench cfg4 random S"; timeout 600 python bench.py --random-steps --no-cpu-baseline --no-eval 2>&1 | tail -1 | tee $OUT/bench_cfg4_randomS.json | cut -c1-160
echo "== bench cfg4 B=1024"; timeout 600 python bench.py --batch 1024 --steps 10 --no-cpu-baseline --no-eval 2>&1 | tail -1 | tee $OUT/bench_cfg4_b1024.json | cut -c1-160
echo "== k4 roofline"; timeout 300 python scripts/k4_roofline.py 2>&1 | tail -1 | tee $OUT/k4_roofline.json | cut -c1-300
echo "== ncu traffic cfg4"; timeout 900 ncu --set full --clock-control none -k regex:"tc_gemm|rw_wgrad|umnn_fwd_tc3|dag_l1" -s 56 -c 14 -o $OUT/prof_cfg4 python bench.py --steps 3 --warmup 3 --no-eval --no-cpu-baseline --cuda-graph off > $OUT/ncu_cfg4.log 2>&1; tail -2 $OUT/ncu_cfg4.log | cut -c1-200
ncu -i $OUT/prof_cfg4.ncu-rep --page raw --csv > $OUT/prof_cfg4_raw.csv 2>/dev/null; rm -f $OUT/prof_cfg4.ncu-rep   # gpurun_out travels back only below 64 MiB
echo "== ncu traffic cfg5"; timeout 900 ncu --set full --clock-control none -k regex:"tc_gemm|dag_l1" -s 36 -c 9 -o $OUT/prof_cfg5 python bench.py --config cfg5 --steps 3 --warmup 3 --no-eval --no-cpu-baseline --cuda-graph off > $OUT/ncu_cfg5.log 2>&1; tail -2 $OUT/ncu_cfg5.log | cut -c1-200
ncu -i $OUT/prof_cfg5.ncu-rep --page raw --csv > $OUT/prof_cfg5_raw.csv 2>/dev/null; rm -f $OUT/prof_cfg5.ncu-rep
ls -la $OUT
