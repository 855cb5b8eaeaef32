#!/bin/bash
# One gpurun call for the round's evidence: GPU parity suite, smoke, both bench arms, ncu launch list + full captures.
TAG=${1:-r01zc}
OUT=gpurun_out/$TAG
mkdir -p $OUT
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw,memory.total --format=csv > $OUT/gpu.txt 2>&1
echo "== pytest -m gpu"; timeout 1200 python -m pytest tests -m gpu -q -p no:cacheprovider 2>&1 | tail -5 | tee $OUT/pytest_gpu.txt
echo "== smoke"; timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee $OUT/smoke.txt
echo "== bench default"; timeout 600 python bench.py 2>&1 | tail -1 | tee $OUT/bench_default.json
echo "== bench reference"; timeout 600 python bench.py --impl reference --steps 5 --warmup 3 2>&1 | tail -1 | tee $OUT/bench_reference.json
echo "== bench fused engine"; timeout 600 python bench.py --umnn-engine fused --gemm ffma --no-cpu-baseline --no-eval 2>&1 | tail -1 | tee $OUT/bench_ffma_only.json
echo "== bench B=1024"; timeout 600 python bench.py --batch 1024 --steps 10 --no-cpu-baseline --no-eval 2>&1 | tail -1 | tee $OUT/bench_b1024.json
echo "== bench cfg2/cfg3/cfg5/cfg1"
timeout 600 python bench.py --config cfg2 --steps 20 --no-cpu-baseline 2>&1 | tail -1 | tee $OUT/bench_cfg2.json
timeout 600 python bench.py --config cfg3 --steps 5 --no-cpu-baseline 2>&1 | tail -1 | tee $OUT/bench_cfg3.json
timeout 600 python bench.py --config cfg5 --steps 5 --no-cpu-baseline 2>&1 | tail -1 | tee $OUT/bench_cfg5.json
timeout 600 python bench.py --config cfg1 --steps 30 --no-cpu-baseline 2>&1 | tail -1 | tee $OUT/bench_cfg1.json
echo "== ncu launch list"
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 1200 --csv --log-file $OUT/launches.csv \
  python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-eval --cuda-graph off > $OUT/ncu_launches.log 2>&1
echo "== ncu full: tcgen05 GEMM kernels"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:"tc_gemm|rw_wgrad_kernel" -s 36 -c 12 -o $OUT/prof_gemms -f \
  python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-eval --cuda-graph off > $OUT/ncu_gemms.log 2>&1
tail -2 $OUT/ncu_gemms.log
ls -la $OUT
