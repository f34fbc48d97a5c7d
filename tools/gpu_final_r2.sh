#!/bin/bash
# Round-2 single-GPU validation on a B200 box (run through gpurun): smoke, parity suite, every single-GPU BASELINE config through
# bench.py, the reference arm, projection and training timings, launch lists and ncu --set full captures of the hot kernels.
# Everything lands under gpurun_out/; what should be judged is copied into profiles/ afterwards.
mkdir -p gpurun_out
O=gpurun_out
echo "== smoke"; timeout 300 python __graft_entry__.py smoke 2>&1 | tail -2
echo "== pytest -m gpu"; timeout 900 python -m pytest tests -m gpu -q > $O/r2_pytest_gpu.log 2>&1; echo "rc=$?"; tail -3 $O/r2_pytest_gpu.log
echo "== bench headline"; timeout 600 python bench.py --steps 10 --warmup 3 > $O/r2_bench_headline.json 2> $O/r2_bench_headline.err; echo "rc=$?"; cut -c1-200 $O/r2_bench_headline.json
echo "== reference arm"; timeout 600 python bench.py --impl reference --steps 2 --warmup 1 > $O/r2_bench_reference.json 2> $O/r2_bench_reference.err; echo "rc=$?"; cut -c1-200 $O/r2_bench_reference.json
for c in cfg1 cfg2 cfg3 cfg4; do
  echo "== bench $c"; timeout 600 python bench.py --config $c --steps 10 --warmup 3 > $O/r2_$c.json 2> $O/r2_$c.err; echo "rc=$?"; cut -c1-160 $O/r2_$c.json
done
echo "== gemm"; timeout 200 python tools/bench_gemm.py > $O/r2_gemm.log 2>&1; cp $O/bench_gemm.json $O/r2_gemm_proj.json
echo "== train"; timeout 300 python tools/bench_train.py --steps 5 > $O/r2_train_step.json 2> $O/r2_train.err; cut -c1-300 $O/r2_train_step.json
if [ "$1" == "--ncu" ]; then
  echo "== launch list headline"; timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/r2_launches_headline.csv python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-e2e > /dev/null 2> $O/ncu1.err; echo "rc=$?"
  echo "== launch list cfg4"; timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file $O/r2_launches_cfg4.csv python bench.py --config cfg4 --steps 2 --warmup 3 --no-cpu-baseline --no-e2e > /dev/null 2> $O/ncu1b.err; echo "rc=$?"
  echo "== ncu --set full headline kernels"; timeout 900 ncu --set full --clock-control none --import-source on -k regex:"gat_gather4_kernel|gat_async_kernel|spmm_gather4_kernel|spmm_async_kernel|gemm_proj_ts_kernel" -s 12 -c 4 -o $O/r2_prof_headline -f python bench.py --steps 1 --warmup 3 --no-cpu-baseline --no-e2e > /dev/null 2> $O/ncu2.err; echo "rc=$?"
  echo "== ncu --set full training kernels"; timeout 900 ncu --set full --clock-control none --import-source on -k regex:"gat_bwd_kernel|spmm_gather4_kernel" -s 6 -c 4 -o $O/r2_prof_train -f python tools/ncu_train.py > /dev/null 2> $O/ncu3.err; echo "rc=$?"
  for r in r2_prof_headline r2_prof_train; do python tools/ncu_summary.py $O/$r.ncu-rep > $O/$r.json 2>/dev/null; done
fi
