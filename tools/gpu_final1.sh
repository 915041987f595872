#!/bin/bash
# round-2 final single-GPU session: full GPU suite, bench line, launch list, ncu capture of the walk
set -u
O=gpurun_out
mkdir -p $O
timeout 2400 python -m pytest tests -m gpu -x -q > $O/pytest_gpu_final.log 2>&1; echo "pytest rc=$?" > $O/final1.log
python bench.py > $O/bench_final_1gpu.json 2> $O/bench_final_1gpu.err; echo "bench rc=$?" >> $O/final1.log
python bench.py --impl reference --steps 3 --warmup 1 > $O/bench_final_ref.json 2> $O/bench_final_ref.err; echo "bench ref rc=$?" >> $O/final1.log
python -c "import __graft_entry__ as g; g.smoke()" > $O/smoke_final.log 2>&1; echo "smoke rc=$?" >> $O/final1.log
ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv --log-file $O/r2_bench_launches.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu --no-c5 > $O/ncu_bench_final.log 2>&1; echo "ncu list rc=$?" >> $O/final1.log
ncu --set full --clock-control none --import-source on -k regex:walk_warp2 -c 1 -f -o $O/r2_walk_final \
    python tools/tree_bench.py > $O/ncu_walk_final.log 2>&1; echo "ncu walk rc=$?" >> $O/final1.log
python tools/tree_bench.py > $O/tree_bench_final.log 2>&1
python tools/tree_bench.py --dist clustered >> $O/tree_bench_final.log 2>&1
python tools/tree_bench.py --dist box >> $O/tree_bench_final.log 2>&1
python tools/tree_bench.py --n 16777216 >> $O/tree_bench_final.log 2>&1
cat $O/final1.log; tail -3 $O/pytest_gpu_final.log; cat $O/smoke_final.log | tail -2; grep "build\|^walk " $O/tree_bench_final.log | cut -c1-110
