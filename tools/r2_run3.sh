#!/bin/bash
# Runs ON THE GPU BOX: parity tests, default bench (all legs), gather microbenchmark, binary-level end to end, ncu captures.
mkdir -p gpurun_out; O=gpurun_out; T=${1:-r2c}
( timeout 1700 python -m pytest tests -m gpu -x -q 2>&1 | tail -15 ) | tee $O/${T}_pytest.log
timeout 900 python bench.py --steps 5 --warmup 3 > $O/${T}_bench.json 2> $O/${T}_bench.err || tail -20 $O/${T}_bench.err
python tools/bench_summary.py $O/${T}_bench.json
timeout 900 python tools/exp_r2c.py > $O/${T}_exp.jsonl 2> $O/${T}_exp.err || tail -5 $O/${T}_exp.err
cat $O/${T}_exp.jsonl | cut -c1-200
timeout 1200 python tools/e2e_binaries.py --config c2 --reads 4000000 --ref-reads 40000 --out $O/${T}_e2e_binaries.json 2>&1 | tail -12
timeout 900 ncu --set full --clock-control none --import-source on -k regex:search_kernel -s 1 -c 1 -f -o $O/${T}_c2_search_count \
    python bench.py --mode count --legs '' --steps 1 --warmup 1 --no-cpu-baseline --no-gather > $O/${T}_ncu_search.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:locate_kernel -s 1 -c 1 -f -o $O/${T}_c2_locate_kernel \
    python bench.py --mode locate --legs '' --steps 1 --warmup 1 --no-cpu-baseline --no-gather > $O/${T}_ncu_locate.log 2>&1
ls -la $O | tail -8
