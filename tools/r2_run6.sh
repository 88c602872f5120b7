#!/bin/bash
# Runs ON THE GPU BOX: parity tests, call-latency experiment.
mkdir -p gpurun_out; O=gpurun_out; T=${1:-r2f}
( timeout 1700 python -m pytest tests -m gpu -x -q 2>&1 | tail -15 ) | tee $O/${T}_pytest.log
timeout 1200 python tools/exp_r2e.py > $O/${T}_exp.jsonl 2> $O/${T}_exp.err || tail -5 $O/${T}_exp.err
python - <<PY
import json
for ln in open("$O/${T}_exp.jsonl"):
    d = json.loads(ln)
    print("call %-6s %8d reads x %d threads: %.3f ms per call  %.3g reads/s" % (d["mode"], d["reads"], d["host_threads"], d["ms_per_call"], d["reads_per_s"]))
PY
