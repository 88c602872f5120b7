#!/usr/bin/env python3
"""Times the GPU marker-array builder (rowbowt_b200.build_marker_array: .mps + index phi -> .ma + .mab) on `small`, and on
c2 / c5w when data/ holds them: wall time split (read / layout / write), CUDA-event time of ma_rows_kernel and of the
block stage, rows/s and phi steps/s of ma_rows_kernel, records and words.  Two runs of each configuration, alternated.
The card name and power limit are read in the same call.  One JSON line per run to <out>/ma_build_<cfg>.jsonl.

    python tools/exp_ma_build.py [--out profiles] [--configs small,c2,c5w]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import rowbowt_b200 as rb  # noqa: E402
from tools import synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--configs", default="small,c2,c5w")
    ap.add_argument("--runs", type=int, default=2)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    tmp = tempfile.mkdtemp(prefix="ma_build_")
    where = {}
    for cfg in a.configs.split(","):
        pre = os.path.join(ROOT, "data", cfg, cfg)
        if not os.path.exists(pre + ".tsa"):
            if cfg != "small":
                print("%s: data/%s not present, skipped" % (cfg, cfg), file=sys.stderr)
                continue
            pre = os.path.join(tmp, cfg)
            synth.build_index_gpu(synth.make_panel(*synth.CONFIGS[cfg]), pre, markers=True)
        mps = os.path.join(tmp, cfg + ".mps")
        synth.write_mps(synth.make_panel(*synth.CONFIGS[cfg]), mps)
        where[cfg] = (pre, mps)
    gpu = card()
    for run in range(a.runs):
        for cfg, (pre, mps) in where.items():
            ma, mab = os.path.join(tmp, cfg + ".ma"), os.path.join(tmp, cfg + ".mab")
            st = rb.build_marker_array(pre, mps, ma, mab)
            rec = dict(config=cfg, run=run, **gpu, **st.as_dict())
            rec["rows_per_s_rows_kernel"] = st.rows / (st.ms_rows_kernel / 1e3)
            rec["phi_steps_per_s_rows_kernel"] = st.phi_steps / (st.ms_rows_kernel / 1e3)
            if os.path.exists(pre + ".mab"):
                with open(pre + ".mab", "rb") as f1, open(mab, "rb") as f2:
                    rec["mab_equals_index"] = f1.read() == f2.read()
            line = json.dumps(rec)
            print(line)
            with open(os.path.join(a.out, "ma_build_%s.jsonl" % cfg), "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
