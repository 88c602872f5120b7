#!/usr/bin/env python3
"""Times the GPU BWT builder (rowbowt_b200.build_bwt: FASTA -> .bwt/.ssa/.esa/.docs) on the benchmark panels: n, r, the
doubling rounds and the suffixes each round sorted, wall time per stage (parse / device / write), CUDA-event time of the
sort (initial sort + rounds) and of the BWT stage, and the device memory the build allocates.  The FASTA is written by
tools/synth.write_fasta to a temporary directory first (not timed as part of the build).  The card name and power limit
are read in the same call.  One JSON line per build to <out>/bwt_build.jsonl.

--builders u32,wide builds every config with each builder in turn (alternated, `RBG_BWT_WIDE=1` forcing the u64 builder;
configs of n >= 2^32 such as c5w always take it) and writes to <out>/bwt_build_wide.jsonl, every stats field included.

    python tools/exp_bwt_build.py [--out profiles] [--configs small,medium,c2] [--builders u32,wide] [--repeat 1]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

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
    ap.add_argument("--configs", default="small,medium,c2")
    ap.add_argument("--builders", default="", help="u32,wide: alternate the two builders (default: the library's choice)")
    ap.add_argument("--repeat", type=int, default=1)
    a = ap.parse_args()
    builders = [b for b in a.builders.split(",") if b] or [""]
    out_name = "bwt_build_wide.jsonl" if a.builders else "bwt_build.jsonl"
    os.makedirs(a.out, exist_ok=True)
    gpu = card()
    tmp = tempfile.mkdtemp(prefix="bwt_build_")
    try:
        for cfg in a.configs.split(","):
            panel = synth.make_panel(*synth.CONFIGS[cfg])
            fa = os.path.join(tmp, cfg + ".fa")
            t0 = time.time()
            synth.write_fasta(panel, fa)
            s_fasta = time.time() - t0
            pre = os.path.join(tmp, cfg)
            for rep in range(a.repeat):
                for b in builders:
                    if b == "wide":
                        os.environ["RBG_BWT_WIDE"] = "1"
                    else:
                        os.environ.pop("RBG_BWT_WIDE", None)
                    st = rb.build_bwt(fa, pre)
                    rec = dict(config=cfg, builder=b or "auto", rep=rep, **gpu, s_write_fasta=s_fasta, **st.as_dict())
                    rec["positions_per_s_sort"] = st.n / st.s_sort
                    line = json.dumps(rec)
                    print(line, flush=True)
                    with open(os.path.join(a.out, out_name), "a") as f:
                        f.write(line + "\n")
            os.environ.pop("RBG_BWT_WIDE", None)
            for suf in (".fa", ".bwt", ".ssa", ".esa", ".docs"):
                os.remove(pre + suf)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
