#!/usr/bin/env python3
"""search_kernel alone on the three directories the `small` index that bench.py builds can open with, alternated: layout 5
without the pair directory (RBG_LAYOUT=5 RBG_PAIR=0), layout 5 with it (RBG_PAIR=1) and the automatic choice (layout 7, plain
2-bit lines).  150 bp exact and noisy (1 % substitutions, 0.1 % N) reads, seed table k = 10, count and toehold search.  All
three must give the same checksum and count the same LF steps.

  python tools/exp_plain_layout.py [--reads 4000000] [--rounds 5] [--out profiles/plain_layout_small.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools import synth  # noqa: E402

import rowbowt_b200 as rb  # noqa: E402
from rowbowt_b200 import RBG_COUNT, RBG_LOCATE  # noqa: E402

FORMS = (("layout5", {"RBG_LAYOUT": "5", "RBG_PAIR": "0"}), ("pair", {"RBG_PAIR": "1"}), ("plain", {}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4_000_000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "plain_layout_small.jsonl"))
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    recs = []
    with tempfile.TemporaryDirectory() as tmp:
        panel = synth.make_panel(*synth.CONFIGS["small"])
        prefix = os.path.join(tmp, "small")
        synth.build_index_gpu(panel, prefix, markers=False)
        ix = {}
        for name, env in FORMS:
            for k in ("RBG_LAYOUT", "RBG_PAIR"):
                os.environ.pop(k, None)
            os.environ.update(env)
            ix[name] = rb.GpuIndex.open(prefix, sa=True)
            ix[name].build_ftab(10)
        for k in ("RBG_LAYOUT", "RBG_PAIR"):
            os.environ.pop(k, None)
        head = {"gpu": gpu}
        for name in ix:
            info = ix[name].info()
            head[name] = {"layout": info.layout, "window": info.window, "dir_bytes": info.dir_bytes, "pair_bytes": info.pair_bytes,
                          "n_lines": info.n_lines}
        head.update(n=ix["plain"].info().n, R=ix["plain"].info().r)
        assert head["plain"]["layout"] == 7 and head["pair"]["pair_bytes"] > 0 and head["layout5"]["pair_bytes"] == 0
        print(json.dumps(head), flush=True)
        recs.append(head)
        for reads_name, err, nr in (("exact", 0.0, 0.0), ("noisy", 0.01, 0.001)):
            reads = synth.make_reads(panel, a.reads, err_rate=err, n_rate=nr)[0]
            batch = (reads.reshape(-1), np.arange(0, reads.size + 1, reads.shape[1], dtype=np.uint64))
            staged = {p: ix[p].upload(batch) for p in ix}
            for mode_name, mode in (("count", RBG_COUNT), ("locate", RBG_LOCATE)):
                forms = list(ix) if mode == RBG_COUNT else ["layout5", "plain"]      # the pair directory serves counts only
                for p in forms:                                     # warm-up
                    ix[p].query_staged(staged[p], mode)
                sums = {p: ix[p].query_staged(staged[p], mode, checksum=True) for p in forms}
                assert len(set(sums.values())) == 1, (reads_name, mode_name, sums)
                ms = {p: [] for p in forms}
                steps, lines = {}, {}
                for _ in range(a.rounds):
                    for p in forms:
                        ix[p].query_staged(staged[p], mode)
                        st = ix[p].stats()
                        ms[p].append(st.ms_search)
                        steps[p], lines[p] = st.lf_steps, st.lf_lines
                assert len(set(steps.values())) == 1, (reads_name, mode_name, steps)
                rec = {"reads": reads_name, "mode": mode_name, "n_reads": a.reads, "lf_steps": steps["plain"], "checksum": sums["plain"],
                       "ms_search": ms, "median_ms": {p: float(np.median(ms[p])) for p in forms}, "lf_lines": lines,
                       "speedup_plain_vs": {p: float(np.median(ms[p]) / np.median(ms["plain"])) for p in forms if p != "plain"}}
                print(json.dumps(rec), flush=True)
                recs.append(rec)
            for p in ix:
                staged[p].free()
        for p in ix:
            ix[p].close()
    with open(a.out, "w") as f:
        for r in recs:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
