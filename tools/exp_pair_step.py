#!/usr/bin/env python3
"""search_kernel alone with and without the pair directory (RBG_PAIR=0 / 1), alternated, on the `small` index that
bench.py builds: 150 bp exact and noisy (1 % substitutions, 0.1 % N) reads, seed table k = 10, count only.  Also checks the
pair decode at sampled positions of the index (rbg_selftest_pair) and records R2 / R and the directory sizes.

  python tools/exp_pair_step.py [--reads 4000000] [--rounds 5] [--out profiles/pair_step_small.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import rbformats as F  # noqa: E402
from tools import synth  # noqa: E402

import rowbowt_b200 as rb  # noqa: E402
from rowbowt_b200 import RBG_COUNT  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4_000_000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pair_step_small.jsonl"))
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    recs = []
    with tempfile.TemporaryDirectory() as tmp:
        panel = synth.make_panel(*synth.CONFIGS["small"])
        prefix = os.path.join(tmp, "small")
        synth.build_index_gpu(panel, prefix, markers=False)
        bwt = F.read_rbwt(prefix + ".rbwt")
        heads, lens = np.ascontiguousarray(bwt.heads, np.uint8), np.ascontiguousarray(bwt.lens, np.uint64)
        codes = np.zeros(bwt.n, np.uint8)
        chk, nl, nc = C.c_uint64(), C.c_uint64(), C.c_uint64()
        rc = rb.lib().rbg_selftest_pair(bwt.n, heads.ctypes.data, lens.ctypes.data, bwt.R, 0, 9973, codes.ctypes.data,
                                        C.byref(chk), C.byref(nl), C.byref(nc))
        assert rc == 0, rc
        r2 = 1 + int(np.count_nonzero(np.diff(codes)))
        ix = {}
        for pair in ("0", "1"):
            os.environ["RBG_PAIR"] = pair
            ix[pair] = rb.GpuIndex.open(prefix)
            ix[pair].build_ftab(10)
        del os.environ["RBG_PAIR"]
        info = ix["1"].info()
        head = {"gpu": gpu, "n": bwt.n, "R": bwt.R, "R2": r2, "R2_over_R": r2 / bwt.R, "pair_bytes": info.pair_bytes,
                "pair_window": info.pair_window, "dir_bytes": info.dir_bytes, "window": info.window,
                "pair_lines": nl.value, "pair_cluster_windows": nc.value, "selftest_checks": chk.value}
        assert info.pair_bytes > 0 and ix["0"].info().pair_bytes == 0
        print(json.dumps(head), flush=True)
        recs.append(head)
        for name, err, nr in (("exact", 0.0, 0.0), ("noisy", 0.01, 0.001)):
            reads = synth.make_reads(panel, a.reads, err_rate=err, n_rate=nr)[0]
            batch = (reads.reshape(-1), np.arange(0, reads.size + 1, reads.shape[1], dtype=np.uint64))
            staged = {p: ix[p].upload(batch) for p in ix}
            for p in ix:                                            # warm-up
                ix[p].query_staged(staged[p], RBG_COUNT)
            sums = {p: ix[p].query_staged(staged[p], RBG_COUNT, checksum=True) for p in ix}
            assert sums["0"] == sums["1"], name
            ms = {p: [] for p in ix}
            steps, lines = {}, {}
            for _ in range(a.rounds):
                for p in ix:
                    ix[p].query_staged(staged[p], RBG_COUNT)
                    st = ix[p].stats()
                    ms[p].append(st.ms_search)
                    steps[p], lines[p] = st.lf_steps, st.lf_lines
            assert steps["0"] == steps["1"], name
            rec = {"reads": name, "n_reads": a.reads, "ms_search_single": ms["0"], "ms_search_pair": ms["1"],
                   "median_speedup": float(np.median(ms["0"]) / np.median(ms["1"])), "lf_steps": steps["0"],
                   "lf_lines_single": lines["0"], "lf_lines_pair": lines["1"], "checksum": sums["1"]}
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
