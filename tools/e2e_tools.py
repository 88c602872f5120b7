#!/usr/bin/env python3
"""Binary-level measurement of the two widened tools (SURVEY 8(f) rows 1 and 4), ON THE GPU BOX, next to the
unmodified reference binaries under oracle/_ref:

  rb_markers  greedy-seeding genotyping of N reads: ours (GPU) vs the reference with all host threads; the
              per-read output lines are compared as a multiset (the reference's order depends on thread timing)
  rb_build    raw .bwt/.ssa/.esa/.ma -> .rbwt/.tsa/.mab: ours (GPU) vs the reference; outputs compared with cmp

  python tools/e2e_tools.py [--markers-config c2] [--reads 1000000] [--ref-reads 100000]
                            [--build-config medium] [--out gpurun_out/e2e_tools.json]

--bin-dir times the rb_markers / rb_build of another build (for instance the parent commit's, built with
`make -C rowbowt_b200/csrc OUTDIR=DIR`), so that two builds can be alternated on the same machine.
"""
import argparse
import filecmp
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools import synth  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref")


def timed(cmd, out_path=None):
    t0 = time.perf_counter()
    with open(out_path or os.devnull, "wb") as f:
        p = subprocess.run(cmd, stdout=f, stderr=subprocess.PIPE)
    wall = time.perf_counter() - t0
    err = p.stderr.decode(errors="replace")
    if p.returncode != 0:
        raise RuntimeError("%s failed: %s" % (cmd, err[-800:]))
    return wall, err


def seconds(err, what):
    m = re.search(what + r"[^0-9]*([0-9.eE+-]+) seconds", err)
    return float(m.group(1)) if m else None


def markers(a, res):
    if a.markers_config not in synth.CONFIGS:
        res["rb_markers"] = {"skipped": "no config"}
        return
    L, H = synth.CONFIGS[a.markers_config]
    prefix = os.path.join(ROOT, "data", a.markers_config, a.markers_config)
    if not os.path.exists(prefix + ".mab"):
        res["rb_markers"] = {"skipped": "no .mab for %s" % a.markers_config}
        return
    panel = synth.make_panel(L, H)
    reads, _, _ = synth.make_reads(panel, a.reads, 150, seed=7, err_rate=0.005)
    fq, fq_ref = os.path.join(a.tmp, "mk.fq"), os.path.join(a.tmp, "mk_ref.fq")
    synth.write_fastq(reads, fq)
    synth.write_fastq(reads[:a.ref_reads], fq_ref)
    cores = os.cpu_count() or 1
    out = {"config": a.markers_config, "bin_dir": a.bin_dir, "reads": a.reads, "ref_reads": a.ref_reads, "host_cores": cores, "runs": []}
    for extra in ([], ["--heuristic", "--read-len", "150"]):
        o_all = os.path.join(a.tmp, "mk_ours.txt")
        wall, err = timed([os.path.join(a.bin_dir, "rb_markers")] + extra + [prefix, fq], o_all)
        q = seconds(err, "counting markers took")
        row = {"flags": " ".join(extra), "ours": {"wall_s": wall, "query_s": q, "reads_per_s_query": a.reads / q if q else None}}
        if os.path.exists(os.path.join(REF, "rb_markers")):
            o_ref, o_sub = os.path.join(a.tmp, "mk_ref.txt"), os.path.join(a.tmp, "mk_ours_sub.txt")
            rwall, rerr = timed([os.path.join(REF, "rb_markers"), "--threads", str(cores)] + extra + [prefix, fq_ref], o_ref)
            rq = seconds(rerr, "counting markers took")
            timed([os.path.join(a.bin_dir, "rb_markers")] + extra + [prefix, fq_ref], o_sub)
            same = sorted(open(o_ref, "rb").read().split(b"\n")) == sorted(open(o_sub, "rb").read().split(b"\n"))
            row["reference"] = {"wall_s": rwall, "query_s": rq, "threads": cores, "reads_per_s_query": a.ref_reads / rq if rq else None}
            row["lines_identical_as_multiset"] = bool(same)
            if q and rq:
                row["speedup_query"] = (a.reads / q) / (a.ref_reads / rq)
        out["runs"].append(row)
        print(json.dumps(row), flush=True)
    res["rb_markers"] = out


def build(a, res):
    prefix = os.path.join(ROOT, "data", a.build_config, a.build_config)
    if not os.path.exists(prefix + ".bwt"):
        res["rb_build"] = {"skipped": "no raw %s.bwt (python tools/synth.py %s data/%s --keep)" % (prefix, a.build_config, a.build_config)}
        return
    flags = ["-s"] + (["-m"] if os.path.exists(prefix + ".ma") else [])
    o_pre, r_pre = os.path.join(a.tmp, "b_ours"), os.path.join(a.tmp, "b_ref")
    out = {"config": a.build_config, "bwt_bytes": os.path.getsize(prefix + ".bwt"), "flags": " ".join(flags)}
    timed([os.path.join(a.bin_dir, "rb_build")] + flags + ["-o", o_pre, prefix])          # warm the page cache / the driver
    wall, err = timed([os.path.join(a.bin_dir, "rb_build")] + flags + ["-o", o_pre, prefix])
    out["ours"] = {"wall_s": wall, "stderr_summary": err.strip().split("\n")[-1]}
    if os.path.exists(os.path.join(REF, "rb_build")):
        rwall, _ = timed([os.path.join(REF, "rb_build")] + flags + ["-o", r_pre, prefix])
        out["reference"] = {"wall_s": rwall}
        out["speedup_wall"] = rwall / wall
        out["byte_identical"] = {suf: filecmp.cmp(o_pre + suf, r_pre + suf, shallow=False)
                                 for suf in (".rbwt", ".tsa", ".mab") if os.path.exists(r_pre + suf)}
    print(json.dumps(out), flush=True)
    res["rb_build"] = out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--markers-config", default="c2")
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--ref-reads", type=int, default=100_000)
    ap.add_argument("--build-config", default="medium")
    ap.add_argument("--bin-dir", default=os.path.join(ROOT, "rowbowt_b200"), help="directory of the rb_markers / rb_build to time")
    ap.add_argument("--tmp", default="/tmp/rbg_e2e")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "e2e_tools.json"))
    a = ap.parse_args()
    a.bin_dir = os.path.abspath(a.bin_dir)
    os.makedirs(a.tmp, exist_ok=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    res = {}
    markers(a, res)
    build(a, res)
    json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
