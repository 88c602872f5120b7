#!/usr/bin/env python3
"""Binary-level end to end, ON THE GPU BOX: FASTQ file -> rb_align stdout, this repo's host driver
(rowbowt_b200/rb_align over librowbowt_gpu.so) next to the unmodified reference binary
(oracle/_ref/rb_align), same index, same FASTQ.

  python tools/e2e_binaries.py [--config c2] [--reads 2000000] [--ref-reads 40000] [--out gpurun_out/e2e.json]

--bin-dir times the rb_align of another build (for instance the parent commit's, built with
`make -C rowbowt_b200/csrc OUTDIR=DIR`), so that two builds can be alternated on the same machine.

For every flag set ("", -s, -m, -s -m):
  * wall time of our rb_align over the whole FASTQ (stdout to a file on the box's disk),
    its own "<load_s> <query_s>" stderr line, reads/s from both;
  * the reference over the FIRST --ref-reads records (it is single-threaded: ~10^4 reads/s), its own query time;
  * byte comparison of the reference's stdout with the head of ours (parity at BASELINE scale: identical text).
Nothing here is a bench.py number; the JSON goes to profiles/ as the host-pipeline record.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools import synth  # noqa: E402


def run(cmd, out_path):
    t0 = time.perf_counter()
    with open(out_path, "wb") as f:
        p = subprocess.run(cmd, stdout=f, stderr=subprocess.PIPE)
    wall = time.perf_counter() - t0
    err = p.stderr.decode(errors="replace").strip().split("\n")
    if p.returncode != 0:
        raise RuntimeError("%s failed: %s" % (cmd[0], err[-3:]))
    load_s, query_s = (float(x) for x in err[-1].split()[:2])
    run.host_stats = next((ln for ln in err if ln.startswith("host stages")), None)      # RBG_HOST_STATS=1
    return wall, load_s, query_s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2")
    ap.add_argument("--reads", type=int, default=2_000_000)
    ap.add_argument("--ref-reads", type=int, default=40_000)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--skip-locate", action="store_true", help="leave out the -s runs (their text output is ~1.4 KB per read)")
    ap.add_argument("--bin-dir", default=os.path.join(ROOT, "rowbowt_b200"), help="directory of the rb_align to time")
    ap.add_argument("--tmp", default="/tmp/rbg_e2e")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "e2e_binaries.json"))
    a = ap.parse_args()
    os.makedirs(a.tmp, exist_ok=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    L, H = synth.CONFIGS[a.config]
    prefix = os.path.join(ROOT, "data", a.config, a.config)
    panel = synth.make_panel(L, H)
    reads, _, _ = synth.make_reads(panel, a.reads, 150, seed=3)
    fq = os.path.join(a.tmp, "reads.fq")
    fq_ref = os.path.join(a.tmp, "reads_ref.fq")
    synth.write_fastq(reads, fq)
    synth.write_fastq(reads[:a.ref_reads], fq_ref)
    ours = os.path.join(os.path.abspath(a.bin_dir), "rb_align")
    ref = os.path.join(ROOT, "oracle", "_ref", "rb_align")
    have_ma = os.path.exists(prefix + ".mab")
    have_sa = os.path.exists(prefix + ".tsa")
    res = {"config": a.config, "bin_dir": os.path.dirname(ours), "reads": a.reads, "ref_reads": a.ref_reads, "gpus": a.gpus, "host_cores": os.cpu_count(),
           "fastq_bytes": os.path.getsize(fq), "runs": []}
    for flags in ([], ["-s"], ["-m"], ["-s", "-m"]):
        if ("-s" in flags and (not have_sa or a.skip_locate)) or ("-m" in flags and not have_ma):
            continue
        tag = "".join(f.strip("-") for f in flags) or "count"
        o_out = os.path.join(a.tmp, "ours_%s.txt" % tag)
        wall, load_s, query_s = run([ours] + flags + ["--gpus", str(a.gpus), prefix, fq], o_out)
        row = {"flags": " ".join(flags), "ours": {"wall_s": wall, "load_s": load_s, "query_s": query_s,
                                                    "reads_per_s_query": a.reads / query_s, "stdout_bytes": os.path.getsize(o_out)}}
        if run.host_stats:
            row["ours"]["host_stats"] = run.host_stats
        if os.path.exists(ref):
            r_out = os.path.join(a.tmp, "ref_%s.txt" % tag)
            rwall, rload, rquery = run([ref] + flags + [prefix, fq_ref], r_out)
            want = open(r_out, "rb").read()
            got = open(o_out, "rb").read(len(want))
            row["reference"] = {"wall_s": rwall, "load_s": rload, "query_s": rquery, "reads_per_s_query": a.ref_reads / rquery,
                                "stdout_bytes": len(want)}
            row["stdout_identical_on_ref_reads"] = bool(want == got)
            row["speedup_query"] = (a.reads / query_s) / (a.ref_reads / rquery)
        res["runs"].append(row)
        print(json.dumps(row), flush=True)
    json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
