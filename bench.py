#!/usr/bin/env python3
"""Benchmark of the rb_align query path on B200 (BASELINE.json metric: 150bp reads/s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--mode count|locate|markers|all]
                  [--impl reference] [--config c2|medium|small] [--reads R] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic reads (the whole
BASELINE config: 10M x 150bp reads against the 50 Mbp x 64 haplotype pfbwt-f index,
count-only by default = configs[1]).  `value` is measured with the batch resident in HBM;
`e2e` goes through the public C-ABI call rbg_query with pinned HOST buffers (H2D of the
reads and D2H of the results inside the timed region).  With --gpus N (launched under
torchrun) every rank holds an index replica and its own batch: weak scaling, no collective
on the data path (SURVEY.md §8(e)); torch.distributed is used only for the barrier and the
max-over-ranks of the device time.

--impl reference times the UNMODIFIED reference rb_align (oracle/_ref, compiled from
/root/reference by oracle/Makefile) on the host cores, same index, same reads.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from tools import synth  # noqa: E402

READ_LEN = 150
DATA = os.path.join(ROOT, "data")
MODES = {"count": 0, "locate": 1, "markers": 2, "all": 3}


# ------------------------------------------------------------------------------------------
def workload(config: str, log, tmpdir):
    """(name, index prefix, panel).  A config built by tools/synth.py and cached under data/ (git-ignored) is
    used as it is; otherwise `small` is built into tmpdir without the reference (synth.build_index_gpu, about a
    minute), so that a fresh checkout benchmarks the same index every time and writes nothing into the tree."""
    order = [config] if config != "auto" else ["c2", "medium", "small"]
    for cfg in order:
        prefix = os.path.join(DATA, cfg, cfg)
        if os.path.exists(prefix + ".rbwt"):
            L, H = synth.CONFIGS[cfg]
            return cfg, prefix, synth.make_panel(L, H)
    cfg = order[-1] if config != "auto" else "small"
    if cfg != "small":
        raise SystemExit("data/%s is not built: run `python tools/synth.py %s data/%s`" % (cfg, cfg, cfg))
    L, H = synth.CONFIGS[cfg]
    panel = synth.make_panel(L, H)
    prefix = os.path.join(tmpdir, cfg)
    print("bench: building the %s index in %s ..." % (cfg, tmpdir), file=log)
    synth.build_index_gpu(panel, prefix, markers=True, device=int(os.environ.get("LOCAL_RANK", "0")), log=log)
    return cfg, prefix, panel


def describe(cfg, n_reads):
    L, H = synth.CONFIGS[cfg]
    full = "" if (cfg == "c2" and n_reads == 10_000_000) else " [REDUCED: not the BASELINE config]"
    if cfg == "c5s":
        full = " [1/10-scale stand-in for BASELINE config 5 (64 Mbp x 2504): n > 2^32 rows]"
    return "synthetic %d bp reference x %d haplotypes (pfbwt-f index), %d x %dbp exact reads%s" % (L, H, n_reads, READ_LEN, full)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_ev = gpu, [], threading.Event()

    def run(self):
        while not self.stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_ev.wait(0.2)

    def summary(self):
        self.stop_ev.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, streaming copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def bind_to_gpu_numa_node(gpu: int):
    """Pins this process (its pinned staging buffers are first-touched by it) to the CPUs of the NUMA node the GPU
    hangs off, when the platform tells (sysfs).  Returns what was done, for the bench record."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(gpu), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        bdf = out.lower()[-12:] if out else None               # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return {"gpu_numa_node": node, "bound": False}
        cpus = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        allowed = ids & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"gpu_numa_node": node, "cpus": cpus, "bound": bool(allowed)}
    except Exception as e:          # noqa: BLE001
        return {"bound": False, "why": repr(e)[:80]}


def pinned_array(lib, nbytes, dtype):
    p = lib.rbg_host_alloc(nbytes)
    if not p:
        raise MemoryError("rbg_host_alloc")
    buf = (C.c_uint8 * nbytes).from_address(p)
    return np.frombuffer(buf, dtype=dtype), p


# ------------------------------------------------------------------------------------------
def reference_cmd(prefix, fq, mode):
    cmd = [os.path.join(ROOT, "oracle", "_ref", "rb_align")]
    if mode & 1:
        cmd.append("-s")
    if mode & 2:
        cmd.append("-m")
    return cmd + [prefix, fq]


def run_reference_shards(prefix, reads, mode, procs, tmpdir):
    """The reference rb_align is single-threaded (src/rb_align.cpp:162-193); all-core = one process
    per contiguous shard (BASELINE.md §3).  Returns (reads/s, slowest shard's own query seconds)."""
    from rowbowt_b200.shard import shard_bounds      # the same contiguous, order-preserving blocks the multi-rank path uses
    fqs = []
    for i in range(procs):
        a, b = shard_bounds(len(reads), procs, i)
        fq = os.path.join(tmpdir, "shard%d.fq" % i)
        synth.write_fastq(reads[a:b], fq, start_id=a)
        fqs.append(fq)
    ps = [subprocess.Popen(reference_cmd(prefix, fq, mode), stdout=subprocess.DEVNULL, stderr=subprocess.PIPE) for fq in fqs]
    qt = []
    for p in ps:
        err = p.communicate()[1].decode().strip().split("\n")
        if p.returncode != 0:
            raise RuntimeError("reference rb_align failed: %s" % err[-1])
        qt.append(float(err[-1].split()[1]))          # "<index_load_time> <total_query_time>"
    return len(reads) / max(qt), max(qt)


def reference_arm(args, rank, world, log, emit, tmpdir):
    if rank != 0:
        return
    mode = MODES[args.mode]
    base = {"impl": "reference", "metric": "150bp reads/s (%s)" % args.mode, "unit": "reads/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic"}
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "rb_align")):
        emit({"impl": "reference", "unavailable": "oracle/_ref/rb_align not built (run make -C oracle ref where /root/reference exists)"})
        return
    cfg, prefix, panel = workload(args.config, log, tmpdir)
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, args.ref_procs or cores))
    per_proc = args.ref_reads_per_proc
    n = per_proc * procs
    reads, _, _ = synth.make_reads(panel, n, READ_LEN, seed=3)
    vals = []
    with tempfile.TemporaryDirectory() as td:
        for it in range(args.warmup + args.steps):
            v, _ = run_reference_shards(prefix, reads, mode, procs, td)
            if it >= args.warmup:
                vals.append(v)
    v = float(np.mean(vals))
    sample = "%d reads (%d per process x %d processes) of the same workload per step" % (n, per_proc, procs)
    base.update({"value": v, "ms_per_step": 1e3 * n / v,
                 "config": {"workload": describe(cfg, args.reads), "mode": args.mode, "sample": sample},
                 "cpu_baseline": {"value": v, "unit": "reads/s", "cores": procs, "kind": "reference", "sample": sample},
                 "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    emit(base)


# ------------------------------------------------------------------------------------------
KERNEL_SOURCES = ("kernels.cu", "device_index.cuh", "leaf.cuh", "phi_slot.cuh", "layout.cpp", "layout.hpp")


def kernel_source_hash():
    """sha256 over the sources that define the kernels and the device layout: profiles/ncu_traffic.json entries carry
    the hash they were captured at, so a stale ncu figure is dropped instead of reported (VERDICT r1 weak #11)."""
    import hashlib
    h = hashlib.sha256()
    for f in KERNEL_SOURCES:
        h.update(open(os.path.join(ROOT, "rowbowt_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic(cfg, leg, n_reads, kernel):
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(tpath):
        return None, None
    t_ = json.load(open(tpath)).get("%s:%s:%d:%s" % (cfg, leg, n_reads, kernel))
    if not t_:
        return None, None
    if t_.get("src_hash") != kernel_source_hash():
        return None, "stale: %s was captured at kernel sources %s" % (t_.get("source"), t_.get("src_hash"))
    return t_["dram_bytes"], t_["source"]


class Workload:
    """One index resident on this rank's GPU + its synthetic read sets in pinned host buffers (raw and 2-bit packed)."""

    def __init__(self, rb, lib, cfg, prefix, panel, local, rank, n_reads, ftab_k, log):
        self.rb, self.lib, self.cfg, self.panel, self.n_reads = rb, lib, cfg, panel, n_reads
        self.has_sa, self.has_ma = os.path.exists(prefix + ".tsa"), os.path.exists(prefix + ".mab")
        t0 = time.time()
        self.ix = rb.GpuIndex.open(prefix, sa=self.has_sa, markers=self.has_ma, device=local)
        self.t_open = time.time() - t0
        t0 = time.time()
        self.ix.build_ftab(ftab_k)
        self.t_ftab = time.time() - t0
        self.info = self.ix.info()
        self.sets = {}
        self._keep = []
        self.rank = rank

    def add_reads(self, name, seed, **kw):
        """Generates the read set, stages it in pinned memory in both forms; returns the host pack time."""
        rb, lib, n = self.rb, self.lib, self.n_reads
        t0 = time.time()
        reads, _, _ = synth.make_reads(self.panel, n, READ_LEN, seed=seed + self.rank, **kw)     # a different batch on every rank
        t_make = time.time() - t0
        bases, p1 = pinned_array(lib, n * READ_LEN + 64, np.uint8)
        offs, p2 = pinned_array(lib, (n + 1) * 8, np.uint64)
        bases[:n * READ_LEN] = reads.reshape(-1)
        offs[:] = np.arange(n + 1, dtype=np.uint64) * np.uint64(READ_LEN)
        del reads
        packed, p3 = pinned_array(lib, ((n * READ_LEN + 31) // 32 + 2) * 8, np.uint64)
        flags, p4 = pinned_array(lib, n + 8, np.uint8)
        threads = max(1, min(16, (os.cpu_count() or 1)))
        t0 = time.perf_counter()
        pb, keep = self.ix.pack((bases[:n * READ_LEN], offs), threads=threads, out=(packed, flags))
        t_pack = time.perf_counter() - t0
        self._keep += [p1, p2, p3, p4, keep]
        self.sets[name] = dict(bases=bases, offs=offs, batch=rb.binding._Batch(n, bases.ctypes.data, offs.ctypes.data), packed=pb,
                               t_make=t_make, host_pack_s=t_pack, host_pack_threads=threads,
                               dead_reads=int(np.count_nonzero(flags[:n] & 1)))
        return self.sets[name]

    def close(self):
        self.ix.close()
        for p in self._keep:
            if isinstance(p, int):
                self.lib.rbg_host_free(p)
        self._keep, self.sets = [], {}


def run_leg(w, read_set, mode, steps, warmup, barrier, ascii_e2e=True, fetch=False):
    """One leg of the metric on this rank: device-resident steps (raw input: pack_kernel inside; and 2-bit input),
    then end to end through rbg_query_packed / rbg_query with pinned host buffers.  Returns per-rank numbers; with
    `fetch`, also out["result"]: what the last timed device-resident step computed, copied to the host after the timing."""
    ix, rs = w.ix, w.sets[read_set]
    e2e_mode = mode | (w.rb.RBG_NARROW_LOCS if mode & 1 else 0) | w.rb.RBG_NARROW_RANGES     # the narrow wire forms rb_align asks for
    out = {}
    staged = ix.upload((rs["bases"][:w.n_reads * READ_LEN], rs["offs"]))
    for _ in range(warmup):
        ix.query_staged(staged, mode)
    barrier()
    dev_ms, search_ms, phi_ms, launches = [], [], [], 0
    w0 = time.perf_counter()
    for _ in range(steps):
        ix.query_staged(staged, mode)
        st = ix.stats()
        dev_ms.append(st.ms_total)
        search_ms.append(st.ms_search)
        phi_ms.append(st.ms_phi)
        launches += st.launches
    barrier()
    out["wall_ms"] = (time.perf_counter() - w0) * 1e3 / steps
    out.update(dev_ms=float(np.mean(dev_ms)), search_ms=float(np.mean(search_ms)), phi_ms=float(np.mean(phi_ms)), launches=launches,
               lf_steps=st.lf_steps, lf_lines=st.lf_lines, phi_steps=st.phi_steps, marker_words=st.marker_words,
               kernel_ms={k: getattr(st, k) for k in ("ms_pack", "ms_search", "ms_locate", "ms_phi", "ms_markers", "ms_total")})
    if fetch:
        out["result"] = ix.fetch(staged, mode)
    out["checksum"] = ix.query_staged(staged, mode, checksum=True)
    staged.free()
    # the same kernels over a batch that arrived 2-bit packed (no pack_kernel), locations narrow
    h = C.c_void_p()
    w.rb.binding._check(w.lib.rbg_reads_upload_packed(ix.h, C.byref(rs["packed"]), C.byref(h)))
    pstaged = w.rb.StagedReads(ix, h)
    for _ in range(min(warmup, 2)):
        ix.query_staged(pstaged, e2e_mode)
    barrier()
    pk, pk_phi, pk_search = [], [], []
    for _ in range(steps):
        ix.query_staged(pstaged, e2e_mode)
        pk.append(ix.stats().ms_total)
        pk_phi.append(ix.stats().ms_phi)
        pk_search.append(ix.stats().ms_search)
        out["launches"] += ix.stats().launches
    barrier()
    out["dev_packed_ms"] = float(np.mean(pk))
    out["phi_narrow_ms"], out["search_packed_ms"] = float(np.mean(pk_phi)), float(np.mean(pk_search))
    out["checksum_packed"] = ix.query_staged(pstaged, e2e_mode, checksum=True)
    pstaged.free()
    # end to end: host buffers in, host results out
    for key, batch in (("e2e_ms", rs["packed"]), ("e2e_ascii_ms", rs["batch"])):
        if key == "e2e_ascii_ms" and not ascii_e2e:
            out[key], out[key + "_stages"] = out["e2e_ms"], None
            continue
        for _ in range(min(warmup, 2)):
            ix.query_raw(batch, e2e_mode)
        barrier()
        e0 = time.perf_counter()
        for _ in range(steps):
            ix.query_raw(batch, e2e_mode)
            out["launches"] += ix.stats().launches
        barrier()
        out[key] = (time.perf_counter() - e0) * 1e3 / steps
        out[key + "_stages"] = {k: getattr(ix.stats(), k) for k in ("ms_h2d", "ms_search", "ms_d2h", "ms_total")}
    return out


def dump_outputs(out_dir, res, budget=64 << 20):
    """Writes a QueryResult as float64 .npy files under out_dir: lo / hi (and toehold, per-read location counts and the
    locations; per-read marker counts and the marker words split into 32-bit halves, which float64 holds exactly) of a
    fixed seeded sample of reads -- all of them when everything fits in `budget` bytes -- plus the sampled read indices."""
    n = res.n
    # (name, offsets, values, float64 words per value)
    segs = [s for s in (("loc", res.loc_off, res.locs, 1), ("marker", res.mk_off, res.markers, 2)) if s[1] is not None]
    k = n
    while True:
        idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
        counts = [(off[idx + 1] - off[idx]).astype(np.int64) for _, off, _, _ in segs]
        per_read = 3 + (res.toehold is not None) + len(segs)
        total = 8 * (k * per_read + sum(int(c.sum()) * words for c, (_, _, _, words) in zip(counts, segs)))
        if total <= budget or k == 1:
            break
        k //= 2
    arrays = {"read_index": idx, "lo": res.lo[idx], "hi": res.hi[idx]}
    if res.toehold is not None:
        arrays["toehold"] = res.toehold[idx]
    for (name, off, vals, _), cnt in zip(segs, counts):
        first = np.repeat(off[idx].astype(np.int64) - np.concatenate([[0], np.cumsum(cnt)[:-1]]), cnt)
        picked = vals[first + np.arange(int(cnt.sum()))]
        arrays[name + "_count"] = cnt
        if name == "marker":
            arrays["markers_lo32"] = picked & np.uint64(0xFFFFFFFF)
            arrays["markers_hi32"] = picked >> np.uint64(32)
        else:
            arrays["locs"] = picked
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a).astype(np.float64))
    return {"dir": out_dir, "reads": int(k), "of": int(n), "bytes": int(sum(8 * len(a) for a in arrays.values()))}


def leg_record(w, name, read_set, mode, m, world, peak, peak_src, gather):
    """The JSON object of one leg from max-over-ranks timings `m`."""
    n, info = w.n_reads, w.info
    total = n * world
    wide = info.n >> 32
    loc_b = 5 if wide else 4
    rec = {"mode": name, "reads": read_set, "ms_per_step": m["dev_ms"], "value": total / (m["dev_ms"] * 1e-3), "unit": "reads/s",
           "ms_per_step_packed_input": m["dev_packed_ms"], "value_packed_input": total / (m["dev_packed_ms"] * 1e-3),
           "lf_steps_per_step": m["lf_steps"], "phi_steps_per_step": m["phi_steps"], "marker_words_per_step": m["marker_words"],
           "kernel_ms": m["kernel_ms"], "checksum": m["checksum"], "checksum_equal_packed_narrow": m["checksum"] == m["checksum_packed"]}
    # search_kernel: 64 B per distinct directory line an LF step loads + 38 B of 2-bit read + 16 B of range (24 with toehold) per read
    alg = m["lf_lines"] * 64 + n * (38 + (24 if mode & 1 else 16))
    ach = alg / (m["search_ms"] * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": "search_kernel<toehold>" if mode & 1 else "search_kernel", "achieved": ach, "peak": peak,
            "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "kernel_ms": m["search_ms"],
            "lf_steps_per_s": m["lf_steps"] / (m["search_ms"] * 1e-3), "lines_per_lf_step": m["lf_lines"] / max(1, m["lf_steps"])}
    roof["traffic"], src = ncu_traffic(w.cfg, name, n, "search_kernel")
    if src:
        roof["traffic_source"] = src
    if gather.get("dir"):
        line_gbs = m["lf_lines"] * 64 / (m["search_ms"] * 1e-3) / 1e9
        roof.update(random_gather_64B_gbs_at_dir_footprint=gather["dir"], random_gather_64B_gbs_8GB=gather.get("big"),
                    line_gbs=line_gbs, frac_of_random_gather=line_gbs / gather["dir"])
    rec["roofline"] = roof
    if mode & 1 and m["phi_steps"]:
        # locate_kernel<narrow> (what rbg_query_packed / rb_align run): per phi step one 32-byte slot + the 8-byte l1 word
        # + one location written (4 B, 5 B when n > 2^32); per read 8 B toehold + 16 B of offsets.  The u64-location form
        # (8 B written per step) is reported beside it.
        alg = m["phi_steps"] * (32 + 8 + loc_b) + n * 24
        ach = alg / (m["phi_narrow_ms"] * 1e-3) / 1e9
        alg_w = m["phi_steps"] * (32 + 8 + 8) + n * 24
        r2 = {"bound": "hbm", "kernel": "locate_kernel<narrow>", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
              "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "kernel_ms": m["phi_narrow_ms"],
              "phi_steps_per_s": m["phi_steps"] / (m["phi_narrow_ms"] * 1e-3),
              "wide_locations": {"kernel_ms": m["phi_ms"], "algorithmic_bytes_per_launch": alg_w,
                                 "achieved": alg_w / (m["phi_ms"] * 1e-3) / 1e9, "frac": alg_w / (m["phi_ms"] * 1e-3) / 1e9 / peak},
              "footprint_MB": {"phi": info.phi_bytes / 1e6, "toehold": info.toehold_bytes / 1e6}}
        r2["traffic"], src = ncu_traffic(w.cfg, name, n, "locate_kernel")
        if src:
            r2["traffic_source"] = src
        if gather.get("phi"):
            r2.update(random_gather_32B_gbs_at_phi_footprint=gather["phi"],
                      slot_gbs=m["phi_steps"] * 32 / (m["phi_narrow_ms"] * 1e-3) / 1e9,
                      frac_of_random_gather=m["phi_steps"] * 32 / (m["phi_narrow_ms"] * 1e-3) / 1e9 / gather["phi"])
        rec["roofline_locate"] = r2
    h2d_packed = ((n * READ_LEN + 31) // 32) * 8 + (n + 1) * 8 + n
    h2d_ascii = n * READ_LEN + (n + 1) * 8
    rg_b = 16 if wide else 8                              # lo + hi per read: u32 planes when n <= 2^32 (RBG_NARROW_RANGES)
    d2h = rg_b * n + ((8 * n + 8 * (n + 1) + loc_b * m["phi_steps"] + loc_b * n) if mode & 1 else 0) + ((8 * (n + 1) + 8 * m["marker_words"]) if mode & 2 else 0)
    rec["e2e"] = {"value": total / (m["e2e_ms"] * 1e-3), "unit": "reads/s", "ms_per_step": m["e2e_ms"], "call": "rbg_query_packed",
                  "input": "2-bit packed reads + offsets + flags in pinned host memory (packed by rbg_pack_bytes, as rb_align's parser threads do)",
                  "locations": "narrow (%d B each)" % loc_b if mode & 1 else None, "ranges": "%d B per read" % rg_b,
                  "h2d_bytes_per_step": h2d_packed, "d2h_bytes_per_step": d2h, "stages_ms": m["e2e_ms_stages"]}
    rec["e2e_ascii"] = {"value": total / (m["e2e_ascii_ms"] * 1e-3), "unit": "reads/s", "ms_per_step": m["e2e_ascii_ms"], "call": "rbg_query",
                        "input": "raw read bytes + offsets in pinned host memory (pack_kernel on the device)",
                        "h2d_bytes_per_step": h2d_ascii, "d2h_bytes_per_step": d2h, "stages_ms": m["e2e_ascii_ms_stages"]}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="count", choices=sorted(MODES), help="the leg reported as the headline (all legs are always measured)")
    ap.add_argument("--legs", default="locate,markers,all,count_noisy,c5", help="extra legs besides the headline ('' = none)")
    ap.add_argument("--config", default="auto", choices=["auto"] + sorted(synth.CONFIGS))
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--c5-reads", type=int, default=0, help="reads per GPU of the config-5 leg (0 = 500 k on c5w: every read occurs ~2000 times, "
                    "1e9 locations = 5 GB per step and GPU; 2 M on c5s)")
    ap.add_argument("--cpu-sample", type=int, default=100_000, help="reads timed through the reference for cpu_baseline")
    ap.add_argument("--ref-procs", type=int, default=0)
    ap.add_argument("--ref-reads-per-proc", type=int, default=50_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--ftab-k", type=int, default=10, help="k of the k-mer seed table built on the GPU at open (0 = none)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the headline leg's results of its last "
                    "step as DIR/<name>.npy (float64; a fixed sample of reads when all of them exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    log = sys.stderr
    tmp = tempfile.TemporaryDirectory(prefix="rowbowt_bench_")      # an index built at run time; removed at exit
    # stdout carries exactly ONE line, the JSON record: whatever a library prints there (NCCL's version banner, torchrun
    # notices) is sent to stderr for the whole run, the record is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank, world, log, emit, tmp.name)
        return

    import torch
    import torch.distributed as dist
    import rowbowt_b200 as rb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    lib = rb.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(m):
        keys = ("dev_ms", "dev_packed_ms", "search_ms", "phi_ms", "phi_narrow_ms", "search_packed_ms", "wall_ms", "e2e_ms", "e2e_ascii_ms")
        t = torch.tensor([m[k] for k in keys], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        m = dict(m)
        m.update({k: float(v) for k, v in zip(keys, t.tolist())})
        return m

    cfg, prefix, panel = workload(args.config, log, tmp.name)
    w = Workload(rb, lib, cfg, prefix, panel, local, rank, args.reads, args.ftab_k, log)
    info = w.info
    exact = w.add_reads("exact", 3)
    k_cpu = min(args.cpu_sample, args.reads)
    cpu_sample_reads = np.array(exact["bases"][:k_cpu * READ_LEN]).reshape(k_cpu, READ_LEN) if rank == 0 else None
    extra = [x for x in args.legs.split(",") if x]
    plan = [(args.mode, "exact", MODES[args.mode])]
    for name in extra:
        if name in MODES and name != args.mode and ((MODES[name] & 1) <= w.has_sa) and ((MODES[name] >> 1) <= w.has_ma):
            plan.append((name, "exact", MODES[name]))
    if "count_noisy" in extra:
        # the second read set of SURVEY 8(d): 1 % substitutions, 0.1 % N -> early exits, dead reads
        w.add_reads("noisy", 5, err_rate=0.01, n_rate=0.001)
        plan.append(("count_noisy", "noisy", 0))

    gather = {}
    if not args.no_gather and rank == 0:
        # the ceilings that actually bind these kernels: random 64-byte lines over a buffer as large as the rank
        # directory (and over 8 GB, beyond the TLB reach); random 32-byte sectors over the phi structures
        gather["dir"] = lib.rbg_gather_roofline(local, max(int(info.dir_bytes), 1 << 20), 64, 256)
        gather["big"] = lib.rbg_gather_roofline(local, 8 << 30, 64, 256)
        if w.has_sa:
            gather["phi"] = lib.rbg_gather_roofline(local, max(int(info.phi_bytes), 1 << 20), 32, 256)

    sampler = ClockSampler(local)
    sampler.start()
    measured = {}
    for name, rset, mode in plan:
        measured[name] = max_over_ranks(run_leg(w, rset, mode, args.steps, args.warmup, barrier,
                                                fetch=bool(args.dump_outputs) and name == args.mode and rank == 0))
    clocks = sampler.summary()

    # ---- BASELINE config 5 family (n > 2^32), -s [-m], when its index travelled with the repo --------------------
    c5 = None
    # c5w = config 5's 2504 haplotypes over a 1.75 Mbp reference (n = 4.38e9 rows; small enough to travel beside c2 in the
    # 512 MiB snapshot: the one the driver's runs see); c5s = its 64 Mbp reference x 256 haplotypes (n = 1.64e10; builder box only)
    c5_cfg = next((c for c in ("c5w", "c5s") if os.path.exists(os.path.join(DATA, c, c + ".tsa"))), None)
    have_c5 = torch.tensor([1 if ("c5" in extra and c5_cfg) else 0, {"c5w": 1, "c5s": 2}.get(c5_cfg, 0)], device="cuda")
    if world > 1:
        dist.all_reduce(have_c5, op=dist.ReduceOp.MIN)
    if int(have_c5[0].item()) and int(have_c5[1].item()):
        c5_cfg = {1: "c5w", 2: "c5s"}[int(have_c5[1].item())]
        c5_prefix = os.path.join(DATA, c5_cfg, c5_cfg)
        c5_reads = args.c5_reads or (500_000 if c5_cfg == "c5w" else 2_000_000)
        w.close()
        L5, H5 = synth.CONFIGS[c5_cfg]
        w5 = Workload(rb, lib, c5_cfg, c5_prefix, synth.make_panel(L5, H5), local, rank, c5_reads, args.ftab_k, log)
        w5.add_reads("exact", 4)
        mode5 = 1 | (2 if w5.has_ma else 0)
        g5 = {}
        if not args.no_gather and rank == 0:
            g5["dir"] = lib.rbg_gather_roofline(local, max(int(w5.info.dir_bytes), 1 << 20), 64, 256)
            g5["phi"] = lib.rbg_gather_roofline(local, max(int(w5.info.phi_bytes), 1 << 20), 32, 256)
        m5 = max_over_ranks(run_leg(w5, "exact", mode5, args.steps, 2, barrier, ascii_e2e=False))
        if rank == 0:
            peak, peak_src = measured_peaks()
            c5 = leg_record(w5, "all" if mode5 == 3 else "locate", "exact", mode5, m5, world, peak, peak_src, g5)
            c5.pop("e2e_ascii", None)
            i5 = w5.info
            c5["workload"] = ("BASELINE config 5 family: synthetic %d bp reference x %d haplotypes (config 5 is 64 Mbp x 2504; n = %d > 2^32 rows), "
                              "%d x 150bp exact reads per GPU, -s%s: %d locations per step and GPU (5 B each); they stay on the device in the "
                              "staged number and are copied out in e2e" % (L5, H5, i5.n, c5_reads, " -m" if w5.has_ma else " (no .mab built for this index)",
                                                                         m5["phi_steps"] + c5_reads))
            c5["index"] = {"config": c5_cfg, "n": i5.n, "r": i5.r, "window": i5.window, "dir_MB": i5.dir_bytes / 1e6, "phi_MB": i5.phi_bytes / 1e6,
                           "toehold_MB": i5.toehold_bytes / 1e6}
        w5.close()

    if rank == 0:
        peak, peak_src = measured_peaks()
        legs = {name: leg_record(w, name, rset, mode, measured[name], world, peak, peak_src, gather) for name, rset, mode in plan}
        head = legs[args.mode]
        m = measured[args.mode]
        n_reads = args.reads
        total_launches = sum(measured[k]["launches"] for k in measured) + (m5["launches"] if c5 else 0)
        out = {"metric": "150bp reads/s (%s)" % args.mode, "value": head["value"], "unit": "reads/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
               "wall_ms_per_step": m["wall_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "u64", "data": "synthetic",
               "config": {"workload": describe(cfg, n_reads), "mode": args.mode, "reads_per_gpu": n_reads, "read_len": READ_LEN,
                          "index": {"n": info.n, "r": info.r, "layout": info.layout, "window": info.window, "lines": info.n_lines,
                                    "cluster_windows": info.n_cluster, "dir_MB": info.dir_bytes / 1e6,
                                    "phi_MB": info.phi_bytes / 1e6, "toehold_MB": info.toehold_bytes / 1e6,
                                    "ftab_k": info.ftab_k, "ftab_MB": info.ftab_bytes / 1e6,
                                    "l2_window_MB": info.hot_bytes / 1e6, "l2_persisting_MB": info.l2_pinned_bytes / 1e6},
                          "l2": "inputs larger than L2 (%.0f MB index + %.0f MB reads per step)" % (
                              info.dir_bytes / 1e6, n_reads * READ_LEN / 1e6),
                          "parallelism": "replicated index, reads sharded, no collective",
                          "legs": "every leg = %d timed steps after %d warm-up steps over the same index" % (args.steps, args.warmup),
                          "numa": numa},
               "lf_steps_per_s": m["lf_steps"] * world / (head["ms_per_step"] * 1e-3), "lf_steps_per_step": m["lf_steps"],
               "phi_steps_per_step": m["phi_steps"], "marker_words_per_step": m["marker_words"],
               "kernel_ms": head["kernel_ms"], "checksum": head["checksum"], "gpu_launches": total_launches, "clocks": clocks,
               "roofline": head["roofline"], "e2e": head["e2e"], "e2e_ascii": head["e2e_ascii"],
               "value_packed_input": head["value_packed_input"],
               "legs": {k: v for k, v in legs.items() if k != args.mode},
               "host_pack": {"gb_per_s": n_reads * READ_LEN / exact["host_pack_s"] / 1e9, "threads": exact["host_pack_threads"],
                             "note": "rbg_pack_bytes over the step's batch, outside the timed region (the FASTQ parser's job)"},
               "kernel_source_hash": kernel_source_hash(),
               "setup_s": {"index_open": w.t_open, "ftab_build": w.t_ftab, "make_reads": exact["t_make"]}}
        if "roofline_locate" in head:
            out["roofline_locate"] = head["roofline_locate"]
        if c5:
            out["legs"]["c5"] = c5
        if args.dump_outputs:
            out["dump_outputs"] = dump_outputs(args.dump_outputs, m.pop("result"))
        # CPU baseline beside it: the unmodified reference on a bounded sample, one process (as shipped)
        if not args.no_cpu_baseline and world == 1 and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "rb_align")):
            k = k_cpu
            with tempfile.TemporaryDirectory() as td:
                v, qt = run_reference_shards(prefix, cpu_sample_reads, MODES[args.mode], 1, td)
            out["cpu_baseline"] = {"value": v, "unit": "reads/s", "cores": 1, "kind": "reference",
                                   "sample": "first %d reads of the step's batch through oracle/_ref/rb_align (its own total_query_time %.2f s)" % (k, qt)}
        elif world == 1:
            out["cpu_baseline"] = {"value": None, "unit": "reads/s", "cores": 0, "kind": "reference", "sample": "oracle/_ref not present"}
        emit(out)
    if w.ix.h:
        w.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
