#!/usr/bin/env python3
"""Synthetic pangenome workloads for tests and bench (SURVEY.md §8(d)).

Generates: a uniform-random reference, a SNP panel, H haplotypes, the FASTA the
reference's index builder consumes, marker positions, and simulated reads.
`build_index` shells out to the UNMODIFIED reference builder binaries compiled
by oracle/Makefile into oracle/_ref/ (pfbwt-f64, rb_build, mps_to_ma and the
write_mps driver around MarkerPositionsWriter), following the reference's
scripts/fa_to_rowbowt.sh.  `build_index_from_fasta_gpu` (`--gpu`) builds the same
files from the same FASTA with this project's GPU builders alone.  The files
produced (.rbwt/.tsa/.mab/.docs) are the reference's own on-disk formats and are
what both the GPU library and the reference rb_align consume.

Seeds (§8(d)): reference seed=1, panel/genotypes seed=2, reads seed=3.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from dataclasses import dataclass

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFBIN = os.path.join(ROOT, "oracle", "_ref")

# the compressible index files travel to the GPU box as zstd frames (tools/datafiles.py): restore them before anyone looks
try:
    from tools.datafiles import inflate_data
except ImportError:          # run as a script from tools/
    from datafiles import inflate_data
inflate_data()
PAD = 10  # pfbwt-f appends w=10 'A's to every sequence (pfbwt-f/README.md "padding")
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


@dataclass
class Panel:
    L: int
    H: int
    ref: np.ndarray      # uint8[L] ASCII
    sites: np.ndarray    # int64[S] sorted
    alts: np.ndarray     # uint8[S] ASCII, != ref[site]
    gt: np.ndarray       # bool[H, S]; haplotype h carries alt at site s

    @property
    def nseq(self) -> int:
        return self.H + 1

    def seq_start(self, h: int) -> int:
        """Text offset of sequence h (0 = reference, 1..H = haplotypes)."""
        return h * (self.L + PAD)

    def sequence(self, h: int) -> np.ndarray:
        s = self.ref.copy()
        if h > 0:
            carry = self.gt[h - 1]
            s[self.sites[carry]] = self.alts[carry]
        return s


def make_panel(L: int, H: int, site_every: int = 500, p_alt: float = 0.3,
               seed_ref: int = 1, seed_panel: int = 2) -> Panel:
    rng = np.random.default_rng(seed_ref)
    ref = ACGT[rng.integers(0, 4, size=L, dtype=np.uint8)]
    rng = np.random.default_rng(seed_panel)
    nsites = max(1, L // site_every)
    sites = np.sort(rng.choice(L, size=nsites, replace=False)).astype(np.int64)
    # alt = a different base: shift the ref code by 1..3
    code = np.searchsorted(ACGT, ref[sites])
    alts = ACGT[(code + rng.integers(1, 4, size=nsites)) % 4]
    gt = rng.random((H, nsites)) < p_alt
    return Panel(L, H, ref, sites, alts, gt)


def write_fasta(panel: Panel, path: str) -> None:
    with open(path, "wb") as f:
        for h in range(panel.nseq):
            name = b"ref" if h == 0 else b"h%d" % h
            f.write(b">" + name + b"\n")
            f.write(panel.sequence(h).tobytes())
            f.write(b"\n")


def write_marker_positions(panel: Panel, path: str, wsize: int = 10) -> None:
    """.mps through the reference's MarkerPositionsWriter: every sequence
    (reference included) gets one marker per site with its own allele."""
    p = subprocess.Popen([os.path.join(REFBIN, "write_mps"), str(wsize), path],
                         stdin=subprocess.PIPE)
    for h in range(panel.nseq):
        base = panel.seq_start(h)
        g = np.zeros(len(panel.sites), dtype=np.int64) if h == 0 else panel.gt[h - 1].astype(np.int64)
        arr = np.stack([panel.sites + base, panel.sites, g], axis=1)
        p.stdin.write(b"\n".join(b"%d %d %d" % tuple(r) for r in arr.tolist()))
        p.stdin.write(b"\n-\n")
    p.stdin.close()
    if p.wait() != 0:
        raise RuntimeError("write_mps failed")


def _run(cmd, **kw):
    t0 = time.time()
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, **kw)
    if r.returncode != 0:
        sys.stderr.write(r.stderr.decode(errors="replace")[-4000:])
        raise RuntimeError("command failed: %s" % (cmd,))
    return time.time() - t0


def build_index(panel: Panel, prefix: str, markers: bool = True, wsize: int = 10,
                keep_fasta: bool = False, log=sys.stderr) -> dict:
    """FASTA -> pfbwt-f64 -> rb_build, exactly scripts/fa_to_rowbowt.sh plus the
    marker pipeline of SURVEY.md Appendix C.  Returns timings."""
    t = {}
    fa = prefix  # pfbwt-f64 -o P P.fa; we name the FASTA == prefix like the reference's scripts
    t0 = time.time(); write_fasta(panel, fa); t["fasta"] = time.time() - t0
    pf = os.path.join(REFBIN, "pfbwt-f64")
    t["pfbwt"] = _run([pf, "--non-acgt-to-a", "--print-docs", "-r", "-o", prefix, fa])
    rb = [os.path.join(REFBIN, "rb_build"), "-s", "-l"]
    if markers:
        t0 = time.time(); write_marker_positions(panel, prefix + ".mps", wsize); t["mps"] = time.time() - t0
        t0 = time.time()
        p1 = subprocess.Popen([pf, "--non-acgt-to-a", "--pfbwt-only", "-o", prefix, "-s", "--stdout", "sa", fa],
                              stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
        p2 = subprocess.Popen([os.path.join(REFBIN, "mps_to_ma"), "-o", prefix + ".ma", prefix + ".mps", "-"],
                              stdin=p1.stdout, stderr=subprocess.DEVNULL)
        p1.stdout.close()
        if p2.wait() != 0 or p1.wait() != 0:
            raise RuntimeError("marker array pipeline failed")
        t["ma"] = time.time() - t0
        rb.append("-m")
    t["rb_build"] = _run(rb + ["-o", prefix, prefix])
    if not keep_fasta:
        for suf in ("", ".bwt", ".ssa", ".esa", ".dict", ".parse", ".occ", ".ilist", ".bwlast",
                    ".bwsai", ".sai", ".mps", ".ma", ".n", ".last", ".parse_old", ".ntab", ".log"):
            try:
                os.remove(prefix + suf)
            except FileNotFoundError:
                pass
    print("build_index %s: %s" % (prefix, {k: round(v, 1) for k, v in t.items()}), file=log)
    return t


def panel_text(panel: Panel) -> np.ndarray:
    """The text pfbwt-f indexes: every sequence followed by PAD 'A's, then the terminator (byte 0)."""
    pad = np.full(PAD, ord("A"), np.uint8)
    return np.concatenate([x for h in range(panel.nseq) for x in (panel.sequence(h), pad)] + [np.zeros(1, np.uint8)])


def suffix_array(text: np.ndarray) -> np.ndarray:
    """int64 suffix array of an ACGT text ending in a unique byte 0, by prefix doubling from 27-mer keys."""
    n = len(text)
    code = np.searchsorted(np.frombuffer(b"\0ACGT", np.uint8), text).astype(np.int64)
    K = 27                                                   # 27 base-5 digits fit in 63 bits
    padded = np.concatenate([code, np.zeros(K, np.int64)])
    key = np.zeros(n, np.int64)
    for j in range(K):
        key = key * 5 + padded[j:j + n]
    rank = np.empty(n, np.int64)
    h = K
    while True:
        order = np.argsort(key, kind="stable")
        sk = key[order]
        rank[order] = np.concatenate([[0], np.cumsum(sk[1:] != sk[:-1])])
        if rank[order[-1]] == n - 1:
            return order
        nxt = np.zeros(n, np.int64)
        nxt[:n - h] = rank[h:] + 1
        key = rank * (n + 1) + nxt
        h *= 2


def write_raw_index(panel: Panel, prefix: str, markers: bool = True, wsize: int = 10) -> None:
    """rb_build's inputs as pfbwt-f64 / mps_to_ma write them, computed here without the reference:
    <prefix>.bwt (one byte per row), .ssa / .esa (row, SA) at the first / last row of every run, .docs and,
    with markers, .ma (`first_row last_row marker* ~0` for every maximal block of consecutive rows whose
    suffix starts within wsize before the same panel-site markers).  tests/test_rb_build.py checks the files
    against the reference's own for the `tiny` panel, byte for byte."""
    text = panel_text(panel)
    n = len(text)
    sa = suffix_array(text)
    bwt = text[sa - 1]                                        # sa - 1 = -1 at the terminator's row wraps to it
    bwt.tofile(prefix + ".bwt")
    starts = np.concatenate([[0], np.nonzero(bwt[1:] != bwt[:-1])[0] + 1])
    ends = np.concatenate([starts[1:] - 1, [n - 1]])
    for suf, rows in ((".ssa", starts), (".esa", ends)):
        np.stack([rows, sa[rows]], axis=1).astype(np.uint64).tofile(prefix + suf)
    with open(prefix + ".docs", "w") as f:
        f.write("".join("%s %d\n" % ("ref" if h == 0 else "h%d" % h, panel.seq_start(h)) for h in range(panel.nseq)))
    if not markers:
        return
    # MarkerT words (pfbwt-f/include/marker.hpp): allele << 60 | reference position, in text order
    pos = np.concatenate([panel.sites + panel.seq_start(h) for h in range(panel.nseq)])
    alleles = np.concatenate([np.zeros(len(panel.sites), np.uint64)] + [g.astype(np.uint64) for g in panel.gt])
    words = (alleles << np.uint64(60)) | np.tile(panel.sites.astype(np.uint64), panel.nseq)
    a, b = np.searchsorted(pos, sa), np.searchsorted(pos, sa + wsize)
    out, block = [], None
    for row in np.nonzero(b > a)[0].tolist():
        ws = words[a[row]:b[row]].tolist()
        if block and block[1] == row - 1 and block[2] == ws:
            block[1] = row
            continue
        if block:
            out += block[:2] + block[2] + [0xFFFFFFFFFFFFFFFF]
        block = [row, row, ws]
    if block:
        out += block[:2] + block[2] + [0xFFFFFFFFFFFFFFFF]
    np.array(out, np.uint64).tofile(prefix + ".ma")


def _marker_words(panel: Panel):
    """Text positions of every marker (reference included, text order) and their MarkerT words."""
    pos = np.concatenate([panel.sites + panel.seq_start(h) for h in range(panel.nseq)])
    alleles = np.concatenate([np.zeros(len(panel.sites), np.uint64)] + [g.astype(np.uint64) for g in panel.gt])
    return pos, (alleles << np.uint64(60)) | np.tile(panel.sites.astype(np.uint64), panel.nseq)


def write_mps(panel: Panel, path: str, wsize: int = 10) -> None:
    """The panel's .mps without the reference: `first last word* ~0` for every maximal run of text positions p with the same
    non-empty list of markers in [p, p + wsize).  The list only changes where a marker at q enters (p = q - wsize + 1) or
    leaves (p = q + 1), so the records come from those breakpoints, never from the n positions."""
    n = panel.nseq * (panel.L + PAD) + 1
    pos, words = _marker_words(panel)
    cuts = np.unique(np.clip(np.concatenate([[0], pos - wsize + 1, pos + 1]), 0, n - 1))    # segment i: [cuts[i], cuts[i + 1])
    a, b = np.searchsorted(pos, cuts), np.searchsorted(pos, cuts + wsize)
    keep = b > a
    same = np.zeros(len(cuts) + 1, bool)                     # segment i continues the record of segment i - 1
    same[1:-1] = keep[1:] & keep[:-1] & (a[1:] == a[:-1]) & (b[1:] == b[:-1])
    first, last = np.nonzero(keep & ~same[:-1])[0], np.nonzero(keep & ~same[1:])[0]
    seg_end = np.append(cuts[1:], n) - 1
    out = []
    for f, l in zip(first.tolist(), last.tolist()):
        out += [int(cuts[f]), int(seg_end[l])] + words[a[f]:b[f]].tolist() + [0xFFFFFFFFFFFFFFFF]
    np.array(out, np.uint64).tofile(path)


def ma_from_mps(sa_rows: np.ndarray, row0: int, mps_words: np.ndarray) -> np.ndarray:
    """The .ma of rows [row0, row0 + len(sa_rows)) with SA values sa_rows, from the words of a .mps: row i gets the list of the
    record whose [first, last] holds SA[i] (none without one); a .ma record is a maximal run of consecutive rows whose lists
    are non-empty and equal by value, words in the .mps record's order."""
    w = np.asarray(mps_words, np.uint64)
    ends = np.nonzero(w == np.uint64(0xFFFFFFFFFFFFFFFF))[0]
    starts = np.concatenate([[0], ends[:-1] + 1]).astype(np.int64)
    firsts, lasts = w[starts], w[starts + 1]
    lists, lid = {}, np.empty(len(starts), np.int64)
    for k, (s, e) in enumerate(zip(starts.tolist(), ends.tolist())):
        ws = tuple(w[s + 2:e].tolist())
        lid[k] = lists.setdefault(ws, len(lists)) if ws else -1
    by_id = {v: list(k) for k, v in lists.items()}
    sa = np.asarray(sa_rows, np.uint64)
    ids = np.full(len(sa), -1, np.int64)
    if len(firsts):
        k = np.searchsorted(firsts, sa, side="right") - 1
        hit = (k >= 0) & (sa <= lasts[np.clip(k, 0, None)])
        ids[hit] = lid[k[hit]]
    change = np.nonzero(np.diff(ids) != 0)[0] + 1
    b0 = np.concatenate([[0], change])
    b1 = np.append(change, len(ids)) - 1
    out = []
    for f, l in zip(b0.tolist(), b1.tolist()):
        if ids[f] >= 0:
            out += [row0 + f, row0 + l] + by_id[int(ids[f])] + [0xFFFFFFFFFFFFFFFF]
    return np.array(out, np.uint64)


def build_index_gpu(panel: Panel, prefix: str, markers: bool = True, device: int = 0, log=sys.stderr) -> dict:
    """The same index files as build_index, without the reference: write_raw_index, then the project's own
    rb_build on the GPU (rowbowt_b200.build_index).  Returns timings."""
    import rowbowt_b200 as rb
    t = {}
    t0 = time.time(); write_raw_index(panel, prefix, markers=markers); t["raw"] = time.time() - t0
    t0 = time.time(); rb.build_index(prefix, prefix, sa=True, markers=markers, device=device); t["rb_build"] = time.time() - t0
    for suf in (".bwt", ".ssa", ".esa", ".ma"):
        if os.path.exists(prefix + suf):
            os.remove(prefix + suf)
    print("build_index_gpu %s: %s" % (prefix, {k: round(v, 1) for k, v in t.items()}), file=log)
    return t


def build_index_from_fasta_gpu(panel: Panel, prefix: str, markers: bool = True, device: int = 0, log=sys.stderr) -> dict:
    """The same index files as build_index, from the panel's FASTA with the project's GPU builders alone: write_fasta ->
    build_bwt (.bwt/.ssa/.esa/.docs) -> build_index (.rbwt/.tsa) -> write_mps -> build_marker_array (.ma, .mab); the FASTA
    and the raw files are removed afterwards.  Returns timings."""
    import rowbowt_b200 as rb
    t = {}
    fa = prefix + ".fa"
    t0 = time.time(); write_fasta(panel, fa); t["fasta"] = time.time() - t0
    t0 = time.time(); st = rb.build_bwt(fa, prefix, device=device); t["bwt"] = time.time() - t0
    print("build_bwt %s" % json.dumps(st.as_dict()), file=log, flush=True)
    t0 = time.time(); rb.build_index(prefix, prefix, sa=True, device=device); t["rb_build"] = time.time() - t0
    if markers:
        t0 = time.time(); write_mps(panel, prefix + ".mps"); t["mps"] = time.time() - t0
        t0 = time.time()
        rb.build_marker_array(prefix, prefix + ".mps", prefix + ".ma", mab=prefix + ".mab", device=device)
        t["ma"] = time.time() - t0
    for path in (fa, prefix + ".bwt", prefix + ".ssa", prefix + ".esa", prefix + ".mps", prefix + ".ma"):
        if os.path.exists(path):
            os.remove(path)
    print("build_index_from_fasta_gpu %s: %s" % (prefix, {k: round(v, 1) for k, v in t.items()}), file=log)
    return t


def make_reads(panel: Panel, n_reads: int, read_len: int = 150, seed: int = 3,
               err_rate: float = 0.0, n_rate: float = 0.0, chunk: int = 1 << 20):
    """uint8[n_reads, read_len] ASCII reads: uniform substrings of uniformly
    chosen sequences (reference or haplotype).  Returns (reads, seq_id, start)."""
    rng = np.random.default_rng(seed)
    out = np.empty((n_reads, read_len), dtype=np.uint8)
    hs = rng.integers(0, panel.nseq, size=n_reads)
    starts = rng.integers(0, panel.L - read_len + 1, size=n_reads)
    ar = np.arange(read_len, dtype=np.int64)
    for a in range(0, n_reads, chunk):
        b = min(n_reads, a + chunk)
        st = starts[a:b]
        blk = panel.ref[st[:, None] + ar]
        first = np.searchsorted(panel.sites, st)
        last = np.searchsorted(panel.sites, st + read_len)
        k = 0
        while True:
            m = first + k < last
            if not m.any():
                break
            rows = np.nonzero(m)[0]
            si = first[rows] + k
            h = hs[a:b][rows]
            carry = (h > 0) & panel.gt[np.maximum(h, 1) - 1, si]
            rows, si = rows[carry], si[carry]
            blk[rows, panel.sites[si] - st[rows]] = panel.alts[si]
            k += 1
        out[a:b] = blk
    if err_rate > 0:
        m = rng.random(out.shape) < err_rate
        code = np.searchsorted(ACGT, out[m])
        out[m] = ACGT[(code + rng.integers(1, 4, size=code.shape)) % 4]
    if n_rate > 0:
        out[rng.random(out.shape) < n_rate] = ord("N")
    return out, hs, starts


def write_fastq(reads: np.ndarray, path: str, start_id: int = 0) -> None:
    n, m = reads.shape
    qual = b"I" * m
    with open(path, "wb") as f:
        for a in range(0, n, 65536):
            b = min(n, a + 65536)
            f.write(b"".join(b"@r%d\n%s\n+\n%s\n" % (start_id + i, reads[i].tobytes(), qual)
                             for i in range(a, b)))


CONFIGS = {
    # name: (L, H)   — C2..C4 of BASELINE.json: 50 Mbp x 64 haplotypes
    "tiny": (20_000, 4),
    "small": (1_000_000, 16),
    "medium": (8_000_000, 32),
    "c2": (50_000_000, 64),
    # 1/10-scale stand-in for BASELINE config 5 (64 Mbp x 2504): n = 1.64e10 > 2^32 rows in a REAL index
    "c5s": (64_000_000, 256),
    # smallest member of the same family that still has n > 2^32 rows AND an index (.rbwt + .tsa) small enough to
    # travel to the GPU box: the -s path over a real wide index
    "c5m": (20_000_000, 256),
    # the OTHER axis of config 5: its 2504 haplotypes (an exact read occurs up to 2505 times) over a 1.75 Mbp reference,
    # n = 4.38e9 > 2^32 rows; the only member of the family whose .rbwt + .tsa + .mab fit beside c2 in the 512 MiB
    # snapshot that travels to the GPU box, so it is the one the driver's own runs see
    "c5w": (1_750_000, 2504),
}


def parity_sample_sizes(nseq: int) -> dict:
    """Reads in the committed parity samples of a full-size workload (tools/make_fullsize_sample.py,
    tools/make_fullsize_oracle.py, tests/test_full_size.py).  -s prints ~28 bytes per occurrence and an exact read
    occurs in up to nseq sequences: panels with thousands of haplotypes get fewer reads so the files stay ~1 MB."""
    if nseq < 1000:
        return {"count": 600, "s": 120, "m": 600, "exact": 300, "noisy": 300, "noisy_text": 600}
    return {"count": 600, "s": 8, "m": 600, "exact": 20, "noisy": 60, "noisy_text": 40}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("config", choices=sorted(CONFIGS))
    ap.add_argument("outdir")
    ap.add_argument("--no-markers", action="store_true")
    ap.add_argument("--reads", type=int, default=0, help="also write N reads as FASTQ")
    ap.add_argument("--keep", action="store_true")
    ap.add_argument("--gpu", action="store_true", help="build on the GPU with this project's builders, without the reference")
    a = ap.parse_args()
    L, H = CONFIGS[a.config]
    os.makedirs(a.outdir, exist_ok=True)
    prefix = os.path.join(a.outdir, a.config)
    panel = make_panel(L, H)
    if a.gpu:
        if ROOT not in sys.path:          # run as a script from tools/: the package is imported from the repository root
            sys.path.insert(0, ROOT)
        build_index_from_fasta_gpu(panel, prefix, markers=not a.no_markers)
    else:
        build_index(panel, prefix, markers=not a.no_markers, keep_fasta=a.keep)
    if a.reads:
        reads, _, _ = make_reads(panel, a.reads)
        write_fastq(reads, prefix + ".reads.fq")


if __name__ == "__main__":
    main()
