"""The u64 BWT builder (csrc/bwt_build_wide.cu): the suffix array sorted in parts of at most M rows, certified before any
file is written.  rbg_build_bwt takes it from n = 2^32 on; RBG_BWT_WIDE=1 forces it at any n and RBG_BWT_PART_ROWS caps M,
so small texts reach the real key packing (at least 33 rank bits) and many parts.

CPU part: the text entry point keeps its 2^32 cap when the wide builder is forced, refusals before any CUDA call, the numpy
mirror of the certificate against synth.suffix_array.
GPU part: the adversarial texts of test_bwt_build in one and several parts against numpy and the u32 builder, the refusal of
a prefix bucket larger than a part, the reference's tiny files, small in at least 4 parts, rbg_check_suffix_array.
RBG_TEST_WIDE_BUILD=1 adds c5w (n = 4.38e9) built from its FASTA in a temporary directory and checked against the reference's
committed rb_align output (minutes, about 10 GB of disk)."""
import filecmp
import gzip
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

import rowbowt_b200 as rb
from tools import synth
from test_bwt_build import RAW, TINY, _adversarial, _as_n, _expected, _fasta, _same, _tiny_records

E_ALPHABET, E_ARG, E_NOMEM = -3, -5, -6
PREFIX_K = 11


def _codes(text):
    return np.searchsorted(np.frombuffer(b"\0ACGT", np.uint8), np.concatenate([np.frombuffer(text, np.uint8), np.zeros(1, np.uint8)]))


def _buckets(text):
    """Suffixes per 11-symbol base-5 prefix (terminator and past the end 0), as (sorted bucket ids, counts)."""
    c = np.concatenate([_codes(text), np.zeros(PREFIX_K, np.int64)]).astype(np.int64)
    n = len(text) + 1
    key = np.zeros(n, np.int64)
    for j in range(PREFIX_K):
        key = key * 5 + c[j:j + n]
    return np.unique(key, return_counts=True)


def _parts(counts, cap):
    """Rows per part of the greedy cut at bucket boundaries into parts of at most cap rows (None when a bucket exceeds cap)."""
    if counts.max() > cap:
        return None
    out = [0]
    for c in counts.tolist():
        if out[-1] + c > cap:
            out.append(0)
        out[-1] += c
    return out


def _first_bad(text, sa):
    """Host mirror of rbg_check_suffix_array: the smallest row i where sa[i] >= n, sa[i] is held by an earlier row, or
    (T[sa[i]], rank[sa[i] + 1]) is not below row i + 1's pair, rank being the first row of each value; n when none."""
    code = _codes(text)
    n = len(code)
    sa = np.asarray(sa, np.uint64)
    rows = np.arange(n, dtype=np.uint64)
    valid = sa < np.uint64(n)
    rank = np.full(n + 1, np.iinfo(np.uint64).max, np.uint64)
    np.minimum.at(rank, sa[valid].astype(np.int64), rows[valid])
    sv = np.where(valid, sa, 0).astype(np.int64)
    bad = ~valid | (rank[sv] != rows)
    p, q = sv[:-1], sv[1:]
    cp, cq = code[p], code[q]
    rp, rq = rank[p + 1], rank[q + 1]
    bad[:-1] |= valid[:-1] & valid[1:] & ((cp > cq) | ((cp == cq) & ((cp == 0) | (rp >= rq))))
    nz = np.nonzero(bad)[0]
    return int(nz[0]) if len(nz) else n


def _rand_text(m, seed):
    return synth.ACGT[np.random.default_rng(seed).integers(0, 4, m)].tobytes()


def _corruptions(n):
    """(name, function of a suffix array returning a corrupted copy)."""
    def swap(i, j):
        def f(sa):
            sa = sa.copy()
            sa[[i, j]] = sa[[j, i]]
            return sa
        return f

    def put(i, v):
        def f(sa):
            sa = sa.copy()
            sa[i] = v(sa)
            return sa
        return f
    return [("adjacent", swap(n // 2, n // 2 + 1)), ("distant", swap(n // 10, 9 * n // 10)),
            ("repeated", put(2 * n // 3, lambda sa: sa[n // 3])), ("too_large", put(2 * n // 5, lambda sa: n + 5)),
            ("last_is_n", put(n - 1, lambda sa: n))]


# ---- CPU ----------------------------------------------------------------------------------------------------------------

def test_text_entry_keeps_its_cap_when_wide_is_forced(tmp_path, monkeypatch):
    monkeypatch.setenv("RBG_BWT_WIDE", "1")
    buf = np.zeros(1, np.uint8) + ord("A")
    rc = rb.lib().rbg_build_bwt_text(buf.ctypes.data, 1 << 32, str(tmp_path / "o").encode(), 0, None)
    assert rc == E_ARG
    msg = rb.lib().rbg_last_error().decode()
    assert "2^32" in msg and str(0xFFFFFFFF) in msg, msg
    assert os.listdir(tmp_path) == []


def test_check_suffix_array_refuses_before_cuda():
    with pytest.raises(rb.RbgError) as e:
        rb.check_suffix_array(np.frombuffer(b"ACNT", np.uint8), np.arange(5, dtype=np.uint64))
    assert e.value.code == E_ALPHABET and "offset 2" in str(e.value)
    with pytest.raises(ValueError):
        rb.check_suffix_array(np.frombuffer(b"ACGT", np.uint8), np.arange(4, dtype=np.uint64))


def test_usage_has_no_length_cap():
    r = subprocess.run([os.path.join(ROOT, "rowbowt_b200", "fa_to_bwt")], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"Usage: fa_to_bwt" in r.stderr and b"2^32" not in r.stderr


@pytest.mark.parametrize("seed", [1, 2])
def test_certificate_mirror(seed):
    """The mirror accepts suffix arrays and flags every corruption at or before the first row it touches."""
    for text in (_rand_text(3000, seed), b"ACG" * 700, b"A" * 500):
        t = np.concatenate([np.frombuffer(text, np.uint8), np.zeros(1, np.uint8)])
        sa = synth.suffix_array(t).astype(np.uint64)
        n = len(sa)
        assert _first_bad(text, sa) == n
        for name, f in _corruptions(n):
            bad = _first_bad(text, f(sa))
            assert bad < n, name


def test_part_cut_mirror():
    text = _rand_text(1 << 14, 3)
    ids, counts = _buckets(text)
    assert counts.sum() == len(text) + 1 and np.all(np.diff(ids) > 0)
    parts = _parts(counts, 4096)
    assert parts and sum(parts) == len(text) + 1 and max(parts) <= 4096 and len(parts) >= 5
    assert _parts(_buckets(b"A" * 5000)[1], 4096) is None


# ---- GPU ----------------------------------------------------------------------------------------------------------------

_U32 = {}


def _u32_build(case, tmp_path, monkeypatch):
    """Files and stats of the u32 builder for an adversarial text (once per session)."""
    if case not in _U32:
        monkeypatch.delenv("RBG_BWT_WIDE", raising=False)
        out = str(tmp_path / "u32")
        st = rb.build_bwt_text(np.frombuffer(_adversarial()[case][0], np.uint8), out)
        files = []
        for suf in (".bwt", ".ssa", ".esa"):
            with open(out + suf, "rb") as f:
                files.append(f.read())
            os.remove(out + suf)
        _U32[case] = (files, st.rounds)
    return _U32[case]


def _caps(case):
    """Part caps for an adversarial text: none, the largest bucket or 4096 rows (whichever is larger), and a cap landing
    exactly on a bucket boundary near a third of the rows."""
    text = _adversarial()[case][0]
    counts = _buckets(text)[1]
    cum = np.cumsum(counts)
    edge = int(cum[np.searchsorted(cum, len(text) // 3)])
    return {"whole": None, "4096": max(4096, int(counts.max())), "edge": max(edge, int(counts.max()))}


CAP_CASES = [(c, k) for c in sorted(_adversarial()) for k in ("whole", "4096", "edge")]


@pytest.mark.gpu
@pytest.mark.parametrize("case,cap", CAP_CASES, ids=["%s-%s" % x for x in CAP_CASES])
def test_adversarial_texts_in_parts(tmp_path, monkeypatch, case, cap):
    text = _adversarial()[case][0]
    exp_files, u32_rounds = _u32_build(case, tmp_path, monkeypatch)
    rows = _caps(case)[cap]
    monkeypatch.setenv("RBG_BWT_WIDE", "1")
    if rows is not None:
        monkeypatch.setenv("RBG_BWT_PART_ROWS", str(rows))
    out = str(tmp_path / "o")
    st = rb.build_bwt_text(np.frombuffer(text, np.uint8), out)
    for suf, exp, u32 in zip((".bwt", ".ssa", ".esa"), _expected(text), exp_files):
        with open(out + suf, "rb") as f:
            got = f.read()
        assert got == exp, suf
        assert got == u32, suf
    n = len(text) + 1
    parts = _parts(_buckets(text)[1], rows if rows is not None else n)
    assert st.wide == 1 and st.n == n and st.r == os.path.getsize(out + ".ssa") // 16
    assert st.parts == len(parts) and st.part_rows == max(parts), st.as_dict()
    if rows is not None and n > rows:
        assert st.parts > 1
    assert st.rounds <= u32_rounds, (st.rounds, u32_rounds)
    active = list(st.active)[:st.rounds]
    assert all(a > 0 for a in active) and st.max_active == max(active, default=0)
    assert st.ms_verify > 0 and st.peak_bytes >= 21 * n


@pytest.mark.gpu
def test_bucket_larger_than_a_part_is_refused(tmp_path, monkeypatch):
    monkeypatch.setenv("RBG_BWT_WIDE", "1")
    monkeypatch.setenv("RBG_BWT_PART_ROWS", "1000")
    with pytest.raises(rb.RbgError) as e:
        rb.build_bwt_text(np.frombuffer(b"A" * (1 << 16), np.uint8), str(tmp_path / "o"))
    assert e.value.code == E_NOMEM, str(e.value)
    assert "AAAAAAAAAAA" in str(e.value) and "1000" in str(e.value), str(e.value)
    assert os.listdir(tmp_path) == []


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["plain", "wrapped", "gzip", "bgzf", "iupac"])
def test_tiny_equals_reference_files(tmp_path, monkeypatch, form):
    monkeypatch.setenv("RBG_BWT_WIDE", "1")
    monkeypatch.setenv("RBG_BWT_PART_ROWS", "4096")
    names, seqs = _tiny_records()
    if form == "iupac":
        seqs = [_as_n(s) for s in seqs]
    data = _fasta(names, seqs, width=60 if form in ("wrapped", "bgzf") else 0)
    fa = str(tmp_path / "tiny.fa")
    if form == "gzip":
        data = gzip.compress(data)
    with open(fa, "wb") as f:
        f.write(data)
    if form == "bgzf":
        from tools.e2e_inputs import write_bgzf
        write_bgzf(fa, fa + ".gz", block=4096)
        fa += ".gz"
    out = str(tmp_path / "o")
    st = rb.build_bwt(fa, out)
    _same(RAW, out, (".bwt", ".ssa", ".esa"))
    assert filecmp.cmp(TINY + ".docs", out + ".docs", shallow=False)
    assert st.wide == 1 and st.parts > 1 and st.records == len(names)
    rb.build_index(out, out, sa=True)
    _same(TINY, out, (".rbwt", ".tsa"))


@pytest.mark.gpu
def test_small_in_parts_equals_write_raw_index(tmp_path, monkeypatch):
    panel = synth.make_panel(*synth.CONFIGS["small"])
    exp = str(tmp_path / "exp")
    synth.write_raw_index(panel, exp, markers=False)
    fa = str(tmp_path / "small.fa")
    synth.write_fasta(panel, fa)
    n = os.path.getsize(exp + ".bwt")
    monkeypatch.setenv("RBG_BWT_WIDE", "1")
    monkeypatch.setenv("RBG_BWT_PART_ROWS", str(n // 5))
    out = str(tmp_path / "o")
    st = rb.build_bwt(fa, out)
    _same(exp, out, (".bwt", ".ssa", ".esa", ".docs"))
    assert st.wide == 1 and st.parts >= 4 and st.part_rows <= n // 5 and st.n == n


@pytest.mark.gpu
def test_check_suffix_array(tmp_path):
    for text in (_rand_text(5000, 4), b"ACGT" * 1000, _adversarial()["fibonacci"][0][:20000], b"T"):
        t = np.concatenate([np.frombuffer(text, np.uint8), np.zeros(1, np.uint8)])
        sa = synth.suffix_array(t).astype(np.uint64)
        n = len(sa)
        assert rb.check_suffix_array(np.frombuffer(text, np.uint8), sa) == n
        if n < 10:
            continue
        for name, f in _corruptions(n):
            bad = f(sa)
            assert rb.check_suffix_array(np.frombuffer(text, np.uint8), bad) == _first_bad(text, bad), name


# ---- c5w from its FASTA (RBG_TEST_WIDE_BUILD=1) ------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.skipif(os.environ.get("RBG_TEST_WIDE_BUILD") != "1", reason="RBG_TEST_WIDE_BUILD=1: minutes and about 10 GB of disk")
def test_c5w_from_fasta_equals_reference_output(tmp_path):
    """python tools/synth.py c5w DIR --gpu (n = 4.38e9: the wide builder without forcing), then rb_align over the index it
    made prints what the unmodified reference printed over its own c5w index, on exact and noisy reads."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "synth.py"), "c5w", str(tmp_path), "--gpu"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=ROOT)
    log = r.stderr.decode(errors="replace")
    print(log)
    assert r.returncode == 0, log[-4000:]
    stats = json.loads(next(line for line in log.splitlines() if line.startswith("build_bwt "))[len("build_bwt "):])
    assert stats["wide"] == 1 and stats["n"] > 1 << 32 and stats["ms_verify"] > 0
    prefix = str(tmp_path / "c5w")
    panel = synth.make_panel(*synth.CONFIGS["c5w"])
    sizes = synth.parity_sample_sizes(panel.nseq)
    exp_dir = os.path.join(GOLDEN, "expected")
    n_reads = json.load(open(os.path.join(exp_dir, "c5w.sample.json")))["n_reads"]
    reads = synth.make_reads(panel, n_reads, 150, seed=3)[0]
    noisy = synth.make_reads(panel, sizes["noisy_text"], 150, seed=5, err_rate=0.01, n_rate=0.001)[0]
    rb_align = os.path.join(ROOT, "rowbowt_b200", "rb_align")
    runs = [("sample", tag, flags, reads[:sizes[k]]) for tag, flags, k in (("count", [], "count"), ("s", ["-s"], "s"), ("m", ["-m"], "m"))]
    runs += [("noisy", tag, flags, noisy) for tag, flags in (("count", []), ("s", ["-s"]), ("m", ["-m"]), ("sm", ["-s", "-m"]))]
    for kind, tag, flags, batch in runs:
        fq = str(tmp_path / ("%s_%s.fq" % (kind, tag)))
        synth.write_fastq(batch, fq)
        p = subprocess.run([rb_align] + flags + [prefix, fq], capture_output=True)
        assert p.returncode == 0, p.stderr.decode()
        with open(os.path.join(exp_dir, "c5w.%s.%s.txt" % (kind, tag)), "rb") as f:
            assert p.stdout == f.read(), (kind, tag)
