"""The BWT of a FASTA built on the GPU (rbg_build_bwt / fa_to_bwt): the raw files pfbwt-f64 --non-acgt-to-a --print-docs -r
writes (.bwt, .ssa, .esa, .docs), for texts below 2^32 positions.

CPU part: inputs refused before any CUDA call (this runs without a GPU), the binary's usage.
GPU part: the reference's own files (tiny), the committed indexes rebuilt from the FASTAs their texts invert to,
tools/synth.write_raw_index (small), adversarial texts against tools/synth.suffix_array, the binary, and synth.py --gpu."""
import filecmp
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

import rowbowt_b200 as rb
from oracle import rbformats as F
from tools import synth

FA_TO_BWT = os.path.join(ROOT, "rowbowt_b200", "fa_to_bwt")
RAW = os.path.join(GOLDEN, "raw", "tiny")
TINY = os.path.join(GOLDEN, "tiny", "tiny")
E_IO, E_FORMAT, E_ALPHABET, E_ARG = -1, -2, -3, -5


def _refused(tmp_path, data, code, *words):
    path = str(tmp_path / "in.fa")
    if data is not None:
        with open(path, "wb") as f:
            f.write(data)
    with pytest.raises(rb.RbgError) as e:
        rb.build_bwt(path, str(tmp_path / "out"))
    assert e.value.code == code, str(e.value)
    for w in words:
        assert w in str(e.value), str(e.value)
    assert sorted(os.listdir(tmp_path)) == ([] if data is None else ["in.fa"])       # nothing written


# ---- CPU ----------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case,data,code,words", [
    ("missing", None, E_IO, ()),
    ("empty", b"", E_FORMAT, ("no FASTA records",)),
    ("header_only", b">only one\n", E_FORMAT, ("'only'", "no bases")),
    ("record_without_bases", b">a\nACGT\n>b\n>c\nGATTACA\n", E_FORMAT, ("'b'", "no bases")),
    ("lowercase", b">a\nACGT\n>chr2 soft\nACGTNNacgt\n", E_ALPHABET, ("'chr2'", "offset 6", "uppercase")),
    ("star", b">a\nACG*T\n", E_ALPHABET, ("'a'", "'*'", "offset 3")),
])
def test_refused_before_cuda(tmp_path, case, data, code, words):
    _refused(tmp_path, data, code, *words)


def test_text_length_is_checked_before_the_buffer_is_read(tmp_path):
    """len = 2^32 bases on a 1-byte buffer: the terminator would make n = 2^32 + 1."""
    buf = np.zeros(1, np.uint8) + ord("A")
    rc = rb.lib().rbg_build_bwt_text(buf.ctypes.data, 1 << 32, str(tmp_path / "o").encode(), 0, None)
    assert rc == E_ARG
    msg = rb.lib().rbg_last_error().decode()
    assert "2^32" in msg and str(0xFFFFFFFF) in msg, msg
    with pytest.raises(rb.RbgError) as e:
        rb.build_bwt_text(np.frombuffer(b"ACGTX", np.uint8), str(tmp_path / "o"))
    assert e.value.code == E_ALPHABET and "offset 4" in str(e.value)
    assert os.listdir(tmp_path) == []


def test_binary_usage():
    r = subprocess.run([FA_TO_BWT], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"Usage: fa_to_bwt" in r.stderr


# ---- GPU ----------------------------------------------------------------------------------------------------------------

def _fasta(names, seqs, width=0):
    out = []
    for name, s in zip(names, seqs):
        out.append(b">" + name.encode() + b"\n")
        if width:
            out += [s[i:i + width] + b"\n" for i in range(0, len(s), width)]
        else:
            out.append(s + b"\n")
    return b"".join(out)


def _tiny_records():
    panel = synth.make_panel(*synth.CONFIGS["tiny"])
    return ["ref"] + ["h%d" % h for h in range(1, panel.nseq)], [panel.sequence(h).tobytes() for h in range(panel.nseq)]


def _as_n(seq):
    """'N' (and one 'R') where the text has 'A': --non-acgt-to-a maps them back."""
    a = np.frombuffer(seq, np.uint8).copy()
    idx = np.nonzero(a == ord("A"))[0]
    a[idx[::3]] = ord("N")
    a[idx[1]] = ord("R")
    return a.tobytes()


def _same(a, b, sufs):
    for suf in sufs:
        assert filecmp.cmp(a + suf, b + suf, shallow=False), suf


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["plain", "wrapped", "gzip", "bgzf", "iupac"])
def test_tiny_equals_reference_files(tmp_path, form):
    """.bwt/.ssa/.esa are the reference pfbwt-f64's, .docs its --print-docs list, and rb_build over them gives the committed
    .rbwt/.tsa, whatever the FASTA's line width and compression, and with N for A."""
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
    assert (st.n, st.r, st.records) == (os.path.getsize(RAW + ".bwt"), os.path.getsize(RAW + ".ssa") // 16, len(names))
    assert st.peak_bytes >= 37 * st.n
    rb.build_index(out, out, sa=True)
    _same(TINY, out, (".rbwt", ".tsa"))


def _invert(prefix):
    """The text of a committed index, by inverse BWT: row i's suffix is followed by the one at row order[i]."""
    b = F.read_rbwt(prefix + ".rbwt")
    last = np.repeat(b.heads, b.lens.astype(np.int64))
    last[last == 1] = 0                                            # the terminator is stored as byte 1
    order = np.argsort(last, kind="stable").tolist()
    L = last.tolist()
    i = L.index(0)
    text = bytearray(b.n)
    for k in range(b.n):
        i = order[i]
        text[k] = L[i]
    assert text[-1] == 0 and text.count(0) == 1
    return bytes(text[:-1])


@pytest.mark.gpu
@pytest.mark.parametrize("pre", ["toy/small.fa", "greedy/ref.fa"])
def test_committed_indexes_from_their_inverted_text(tmp_path, pre):
    """Indexes the reference built from FASTAs this repository does not have: their texts, split at the .docs starts and
    stripped of the padding, rebuild the committed .rbwt/.tsa byte for byte."""
    src = os.path.join(GOLDEN, pre)
    text = _invert(src)
    names, starts = F.read_docs(src + ".docs")
    bounds = starts.tolist() + [len(text)]
    seqs = []
    for k in range(len(names)):
        rec = text[bounds[k]:bounds[k + 1]]
        assert rec.endswith(b"A" * synth.PAD), names[k]
        seqs.append(rec[:-synth.PAD])
    fa = str(tmp_path / "in.fa")
    with open(fa, "wb") as f:
        f.write(_fasta(names, seqs, width=70))
    out = str(tmp_path / "o")
    rb.build_bwt(fa, out)
    rb.build_index(out, out, sa=True)
    _same(src, out, (".rbwt", ".tsa", ".docs"))


def _expected(text):
    """(.bwt, .ssa, .esa) bytes of an ACGT text + terminator, derived as write_raw_index derives them."""
    t = np.concatenate([np.frombuffer(text, np.uint8), np.zeros(1, np.uint8)])
    sa = synth.suffix_array(t)
    bwt = t[sa - 1]
    starts = np.concatenate([[0], np.nonzero(bwt[1:] != bwt[:-1])[0] + 1])
    ends = np.concatenate([starts[1:] - 1, [len(t) - 1]])
    return [bwt.tobytes()] + [np.stack([rows, sa[rows]], axis=1).astype(np.uint64).tobytes() for rows in (starts, ends)]


def _check_files(out, text):
    for suf, exp in zip((".bwt", ".ssa", ".esa"), _expected(text)):
        with open(out + suf, "rb") as f:
            assert f.read() == exp, suf


def _fibonacci(n):
    a, b = b"A", b"AC"
    while len(b) < n:
        a, b = b, b + a
    return b[:n]


def _adversarial():
    rng = np.random.default_rng(7)
    rand = lambda m: synth.ACGT[rng.integers(0, 4, m)].tobytes()
    unit = rand(5000)
    return {
        "all_A": (b"A" * (1 << 20), 16),
        "period2": (b"AC" * 60000, None),
        "period3": (b"ACG" * 40000, None),
        "period7": (b"ACGTTGA" * 20000, None),
        "fibonacci": (_fibonacci(150000), None),
        "repeats": (unit * 200, 16),
        "one": (b"G", 0),
        "two": (b"TA", 0),
        "three": (b"CCC", 0),
        **{"len%d" % m: (rand(m), None) for m in (26, 27, 28, 53, 54, 55)},
        "random": (rand(1 << 20), None),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(_adversarial()))
def test_adversarial_texts(tmp_path, case):
    text, rounds = _adversarial()[case]
    out = str(tmp_path / "o")
    st = rb.build_bwt_text(np.frombuffer(text, np.uint8), out)
    _check_files(out, text)
    assert not os.path.exists(out + ".docs")
    assert st.n == len(text) + 1 and st.r == os.path.getsize(out + ".ssa") // 16
    if rounds is not None:
        assert st.rounds == rounds, st.as_dict()
    active = list(st.active)[:st.rounds]
    assert all(a > 0 for a in active) and st.max_active == max(active, default=0)
    if case == "repeats":                                        # every suffix but the last copy's waits for the long rounds
        assert st.max_active > len(text) // 2


@pytest.mark.gpu
def test_binary_equals_abi(tmp_path):
    names, seqs = _tiny_records()
    fa = str(tmp_path / "tiny.fa")
    with open(fa, "wb") as f:
        f.write(_fasta(names, seqs))
    r = subprocess.run([FA_TO_BWT, "-o", str(tmp_path / "b"), fa], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode()
    assert b"rounds" in r.stderr
    rb.build_bwt(fa, str(tmp_path / "a"))
    _same(str(tmp_path / "a"), str(tmp_path / "b"), (".bwt", ".ssa", ".esa", ".docs"))
    r = subprocess.run([FA_TO_BWT, fa], stdout=subprocess.PIPE, stderr=subprocess.PIPE)    # default prefix: the input path
    assert r.returncode == 0, r.stderr.decode()
    _same(str(tmp_path / "a"), fa, (".bwt", ".ssa", ".esa", ".docs"))


@pytest.mark.gpu
def test_one_base_records(tmp_path):
    """Records of one base each: every record is mostly padding, so many suffixes share long prefixes across records."""
    rng = np.random.default_rng(5)
    seqs = [bytes([b]) for b in synth.ACGT[rng.integers(0, 4, 300)].tolist()]
    names = ["r%d" % i for i in range(len(seqs))]
    fa = str(tmp_path / "in.fa")
    with open(fa, "wb") as f:
        f.write(_fasta(names, seqs))
    out = str(tmp_path / "o")
    st = rb.build_bwt(fa, out)
    text = b"".join(s + b"A" * synth.PAD for s in seqs)
    _check_files(out, text)
    with open(out + ".docs") as f:
        assert f.read() == "".join("%s %d\n" % (nm, i * (1 + synth.PAD)) for i, nm in enumerate(names))
    assert st.records == len(seqs) and st.n == len(text) + 1


@pytest.mark.gpu
def test_small_equals_write_raw_index(tmp_path, small_index):
    panel = synth.make_panel(*synth.CONFIGS["small"])
    exp = str(tmp_path / "exp")
    synth.write_raw_index(panel, exp, markers=False)
    fa = str(tmp_path / "small.fa")
    synth.write_fasta(panel, fa)
    out = str(tmp_path / "o")
    st = rb.build_bwt(fa, out)
    _same(exp, out, (".bwt", ".ssa", ".esa", ".docs"))
    ix = rb.GpuIndex.open(small_index)
    info = ix.info()
    ix.close()
    assert (st.n, st.r) == (info.n, info.r)
    assert st.rounds > 0 and st.max_active > 0


@pytest.mark.gpu
def test_synth_gpu_build_equals_build_index_gpu(tmp_path, small_index):
    """python tools/synth.py small DIR --gpu: FASTA -> build_bwt -> build_index -> write_mps -> build_marker_array gives the
    small index's files, and leaves only them."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "synth.py"), "small", str(tmp_path), "--gpu"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, cwd=ROOT)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    _same(small_index, str(tmp_path / "small"), (".rbwt", ".tsa", ".mab", ".docs"))
    assert sorted(os.listdir(tmp_path)) == ["small.docs", "small.mab", "small.rbwt", "small.tsa"]
