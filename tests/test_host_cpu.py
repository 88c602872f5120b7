"""CPU-only checks of the product's host side: the C-ABI library loads and exports what
include/rowbowt_gpu.h declares, the load-time re-layout decodes to the right ranks (no GPU
compute), the file readers reject garbage, the FASTX reader matches kseq, and the library
refuses to run without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, read_fastx
from oracle import oracle as O

import rowbowt_b200 as rb

HEADER = os.path.join(ROOT, "include", "rowbowt_gpu.h")
RB_ALIGN = os.path.join(ROOT, "rowbowt_b200", "rb_align")


def declared_symbols():
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(rbg_[a-z_0-9]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    L = rb.lib()
    syms = declared_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(L, s), "librowbowt_gpu.so does not export %s" % s


def test_no_oracle_in_product():
    """The product never links or imports the oracle."""
    out = subprocess.run(["ldd", rb.lib_path()], capture_output=True, text=True).stdout
    assert "oracle" not in out
    for root, _, files in os.walk(os.path.join(ROOT, "rowbowt_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp")):
                src = open(os.path.join(root, f)).read()
                assert "liboracle" not in src and "from oracle" not in src and "import oracle" not in src, f


@pytest.mark.parametrize("pre", ["toy/small.fa", "tiny/tiny", "greedy/ref.fa"])
@pytest.mark.parametrize("window", [0, 16, 24, 37, 64, 100, 256, 1000, 4096, 32767])
@pytest.mark.parametrize("layout", [4, 5])
def test_layout_selftest(pre, window, layout):
    """rank_c at every p and p+1 (hence BWT[p]==c) decoded from the 64-byte mixed leaves and the
    superblock array -- cluster windows with raw children (forced by the larger windows on these
    dense BWTs), non-power-of-two windows (magic division) and the terminator line included --
    equals a direct count over the runs."""
    chk, nl, nc = C.c_uint64(), C.c_uint64(), C.c_uint64()
    rc = rb.lib().rbg_selftest_layout(os.path.join(GOLDEN, pre).encode(), window | (layout << 16), 1, C.byref(chk), C.byref(nl), C.byref(nc))
    assert rc == 0 and chk.value > 0 and nl.value > 0
    if window >= 256:
        assert nc.value > 0


@pytest.mark.parametrize("pre", ["toy/small.fa", "tiny/tiny", "greedy/ref.fa"])
@pytest.mark.parametrize("shift", [0, 1, 2, 3, 5, 6, 7, 8, 12, 16, (4096 << 8), (1 << 8)])
def test_phi_slot_selftest(pre, shift):
    """phi(i) decoded from the 32-byte slots (the code locate_kernel runs) equals ToeholdSA::phi over the
    .tsa arrays for every text position: INLINE slots, BITMAP slots (shift <= 7), SEARCH slots (shift > 7,
    also chosen automatically under a small memory budget: the last two cases), empty slots (carry only)."""
    chk, ns, no = C.c_uint64(), C.c_uint64(), C.c_uint64()
    rc = rb.lib().rbg_selftest_phi(os.path.join(GOLDEN, pre).encode(), shift, 1, C.byref(chk), C.byref(ns), C.byref(no))
    assert rc == 0 and chk.value > 0 and ns.value > 0
    if 5 <= shift <= 16:
        assert no.value > 0
    if shift == 1:
        assert no.value == 0
    if shift >> 8:
        assert ns.value * 32 <= max(shift >> 8, 128)       # the budget was honoured (or shift hit 16: buckets + sentinel)


def test_layout_selftest_rejects_missing_file():
    chk, nl, ns = C.c_uint64(), C.c_uint64(), C.c_uint64()
    assert rb.lib().rbg_selftest_layout(b"/nonexistent/prefix", 0, 1, C.byref(chk), C.byref(nl), C.byref(ns)) != 0


@pytest.mark.skipif(rb.lib().rbg_device_count() > 0, reason="a GPU is present")
def test_fails_loudly_without_gpu():
    with pytest.raises(rb.RbgError) as e:
        rb.GpuIndex.open(os.path.join(GOLDEN, "toy", "small.fa"))
    assert e.value.code == -4 and "no CPU fallback" in str(e.value)
    p = subprocess.run([RB_ALIGN, os.path.join(GOLDEN, "toy", "small.fa"), os.path.join(GOLDEN, "toy", "simple_query.fq")],
                       capture_output=True, text=True)
    assert p.returncode == 1 and p.stdout == "" and "no CUDA device" in p.stderr


def test_open_errors_are_codes_not_aborts(tmp_path):
    h = C.c_void_p()
    assert rb.lib().rbg_index_open(b"/nonexistent/prefix", 0, 0, C.byref(h)) == -1      # RBG_E_IO
    bad = tmp_path / "bad.rbwt"
    bad.write_bytes(b"\x05" * 100)
    assert rb.lib().rbg_index_open(str(tmp_path / "bad").encode(), 0, 0, C.byref(h)) in (-2, -1)
    assert rb.lib().rbg_last_error()


WEIRD = (b">a desc here\r\nACGT\r\nAC\r\n\r\n>b\nTTTT\n@c comment\nACGTACGT\n+c\nIIIIIIII\n"
         b"@d\nAC\nGT\n+\nII\nII\n>e\tx\nGGCAGGCGGA\n\n\n>f\n>g\nA\n")


def parse_only(path, *extra):
    p = subprocess.run([RB_ALIGN, "--parse-only", *extra, path], capture_output=True)
    recs = [ln.split(b"\t") for ln in p.stdout.split(b"\n") if ln]
    return p.returncode, [r[0].decode() for r in recs], [r[1] if len(r) > 1 else b"" for r in recs], p.stderr.decode()


def test_fastx_reader_semantics(tmp_path):
    f = tmp_path / "w.fq"
    f.write_bytes(WEIRD)
    rc, names, seqs, _ = parse_only(str(f))
    assert rc == 0
    assert names == ["a", "b", "c", "d", "e", "f", "g"]
    assert seqs == [b"ACGTAC", b"TTTT", b"ACGTACGT", b"ACGT", b"GGCAGGCGGA", b"", b"A"]
    import gzip
    g = tmp_path / "w.fq.gz"
    g.write_bytes(gzip.compress(WEIRD))
    assert parse_only(str(g))[1:3] == (names, seqs)
    t = tmp_path / "trunc.fq"
    t.write_bytes(b"@r1\nACGT\n+\nIIII\n@r2\nACGT\n+\nII\n")
    rc, names, seqs, err = parse_only(str(t))
    assert rc == 1 and names == ["r1"] and "truncated quality string" in err


@pytest.mark.skipif(not O.have_ref(), reason="compiled reference (oracle/_ref) not present")
def test_fastx_reader_matches_kseq_through_reference(tmp_path):
    """Names and sequences as kseq hands them to the reference: rb_align (reference) on the same
    odd file prints the names we parse, and ranges equal to the oracle on the sequences we parse."""
    f = tmp_path / "w.fq"
    f.write_bytes(WEIRD)
    rc, names, seqs, _ = parse_only(str(f))
    ref = O.ref_rb_align(os.path.join(GOLDEN, "toy", "small.fa"), str(f))
    ix = O.OracleIndex.open(os.path.join(GOLDEN, "toy", "small.fa"))
    assert ix.report(names, seqs) == ref


@pytest.mark.skipif(not O.have_ref(), reason="compiled reference (oracle/_ref) not present")
def test_fastx_reader_matches_kseq_on_random_irregular_input(tmp_path):
    """The same through random FASTQ-like inputs (tools/fuzz_parsers.py's generator: multi-line, CRLF and FASTA records, blank and
    garbage lines, embedded NULs, truncation anywhere): what kseq hands the reference is what the reader here parses -- same report,
    same exit status, same ERROR line.  tools/fuzz_kseq_reference.py is the long-running form (885 inputs, no difference)."""
    import random
    from tools.fuzz_parsers import gen
    toy = os.path.join(GOLDEN, "toy", "small.fa")
    ix = O.OracleIndex.open(toy)
    ref = os.path.join(O.REFBIN, "rb_align")
    f = tmp_path / "r.fq"
    for it in range(30):
        f.write_bytes(gen(random.Random(7_000_000 + it)))
        rc, names, seqs, err = parse_only(str(f), "--threads", "1")
        q = subprocess.run([ref, toy, str(f)], capture_output=True)
        assert ix.report(names, seqs) == q.stdout.decode(errors="replace"), it
        assert (rc != 0) == (q.returncode != 0), it
        assert [ln for ln in err.splitlines() if ln.startswith("ERROR")] == \
               [ln for ln in q.stderr.decode(errors="replace").splitlines() if ln.startswith("ERROR")], it


def _random_fastq(rng, n, irregular):
    """Strict four-line records with hostile quality strings ('@', '+', '>' anywhere, also first);
    with `irregular`, a few FASTA records, multi-line records, CRLF records and blank lines."""
    out = []
    for i in range(n):
        L = int(rng.integers(1, 200))
        seq = bytes(rng.choice(np.frombuffer(b"ACGTN", np.uint8), L))
        qual = bytes(rng.choice(np.frombuffer(b"@+>IJ#!", np.uint8), L))
        name = b"r%d" % i + (b" comment @x +y" if rng.random() < 0.3 else b"")
        r = rng.random() if irregular else 1.0
        if r < 0.004:
            out.append(b">fa%d desc\nACGT\nAC\n\n" % i)
        elif r < 0.008:
            out.append(b"@ml%d\nACGT\nACGT\n+\nIIII\nIIII\n" % i)
        elif r < 0.012:
            out.append(b"@cr%d\r\nACGT\r\n+\r\nIIII\r\n" % i)
        elif r < 0.014:
            out.append(b"\n\n")
        else:
            out.append(b"@" + name + b"\n" + seq + b"\n+" + (name if rng.random() < 0.5 else b"") + b"\n" + qual + b"\n")
    return b"".join(out)


@pytest.mark.parametrize("chunk", [64, 100, 1000, 4096, 100000])
@pytest.mark.parametrize("irregular", [False, True])
def test_parallel_parser_equals_sequential(tmp_path, chunk, irregular):
    """fastx_parallel.hpp: chunked, multi-threaded parsing with verified chunk starts yields exactly the
    records of the sequential kseq-compatible reader, whatever the chunk size; irregular input falls back."""
    rng = np.random.default_rng(chunk + irregular)
    f = tmp_path / "p.fq"
    f.write_bytes(_random_fastq(rng, 4000, irregular))
    rc1, n1, s1, e1 = parse_only(str(f), "-t", "1")
    rc4, n4, s4, e4 = parse_only(str(f), "-t", "4", "-c", str(chunk))
    assert "sequential" in e1 and "parallel" in e4
    assert (rc1, n1, s1) == (rc4, n4, s4) and rc1 == 0 and len(n1) >= 3900
    assert ("1 fallbacks" in e4) == irregular


def test_parallel_parser_edge_files(tmp_path):
    rng = np.random.default_rng(5)
    body = _random_fastq(rng, 500, False)
    cases = {
        "trunc": body + b"@x\nACGT\n+\nII\n",                   # kseq: -2, records before it are kept
        "nonl": body[:-1],                                       # no newline at the end of the file
        "nul": b"@a\x00b\nAC\x00GT\n+\nIIIII\n@c\nACGT\n+\nIIII\n",  # name and sequence are C strings
        "fasta": b">a\nACGT\n>b\nGG\nTT\n" * 50,
        "junk_between": body + b"garbage line\n" + body,
        "empty": b"",
    }
    for tag, data in cases.items():
        f = tmp_path / (tag + ".fq")
        f.write_bytes(data)
        a = parse_only(str(f), "-t", "1")
        b = parse_only(str(f), "-t", "3", "-c", "300")
        assert a[:3] == b[:3], tag
        assert a[0] == (1 if tag == "trunc" else 0), tag
    assert parse_only(str(tmp_path / "nul.fq"), "-t", "3", "-c", "64")[1:3] == (["a", "c"], [b"AC", b"ACGT"])


def test_golden_reader_agrees_with_test_helper():
    for fq in ("toy/simple_query.fq", "tiny/noisy.fq"):
        rc, names, seqs, _ = parse_only(os.path.join(GOLDEN, fq))
        n2, s2 = read_fastx(os.path.join(GOLDEN, fq))
        assert rc == 0 and names == n2 and seqs == s2


def test_result_checksum_is_order_sensitive_per_index():
    lo = np.array([1, 2, 3], np.uint64)
    hi = np.array([4, 5, 6], np.uint64)
    a = rb.result_checksum(lo, hi)
    assert a == rb.result_checksum(lo.copy(), hi.copy())
    assert a != rb.result_checksum(lo[::-1].copy(), hi)


# ---- wt_fbb indexes (`--fbb`, SURVEY 8(f) row 3) ------------------------------------------------------
def test_fbb_index_decodes_to_the_reference_rle_file(tmp_path):
    """tests/golden/fbb/tiny.rbwt is a wt_fbb written by the reference `rb_build --fbb` from raw/tiny.bwt.  The product's
    reader (csrc/formats.cpp read_rbwt_fbb) decodes it into runs; serialized as an rle_string .rbwt they must be,
    byte for byte, the file the reference's plain rb_build wrote for the same BWT (tests/golden/tiny/tiny.rbwt)."""
    out = str(tmp_path / "tiny")
    rc = rb.lib().rbg_selftest_rewrite(os.path.join(GOLDEN, "fbb", "tiny").encode(), out.encode(), 8)
    assert rc == 0
    assert open(out + ".rbwt", "rb").read() == open(os.path.join(GOLDEN, "tiny", "tiny.rbwt"), "rb").read()


def test_fbb_oracle_reader_returns_the_raw_bwt():
    """The oracle's independent numpy/python wt_fbb reader gives back the bytes of the .bwt the index was built from."""
    from oracle import rbformats as F
    text = F.read_fbb_text(os.path.join(GOLDEN, "fbb", "tiny.rbwt"))
    raw = np.fromfile(os.path.join(GOLDEN, "raw", "tiny.bwt"), dtype=np.uint8)
    assert np.array_equal(text, raw)


def test_fbb_reader_rejects_an_rle_file_and_vice_versa(tmp_path):
    lib = rb.lib()
    assert lib.rbg_selftest_rewrite(os.path.join(GOLDEN, "tiny", "tiny").encode(), str(tmp_path / "x").encode(), 8) != 0
    assert lib.rbg_selftest_rewrite(os.path.join(GOLDEN, "fbb", "tiny").encode(), str(tmp_path / "y").encode(), 1) != 0
    # truncated wt_fbb
    data = open(os.path.join(GOLDEN, "fbb", "tiny.rbwt"), "rb").read()
    for cut in (7, 100, 3000, len(data) - 1):
        p = tmp_path / ("cut%d" % cut)
        open(str(p) + ".rbwt", "wb").write(data[:cut])
        assert lib.rbg_selftest_rewrite(str(p).encode(), str(tmp_path / "z").encode(), 8) != 0


def test_fbb_reader_survives_corrupted_files(tmp_path, capfd):
    """Random byte flips in a wt_fbb file: the reader returns an error code or a (different) decode, it never
    crashes -- the C ABI contract (errors are codes, SURVEY 8(b))."""
    import random
    data = open(os.path.join(GOLDEN, "fbb", "tiny.rbwt"), "rb").read()
    rnd = random.Random(7)
    lib = rb.lib()
    rejected = 0
    for it in range(120):
        d = bytearray(data)
        for _ in range(rnd.randint(1, 4)):
            d[rnd.randrange(len(d))] = rnd.randrange(256)
        p = str(tmp_path / "f")
        open(p + ".rbwt", "wb").write(d)
        rejected += lib.rbg_selftest_rewrite(p.encode(), (p + "_o").encode(), 8) != 0
    capfd.readouterr()                     # the selftest hook prints the reader's message; not part of the result
    assert rejected > 0


@pytest.mark.parametrize("parts", ["2", "3", "8", "64"])
@pytest.mark.parametrize("shift", [0, 3, 7, 9])
def test_phi_directory_built_in_parts(parts, shift, monkeypatch):
    """Large indexes build the phi directory on several threads (keys cut at 32-bucket group boundaries, part-local
    value indexes rebased when the parts are joined): forced here on the small fixtures, every position checked."""
    monkeypatch.setenv("RBG_PHI_PARTS", parts)
    for pre in ("toy/small.fa", "tiny/tiny"):
        chk = C.c_uint64()
        rc = rb.lib().rbg_selftest_phi(os.path.join(GOLDEN, pre).encode(), shift, 1, C.byref(chk), None, None)
        assert rc == 0 and chk.value > 0


def test_fbb_multi_superblock_index(tmp_path):
    """A wt_fbb over 2.5 M symbols (three superblocks, partial last block, blocks of every tree height the data has):
    decoded and re-serialized as an rle_string it equals, byte for byte, the reference's plain rb_build output for the
    same text (tests/golden/fbb/multi.rle.rbwt); the oracle's independent reader agrees on the run-length encoding."""
    out = str(tmp_path / "multi")
    assert rb.lib().rbg_selftest_rewrite(os.path.join(GOLDEN, "fbb", "multi").encode(), out.encode(), 8) == 0
    assert open(out + ".rbwt", "rb").read() == open(os.path.join(GOLDEN, "fbb", "multi.rle.rbwt"), "rb").read()
    from oracle import rbformats as F
    text = F.read_fbb_text(os.path.join(GOLDEN, "fbb", "multi.rbwt"))
    assert len(text) == 2_500_123
    heads = text[np.r_[True, text[1:] != text[:-1]]]
    rle = F.read_rbwt(os.path.join(GOLDEN, "fbb", "multi.rle.rbwt"))
    assert np.array_equal(np.where(heads == 0, 1, heads), rle.heads)


@pytest.mark.parametrize("threads", ["1", "2", "3", "8"])
def test_fbb_superblocks_decoded_on_threads(threads, tmp_path, monkeypatch):
    """Large wt_fbb files are decoded superblock groups in parallel and the run lists joined (runs continue across
    group boundaries): forced here on the three-superblock fixture; the result is the reference's rle file again."""
    monkeypatch.setenv("RBG_FBB_THREADS", threads)
    for name, ref in (("multi", os.path.join(GOLDEN, "fbb", "multi.rle.rbwt")), ("tiny", os.path.join(GOLDEN, "tiny", "tiny.rbwt"))):
        out = str(tmp_path / name)
        assert rb.lib().rbg_selftest_rewrite(os.path.join(GOLDEN, "fbb", name).encode(), out.encode(), 8) == 0
        assert open(out + ".rbwt", "rb").read() == open(ref, "rb").read()


# ---- BGZF inputs: blocks inflated on several threads behind the sequential record reader ----------------
def _bgzf(data: bytes, block: int = 60000, eof_block: bool = True) -> bytes:
    import struct
    import zlib
    out = bytearray()
    chunks = [data[a:a + block] for a in range(0, len(data), block)] + ([b""] if eof_block else [])
    for chunk in chunks:
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        cd = c.compress(chunk) + c.flush()
        out += b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, 12 + 6 + len(cd) + 8 - 1)
        out += cd + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk))
    return bytes(out)


@pytest.mark.parametrize("block", [1, 7, 300, 60000])
def test_bgzf_input_equals_plain_input(tmp_path, block):
    """A bgzip-style file (independent gzip members with a 'BC' size field) goes through BgzfSource: same records
    as the plain file and as the one-stream .gz, for block sizes that cut records anywhere."""
    rng = np.random.default_rng(5)
    recs = []
    for i in range(3000 if block >= 300 else 60):
        m = int(rng.integers(1, 260))
        seq = bytes(rng.choice(np.frombuffer(b"ACGTN", np.uint8), m))
        recs.append(b"@r%d some comment\n%s\n+\n%s\n" % (i, seq, b"@" * m))       # '@' qualities: worst case for any guessing
    data = b"".join(recs) + WEIRD
    plain = tmp_path / "p.fq"
    plain.write_bytes(data)
    want = parse_only(str(plain))
    assert want[0] == 0 and len(want[1]) > 60
    for eof_block in (True, False):
        z = tmp_path / ("b%d.fq.gz" % eof_block)
        z.write_bytes(_bgzf(data, block, eof_block))
        import gzip
        assert gzip.decompress(z.read_bytes()) == data                       # it IS a valid gzip file
        got = parse_only(str(z))
        assert got[0] == 0 and got[1] == want[1] and got[2] == want[2]
        got = parse_only(str(z), "--threads", "3")
        assert got[1] == want[1] and got[2] == want[2]


@pytest.mark.parametrize("block", [7, 300, 4000, 60000])
@pytest.mark.parametrize("margin", ["0", "40", "700", None])
def test_bgzf_chunk_parser_equals_plain_input(tmp_path, block, margin):
    """BGZF input through the CHUNK parser (block table -> every parser thread inflates the blocks under its chunk into
    a private view): same records as the plain file for chunks and blocks that cut records anywhere, and for view
    margins so small that records run into the end of a view (a bail, never taken for the end of the input)."""
    rng = np.random.default_rng(11)
    recs = []
    for i in range(2500 if block >= 300 else 120):
        m = int(rng.integers(1, 260))
        seq = bytes(rng.choice(np.frombuffer(b"ACGTN", np.uint8), m))
        recs.append(b"@r%d some comment\n%s\n+\n%s\n" % (i, seq, b"@" * m))
    env = dict(os.environ)
    if margin is not None:
        env["RBG_VIEW_MARGIN"] = margin
    for tail in (b"", b"@last\nACGT\n+\nIIII", WEIRD):               # newline-terminated, unterminated last record, kseq oddities
        data = b"".join(recs) + tail
        plain = tmp_path / "p.fq"
        plain.write_bytes(data)
        want = parse_only(str(plain), "--threads", "1")
        assert want[0] == 0
        z = tmp_path / "b.fq.gz"
        z.write_bytes(_bgzf(data, block, eof_block=bool(block % 2)))
        for chunk in ("1500", "40000", "300000"):
            p = subprocess.run([RB_ALIGN, "--parse-only", "--threads", "4", "--chunk-bytes", chunk, str(z)], capture_output=True, env=env)
            got = [ln.split(b"\t") for ln in p.stdout.split(b"\n") if ln]
            assert p.returncode == 0, p.stderr.decode()
            assert [g[0].decode() for g in got] == want[1] and [g[1] if len(g) > 1 else b"" for g in got] == want[2]
            assert b"parallel" in p.stderr


def test_bgzf_chunk_parser_reports_a_bad_block_in_its_place(tmp_path):
    """A block that does not inflate (flipped payload bit) in the middle of a BGZF file read by the chunk parser: every
    record in front of it (up to the 32-block group the sequential reader inflates it in) is delivered, in order, then
    kseq's stream error."""
    data = b"".join(b"@r%d\nACGTACGTAC\n+\nIIIIIIIIII\n" % i for i in range(20000))
    bad = bytearray(_bgzf(data, 5000))
    bad[len(bad) // 2] ^= 0x10
    f = tmp_path / "bad.fq.gz"
    f.write_bytes(bad)
    # which block is broken, and how many records end in front of the group of 32 blocks the sequential reader inflates it in
    import struct
    at, blocks = 0, []
    while at < len(bad):
        blocks.append(at)
        at += struct.unpack_from("<H", bad, at + 16)[0] + 1
    broken = max(i for i, a in enumerate(blocks) if a <= len(bad) // 2)
    ends = np.cumsum([len(b"@r%d\nACGTACGTAC\n+\nIIIIIIIIII\n" % i) for i in range(20000)])
    at_least = int(np.searchsorted(ends, max(0, broken - 32) * 5000, side="right"))
    at_most = int(np.searchsorted(ends, broken * 5000, side="right"))
    assert at_least > 1000
    for chunk in ("3000", "100000", "1000000"):
        rc, names, seqs, err = parse_only(str(f), "--threads", "4", "--chunk-bytes", chunk)
        assert rc == 1 and "error reading stream" in err
        assert at_least <= len(names) <= at_most
        assert names == ["r%d" % i for i in range(len(names))] and all(s == b"ACGTACGTAC" for s in seqs)


def test_bgzf_corruption_is_a_stream_error(tmp_path):
    data = b"".join(b"@r%d\nACGTACGTAC\n+\nIIIIIIIIII\n" % i for i in range(20000))
    good = bytearray(_bgzf(data, 5000))
    # a flipped bit in the middle of the payload of a block: CRC / inflate failure -> kseq's -3
    bad = bytearray(good)
    bad[len(bad) // 2] ^= 0x10
    f = tmp_path / "bad.fq.gz"
    f.write_bytes(bad)
    rc, names, _, err = parse_only(str(f))
    assert rc == 1 and "error reading stream" in err and len(names) < 20000
    # good blocks followed by bytes that are no block
    f2 = tmp_path / "tail.fq.gz"
    f2.write_bytes(bytes(good) + b"garbage-after-the-last-block")
    rc, names, _, err = parse_only(str(f2))
    assert rc == 1 and "error reading stream" in err
    # only the empty end-of-file block
    f3 = tmp_path / "empty.fq.gz"
    f3.write_bytes(_bgzf(b""))
    rc, names, _, _ = parse_only(str(f3))
    assert rc == 0 and names == []


@pytest.mark.parametrize("pre", ["toy/small.fa", "tiny/tiny", "greedy/ref.fa"])
@pytest.mark.parametrize("shift", [0, 1, 3, 8, 9, 16, 17, 24])
def test_toehold_directory_selftest(pre, shift):
    """ToeholdDir (bucket table + keys reduced to 1 / 2 / 4 bytes + samples as a u32 plane): the row LF(end of run j)
    selects samples_last[j] for every run j, for every key width."""
    chk, nbytes = C.c_uint64(), C.c_uint64()
    rc = rb.lib().rbg_selftest_toehold(os.path.join(GOLDEN, pre).encode(), shift, C.byref(chk), C.byref(nbytes))
    assert rc == 0 and chk.value > 1000 and nbytes.value > 0


def _pack_numpy(bases, offs, code_of):
    """Restatement of pack_kernel / rbg_pack_bytes: base at byte x -> bits 2*(x&31) of packed[x>>5]; flags per read."""
    n_bytes = int(offs[-1])
    codes = code_of[bases[:n_bytes]].astype(np.int64)
    good = (codes >= 0) & (codes < 4)
    words = np.zeros((n_bytes + 31) // 32, np.uint64)
    x = np.nonzero(good)[0]
    np.bitwise_or.at(words, x >> 5, codes[x].astype(np.uint64) << (np.uint64(2) * (x & 31).astype(np.uint64)))
    flags = np.zeros(len(offs) - 1, np.uint8)
    owner = np.searchsorted(offs, np.arange(n_bytes), side="right") - 1
    np.bitwise_or.at(flags, owner[codes < 0], 1)
    np.bitwise_or.at(flags, owner[codes == 4], 2)
    return words, flags, int((codes == 4).sum())


@pytest.mark.parametrize("table", ["acgt", "acgt+term", "no-T"])
@pytest.mark.parametrize("threads", [1, 4])
def test_host_packer_equals_restatement(table, threads):
    """rbg_pack_bytes (AVX2/BMI2 fast path + byte-wise path) against a numpy restatement: ragged reads, empty reads,
    bytes without a code (N, lowercase, 0xff, NUL), terminator bytes, an index without 'T', ranges packed by
    several threads at word-aligned cuts."""
    rng = np.random.default_rng(3)
    code_of = np.full(256, -1, np.int8)
    for i, c in enumerate(b"ACGT"):
        code_of[c] = i
    if table == "acgt+term":
        code_of[1] = 4
    if table == "no-T":
        code_of[ord("T")] = -1
    reads = []
    acgt = np.frombuffer(b"ACGT", np.uint8)
    for i in range(3000):
        m = int(rng.integers(0, 260))
        r = acgt[rng.integers(0, 4, m)].copy()
        if m and i % 7 == 0:
            r[rng.integers(0, m, 1 + m // 50)] = rng.choice(np.frombuffer(b"N\x01acgt\xff\x00n", np.uint8))
        reads.append(r)
    lens = np.array([len(r) for r in reads], np.uint64)
    offs = np.zeros(len(reads) + 1, np.uint64)
    np.cumsum(lens, out=offs[1:])
    bases = np.concatenate(reads + [np.zeros(64, np.uint8)])
    n, n_bytes = len(reads), int(offs[-1])
    want_w, want_f, want_ex = _pack_numpy(bases, offs, code_of)
    packed = np.full(len(want_w) + 2, 0xDEADBEEF, np.uint64)
    flags = np.zeros(n + 8, np.uint8)
    ex = C.c_uint64(0)
    cuts = [min(n_bytes, ((n_bytes * t // threads) + 31) // 32 * 32) for t in range(threads)] + [n_bytes]

    def job(t):
        assert rb.lib().rbg_selftest_pack(code_of.ctypes.data, bases.ctypes.data, offs.ctypes.data, n, cuts[t], cuts[t + 1],
                                          packed.ctypes.data, flags.ctypes.data, C.byref(ex)) == 0
    import concurrent.futures as cf
    with cf.ThreadPoolExecutor(threads) as pool:
        list(pool.map(job, range(threads)))
    assert np.array_equal(packed[:len(want_w)], want_w)
    assert packed[len(want_w)] == 0xDEADBEEF                       # nothing written past the last word
    assert np.array_equal(flags[:n], want_f)
    assert ex.value == want_ex
    if table != "acgt+term":
        assert want_ex == 0 and (want_f & 1).any()


@pytest.mark.parametrize("gz", [False, True])
@pytest.mark.parametrize("threads", ["1", "4"])
def test_piped_input_loses_no_reads(tmp_path, gz, threads):
    """A FIFO (what <(zcat x.fq.gz) or /dev/stdin is) must be opened exactly once: every probe of the path would eat
    the head of the stream.  The reference reads pipes through gzopen/kseq without loss (src/rb_align.cpp:169-176)."""
    import gzip
    import threading
    rng = np.random.default_rng(11)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    recs = [(b"r%d" % i, acgt[rng.integers(0, 4, int(rng.integers(20, 200)))].tobytes()) for i in range(2000)]
    data = b"".join(b"@%s\n%s\n+\n%s\n" % (n, s, b"I" * len(s)) for n, s in recs)
    payload = gzip.compress(data) if gz else data
    fifo = str(tmp_path / "pipe.fq")
    os.mkfifo(fifo)

    def feed():
        with open(fifo, "wb") as f:
            f.write(payload)
    t = threading.Thread(target=feed)
    t.start()
    rc, names, seqs, err = parse_only(fifo, "--threads", threads)
    t.join()
    assert rc == 0, err
    assert names == [n.decode() for n, _ in recs]
    assert seqs == [s for _, s in recs]


def test_bgzf_block_smaller_than_its_header_is_a_stream_error(tmp_path):
    """A crafted BGZF block whose BSIZE is smaller than header + trailer must fail as a stream error (kseq's -3),
    not read past the mapping."""
    import struct
    good = _bgzf(b"@r1\nACGT\n+\nIIII\n", eof_block=False)
    # header with XLEN = 200 but BSIZE = 27 (total 28 bytes): 12 + xlen + 8 > bs
    hdr = b"\x1f\x8b\x08\x04" + b"\x00" * 6 + struct.pack("<H", 200) + b"BC" + struct.pack("<HH", 2, 27)
    blob = hdr + b"\x00" * 300
    f = tmp_path / "crafted.fq.gz"
    f.write_bytes(good + blob)
    rc, names, seqs, err = parse_only(str(f), "--threads", "4")
    assert rc == 1 and "error reading stream" in err


def test_report_writers_agree():
    """rb_align --format-selftest: random results (empty / wrapped ranges, u64 and narrow locations, markers, a document
    list with a duplicate start) through the plain report writer and through format_report (report_format.hpp), all four
    flag sets -- byte-identical -- plus put_dec against printf over 2 M values."""
    p = subprocess.run([RB_ALIGN, "--format-selftest", "20000"], capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    assert p.stdout.startswith(b"format-selftest ok")


_SELFTEST_CHILD = """
import sys, ctypes as C
sys.path.insert(0, %r)
import rowbowt_b200 as rb
lib, pre = rb.lib(), sys.argv[1].encode()
a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
print(lib.rbg_selftest_layout(pre, 0, 7, C.byref(a), C.byref(b), C.byref(c)),
      lib.rbg_selftest_toehold(pre, 0, C.byref(a), C.byref(b)),
      lib.rbg_selftest_phi(pre, 0, 7, C.byref(a), C.byref(b), C.byref(c)),
      lib.rbg_selftest_rewrite(pre, (sys.argv[1] + ".out").encode(), 7))
"""


def _selftests_in_a_child(prefix):
    import sys
    p = subprocess.run([sys.executable, "-c", _SELFTEST_CHILD % ROOT, prefix], capture_output=True)
    return p.returncode, p.stdout.decode().split()


def test_corrupted_index_files_end_as_format_errors(tmp_path):
    """Index files with flipped bytes or cut short: the readers and the layout builders (run on the host by the self-checks)
    must refuse them or build a self-consistent layout, never touch memory out of range.  First the case a fuzzing run found: three
    bytes of toy's .rbwt changed so that one run length wraps below zero while the lengths still sum to n modulo 2^64."""
    import random
    import shutil
    toy = os.path.join(GOLDEN, "toy", "small.fa")

    def fresh(src):
        pre = str(tmp_path / "x")
        for suf in (".rbwt", ".tsa", ".mab"):
            shutil.copy(src + suf, pre + suf)
        return pre

    pre = fresh(toy)
    rc, out = _selftests_in_a_child(pre)
    assert rc == 0 and out == ["0", "0", "0", "0"]
    b = bytearray(open(pre + ".rbwt", "rb").read())
    b[3508], b[5103], b[13541] = 0x9B, 0x1E, 0x2F
    open(pre + ".rbwt", "wb").write(b)
    rc, out = _selftests_in_a_child(pre)
    assert rc == 0, "the child crashed (rc %d)" % rc
    assert out[0] == "-1" and out[1] == "-1"                # format_error from validate_runs, not a walk over a wrapped length
    rng = random.Random(20)
    for it in range(24):
        pre = fresh(rng.choice([toy, os.path.join(GOLDEN, "tiny", "tiny")]))
        suf = rng.choice([".rbwt", ".tsa", ".mab"])
        b = bytearray(open(pre + suf, "rb").read())
        if rng.random() < 0.3:
            b = b[:rng.randint(0, len(b))]
        else:
            for _ in range(rng.randint(1, 4)):
                b[rng.randrange(len(b))] = rng.randrange(256)
        open(pre + suf, "wb").write(b)
        rc, out = _selftests_in_a_child(pre)
        assert rc == 0, "the child crashed on corruption %d of %s (rc %d)" % (it, suf, rc)
        assert len(out) == 4


@pytest.mark.parametrize("compiler,std", [("gcc", "-std=c99"), ("g++", "-std=c++11")])
def test_public_header_compiles_as_c_and_cpp_and_links(compiler, std, tmp_path):
    """include/rowbowt_gpu.h is the whole boundary: a plain C99 (and a C++11) translation unit that includes nothing else compiles
    under -Wall -Wextra -pedantic, links against librowbowt_gpu.so, and a call on a missing index comes back as an error code with
    the reference's message -- not an exit, not an exception (no device is touched before the files are read)."""
    src = tmp_path / "client.c"
    src.write_text(
        '#include "rowbowt_gpu.h"\n#include <stdio.h>\n#include <string.h>\n'
        'int main(void) {\n'
        '    rbg_index* ix = NULL;\n'
        '    rbg_result res;\n'
        '    rbg_batch in;\n'
        '    int rc = rbg_index_open("/nonexistent/prefix", RBG_LOAD_SA | RBG_LOAD_MA | RBG_LOAD_CACHE, 0, &ix);\n'
        '    memset(&res, 0, sizeof res); memset(&in, 0, sizeof in);\n'
        '    printf("%d %s\\n", rc, rbg_last_error());\n'
        '    return (rc == RBG_E_IO && ix == NULL && RBG_LOCATE != RBG_MARKERS) ? 0 : 1;\n'
        '}\n')
    exe = str(tmp_path / "client")
    lib_dir = os.path.join(ROOT, "rowbowt_b200")
    cmd = [compiler, std, "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include")]
    cmd += ["-x", "c++"] if compiler == "g++" else []
    cmd += [str(src), "-L", lib_dir, "-lrowbowt_gpu", "-Wl,-rpath," + lib_dir, "-o", exe]
    p = subprocess.run(cmd, capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    p = subprocess.run([exe], capture_output=True)
    assert p.returncode == 0, (p.stdout, p.stderr)
    assert b"bad file" in p.stdout


FAST_DIV_HARNESS = r"""
#include <vector_types.h>
#include <cstdio>
#include <thread>
#include <vector>
#include "device_index.cuh"

// set_fast_div for window W over n positions; the quotient x / m (m = odd part of W) for x = p >> div_k < 2^31
static rbg::DevLeafDir div_for(uint32_t W, uint64_t n) {
    rbg::DevLeafDir D{};
    D.window = W;
    D.n = n;
    rbg::set_fast_div(D);
    return D;
}

int main() {
    const uint64_t top = 1ull << 31;
    long long bad = 0;
    std::vector<uint32_t> mul_of(32768, 0), s_of(32768, 0);
    for (uint32_t W = 16; W <= 32767; ++W) {
        uint32_t k = 0;
        while (!((W >> k) & 1u)) ++k;
        const uint64_t m = W >> k, n_max = (top << k) - 1;       // the largest n with (n >> k) < 2^31
        const rbg::DevLeafDir D = div_for(W, n_max);
        if (!D.div_fast || D.div_k != k) { printf("W=%u: no fast path at n=%llu\n", W, (unsigned long long) n_max); ++bad; continue; }
        if (div_for(W, n_max + 1).div_fast) { printf("W=%u: fast path at n=%llu\n", W, (unsigned long long) (n_max + 1)); ++bad; }
        for (uint64_t x = top - (1ull << 16); x < top; ++x)
            if (((x * D.div_mul) >> D.div_s) != x / m && bad++ < 20) printf("W=%u x=%llu\n", W, (unsigned long long) x);
        if (mul_of[m] && (mul_of[m] != D.div_mul || s_of[m] != D.div_s)) { printf("W=%u: multiplier differs\n", W); ++bad; }
        mul_of[m] = D.div_mul;
        s_of[m] = D.div_s;
    }
    // every x = 0 and x = -1 (mod m) among the top 2^24 values below 2^31, once per odd part m (div_mul / div_s depend on m only)
    const unsigned T = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<long long> wrong(T, 0);
    std::vector<std::thread> th;
    for (unsigned t = 0; t < T; ++t)
        th.emplace_back([&, t] {
            for (uint64_t m = 1 + 2 * t; m < 32768; m += 2 * T) {
                if (!mul_of[m]) continue;
                const uint64_t mul = mul_of[m], s = s_of[m], q0 = (top - (1ull << 24)) / m;
                for (uint64_t q = q0, x = q0 * m; x < top; ++q, x += m) {
                    wrong[t] += ((x * mul) >> s) != q;
                    if (x + m - 1 < top) wrong[t] += (((x + m - 1) * mul) >> s) != q;
                }
            }
        });
    for (auto& x : th) x.join();
    for (long long w : wrong) bad += w;
    printf("%lld wrong\n", bad);
    return bad ? 1 : 0;
}
"""


def test_fast_window_division_is_exact(tmp_path):
    """line_of divides a BWT position by the window with set_fast_div's 32-bit multiplier whenever (n >> k) < 2^31
    (W = m * 2^k, m odd).  The real set_fast_div (device_index.cuh) against exact division for every window in [16, 32767]
    at the largest n that enables the fast path: the top 2^16 quotient arguments below 2^31 and every multiple of m and
    every x = -1 (mod m) among the top 2^24; one step past that n the fast path must be off."""
    import shutil
    cxx = shutil.which("g++") or shutil.which("c++")
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")      # vector_types.h: ulonglong2
    if not cxx or not os.path.exists(os.path.join(cuda_inc, "vector_types.h")):
        pytest.skip("no host C++ compiler or CUDA toolkit headers")
    src = tmp_path / "fast_div.cpp"
    src.write_text(FAST_DIV_HARNESS)
    exe = str(tmp_path / "fast_div")
    p = subprocess.run([cxx, "-O2", "-std=c++17", "-pthread", "-I", cuda_inc, "-I", os.path.join(ROOT, "rowbowt_b200", "csrc"),
                        str(src), "-o", exe], capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    p = subprocess.run([exe], capture_output=True)
    assert p.returncode == 0, p.stdout.decode()
    assert p.stdout.decode().strip() == "0 wrong"
