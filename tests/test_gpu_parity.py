"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the
C ABI, against the oracle on the same inputs and against the committed stdout of the
reference rb_align.  Bit-exact: integer/index work only."""
import os
import subprocess

import numpy as np
import pytest

from conftest import FIXTURES, GOLDEN, ROOT, fixture_cases, read_fastx
from oracle import oracle as O

import rowbowt_b200 as rb
from rowbowt_b200 import RBG_COUNT, RBG_LOCATE, RBG_MARKERS

pytestmark = pytest.mark.gpu
RB_ALIGN = os.path.join(ROOT, "rowbowt_b200", "rb_align")


def compare_with_oracle(gpu_res, orc, seqs, sa, ma):
    lo, hi, k = orc.find_ranges(seqs, toehold=sa)
    assert np.array_equal(gpu_res.lo, lo)
    assert np.array_equal(gpu_res.hi, hi)
    if sa:
        assert np.array_equal(gpu_res.toehold, k)
        for i in range(len(seqs)):
            exp = orc.locate(lo[i], hi[i], k[i])
            assert np.array_equal(gpu_res.locs[gpu_res.loc_off[i]:gpu_res.loc_off[i + 1]], exp), i
    if ma:
        for i in range(len(seqs)):
            exp = orc.markers_at_range(lo[i], hi[i])
            assert np.array_equal(gpu_res.markers[gpu_res.mk_off[i]:gpu_res.mk_off[i + 1]], exp), i
    return lo, hi, k


@pytest.mark.parametrize("d,pre,fq,tag,sa,ma", list(fixture_cases()))
def test_rb_align_binary_matches_reference_stdout(d, pre, fq, tag, sa, ma):
    """The host rb_align over the C ABI prints byte-for-byte what the reference rb_align printed."""
    cmd = [RB_ALIGN] + (["-s"] if sa else []) + (["-m"] if ma else []) + ["--batch", "97",
                                                                          os.path.join(GOLDEN, d, pre), os.path.join(GOLDEN, d, fq)]
    p = subprocess.run(cmd, capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    exp = open(os.path.join(GOLDEN, "expected", "%s.%s.%s.txt" % (d, fq, tag)), "rb").read()
    assert p.stdout == exp
    # stderr ends with "<load_s> <query_s>"
    last = p.stderr.decode().strip().split("\n")[-1].split()
    assert len(last) == 2 and float(last[0]) >= 0 and float(last[1]) >= 0


@pytest.mark.parametrize("d,pre,fq,tag,sa,ma", list(fixture_cases()))
def test_rb_align_parallel_host_pipeline(d, pre, fq, tag, sa, ma):
    """Same bytes through the multi-threaded front end: tiny parser chunks (= GPU batches), 4 parser and
    formatter threads, ordered writer."""
    cmd = [RB_ALIGN] + (["-s"] if sa else []) + (["-m"] if ma else []) + ["--threads", "4", "--chunk-bytes", "2000",
                                                                          os.path.join(GOLDEN, d, pre), os.path.join(GOLDEN, d, fq)]
    p = subprocess.run(cmd, capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    exp = open(os.path.join(GOLDEN, "expected", "%s.%s.%s.txt" % (d, fq, tag)), "rb").read()
    assert p.stdout == exp


@pytest.mark.parametrize("name", sorted(FIXTURES))
@pytest.mark.parametrize("layout", ["4", "5"])
def test_query_matches_oracle(name, layout, monkeypatch):
    monkeypatch.setenv("RBG_LAYOUT", layout)
    d, pre, fqs, has_ma = FIXTURES[name]
    prefix = os.path.join(GOLDEN, d, pre)
    ix = rb.GpuIndex.open(prefix, sa=True, markers=has_ma)
    orc = O.OracleIndex.open(prefix, sa=True, markers=has_ma)
    info = ix.info()
    assert (info.n, info.r) == (orc.bwt.n, orc.bwt.R)
    assert [info.F[c] for c in range(256)] == [orc.F(c) for c in range(256)]
    assert info.toehold0 == O.lib().orc_last_run_sample(orc.h)
    seqs = []
    for fq in fqs:
        seqs += read_fastx(os.path.join(GOLDEN, d, fq))[1]
    mode = RBG_LOCATE | (RBG_MARKERS if has_ma else 0)
    compare_with_oracle(ix.query(seqs, mode), orc, seqs, True, has_ma)
    # count-only kernel variant gives the same ranges
    r = ix.query(seqs, RBG_COUNT)
    lo, hi, _ = orc.find_ranges(seqs)
    assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi)
    st = ix.stats()
    assert st.lf_steps > 0 and st.launches >= 2
    ix.close()


@pytest.mark.parametrize("ftab_k", [0, 3, 10])
@pytest.mark.parametrize("layout", ["4", "5"])
def test_edge_reads_and_ragged_batches(ftab_k, layout, monkeypatch):
    monkeypatch.setenv("RBG_LAYOUT", layout)
    """Empty batch, empty read, 1-base reads, N / lowercase / terminator bytes, ragged lengths --
    with and without the k-mer seed table (reads shorter than k fall back to plain steps)."""
    prefix = os.path.join(GOLDEN, "toy", "small.fa")
    ix = rb.GpuIndex.open(prefix, sa=True, markers=True)
    ix.build_ftab(ftab_k)
    assert ix.info().ftab_k == ftab_k
    orc = O.OracleIndex.open(prefix, sa=True, markers=True)
    r = ix.query([], RBG_LOCATE | RBG_MARKERS)
    assert r.n == 0 and len(r.locs) == 0 and len(r.markers) == 0
    rng = np.random.default_rng(1)
    _, base = read_fastx(os.path.join(GOLDEN, "toy", "simple_query.fq"))
    seqs = [b"A", b"C", b"G", b"T", b"N", b"a", b"\x01", b"\x01A", b"A\x01", b"AC\x01GT", b"\x02", b"\xff", b"\x00",
            b"GGCAGNCGGA", b"ggcaggcgga", b"GGCAGGCGGA", b"TTCGTCGTAA", b"ACGT" * 40, b"A" * 31, b"A" * 32, b"A" * 33,
            b"A" * 64, b"A" * 65, b"AAAAAAAAAA"]
    for s in base:
        for cut in (1, 2, 5, 19, 20):
            seqs.append(s[-cut:])
            seqs.append(s[:cut])
    # random substrings of random lengths (ragged), exact and mutated
    acgt = np.frombuffer(b"ACGT", np.uint8)
    for _ in range(300):
        m = int(rng.integers(1, 200))
        q = acgt[rng.integers(0, 4, m)].tobytes()
        seqs.append(q)
    res = ix.query(seqs, RBG_LOCATE | RBG_MARKERS)
    compare_with_oracle(res, orc, seqs, True, True)
    # an empty read keeps the full range (find_range never enters its loop) -- count only, locating n rows is legal but large
    r = ix.query([b"", b"A", b""], RBG_COUNT)
    assert (int(r.lo[0]), int(r.hi[0])) == (0, orc.n - 1) and (int(r.lo[2]), int(r.hi[2])) == (0, orc.n - 1)
    ix.close()


def test_max_hits_caps_locate():
    prefix = os.path.join(GOLDEN, "toy", "small.fa")
    ix = rb.GpuIndex.open(prefix, sa=True)
    orc = O.OracleIndex.open(prefix, sa=True)
    seqs = [b"A", b"AC", b"GGCAGGCGGA", b"ACGTTTTTTTTTTTTTTTTTTT"]
    for cap in (0, 1, 3, 1000):
        r = ix.query(seqs, RBG_LOCATE, max_hits=cap)
        lo, hi, k = orc.find_ranges(seqs, toehold=True)
        for i in range(len(seqs)):
            exp = orc.locate(lo[i], hi[i], k[i], max_hits=cap)
            assert np.array_equal(r.locs[r.loc_off[i]:r.loc_off[i + 1]], exp)
    ix.close()


def test_open_arrays_equals_open_files():
    from oracle import rbformats as F
    prefix = os.path.join(GOLDEN, "tiny", "tiny")
    b, t, m = F.read_rbwt(prefix + ".rbwt"), F.read_tsa(prefix + ".tsa"), F.read_mab(prefix + ".mab")
    ix = rb.GpuIndex.from_arrays(b.n, b.heads, b.lens, tsa=(t.pred, t.samples_last, t.pred_to_run),
                                 ma=(m.starts, m.ends, m.idxs, m.arr, m.size_starts, m.size_ends, m.size_idxs))
    ix2 = rb.GpuIndex.open(prefix, sa=True, markers=True)
    _, seqs = read_fastx(os.path.join(GOLDEN, "tiny", "marked.fq"))
    a = ix.query(seqs, RBG_LOCATE | RBG_MARKERS)
    c = ix2.query(seqs, RBG_LOCATE | RBG_MARKERS)
    for f in ("lo", "hi", "toehold", "loc_off", "locs", "mk_off", "markers"):
        assert np.array_equal(getattr(a, f), getattr(c, f)), f
    ix.close(); ix2.close()


def test_modes_need_their_parts():
    ix = rb.GpuIndex.open(os.path.join(GOLDEN, "toy", "small.fa"))
    with pytest.raises(rb.RbgError):
        ix.query([b"ACGT"], RBG_LOCATE)
    with pytest.raises(rb.RbgError):
        ix.query([b"ACGT"], RBG_MARKERS)
    ix.close()


def test_unsupported_alphabet_is_an_error():
    heads = np.frombuffer(b"\x01ACGNT", np.uint8)
    lens = np.ones(6, np.uint64)
    with pytest.raises(rb.RbgError) as e:
        rb.GpuIndex.from_arrays(6, heads, lens)
    assert e.value.code == -3


@pytest.mark.parametrize("window", ["16", "24", "40", "64", "100", "256", "1000", "4096"])
@pytest.mark.parametrize("layout", ["4", "5"])
def test_results_do_not_depend_on_window_size(window, layout, monkeypatch):
    """Every window size (powers of two or not), both line layouts (leaf.cuh LeafFmt<4> / <5>); the larger windows make
    every window of this dense BWT a CLUSTER line with raw children, so both the uniform decode and the rare path are compared."""
    monkeypatch.setenv("RBG_WINDOW", window)
    monkeypatch.setenv("RBG_LAYOUT", layout)
    prefix = os.path.join(GOLDEN, "tiny", "tiny")
    ix = rb.GpuIndex.open(prefix, sa=True, markers=True)
    info = ix.info()
    assert info.window == int(window) and info.layout == int(layout)
    if int(window) >= 256:
        assert info.n_cluster > 0
    orc = O.OracleIndex.open(prefix, sa=True, markers=True)
    seqs = read_fastx(os.path.join(GOLDEN, "tiny", "noisy.fq"))[1] + read_fastx(os.path.join(GOLDEN, "tiny", "short.fq"))[1]
    compare_with_oracle(ix.query(seqs, RBG_LOCATE | RBG_MARKERS), orc, seqs, True, True)
    ix.close()


def test_staged_checksum_equals_host_digest_of_oracle_result():
    prefix = os.path.join(GOLDEN, "tiny", "tiny")
    ix = rb.GpuIndex.open(prefix, sa=True, markers=True)
    orc = O.OracleIndex.open(prefix, sa=True, markers=True)
    seqs = read_fastx(os.path.join(GOLDEN, "tiny", "exact.fq"))[1] + read_fastx(os.path.join(GOLDEN, "tiny", "marked.fq"))[1]
    lo, hi, k = orc.find_ranges(seqs, toehold=True)
    locs = [orc.locate(lo[i], hi[i], k[i]) for i in range(len(seqs))]
    mks = [orc.markers_at_range(lo[i], hi[i]) for i in range(len(seqs))]
    loc_off = np.concatenate([[0], np.cumsum([len(x) for x in locs])]).astype(np.uint64)
    mk_off = np.concatenate([[0], np.cumsum([len(x) for x in mks])]).astype(np.uint64)
    st = ix.upload(seqs)
    cs = ix.query_staged(st, RBG_LOCATE | RBG_MARKERS, checksum=True)
    assert cs == rb.result_checksum(lo, hi, k, loc_off, np.concatenate(locs), mk_off, np.concatenate(mks))
    cs2 = ix.query_staged(st, RBG_COUNT, checksum=True)
    lo2, hi2, _ = orc.find_ranges(seqs)
    assert cs2 == rb.result_checksum(lo2, hi2)
    # fetch of a staged run == direct query
    r = ix.fetch(st, RBG_COUNT)
    assert np.array_equal(r.lo, lo2) and np.array_equal(r.hi, hi2)
    st.free()
    ix.close()


# ---- FTab (include/ftab.hpp; RowBowt::build_ftab / search_ftab) ---------------------------------
FTAB_CASES = [("toy", "small.fa", 4), ("toy", "small.fa", 6), ("tiny", "tiny", 5), ("toy", "small.fa", 10),
              ("tiny", "tiny", 10), ("greedy", "ref.fa", 7)]


@pytest.mark.parametrize("d,pre,k", FTAB_CASES)
def test_gpu_ftab_file_equals_reference_rb_build(d, pre, k, tmp_path):
    """rbg_ftab_build + rbg_ftab_save == the file the unmodified `rb_build --ftab-only -k K` wrote."""
    import hashlib
    import json
    ix = rb.GpuIndex.open(os.path.join(GOLDEN, d, pre))
    ix.build_ftab(k)
    out = str(tmp_path / "x.ftab")
    ix.save_ftab(out)
    txt = open(out, "rb").read()
    name = "%s.k%d.ftab" % (d, k)
    sums = json.load(open(os.path.join(GOLDEN, "expected", "ftab_sha256.json")))
    assert hashlib.sha256(txt).hexdigest() == sums[name]["sha256"]
    path = os.path.join(GOLDEN, "expected", name)
    if os.path.exists(path):
        assert txt == open(path, "rb").read()
    # and the file loads back (every entry is verified against the index)
    ix.load_ftab(out)
    assert ix.info().ftab_k == k
    ix.close()


@pytest.mark.parametrize("name", sorted(FIXTURES))
@pytest.mark.parametrize("k", [1, 5, 10, 13])
def test_ftab_seeded_query_equals_oracle(name, k):
    """Seeding from the table changes nothing: ranges, toeholds, locations, markers (SURVEY §8c:
    'k-mer ranges equal to plain search')."""
    d, pre, fqs, has_ma = FIXTURES[name]
    prefix = os.path.join(GOLDEN, d, pre)
    ix = rb.GpuIndex.open(prefix, sa=True, markers=has_ma)
    ix.build_ftab(k)
    orc = O.OracleIndex.open(prefix, sa=True, markers=has_ma)
    seqs = []
    for fq in fqs:
        seqs += read_fastx(os.path.join(GOLDEN, d, fq))[1]
    plain_steps = None
    compare_with_oracle(ix.query(seqs, RBG_LOCATE | (RBG_MARKERS if has_ma else 0)), orc, seqs, True, has_ma)
    seeded_steps = ix.stats().lf_steps
    r = ix.query(seqs, RBG_COUNT)
    lo, hi, _ = orc.find_ranges(seqs)
    assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi)
    ix.build_ftab(0)
    ix.query(seqs, RBG_COUNT)
    plain_steps = ix.stats().lf_steps
    assert seeded_steps < plain_steps            # the table really was used
    ix.close()


def test_search_ftab_goldens_rb_tests_147_173():
    """tests/rb_tests.cpp:147-173 through rbg_ftab_lookup; a k-mer that does not occur -> (full range, 0)."""
    prefix = os.path.join(GOLDEN, "toy", "small.fa")
    ix = rb.GpuIndex.open(prefix)
    ix.build_ftab(10)
    kmers = [b"TTCGTCGTAA", b"CCGCGGACAT", b"GGCAGGCGGA", b"TATCGTGGAA", b"GGAGATATTG", b"GGCAGNCGGA"]
    lo, hi, used = ix.search_ftab(kmers)
    exp = [(28942, 28944), (10673, 10675), (19418, 19423), (24272, 24274), (19097, 19099)]
    assert list(zip(lo.tolist(), hi.tolist()))[:5] == exp and used.tolist()[:5] == [10] * 5
    n = ix.info().n
    assert (int(lo[5]), int(hi[5]), int(used[5])) == (0, n - 1, 0)
    ix.close()


def test_ftab_of_another_index_is_rejected_and_load_flag(tmp_path):
    import shutil
    toy = os.path.join(GOLDEN, "toy", "small.fa")
    tiny = os.path.join(GOLDEN, "tiny", "tiny")
    ix = rb.GpuIndex.open(tiny)
    with pytest.raises(rb.RbgError) as e:
        ix.load_ftab(os.path.join(GOLDEN, "expected", "toy.k6.ftab"))
    assert e.value.code == -2 and ix.info().ftab_k == 0
    with pytest.raises(rb.RbgError) as e:
        ix.load_ftab(str(tmp_path / "missing.ftab"))
    assert e.value.code == -1
    ix.close()
    # LoadRbwtFlag::FT: <prefix>.ftab next to the index files (include/rowbowt_io.hpp:187)
    for suf in (".rbwt", ".tsa", ".mab"):
        shutil.copy(toy + suf, str(tmp_path / ("t" + suf)))
    shutil.copy(os.path.join(GOLDEN, "expected", "toy.k6.ftab"), str(tmp_path / "t.ftab"))
    ix = rb.GpuIndex.open(str(tmp_path / "t"), sa=True, markers=True, ftab=True)
    assert ix.info().ftab_k == 6
    orc = O.OracleIndex.open(toy, sa=True, markers=True)
    seqs = read_fastx(os.path.join(GOLDEN, "toy", "simple_query.fq"))[1]
    compare_with_oracle(ix.query(seqs, RBG_LOCATE | RBG_MARKERS), orc, seqs, True, True)
    ix.close()
    with pytest.raises(rb.RbgError):
        rb.GpuIndex.open(tiny, ftab=True)           # no tiny.ftab: "bad file"


def _wide_synthetic_index(monkeypatch):
    """(GpuIndex, OracleIndex, reads) over a synthetic run sequence with n ~ 5.5*10^10 and fabricated toehold arrays."""
    from oracle import rbformats as F
    with monkeypatch.context() as mp:
        mp.setenv("RBG_PHI_SHIFT", "14")                  # 2^14-position buckets: 3 M slots instead of 400 M
        rng = np.random.default_rng(17)
        R = 200_000
        heads = np.frombuffer(b"ACGT", np.uint8)[np.cumsum(rng.integers(1, 4, R)) % 4].copy()      # adjacent runs differ
        lens = (2.0 ** rng.uniform(0, 22, R)).astype(np.uint64) + np.uint64(1)
        heads[R // 3] = 1                                      # one terminator
        lens[R // 3] = 1
        n = int(lens.sum())
        assert n > 1 << 35
        pred = np.sort(rng.choice(np.arange(0, n - 1, max(1, (n - 1) // (4 * R)), dtype=np.uint64), R - 1, replace=False))
        pred = np.concatenate([pred, [np.uint64(n - 1)]]).astype(np.uint64)      # the last text position is always sampled
        samples_last = rng.integers(0, n, R, dtype=np.uint64)
        pred_to_run = rng.integers(1, R, R, dtype=np.uint64)
        bwt = F.Rlbwt(n=n, R=R, B=2, heads=heads, lens=lens)
        tsa = F.Toehold(r=R, n=n, pred=pred, samples_last=samples_last, pred_to_run=pred_to_run)
        orc = O.OracleIndex(bwt, tsa)
        ix = rb.GpuIndex.from_arrays(n, heads, lens, tsa=(pred, samples_last, pred_to_run))
    acgt = np.frombuffer(b"ACGT", np.uint8)
    seqs = [acgt[rng.integers(0, 4, int(m))].tobytes() for m in rng.integers(1, 22, 4000)]
    seqs += [b"A", b"C", b"G", b"T", b"\x01", b"A\x01", b"N"]
    return ix, orc, seqs, n


@pytest.mark.parametrize("ftab_k", [0, 8])
def test_wide_positions_synthetic_index(ftab_k, monkeypatch):
    """Positions beyond 2^32 (BASELINE config 5 needs 38 bits; SURVEY §7 'position width'): a synthetic run
    sequence with n ~ 5.5*10^10 and fabricated toehold arrays.  find_range / LF_w_loc / phi are pure rank
    arithmetic over the arrays, so the oracle defines the answer for any such input."""
    ix, orc, seqs, n = _wide_synthetic_index(monkeypatch)
    ix.build_ftab(ftab_k)
    info = ix.info()
    assert info.n == n and info.window == 32767
    r = ix.query(seqs, RBG_LOCATE, max_hits=4)
    lo, hi, k = orc.find_ranges(seqs, toehold=True)
    assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi) and np.array_equal(r.toehold, k)
    assert int(hi.max()) > 1 << 35                         # the wide paths were exercised
    alive = int((hi >= lo).sum())
    assert alive > 500
    for i in range(len(seqs)):
        exp = orc.locate(lo[i], hi[i], k[i], max_hits=4)
        assert np.array_equal(r.locs[r.loc_off[i]:r.loc_off[i + 1]], exp), i
    ix.close()


# ---- wt_fbb indexes (`--fbb`, SURVEY 8(f) row 3) ------------------------------------------------------
FBB = os.path.join(GOLDEN, "fbb", "tiny")


@pytest.mark.parametrize("fq_dir,fq,exp_prefix", [("tiny", "exact.fq", "tiny"), ("tiny", "noisy.fq", "tiny"), ("tiny", "short.fq", "tiny"),
                                                  ("tiny", "marked.fq", "tiny"), ("fbb", "edge.fq", "fbb")])
@pytest.mark.parametrize("tag,flags", [("count", []), ("m", ["-m"])])
def test_rb_align_fbb_matches_reference_stdout(fq_dir, fq, exp_prefix, tag, flags):
    """`rb_align --fbb [-m]` over the wt_fbb index prints what the reference `rb_align --fbb` printed
    (tests/golden/make_fbb_golden.py; for the regular query files that is also what it prints without --fbb)."""
    p = subprocess.run([RB_ALIGN, "--fbb"] + flags + ["--batch", "61", FBB, os.path.join(GOLDEN, fq_dir, fq)], capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    assert p.stdout == open(os.path.join(GOLDEN, "expected", "%s.%s.%s.txt" % (exp_prefix, fq, tag)), "rb").read()


def test_fbb_index_equals_rle_index_except_for_byte_1():
    rle = rb.GpuIndex.open(os.path.join(GOLDEN, "tiny", "tiny"), markers=True)
    fbb = rb.GpuIndex.open(FBB, markers=True, fbb=True)
    a, b = rle.info(), fbb.info()
    assert (a.n, a.r, a.window, a.n_lines) == (b.n, b.r, b.window, b.n_lines)
    assert [a.F[c] for c in range(256)] == [b.F[c] for c in range(256)]
    seqs = []
    for fq in ("exact.fq", "noisy.fq", "short.fq", "marked.fq"):
        seqs += read_fastx(os.path.join(GOLDEN, "tiny", fq))[1]
    for k in (0, 10):
        rle.build_ftab(k)
        fbb.build_ftab(k)
        x, y = rle.query(seqs, RBG_MARKERS), fbb.query(seqs, RBG_MARKERS)
        assert np.array_equal(x.lo, y.lo) and np.array_equal(x.hi, y.hi)
        assert np.array_equal(x.mk_off, y.mk_off) and np.array_equal(x.markers, y.markers)
    # the terminator: byte 1 is a symbol of an rle_string index (include/rle_string.hpp:59-62) and of no wt_fbb index
    x, y = rle.query([b"\x01", b"A\x01"], RBG_COUNT), fbb.query([b"\x01", b"A\x01"], RBG_COUNT)
    assert (int(x.lo[0]), int(x.hi[0])) == (0, 0)
    assert [(int(y.lo[i]), int(y.hi[i])) for i in range(2)] == [(1, 0), (1, 0)]
    rle.close()
    fbb.close()


def test_fbb_refuses_the_toehold_sa():
    with pytest.raises(rb.RbgError):
        rb.GpuIndex.open(FBB, sa=True, fbb=True)
    p = subprocess.run([RB_ALIGN, "--fbb", "-s", FBB, os.path.join(GOLDEN, "tiny", "exact.fq")], capture_output=True)
    assert p.returncode == 1 and b"fbb" in p.stderr


@pytest.mark.parametrize("chunks,est", [("1", None), ("7", None), ("7", "1"), ("16", "37"), ("64", "1")])
def test_pipelined_locate_output_with_regrowth(chunks, est, monkeypatch):
    """rbg_query streams the locations out chunk by chunk (device-continued scan, buffers sized from the first
    chunks): same arrays for any chunking, also when every chunk has to grow the buffers (RBG_LOC_EST forces a
    hopeless first guess) -- on fresh and on reused scratch buffers."""
    monkeypatch.setenv("RBG_CHUNKS", chunks)
    if est:
        monkeypatch.setenv("RBG_LOC_EST", est)
    prefix = os.path.join(GOLDEN, "tiny", "tiny")
    ix = rb.GpuIndex.open(prefix, sa=True, markers=True)
    orc = O.OracleIndex.open(prefix, sa=True, markers=True)
    seqs = []
    for fq in ("exact.fq", "noisy.fq", "short.fq", "marked.fq"):
        seqs += read_fastx(os.path.join(GOLDEN, "tiny", fq))[1]
    seqs += [b"A", b"", b"ACGT", b"N"] * 3
    for rep in range(2):
        compare_with_oracle(ix.query(seqs, RBG_LOCATE | RBG_MARKERS), orc, seqs, True, True)
        r = ix.query(seqs[:5], RBG_LOCATE, max_hits=2)
        assert np.all(np.diff(r.loc_off) <= 2)
    r = ix.query([], RBG_LOCATE)
    assert r.n == 0 and len(r.locs) == 0
    ix.close()
