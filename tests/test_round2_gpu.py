"""Round-2 additions to the C ABI, through the C ABI (-m gpu): narrow locations, 2-bit packed batches packed on
the host, concurrent calls on one handle, the host binary's multi-worker path."""
import os
import subprocess
import threading

import numpy as np
import pytest

from conftest import FIXTURES, GOLDEN, ROOT, fixture_cases, read_fastx
from oracle import oracle as O

import rowbowt_b200 as rb
from rowbowt_b200 import RBG_COUNT, RBG_LOCATE, RBG_MARKERS, RBG_NARROW_LOCS, RBG_NARROW_RANGES, RBG_READ_DEAD, RBG_READ_EXOTIC

pytestmark = pytest.mark.gpu
RB_ALIGN = os.path.join(ROOT, "rowbowt_b200", "rb_align")

EDGE = [b"A", b"C", b"G", b"T", b"N", b"a", b"\x01", b"\x01A", b"A\x01", b"AC\x01GT", b"\x02", b"\xff", b"\x00", b"",
        b"GGCAGNCGGA", b"ggcaggcgga", b"GGCAGGCGGA", b"TTCGTCGTAA", b"ACGT" * 40, b"A" * 31, b"A" * 32, b"A" * 33,
        b"A" * 64, b"A" * 65, b"AAAAAAAAAA", b"", b"T"]


def _fixture_reads(name):
    d, pre, fqs, has_ma = FIXTURES[name]
    seqs = []
    for fq in fqs:
        seqs += read_fastx(os.path.join(GOLDEN, d, fq))[1]
    return os.path.join(GOLDEN, d, pre), seqs, has_ma


def _same(a, b, mode):
    assert np.array_equal(a.lo, b.lo) and np.array_equal(a.hi, b.hi)
    if mode & RBG_LOCATE:
        assert np.array_equal(a.toehold, b.toehold) and np.array_equal(a.loc_off, b.loc_off) and np.array_equal(a.locs, b.locs)
    if mode & RBG_MARKERS:
        assert np.array_equal(a.mk_off, b.mk_off) and np.array_equal(a.markers, b.markers)


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_narrow_locations_equal_wide(name, monkeypatch):
    prefix, seqs, has_ma = _fixture_reads(name)
    ix = rb.GpuIndex.open(prefix, sa=True, markers=has_ma)
    mode = RBG_LOCATE | (RBG_MARKERS if has_ma else 0)
    wide = ix.query(seqs, mode)
    narrow = ix.query(seqs, mode | RBG_NARROW_LOCS)
    assert narrow.narrow_bytes == 4                  # n < 2^32: no high plane
    _same(wide, narrow, mode)
    monkeypatch.setenv("RBG_LOC_EST", "1")           # force the location buffers to regrow chunk after chunk
    monkeypatch.setenv("RBG_CHUNKS", "5")
    _same(wide, ix.query(seqs, mode | RBG_NARROW_LOCS), mode)
    # staged (device-resident) form: same digest, same fetched arrays
    st = ix.upload(seqs)
    cs_wide = ix.query_staged(st, mode, checksum=True)
    cs_narrow = ix.query_staged(st, mode | RBG_NARROW_LOCS, checksum=True)
    assert cs_wide == cs_narrow
    _same(wide, ix.fetch(st, mode | RBG_NARROW_LOCS), mode)
    st.free()
    ix.close()


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_narrow_ranges_equal_wide(name, monkeypatch):
    """RBG_NARROW_RANGES: lo / hi as u32 planes on the wire (n <= 2^32) -- same values, empty ranges still (1,0), with every
    other mode bit, raw and packed input, one chunk and several."""
    prefix, seqs, has_ma = _fixture_reads(name)
    seqs = seqs + [b"N", b"A" * 40, b"ACGTN" * 9]
    ix = rb.GpuIndex.open(prefix, sa=True, markers=has_ma)
    for mode in (RBG_COUNT, RBG_LOCATE | RBG_NARROW_LOCS | (RBG_MARKERS if has_ma else 0), RBG_LOCATE):
        wide = ix.query(seqs, mode)
        assert not wide.narrow_ranges
        for chunks in ("1", "4"):
            monkeypatch.setenv("RBG_CHUNKS", chunks)
            for r in (ix.query(seqs, mode | RBG_NARROW_RANGES), ix.query_packed(seqs, mode | RBG_NARROW_RANGES, threads=2)):
                assert r.narrow_ranges
                _same(wide, r, mode)
        monkeypatch.delenv("RBG_CHUNKS")
    assert int((wide.hi < wide.lo).sum()) >= 2            # the dead reads came back as (1,0)
    ix.close()


@pytest.mark.parametrize("threads", [1, 3])
@pytest.mark.parametrize("ftab_k", [0, 5])
def test_packed_batch_equals_raw_batch(threads, ftab_k, monkeypatch):
    """rbg_pack_bytes + rbg_query_packed == rbg_query on the raw bytes, dead (N, lowercase, 0xff) and exotic
    (terminator byte) reads included, whole-batch and chunked."""
    prefix = os.path.join(GOLDEN, "toy", "small.fa")
    ix = rb.GpuIndex.open(prefix, sa=True, markers=True)
    ix.build_ftab(ftab_k)
    orc = O.OracleIndex.open(prefix, sa=True, markers=True)
    rng = np.random.default_rng(7)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    seqs = list(EDGE) + read_fastx(os.path.join(GOLDEN, "toy", "simple_query.fq"))[1]
    for _ in range(400):
        seqs.append(acgt[rng.integers(0, 4, int(rng.integers(1, 200)))].tobytes())
    full = [s for s in seqs if len(s)]               # locating the full range of an empty read is legal but huge
    mode = RBG_LOCATE | RBG_MARKERS | RBG_NARROW_LOCS
    raw = ix.query(full, mode)
    pb, keep = ix.pack(full, threads)
    flags = keep[1][:len(full)]
    assert pb.n_exotic == sum(1 for s in full if b"\x01" in s)
    for i, s in enumerate(full):
        dead = any(c not in b"ACGT\x01" for c in s)
        assert bool(flags[i] & RBG_READ_DEAD) == dead and bool(flags[i] & RBG_READ_EXOTIC) == (b"\x01" in s), (i, s)
    _same(raw, ix.query_packed(full, mode, threads=threads), mode)
    monkeypatch.setenv("RBG_CHUNKS", "7")
    _same(raw, ix.query_packed(full, mode, threads=threads), mode)
    monkeypatch.delenv("RBG_CHUNKS")
    # against the oracle, count-only, empty reads included
    r = ix.query_packed(seqs, RBG_COUNT, threads=threads)
    lo, hi, _ = orc.find_ranges(seqs)
    assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi)
    # staged form
    st = ix.upload_packed(full, threads)
    assert ix.query_staged(st, mode, checksum=True) == rb.result_checksum(raw.lo, raw.hi, raw.toehold, raw.loc_off, raw.locs, raw.mk_off, raw.markers)
    st.free()
    # an empty packed batch
    r = ix.query_packed([], RBG_LOCATE | RBG_MARKERS)
    assert r.n == 0 and len(r.locs) == 0
    ix.close()


def test_packed_batch_argument_errors():
    prefix = os.path.join(GOLDEN, "toy", "small.fa")
    ix = rb.GpuIndex.open(prefix)
    import ctypes as C
    pb, keep = ix.pack([b"ACGT", b"A\x01"])
    assert pb.n_exotic == 1
    pb.bases = None                                  # exotic reads without their bytes
    res = rb.binding._Result()
    assert rb.lib().rbg_query_packed(ix.h, C.byref(pb), 0, 1, C.byref(res)) == -5
    offs = keep[3] + np.uint64(3)
    pb2 = rb.binding._PackedBatch(2, keep[0].ctypes.data, offs.ctypes.data, None, 0, None)
    assert rb.lib().rbg_query_packed(ix.h, C.byref(pb2), 0, 1, C.byref(res)) == -5      # offsets[0] != 0
    ix.close()


def test_concurrent_calls_on_one_handle():
    """Two host threads interleave -s and count batches on ONE handle (the reference shares one const RowBowt&
    among its workers, src/rb_markers.cpp:321-326): every result equals the oracle's."""
    prefix, seqs, _ = _fixture_reads("tiny")
    ix = rb.GpuIndex.open(prefix, sa=True, markers=True)
    ix.build_ftab(4)
    orc = O.OracleIndex.open(prefix, sa=True, markers=True)
    lo, hi, k = orc.find_ranges(seqs, toehold=True)
    locs = [orc.locate(lo[i], hi[i], k[i]) for i in range(len(seqs))]
    errors = []

    def worker(tid):
        try:
            rng = np.random.default_rng(tid)
            for it in range(40):
                sel = rng.permutation(len(seqs))[: int(rng.integers(1, len(seqs)))]
                batch = [seqs[i] for i in sel]
                if (it + tid) % 2:
                    r = ix.query(batch, RBG_LOCATE | RBG_MARKERS | (RBG_NARROW_LOCS if it % 4 < 2 else 0))
                    assert np.array_equal(r.toehold, k[sel])
                    for j, i in enumerate(sel):
                        assert np.array_equal(r.locs[r.loc_off[j]:r.loc_off[j + 1]], locs[i])
                else:
                    r = ix.query_packed(batch, RBG_COUNT) if it % 3 == 0 else ix.query(batch, RBG_COUNT)
                assert np.array_equal(r.lo, lo[sel]) and np.array_equal(r.hi, hi[sel])
        except Exception as e:            # noqa: BLE001
            errors.append((tid, repr(e)))

    th = [threading.Thread(target=worker, args=(t,)) for t in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors
    ix.close()


@pytest.mark.parametrize("d,pre,fq,tag,sa,ma", list(fixture_cases()))
@pytest.mark.parametrize("host_pack", ["1", "0"])
def test_rb_align_three_workers_ordered_reassembly(d, pre, fq, tag, sa, ma, host_pack):
    """rb_align --gpus 3 with tiny parser chunks: three GPU workers (mapped onto the visible devices modulo their
    number, RBG_GPU_MODULO) feed the formatter pool and the ordered writer; stdout must still be the reference's."""
    env = dict(os.environ, RBG_GPU_MODULO="1", RBG_HOST_PACK=host_pack)
    cmd = [RB_ALIGN] + (["-s"] if sa else []) + (["-m"] if ma else []) + ["--gpus", "3", "--threads", "4", "--chunk-bytes", "2000",
                                                                          os.path.join(GOLDEN, d, pre), os.path.join(GOLDEN, d, fq)]
    p = subprocess.run(cmd, capture_output=True, env=env)
    assert p.returncode == 0, p.stderr.decode()
    assert p.stdout == open(os.path.join(GOLDEN, "expected", "%s.%s.%s.txt" % (d, fq, tag)), "rb").read()


@pytest.mark.parametrize("d,pre,fq,tag,sa,ma", list(fixture_cases()))
def test_rb_align_stdout_to_a_file_is_the_same_report(d, pre, fq, tag, sa, ma, tmp_path):
    """stdout redirected to a regular file takes the positional writer (slices pwritten concurrently at their offsets):
    from offset 0, behind bytes already in the file, and -- opened O_APPEND, where pwrite ignores offsets -- the
    sequential writer; the file must hold exactly the reference's report every time."""
    want = open(os.path.join(GOLDEN, "expected", "%s.%s.%s.txt" % (d, fq, tag)), "rb").read()
    cmd = [RB_ALIGN] + (["-s"] if sa else []) + (["-m"] if ma else []) + ["--threads", "4", "--chunk-bytes", "1500",
                                                                          os.path.join(GOLDEN, d, pre), os.path.join(GOLDEN, d, fq)]
    out = str(tmp_path / "report.txt")
    with open(out, "wb") as f:
        assert subprocess.run(cmd, stdout=f, stderr=subprocess.PIPE).returncode == 0
    assert open(out, "rb").read() == want
    fd = os.open(out, os.O_WRONLY | os.O_CREAT | os.O_TRUNC)
    os.write(fd, b"header line\n")
    assert subprocess.run(cmd, stdout=fd, stderr=subprocess.PIPE).returncode == 0
    os.write(fd, b"trailer\n")                        # the shared file position was left behind the report
    os.close(fd)
    assert open(out, "rb").read() == b"header line\n" + want + b"trailer\n"
    with open(out, "ab") as f:
        assert subprocess.run(cmd, stdout=f, stderr=subprocess.PIPE).returncode == 0
    assert open(out, "rb").read() == b"header line\n" + want + b"trailer\n" + want


def test_wide_index_narrow_locations_have_a_high_plane(monkeypatch):
    """An index with n > 2^32 (fabricated arrays as in test_wide_positions_synthetic_index): 5-byte locations."""
    from test_gpu_parity import _wide_synthetic_index
    ix, orc, seqs, n = _wide_synthetic_index(monkeypatch)
    wide = ix.query(seqs, RBG_LOCATE, max_hits=6)
    narrow = ix.query(seqs, RBG_LOCATE | RBG_NARROW_LOCS, max_hits=6)
    assert narrow.narrow_bytes == 5
    _same(wide, narrow, RBG_LOCATE)
    assert wide.locs.max() >> 32
    r = ix.query(seqs, RBG_LOCATE | RBG_NARROW_RANGES, max_hits=6)       # n > 2^32: the bit is ignored, ranges stay u64
    assert not r.narrow_ranges
    _same(wide, r, RBG_LOCATE)
    ix.close()


def _copy_index(prefix, dst_dir):
    import glob
    import shutil
    out = os.path.join(str(dst_dir), os.path.basename(prefix))
    for f in glob.glob(prefix + ".*"):                       # .rbwt / .tsa / .mab / .docs / .ftab ...
        if os.path.isfile(f) and not f.endswith(".rbgcache"):
            shutil.copy(f, out + f[len(prefix):])
    return out


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_layout_cache_opens_the_same_index(name, tmp_path, monkeypatch):
    """RBG_LOAD_CACHE: the first open writes <prefix>.rbgcache, the second uploads it as it is (info.from_cache) and
    answers every query like an index decoded from the files; other load flags, touched index files, a truncated cache or
    other layout knobs are not served from it."""
    src, seqs, has_ma = _fixture_reads(name)
    prefix = _copy_index(src, tmp_path)
    seqs = seqs + EDGE
    mode = RBG_LOCATE | (RBG_MARKERS if has_ma else 0)
    plain = rb.GpuIndex.open(prefix, sa=True, markers=has_ma)
    want, want_info = plain.query(seqs, mode), plain.info()
    plain.close()
    assert not os.path.exists(prefix + ".rbgcache")          # not asked for: nothing written
    first = rb.GpuIndex.open(prefix, sa=True, markers=has_ma, cache=True)
    assert first.info().from_cache == 0 and os.path.exists(prefix + ".rbgcache")
    _same(want, first.query(seqs, mode), mode)
    first.close()
    second = rb.GpuIndex.open(prefix, sa=True, markers=has_ma, cache=True)
    info = second.info()
    assert info.from_cache == 1
    for f in ("n", "r", "window", "n_lines", "n_cluster", "dir_bytes", "phi_bytes", "toehold_bytes", "marker_bytes", "layout",
              "phi_shift", "phi_overflow", "has_sa", "has_ma", "toehold0", "wsize"):
        assert getattr(info, f) == getattr(want_info, f), f
    assert list(info.F) == list(want_info.F)
    _same(want, second.query(seqs, mode), mode)
    second.build_ftab(5)                                      # the seed table is rebuilt on top of a cached layout
    _same(want, second.query_packed(seqs, mode | RBG_NARROW_LOCS, threads=2), mode)
    second.close()
    # other load flags: a different cache (rewritten), still the right answers
    count_only = rb.GpuIndex.open(prefix, cache=True)
    assert count_only.info().from_cache == 0 and count_only.info().has_sa == 0
    c = count_only.query(seqs, RBG_COUNT)
    assert np.array_equal(c.lo, want.lo) and np.array_equal(c.hi, want.hi)
    count_only.close()
    again = rb.GpuIndex.open(prefix, cache=True)
    assert again.info().from_cache == 1
    again.close()
    # an index file that changed (mtime) invalidates the cache
    os.utime(prefix + ".rbwt", ns=(1, 1))
    stale = rb.GpuIndex.open(prefix, cache=True)
    assert stale.info().from_cache == 0
    stale.close()
    # a truncated cache file is rebuilt, not trusted
    size = os.path.getsize(prefix + ".rbgcache")
    with open(prefix + ".rbgcache", "r+b") as f:
        f.truncate(size // 2)
    trunc = rb.GpuIndex.open(prefix, cache=True)
    assert trunc.info().from_cache == 0
    c = trunc.query(seqs, RBG_COUNT)
    assert np.array_equal(c.lo, want.lo) and np.array_equal(c.hi, want.hi)
    trunc.close()
    assert os.path.getsize(prefix + ".rbgcache") == size
    # other layout knobs: not this cache
    monkeypatch.setenv("RBG_LAYOUT", "4")
    other = rb.GpuIndex.open(prefix, cache=True)
    assert other.info().from_cache == 0 and other.info().layout == 4
    c = other.query(seqs, RBG_COUNT)
    assert np.array_equal(c.lo, want.lo) and np.array_equal(c.hi, want.hi)
    other.close()


def test_layout_cache_concurrent_first_opens(tmp_path):
    """Several handles of one prefix opened at the same time with RBG_LOAD_CACHE (rb_align --gpus N does that): every open
    succeeds, the cache file that remains is whole, the next open is served from it."""
    src, seqs, has_ma = _fixture_reads("tiny")
    prefix = _copy_index(src, tmp_path)
    handles, errors = [None] * 4, []

    def work(i):
        try:
            handles[i] = rb.GpuIndex.open(prefix, sa=True, markers=has_ma, cache=True)
        except Exception as e:                                   # noqa: BLE001
            errors.append(repr(e))
    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors
    want = handles[0].query(seqs, RBG_LOCATE)
    for h in handles[1:]:
        _same(want, h.query(seqs, RBG_LOCATE), RBG_LOCATE)
    for h in handles:
        h.close()
    assert not [f for f in os.listdir(str(tmp_path)) if ".tmp." in f]
    again = rb.GpuIndex.open(prefix, sa=True, markers=has_ma, cache=True)
    assert again.info().from_cache == 1
    _same(want, again.query(seqs, RBG_LOCATE), RBG_LOCATE)
    again.close()


def test_rb_align_layout_cache_same_stdout(tmp_path):
    """rb_align --layout-cache: the run that writes the cache and the run that opens from it print the reference's report."""
    d, pre, fq, tag, sa, ma = [c.values for c in fixture_cases() if c.values[4] and c.values[5]][0]
    prefix = _copy_index(os.path.join(GOLDEN, d, pre), tmp_path)
    want = open(os.path.join(GOLDEN, "expected", "%s.%s.%s.txt" % (d, fq, tag)), "rb").read()
    cmd = [RB_ALIGN, "-s", "-m", "--layout-cache", "--threads", "2", prefix, os.path.join(GOLDEN, d, fq)]
    for _ in range(2):
        p = subprocess.run(cmd, capture_output=True)
        assert p.returncode == 0, p.stderr.decode()
        assert p.stdout == want
    assert os.path.exists(prefix + ".rbgcache")


def test_chunk_boundary_words_survive_any_stream_order(monkeypatch):
    """rbg_query packs raw bytes chunk by chunk on two alternating streams, and the 2-bit word a chunk boundary falls into is
    written by both neighbours (incomplete by the earlier one).  RBG_TEST_STALL holds the even chunks' stream back in front
    of their pack and the odd chunks' stream between pack and search -- the order in which an unordered earlier pack would
    land on top of the complete word before the later chunk reads it.  Results must not depend on it."""
    prefix, seqs, has_ma = _fixture_reads("tiny")
    seqs = [s[:75 + (i % 9)] for i, s in enumerate(seqs) if len(s) >= 90][:400]        # lengths that are no multiple of 32 bases
    ix = rb.GpuIndex.open(prefix, sa=True, markers=has_ma)
    mode = RBG_LOCATE | (RBG_MARKERS if has_ma else 0)
    monkeypatch.setenv("RBG_CHUNKS", "1")
    want = ix.query(seqs, mode)
    orc = O.OracleIndex.open(prefix, sa=True, markers=has_ma)
    lo, hi, k = orc.find_ranges(seqs, toehold=True)
    assert np.array_equal(want.lo, lo) and np.array_equal(want.hi, hi) and np.array_equal(want.toehold, k)
    assert int((hi >= lo).sum()) > 100
    monkeypatch.setenv("RBG_CHUNKS", "16")
    for stall in ("0,0", "2000,4000", "4000,0", "0,3000"):
        monkeypatch.setenv("RBG_TEST_STALL", stall)
        for _ in range(2):
            _same(want, ix.query(seqs, mode), mode)
            _same(want, ix.query(seqs, mode | RBG_NARROW_RANGES | RBG_NARROW_LOCS), mode)
    ix.close()
