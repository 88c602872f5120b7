"""Full-size parity through size-independent properties (run with -m gpu on the B200 box).

At BASELINE sizes (data/c2: 50 Mbp x 64 haplotypes, millions of 150 bp reads) the oracle is too slow to
be the checker, so the GPU result is checked against facts that follow from how the synthetic panel was
made (tools/synth.py), independently of any BWT code:
  * an exact read drawn from sequence h at offset s occurs exactly in the sequences that carry the same
    alleles as h at the panel sites inside [s, s+150) -- so count == |that set| (a 150-mer of a uniform
    random reference does not repeat by chance), and
  * the locations reported by -s are exactly {h' * (L+10) + s} over that set (text layout: every
    sequence is followed by 10 'A's, pfbwt-f README "padding"), each with the right haplotype, and
  * markers reported by -m are words of the panel sites within wsize of the read start (allele of h').
Plus: a sample of the batch bit-exact against the oracle; seed table on/off and 1 vs N chunks give the
same device digest.  Falls back to the `small` index when data/c2 has not been built: data/small when present,
else built once per session without the reference (conftest.small_index).
"""
import os

import numpy as np
import pytest

from conftest import ROOT

import rowbowt_b200 as rb
from rowbowt_b200 import RBG_COUNT, RBG_LOCATE, RBG_MARKERS
from tools import synth

pytestmark = pytest.mark.gpu
READ_LEN = 150


def _workloads():
    """The BASELINE index (c2; data/small when it has not been built) and, when present, the config-5 family index c5w
    (1.75 Mbp x 2504 haplotypes: n = 4.38e9 > 2^32 rows, 5-byte locations, up to 2505 occurrences per read -- the member of
    the family that fits beside c2 in the snapshot the GPU box receives).  RBG_TEST_CONFIG / RBG_TEST_READS select one
    explicitly (c5s, c5m: builder-box runs)."""
    if os.environ.get("RBG_TEST_CONFIG"):
        return [(os.environ["RBG_TEST_CONFIG"], int(os.environ.get("RBG_TEST_READS", "1000000")))]
    have = lambda cfg: os.path.exists(os.path.join(ROOT, "data", cfg, cfg + ".rbwt"))
    out = [("c2", 2_000_000)] if have("c2") else [("small", 500_000)]
    if have("c5w"):
        out.append(("c5w", 100_000))
    return out


def _carriers(panel, hs, starts):
    """bool[n_reads, nseq]: sequence h' spells the same 150-mer as the read's source sequence."""
    gt = np.vstack([np.zeros((1, len(panel.sites)), bool), panel.gt])          # row 0 = the reference
    first = np.searchsorted(panel.sites, starts)
    last = np.searchsorted(panel.sites, starts + READ_LEN)
    same = np.ones((len(hs), panel.nseq), bool)
    k = 0
    while True:
        m = first + k < last
        if not m.any():
            break
        rows = np.nonzero(m)[0]
        si = first[rows] + k
        same[rows] &= gt[:, si].T == gt[hs[rows], si][:, None]
        k += 1
    return same


@pytest.fixture(scope="module", params=_workloads(), ids=lambda w: w[0])
def full(request):
    cfg, n_reads = request.param
    prefix = os.path.join(ROOT, "data", cfg, cfg) if cfg != "small" else request.getfixturevalue("small_index")
    L, H = synth.CONFIGS[cfg]
    panel = synth.make_panel(L, H)
    reads, hs, starts = synth.make_reads(panel, n_reads, READ_LEN, seed=3)
    has_sa, has_ma = os.path.exists(prefix + ".tsa"), os.path.exists(prefix + ".mab")
    ix = rb.GpuIndex.open(prefix, sa=has_sa, markers=has_ma)
    yield dict(cfg=cfg, prefix=prefix, panel=panel, reads=reads, hs=hs, starts=starts, ix=ix, sa=has_sa, ma=has_ma)
    ix.close()


def test_counts_equal_number_of_carrier_sequences(full):
    ix, panel = full["ix"], full["panel"]
    same = _carriers(panel, full["hs"], full["starts"])
    r = ix.query(full["reads"], RBG_COUNT)
    assert np.all(r.hi >= r.lo)
    assert np.array_equal((r.hi - r.lo + np.uint64(1)).astype(np.int64), same.sum(axis=1))
    st = ix.stats()
    assert st.lf_steps == len(full["reads"]) * READ_LEN          # exact reads never stop early (no seed table yet)


def test_seed_table_and_chunking_do_not_change_the_digest(full, monkeypatch):
    ix = full["ix"]
    mode = (RBG_LOCATE if full["sa"] else 0) | (RBG_MARKERS if full["ma"] else 0)
    staged = ix.upload(full["reads"])
    ix.build_ftab(0)
    plain = ix.query_staged(staged, mode, checksum=True)
    steps_plain = ix.stats().lf_steps
    for k in (10, 12):
        ix.build_ftab(k)
        assert ix.query_staged(staged, mode, checksum=True) == plain
        assert ix.stats().lf_steps == steps_plain - len(full["reads"]) * k
    # the pipelined host-buffer call (16 chunks) returns the same arrays as the staged one
    a = ix.query(full["reads"][:300_000], RBG_COUNT)
    monkeypatch.setenv("RBG_CHUNKS", "1")
    b = ix.query(full["reads"][:300_000], RBG_COUNT)
    assert np.array_equal(a.lo, b.lo) and np.array_equal(a.hi, b.hi)
    assert rb.result_checksum(a.lo, a.hi) == ix.query_staged(ix.upload(full["reads"][:300_000]), RBG_COUNT, checksum=True)
    staged.free()
    ix.build_ftab(0)


def test_locations_are_exactly_the_carrier_copies(full):
    if not full["sa"]:
        pytest.skip("index without .tsa")
    ix, panel = full["ix"], full["panel"]
    m = min(len(full["reads"]), 400_000 if panel.nseq < 1000 else 20_000)         # c5w: ~2000 locations per read
    reads, hs, starts = full["reads"][:m], full["hs"][:m], full["starts"][:m]
    same = _carriers(panel, hs, starts)
    ix.build_ftab(10)
    r = ix.query(reads, RBG_LOCATE)
    ix.build_ftab(0)
    cnt = np.diff(r.loc_off).astype(np.int64)
    assert np.array_equal(cnt, same.sum(axis=1))
    owner = np.repeat(np.arange(m), cnt)
    seq = (r.locs // np.uint64(panel.L + synth.PAD)).astype(np.int64)
    off = (r.locs % np.uint64(panel.L + synth.PAD)).astype(np.int64)
    assert np.array_equal(off, starts[owner])                      # every copy at the read's own offset
    assert np.all(same[owner, seq])                                # ... in a sequence that carries the same alleles
    key = owner * panel.nseq + seq                                 # ... each such sequence exactly once
    assert len(np.unique(key)) == len(key)
    assert np.array_equal(r.locs[r.loc_off[:-1][cnt > 0].astype(np.int64)], r.toehold[cnt > 0])   # first location = SA[hi]


def test_markers_are_panel_sites_near_the_read_start(full):
    if not full["ma"]:
        pytest.skip("index without .mab")
    ix, panel = full["ix"], full["panel"]
    m = min(len(full["reads"]), 1_000_000)
    starts, hs = full["starts"][:m], full["hs"][:m]
    r = ix.query(full["reads"][:m], RBG_MARKERS)
    cnt = np.diff(r.mk_off).astype(np.int64)
    assert cnt.sum() > 0
    owner = np.repeat(np.arange(m), cnt)
    pos = (r.markers & np.uint64(0x00000FFFFFFFFFFF)).astype(np.int64)          # MarkerT pos, pfbwt-f/include/marker.hpp:11
    allele = (r.markers >> np.uint64(60)).astype(np.int64)
    # the site is a panel site at or after the read start, within the marker window (wsize = 10)
    si = np.searchsorted(panel.sites, pos)
    assert np.all(panel.sites[np.minimum(si, len(panel.sites) - 1)] == pos)
    d = pos - starts[owner]
    assert np.all((d >= 0) & (d < 10))
    # its allele is one that a carrier of the read has at that site; all carriers agree inside the read
    gt = np.vstack([np.zeros((1, len(panel.sites)), bool), panel.gt])
    assert np.array_equal(allele, gt[hs[owner], si].astype(np.int64))
    # reads with a site in their first wsize bases do report it
    nxt = np.searchsorted(panel.sites, starts)
    near = (nxt < len(panel.sites)) & (panel.sites[np.minimum(nxt, len(panel.sites) - 1)] - starts < 10)
    assert np.all(cnt[near] > 0)


def test_sample_bit_exact_against_oracle(full):
    """300 exact + 300 noisy reads (1 % substitutions, 0.1 % N: early exits, dead reads) bit-exact against the oracle.
    For c2 the oracle's answers were computed in the build container and committed (tools/make_fullsize_oracle.py ->
    tests/golden/expected/c2.oracle.npz: loading that index into the numpy readers takes minutes); other configs
    run the oracle live."""
    import json
    from conftest import GOLDEN
    from rowbowt_b200 import RBG_NARROW_LOCS
    sizes = synth.parity_sample_sizes(full["panel"].nseq)
    seqs = [bytes(x) for x in full["reads"][:sizes["exact"]]]
    noisy, _, _ = synth.make_reads(full["panel"], sizes["noisy"], READ_LEN, seed=5, err_rate=0.01, n_rate=0.001)
    seqs += [bytes(x) for x in noisy]
    mode = (RBG_LOCATE if full["sa"] else 0) | (RBG_MARKERS if full["ma"] else 0)
    cache = os.path.join(GOLDEN, "expected", "%s.oracle.npz" % full["cfg"])
    meta = os.path.join(GOLDEN, "expected", "%s.oracle.json" % full["cfg"])
    have = json.load(open(meta)) if os.path.exists(cache) else {}
    if have.get("n_reads") == len(full["reads"]) and have.get("has_sa") == full["sa"] and have.get("has_ma") == full["ma"]:
        z = np.load(cache)
        lo, hi, k = z["lo"], z["hi"], z["k"]
        locate = lambda i: z["locs"][int(z["loc_off"][i]):int(z["loc_off"][i + 1])]
        markers_of = lambda i: z["markers"][int(z["mk_off"][i]):int(z["mk_off"][i + 1])]
    else:
        from oracle import oracle as O
        orc = O.OracleIndex.open(full["prefix"], sa=full["sa"], markers=full["ma"])
        lo, hi, k = orc.find_ranges(seqs, toehold=full["sa"])
        locate = lambda i: orc.locate(lo[i], hi[i], k[i])
        markers_of = lambda i: orc.markers_at_range(lo[i], hi[i])
    assert int((hi < lo).sum()) > sizes["noisy"] // 3  # the noisy half really exercises the early exit
    for ftab_k in (0, 10):
        full["ix"].build_ftab(ftab_k)
        for m in (mode, mode | RBG_NARROW_LOCS) if full["sa"] else (mode,):
            for r in (full["ix"].query(seqs, m), full["ix"].query_packed(seqs, m, threads=2)):
                assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi)
                if full["sa"]:
                    assert np.array_equal(r.toehold, k)
                for i in range(len(seqs)):
                    if full["sa"]:
                        assert np.array_equal(r.locs[r.loc_off[i]:r.loc_off[i + 1]], locate(i)), i
                    if full["ma"]:
                        assert np.array_equal(r.markers[r.mk_off[i]:r.mk_off[i + 1]], markers_of(i)), i
    full["ix"].build_ftab(0)


def test_binary_stdout_equals_committed_reference_sample(full, tmp_path):
    """tests/golden/expected/<cfg>.sample.<tag>.txt holds what the UNMODIFIED reference rb_align printed, in the build
    container, for the first 600 reads (120 with -s) of this workload (tools/make_fullsize_sample.py): the host binary must print
    the same bytes from the same index on the GPU box."""
    import json
    import subprocess
    from conftest import GOLDEN
    meta = os.path.join(GOLDEN, "expected", "%s.sample.json" % full["cfg"])
    if not os.path.exists(meta) or json.load(open(meta))["n_reads"] != len(full["reads"]):
        pytest.skip("no committed reference sample for %s at this batch size" % full["cfg"])
    ran = 0
    sizes = synth.parity_sample_sizes(full["panel"].nseq)               # as tools/make_fullsize_sample.py
    for tag, flags, need, k in (("count", [], True, sizes["count"]), ("s", ["-s"], full["sa"], sizes["s"]), ("m", ["-m"], full["ma"], sizes["m"])):
        exp = os.path.join(GOLDEN, "expected", "%s.sample.%s.txt" % (full["cfg"], tag))
        if not need or not os.path.exists(exp):
            continue
        fq = str(tmp_path / ("sample_%s.fq" % tag))
        synth.write_fastq(full["reads"][:k], fq)
        p = subprocess.run([os.path.join(ROOT, "rowbowt_b200", "rb_align")] + flags + [full["prefix"], fq], capture_output=True)
        assert p.returncode == 0, p.stderr.decode()
        assert p.stdout == open(exp, "rb").read(), tag
        ran += 1
    if not ran:
        pytest.skip("no committed reference sample for %s" % full["cfg"])


def test_binary_stdout_on_noisy_reads_equals_reference(full, tmp_path):
    """The second read set of SURVEY 8(d) -- 1 % substitutions, 0.1 % N (seed 5) -- through the host binary, every flag
    set, against what the UNMODIFIED reference printed for the same 600 reads (tools/make_fullsize_oracle.py)."""
    import subprocess
    from conftest import GOLDEN
    noisy = synth.make_reads(full["panel"], synth.parity_sample_sizes(full["panel"].nseq)["noisy_text"], READ_LEN, seed=5, err_rate=0.01, n_rate=0.001)[0]
    fq = str(tmp_path / "noisy.fq")
    synth.write_fastq(noisy, fq)
    ran = 0
    for tag, flags, need in (("count", [], True), ("s", ["-s"], full["sa"]), ("m", ["-m"], full["ma"]), ("sm", ["-s", "-m"], full["sa"] and full["ma"])):
        exp = os.path.join(GOLDEN, "expected", "%s.noisy.%s.txt" % (full["cfg"], tag))
        if not need or not os.path.exists(exp):
            continue
        for extra in ([], ["--threads", "3", "--chunk-bytes", "30000"]):
            p = subprocess.run([os.path.join(ROOT, "rowbowt_b200", "rb_align")] + flags + extra + [full["prefix"], fq], capture_output=True)
            assert p.returncode == 0, p.stderr.decode()
            assert p.stdout == open(exp, "rb").read(), (tag, extra)
        ran += 1
    if not ran:
        pytest.skip("no committed noisy reference sample for %s" % full["cfg"])


def test_device_layout_walked_on_the_host(full):
    """The host-side self-checks (csrc/selftest.cpp: the SAME decode code the kernels run, over the SAME layout the
    index open builds) at full size: rank_c at every 61st position of every run plus the run boundaries against the flat
    runs (all CLUSTER windows, their RAW children and the TERM window included), the toehold sample of EVERY run
    end's LF image, phi at every 53rd text position plus the neighbours of every sample against the flat arrays."""
    import ctypes as C
    lib, pre = rb.lib(), full["prefix"].encode()
    chk, nl, nc = C.c_uint64(), C.c_uint64(), C.c_uint64()
    assert lib.rbg_selftest_layout(pre, 0, 61, C.byref(chk), C.byref(nl), C.byref(nc)) == 0, lib.rbg_last_error()
    info = full["ix"].info()
    assert chk.value > info.r and nl.value == info.n_lines and nc.value == info.n_cluster
    if full["sa"]:
        nb = C.c_uint64()
        assert lib.rbg_selftest_toehold(pre, 0, C.byref(chk), C.byref(nb)) == 0, lib.rbg_last_error()
        assert chk.value == info.r and nb.value == info.toehold_bytes
        ns, no = C.c_uint64(), C.c_uint64()
        assert lib.rbg_selftest_phi(pre, 0, 53, C.byref(chk), C.byref(ns), C.byref(no)) == 0, lib.rbg_last_error()
        assert chk.value > info.n // 53
