"""rb_markers greedy-seeding marker genotyping (SURVEY.md §8(f) row 1).

CPU (-m "not gpu"): the oracle's restatement of get_markers_greedy_seeding + the rb_markers worker
(oracle/rlbwt_oracle.c) against the committed stdout of the UNMODIFIED reference binary
(tests/golden/expected/rbm.*.txt, made by tests/golden/make_rb_markers_golden.py), and against the
live binary when oracle/_ref is present.
GPU (-m gpu): rbg_markers_greedy through the C ABI against the oracle (every seed record and marker
word, bit-exact) and the host rb_markers binary against the reference's stdout, byte for byte.
"""
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, read_fastx
from oracle import oracle as O

import rowbowt_b200 as rb

EXP = os.path.join(GOLDEN, "expected")
CASES = json.load(open(os.path.join(EXP, "rb_markers_cases.json")))
RB_MARKERS = os.path.join(ROOT, "rowbowt_b200", "rb_markers")


def case_id(c):
    return c["out"][4:-4] + ":" + "".join(c["flags"])


def parse_flags(flags):
    """wsize / max_range / min_range of a reference command line; None when a host-side filter is on."""
    kw = {"wsize": 19, "max_range": 1000, "min_range": 0}
    it = iter(flags)
    for f in it:
        if f == "-w":
            kw["wsize"] = int(next(it))
        elif f == "-r":
            kw["max_range"] = int(next(it))
        elif f == "-m":
            kw["min_range"] = int(next(it))
        elif f == "--ftab":
            pass
        else:
            return None
    return kw


PLAIN = [c for c in CASES if parse_flags(c["flags"]) is not None]


@pytest.mark.parametrize("c", PLAIN, ids=case_id)
def test_oracle_matches_reference_rb_markers_stdout(c):
    prefix = os.path.join(GOLDEN, c["fixture"], c["prefix"])
    orc = O.OracleIndex.open(prefix, markers=True)
    names, seqs = read_fastx(os.path.join(GOLDEN, c["fixture"], c["fastq"]))
    got = orc.rb_markers_text(names, seqs, ftab_k=c["ftab_k"], **parse_flags(c["flags"]))
    assert got == open(os.path.join(EXP, c["out"])).read()


def test_oracle_reports_the_reference_error_exits():
    orc = O.OracleIndex.open(os.path.join(GOLDEN, "toy", "small.fa"), markers=True)
    with pytest.raises(ValueError):
        orc.rb_markers([b"ACGTACGTACGT"], wsize=2, ftab_k=4)          # k - 1 > wsize: include/rowbowt.hpp:423-426
    with pytest.raises(ValueError):
        orc.rb_markers([b"ACG"], wsize=10, ftab_k=4)                  # read shorter than k: substr throws at :431


@pytest.mark.skipif(not os.path.exists(os.path.join(O.REFBIN, "rb_markers")), reason="compiled reference not present")
def test_oracle_matches_live_reference_on_random_reads(tmp_path):
    """Reads the goldens do not hold: random mutations of genuine substrings, both strands, all window sizes."""
    prefix = os.path.join(GOLDEN, "tiny", "tiny")
    orc = O.OracleIndex.open(prefix, markers=True)
    _, base = read_fastx(os.path.join(GOLDEN, "tiny", "exact.fq"))
    rng = np.random.default_rng(21)
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    seqs = []
    for i, s in enumerate(base[:120]):
        a = bytearray(s if i % 2 else s.translate(comp)[::-1])
        for _ in range(int(rng.integers(0, 4))):
            a[int(rng.integers(0, len(a)))] = b"ACGTN"[int(rng.integers(0, 5))]
        seqs.append(bytes(a))
    names = ["q%d" % i for i in range(len(seqs))]
    fq = tmp_path / "q.fq"
    fq.write_bytes(b"".join(b"@%s\n%s\n+\n%s\n" % (n.encode(), s, b"I" * len(s)) for n, s in zip(names, seqs)))
    for w, mr, mn in ((1, 1000, 0), (5, 3, 0), (12, 1000, 2), (30, 1000, 0), (200, 1000, 0)):
        assert orc.rb_markers_text(names, seqs, wsize=w, max_range=mr, min_range=mn) == \
            O.ref_rb_markers(prefix, str(fq), w, mr, mn)


# ---- GPU ----------------------------------------------------------------------------------------------------

def assert_same_seeds(got, exp):
    g_off, g_seeds, g_words = got
    e_off, e_seeds, e_words = exp
    assert np.array_equal(g_off, e_off)
    for f in ("lo", "hi", "qstart", "qlen", "mk_raw", "mk_cnt", "mk_off"):
        assert np.array_equal(g_seeds[f], e_seeds[f]), f
    for s in np.nonzero(e_seeds["mk_cnt"])[0]:
        o, c = int(e_seeds["mk_off"][s]), int(e_seeds["mk_cnt"][s])
        assert np.array_equal(g_words[o:o + c], e_words[o:o + c]), s


@pytest.mark.gpu
@pytest.mark.parametrize("c", PLAIN, ids=case_id)
def test_gpu_seeds_match_oracle_and_reference_stdout(c):
    prefix = os.path.join(GOLDEN, c["fixture"], c["prefix"])
    kw = parse_flags(c["flags"])
    names, seqs = read_fastx(os.path.join(GOLDEN, c["fixture"], c["fastq"]))
    ix = rb.GpuIndex.open(prefix, markers=True)
    if c["ftab_k"]:
        ix.build_ftab(c["ftab_k"])
    got = ix.markers_greedy(seqs, use_ftab=bool(c["ftab_k"]), **kw)
    st = ix.stats()
    assert st.lf_steps > 0 and st.launches >= 4
    orc = O.OracleIndex.open(prefix, markers=True)
    assert_same_seeds(got, orc.rb_markers(seqs, ftab_k=c["ftab_k"], **kw))
    assert O.render_seeds(names, *got) == open(os.path.join(EXP, c["out"])).read()
    ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_rb_markers_binary_matches_reference_stdout(c, tmp_path):
    """The host rb_markers over the C ABI prints byte-for-byte what the reference printed at --threads 1,
    including the --heuristic post-filters (random first strand, best strand, conflicting / identical markers)."""
    prefix = os.path.join(GOLDEN, c["fixture"], c["prefix"])
    if c["ftab_k"]:
        for suf in (".rbwt", ".mab"):
            shutil.copy(prefix + suf, tmp_path / (c["prefix"] + suf))
        shutil.copy(os.path.join(EXP, "%s.k%d.ftab" % (c["fixture"], c["ftab_k"])), tmp_path / (c["prefix"] + ".ftab"))
        prefix = str(tmp_path / c["prefix"])
    for batch in ("37", "100000"):
        p = subprocess.run([RB_MARKERS, "--batch", batch] + c["flags"] + [prefix, os.path.join(GOLDEN, c["fixture"], c["fastq"])],
                           capture_output=True)
        assert p.returncode == 0, p.stderr.decode()
        assert p.stdout == open(os.path.join(EXP, c["out"]), "rb").read()


@pytest.mark.gpu
def test_gpu_greedy_edge_cases():
    prefix = os.path.join(GOLDEN, "toy", "small.fa")
    ix = rb.GpuIndex.open(prefix, markers=True)
    orc = O.OracleIndex.open(prefix, markers=True)
    seqs = [b"", b"A", b"N", b"n", b"a", b"R", b"\x01", b"\xff", b"AC", b"ACGT" * 50, b"A" * 31, b"A" * 32, b"A" * 33, b"T" * 64,
            b"NNNNNNNNNNNN", b"GGCAGGCGGA", b"ggcaggcgga", b"GGCAGNCGGA", b"GGCAG-CGGATTCGTCGTAA", b"TTCGTCGTAA" * 3]
    rng = np.random.default_rng(5)
    acgt = np.frombuffer(b"ACGTN", np.uint8)
    for _ in range(200):
        seqs.append(acgt[rng.integers(0, 5, int(rng.integers(1, 180))) % (4 + (rng.random() < 0.3))].tobytes())
    for w, mr, mn in ((0, 1000, 0), (1, 1000, 0), (3, 2, 0), (10, 1000, 0), (10, 1000, 5), (19, 10 ** 9, 0)):
        assert_same_seeds(ix.markers_greedy(seqs, wsize=w, max_range=mr, min_range=mn), orc.rb_markers(seqs, wsize=w, max_range=mr, min_range=mn))
    # empty batch
    off, seeds, words = ix.markers_greedy([])
    assert len(off) == 1 and len(seeds) == 0 and len(words) == 0
    # with the seed table: every k, reads at least k long
    longer = [s for s in seqs if len(s) >= 6]
    for k in (1, 3, 6):
        ix.build_ftab(k)
        assert_same_seeds(ix.markers_greedy(longer, wsize=7, use_ftab=True), orc.rb_markers(longer, wsize=7, ftab_k=k))
    # the reference's error exits come back as error codes
    ix.build_ftab(6)
    with pytest.raises(rb.RbgError):
        ix.markers_greedy(longer, wsize=4, use_ftab=True)             # k - 1 > wsize
    with pytest.raises(rb.RbgError):
        ix.markers_greedy([b"ACG"], wsize=10, use_ftab=True)          # read shorter than k
    ix.build_ftab(0)
    with pytest.raises(rb.RbgError):
        ix.markers_greedy(longer, use_ftab=True)                      # no table resident
    ix.close()
    ix = rb.GpuIndex.open(prefix)
    with pytest.raises(rb.RbgError):
        ix.markers_greedy(seqs)                                       # index opened without the marker array
    ix.close()


@pytest.mark.gpu
def test_gpu_greedy_larger_index_sample(small_index):
    """The `small` index (1 Mbp x 16 haplotypes): 3000 noisy 150 bp reads, both the plain and the ftab-seeded walk,
    against the oracle."""
    from tools import synth
    prefix = small_index
    panel = synth.make_panel(*synth.CONFIGS["small"])
    reads, _, _ = synth.make_reads(panel, 3000, 150, seed=17, err_rate=0.01, n_rate=0.001)
    ix = rb.GpuIndex.open(prefix, markers=True)
    orc = O.OracleIndex.open(prefix, markers=True)
    assert_same_seeds(ix.markers_greedy(reads, wsize=10), orc.rb_markers(reads, wsize=10))
    ix.build_ftab(10)
    assert_same_seeds(ix.markers_greedy(reads, wsize=19, use_ftab=True), orc.rb_markers(reads, wsize=19, ftab_k=10))
    ix.close()
