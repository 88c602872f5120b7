"""Two bases per LF step in the count search: the pair directory over P[j] = (BWT[LF(j)], BWT[j]).

CPU: the pair runs the library builds from the BWT runs alone equal the pair sequence read off a suffix array, and the
host mirror of the pair decode (rbg_selftest_pair: the leaf.cuh code the kernel runs) answers K[p] + rank_p at every
position, CLUSTER windows and the terminator rows included.  GPU: the count search with the pair directory (RBG_PAIR=1)
and without it (RBG_PAIR=0) return the oracle's ranges and count the same LF steps, on the tiny fixture and on synthetic
indexes with 1 and 8 terminators, without 'T', and with dense CLUSTER stretches."""
import ctypes as C
import os

import numpy as np
import pytest

import rowbowt_b200 as rb
from rowbowt_b200 import RBG_COUNT
from tools import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CODE = np.full(256, 4, np.int64)
CODE[list(b"ACGT")] = np.arange(4)


def _selftest(n, heads, lens, window=0, stride=1, codes=False):
    heads = np.ascontiguousarray(heads, np.uint8)
    lens = np.ascontiguousarray(lens, np.uint64)
    out = np.zeros(n, np.uint8) if codes else None
    chk, nl, nc = C.c_uint64(), C.c_uint64(), C.c_uint64()
    rc = rb.lib().rbg_selftest_pair(n, heads.ctypes.data, lens.ctypes.data, len(heads), window, stride,
                                    out.ctypes.data if codes else None, C.byref(chk), C.byref(nl), C.byref(nc))
    return rc, chk.value, nc.value, out


def _runs(bwt):
    starts = np.concatenate([[0], np.flatnonzero(np.diff(bwt)) + 1])
    return bwt[starts], np.diff(np.concatenate([starts, [len(bwt)]])).astype(np.uint64)


def _panel(name):
    if name == "tiny":
        return synth.make_panel(*synth.CONFIGS["tiny"])
    return synth.make_panel(4000, 24, site_every=5, p_alt=0.5)         # a variant every 5 bases: dense CLUSTER stretches


def _bwt_and_pairs(panel):
    text = synth.panel_text(panel)
    sa = synth.suffix_array(text)
    text = np.where(text == 0, 1, text).astype(np.uint8)                # the index's terminator byte
    n = len(text)
    bwt = text[(sa - 1) % n]
    c2, c1 = CODE[bwt], CODE[text[(sa - 2) % n]]
    return bwt, np.where((c1 < 4) & (c2 < 4), 4 * c1 + c2, 16).astype(np.uint8)


@pytest.mark.parametrize("name", ["tiny", "dense"])
def test_pair_runs_equal_suffix_array_pairs(name):
    bwt, pairs = _bwt_and_pairs(_panel(name))
    heads, lens = _runs(bwt)
    rc, chk, _, codes = _selftest(len(bwt), heads, lens, codes=True)
    assert rc == 0 and chk == 16 * (len(bwt) + 1)
    assert np.array_equal(codes, pairs)


@pytest.mark.parametrize("window", [0, 16, 30, 128, 130, 256])
@pytest.mark.parametrize("name", ["tiny", "dense"])
def test_pair_decode_every_position(name, window):
    bwt, _ = _bwt_and_pairs(_panel(name))
    heads, lens = _runs(bwt)
    rc, chk, n_cluster, _ = _selftest(len(bwt), heads, lens, window=window)
    assert rc == 0 and chk == 16 * (len(bwt) + 1)
    if name == "dense" and window >= 128:
        assert n_cluster > 0


def _synthetic_runs(n, terms, alphabet, seed):
    from test_synthetic_parity import _insert_terminators, _place_terms, _runs as runs
    rng = np.random.default_rng(seed)
    heads, lens, dense_at = runs(rng, n, alphabet, n_long=20_000, n_dense=100, dense_runs=600)
    return _insert_terminators(heads, lens, _place_terms(rng, n, lens, dense_at, terms))


TERMS8 = [("at0", 1), ("last", 1), ("cluster", 1), ("cluster", 1), ("run2", 2), ("boundary", 4096), ("boundary", 64)]


@pytest.mark.parametrize("terms,alphabet", [([("at0", 1)], b"ACGT"), (TERMS8, b"ACGT"), ([("last", 1), ("run2", 2)], b"ACG")],
                         ids=["1term", "8term", "noT"])
def test_pair_decode_synthetic(terms, alphabet):
    heads, lens = _synthetic_runs(400_003, terms, alphabet, 11)
    for window in (0, 256):
        rc, chk, n_cluster, _ = _selftest(400_003, heads, lens, window=window, stride=7)
        assert rc == 0 and chk > 16 * 400_003 // 7
        assert n_cluster > 0


# ---- GPU ----------------------------------------------------------------------------------------------------------

def _read_fq(path):
    with open(path, "rb") as f:
        lines = f.read().split(b"\n")
    return [lines[i] for i in range(1, len(lines), 4) if i < len(lines)]


def _both(open_ix, monkeypatch, queries):
    """queries(ix) -> list of (lo, hi, lf_steps); the same with and without the pair directory."""
    out = []
    for pair in ("0", "1"):
        with monkeypatch.context() as mp:
            mp.setenv("RBG_PAIR", pair)
            ix = open_ix()
            try:
                assert (ix.info().pair_bytes > 0) == (pair == "1")
                out.append(queries(ix))
            finally:
                ix.close()
    return out


@pytest.mark.gpu
def test_pair_search_tiny_equals_oracle(monkeypatch):
    from oracle import oracle as O
    pre = os.path.join(GOLDEN, "tiny", "tiny")
    seqs = []
    for f in ("exact.fq", "noisy.fq", "short.fq", "marked.fq"):
        seqs += _read_fq(os.path.join(GOLDEN, "tiny", f))
    exact = _read_fq(os.path.join(GOLDEN, "tiny", "exact.fq"))
    seqs += [exact[i % len(exact)][: 1 + i % 15] for i in range(60)]           # lengths 1 .. 15: below, at and above k
    seqs += [exact[i % len(exact)][: 2 * (i % 40) + 1] for i in range(80)]     # odd lengths
    seqs += [b"", b"A", b"ACGNT", b"NNNN"]
    orc = O.OracleIndex.open(pre)
    lo, hi = orc.find_ranges(seqs)[:2]

    def queries(ix):
        got = []
        for k in (0, 1, 7, 10, 13):
            ix.build_ftab(k)
            r = ix.query(seqs, RBG_COUNT)
            assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi), k
            steps = ix.stats().lf_steps
            p = ix.query_packed(seqs, RBG_COUNT, threads=2)
            assert np.array_equal(p.lo, lo) and np.array_equal(p.hi, hi), k
            for chunks in ("1", "16"):
                with monkeypatch.context() as mp:
                    mp.setenv("RBG_CHUNKS", chunks)
                    r = ix.query(seqs, RBG_COUNT)
                    assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi), (k, chunks)
            st = ix.upload(seqs)
            assert ix.query_staged(st, RBG_COUNT, checksum=True) == rb.result_checksum(lo, hi)
            st.free()
            got.append(steps)
        return got

    single, pair = _both(lambda: rb.GpuIndex.open(pre), monkeypatch, queries)
    assert single == pair


@pytest.mark.gpu
@pytest.mark.parametrize("terms,alphabet,window", [([("at0", 1)], b"ACGT", None), (TERMS8, b"ACGT", None),
                                                   (TERMS8, b"ACGT", "256"), ([("last", 1), ("run2", 2)], b"ACG", None)],
                         ids=["1term", "8term", "8term-W256", "noT"])
def test_pair_search_synthetic_equals_oracle(terms, alphabet, window, monkeypatch):
    from oracle import oracle as O
    from oracle import rbformats as F
    from test_synthetic_parity import _reads
    n = 400_003
    heads, lens = _synthetic_runs(n, terms, alphabet, 11)
    orc = O.OracleIndex(F.Rlbwt(n=n, R=len(heads), B=2, heads=heads, lens=lens), None, None)
    rng = np.random.default_rng(5)
    seqs = _reads(rng, alphabet) + [b"", b"A", b"C"]
    lo, hi = orc.find_ranges(seqs)[:2]
    if window:
        monkeypatch.setenv("RBG_PAIR_WINDOW", window)

    def queries(ix):
        if window and ix.info().pair_bytes:
            assert ix.info().pair_window == int(window)
        got = []
        for k in (0, 1, 7, 13):
            ix.build_ftab(k)
            r = ix.query(seqs, RBG_COUNT)
            assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi), k
            got.append(ix.stats().lf_steps)
        return got

    single, pair = _both(lambda: rb.GpuIndex.from_arrays(n, heads, lens), monkeypatch, queries)
    assert single == pair
