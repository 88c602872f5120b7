"""Layout 7: the BWT at 2 bits per row in 32-byte lines of 64 rows, for indexes small enough to stay in L2.

CPU: the host mirror of the plain-line decode (rbg_selftest_layout[_runs], the leaf.cuh code the kernels run) answers rank_c
at every position for all four symbols, and BWT[i] as the toehold step reads it, on the tiny fixture, on a dense pangenome
panel and on synthetic runs with terminators at row 0, at the last row and on line boundaries; the automatic choice takes
layout 7 up to its byte budget and below 2^31 rows, and RBG_PAIR=1 keeps layout 5 under the pair directory.  GPU: counts and
toehold searches with locations on layout 7 equal the oracle, count the same LF steps as layout 5 and build the same seed
tables."""
import ctypes as C
import os

import numpy as np
import pytest

import rowbowt_b200 as rb
from rowbowt_b200 import RBG_COUNT, RBG_LOCATE
from tools import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
TERM = 1
PLAIN_MAX_BYTES = 32 << 20                  # layout.hpp kPlainMaxBytes
PLAIN_MAX_N = PLAIN_MAX_BYTES // 32 * 64    # rows of the largest index the automatic choice lays out plain
N_SYN = 400_003


def _selftest_runs(n, heads, lens, layout=0, stride=1):
    heads = np.ascontiguousarray(heads, np.uint8)
    lens = np.ascontiguousarray(lens, np.uint64)
    chk, nl, lay = C.c_uint64(), C.c_uint64(), C.c_uint32()
    rc = rb.lib().rbg_selftest_layout_runs(n, heads.ctypes.data, lens.ctypes.data, len(heads), layout << 16, stride,
                                           C.byref(chk), C.byref(nl), C.byref(lay))
    return rc, chk.value, nl.value, lay.value


def _runs_of(bwt):
    starts = np.concatenate([[0], np.flatnonzero(np.diff(bwt)) + 1])
    return bwt[starts], np.diff(np.concatenate([starts, [len(bwt)]])).astype(np.uint64)


def _dense_runs():
    """The BWT of a panel with a variant every 5 bases (dense CLUSTER stretches in the run-length layouts)."""
    text = synth.panel_text(synth.make_panel(4000, 24, site_every=5, p_alt=0.5))
    sa = synth.suffix_array(text)
    text = np.where(text == 0, TERM, text).astype(np.uint8)
    bwt = text[(sa - 1) % len(text)]
    return (len(bwt),) + _runs_of(bwt)


# terminator places (row, length) of the synthetic indexes; rows 63-64 and 127 sit on line boundaries
CASES = {
    "1term-row0": ([(0, 1)], b"ACGT"),
    "1term-last": ([(N_SYN - 1, 1)], b"ACGT"),
    "8term": ([(0, 1), (63, 2), (127, 1), (4096 * 40, 1), (64 * 3001, 1), (N_SYN // 2 + 17, 1), (N_SYN - 1, 1)], b"ACGT"),
    "noT": ([(64, 1), (N_SYN - 1, 1)], b"ACG"),
}


def _synthetic(case):
    """Long runs alternating with dense stretches (test_synthetic_parity._runs) behind one 200-row run that holds the
    terminators placed in the first lines; every terminator replaces rows of a non-terminator run."""
    from test_synthetic_parity import _insert_terminators, _runs
    places, alphabet = CASES[case]
    rng = np.random.default_rng(sum(case.encode()))
    heads, lens, _ = _runs(rng, N_SYN - 200, alphabet, n_long=20_000, n_dense=100, dense_runs=600)
    first = b"C" if heads[0] != ord("C") else b"G"
    heads = np.concatenate([np.frombuffer(first, np.uint8), heads])
    lens = np.concatenate([np.array([200], np.uint64), lens])
    heads, lens = _insert_terminators(heads, lens, places)
    assert int(lens.sum()) == N_SYN and int(np.count_nonzero(heads == TERM)) >= 1
    return heads, lens


# ---- CPU ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pre", ["tiny/tiny", "toy/small.fa", "greedy/ref.fa"])
def test_plain_decode_fixtures(pre):
    chk, nl, nc = C.c_uint64(), C.c_uint64(), C.c_uint64()
    rc = rb.lib().rbg_selftest_layout(os.path.join(GOLDEN, pre).encode(), 7 << 16, 1, C.byref(chk), C.byref(nl), C.byref(nc))
    assert rc == 0 and chk.value > 0 and nl.value > 0 and nc.value == 0


def test_plain_decode_dense_panel():
    n, heads, lens = _dense_runs()
    rc, chk, nl, lay = _selftest_runs(n, heads, lens, layout=7)
    assert rc == 0 and lay == 7 and nl == (n + 63) // 64 and chk > 0


@pytest.mark.parametrize("case", sorted(CASES))
def test_plain_decode_synthetic(case):
    heads, lens = _synthetic(case)
    rc, chk, nl, lay = _selftest_runs(N_SYN, heads, lens, layout=7)
    assert rc == 0 and lay == 7 and nl == (N_SYN + 63) // 64
    symbols = 3 if case == "noT" else 4
    assert chk >= symbols * (N_SYN - 8)                  # every row, every symbol present in the BWT


def _long_runs(n, n_runs=1000):
    """n rows in n_runs long runs of A, C, G, T in turn, one of them a single terminator row."""
    lens = np.full(n_runs, n // n_runs, np.uint64)
    lens[n_runs // 2] = 1
    lens[-1] += np.uint64(n - int(lens.sum()))
    heads = np.frombuffer(b"ACGT", np.uint8)[np.arange(n_runs) % 4].copy()
    heads[n_runs // 2] = TERM
    return heads, lens


@pytest.mark.parametrize("n,layout", [(PLAIN_MAX_N, 7), (PLAIN_MAX_N + 1, 5), (1 << 31, 5)])
def test_automatic_layout_follows_the_budget(n, layout, monkeypatch):
    for knob in ("RBG_LAYOUT", "RBG_WINDOW", "RBG_PAIR"):
        monkeypatch.delenv(knob, raising=False)
    heads, lens = _long_runs(n)
    rc, chk, _, lay = _selftest_runs(n, heads, lens, stride=1 << 16)
    assert rc == 0 and chk > 0 and lay == layout


def test_layout7_refuses_2_pow_31_rows(monkeypatch):
    monkeypatch.delenv("RBG_LAYOUT", raising=False)
    heads, lens = _long_runs(1 << 31)
    assert _selftest_runs(1 << 31, heads, lens, layout=7, stride=1 << 20)[0] != 0


def test_pair_knob_and_forced_layouts(monkeypatch):
    """RBG_PAIR=1 asks for the pair directory, which lives over layout 5; RBG_LAYOUT forces any of the three; a forced
    window asks for a run-length layout."""
    n, heads, lens = _dense_runs()
    for knob in ("RBG_LAYOUT", "RBG_WINDOW", "RBG_PAIR"):
        monkeypatch.delenv(knob, raising=False)
    assert _selftest_runs(n, heads, lens)[3] == 7
    monkeypatch.setenv("RBG_PAIR", "0")
    assert _selftest_runs(n, heads, lens)[3] == 7
    monkeypatch.setenv("RBG_PAIR", "1")
    assert _selftest_runs(n, heads, lens)[3] == 5
    monkeypatch.setenv("RBG_LAYOUT", "7")
    assert _selftest_runs(n, heads, lens)[3] == 7
    monkeypatch.delenv("RBG_PAIR")
    for layout in ("4", "5"):
        monkeypatch.setenv("RBG_LAYOUT", layout)
        rc, _, _, lay = _selftest_runs(n, heads, lens)
        assert rc == 0 and lay == int(layout)
    monkeypatch.delenv("RBG_LAYOUT")
    monkeypatch.setenv("RBG_WINDOW", "256")
    assert _selftest_runs(n, heads, lens)[3] == 5


# ---- GPU ----------------------------------------------------------------------------------------------------------

KS = (0, 1, 7, 10, 13)


def _open_both(open_ix, monkeypatch):
    """The same index opened in the automatic layout (7 here) and in layout 5 without the pair directory."""
    out = {}
    for name, env in (("plain", {}), ("layout5", {"RBG_LAYOUT": "5", "RBG_PAIR": "0"})):
        with monkeypatch.context() as mp:
            for knob in ("RBG_LAYOUT", "RBG_WINDOW", "RBG_PAIR"):
                mp.delenv(knob, raising=False)
            for k, v in env.items():
                mp.setenv(k, v)
            out[name] = open_ix()
    assert out["plain"].info().layout == 7 and out["layout5"].info().layout == 5
    info = out["plain"].info()
    assert info.window == 64 and info.n_cluster == 0 and info.pair_bytes == 0 and info.n_lines == (info.n + 63) // 64
    assert info.dir_bytes >= info.n_lines * 32
    return out


def _parity(ixs, seqs, lo, hi, k_toe, locs_expected, tmp_path, max_hits=rb.binding.U64_MAX):
    """Count and toehold search on both layouts for every seed-table k: oracle ranges, toeholds and locations, equal LF
    steps, identical seed tables."""
    steps = {}
    for name, ix in ixs.items():
        for k in KS:
            ix.build_ftab(k)
            r = ix.query(seqs, RBG_COUNT)
            assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi), (name, k)
            steps[name, k, "count"] = ix.stats().lf_steps
            p = ix.query_packed(seqs, RBG_COUNT, threads=2)
            assert np.array_equal(p.lo, lo) and np.array_equal(p.hi, hi), (name, k)
            if k_toe is not None:
                r = ix.query(seqs, RBG_LOCATE, max_hits=max_hits)
                assert np.array_equal(r.lo, lo) and np.array_equal(r.hi, hi) and np.array_equal(r.toehold, k_toe), (name, k)
                if locs_expected is not None:
                    assert np.array_equal(r.loc_off, locs_expected[0]) and np.array_equal(r.locs, locs_expected[1]), (name, k)
                steps[name, k, "locate"] = ix.stats().lf_steps
            if 0 < k <= 10:
                ix.save_ftab(str(tmp_path / ("%s.k%d.ftab" % (name, k))))
    for key in [x for x in steps if x[0] == "plain"]:
        assert steps[key] == steps[("layout5",) + key[1:]], key
    for k in KS:
        if 0 < k <= 10:
            a = (tmp_path / ("plain.k%d.ftab" % k)).read_bytes()
            assert a == (tmp_path / ("layout5.k%d.ftab" % k)).read_bytes(), k


def _fq(path):
    with open(path, "rb") as f:
        lines = f.read().split(b"\n")
    return [lines[i] for i in range(1, len(lines), 4) if i < len(lines)]


@pytest.mark.gpu
@pytest.mark.parametrize("pre,queries", [("tiny/tiny", ("tiny/exact.fq", "tiny/noisy.fq", "tiny/short.fq", "tiny/marked.fq")),
                                         ("toy/small.fa", ("toy/simple_query.fq", "toy/error_query.fq", "toy/edge_query.fq"))])
def test_plain_search_fixtures_equal_oracle(pre, queries, monkeypatch, tmp_path):
    from oracle import oracle as O
    prefix = os.path.join(GOLDEN, pre)
    seqs = []
    for q in queries:
        seqs += _fq(os.path.join(GOLDEN, q))
    seqs += [s[: 1 + i % 15] for i, s in enumerate(seqs[:60])] + [b"", b"A", b"ACGNT", b"NNNN"]
    orc = O.OracleIndex.open(prefix, sa=True)
    lo, hi, k_toe = orc.find_ranges(seqs, toehold=True)
    locs = [orc.locate(lo[i], hi[i], k_toe[i]) for i in range(len(seqs))]
    loc_off = np.concatenate([[0], np.cumsum([len(x) for x in locs])]).astype(np.uint64)
    ixs = _open_both(lambda: rb.GpuIndex.open(prefix, sa=True), monkeypatch)
    try:
        _parity(ixs, seqs, lo, hi, k_toe, (loc_off, np.concatenate(locs).astype(np.uint64)), tmp_path)
    finally:
        for ix in ixs.values():
            ix.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_plain_search_synthetic_equals_oracle(case, monkeypatch, tmp_path):
    from oracle import oracle as O
    from oracle import rbformats as F
    from test_synthetic_parity import MAX_HITS, _reads, _toehold
    heads, lens = _synthetic(case)
    rng = np.random.default_rng(7)
    tsa = _toehold(rng, N_SYN, len(heads))
    orc = O.OracleIndex(F.Rlbwt(n=N_SYN, R=len(heads), B=2, heads=heads, lens=lens), F.Toehold(len(heads), N_SYN, *tsa), None)
    seqs = _reads(rng, CASES[case][1]) + [b"", b"A", b"C"]
    lo, hi, k_toe = orc.find_ranges(seqs, toehold=True)
    ixs = _open_both(lambda: rb.GpuIndex.from_arrays(N_SYN, heads, lens, tsa=tsa), monkeypatch)
    try:
        _parity(ixs, seqs, lo, hi, k_toe, None, tmp_path, max_hits=MAX_HITS)
        # locations on a bounded number of hits per read (long phi chains over the random toehold arrays)
        ix = ixs["plain"]
        ix.build_ftab(7)
        r = ix.query(seqs, RBG_LOCATE, max_hits=MAX_HITS)
        for i in range(len(seqs)):
            assert np.array_equal(r.locs[r.loc_off[i]:r.loc_off[i + 1]], orc.locate(lo[i], hi[i], k_toe[i], max_hits=MAX_HITS)), i
    finally:
        for ix in ixs.values():
            ix.close()


@pytest.mark.gpu
def test_pair_knob_opens_layout5_with_the_pair_directory(monkeypatch):
    monkeypatch.delenv("RBG_LAYOUT", raising=False)
    monkeypatch.setenv("RBG_PAIR", "1")
    ix = rb.GpuIndex.open(os.path.join(GOLDEN, "tiny", "tiny"))
    try:
        assert ix.info().layout == 5 and ix.info().pair_bytes > 0
    finally:
        ix.close()
