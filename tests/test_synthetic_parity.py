"""Synthetic indexes against the oracle (run with -m gpu): run arrays, toehold arrays and marker arrays with properties the
committed fixtures do not have -- n on both sides of 2^32 and up to just under the layout-5 cap of ~2^40, 1, 2 or 8
terminators (at 0, at n-1, on a window boundary, inside a collapsed CLUSTER stretch, as one run of length 2), an index
without 'T', phi buckets with more than three samples -- opened with GpuIndex.from_arrays.  The oracle is pure rank / phi
arithmetic over the same arrays, so it defines the answer for any such input, bit for bit.

Every build runs the search with and without the toehold and the seed table, both locate forms (static / drawing, each at
the CTAs per SM it is built for, u64 / narrow locations), every entry point (query, query_packed, staged + checksum, 1 and
16 chunks, narrow ranges) and greedy seeding.  What each case is meant to
reach (layout, window, CLUSTER lines, phi overflow slots, the high planes) is asserted, not assumed."""
import numpy as np
import pytest

from oracle import oracle as O
from oracle import rbformats as F

import rowbowt_b200 as rb
from rowbowt_b200 import RBG_COUNT, RBG_LOCATE, RBG_MARKERS, RBG_NARROW_LOCS, RBG_NARROW_RANGES

pytestmark = pytest.mark.gpu

L_MAX = 64                                  # longest read
MAX_HITS = 300                              # locations per read: long phi chains, small output
LAYOUT5_CAP = 256 * 32767 << 17             # layout 5: at most 256 superblocks of 32767 * 2^17 positions (W = 32767)
TERM = 1

# name: n, terminators as (kind, length), alphabet, phi bucket shift (None: the library's choice)
SPECS = {
    "mega": (1_000_003, [("at0", 1)], b"ACGT", None),
    "b32m": ((1 << 32) - 1, [("last", 1), ("cluster", 1)], b"ACGT", 12),
    "b32": (1 << 32, [("at0", 1), ("last", 1), ("boundary", 32766), ("boundary", 32764), ("boundary", 16384),
                      ("cluster", 1), ("run2", 2)], b"ACGT", 12),
    "b32p": ((1 << 32) + 1, [("boundary", 16384)], b"ACG", 12),
    "w36": ((1 << 36) + 12345, [("at0", 1), ("run2", 2)], b"ACGT", 13),
    "top": (LAYOUT5_CAP - 1000, [("cluster", 1)], b"ACGT", 14),
}

# (index, RBG_LAYOUT, RBG_WINDOW or None).  Windows above 2^32: the fast division needs (n >> k) < 2^31 for W = m * 2^k
# (m odd): 32764 = 8191 * 4 below 2^33 and 32256 = 63 * 512 below 2^40 take it, odd 32767 never does, 32766 = 16383 * 2
# sits on the switch (n = 2^32 - 1: (n >> 1) = 2^31 - 1, fast; n = 2^32: 2^31, the fallback), 16384 is a power of two
# (layout 5: superblocks of exactly 2^32 positions).  Just under the layout-5 cap only W = 32767 (or a power of two, at twice
# the lines) keeps layout 5 within 256 superblocks, so the fast division at ~2^40 runs in layout 4.
BUILDS = [
    ("mega", 4, None), ("mega", 5, None), ("mega", 5, 64),
    ("b32m", 5, 32766), ("b32m", 4, 32767),
    ("b32", 5, 32766), ("b32", 4, 32764),
    ("b32p", 5, 32764), ("b32p", 4, 16384),
    ("w36", 5, 16384), ("w36", 4, 32256), ("w36", 5, 32767),
    ("top", 5, 32767), ("top", 4, 32256),
]


def _fast_div(n, window):
    k = (window & -window).bit_length() - 1
    return (n >> k) < (1 << 31)


def _runs(rng, n, alphabet, n_long, n_dense, dense_runs):
    """Long runs (log-uniform lengths) alternating with dense stretches of runs of length 1-3; adjacent heads differ.
    Returns heads, lens and the first run of every dense stretch."""
    dense = [rng.integers(1, 4, dense_runs).astype(np.uint64) for _ in range(n_dense)]
    rest = n - int(sum(int(d.sum()) for d in dense))
    w = 2.0 ** rng.uniform(0, 16, n_long)
    lens_long = (np.floor(w / w.sum() * (rest - n_long))).astype(np.uint64) + np.uint64(1)
    lens_long[int(np.argmax(lens_long))] += np.uint64(rest - int(lens_long.sum()))
    parts, dense_at, at = [], [], 0
    for i in range(n_long):
        parts.append(lens_long[i:i + 1])
        at += 1
        if i < n_dense:
            dense_at.append(at)
            parts.append(dense[i])
            at += dense_runs
    lens = np.concatenate(parts)
    a = len(alphabet)
    codes = np.cumsum(rng.integers(1, a, len(lens))) % a
    heads = np.frombuffer(alphabet, np.uint8)[codes].copy()
    assert int(lens.sum()) == n
    return heads, lens, dense_at


def _insert_terminators(heads, lens_in, places):
    """Turns the positions [p, p + length) of the (non-terminator) run holding them into one terminator run."""
    ends = np.cumsum(lens_in.astype(np.int64))
    heads, lens = list(heads), [int(x) for x in lens_in]
    for p, tl in sorted(places, reverse=True):                  # back to front: earlier runs keep their index and start
        j = int(np.searchsorted(ends, p, side="right"))
        s = int(ends[j]) - int(lens_in[j])
        e = s + lens[j]
        assert heads[j] != TERM and p + tl <= e, (p, tl)
        pieces = [(heads[j], p - s), (TERM, tl), (heads[j], e - p - tl)]
        pieces = [x for x in pieces if x[1] > 0]
        heads[j:j + 1] = [h for h, _ in pieces]
        lens[j:j + 1] = [ln for _, ln in pieces]
    heads, lens = np.array(heads, np.uint8), np.array(lens, np.uint64)
    is_t = heads == TERM
    assert not (is_t[1:] & is_t[:-1]).any()                     # no two terminator runs touch
    return heads, lens


def _place_terms(rng, n, lens, dense_at, terms):
    ends = np.cumsum(lens.astype(np.int64))
    starts = ends - lens.astype(np.int64)
    places = []
    for kind, arg in terms:
        if kind == "at0":
            places.append((0, 1))
        elif kind == "last":
            places.append((n - 1, 1))
        elif kind == "boundary":                                # the first position of some window of size `arg`
            p = (n // 3 // arg + len(places)) * arg
            places.append((p, 1))
        elif kind == "cluster":                                 # the middle run of a dense stretch
            j = dense_at[len(dense_at) // 2 + len(places)] + 150
            places.append((int(starts[j]), 1))
        elif kind == "run2":                                    # two positions in the middle of the longest run
            j = int(np.argmax(lens))
            places.append((int(starts[j] + lens[j] // 2), 2))
    return places


def _toehold(rng, n, r):
    """pred: r - 1 sorted positions in groups of 1..12 consecutive ones (phi buckets with > 3 samples), then n - 1;
    pred_to_run in [1, r]; samples_last in [L_MAX + 1, n - 2], so that every toehold sample - since lies in [0, n)."""
    sizes = []
    while sum(sizes) < r - 1:
        sizes.append(int(rng.integers(1, 13)))
    sizes[-1] -= sum(sizes) - (r - 1)
    sizes = np.array([s for s in sizes if s > 0], np.int64)
    g = len(sizes)
    first = np.sort(rng.integers(0, n - 1 - (r - 1), g)) + np.concatenate([[0], np.cumsum(sizes)[:-1]])
    pred = (np.repeat(first, sizes) + (np.arange(r - 1) - np.repeat(np.cumsum(sizes) - sizes, sizes))).astype(np.uint64)
    pred = np.concatenate([pred, [np.uint64(n - 1)]]).astype(np.uint64)
    samples_last = rng.integers(L_MAX + 1, n - 1, r, dtype=np.uint64)
    pred_to_run = rng.integers(1, r + 1, r, dtype=np.uint64)
    assert np.all(np.diff(pred.astype(np.int64)) > 0) and int(pred[-1]) == n - 1
    assert int(pred_to_run.min()) >= 1 and int(pred_to_run.max()) <= r
    assert int(samples_last.min()) > L_MAX and int(samples_last.max()) < n - 1
    return pred, samples_last, pred_to_run


def _markers(rng, n, n_win):
    """A .mab-shaped window array: ascending windows [start, end] inside [0, n), 1..4 words each, size_idxs = len(arr),
    marker words with 44-bit positions above 2^32."""
    starts = np.unique(rng.integers(1, n - 1, n_win - 1, dtype=np.uint64))
    starts = np.concatenate([[np.uint64(0)], starts]).astype(np.uint64)
    nxt = np.concatenate([starts[1:], [np.uint64(n)]]).astype(np.uint64)
    span = (nxt - starts).astype(np.float64)
    ends = starts + np.floor(rng.uniform(0, 1, len(starts)) * span).astype(np.uint64)
    ends = np.minimum(ends, nxt - np.uint64(1))
    ends[-1] = np.uint64(n - 1)
    cnt = rng.integers(1, 5, len(starts))
    idxs = np.concatenate([[0], np.cumsum(cnt)[:-1]]).astype(np.uint64)
    m = int(cnt.sum())
    pos = rng.integers((1 << 32) + 1, 1 << 44, m, dtype=np.uint64)
    seq = rng.integers(0, 1 << 16, m, dtype=np.uint64)
    allele = rng.integers(0, 16, m, dtype=np.uint64)
    arr = pos | (seq << np.uint64(44)) | (allele << np.uint64(60))
    assert np.all(np.diff(starts.astype(np.int64)) > 0) and np.all(np.diff(ends.astype(np.int64)) > 0)
    assert np.all(ends >= starts) and int(ends[-1]) < n
    return F.MarkerWindows(n, n, m, starts, ends, idxs, arr, 19)


def _reads(rng, alphabet):
    acgt = np.frombuffer(b"ACGT", np.uint8)
    seqs = []
    for _ in range(700):
        m = int(rng.integers(1, 13)) if rng.random() < 0.6 else int(rng.integers(1, L_MAX + 1))
        seqs.append(acgt[rng.integers(0, 4, m)].tobytes())
    seqs += [b"A", b"C", b"G", b"T", b"AA", b"CA", b"GA", b"TA", b"N", b"ACGN", b"NACG", b"a", b"acgt", b"ACgT",
             b"\x01", b"\x01\x01", b"A\x01", b"\x01A", b"AC\x01\x01GT", b"\x01\x01A", b"A" * L_MAX, b"T" * L_MAX]
    missing = bytes(c for c in b"ACGT" if c not in alphabet)
    for c in missing:
        seqs += [bytes([c]), b"A" + bytes([c]), bytes([c]) + b"ACG", b"\x01" + bytes([c])]
    seqs.append(b"C")                       # the last read of the batch has a full chain of locations
    assert max(len(s) for s in seqs) <= L_MAX
    return seqs


class Synthetic:
    """Host arrays, oracle and expected results of one SPECS entry (shared by its builds)."""

    def __init__(self, name):
        n, terms, alphabet, phi_shift = SPECS[name]
        rng = np.random.default_rng(sum(name.encode()) * 7919)
        self.name, self.n, self.alphabet, self.phi_shift = name, n, alphabet, phi_shift
        if n < 1 << 24:
            heads, lens, dense_at = _runs(rng, n, alphabet, n_long=60_000, n_dense=200, dense_runs=600)
        else:
            heads, lens, dense_at = _runs(rng, n, alphabet, n_long=120_000, n_dense=64, dense_runs=600)
        self.places = _place_terms(rng, n, lens, dense_at, terms)
        self.heads, self.lens = _insert_terminators(heads, lens, self.places)
        self.n_term = sum(tl for _, tl in self.places)
        self.R = len(self.heads)
        assert self.R <= 200_000 and 1 <= self.n_term <= 8
        self.tsa = _toehold(rng, n, self.R)
        self.ma = _markers(rng, n, 600)
        bwt = F.Rlbwt(n=n, R=self.R, B=2, heads=self.heads, lens=self.lens)
        self.orc = O.OracleIndex(bwt, F.Toehold(self.R, n, *self.tsa), self.ma)
        self.seqs = _reads(rng, alphabet)
        lo, hi, k = self.orc.find_ranges(self.seqs, toehold=True)
        alive = hi >= lo
        # safety before any locate on the device: every toehold and every location is a text position
        assert np.all(k[alive] < np.uint64(n)) and np.all(hi[alive] < np.uint64(n))
        locs = [self.orc.locate(lo[i], hi[i], k[i], max_hits=MAX_HITS) for i in range(len(self.seqs))]
        mks = [self.orc.markers_at_range(lo[i], hi[i]) for i in range(len(self.seqs))]
        self.lo, self.hi, self.k = lo, hi, k
        self.loc_off = np.concatenate([[0], np.cumsum([len(x) for x in locs])]).astype(np.uint64)
        self.locs = np.concatenate(locs).astype(np.uint64)
        self.mk_off = np.concatenate([[0], np.cumsum([len(x) for x in mks])]).astype(np.uint64)
        self.mks = np.concatenate(mks).astype(np.uint64)
        assert np.all(self.locs < np.uint64(n))
        assert int(alive.sum()) > 100 and len(self.locs) > 20_000 and len(self.mks) > 0
        # count only: the empty read keeps the full range
        self.count_seqs = self.seqs + [b"", b"A", b""]
        self.clo, self.chi, _ = self.orc.find_ranges(self.count_seqs)
        assert (int(self.clo[-1]), int(self.chi[-1])) == (0, n - 1)
        self.greedy = [s for s in self.seqs if len(s) >= 7 and set(s) <= set(b"ACGT")]

    def open(self, monkeypatch, layout, window):
        monkeypatch.setenv("RBG_LAYOUT", str(layout))
        if window:
            monkeypatch.setenv("RBG_WINDOW", str(window))
        else:
            monkeypatch.delenv("RBG_WINDOW", raising=False)
        if self.phi_shift:
            monkeypatch.setenv("RBG_PHI_SHIFT", str(self.phi_shift))      # 2^s-position buckets keep the l1 words small
        ma = self.ma
        return rb.GpuIndex.from_arrays(self.n, self.heads, self.lens, tsa=self.tsa,
                                       ma=(ma.starts, ma.ends, ma.idxs, ma.arr, ma.size_starts, ma.size_ends, ma.size_idxs))

    def check(self, r, locate=True, markers=True):
        assert np.array_equal(r.lo, self.lo) and np.array_equal(r.hi, self.hi)
        if locate:
            assert np.array_equal(r.toehold, self.k)
            assert np.array_equal(r.loc_off, self.loc_off)
            assert np.array_equal(r.locs, self.locs)
        if markers:
            assert np.array_equal(r.mk_off, self.mk_off)
            assert np.array_equal(r.markers, self.mks)

    def check_count(self, r):
        assert np.array_equal(r.lo, self.clo) and np.array_equal(r.hi, self.chi)


_CACHE = {}


def synthetic(name):
    if name not in _CACHE:
        _CACHE.clear()                                          # one index's host arrays at a time
        _CACHE[name] = Synthetic(name)
    return _CACHE[name]


@pytest.mark.parametrize("name,layout,window", BUILDS, ids=["%s-L%d-W%s" % b for b in BUILDS])
def test_synthetic_index_equals_oracle(name, layout, window, monkeypatch):
    s = synthetic(name)
    n = s.n
    ix = s.open(monkeypatch, layout, window)
    try:
        info = ix.info()
        assert (info.n, info.r, info.layout) == (n, s.R, layout)
        if window:
            assert info.window == window
        assert info.n_cluster > 0                               # CLUSTER lines with RAW children
        assert info.phi_overflow > 0                            # BITMAP (shift <= 7) or SEARCH (shift > 7) phi slots
        assert info.phi_shift == (s.phi_shift or 7)
        assert [info.F[c] for c in range(256)] == [s.orc.F(c) for c in range(256)]
        assert info.toehold0 == O.lib().orc_last_run_sample(s.orc.h)
        if name == "b32m" and window == 32766:
            assert _fast_div(n, info.window)                    # the last n of the fast division ...
        if name == "b32" and window == 32766:
            assert not _fast_div(n, info.window)                # ... and the first of the fallback
        if name == "top" and layout == 4:
            assert _fast_div(n, info.window)
        mode = RBG_LOCATE | RBG_MARKERS

        # search x toehold x seed table
        for k in (0, 1, 7, 13):
            ix.build_ftab(k)
            assert ix.info().ftab_k == k
            s.check(ix.query(s.seqs, mode, max_hits=MAX_HITS))
            st = ix.stats()
            assert st.lf_steps > 0 and st.phi_steps > 0
            s.check_count(ix.query(s.count_seqs, RBG_COUNT))
        ix.build_ftab(0)

        # locate forms: static / drawing kernel, u64 / narrow locations (+ the high plane above 2^32)
        for draw in ("0", "1"):
            with monkeypatch.context() as mp:
                mp.setenv("RBG_LOC_DRAW", draw)
                s.check(ix.query(s.seqs, RBG_LOCATE, max_hits=MAX_HITS), markers=False)
                assert ix.stats().phi_steps == len(s.locs) - int(np.count_nonzero(np.diff(s.loc_off)))
                r = ix.query(s.seqs, RBG_LOCATE | RBG_NARROW_LOCS, max_hits=MAX_HITS)
                s.check(r, markers=False)
                assert r.narrow_bytes == (5 if n >> 32 else 4)

        # entry points
        for threads in (1, 3):
            s.check(ix.query_packed(s.seqs, mode, max_hits=MAX_HITS, threads=threads))
            s.check_count(ix.query_packed(s.count_seqs, RBG_COUNT, threads=threads))
        st = ix.upload(s.seqs)
        cs = ix.query_staged(st, mode, max_hits=MAX_HITS, checksum=True)
        assert cs == rb.result_checksum(s.lo, s.hi, s.k, s.loc_off, s.locs, s.mk_off, s.mks)
        assert ix.query_staged(st, RBG_COUNT, checksum=True) == rb.result_checksum(s.lo, s.hi)
        st.free()
        for chunks in ("1", "16"):
            with monkeypatch.context() as mp:
                mp.setenv("RBG_CHUNKS", chunks)
                s.check(ix.query(s.seqs, mode, max_hits=MAX_HITS))
        r = ix.query(s.count_seqs, RBG_COUNT | RBG_NARROW_RANGES)
        assert r.narrow_ranges == (n < 1 << 32)                 # u32 planes on the wire only below 2^32
        s.check_count(r)

        # greedy seeding, with and without the seed table
        for k in (0, 7):
            ix.build_ftab(k)
            got = ix.markers_greedy(s.greedy, max_range=1 << 41, use_ftab=bool(k))      # every seed collects its markers
            exp = s.orc.rb_markers(s.greedy, max_range=1 << 41, ftab_k=k)
            assert np.array_equal(got[0], exp[0])
            for f in ("lo", "hi", "qstart", "qlen", "mk_raw", "mk_cnt", "mk_off"):
                assert np.array_equal(got[1][f], exp[1][f]), f
            assert np.array_equal(got[2], exp[2])

        if name == "top":                                       # position bits 36..39 are in play
            assert int(s.hi.max()) >= 1 << 39 and int(s.locs.max()) >= 1 << 39
    finally:
        ix.close()


def test_layout5_past_256_superblocks_is_an_error(monkeypatch):
    """W = 32766 makes superblocks of 32766 * 2^17 positions: the top index then needs 257 of them."""
    s = synthetic("top")
    monkeypatch.setenv("RBG_LAYOUT", "5")
    monkeypatch.setenv("RBG_WINDOW", "32766")
    with pytest.raises(rb.RbgError):
        rb.GpuIndex.from_arrays(s.n, s.heads, s.lens)


def test_arrays_that_would_index_out_of_bounds_are_rejected():
    """Validation runs on the host before anything is uploaded: a run-end sample >= n (it would become a toehold and a
    phi argument) and a marker index universe beyond the marker words (it ends the last window's gather)."""
    s = synthetic("mega")
    pred, samples_last, pred_to_run = s.tsa
    bad = samples_last.copy()
    bad[len(bad) // 2] = np.uint64(s.n)
    with pytest.raises(rb.RbgError) as e:
        rb.GpuIndex.from_arrays(s.n, s.heads, s.lens, tsa=(pred, bad, pred_to_run))
    assert e.value.code == -2
    ma = s.ma
    with pytest.raises(rb.RbgError) as e:
        rb.GpuIndex.from_arrays(s.n, s.heads, s.lens,
                                ma=(ma.starts, ma.ends, ma.idxs, ma.arr, ma.size_starts, ma.size_ends, len(ma.arr) + 1))
    assert e.value.code == -2
    # the same arrays with the bounds kept open fine
    rb.GpuIndex.from_arrays(s.n, s.heads, s.lens, tsa=s.tsa,
                            ma=(ma.starts, ma.ends, ma.idxs, ma.arr, ma.size_starts, ma.size_ends, len(ma.arr))).close()
