"""The marker array (.ma) built on the GPU from a .mps and the index's own phi (mps_to_ma without the suffix-array stream).

CPU part: the numpy restatement of the mapping (tools/synth.ma_from_mps over a numpy SA, the .mps from tools/synth.write_mps)
reproduces the reference mps_to_ma's tiny.ma and write_raw_index's .ma; malformed .mps files and bad arguments are refused
before any CUDA call; the binary refuses the suffix-array stream.
GPU part: the builder against the reference's files (tiny), write_raw_index (small), and the oracle's phi on synthetic
indexes with positions past 2^32."""
import filecmp
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

import rowbowt_b200 as rb
from oracle import oracle as O
from oracle import rbformats as F
from tools import synth

MPS_TO_MA = os.path.join(ROOT, "rowbowt_b200", "mps_to_ma")
RAW = os.path.join(GOLDEN, "raw", "tiny")
TINY = os.path.join(GOLDEN, "tiny", "tiny")
DELIM = 0xFFFFFFFFFFFFFFFF


def _records(words):
    """.ma / .mps words -> [(first, last, (word, ...))]"""
    w = np.asarray(words, np.uint64)
    ends = np.nonzero(w == np.uint64(DELIM))[0].tolist()
    out, s = [], 0
    for e in ends:
        out.append((int(w[s]), int(w[s + 1]), tuple(w[s + 2:e].tolist())))
        s = e + 1
    return out


def _tiny_mps(path):
    synth.write_mps(synth.make_panel(*synth.CONFIGS["tiny"]), path)
    return path


# ---- CPU ----------------------------------------------------------------------------------------------------------------

def test_mps_mapping_reproduces_reference_tiny_ma(tmp_path):
    """write_mps(tiny) mapped through the numpy SA is the unmodified mps_to_ma's tiny.ma, byte for byte."""
    panel = synth.make_panel(*synth.CONFIGS["tiny"])
    mps = _tiny_mps(str(tmp_path / "tiny.mps"))
    sa = synth.suffix_array(synth.panel_text(panel))
    got = synth.ma_from_mps(sa, 0, np.fromfile(mps, np.uint64))
    assert np.array_equal(got, np.fromfile(RAW + ".ma", np.uint64))


def _dense_panel(seed, L, H, wsize):
    """Sites closer than wsize (records with several words) and within wsize of every sequence start (windows that cross
    the padding of the sequence before)."""
    rng = np.random.default_rng(seed)
    ref = synth.ACGT[rng.integers(0, 4, L)]
    gaps = rng.integers(1, 2 * wsize, L)
    sites = np.unique(np.concatenate([[int(rng.integers(0, 3))], rng.integers(0, wsize, 2), np.cumsum(gaps)]))
    sites = sites[sites < L].astype(np.int64)
    code = np.searchsorted(synth.ACGT, ref[sites])
    alts = synth.ACGT[(code + rng.integers(1, 4, len(sites))) % 4]
    gt = rng.random((H, len(sites))) < 0.4
    return synth.Panel(L, H, ref, sites, alts, gt)


@pytest.mark.parametrize("seed,wsize", [(11, 5), (12, 10), (13, 19)])
def test_mps_mapping_equals_write_raw_index(tmp_path, seed, wsize):
    panel = _dense_panel(seed, 1500, 3, wsize)
    pre = str(tmp_path / "p")
    synth.write_raw_index(panel, pre, wsize=wsize)
    synth.write_mps(panel, pre + ".mps", wsize=wsize)
    mps = np.fromfile(pre + ".mps", np.uint64)
    assert any(len(ws) > 1 for _, _, ws in _records(mps))                       # several words in one record
    sa = synth.suffix_array(synth.panel_text(panel))
    got = synth.ma_from_mps(sa, 0, mps)
    assert np.array_equal(got, np.fromfile(pre + ".ma", np.uint64))


def _small_arrays():
    """n = 100: two runs, one toehold sample each."""
    heads = np.array([ord("A"), ord("C")], np.uint8)
    lens = np.array([50, 50], np.uint64)
    tsa = (np.array([10, 99], np.uint64), np.array([5, 60], np.uint64), np.array([1, 2], np.uint64))
    return 100, heads, lens, tsa


MALFORMED = {
    "cut_tail": ([3, 4, 7, DELIM, 10, 12, 7], "record 1"),
    "cut_word": (None, "record 1"),
    "first_after_last": ([3, 4, 7, DELIM, 12, 10, 7, DELIM], "record 1"),
    "overlap": ([3, 10, 7, DELIM, 10, 12, 7, DELIM], "record 1"),
    "unsorted": ([20, 30, 7, DELIM, 3, 4, 7, DELIM], "record 1"),
    "last_beyond_n": ([3, 4, 7, DELIM, 10, 100, 7, DELIM], "record 1"),
}


@pytest.mark.parametrize("case", sorted(MALFORMED))
def test_malformed_mps_refused_before_cuda(tmp_path, case):
    """Refused with RBG_E_FORMAT naming the record, before any CUDA call: this runs without a GPU."""
    words, where = MALFORMED[case]
    path = str(tmp_path / "bad.mps")
    if words is None:
        with open(path, "wb") as f:
            f.write(np.array([3, 4, 7, DELIM, 10, 12], np.uint64).tobytes() + b"\x07\x00\x00")
    else:
        np.array(words, np.uint64).tofile(path)
    n, heads, lens, tsa = _small_arrays()
    with pytest.raises(rb.RbgError) as e:
        rb.build_marker_array_arrays(n, heads, lens, tsa, path, str(tmp_path / "o.ma"))
    assert e.value.code == -2 and where in str(e.value), str(e.value)
    with pytest.raises(rb.RbgError) as e:                                     # the same through the index files
        rb.build_marker_array(TINY, path if case != "last_beyond_n" else _beyond(tmp_path), str(tmp_path / "o.ma"))
    assert e.value.code == -2, str(e.value)
    assert not os.path.exists(str(tmp_path / "o.ma"))


def _beyond(tmp_path):
    n = os.path.getsize(RAW + ".bwt")
    path = str(tmp_path / "beyond.mps")
    np.array([3, 4, 7, DELIM, 10, n, 7, DELIM], np.uint64).tofile(path)
    return path


def test_empty_records_are_accepted_before_cuda(tmp_path):
    """A record without words passes the reader (its rows get no list): the call gets as far as the device."""
    path = str(tmp_path / "ok.mps")
    np.array([3, 4, DELIM, 10, 12, 7, DELIM], np.uint64).tofile(path)
    n, heads, lens, tsa = _small_arrays()
    if rb.lib().rbg_device_count() > 0:
        rb.build_marker_array_arrays(n, heads, lens, tsa, path, str(tmp_path / "o.ma"))
        return
    with pytest.raises(rb.RbgError) as e:
        rb.build_marker_array_arrays(n, heads, lens, tsa, path, str(tmp_path / "o.ma"))
    assert e.value.code == -4


def test_argument_errors_before_cuda(tmp_path):
    mps = _tiny_mps(str(tmp_path / "tiny.mps"))
    out = str(tmp_path / "o.ma")
    # no .tsa beside the .rbwt
    for suf in (".rbwt",):
        os.symlink(TINY + suf, str(tmp_path / "notsa") + suf)
    with pytest.raises(rb.RbgError) as e:
        rb.build_marker_array(str(tmp_path / "notsa"), mps, out)
    assert e.value.code == -1
    # raw inputs without .esa
    for suf in (".bwt", ".ssa"):
        os.symlink(RAW + suf, str(tmp_path / "noesa") + suf)
    with pytest.raises(rb.RbgError) as e:
        rb.build_marker_array(str(tmp_path / "noesa"), mps, out)
    assert e.value.code == -1
    n = os.path.getsize(RAW + ".bwt")
    for rows in ((5, 5), (7, 3), (n, n + 10), (n + 1, 2 * n)):                  # empty or inverted windows
        with pytest.raises(rb.RbgError) as e:
            rb.build_marker_array(TINY, mps, out, rows=rows)
        assert e.value.code == -5, rows
    n_small, heads, lens, tsa = _small_arrays()
    np.array([3, 4, 7, DELIM], np.uint64).tofile(str(tmp_path / "s.mps"))
    with pytest.raises(rb.RbgError) as e:                                     # r != R
        rb.build_marker_array_arrays(n_small, heads, lens, tuple(x[:1] for x in tsa), str(tmp_path / "s.mps"), out)
    assert e.value.code == -5
    assert not os.path.exists(out)


def test_binary_refuses_the_sa_stream(tmp_path):
    mps = _tiny_mps(str(tmp_path / "tiny.mps"))
    r = subprocess.run([MPS_TO_MA, "-o", str(tmp_path / "o.ma"), mps, "-"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"stream is not read" in r.stderr
    assert not os.path.exists(str(tmp_path / "o.ma"))


# ---- GPU: reference files -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("source,chunk_rows", [("rbwt", None), ("rbwt", "1000"), ("rbwt", "1"), ("raw", None), ("raw", "1000")])
def test_tiny_equals_reference_files(tmp_path, monkeypatch, source, chunk_rows):
    """The .ma equals the reference mps_to_ma's, the .mab the reference rb_build -m's, with any number of chunk seams."""
    if chunk_rows:
        monkeypatch.setenv("RBG_MA_CHUNK_ROWS", chunk_rows)
    mps = _tiny_mps(str(tmp_path / "tiny.mps"))
    ma, mab = str(tmp_path / "o.ma"), str(tmp_path / "o.mab")
    st = rb.build_marker_array(TINY if source == "rbwt" else RAW, mps, ma, mab)
    assert filecmp.cmp(ma, RAW + ".ma", shallow=False)
    assert filecmp.cmp(mab, TINY + ".mab", shallow=False)
    n = os.path.getsize(RAW + ".bwt")
    assert st.n == n and st.rows == n and st.phi_steps == n - st.r
    assert st.ma_records == len(_records(np.fromfile(ma, np.uint64)))
    assert sorted(os.listdir(tmp_path)) == ["o.ma", "o.mab", "tiny.mps"]      # no temporary file left behind


@pytest.mark.gpu
def test_tiny_binary(tmp_path):
    mps = _tiny_mps(str(tmp_path / "tiny.mps"))
    ma, mab = str(tmp_path / "o.ma"), str(tmp_path / "o.mab")
    r = subprocess.run([MPS_TO_MA, "-o", ma, "--mab", mab, mps, TINY], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode()
    assert b"phi steps" in r.stderr
    assert filecmp.cmp(ma, RAW + ".ma", shallow=False) and filecmp.cmp(mab, TINY + ".mab", shallow=False)


@pytest.mark.gpu
def test_mab_refuses_a_record_at_row_zero(tmp_path):
    """.mps records over the whole text give every row, row 0 included, a list: the .ma has a record at row 0, which
    rb_build -m refuses (RBG_E_FORMAT); the .ma is still written."""
    n, heads, lens, tsa = _small_arrays()
    path = str(tmp_path / "all.mps")
    np.array([0, 49, 7, 8, DELIM, 50, n - 1, 9, DELIM], np.uint64).tofile(path)
    ma, mab = str(tmp_path / "o.ma"), str(tmp_path / "o.mab")
    with pytest.raises(rb.RbgError) as e:
        rb.build_marker_array_arrays(n, heads, lens, tsa, path, ma, mab)
    assert e.value.code == -2 and "row 0" in str(e.value), str(e.value)
    recs = _records(np.fromfile(ma, np.uint64))
    assert len(recs) >= 2 and recs[0][0] == 0 and recs[-1][1] == n - 1
    assert not os.path.exists(mab)


# ---- GPU: the small benchmark index against write_raw_index ------------------------------------------------------------

@pytest.fixture(scope="module")
def small_raw(tmp_path_factory):
    """write_raw_index's files (.ma from a numpy SA) and write_mps of the `small` panel."""
    pre = str(tmp_path_factory.mktemp("small_raw") / "small")
    panel = synth.make_panel(*synth.CONFIGS["small"])
    synth.write_raw_index(panel, pre)
    synth.write_mps(panel, pre + ".mps")
    return pre


def _join(parts):
    """.ma words of consecutive row windows -> the .ma of their union (a record cut at a seam is joined again)."""
    recs = []
    for p in parts:
        for r in _records(p):
            if recs and recs[-1][1] + 1 == r[0] and recs[-1][2] == r[2]:
                recs[-1] = (recs[-1][0], r[1], r[2])
            else:
                recs.append(r)
    return np.array([x for f, l, ws in recs for x in (f, l) + ws + (DELIM,)], np.uint64)


@pytest.mark.gpu
def test_small_equals_numpy_ma(tmp_path, small_index, small_raw):
    ma, mab = str(tmp_path / "o.ma"), str(tmp_path / "o.mab")
    st = rb.build_marker_array(small_index, small_raw + ".mps", ma, mab)
    whole = np.fromfile(ma, np.uint64)
    assert np.array_equal(whole, np.fromfile(small_raw + ".ma", np.uint64))
    assert filecmp.cmp(mab, small_index + ".mab", shallow=False)
    n = os.path.getsize(small_raw + ".bwt")
    assert st.n == n and st.rows == n and st.phi_steps == n - st.r
    rng = np.random.default_rng(5)
    for split in range(3):
        cuts = [0] + sorted(rng.choice(np.arange(1, n), size=int(rng.integers(1, 6)), replace=False).tolist()) + [n]
        parts = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            p = str(tmp_path / ("w%d_%d.ma" % (split, a)))
            s = rb.build_marker_array(small_index, small_raw + ".mps", p, rows=(a, b))
            assert s.rows == b - a
            parts.append(np.fromfile(p, np.uint64))
        assert np.array_equal(_join(parts), whole), cuts


@pytest.mark.gpu
def test_small_from_raw_inputs(tmp_path, small_raw):
    ma = str(tmp_path / "o.ma")
    rb.build_marker_array(small_raw, small_raw + ".mps", ma)
    assert filecmp.cmp(ma, small_raw + ".ma", shallow=False)


# ---- GPU: synthetic indexes with positions past 2^32, against the oracle's phi -----------------------------------------

def _fill(rng, total, lo, hi):
    """Run lengths in [lo, hi] summing to total."""
    lens = rng.integers(lo, hi + 1, total // lo + 2).astype(np.int64)
    c = np.cumsum(lens)
    m = int(np.searchsorted(c, total))
    lens = lens[:m + 1]
    lens[-1] -= int(c[m]) - total
    return lens[lens > 0]


class Wide:
    """Runs of 1..64 rows around row 2^32 and at the top (the windows compared with the oracle), of 2^14..2^16 rows
    elsewhere; one toehold sample per run (r == R); a .mps whose records cover about `cover` of the text, several above
    2^32 and one ending at n - 1, with lists from a small pool (adjacent rows merge by value) and one record without words."""

    def __init__(self, n, seed, cover, n_records):
        rng = np.random.default_rng(seed)
        z = 1 << 21
        short = [((1 << 32) - z, min(n, (1 << 32) + z))]
        short = short + [(n - z, n)] if n - z > short[0][1] else [(short[0][0], n)]
        zones, at = [], 0
        for a, b in short:
            zones += ([(at, a, False)] if a > at else []) + [(a, b, True)]
            at = b
        self.lens = np.concatenate([_fill(rng, b - a, 1, 64) if sh else _fill(rng, b - a, 1 << 14, 1 << 16)
                                    for a, b, sh in zones]).astype(np.uint64)
        self.n, self.R = n, len(self.lens)
        assert int(self.lens.sum()) == n
        self.heads = synth.ACGT[np.cumsum(rng.integers(1, 4, self.R)) % 4].copy()
        cand = np.unique(rng.integers(0, n - 1, int(self.R * 1.3) + 16, dtype=np.uint64))
        pred = np.sort(rng.choice(cand, self.R - 1, replace=False))
        self.tsa = (np.append(pred, np.uint64(n - 1)).astype(np.uint64), rng.integers(0, n, self.R, dtype=np.uint64),
                    rng.integers(1, self.R + 1, self.R, dtype=np.uint64))
        self.start = np.concatenate([[0], np.cumsum(self.lens.astype(np.int64))])
        # records: ascending first, gaps of ~n / n_records, widths a fraction `cover` of the gap
        firsts = np.unique(rng.integers(0, n - 2000, n_records, dtype=np.uint64))
        nxt = np.append(firsts[1:], np.uint64(n - 1000))
        width = np.floor((nxt - firsts).astype(np.float64) * rng.uniform(0, 2 * cover, len(firsts))).astype(np.uint64)
        lasts = np.minimum(firsts + width, nxt - np.uint64(1))
        pool = [[], [7], [(5 << 60) | (1 << 40) | 3], [1, 2], [(1 << 33) + 9, 4, (3 << 60) | ((1 << 32) + 1)]]
        pick = rng.integers(0, len(pool), len(firsts))
        words = []
        for f, l, k in zip(firsts.tolist(), lasts.tolist(), pick.tolist()):
            words += [f, l] + pool[k] + [DELIM]
        words += [n - 1000, n - 1, 11, DELIM]                                   # a record ending at n - 1
        self.mps = np.array(words, np.uint64)
        assert n < 1 << 33 or np.count_nonzero(firsts > np.uint64(1 << 32)) > 1000      # at 2^32 + 1 only the last record is
        assert any(not ws for _, _, ws in _records(self.mps))
        self.orc = O.OracleIndex(F.Rlbwt(n=n, R=self.R, B=2, heads=self.heads, lens=self.lens), F.Toehold(self.R, n, *self.tsa))

    def sa_rows(self, a, b):
        """SA[a..b) from the oracle's phi: every run overlapping the window, from (samples_last[j] + 1) mod n at its last row."""
        out = np.empty(b - a, np.uint64)
        j = int(np.searchsorted(self.start, a, side="right")) - 1
        while j < self.R and self.start[j] < b:
            s, e = int(self.start[j]), int(self.start[j + 1]) - 1
            chain = self.orc.locate(s, e, (int(self.tsa[1][j]) + 1) % self.n)      # SA[e], SA[e-1], ..., SA[s]
            rows = np.arange(e, s - 1, -1)
            keep = (rows >= a) & (rows < b)
            out[rows[keep] - a] = chain[keep]
            j += 1
        return out

    def build(self, tmp_path, rows=None, name="o"):
        mps = str(tmp_path / (name + ".mps"))
        self.mps.tofile(mps)
        ma = str(tmp_path / (name + ".ma"))
        st = rb.build_marker_array_arrays(self.n, self.heads, self.lens, self.tsa, mps, ma, rows=rows)
        return st, np.fromfile(ma, np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [(1 << 32) + 1, (1 << 36) + 12345])
def test_wide_windows_against_oracle(tmp_path, n):
    w = Wide(n, seed=n % 1000, cover=0.5, n_records=200_000)
    for a, b in (((1 << 32) - 500_000, (1 << 32) + 500_000), (n - 1_000_000, n)):
        st, got = w.build(tmp_path, rows=(a, b), name="w%d" % a)
        end = min(b, n)                                                     # a window past the last row stops at n
        want = synth.ma_from_mps(w.sa_rows(a, end), a, w.mps)
        assert st.rows == end - a
        assert len(_records(want)) > 1000 and np.array_equal(got, want), (a, b)
        if end == n:
            assert _records(got)[-1][1] <= n - 1


@pytest.mark.gpu
def test_wide_full_range(tmp_path):
    """The whole 2^32 + 1 rows in one call (several chunks): every row walked, n - R phi steps; the rows around 2^32 agree
    with a window build."""
    n = (1 << 32) + 1
    w = Wide(n, seed=3, cover=1 / 8192, n_records=4000)
    st, whole = w.build(tmp_path, name="all")
    assert st.rows == n and st.phi_steps == n - w.R and st.ma_records > 0
    a, b = (1 << 32) - 500_000, (1 << 32) + 500_000
    _, part = w.build(tmp_path, rows=(a, b), name="part")
    inside = [r for r in _records(whole) if r[0] >= a and r[1] < b]
    assert [r for r in _records(part) if r[0] > a and r[1] < b - 1] == [r for r in inside if r[0] > a and r[1] < b - 1]


# ---- GPU: full-size data (skipped without data/<cfg>) ------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["c2", "c5w"])
def test_full_size_mab_equals_reference(tmp_path, cfg):
    """write_mps(panel) + this builder give the .mab the reference's write_mps + mps_to_ma + rb_build wrote."""
    pre = os.path.join(ROOT, "data", cfg, cfg)
    if not (os.path.exists(pre + ".rbwt") and os.path.exists(pre + ".tsa") and os.path.exists(pre + ".mab")):
        pytest.skip("data/%s not built" % cfg)
    mps = str(tmp_path / (cfg + ".mps"))
    synth.write_mps(synth.make_panel(*synth.CONFIGS[cfg]), mps)
    ma, mab = str(tmp_path / "o.ma"), str(tmp_path / "o.mab")
    rb.build_marker_array(pre, mps, ma, mab)
    assert filecmp.cmp(mab, pre + ".mab", shallow=False)
