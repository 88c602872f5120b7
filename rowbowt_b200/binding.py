"""ctypes binding of include/rowbowt_gpu.h.  Mirrors the reference's RowBowt query
interface (include/rowbowt.hpp) at batch granularity: find_range / find_range_w_toehold
/ locs_at / markers_at become one `query(reads, mode)` call."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
RBG_COUNT, RBG_LOCATE, RBG_MARKERS, RBG_NARROW_LOCS, RBG_NARROW_RANGES = 0, 1, 2, 4, 8
RBG_READ_DEAD, RBG_READ_EXOTIC = 1, 2
RBG_LOAD_SA, RBG_LOAD_MA, RBG_LOAD_DL, RBG_LOAD_FT, RBG_LOAD_FBB, RBG_LOAD_CACHE = 1, 2, 4, 8, 16, 32
U64_MAX = 0xFFFFFFFFFFFFFFFF
u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)
u8p = C.POINTER(C.c_uint8)


class RbgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("rowbowt_gpu error %d: %s" % (code, msg))
        self.code = code


class _Desc(C.Structure):
    _fields_ = [("n", C.c_uint64), ("R", C.c_uint64), ("run_heads", C.c_void_p), ("run_lens", C.c_void_p),
                ("r", C.c_uint64), ("pred", C.c_void_p), ("samples_last", C.c_void_p), ("pred_to_run", C.c_void_p),
                ("n_windows", C.c_uint64), ("arr_size", C.c_uint64),
                ("size_starts", C.c_uint64), ("size_ends", C.c_uint64), ("size_idxs", C.c_uint64),
                ("win_starts", C.c_void_p), ("win_ends", C.c_void_p), ("win_idxs", C.c_void_p), ("arr", C.c_void_p)]


class _Batch(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("bases", C.c_void_p), ("offsets", C.c_void_p)]


class _Result(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("lo", u64p), ("hi", u64p), ("toehold", u64p), ("loc_off", u64p),
                ("locs", u64p), ("mk_off", u64p), ("markers", u64p), ("_owner", C.c_void_p),
                ("locs_lo32", u32p), ("locs_hi8", u8p), ("lo32", u32p), ("hi32", u32p)]


class _PackedBatch(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("packed", C.c_void_p), ("offsets", C.c_void_p), ("flags", C.c_void_p),
                ("n_exotic", C.c_uint64), ("bases", C.c_void_p)]


class _GreedyParams(C.Structure):
    _fields_ = [("wsize", C.c_uint64), ("max_range", C.c_uint64), ("min_range", C.c_uint64), ("use_ftab", C.c_uint32),
                ("_pad", C.c_uint32)]


class _SeedResult(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("seed_off", u64p), ("seeds", C.c_void_p), ("n_seeds", C.c_uint64),
                ("markers", u64p), ("n_marker_words", C.c_uint64), ("_owner", C.c_void_p)]


# rbg_seed (include/rowbowt_gpu.h)
SEED_DTYPE = np.dtype([("lo", "<u8"), ("hi", "<u8"), ("mk_off", "<u8"), ("qstart", "<u4"), ("qlen", "<u4"),
                       ("mk_raw", "<u4"), ("mk_cnt", "<u4")])


class Info(C.Structure):
    _fields_ = [("n", C.c_uint64), ("r", C.c_uint64), ("F", C.c_uint64 * 256), ("toehold0", C.c_uint64),
                ("has_sa", C.c_uint32), ("has_ma", C.c_uint32), ("wsize", C.c_int32), ("window", C.c_uint32),
                ("n_lines", C.c_uint64), ("n_cluster", C.c_uint64), ("dir_bytes", C.c_uint64),
                ("phi_bytes", C.c_uint64), ("toehold_bytes", C.c_uint64), ("marker_bytes", C.c_uint64),
                ("ftab_k", C.c_uint32), ("layout", C.c_uint32), ("ftab_bytes", C.c_uint64), ("hot_bytes", C.c_uint64),
                ("l2_pinned_bytes", C.c_uint64), ("phi_shift", C.c_uint32), ("from_cache", C.c_uint32),
                ("phi_overflow", C.c_uint64), ("pair_bytes", C.c_uint64), ("pair_window", C.c_uint32)]


class BuildStats(C.Structure):
    _fields_ = [("n", C.c_uint64), ("r", C.c_uint64), ("s_bwt_read", C.c_double), ("s_rle", C.c_double),
                ("ms_rle_kernels", C.c_float), ("s_samples", C.c_double), ("s_markers", C.c_double),
                ("s_write", C.c_double), ("s_total", C.c_double)]


class MaStats(C.Structure):
    _fields_ = [("n", C.c_uint64), ("r", C.c_uint64), ("rows", C.c_uint64), ("phi_steps", C.c_uint64),
                ("mps_records", C.c_uint64), ("lists", C.c_uint64), ("ma_records", C.c_uint64), ("ma_words", C.c_uint64),
                ("s_read", C.c_double), ("s_layout", C.c_double), ("s_write", C.c_double), ("s_total", C.c_double),
                ("ms_rows_kernel", C.c_float), ("ms_blocks", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


BWT_MAX_ROUNDS = 32       # RBG_BWT_MAX_ROUNDS


class BwtStats(C.Structure):
    _fields_ = [("n", C.c_uint64), ("r", C.c_uint64), ("records", C.c_uint64), ("rounds", C.c_uint32), ("_pad", C.c_uint32),
                ("max_active", C.c_uint64), ("active", C.c_uint64 * BWT_MAX_ROUNDS),
                ("s_parse", C.c_double), ("s_sort", C.c_double), ("s_write", C.c_double), ("s_total", C.c_double),
                ("ms_sort", C.c_float), ("ms_gather", C.c_float), ("peak_bytes", C.c_uint64),
                ("wide", C.c_uint32), ("parts", C.c_uint32), ("part_rows", C.c_uint64), ("ms_verify", C.c_float),
                ("_pad2", C.c_uint32)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k not in ("_pad", "_pad2", "active")}
        d["active"] = list(self.active)[:min(self.rounds, BWT_MAX_ROUNDS)]
        return d


class Stats(C.Structure):
    _fields_ = [("reads", C.c_uint64), ("bases", C.c_uint64), ("lf_steps", C.c_uint64), ("lf_lines", C.c_uint64),
                ("phi_steps", C.c_uint64), ("marker_words", C.c_uint64),
                ("ms_pack", C.c_float), ("ms_search", C.c_float), ("ms_toehold", C.c_float), ("ms_locate", C.c_float),
                ("ms_markers", C.c_float), ("ms_h2d", C.c_float), ("ms_d2h", C.c_float), ("ms_total", C.c_float),
                ("launches", C.c_uint32), ("ms_phi", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def lib_path() -> str:
    # RBG_LIB: another build of the SAME library, e.g. one made at another commit, so that bench.py or a tool can A/B
    # the two on the same inputs; never a fallback
    return os.environ.get("RBG_LIB") or os.path.join(HERE, "librowbowt_gpu.so")


_lib = None


def lib():
    """Loads librowbowt_gpu.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        p = lib_path()
        if not os.path.exists(p):
            raise RbgError(-4, "%s not built: run `python -c 'import __graft_entry__ as g; g.build()'`" % p)
        L = C.CDLL(p)
        L.rbg_last_error.restype = C.c_char_p
        L.rbg_index_open.argtypes = [C.c_char_p, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.rbg_index_open_arrays.argtypes = [C.POINTER(_Desc), C.c_int, C.POINTER(C.c_void_p)]
        L.rbg_index_open_raw.argtypes = [C.c_char_p, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.rbg_build_index.argtypes = [C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(BuildStats)]
        L.rbg_build_marker_array.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_int,
                                             C.POINTER(MaStats)]
        L.rbg_build_marker_array_arrays.argtypes = [C.POINTER(_Desc), C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint64, C.c_uint64,
                                                    C.c_int, C.POINTER(MaStats)]
        L.rbg_build_bwt.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.POINTER(BwtStats)]
        L.rbg_build_bwt_text.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p, C.c_int, C.POINTER(BwtStats)]
        L.rbg_index_close.argtypes = [C.c_void_p]
        L.rbg_index_info.argtypes = [C.c_void_p, C.POINTER(Info)]
        L.rbg_last_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.rbg_ftab_build.argtypes = [C.c_void_p, C.c_uint32]
        L.rbg_ftab_load.argtypes = [C.c_void_p, C.c_char_p]
        L.rbg_ftab_save.argtypes = [C.c_void_p, C.c_char_p]
        L.rbg_ftab_lookup.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, u64p, u64p, u64p]
        L.rbg_query.argtypes = [C.c_void_p, C.POINTER(_Batch), C.c_uint32, C.c_uint64, C.POINTER(_Result)]
        L.rbg_result_free.argtypes = [C.POINTER(_Result)]
        L.rbg_query_packed.argtypes = [C.c_void_p, C.POINTER(_PackedBatch), C.c_uint32, C.c_uint64, C.POINTER(_Result)]
        L.rbg_pack_bytes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p,
                                     C.c_void_p, u64p]
        L.rbg_reads_upload_packed.argtypes = [C.c_void_p, C.POINTER(_PackedBatch), C.POINTER(C.c_void_p)]
        L.rbg_markers_greedy.argtypes = [C.c_void_p, C.POINTER(_Batch), C.POINTER(_GreedyParams), C.POINTER(_SeedResult)]
        L.rbg_seed_result_free.argtypes = [C.POINTER(_SeedResult)]
        L.rbg_reads_upload.argtypes = [C.c_void_p, C.POINTER(_Batch), C.POINTER(C.c_void_p)]
        L.rbg_query_staged.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, u64p]
        L.rbg_reads_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(_Result)]
        L.rbg_reads_free.argtypes = [C.c_void_p]
        L.rbg_host_alloc.restype = C.c_void_p
        L.rbg_host_alloc.argtypes = [C.c_size_t]
        L.rbg_host_free.argtypes = [C.c_void_p]
        L.rbg_gather_roofline.restype = C.c_double
        L.rbg_gather_roofline.argtypes = [C.c_int, C.c_size_t, C.c_int, C.c_int]
        L.rbg_check_suffix_array.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, u64p]
        L.rbg_selftest_layout.argtypes = [C.c_char_p, C.c_uint32, C.c_uint64, u64p, u64p, u64p]
        L.rbg_selftest_layout_runs.argtypes = [C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, u64p, u64p,
                                               C.POINTER(C.c_uint32)]
        L.rbg_selftest_phi.argtypes = [C.c_char_p, C.c_uint32, C.c_uint64, u64p, u64p, u64p]
        L.rbg_selftest_rewrite.argtypes = [C.c_char_p, C.c_char_p, C.c_uint32]
        L.rbg_selftest_toehold.argtypes = [C.c_char_p, C.c_uint32, u64p, u64p]
        L.rbg_selftest_pair.argtypes = [C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, C.c_void_p, u64p, u64p, u64p]
        L.rbg_selftest_pack.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p,
                                        C.c_void_p, u64p]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise RbgError(rc, lib().rbg_last_error().decode(errors="replace"))


def _as_batch(reads):
    """list[bytes] | uint8[n,m] | (bases uint8[], offsets uint64[n+1]) -> (_Batch, keepalive)"""
    if isinstance(reads, tuple):
        bases, offs = reads
    elif isinstance(reads, np.ndarray) and reads.ndim == 2:
        n, m = reads.shape
        bases = np.ascontiguousarray(reads).reshape(-1)
        offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(m)
    else:
        lens = np.fromiter((len(r) for r in reads), dtype=np.uint64, count=len(reads))
        offs = np.zeros(len(reads) + 1, dtype=np.uint64)
        np.cumsum(lens, out=offs[1:])
        bases = np.frombuffer(b"".join(reads), dtype=np.uint8)
    if bases.size == 0:
        bases = np.zeros(1, np.uint8)
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    b = _Batch(len(offs) - 1, bases.ctypes.data, offs.ctypes.data)
    return b, (bases, offs)


class QueryResult:
    """numpy copies of one rbg_result (lo, hi[, toehold, loc_off, locs][, mk_off, markers])."""

    def __init__(self, res: _Result, mode: int):
        n = res.n_reads
        take = lambda p, m: np.ctypeslib.as_array(p, shape=(m,)).copy() if m else np.zeros(0, np.uint64)
        self.n = n
        self.narrow_ranges = bool(res.lo32)          # RBG_NARROW_RANGES on an index with n <= 2^32: u32 planes on the wire
        if self.narrow_ranges:
            assert not res.lo and not res.hi
            widen = lambda p: np.ctypeslib.as_array(p, shape=(n,)).astype(np.uint64) if n else np.zeros(0, np.uint64)
            self.lo, self.hi = widen(res.lo32), widen(res.hi32)
        else:
            self.lo, self.hi = take(res.lo, n), take(res.hi, n)
        self.toehold = self.loc_off = self.locs = self.mk_off = self.markers = None
        if mode & RBG_LOCATE:
            self.toehold = take(res.toehold, n)
            self.loc_off = np.ctypeslib.as_array(res.loc_off, shape=(n + 1,)).copy()
            m = int(self.loc_off[n])
            if mode & RBG_NARROW_LOCS:        # widen: locs_lo32 | locs_hi8 << 32
                self.locs = np.ctypeslib.as_array(res.locs_lo32, shape=(m,)).astype(np.uint64) if m else np.zeros(0, np.uint64)
                self.narrow_bytes = 4
                if m and res.locs_hi8:
                    self.locs |= np.ctypeslib.as_array(res.locs_hi8, shape=(m,)).astype(np.uint64) << np.uint64(32)
                    self.narrow_bytes = 5
                assert not res.locs
            else:
                self.locs = take(res.locs, m)
        if mode & RBG_MARKERS:
            self.mk_off = np.ctypeslib.as_array(res.mk_off, shape=(n + 1,)).copy()
            self.markers = take(res.markers, int(self.mk_off[n]))


def build_index(in_prefix: str, out_prefix: str, sa: bool = False, markers: bool = False, ftab_k: int = 0, device: int = 0) -> "BuildStats":
    """rb_build on the GPU (rbwt::construct_and_serialize_rowbowt, include/rowbowt_io.hpp:49-89): <in>.bwt[.ssa/.esa/.ma]
    -> <out>.rbwt[.tsa/.mab/.ftab], byte-identical to the reference builder's files."""
    st = BuildStats()
    flags = (RBG_LOAD_SA if sa else 0) | (RBG_LOAD_MA if markers else 0) | (RBG_LOAD_FT if ftab_k else 0)
    _check(lib().rbg_build_index(in_prefix.encode(), out_prefix.encode(), flags, ftab_k, device, C.byref(st)))
    return st


def build_bwt(fasta: str, out_prefix: str, device: int = 0) -> "BwtStats":
    """pfbwt-f64 --non-acgt-to-a --print-docs -r on the GPU: a FASTA (plain, gzip or BGZF) -> <out>.bwt/.ssa/.esa/.docs, the
    files rb_build reads.  The text is every record followed by 10 'A's, then the terminator; it must have n < 2^40 (from
    2^32 on, u64 positions and the suffix array sorted in parts: `stats.wide`)."""
    st = BwtStats()
    _check(lib().rbg_build_bwt(fasta.encode(), out_prefix.encode(), device, C.byref(st)))
    return st


def build_bwt_text(text: np.ndarray, out_prefix: str, device: int = 0) -> "BwtStats":
    """The same for one ACGT text (uint8 ASCII, without the terminator, which is appended): <out>.bwt/.ssa/.esa, no .docs."""
    t = np.ascontiguousarray(text, np.uint8)
    st = BwtStats()
    _check(lib().rbg_build_bwt_text(t.ctypes.data, len(t), out_prefix.encode(), device, C.byref(st)))
    return st


def check_suffix_array(text: np.ndarray, sa: np.ndarray, device: int = 0) -> int:
    """The BWT builder's suffix-array certificate on the GPU over sa (len(text) + 1 values) of an ACGT text + terminator:
    len(sa) when sa is its suffix array, else the smallest failing row (rbg_check_suffix_array)."""
    t = np.ascontiguousarray(text, np.uint8)
    a = np.ascontiguousarray(sa, np.uint64)
    if len(a) != len(t) + 1:
        raise ValueError("sa must hold len(text) + 1 values")
    bad = C.c_uint64(0)
    _check(lib().rbg_check_suffix_array(t.ctypes.data, len(t), a.ctypes.data, device, C.byref(bad)))
    return bad.value


def _ma_window(rows):
    return (0, U64_MAX) if rows is None else (int(rows[0]), int(rows[1]))


def build_marker_array(prefix: str, mps: str, ma: str, mab: str | None = None, rows=None, device: int = 0) -> "MaStats":
    """mps_to_ma on the GPU: <mps> -> <ma> (and, with `mab`, the .mab rb_build -m makes from it), SA taken from the index's
    phi (<prefix>.rbwt + .tsa, else the raw <prefix>.bwt/.ssa/.esa).  rows = (begin, end): only rows [begin, min(end, n))."""
    st = MaStats()
    r0, r1 = _ma_window(rows)
    _check(lib().rbg_build_marker_array(prefix.encode(), mps.encode(), ma.encode(), mab.encode() if mab else None, r0, r1, device,
                                        C.byref(st)))
    return st


def build_marker_array_arrays(n, heads, lens, tsa, mps: str, ma: str, mab: str | None = None, rows=None,
                              device: int = 0) -> "MaStats":
    """The same over flat arrays: runs (heads, lens) and tsa = (pred, samples_last, pred_to_run) with one sample per run."""
    keep = [np.ascontiguousarray(heads, np.uint8), np.ascontiguousarray(lens, np.uint64)] + [np.ascontiguousarray(x, np.uint64) for x in tsa]
    d = _Desc()
    d.n, d.R, d.r = int(n), len(keep[0]), len(keep[2])
    d.run_heads, d.run_lens, d.pred, d.samples_last, d.pred_to_run = (x.ctypes.data for x in keep)
    st = MaStats()
    r0, r1 = _ma_window(rows)
    _check(lib().rbg_build_marker_array_arrays(C.byref(d), mps.encode(), ma.encode(), mab.encode() if mab else None, r0, r1, device,
                                               C.byref(st)))
    return st


class StagedReads:
    def __init__(self, ix: "GpuIndex", handle):
        self.ix, self.h = ix, handle

    def free(self):
        if self.h:
            lib().rbg_reads_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class GpuIndex:
    """One index resident on one GPU: load_rowbowt (include/rowbowt_io.hpp:176-189) + RowBowt's
    const query methods (include/rowbowt.hpp) at batch granularity."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def open(cls, prefix: str, sa: bool = False, markers: bool = False, device: int = 0, ftab: bool = False,
             fbb: bool = False, cache: bool = False) -> "GpuIndex":
        h = C.c_void_p()
        flags = ((RBG_LOAD_SA if sa else 0) | (RBG_LOAD_MA if markers else 0) | (RBG_LOAD_FT if ftab else 0) | (RBG_LOAD_FBB if fbb else 0) |
                 (RBG_LOAD_CACHE if cache else 0))
        _check(lib().rbg_index_open(prefix.encode(), flags, device, C.byref(h)))
        return cls(h)

    @classmethod
    def open_raw(cls, prefix: str, sa: bool = False, markers: bool = False, device: int = 0) -> "GpuIndex":
        """Straight from rb_build's inputs (<prefix>.bwt, .ssa/.esa, .ma): run-length kernels -> device layout."""
        h = C.c_void_p()
        flags = (RBG_LOAD_SA if sa else 0) | (RBG_LOAD_MA if markers else 0)
        _check(lib().rbg_index_open_raw(prefix.encode(), flags, device, C.byref(h)))
        return cls(h)

    @classmethod
    def from_arrays(cls, n, heads, lens, tsa=None, ma=None, device: int = 0) -> "GpuIndex":
        """tsa = (pred, samples_last, pred_to_run); ma = (starts, ends, idxs, arr, size_starts, size_ends, size_idxs)"""
        keep = [np.ascontiguousarray(heads, np.uint8), np.ascontiguousarray(lens, np.uint64)]
        d = _Desc()
        d.n, d.R = int(n), len(keep[0])
        d.run_heads, d.run_lens = keep[0].ctypes.data, keep[1].ctypes.data
        if tsa is not None:
            a = [np.ascontiguousarray(x, np.uint64) for x in tsa]
            keep += a
            d.r = len(a[0])
            d.pred, d.samples_last, d.pred_to_run = (x.ctypes.data for x in a)
        if ma is not None:
            a = [np.ascontiguousarray(x, np.uint64) for x in ma[:4]]
            keep += a
            d.n_windows, d.arr_size = len(a[0]), len(a[3])
            d.win_starts, d.win_ends, d.win_idxs, d.arr = (x.ctypes.data for x in a)
            d.size_starts, d.size_ends, d.size_idxs = (int(x) for x in ma[4:7])
        h = C.c_void_p()
        _check(lib().rbg_index_open_arrays(C.byref(d), device, C.byref(h)))
        return cls(h)

    def close(self):
        if self.h:
            lib().rbg_index_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self) -> Info:
        i = Info()
        _check(lib().rbg_index_info(self.h, C.byref(i)))
        return i

    # FTab (include/ftab.hpp) -------------------------------------------------------------------
    def build_ftab(self, k: int = 10) -> None:
        """RowBowt::build_ftab(k) on the GPU; k = 0 drops the table.  Queries use it from then on."""
        _check(lib().rbg_ftab_build(self.h, k))

    def load_ftab(self, path: str) -> None:
        _check(lib().rbg_ftab_load(self.h, path.encode()))

    def save_ftab(self, path: str) -> None:
        _check(lib().rbg_ftab_save(self.h, path.encode()))

    def search_ftab(self, kmers):
        """RowBowt::search_ftab for a list of k-mers (bytes, each exactly k long) -> (lo, hi, consumed)."""
        n = len(kmers)
        lo, hi, used = (np.zeros(n, np.uint64) for _ in range(3))
        _check(lib().rbg_ftab_lookup(self.h, b"".join(kmers), n, lo.ctypes.data_as(u64p), hi.ctypes.data_as(u64p),
                                     used.ctypes.data_as(u64p)))
        return lo, hi, used

    def stats(self) -> Stats:
        s = Stats()
        _check(lib().rbg_last_stats(self.h, C.byref(s)))
        return s

    def query(self, reads, mode: int = RBG_COUNT, max_hits: int = U64_MAX) -> QueryResult:
        b, keep = _as_batch(reads)
        res = _Result()
        _check(lib().rbg_query(self.h, C.byref(b), mode, max_hits, C.byref(res)))
        try:
            return QueryResult(res, mode)
        finally:
            lib().rbg_result_free(C.byref(res))

    def query_raw(self, batch, mode: int, max_hits: int = U64_MAX) -> None:
        """rbg_query / rbg_query_packed + rbg_result_free without copying results into numpy (timing loops)."""
        res = _Result()
        if isinstance(batch, _PackedBatch):
            _check(lib().rbg_query_packed(self.h, C.byref(batch), mode, max_hits, C.byref(res)))
        else:
            _check(lib().rbg_query(self.h, C.byref(batch), mode, max_hits, C.byref(res)))
        lib().rbg_result_free(C.byref(res))

    # 2-bit packed batches (rbg_packed_batch) ------------------------------------------------------
    def pack(self, reads, threads: int = 1, out=None):
        """rbg_pack_bytes over the whole batch -> (_PackedBatch, keepalive).  `out` = (packed uint64[], flags uint8[])
        preallocated (e.g. pinned) buffers; `threads` byte ranges are packed concurrently."""
        b, keep = _as_batch(reads)
        bases, offs = keep
        if offs[0] != 0:
            bases, offs = bases[int(offs[0]):], offs - offs[0]
        n, n_bytes = len(offs) - 1, int(offs[-1])
        words = (n_bytes + 31) // 32
        packed, flags = out if out is not None else (np.zeros(words + 1, np.uint64), np.zeros(n + 8, np.uint8))
        flags[:n] = 0
        ex = C.c_uint64(0)
        cuts = [min(n_bytes, ((n_bytes * t // threads) + 31) // 32 * 32) for t in range(threads)] + [n_bytes]

        def job(t):
            _check(lib().rbg_pack_bytes(self.h, bases.ctypes.data, offs.ctypes.data, n, cuts[t], cuts[t + 1],
                                        packed.ctypes.data, flags.ctypes.data, C.byref(ex)))
        if threads > 1:
            import concurrent.futures as cf
            with cf.ThreadPoolExecutor(threads) as ex_:
                list(ex_.map(job, range(threads)))
        else:
            job(0)
        n_exotic = int(np.count_nonzero(flags[:n] & RBG_READ_EXOTIC)) if ex.value else 0
        pb = _PackedBatch(n, packed.ctypes.data, offs.ctypes.data, flags.ctypes.data, n_exotic, bases.ctypes.data)
        return pb, (packed, flags, bases, offs)

    def query_packed(self, reads, mode: int = RBG_COUNT, max_hits: int = U64_MAX, threads: int = 1) -> QueryResult:
        pb, keep = self.pack(reads, threads)
        res = _Result()
        _check(lib().rbg_query_packed(self.h, C.byref(pb), mode, max_hits, C.byref(res)))
        try:
            return QueryResult(res, mode)
        finally:
            lib().rbg_result_free(C.byref(res))

    def upload_packed(self, reads, threads: int = 1) -> "StagedReads":
        pb, keep = self.pack(reads, threads)
        h = C.c_void_p()
        _check(lib().rbg_reads_upload_packed(self.h, C.byref(pb), C.byref(h)))
        return StagedReads(self, h)

    def markers_greedy(self, reads, wsize: int = 19, max_range: int = 1000, min_range: int = 0, use_ftab: bool = False):
        """The rb_markers worker (src/rb_markers.cpp:347-415) for a batch: both strands of every read through
        get_markers_greedy_seeding (include/rowbowt.hpp:406-482).  Returns (seed_off uint64[2n+1], seeds SEED_DTYPE[],
        markers uint64[]); the defaults are rb_markers' own (RbAlignArgs, src/rb_markers.cpp:21-39)."""
        b, keep = _as_batch(reads)
        gp = _GreedyParams(wsize, max_range, min_range, 1 if use_ftab else 0, 0)
        res = _SeedResult()
        _check(lib().rbg_markers_greedy(self.h, C.byref(b), C.byref(gp), C.byref(res)))
        try:
            n = res.n_reads
            seed_off = np.ctypeslib.as_array(res.seed_off, shape=(2 * n + 1,)).copy()
            if res.n_seeds:
                raw = (C.c_uint8 * (res.n_seeds * SEED_DTYPE.itemsize)).from_address(res.seeds)
                seeds = np.frombuffer(raw, dtype=SEED_DTYPE).copy()
            else:
                seeds = np.zeros(0, SEED_DTYPE)
            words = (np.ctypeslib.as_array(res.markers, shape=(res.n_marker_words,)).copy() if res.n_marker_words
                     else np.zeros(0, np.uint64))
            return seed_off, seeds, words
        finally:
            lib().rbg_seed_result_free(C.byref(res))

    # RowBowt-shaped conveniences ------------------------------------------------------------
    def find_range(self, reads):
        r = self.query(reads, RBG_COUNT)
        return r.lo, r.hi

    def find_range_w_toehold(self, reads):
        r = self.query(reads, RBG_LOCATE, max_hits=0)
        return r.lo, r.hi, r.toehold

    # device-resident path ----------------------------------------------------------------------
    def upload(self, reads) -> StagedReads:
        b, keep = _as_batch(reads)
        h = C.c_void_p()
        _check(lib().rbg_reads_upload(self.h, C.byref(b), C.byref(h)))
        return StagedReads(self, h)

    def query_staged(self, staged: StagedReads, mode: int = RBG_COUNT, max_hits: int = U64_MAX, checksum: bool = False):
        cs = C.c_uint64(0)
        _check(lib().rbg_query_staged(self.h, staged.h, mode, max_hits, C.byref(cs) if checksum else None))
        return cs.value if checksum else None

    def fetch(self, staged: StagedReads, mode: int) -> QueryResult:
        res = _Result()
        _check(lib().rbg_reads_fetch(self.h, staged.h, mode, C.byref(res)))
        try:
            return QueryResult(res, mode)
        finally:
            lib().rbg_result_free(C.byref(res))


_M1, _M2, _G = 0xBF58476D1CE4E5B9, 0x94D049BB133111EB, 0x9E3779B97F4A7C15


def _mix(z):
    z = (z + np.uint64(_G))
    z = (z ^ (z >> np.uint64(30))) * np.uint64(_M1)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(_M2)
    return z ^ (z >> np.uint64(31))


def _digest(tag, vals):
    vals = np.asarray(vals, dtype=np.uint64)
    idx = np.arange(len(vals), dtype=np.uint64)
    with np.errstate(over="ignore"):
        return int(_mix(_mix(vals) ^ (idx * np.uint64(_G) + np.uint64(tag))).sum(dtype=np.uint64))


def result_checksum(lo, hi, toehold=None, loc_off=None, locs=None, mk_off=None, markers=None) -> int:
    """Host restatement of the device digest (csrc/kernels.cu checksum_kernel) so that any
    reference result (oracle or rb_align) can be compared with a device-resident one."""
    s = _digest(1, lo) + _digest(2, hi)
    if toehold is not None:
        s += _digest(3, toehold)
    if loc_off is not None:
        s += _digest(4, np.diff(np.asarray(loc_off, dtype=np.uint64))) + _digest(5, locs)
    if mk_off is not None:
        s += _digest(7, np.diff(np.asarray(mk_off, dtype=np.uint64))) + _digest(6, markers)
    return s & U64_MAX
