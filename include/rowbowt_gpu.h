/*
 * rowbowt_gpu.h — C ABI of librowbowt_gpu.so, the B200 (sm_100a) implementation of
 * rowbowt's batched RLBWT query path (rb_align: count, -s locate, -m markers).
 *
 * The reference (alshai/rowbowt) has no FFI; the seam this library replaces is the set
 * of `RowBowt` const methods that rb_align calls per read, and the loader that feeds
 * them.  Each entry point names the reference interface it stands in for
 * (paths relative to the reference checkout).  Plain pointers and sizes only.
 *
 * Conventions carried over bit-exactly (SURVEY.md Appendix B):
 *   - ranges are inclusive [lo,hi]; the empty range is exactly (1,0)
 *   - toehold k == SA[hi]; a failed search returns (1,0) with k == 0
 *   - locations are emitted SA[hi], SA[hi-1], ..., SA[lo] (phi iteration), at most max_hits
 *   - marker words are opaque u64 (allele[63:60] | seq | pos[43:0]), window order, duplicates kept
 * There is no CPU fallback: every query runs on the GPU or fails with an error code.
 */
#ifndef ROWBOWT_GPU_H
#define ROWBOWT_GPU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rbg_index rbg_index;     /* one index resident on one GPU */
typedef struct rbg_reads rbg_reads;     /* a read batch staged in device memory */

/* error codes (0 = success). rbg_last_error() holds the message of the calling thread. */
enum {
    RBG_OK = 0,
    RBG_E_IO = -1,          /* missing / unreadable / truncated index file ("bad file" in rowbowt_io.hpp:166-169) */
    RBG_E_FORMAT = -2,      /* file does not parse as the reference's serialization */
    RBG_E_ALPHABET = -3,    /* BWT symbols outside {terminator,A,C,G,T} (build with pfbwt-f --non-acgt-to-a) */
    RBG_E_CUDA = -4,        /* CUDA runtime failure, including "no device" */
    RBG_E_ARG = -5,         /* invalid argument / mode needs a part that was not loaded */
    RBG_E_NOMEM = -6,
    RBG_E_INTERNAL = -7     /* a result failed its own check (the BWT builder's suffix-array certificate); nothing was written */
};

/* rbwt::LoadRbwtFlag, include/rowbowt_io.hpp:146-158 (same numeric values) */
enum { RBG_LOAD_NONE = 0, RBG_LOAD_SA = 1, RBG_LOAD_MA = 2, RBG_LOAD_DL = 4, RBG_LOAD_FT = 8,
       /* not a LoadRbwtFlag: the template argument of load_rowbowt<ri::fbb_string> (src/rb_align.cpp:195-202,
        * `--fbb`): <prefix>.rbwt holds a wt_fbb (include/fbb_string.hpp).  Decoded at load into the same device
        * layout; byte 1 in a read is then an absent symbol (the wt_fbb keeps the terminator as byte 0).
        * RBG_LOAD_SA is refused with RBG_E_ARG: the reference has no toehold search over fbb_string
        * (include/rowbowt_io.hpp:107, src/rb_align.cpp:110-116 leaves the toehold uninitialised). */
       RBG_LOAD_FBB = 16,
       /* not a LoadRbwtFlag: keep the finished GPU layout next to the index as <prefix>.rbgcache (written on the first open,
        * uploaded as it is by later ones: the BASELINE index opens in a few tenths of a second instead of ~2 s).  Valid only
        * for exactly these index files (size + mtime), load flags, library layout version and layout knobs; otherwise rebuilt. */
       RBG_LOAD_CACHE = 32 };

/* query modes: what rb_report asks of the index, src/rb_align.cpp:118-145 */
enum {
    RBG_COUNT = 0,          /* RowBowt::find_range                      include/rowbowt.hpp:121-131 */
    RBG_LOCATE = 1,         /* find_range_w_toehold + locs_at           include/rowbowt.hpp:169-184,613-621 ; include/toehold_sa.hpp:37-72 */
    RBG_MARKERS = 2,        /* markers_at(range) -> at_range            include/rowbowt.hpp:282-285 ; pfbwt-f/include/rle_window_array.hpp:130-154 */
    /* not a reference option: with RBG_LOCATE the locations come back NARROW -- rbg_result.locs_lo32 (low 32 bits)
     * plus, only for an index with n > 2^32, rbg_result.locs_hi8 (bits 32..39) -- instead of 8 bytes each in `locs`.
     * Location j is locs_lo32[j] | (uint64_t) locs_hi8[j] << 32.  Halves the D2H volume that bounds -s end to end. */
    RBG_NARROW_LOCS = 4,
    /* not a reference option: on an index with n <= 2^32 the ranges come back as two u32 planes, rbg_result.lo32 / hi32
     * (the empty range is still (1,0)), and rbg_result.lo / hi are NULL; ignored (u64 as usual) when n > 2^32.  8 instead
     * of 16 bytes per read leave the device: with several GPUs on one host the PCIe volume bounds the end-to-end rate. */
    RBG_NARROW_RANGES = 8
};

/* Flat description of an index (SURVEY.md Appendix B.8) for rbg_index_open_arrays.
 * Mirrors the members of rle_string (include/rle_string.hpp:385-395), ToeholdSA
 * (include/toehold_sa.hpp:157-161) and rle_window_arr (rle_window_array.hpp:258-264). */
typedef struct {
    uint64_t n, R;
    const uint8_t*  run_heads;      /* [R] BWT symbol of each run; terminator as byte 1 */
    const uint64_t* run_lens;       /* [R] */
    /* optional toehold SA (NULL/0 when absent) */
    uint64_t r;
    const uint64_t* pred;           /* [r] sorted text positions (ones of pred_) */
    const uint64_t* samples_last;   /* [r] */
    const uint64_t* pred_to_run;    /* [r] */
    /* optional marker windows */
    uint64_t n_windows, arr_size;
    uint64_t size_starts, size_ends, size_idxs;   /* bit-vector lengths: they clamp rank/select (rle_window_array.hpp:202-232) */
    const uint64_t* win_starts;     /* [n_windows] sorted */
    const uint64_t* win_ends;       /* [n_windows] sorted */
    const uint64_t* win_idxs;       /* [n_windows] sorted offsets into arr */
    const uint64_t* arr;            /* [arr_size] marker words */
} rbg_index_desc;

/* A batch of reads exactly as kseq hands them to rb_report (seq->seq.s, raw bytes,
 * no case folding): read i is bases[offsets[i] .. offsets[i+1]).  Caller-owned. */
typedef struct {
    uint64_t n_reads;
    const char* bases;
    const uint64_t* offsets;        /* [n_reads+1], offsets[0] may be non-zero */
} rbg_batch;

/* Results, library-owned pinned host memory, valid until rbg_result_free. */
typedef struct {
    uint64_t n_reads;
    uint64_t* lo;                   /* [n]   range_t.first  */
    uint64_t* hi;                   /* [n]   range_t.second */
    uint64_t* toehold;              /* [n]   LFData::ssamp (LOCATE), else NULL */
    uint64_t* loc_off;              /* [n+1] (LOCATE) locs of read i = locs[loc_off[i]..loc_off[i+1]) */
    uint64_t* locs;
    uint64_t* mk_off;               /* [n+1] (MARKERS) */
    uint64_t* markers;
    void* _owner;                   /* internal */
    uint32_t* locs_lo32;            /* (LOCATE | NARROW_LOCS) low 32 bits of every location; `locs` is NULL then */
    uint8_t*  locs_hi8;             /* ... bits 32..39, NULL when the index has n <= 2^32 */
    uint32_t* lo32;                 /* (NARROW_RANGES, n <= 2^32) range_t.first / .second as u32; `lo` and `hi` are NULL then */
    uint32_t* hi32;
} rbg_result;

/* The same batch with the bases already 2-bit packed on the host (SURVEY.md 8(f) row 2; what pack_kernel produces
 * from an rbg_batch): the base at batch byte x, counted from offsets[0] == 0, sits at bits 2*(x & 31) of
 * packed[x >> 5], A=0 C=1 G=2 T=3.  46 bytes per 150 bp read cross PCIe instead of 158.  rbg_pack_bytes fills
 * `packed` and `flags` from raw bytes exactly as the device would. */
enum {
    RBG_READ_DEAD = 1,      /* the read holds a byte that is no symbol of this index: its result is (1,0) (SURVEY.md B.1) */
    RBG_READ_EXOTIC = 2     /* the read holds byte 1 (the terminator, a legal BWT symbol without a 2-bit code): searched byte-wise */
};
typedef struct {
    uint64_t n_reads;
    const uint64_t* packed;         /* [(offsets[n_reads] + 31) / 32] */
    const uint64_t* offsets;        /* [n_reads+1], offsets[0] == 0 */
    const uint8_t* flags;           /* [n_reads] RBG_READ_*; NULL = no read flagged */
    uint64_t n_exotic;              /* reads flagged RBG_READ_EXOTIC (0 = the library need not look) */
    const char* bases;              /* raw bytes of the batch as in rbg_batch; only read for RBG_READ_EXOTIC reads, may be NULL when n_exotic == 0 */
} rbg_packed_batch;

typedef struct {
    uint64_t n, r;                  /* text length, BWT runs */
    uint64_t F[256];                /* RowBowt::f_, include/rowbowt.hpp:770-778 */
    uint64_t toehold0;              /* ToeholdSA::get_last_run_sample(), include/toehold_sa.hpp:97-99 */
    uint32_t has_sa, has_ma;
    int32_t  wsize;                 /* rle_window_arr::wsize_ */
    uint32_t window;                /* GPU layout: BWT positions per 64-byte rank-directory line */
    uint64_t n_lines;               /* 64-byte rank-directory lines (direct + raw children of cluster windows) */
    uint64_t n_cluster;             /* windows with more than 24 runs (densest stretch summarised, detail in raw children) */
    uint64_t dir_bytes, phi_bytes, toehold_bytes, marker_bytes;   /* device footprint */
    uint32_t ftab_k;                /* FTab::get_k() of the resident k-mer seed table, 0 = none */
    uint32_t layout;                /* GPU layout of the rank directory: 4 (24 runs per line + L2-resident superblock counts), 5 (20 runs, u32 counts in the line)
                                       or 7 (the BWT at 2 bits per row, 32-byte lines of 64 rows: indexes below 2^31 rows whose lines fit 32 MB) */
    uint64_t ftab_bytes;            /* seed table footprint */
    uint64_t hot_bytes;             /* superblock counts + seed table, held in one device allocation */
    uint64_t l2_pinned_bytes;       /* always 0: no persisting-L2 window is set (the field keeps the struct layout) */
    uint32_t phi_shift;             /* GPU layout: one 32-byte phi slot per 2^phi_shift text positions */
    uint32_t from_cache;            /* 1: this handle was opened from <prefix>.rbgcache (RBG_LOAD_CACHE) */
    uint64_t phi_overflow;          /* slots whose bucket holds more than 3 samples (side array, binary search) */
    uint64_t pair_bytes;            /* pair directory (two bases per LF step in the count search); 0 = not built, see RBG_PAIR */
    uint32_t pair_window;           /* its BWT positions per line */
} rbg_info;

typedef struct {
    uint64_t reads, bases;
    uint64_t lf_steps;              /* LF(range,c) executed (a2 in SURVEY §8) */
    uint64_t lf_lines;              /* distinct 64-byte rank lines those steps used (1 or 2 per step) */
    uint64_t phi_steps;             /* phi evaluations */
    uint64_t marker_words;
    float ms_pack, ms_search, ms_toehold, ms_locate, ms_markers;   /* CUDA-event time of each kernel stage, last call */
    float ms_h2d, ms_d2h, ms_total;
    uint32_t launches;              /* kernels launched by the last call */
    float ms_phi;                   /* locate_kernel alone (staged calls; ms_locate also holds the count + scan in front of it) */
} rbg_stats;

const char* rbg_last_error(void);
int rbg_device_count(void);

/* rbwt::load_rowbowt<rle_string_sd>(prefix, flags), include/rowbowt_io.hpp:176-189:
 * reads <prefix>.rbwt (+ .tsa with RBG_LOAD_SA, + .mab with RBG_LOAD_MA, + .ftab with RBG_LOAD_FT; DL is
 * host-side and ignored here), re-lays the index out for the GPU and uploads it to `device`. */
int rbg_index_open(const char* prefix, uint32_t flags, int device, rbg_index** out);
/* Same from flat arrays (tests; the RowBowt(bwt, ma, tsa, ...) constructor, include/rowbowt.hpp:33-61). */
int rbg_index_open_arrays(const rbg_index_desc* desc, int device, rbg_index** out);
void rbg_index_close(rbg_index* ix);
int rbg_index_info(const rbg_index* ix, rbg_info* info);

/* rb_build's work on the GPU (rbwt::construct_and_serialize_rowbowt<rle_string_sd>, include/rowbowt_io.hpp:49-89;
 * rle_string(fname) include/rle_string.hpp:44-97; ToeholdSA(n,r,ssa,esa) include/toehold_sa.hpp:28-36,105-156;
 * rle_window_arr(fname) pfbwt-f/include/rle_window_array.hpp:15-50).  Inputs are the builder's raw files:
 * <prefix>.bwt (one byte per row, terminator 0), with RBG_LOAD_SA <prefix>.ssa/.esa, with RBG_LOAD_MA <prefix>.ma.
 *   rbg_build_index      writes <out_prefix>.rbwt [.tsa] [.mab], byte-identical to the reference's rb_build
 *                        (sdsl serialization restated in csrc/sdsl_writer.hpp); RBG_LOAD_FT also writes
 *                        <out_prefix>.ftab for k = ftab_k (rb_build -f).  `stats` may be NULL.
 *   rbg_index_open_raw   skips the files: raw inputs -> run-length kernels -> device layout. */
typedef struct {
    uint64_t n, r;                  /* BWT length (terminator included), runs */
    double s_bwt_read;              /* fread of the .bwt into pinned memory */
    double s_rle;                   /* wall time of the run-length pass (read + H2D + kernels + D2H) */
    float  ms_rle_kernels;          /* CUDA-event time of H2D + run-length kernels */
    double s_samples;               /* .ssa/.esa -> ToeholdSA arrays (GPU radix sort) */
    double s_markers;               /* .ma -> window arrays */
    double s_write;                 /* serialization of the output files */
    double s_total;
} rbg_build_stats;
int rbg_build_index(const char* in_prefix, const char* out_prefix, uint32_t flags, uint32_t ftab_k, int device, rbg_build_stats* stats);
int rbg_index_open_raw(const char* prefix, uint32_t flags, int device, rbg_index** out);

/* mps_to_ma (pfbwt-f/src/mps_to_ma.cpp) with SA taken from the index's phi instead of a suffix-array stream: the marker
 * array (.ma) of a .mps (`first last word* ~0` records over inclusive ranges of text positions).  Row i gets the words of
 * the record whose range holds SA[i]; a .ma record is a maximal run of rows whose lists are non-empty and equal by value.
 * Index from <prefix>.rbwt + .tsa when present, else the raw <prefix>.bwt/.ssa/.esa (as rb_build --ftab-only chooses).
 * Rows [row_begin, min(row_end, n)); blocks are cut at the window edges.  mab_path may be NULL; otherwise the .mab
 * that rb_build -m would make from this .ma is written too.  Outputs are written to a temporary file and renamed.
 * Errors: no .tsa (.ssa/.esa) RBG_E_IO; r != R or an empty window RBG_E_ARG; a malformed .mps RBG_E_FORMAT naming the
 * record (checked, with the index files read, before any CUDA call except for the raw .bwt); with mab_path, a .ma
 * record at row 0 RBG_E_FORMAT as rb_build -m refuses it (the .ma is still written).
 * RBG_MA_CHUNK_ROWS in the environment caps the rows of one device pass (tests: many chunk seams). */
typedef struct {
    uint64_t n, r, rows, phi_steps;          /* rows walked in the window; phi_step calls */
    uint64_t mps_records, lists, ma_records, ma_words;
    double s_read, s_layout, s_write, s_total;
    float ms_rows_kernel, ms_blocks;          /* CUDA-event time, summed over chunks */
} rbg_ma_stats;
int rbg_build_marker_array(const char* index_prefix, const char* mps_path, const char* ma_path, const char* mab_path,
                           uint64_t row_begin, uint64_t row_end, int device, rbg_ma_stats* stats);
/* Same over flat arrays (tests): desc needs the runs and the toehold arrays with r == R; its marker fields are ignored. */
int rbg_build_marker_array_arrays(const rbg_index_desc* desc, const char* mps_path, const char* ma_path, const char* mab_path,
                                  uint64_t row_begin, uint64_t row_end, int device, rbg_ma_stats* stats);

/* The builder's raw outputs from a FASTA, on the GPU: what `pfbwt-f64 --non-acgt-to-a --print-docs -r -o P P.fa` writes and
 * rbg_build_index / rbg_build_marker_array read.  The text T is, for each record in file order, its bases followed by 10 'A's,
 * then one byte 0 (the terminator): n = sum(len + 10) + 1.
 *   <out>.bwt   n bytes, BWT[i] = T[SA[i] - 1] (0 at the row where SA[i] = 0), bases as ASCII
 *   <out>.ssa   per maximal run of equal BWT bytes, in row order: (first row, SA[first row]), two little-endian u64
 *   <out>.esa   the same with the run's last row
 *   <out>.docs  `name start` per record: the header up to the first whitespace, the offset of its first base in T
 * Input: FASTA, plain, gzip or BGZF, multi-line records joined.  Uppercase A C G T are kept, any other uppercase letter
 * becomes 'A'.  Refused before any CUDA call: a missing or unreadable file RBG_E_IO; no records, or a record without bases
 * RBG_E_FORMAT; a lowercase letter or a non-letter byte in a sequence RBG_E_ALPHABET (record and offset named: soft-masked
 * input must be uppercased first); n >= 2^40 RBG_E_ARG.  When the build does not fit the device's free memory RBG_E_NOMEM
 * (the bytes needed are named), before anything is allocated.  Outputs are written to temporary files and renamed.
 * Below 2^32 positions the build keeps positions and ranks in u32 (37 bytes of device memory per position); from 2^32 on
 * (or at any n with RBG_BWT_WIDE=1 in the environment) in u64, with the suffix array sorted in parts of at most M rows:
 * 21 bytes per position + 32 per part row + 391 MB of prefix counts + scratch, M taken from the free memory (capped by
 * RBG_BWT_PART_ROWS).  An 11-symbol prefix shared by more than M suffixes is refused with RBG_E_NOMEM naming it.  That
 * build certifies its suffix array before writing anything; a failure is RBG_E_INTERNAL naming the row.
 * rbg_build_bwt_text takes len ACGT bytes without the terminator (tests) and writes no .docs; len (n < 2^32) is checked
 * before the buffer is read.  `stats` may be NULL. */
#define RBG_BWT_MAX_ROUNDS 32
typedef struct {
    uint64_t n, r;                  /* text length (terminator included), BWT runs */
    uint64_t records;               /* FASTA records (0 for rbg_build_bwt_text) */
    uint32_t rounds;                /* prefix-doubling rounds after the initial sort by the first 27 symbols */
    uint32_t _pad;
    uint64_t max_active;            /* most suffixes one round sorted */
    uint64_t active[RBG_BWT_MAX_ROUNDS];   /* suffixes round i sorted (i < rounds): those whose group was still larger than 1 */
    double s_parse, s_sort, s_write, s_total;   /* wall time: FASTA -> text; upload, sort, BWT and samples back; file writes; all */
    float ms_sort, ms_gather;       /* CUDA-event time of the initial sort + rounds, and of the BWT gather + run boundaries + samples
                                       (the u64 build: with the copy of the BWT to the host, which its run chunks are cut by) */
    uint64_t peak_bytes;            /* device memory the build allocates (checked against the free memory first) */
    uint32_t wide;                  /* 1: u64 positions and ranks, the suffix array sorted in parts */
    uint32_t parts;                 /* parts the rows were cut into (1 for the u32 build) */
    uint64_t part_rows;             /* rows of the largest part */
    float ms_verify;                /* CUDA-event time of the suffix-array certificate (0 for the u32 build, which has none) */
    uint32_t _pad2;
} rbg_bwt_stats;
int rbg_build_bwt(const char* fasta_path, const char* out_prefix, int device, rbg_bwt_stats* stats);
int rbg_build_bwt_text(const uint8_t* text, uint64_t len, const char* out_prefix, int device, rbg_bwt_stats* stats);

/* The k-mer seed table (FTab, include/ftab.hpp:12-40).  Once resident, every query of a read of
 * at least k bases starts from the table entry of its last k bases instead of k LF steps; results
 * are identical by construction (entry = find_range(kmer), rb_tests.cpp:147-173).
 *   rbg_ftab_build   RowBowt::build_ftab(k), include/rowbowt.hpp:726-743, on the GPU (k = 0 drops the table)
 *   rbg_ftab_load    FTab::load, include/ftab.hpp:15-28 (also: RBG_LOAD_FT in rbg_index_open reads <prefix>.ftab);
 *                    entries are verified against the index, RBG_E_FORMAT on mismatch
 *   rbg_ftab_save    FTab::serialize, include/ftab.hpp:30-34 (what `rb_build --ftab` writes, byte for byte)
 *   rbg_ftab_lookup  RowBowt::search_ftab, include/rowbowt.hpp:745-758: n_kmers strings of exactly k bases,
 *                    concatenated; a miss yields (full range, consumed 0) */
int rbg_ftab_build(rbg_index* ix, uint32_t k);
int rbg_ftab_load(rbg_index* ix, const char* path);
int rbg_ftab_save(const rbg_index* ix, const char* path);
int rbg_ftab_lookup(const rbg_index* ix, const char* kmers, uint64_t n_kmers, uint64_t* lo, uint64_t* hi, uint64_t* consumed);

/* One batched call = the body of rb_align's per-read loop (src/rb_align.cpp:176-178) for
 * every read of `in`: mode is an OR of RBG_LOCATE / RBG_MARKERS (0 = count only).
 * max_hits as in locs_at (rb_align passes UINT64_MAX, src/rb_align.cpp:125).
 * Host buffers in, pinned host buffers out (H2D, kernels, D2H inside the call). */
int rbg_query(rbg_index* ix, const rbg_batch* in, uint32_t mode, uint64_t max_hits, rbg_result* out);
void rbg_result_free(rbg_result* res);
/* Calls on one handle may run concurrently from several host threads, as the reference's const RowBowt& is shared by
 * the rb_markers workers (src/rb_markers.cpp:321-326,534): each call in flight owns a "lane" (three streams, events,
 * device scratch); up to RBG_LANES (default 2) run at once, further callers wait.  rbg_ftab_build / rbg_ftab_load
 * wait for the lanes to drain.  rbg_last_stats reports the call that finished last.
 * RBG_BLOCKING_SYNC=1 in the environment (read when a lane is created): the calling thread sleeps while it waits for
 * the GPU instead of spinning -- for hosts that keep every core busy beside the caller, as rb_align does. */

/* Same call for a batch packed on the host.  Results are identical to rbg_query on the raw bytes. */
int rbg_query_packed(rbg_index* ix, const rbg_packed_batch* in, uint32_t mode, uint64_t max_hits, rbg_result* out);
/* Host-side packer (CPU, no CUDA call): batch bytes [x0, x1) of bases/offsets (offsets[0] == 0; x0 a multiple of 32)
 * -> packed[x0/32 .. ceil(x1/32)) and, OR-ed in atomically, flags[read] for bytes without a 2-bit code in THIS index.
 * Disjoint byte ranges may be packed by different threads at the same time; `flags` must start zeroed.
 * *n_exotic (may be NULL) is incremented by the number of terminator bytes seen. */
int rbg_pack_bytes(const rbg_index* ix, const char* bases, const uint64_t* offsets, uint64_t n_reads,
                   uint64_t x0, uint64_t x1, uint64_t* packed, uint8_t* flags, uint64_t* n_exotic);

/* Device-resident variant for kernel-only measurement: stage a batch once, run the
 * kernels any number of times.  Results stay on the device; `checksum` (may be NULL)
 * receives an order-independent digest of (lo,hi[,toehold,locs,markers]) for parity. */
int rbg_reads_upload(rbg_index* ix, const rbg_batch* in, rbg_reads** out);
int rbg_reads_upload_packed(rbg_index* ix, const rbg_packed_batch* in, rbg_reads** out);
int rbg_query_staged(rbg_index* ix, rbg_reads* reads, uint32_t mode, uint64_t max_hits, uint64_t* checksum);
int rbg_reads_fetch(rbg_index* ix, rbg_reads* reads, uint32_t mode, rbg_result* out);   /* D2H of the last staged run */
void rbg_reads_free(rbg_reads* reads);

int rbg_last_stats(const rbg_index* ix, rbg_stats* st);

/* ---- rb_markers: greedy-seeding marker genotyping (src/rb_markers.cpp; SURVEY.md §8(f) row 1) ----
 * One seed = one fn(range, (q.first, q.second), mbuf) call of RowBowt::get_markers_greedy_seeding
 * (include/rowbowt.hpp:406-482) as the rb_markers worker records it (MarkerSeed / out_fn,
 * src/rb_markers.cpp:255-275,356-373): markers already sorted by marker_cmp (:243-251) and
 * std::unique'd, dropped when range_size < min_range. */
typedef struct {
    uint64_t lo, hi;                /* SA range of the seed; MarkerSeed::range_size = hi - lo + 1 */
    uint64_t mk_off;                /* markers of this seed: markers[mk_off .. mk_off + mk_cnt) */
    uint32_t query_start;           /* MarkerSeed::query_start (the reference's size_t(-1) is 0xFFFFFFFF here) */
    uint32_t query_len;             /* MarkerSeed::query_len */
    uint32_t mk_raw;                /* words gathered along the seed (slots reserved at mk_off) */
    uint32_t mk_cnt;                /* words left after sort + unique */
} rbg_seed;

typedef struct {
    uint64_t wsize;                 /* --wsize     (default 19): marker query every wsize bases of a seed */
    uint64_t max_range;             /* --max-range (default 1000): no marker query for wider ranges */
    uint64_t min_range;             /* --min-range (default 0): seeds with a narrower range report no markers */
    uint32_t use_ftab;              /* --ftab: seed and re-seed through the resident k-mer table (rowbowt.hpp:430-433,454-464) */
    uint32_t _pad;
} rbg_greedy_params;

/* Library-owned pinned host memory, valid until rbg_seed_result_free.  Seeds of read i on strand s
 * (0 = the read as given, 1 = its reverse complement) are seeds[seed_off[2i+s] .. seed_off[2i+s+1]),
 * in the order the reference generates them. */
typedef struct {
    uint64_t n_reads;
    uint64_t* seed_off;             /* [2 n_reads + 1] */
    rbg_seed* seeds;
    uint64_t n_seeds;
    uint64_t* markers;
    uint64_t n_marker_words;        /* slots in `markers` (sum of mk_raw) */
    void* _owner;                   /* internal */
} rbg_seed_result;

/* The body of the rb_markers worker (src/rb_markers.cpp:375-404) for every read of `in`: bytes are
 * mapped through seq_ntoa_table (:135-152: acgt -> ACGT, n/N -> A, anything else never matches), then
 * both strands go through get_markers_greedy_seeding.  Needs RBG_LOAD_MA; use_ftab needs a resident
 * seed table with k - 1 <= wsize and every read at least k bases long (the reference exits / throws
 * there; this call returns RBG_E_ARG). */
int rbg_markers_greedy(rbg_index* ix, const rbg_batch* in, const rbg_greedy_params* params, rbg_seed_result* out);
void rbg_seed_result_free(rbg_seed_result* res);

/* Pinned host allocations for callers that want zero-copy staging of `bases`/`offsets`. */
void* rbg_host_alloc(size_t bytes);
void rbg_host_free(void* p);

/* Random 64-byte-line gather microbenchmark over `footprint_bytes` of HBM (the roofline
 * denominator of SURVEY §8(d)); returns achieved GB/s of useful lines, <0 on error.  line_bytes 32 / 64 / 128: every
 * thread reads whole lines (as the kernels do); -64: 64-byte lines read by lane pairs, one request per line;
 * iters < 0: each address depends on the data just read. */
double rbg_gather_roofline(int device, size_t footprint_bytes, int line_bytes, int iters);

/* The BWT builder's suffix-array certificate over a caller's suffix array: sa[0, len + 1) of text[0, len) (A, C, G, T) + the
 * terminator.  *first_bad = len + 1 when sa is the suffix array, else the smallest row i where sa[i] >= len + 1, sa[i]
 * appeared at an earlier row, or (T[sa[i]], rank[sa[i] + 1]) is not below (T[sa[i + 1]], rank[sa[i + 1] + 1]) -- rank being
 * the first row holding each value, the terminator the smallest symbol. */
int rbg_check_suffix_array(const uint8_t* text, uint64_t len, const uint64_t* sa, int device, uint64_t* first_bad);

/* ---- diagnostics (host only, no CUDA call): the load-time re-layout checked against the flat arrays ----------
 * Each walks the SAME decode code the kernels run (csrc/leaf.cuh, csrc/phi_slot.cuh, the ToeholdDir lookup) on the
 * host over <prefix>.rbwt / .tsa and compares with a direct computation; 0 = every probe agreed.
 *   rbg_selftest_layout   rank_c(p), rank_c(p+1) for every stride-th position of every run (window & 0xFFFF = 0: automatic;
 *                         window >> 16 = 4, 5 or 7 forces that line layout; layout 7 also checks BWT[p] as the toehold reads it)
 *   rbg_selftest_layout_runs  the same over caller-supplied runs (n, heads, lens, R); *layout = the line layout built
 *   rbg_selftest_phi      phi(i) for every stride-th text position and the neighbours of every sample
 *   rbg_selftest_toehold  the toehold sample of every run end's LF image (shift = 0: automatic bucket width)
 *   rbg_selftest_rewrite  decode + re-serialize the index files (parts: 1 .rbwt, 2 .tsa, 4 .mab, 8 .rbwt is a wt_fbb)
 *   rbg_selftest_pack     rbg_pack_bytes with an explicit byte -> code table instead of an index handle */
int rbg_selftest_layout(const char* prefix, uint32_t window, uint64_t stride, uint64_t* checked, uint64_t* n_lines, uint64_t* n_cluster);
int rbg_selftest_layout_runs(uint64_t n, const uint8_t* heads, const uint64_t* lens, uint64_t R, uint32_t window, uint64_t stride,
                             uint64_t* checked, uint64_t* n_lines, uint32_t* layout);
int rbg_selftest_phi(const char* prefix, uint32_t shift, uint64_t stride, uint64_t* checked, uint64_t* n_slots, uint64_t* n_overflow);
int rbg_selftest_toehold(const char* prefix, uint32_t shift, uint64_t* checked, uint64_t* dir_bytes);
int rbg_selftest_rewrite(const char* prefix, const char* out_prefix, uint32_t parts);
int rbg_selftest_pack(const int8_t* code_of, const char* bases, const uint64_t* offsets, uint64_t n_reads,
                      uint64_t x0, uint64_t x1, uint64_t* packed, uint8_t* flags, uint64_t* n_exotic);

#ifdef __cplusplus
}
#endif
#endif /* ROWBOWT_GPU_H */
