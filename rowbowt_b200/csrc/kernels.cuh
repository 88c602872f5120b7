// Kernel launch wrappers (definitions in kernels.cu).  All launches go to the given stream.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "device_index.cuh"

namespace rbg {

// per-read flags written by the pack kernel
enum : uint32_t {
    kReadDead = 1,      // contains a byte that is not a BWT symbol -> result (1,0) (SURVEY Appendix B.1)
    kReadExotic = 2     // contains the terminator byte (1): searched by the byte-wise kernel
};

struct CodeTable {
    int8_t code_of[256];
    uint32_t plain;     // set by launch_pack: 'A','C','G','T' -> 0,1,2,3 (pack_kernel's arithmetic fast path applies)
};

struct DevCounters {    // accumulated with atomics by the kernels
    unsigned long long lf_steps, lf_lines, phi_steps, marker_words, checksum;
    unsigned long long cursor[64];      // search_kernel: reads handed out so far, one slot per launch of a call (zeroed with the rest)
    unsigned long long loc_cursor[64];  // locate_draw_kernel: the same for the chains of a launch
};

struct DevBatch {
    const uint8_t* bases;       // raw bytes, read i = bases[offs[i]..offs[i+1])
    const uint64_t* offs;       // [n_reads+1], offs[0] == 0
    uint64_t n_reads;
    uint64_t n_bytes;
    uint64_t r0, r1;            // the reads this launch works on: [r0, r1) (a chunk of the batch, or all of it)
    uint64_t* packed;           // 2-bit codes: base at byte x -> bits 2*(x&31) of packed[x>>5]
    uint8_t* flags;             // [n_reads] kReadDead / kReadExotic (buffer padded to a multiple of 4 bytes)
    uint32_t* bad;              // optional (greedy seeding): bit x&31 of bad[x>>5] = byte x has no 2-bit code; flags stay untouched
};

struct DevResult {
    uint64_t *lo, *hi, *toehold;        // [n_reads]
    uint64_t *loc_cnt, *loc_off, *locs; // [n_reads], [n_reads+1], [total]
    uint32_t* locs_lo;                  // narrow form of the locations (RBG_NARROW_LOCS): low 32 bits ...
    uint8_t* locs_hi;                   // ... and bits 32..39, null when n <= 2^32; locs is unused then
    uint64_t *mk_cnt, *mk_off, *markers;
    uint64_t *mk_first;                 // [n_reads] first window index
};

// grid size for `work_items` threads of work: enough CTAs, at most per_sm per SM
int grid_for(uint64_t work_items, int block, int per_sm);

int launch_pack(const DevBatch& b, const CodeTable& ct, uint64_t approx_bytes, cudaStream_t st);   // reads [b.r0, b.r1)
int launch_search(const DevLeafDir& D, const DevPairDir& PD, const DevToehold* T, const DevFtab& ft, const DevBatch& b, const DevResult& r,
                  DevCounters* ctr, unsigned long long* cursor, cudaStream_t st);     // T == nullptr -> count only (on PD when PD.lines is set); ft.k == 0 -> no seed table; cursor: zeroed device counter of this launch; returns #launches
int launch_ftab_build(const DevLeafDir& D, uint32_t k, bool toehold, ulonglong2* range, uint64_t* toe, cudaStream_t st);
int launch_search_bytes(const DevLeafDir& D, const DevToehold* T, const DevBatch& b, const DevResult& r,
                        const CodeTable& ct, DevCounters* ctr, cudaStream_t st);   // reads flagged kReadExotic
int launch_locate_counts(const DevResult& r, uint64_t r0, uint64_t r1, uint64_t max_hits, cudaStream_t st);
// n_locs: locations reads [r0, r1) will produce (chooses the static or the drawing kernel); force_draw: 0 / 1 forces the static /
// drawing kernel, -1 lets n_locs choose; cursor: zeroed device counter of this launch
int launch_locate(const DevPhi& P, const DevResult& r, uint64_t r0, uint64_t r1, uint64_t n_locs, int force_draw, DevCounters* ctr,
                  unsigned long long* cursor, cudaStream_t st);
int launch_marker_counts(const DevMarkers& M, const DevResult& r, uint64_t r0, uint64_t r1, cudaStream_t st);
int launch_marker_gather(const DevMarkers& M, const DevResult& r, uint64_t r0, uint64_t r1, DevCounters* ctr, cudaStream_t st);
// exclusive prefix sum of cnt[0..n) into off[0..n], total in off[n]
int launch_scan(const uint64_t* cnt, uint64_t* off, uint64_t n, void* tmp, size_t tmp_bytes, cudaStream_t st);
size_t scan_tmp_bytes(uint64_t n);
int launch_scan_from(const uint64_t* cnt, uint64_t* off, uint64_t n, const uint64_t* init, void* tmp, size_t tmp_bytes, cudaStream_t st);
size_t scan_from_tmp_bytes(uint64_t n);
int launch_checksum(const DevResult& r, uint64_t n_reads, bool toehold, bool locs, bool markers,
                    DevCounters* ctr, cudaStream_t st);
// lo / hi of reads [r0, r1) as u32 planes (narrow.cu)
int launch_narrow_ranges(const uint64_t* lo, const uint64_t* hi, uint32_t* lo32, uint32_t* hi32, uint64_t r0, uint64_t r1, cudaStream_t st);
void launch_stall(unsigned long long ns, cudaStream_t st);      // narrow.cu: test scaffolding
// random-gather microbenchmark; returns elapsed ms for `iters` rounds of grid*block lines each
float run_gather(const uint32_t* buf, uint64_t n_lines, int line_bytes, int iters, int dependent, uint64_t* lines_done,
                 cudaStream_t st);

// ---- rb_markers greedy seeding (greedy.cu) --------------------------------------------------------
struct GreedyParams {
    uint64_t wsize, max_range, min_range;
    uint32_t k;                 // k of the seed table to use, 0 = none
};

struct DevSeed {                // == rbg_seed (include/rowbowt_gpu.h)
    uint64_t lo, hi, mk_off;
    uint32_t query_start, query_len, mk_raw, mk_cnt;
};

struct DevSeedOut {
    uint64_t *item_seeds, *item_words;      // [2 n_reads + 1] per (read, strand): seeds / raw marker words (count pass)
    uint64_t *seed_off, *word_off;          // [2 n_reads + 1] their exclusive prefix sums
    DevSeed* seeds;
    uint64_t* words;
};

// get_markers_greedy_seeding over both strands of reads [b.r0, b.r1); emit == false only counts
int launch_greedy(const DevLeafDir& D, const DevFtab& ft, const DevMarkers& M, const DevBatch& b, const GreedyParams& P,
                  const DevSeedOut& o, bool emit, DevCounters* ctr, cudaStream_t st);
// std::sort(marker_cmp) + std::unique of every seed's words, in place
int launch_seed_sort(const DevSeedOut& o, uint64_t n_seeds, cudaStream_t st);

}  // namespace rbg
