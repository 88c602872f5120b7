// Load-time re-layout of the run-length BWT and its locate structures for the GPU.
//
// The reference answers rank_c(i) (include/rle_string.hpp:131-161) with ~10 dependent
// probes into sd_vectors and a wavelet tree.  Here the same function is answered from
// ONE 64-byte line whose address is computed from i alone: BWT position i lives in line
// i / W ("mixed leaf", leaf.cuh: all four symbols, 2 bytes per run), plus one u64 per symbol
// from a small superblock array that stays in L2.  No table in front, no per-symbol
// structure: the whole directory is ~3.8 bytes per BWT run, which keeps the BASELINE index
// (r = 41 M runs) well inside the 256 MB the SM TLBs reach and most of it in L2.
// Windows with more than 24 runs (variant clusters) keep a sorted summary of their densest
// stretch and point to RAW child lines (2 bits per position) behind the direct lines.
//
// Toehold / phi structures are sorted arrays with a radix bucket table in front (PredTable).
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "formats.hpp"
#include "leaf.cuh"

namespace rbg {

struct alphabet_error : std::runtime_error { using std::runtime_error::runtime_error; };

constexpr int kLineWords = 16;          // 64-byte lines
constexpr uint32_t kMinWindow = 16;
constexpr uint32_t kMaxWindow = 32767;  // starts are u16 and values >= 0x8000 must read as "unused"
constexpr int kMaxTerm = 8;             // terminator positions carried in kernel params
constexpr int kMaxSuper5 = 256;         // layout 5: superblocks of 2^32 positions at most, n < 2^40
// Layout 7 (plain 2-bit lines, leaf.cuh) is the automatic choice while its lines stay this small: resident in L2, where the
// search is bound by instructions and a plain rank takes far fewer than a run-length decode.  Needs n < 2^31.
constexpr uint64_t kPlainMaxBytes = 32ull << 20;

struct LeafDir {
    uint64_t n = 0;
    int version = 4;                     // leaf.cuh LeafFmt: 4 (24 entries, u16 counts, L2-resident superblock array) or 5 (20 entries,
                                         // u32 counts); 7: plain 2-bit lines of 64 rows (n_super = 1, super all zero, no children)
    uint32_t window = 0;                 // W: BWT positions per direct line
    uint64_t magic = 0;                  // floor(2^64 / W) + 1: i / W == umul64hi(i, magic) for i * W < 2^64
    uint32_t sb_shift = 0;               // a superblock is 2^sb_shift windows (<= 65535 positions; layout 5: <= 2^32)
    uint64_t n_direct = 0;               // ceil(n / W)
    uint64_t n_super = 0;                // ceil(n_direct / 2^sb_shift)
    uint64_t n_cluster = 0;              // windows with a collapsed stretch (CLUSTER lines)
    std::vector<uint32_t> lines;         // [(n_direct + raw children) * 16]; layout 7: [n_direct * 8]
    std::vector<uint64_t> super;         // [4][n_super]: F[c] + #c in BWT[0, superblock_start) (layout 5: at most 4 x 256, kept in shared memory)
    uint64_t line_words() const { return version == 7 ? kPlainWords : kLineWords; }
    uint64_t n_lines() const { return lines.size() / line_words(); }
    uint64_t F[256] = {0};               // RowBowt::build_f (include/rowbowt.hpp:770-778), by byte value
    uint64_t Fcode[4] = {0, 0, 0, 0};    // F of A,C,G,T
    uint64_t count[4] = {0, 0, 0, 0};    // occurrences of A,C,G,T
    int8_t code_of[256];                 // byte -> 0..3, 4 = terminator (byte 1) present, -1 = not in the BWT
    uint32_t n_term = 0;
    uint64_t term_pos[kMaxTerm] = {0};
};

// Validates the alphabet and builds the rank directory.  window = 0 -> choose automatically; layout = 4, 5 or 7 forces that
// line format; 0 -> 7 when n < 2^31, its lines fit kPlainMaxBytes and no window is forced, else 5 while the directory
// stays small, else 4.
LeafDir build_leaf_dir(const RunsBwt& bwt, uint32_t window, int layout);

// Pair directory (leaf.cuh, LeafFmt<6>): a rank directory over P[j] = (BWT[LF(j)], BWT[j]) with which the count search
// takes two bases per LF step.  Built from the runs alone: the rows of BWT run k map under LF onto one contiguous interval
// of rows, and the first symbols of their pairs are the BWT over that interval -- so the runs of P are each run's image
// interval cut at BWT run boundaries (R2 <= 2R + a few).
struct PairDir {
    uint64_t n = 0;
    uint32_t window = 0;                 // even, <= kPairMaxWindow
    uint32_t sb_shift = 0;               // a superblock is 2^sb_shift windows, (2^sb_shift - 1) * window <= 65535
    uint64_t n_direct = 0, n_super = 0, n_cluster = 0, n_runs = 0;
    std::vector<uint32_t> lines;         // [(n_direct + raw children) * 16]
    std::vector<uint32_t> super;         // [16][n_super]: K[p] + #p in P[0, superblock_start)
    uint32_t n_bad = 0;
    uint32_t bad_pos[kPairMaxBad] = {0}; // rows whose pair holds the terminator, ascending (stored as code 0)
    uint64_t bytes() const { return lines.size() * 4 + super.size() * 4; }
};
// Runs of P in row order: code 0..15, or kPairBad for a row whose pair holds the terminator.
constexpr uint8_t kPairBad = 16;
void pair_runs(const RunsBwt& bwt, const LeafDir& d, std::vector<uint32_t>& lens, std::vector<uint8_t>& codes);
// window = 0 -> choose.  Needs n < 2^32.
PairDir build_pair_dir(const RunsBwt& bwt, const LeafDir& d, uint32_t window);

// Sorted u64 keys with a radix table: table[b] = #keys < (b << shift), b in [0, (universe>>shift)+1].
struct PredTable {
    uint32_t shift = 0;
    std::vector<uint64_t> keys;
    std::vector<uint32_t> table;
};

// Text / BWT positions (< 2^40) as a u32 plane plus, only when the universe exceeds 2^32, a u8 plane:
// 4 bytes per value on the BASELINE index (n < 2^32), 5 on the config-5 family, instead of 8.
struct Packed40 {
    std::vector<uint32_t> lo;
    std::vector<uint8_t> hi;             // empty when every value fits 32 bits
    bool wide = false;
    void init(uint64_t universe, size_t reserve = 0) { wide = (universe >> 32) != 0; lo.reserve(reserve); if (wide) hi.reserve(reserve); }
    void push(uint64_t v) { lo.push_back((uint32_t) v); if (wide) hi.push_back((uint8_t) (v >> 32)); }
    uint64_t get(size_t i) const { return (uint64_t) lo[i] | (wide ? (uint64_t) hi[i] << 32 : 0ull); }
    size_t size() const { return lo.size(); }
    size_t bytes() const { return lo.size() * 4 + hi.size(); }
};

// Toehold resolution: rows of the F column that are LF images of BWT run ends, with the
// SA sample of that run end.  After a non-trivial LF_w_loc step (include/rowbowt.hpp:562-566)
// the new hi IS such a row, and its toehold is samples_last[run] -- one lookup instead of
// rank + select + run_of_position.  Rows are cut into buckets of 2^shift (about three keys each); a key keeps only
// its low `shift` bits (1, 2 or 4 bytes), the bucket table the rest; samples are Packed40: 6.2 bytes per run on the
// BASELINE index where two u64 arrays behind a PredTable took 17.
struct ToeholdDir {
    uint32_t shift = 0;
    uint32_t key_bytes = 1;              // 1 (shift <= 8), 2 (<= 16) or 4
    uint64_t n_keys = 0;
    std::vector<uint32_t> table;         // table[b] = #keys < (b << shift), b in [0, (n >> shift) + 2]
    std::vector<uint8_t> keys;           // [n_keys * key_bytes] low bits of LF(end of run j), ascending by full key
    Packed40 sample;                     // sample[i] = samples_last of the run whose end maps to key i
    uint64_t toehold0 = 0;               // ToeholdSA::get_last_run_sample (include/toehold_sa.hpp:97-99)
    size_t bytes() const { return table.size() * 4 + keys.size() + sample.bytes(); }
};
// #keys < row (host mirror of the device lookup; the self-check and tests use it)
uint64_t toehold_dir_rank(const ToeholdDir& t, uint64_t row);

// phi (include/toehold_sa.hpp:56-72) as direct-addressed 32-byte slots (phi_slot.cuh): slot b answers
// every text position of bucket b; prev = samples_last[pred_to_run[jr] - 1] is fused at load.
struct PhiDir {
    uint32_t shift = 0;                  // bucket = 2^shift text positions
    uint64_t n_buckets = 0;
    uint64_t n_slots = 0;                // NON-EMPTY buckets + 1 sentinel (phi_slot.cuh: only they have a slot)
    std::vector<uint64_t> l1;            // [n_buckets/32 + 1]: bits 0..31 which of 32 buckets hold a sample, bits 32..63 non-empty buckets before
    std::vector<uint64_t> slots;         // [n_slots * 4]
    Packed40 ovf_prev;                   // prev values of the samples in BITMAP / SEARCH buckets, ascending by key
    std::vector<uint64_t> ovf_keys;      // their keys (SEARCH buckets only: shift > 7)
    uint64_t n_overflow = 0;             // BITMAP / SEARCH buckets
};

// shift = 0 -> choose (about three keys per bucket), else buckets of 2^shift rows, shift <= 32
ToeholdDir build_toehold_dir(const RunsBwt& bwt, const uint64_t (&F)[256], const ToeholdArrays& tsa, uint32_t shift);
// shift = 0 -> choose: 7, or the smallest larger one whose slots fit max_slot_bytes.  n_parts = 0 -> choose how many host
// threads build it (several only for large indexes)
PhiDir build_phi_dir(const ToeholdArrays& tsa, uint32_t shift, unsigned n_parts, uint64_t max_slot_bytes);
// phi(i) through the slots on the host (self-check): must equal ToeholdSA::phi for every i != SA[0]
uint64_t phi_dir_eval(const PhiDir& p, uint64_t n, uint64_t i);
PredTable build_pred_table(std::vector<uint64_t>&& keys, uint64_t universe, double keys_per_bucket);

}  // namespace rbg
