// The BWT of a FASTA (or of an ACGT text) and its run-boundary samples, built on the GPU (bwt_build.cu).
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/rowbowt_gpu.h"

namespace rbg {

// build_bwt_files keeps positions and ranks in u32 on the device, so its text (terminator included) holds at most this
// many positions; build_bwt_files_wide keeps them in u64 and takes a FASTA of n < 2^40 (the query path's 5-byte positions).
constexpr uint64_t kBwtMaxN = 0xFFFFFFFFull;
constexpr uint64_t kBwtWideMaxN = (1ull << 40) - 1;
constexpr int kBwtPad = 10;                      // 'A's after every record (pfbwt-f's padding, w = 10)

struct nomem_error : std::runtime_error { using std::runtime_error::runtime_error; };
// A result that failed its own check (the suffix-array certificate): RBG_E_INTERNAL.
struct internal_error : std::runtime_error { using std::runtime_error::runtime_error; };

// The text pfbwt-f64 --non-acgt-to-a indexes, without the terminator: every record's bases (uppercase letters other than
// ACGT become 'A') followed by kBwtPad 'A's, and the offset of each record's first base.  Refuses, with no CUDA call: a
// missing / unreadable file (io_error), no records or a record without bases (format_error), a byte that is not an uppercase
// letter (alphabet_error naming the record and offset), n > max_n (std::invalid_argument naming the cap).
struct FastaText {
    std::vector<uint8_t> text;
    std::vector<std::string> names;
    std::vector<uint64_t> starts;
};
FastaText read_fasta_text(const std::string& path, uint64_t max_n);

// Refuses (std::invalid_argument naming the cap) a text of n > max_n positions; `what` names the text.
void check_bwt_length(uint64_t n, const std::string& what, uint64_t max_n);

// Refuses (alphabet_error) a byte of text[0, len) other than A, C, G, T.  No CUDA call.
void check_acgt(const uint8_t* text, uint64_t len);

// text[0, len) + the terminator (byte 0) on `device` (already selected): writes <out>.bwt, <out>.ssa and <out>.esa, each
// to a temporary file renamed into place.  Before allocating, the peak device memory is checked against what is free
// (nomem_error naming the bytes needed).  Fills n, r, rounds, active, max_active, s_sort, s_write, ms_* and peak_bytes.
void build_bwt_files(const uint8_t* text, uint64_t len, int device, const std::string& out_prefix, rbg_bwt_stats& st);

// The same with u64 positions and ranks and the suffix array sorted in parts of at most part_rows rows (0: as many as the
// free device memory holds), for texts of any n (bwt_build_wide.cu).  Before allocating, 21 bytes per position + 32 per part
// row + the prefix histogram + scratch are checked against what is free (nomem_error); an 11-symbol prefix shared by more
// suffixes than a part holds is refused (nomem_error naming it).  The suffix array is certified before anything is written
// (internal_error naming the first bad row).  Fills, beyond build_bwt_files' fields, wide, parts, part_rows, ms_verify.
void build_bwt_files_wide(const uint8_t* text, uint64_t len, int device, uint64_t part_rows, const std::string& out_prefix,
                          rbg_bwt_stats& st);

// The certificate over a caller's suffix array sa[0, len + 1) of text[0, len) + the terminator: the smallest row i where
// sa[i] >= n, sa[i] is not the first row holding its value, or (T[sa[i]], rank[sa[i] + 1]) is not below the same pair of
// row i + 1; n when there is none.
uint64_t check_suffix_array(const uint8_t* text, uint64_t len, const uint64_t* sa, int device);

// `name start` per record, to a temporary file renamed into place.
void write_docs(const FastaText& ft, const std::string& path);

// The whole file to a temporary name, then renamed into place.
void write_file(const std::string& path, const void* data, size_t bytes);

}  // namespace rbg
