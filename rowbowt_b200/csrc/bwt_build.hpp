// The BWT of a FASTA (or of an ACGT text) and its run-boundary samples, built on the GPU (bwt_build.cu).
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/rowbowt_gpu.h"

namespace rbg {

// Positions and ranks are u32 on the device, so the text (terminator included) holds at most this many positions.
// Every size in the ABI is u64: lifting the cap is a change behind this constant.
constexpr uint64_t kBwtMaxN = 0xFFFFFFFFull;
constexpr int kBwtPad = 10;                      // 'A's after every record (pfbwt-f's padding, w = 10)

struct nomem_error : std::runtime_error { using std::runtime_error::runtime_error; };

// The text pfbwt-f64 --non-acgt-to-a indexes, without the terminator: every record's bases (uppercase letters other than
// ACGT become 'A') followed by kBwtPad 'A's, and the offset of each record's first base.  Refuses, with no CUDA call: a
// missing / unreadable file (io_error), no records or a record without bases (format_error), a byte that is not an uppercase
// letter (alphabet_error naming the record and offset), n >= 2^32 (std::invalid_argument naming the cap).
struct FastaText {
    std::vector<uint8_t> text;
    std::vector<std::string> names;
    std::vector<uint64_t> starts;
};
FastaText read_fasta_text(const std::string& path);

// Refuses (std::invalid_argument naming the cap) a text of n > kBwtMaxN positions; `what` names the text.
void check_bwt_length(uint64_t n, const std::string& what);

// Refuses (alphabet_error) a byte of text[0, len) other than A, C, G, T.  No CUDA call.
void check_acgt(const uint8_t* text, uint64_t len);

// text[0, len) + the terminator (byte 0) on `device` (already selected): writes <out>.bwt, <out>.ssa and <out>.esa, each
// to a temporary file renamed into place.  Before allocating, the peak device memory is checked against what is free
// (nomem_error naming the bytes needed).  Fills n, r, rounds, active, max_active, s_sort, s_write, ms_* and peak_bytes.
void build_bwt_files(const uint8_t* text, uint64_t len, int device, const std::string& out_prefix, rbg_bwt_stats& st);

// `name start` per record, to a temporary file renamed into place.
void write_docs(const FastaText& ft, const std::string& path);

}  // namespace rbg
