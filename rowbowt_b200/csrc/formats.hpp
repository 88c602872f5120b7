// Host-side readers for the reference's serialized index files (.rbwt / .tsa / .mab).
// The on-disk formats stay drop-in (rb_build is unchanged); these readers only DECODE
// them, sequentially, into the flat arrays of SURVEY.md Appendix B.8, from which the
// GPU layout is built (layout.hpp).  No sdsl dependency.
//
// Byte layouts (reference file:line, all little-endian, sdsl = xxsds v3):
//   rle_string::serialize        include/rle_string.hpp:248-260
//   sparse_sd_vector::serialize  include/sparse_sd_vector.hpp:182-189
//   sd_vector::serialize         sdsl-lite/include/sdsl/sd_vector.hpp:374-397
//   int_vector header            sdsl-lite/include/sdsl/int_vector.hpp:813-842
//   select_support_mcl           sdsl-lite/include/sdsl/select_support_mcl.hpp:427-466
//   wt_pc / _byte_tree           sdsl-lite/include/sdsl/wt_pc.hpp:610-623, wt_helper.hpp:117-134,313-340
//   ToeholdSA::serialize         include/toehold_sa.hpp:74-83
//   rle_window_arr::serialize    pfbwt-f/include/rle_window_array.hpp:174-187
//   wt_fbb (`rb_build --fbb`)    faster-minuter/include/wt_fbb.hpp:1849-1861 (top level), :124-146 (superblock
//                                header), :93-101 (block header item), :343-492 (block body + variable header),
//                                :245-267 (canonical codes); sdsl::hyb_vector<16> sdsl/hyb_vector.hpp:31-41,256-357
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

namespace rbg {

struct io_error : std::runtime_error { using std::runtime_error::runtime_error; };
struct format_error : std::runtime_error { using std::runtime_error::runtime_error; };

// Run-length BWT as flat runs.
struct RunsBwt {
    uint64_t n = 0, R = 0;
    std::vector<uint8_t> heads;     // [R]
    std::vector<uint64_t> lens;     // [R]
};

// ToeholdSA members, decoded.
struct ToeholdArrays {
    uint64_t r = 0, n = 0;
    std::vector<uint64_t> pred;          // sorted
    std::vector<uint64_t> samples_last;  // BWT order
    std::vector<uint64_t> pred_to_run;   // text order
};

// rle_window_arr members, decoded.
struct MarkerArrays {
    uint64_t size_starts = 0, size_ends = 0, size_idxs = 0;
    std::vector<uint64_t> starts, ends, idxs, arr;
    int32_t wsize = 10;
};

// Consistency of decoded (or caller-supplied) arrays, checked before any layout is built from them: a corrupted file must end
// as format_error, never as an out-of-range access in the layout builders or on the device.  `what` names the source in the message.
//   runs:    R heads and lengths, every length in [1, n - (sum so far)], lengths sum to n
//   toehold: r sorted sample positions < n, r samples < n, pred_to_run values <= r
//   markers: window starts / ends / indexes ascending inside their universes, indexes and their universe <= the number of
//            marker words
void validate_runs(const RunsBwt& b, const std::string& what);
void validate_toehold(const ToeholdArrays& t, const std::string& what);
void validate_markers(const MarkerArrays& m, const std::string& what);

RunsBwt read_rbwt(const std::string& path);
// The same string out of a wt_fbb .rbwt (include/fbb_string.hpp: `rb_build --fbb` / `rb_align --fbb`), decoded
// sequentially and run-length encoded.  The file holds the raw .bwt bytes (terminator = byte 0); the runs
// returned use the rle_string convention (terminator = byte 1) so that one device layout serves both.
RunsBwt read_rbwt_fbb(const std::string& path);
ToeholdArrays read_tsa(const std::string& path);
MarkerArrays read_mab(const std::string& path);

// A .mps (pfbwt-f's MarkerPositionsWriter; SURVEY.md A.1): records `first last word* ~0`, [first, last] an inclusive range
// of text positions.  Word lists are deduplicated by value into list ids; a record without words has kNoList.
constexpr uint32_t kNoList = 0xFFFFFFFFu;
struct MpsRecords {
    std::vector<uint64_t> first, last;  // [records] ascending, last[k] < first[k + 1]
    std::vector<uint32_t> list;         // [records] list id or kNoList
    std::vector<uint64_t> list_off;     // list i is words[list_off[i] .. list_off[i + 1])
    std::vector<uint64_t> words;
};
// Refuses (format_error naming the record) a truncated record or missing delimiter, first > last, records that do not
// ascend without overlap, last >= n, and 2^32 - 1 or more distinct lists.  No CUDA call.
MpsRecords read_mps(const std::string& path, uint64_t n);

}  // namespace rbg
