// The marker array (.ma) from a .mps and the index's own phi (ma_build.cu).
#pragma once
#include <cstdint>
#include <string>

#include "../../include/rowbowt_gpu.h"
#include "formats.hpp"
#include "layout.hpp"

namespace rbg {

// Rows [row_begin, row_end) (row_begin < row_end <= n; tsa.r == bwt.R): writes ma_path and, when mab_path is not empty, the
// .mab rb_build -m makes from it.  Fills the row, step, record, layout, write and kernel fields of `st` (adding to them).
void build_marker_array(const RunsBwt& bwt, const ToeholdArrays& tsa, const MpsRecords& mps, uint64_t row_begin, uint64_t row_end,
                        int device, const std::string& ma_path, const std::string& mab_path, rbg_ma_stats& st);

}  // namespace rbg
