// The library's environment knobs (INTEGRATION.md, "Environment knobs"): the one place it reads the environment, and so
// the list of every RBG_* variable it reads.  None changes results; tests use them to reach every layout, window, key
// width, chunking and kernel form.  An unset or empty variable means "the library's own choice".
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <optional>

namespace rbg {

// The integer value of `name` when it is set and not empty.
inline std::optional<long long> env_int(const char* name) {
    const char* e = getenv(name);
    if (!e || !*e) return std::nullopt;
    return strtoll(e, nullptr, 10);
}

// What shapes an index's device layout; read once per open and passed to the builders (layout.hpp).  0 = the builder's
// own choice.  The layout cache stamps it, so every field is part of what a cache is valid for.
struct LayoutKnobs {
    int32_t layout = 0;                  // RBG_LAYOUT: 4, 5 or 7 forces the line format of the rank directory
    uint32_t window = 0;                 // RBG_WINDOW: window of the rank directory
    int32_t pair = -1;                   // RBG_PAIR: 0 / 1 builds the pair directory never / whenever allowed; -1 automatic
    uint32_t pair_window = 0;            // RBG_PAIR_WINDOW: window of the pair directory
    uint32_t toehold_shift = 0;          // RBG_TOEHOLD_SHIFT: bucket width 2^s of the toehold directory, 1..32
    uint32_t phi_shift = 0;              // RBG_PHI_SHIFT: bucket width 2^s of the phi directory
    uint32_t phi_parts = 0;              // RBG_PHI_PARTS: parts the phi directory is built in, 1..64

    // The line format asked of build_leaf_dir: RBG_LAYOUT, else layout 5 when RBG_PAIR=1 asks for the pair directory (which
    // is built over layout 5 only), else 0, the builder's own choice.
    int leaf_layout() const { return layout ? layout : pair == 1 ? 5 : 0; }
};

inline LayoutKnobs layout_knobs() {
    LayoutKnobs k;
    if (auto v = env_int("RBG_LAYOUT")) k.layout = *v == 4 || *v == 5 || *v == 7 ? (int32_t) *v : 0;
    if (auto v = env_int("RBG_WINDOW")) k.window = (uint32_t) *v;
    if (auto v = env_int("RBG_PAIR")) k.pair = (int32_t) *v;
    if (auto v = env_int("RBG_PAIR_WINDOW")) k.pair_window = (uint32_t) *v;
    if (auto v = env_int("RBG_TOEHOLD_SHIFT")) k.toehold_shift = (uint32_t) std::clamp(*v, 1ll, 32ll);
    if (auto v = env_int("RBG_PHI_SHIFT")) k.phi_shift = (uint32_t) *v;
    if (auto v = env_int("RBG_PHI_PARTS")) k.phi_parts = (uint32_t) std::clamp(*v, 1ll, 64ll);
    return k;
}

// Read by every query call: tests change them between calls on one handle.
struct QueryKnobs {
    int chunks = 0;                      // RBG_CHUNKS: chunks a batch is cut into, 1..max_chunks (0: automatic)
    int64_t loc_est = -1;                // RBG_LOC_EST: first guess of a batch's locations (-1: extrapolated)
    int loc_draw = -1;                   // RBG_LOC_DRAW: 0 / 1 forces the static / drawing locate kernel (-1: automatic)
    uint64_t stall_ns[2] = {0, 0};       // RBG_TEST_STALL="a,b" (us): stall the even chunks' search stream for a in front of
                                         // their pack, the odd chunks' for b between their pack and their search
};

inline QueryKnobs query_knobs(int max_chunks) {
    QueryKnobs k;
    if (auto v = env_int("RBG_CHUNKS")) k.chunks = (int) std::clamp<long long>(*v, 1, max_chunks);
    if (auto v = env_int("RBG_LOC_EST")) k.loc_est = *v;
    if (auto v = env_int("RBG_LOC_DRAW")) k.loc_draw = *v != 0;
    if (const char* e = getenv("RBG_TEST_STALL")) {
        unsigned long long a = 0, b = 0;
        if (sscanf(e, "%llu,%llu", &a, &b) >= 1) { k.stall_ns[0] = a * 1000ull; k.stall_ns[1] = b * 1000ull; }
    }
    return k;
}

// RBG_LANES: calls that may be in flight on one handle, 1..8 (default 2); read when the handle is opened.
inline int knob_lanes() { return (int) std::clamp(env_int("RBG_LANES").value_or(2), 1ll, 8ll); }

// RBG_BLOCKING_SYNC > 0: a lane's waits sleep instead of spinning; read when the lane is created.
inline bool knob_blocking_sync() { return env_int("RBG_BLOCKING_SYNC").value_or(0) > 0; }

// RBG_FBB_THREADS: threads decoding a wt_fbb .rbwt, 1..64 (0: automatic).
inline unsigned knob_fbb_threads() {
    const auto v = env_int("RBG_FBB_THREADS");
    return v ? (unsigned) std::clamp(*v, 1ll, 64ll) : 0u;
}

// Read by every BWT build (rbg_build_bwt, rbg_build_bwt_text) and passed to the builder.
struct BwtKnobs {
    bool wide = false;                   // RBG_BWT_WIDE=1: the u64 builder (parts) at any n
    uint64_t part_rows = 0;              // RBG_BWT_PART_ROWS: rows of one part of that builder at most, >= 1 (0: from free memory)
};

inline BwtKnobs bwt_knobs() {
    BwtKnobs k;
    if (auto v = env_int("RBG_BWT_WIDE")) k.wide = *v == 1;
    if (auto v = env_int("RBG_BWT_PART_ROWS")) k.part_rows = (uint64_t) std::max(*v, 1ll);
    return k;
}

// RBG_MA_CHUNK_ROWS: rows of one device pass of the marker-array build at most, >= 1 (0: from free device memory).
inline uint64_t knob_ma_chunk_rows() {
    const auto v = env_int("RBG_MA_CHUNK_ROWS");
    return v ? (uint64_t) std::max(*v, 1ll) : 0u;
}

}  // namespace rbg
