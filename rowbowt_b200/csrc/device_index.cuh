// Device-side views of the index (plain structs passed to kernels by value) and the
// per-step device functions: rank-pair / LF, toehold resolution, phi, marker windows.
#pragma once
#include <cstdint>

#include "leaf.cuh"
#include "phi_slot.cuh"

namespace rbg {

constexpr int kDevMaxTerm = 8;
constexpr int kMaxSuper5Dev = 256;      // == kMaxSuper5 (layout.hpp): layout 5 keeps at most 4 x 256 superblock bases
constexpr uint64_t kPairMaxShared = 48 << 10;   // the pair superblock table search_kernel holds in shared memory (16 x 4 x n_super bytes)

// The rank directory (LeafDir, layout.hpp): the line of BWT position p is p / window.
struct DevLeafDir {
    const uint32_t* lines;      // 64-byte mixed leaves: [n_direct] direct, then RAW children of CLUSTER windows (layout 7: 32-byte plain lines)
    const uint64_t* super;      // [4][n_super]: F[c] + #c in BWT[0, superblock_start) (layout 7: unused)
    uint64_t n;
    uint64_t magic;             // i / window == umul64hi(i, magic)
    uint64_t n_super;
    uint32_t window;
    uint32_t sb_shift;
    uint32_t n_term;
    uint32_t version;           // leaf.cuh: LeafFmt 4 or 5, or 7 (plain lines)
    // i / window without the 64 x 64 -> 128 bit product: window = m * 2^div_k (m odd), so i / window = (i >> div_k) / m, and for
    // (n >> div_k) < 2^31 that is ((i >> div_k) * div_mul) >> div_s with a 32-bit multiplier (set_fast_div below):
    // 3 instructions instead of 9, twice per LF step.  div_fast == 0 (odd windows over huge n): umul64hi(i, magic).
    uint32_t div_k, div_mul, div_s, div_fast;
    uint64_t term_pos[kDevMaxTerm];
};

// Fills the fast-division fields for D.window and D.n (host).  Exact for every i <= n: with l = ceil(log2 m) and
// div_mul = floor(2^(31+l) / m) + 1 the error term div_mul * m - 2^(31+l) lies in (0, m] <= 2^l (Granlund-Montgomery).
inline void set_fast_div(DevLeafDir& D) {
    uint32_t k = 0;
    while (!((D.window >> k) & 1u)) ++k;
    const uint64_t m = D.window >> k;
    D.div_k = k;
    D.div_fast = 0;
    D.div_mul = 0;
    D.div_s = 0;
    if ((D.n >> k) >= (1ull << 31)) return;
    uint32_t l = 0;
    while ((1ull << l) < m) ++l;
    D.div_mul = (uint32_t) ((1ull << (31 + l)) / m + 1);
    D.div_s = 31 + l;
    D.div_fast = 1;
}

// The pair directory (PairDir, layout.hpp; lines: leaf.cuh LeafFmt<6>), n < 2^32.  lines == nullptr: not built.
struct DevPairDir {
    const uint32_t* lines;
    const uint32_t* super;      // [16][n_super]: K[p] + #p in P[0, superblock_start), copied to shared memory per CTA
    uint32_t n_super;
    uint32_t window;            // even, so i / window == ((i >> div_k) * div_mul) >> div_s for every i < 2^32 (set_fast_div)
    uint32_t sb_shift;
    uint32_t div_k, div_mul, div_s;
    uint32_t n_child;           // RAW children of a CLUSTER window: ceil(window / 128)
    uint32_t n_bad;
    uint32_t bad_pos[kPairMaxBad];
};

// ToeholdDir (layout.hpp): bucket table over the rows that are LF images of run ends, keys reduced to their low
// `shift` bits, samples as a u32 plane (+ a u8 plane when n > 2^32).
struct DevToehold {
    const uint32_t* table;
    const uint8_t* keys;        // key_bytes per key
    const uint32_t* sample_lo;
    const uint8_t* sample_hi;   // null when n <= 2^32
    uint64_t toehold0;
    uint32_t shift;
    uint32_t key_bytes;         // 1, 2 or 4
};

// phi as direct-addressed 32-byte slots (PhiDir, layout.hpp; decode in phi_slot.cuh)
struct DevPhi {
    const uint64_t* l1;         // [n_buckets/32 + 1] non-empty bitmap | rank (phi_slot.cuh)
    const uint64_t* slots;      // [n_slots][4]: one per non-empty bucket + sentinel
    const uint64_t* ovf_keys;   // keys of SEARCH buckets (shift > 7 only)
    const uint32_t* ovf_prev_lo;   // prev values of the samples in BITMAP / SEARCH buckets: low 32 bits ...
    const uint8_t* ovf_prev_hi;    // ... and bits 32..39 (null when n <= 2^32)
    uint64_t n;
    uint32_t shift;
};

// k-mer seed table (FTab / RowBowt::build_ftab / search_ftab, include/ftab.hpp:12-40,
// include/rowbowt.hpp:726-758): entry x = find_range of the k-mer whose i-th base has code
// (x >> 2i) & 3 -- the reference's own enumeration order -- so the key of a read is the 2k bits of
// its last k bases exactly as pack_kernel laid them out.  (1,0) = k-mer absent.
struct DevFtab {
    const ulonglong2* range;    // [4^k] (lo, hi)
    const uint64_t* toe;        // [4^k] ToeholdTrack after the k steps: row | since << 40 | pending << 63 (null without SA)
    uint32_t k;                 // 0 = no table
};
constexpr uint32_t kFtabMaxK = 13;

struct DevMarkers {
    const uint64_t *starts, *ends, *idxs, *arr;
    uint64_t n_starts, n_ends, n_idxs;
    uint64_t size_starts, size_ends, size_idxs;
};

#if defined(__CUDACC__)

// Line (window) index of BWT position p.
__device__ __forceinline__ uint64_t line_of(const DevLeafDir& D, uint64_t p) {
    if (D.div_fast) return ((uint64_t) (uint32_t) (p >> D.div_k) * D.div_mul) >> D.div_s;      // warp-uniform branch (kernel parameter)
    return __umul64hi(p, D.magic);
}

// One 64-byte line as two 256-bit read-only loads (LDG.E.256 on sm_100a); lines are touched
// once per step and would only evict the table / read words from L1, so no L1 allocation.
__device__ __forceinline__ void load_line(const uint32_t* p, uint32_t (&w)[16]) {
    asm("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
        : "l"(p));
    asm("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(w[8]), "=r"(w[9]), "=r"(w[10]), "=r"(w[11]), "=r"(w[12]), "=r"(w[13]), "=r"(w[14]), "=r"(w[15])
        : "l"(p + 8));
}

// Rare path of one rank: position q of a CLUSTER window that lies strictly inside the collapsed
// stretch is answered from a RAW child line (one more dependent load); a TERM window subtracts the
// terminators it counted as 'A'.  `r` and `rel` are replaced / corrected in place.
template <int V>
__device__ __forceinline__ void leaf_rank_fix(const DevLeafDir& D, const uint32_t (&w)[16], uint32_t c, uint64_t pos_end,
                                              uint32_t q, uint32_t& r, uint32_t& rel) {
    uint64_t from = pos_end - q;                                   // where the counts of the line in use are taken
    if (leaf_inside_cluster(w, q)) {
        const uint32_t s = leaf_cluster_begin(w);
        const uint32_t ch = (q - s) / kRawSymbols, p = (q - s) - ch * kRawSymbols;
        const uint32_t* cw = D.lines + ((uint64_t) leaf_child_ptr(w) + ch) * 16;
        rel = (V == 5 ? rel : 0u) + raw_rel_count(cw, c);           // layout 5: child counts are relative to the window start
        r = raw_rank(cw, leaf_cpat(c), p);
        from += s + ch * kRawSymbols;
    }
    if ((w[15] & kFlagTerm) && c == 0) {
#pragma unroll
        for (uint32_t t = 0; t < (uint32_t) kDevMaxTerm; ++t)      // constant indices: term_pos stays in the parameter bank
            r -= (t < D.n_term && D.term_pos[t] >= from && D.term_pos[t] < pos_end) ? 1u : 0u;
    }
}

// RowBowt::LF(range,c) (include/rowbowt.hpp:74-88) for c in {A,C,G,T} (code 0..3, known present):
// rank_c(lo) from lo's line and rank_c(hi+1) from hi's line -- the same line once the range is
// narrow.  The decode is branch-free and identical for every lane (leaf.cuh).  With TOEHOLD also
// reports BWT[hi]==c (LF_w_loc's trivial-case test, include/rowbowt.hpp:559) as
// rank_c(hi+1) != rank_c(hi).  Returns false when the new range is empty.
template <bool TOEHOLD, int V>
__device__ __forceinline__ bool lf_step_v(const DevLeafDir& D, uint32_t c, uint64_t& lo, uint64_t& hi,
                                          bool& hi_is_c, uint32_t& lines_touched) {
    uint32_t A[16], B[16];
    const uint64_t wa = line_of(D, lo), wb = line_of(D, hi);
    const uint32_t qa = (uint32_t) lo - (uint32_t) wa * D.window, qb = (uint32_t) hi - (uint32_t) wb * D.window + 1u;
    load_line(D.lines + wa * 16, A);
    const uint64_t* sup = D.super + (uint64_t) c * D.n_super;
    const uint64_t base_a = __ldg(sup + (wa >> D.sb_shift));
    uint64_t base_b = base_a;
    if (wb == wa) {
#pragma unroll
        for (int i = 0; i < 16; ++i) B[i] = A[i];
        lines_touched += 1;
    } else {
        load_line(D.lines + wb * 16, B);
        base_b = __ldg(sup + (wb >> D.sb_shift));
        lines_touched += 2;
    }
    const uint32_t cpat = leaf_cpat(c);
    uint32_t ra = leaf_rank<V>(A, cpat, qa);                    // #c in [window start of lo, lo)
    uint32_t xb[6], xs[6];
    leaf_match<V>(B, cpat, xb, xs);
    uint32_t rb = leaf_rank_x<V>(B, xb, xs, qb);                // #c in [window start of hi, hi]
    uint32_t rc = TOEHOLD ? leaf_rank_x<V>(B, xb, xs, qb - 1u) : 0u;
    uint32_t rel_a = leaf_rel_count<V>(A, c), rel_b = leaf_rel_count<V>(B, c), rel_c = rel_b;
    if ((A[15] | B[15]) & kFlagAny) {                           // a variant cluster or the terminator in the window
        const bool term = ((A[15] | B[15]) & kFlagTerm) && c == 0;
        if (term || leaf_inside_cluster(A, qa)) leaf_rank_fix<V>(D, A, c, lo, qa, ra, rel_a);
        if (term || leaf_inside_cluster(B, qb)) leaf_rank_fix<V>(D, B, c, hi + 1, qb, rb, rel_b);
        if (TOEHOLD && (term || leaf_inside_cluster(B, qb - 1u))) leaf_rank_fix<V>(D, B, c, hi, qb - 1u, rc, rel_c);
    }
    const uint64_t new_lo = base_a + rel_a + ra;                 // F[c] + #c in BWT[0,lo)
    const uint64_t new_end = base_b + rel_b + rb;                // F[c] + #c in BWT[0,hi]
    hi_is_c = TOEHOLD ? (uint32_t) (rel_b + rb) != (uint32_t) (rel_c + rc) : false;    // BWT[hi] == c <=> the count grows from hi to hi+1
    if (new_end == new_lo) return false;
    lo = new_lo;
    hi = new_end - 1;
    return true;
}

// 32 bytes as one 256-bit read-only load without L1 allocation (p 32-byte aligned): a plain line (layout 7, leaf.cuh), a
// group of raw read bytes (pack_kernel).
__device__ __forceinline__ void load_nc_32B(const void* p, uint32_t (&w)[8]) {
    asm("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
        : "l"(p));
}

// LF step on the plain lines (layout 7, n < 2^31): rank_c(lo) from lo's line, rank_c(hi+1) from hi's line -- the match word
// and the count of one line serve both once the range is narrow -- and BWT[hi] == c as bit q of hi's match word.  WARP: every
// lane of the warp calls (search_kernel; `act` says whether the lane has a step, an inactive lane reads line 0 and keeps its
// range), so the TERM path costs the common path one flag test and one vote.  Otherwise one thread (lf_step).
template <bool TOEHOLD, bool WARP>
__device__ __forceinline__ bool lf_step_plain(const DevLeafDir& D, uint32_t c, uint64_t& lo, uint64_t& hi, bool act,
                                              bool& hi_is_c, uint32_t& lines_touched) {
    const uint32_t l = act ? (uint32_t) lo : 0u, h = act ? (uint32_t) hi : 0u;
    const uint32_t wa = l >> kPlainShift, wb = h >> kPlainShift, qa = l & (kPlainRows - 1u), qb = h & (kPlainRows - 1u);
    uint32_t A[kPlainWords];
    load_nc_32B(D.lines + (uint64_t) wa * kPlainWords, A);
    const uint64_t ma = plain_match(A, c);
    const uint32_t ca = plain_count(A, c);
    uint64_t mb = ma;
    uint32_t cb = ca, flags = A[0];
    if (wb == wa) {
        lines_touched += act ? 1u : 0u;
    } else {
        uint32_t B[kPlainWords];
        load_nc_32B(D.lines + (uint64_t) wb * kPlainWords, B);
        mb = plain_match(B, c);
        cb = plain_count(B, c);
        flags |= B[0];
        lines_touched += 2;
    }
    uint32_t new_lo = ca + plain_rank_before(ma, qa);            // F[c] + #c in BWT[0, lo)
    uint32_t new_end = cb + plain_rank_upto(mb, qb);             // F[c] + #c in BWT[0, hi]
    hi_is_c = TOEHOLD && ((mb >> qb) & 1ull);
    const bool term = act && (flags & kPlainTerm) && c == 0u;
    if (WARP ? __any_sync(0xFFFFFFFFu, term) : term) {            // a terminator in lo's or hi's line, counted as 'A'
        if (term) {
#pragma unroll
            for (uint32_t t = 0; t < (uint32_t) kDevMaxTerm; ++t) {     // constant indices: term_pos stays in the parameter bank
                const bool on = t < D.n_term;
                const uint64_t p = D.term_pos[t];
                new_lo -= (on && p >= ((uint64_t) wa << kPlainShift) && p < l) ? 1u : 0u;
                new_end -= (on && p >= ((uint64_t) wb << kPlainShift) && p <= h) ? 1u : 0u;
                hi_is_c = hi_is_c && !(on && p == h);
            }
        }
    }
    if (!act || new_end == new_lo) return false;
    lo = new_lo;
    hi = new_end - 1u;
    return true;
}

// One thread, any layout (seed-table build, byte-wise search, greedy seeding: not the hot loop).
template <bool TOEHOLD>
__device__ __forceinline__ bool lf_step(const DevLeafDir& D, uint32_t c, uint64_t& lo, uint64_t& hi,
                                        bool& hi_is_c, uint32_t& lines_touched) {
    if (D.version == 7) return lf_step_plain<TOEHOLD, false>(D, c, lo, hi, true, hi_is_c, lines_touched);
    return D.version == 5 ? lf_step_v<TOEHOLD, 5>(D, c, lo, hi, hi_is_c, lines_touched)
                          : lf_step_v<TOEHOLD, 4>(D, c, lo, hi, hi_is_c, lines_touched);
}

// ---- warp-cooperative form of the rare paths (search_kernel) -----------------------------------
// A warp's 32 reads sit at unrelated BWT positions, so in ~1 of 4 warp steps SOME lane's rank position lies
// strictly inside a collapsed stretch.  Answered lane by lane (leaf_rank_fix) the RAW child walk -- a
// dependent load and up to 14 word iterations -- runs with one lane active and costs the warp ~150 issue
// slots; measured, the rare paths took a third of the kernel's issue slots.  Here the whole warp answers
// each such position together: lanes 0..15 load the 16 words of the child line (one coalesced 64-byte
// request), lanes 2..15 count their word, REDUX adds them up.  ~20 issue slots per position, no loop.
// All 32 lanes must call (inactive ones with in = false).
template <int V>
__device__ __forceinline__ void coop_cluster_fix(const DevLeafDir& D, const uint32_t (&w)[16], uint32_t c, uint32_t q, bool in,
                                                 uint32_t& r, uint32_t& rel, uint32_t& skipped) {
    uint32_t need = __ballot_sync(0xFFFFFFFFu, in);
    if (!need) return;                                             // warp-uniform
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t s = leaf_cluster_begin(w);
    const uint32_t d = in ? q - s : 0u;
    const uint32_t ch = d / kRawSymbols, p = d - ch * kRawSymbols;  // p < 224
    const uint32_t child = leaf_child_ptr(w) + ch;
    const uint32_t pc = p | (c << 8);
    if (in) skipped = s + ch * kRawSymbols;
    const int word_first = 16 * ((int) (lane & 15u) - 2);           // first symbol of this lane's word (lanes 2..15)
    const bool counts = lane >= 2u && lane < 16u;
    do {
        const int src = __ffs(need) - 1;
        need &= need - 1u;
        const uint32_t sc = __shfl_sync(0xFFFFFFFFu, child, src), spc = __shfl_sync(0xFFFFFFFFu, pc, src);
        const uint32_t sp = spc & 0xFFu, cc = spc >> 8;
        const uint32_t word = __ldg(D.lines + (uint64_t) sc * 16 + (lane & 15u));
        const uint32_t x = word ^ leaf_cpat(cc);
        const uint32_t eq = ~(x | (x >> 1)) & 0x55555555u;
        const int rem = (int) sp - word_first;                     // symbols of this word that lie before p
        uint32_t m = rem >= 16 ? 0xFFFFFFFFu : (rem <= 0 ? 0u : (1u << (2 * rem)) - 1u);
        if (!counts) m = 0u;
        const uint32_t total = __reduce_add_sync(0xFFFFFFFFu, (uint32_t) __popc(eq & m));
        const uint32_t pair = __shfl_sync(0xFFFFFFFFu, word, (int) (cc >> 1));      // rel counts: words 0, 1
        if ((int) lane == src) {
            r = total;
            rel = (V == 5 ? rel : 0u) + ((cc & 1u) ? pair >> 16 : pair & 0xFFFFu);     // layout 5: on top of the line's own u32 count
        }
    } while (need);
}

// TERM window: the terminators counted as 'A' between where the counts in use start and pos_end.
__device__ __forceinline__ void term_fix(const DevLeafDir& D, const uint32_t (&w)[16], uint64_t pos_end, uint32_t q,
                                         uint32_t skipped, uint32_t& r) {
    if (!(w[15] & kFlagTerm)) return;
    const uint64_t from = pos_end - q + skipped;
#pragma unroll
    for (uint32_t t = 0; t < (uint32_t) kDevMaxTerm; ++t)
        r -= (t < D.n_term && D.term_pos[t] >= from && D.term_pos[t] < pos_end) ? 1u : 0u;
}

// lf_step for a whole warp: every lane calls, `act` says whether the lane has a step to do (inactive
// lanes read line 0 and keep their range).  Same results as lf_step, lane by lane.

// `sup`: the superblock bases [4][n_super] -- the global array for layout 4 (one L2-resident load per line), a copy
// in shared memory for layout 5 (search_kernel loads its <= 8 KB once per CTA).
template <bool TOEHOLD, int V>
__device__ __forceinline__ bool lf_step_lines(const DevLeafDir& D, const uint64_t* sup, uint32_t c, uint64_t& lo, uint64_t& hi, bool act,
                                              uint64_t wa, uint64_t wb, bool& hi_is_c, uint32_t& lines_touched);

template <bool TOEHOLD, int V>
__device__ __forceinline__ bool lf_step_warp(const DevLeafDir& D, const uint64_t* sup, uint32_t c, uint64_t& lo, uint64_t& hi, bool act,
                                             bool& hi_is_c, uint32_t& lines_touched) {
    if constexpr (V == 7) {
        return lf_step_plain<TOEHOLD, true>(D, c, lo, hi, act, hi_is_c, lines_touched);
    } else {
        const uint64_t l = act ? lo : 0ull, h = act ? hi : 0ull;
        return lf_step_lines<TOEHOLD, V>(D, sup, c, lo, hi, act, line_of(D, l), line_of(D, h), hi_is_c, lines_touched);
    }
}

// Same with the line indexes of lo and hi already known (0, 0 for an inactive lane).
template <bool TOEHOLD, int V>
__device__ __forceinline__ bool lf_step_lines(const DevLeafDir& D, const uint64_t* sup_all, uint32_t c, uint64_t& lo, uint64_t& hi, bool act,
                                              uint64_t wa, uint64_t wb, bool& hi_is_c, uint32_t& lines_touched) {
    uint32_t A[16], B[16];
    const uint64_t l = act ? lo : 0ull, h = act ? hi : 0ull;
    const uint32_t qa = (uint32_t) l - (uint32_t) wa * D.window, qb = (uint32_t) h - (uint32_t) wb * D.window + 1u;
    load_line(D.lines + wa * 16, A);
    const uint64_t* sup = sup_all + (uint64_t) c * D.n_super;
    const uint64_t base_a = V == 5 ? sup[wa >> D.sb_shift] : __ldg(sup + (wa >> D.sb_shift));
    uint64_t base_b = base_a;
    if (wb == wa) {
#pragma unroll
        for (int i = 0; i < 16; ++i) B[i] = A[i];
        lines_touched += act ? 1u : 0u;
    } else {
        load_line(D.lines + wb * 16, B);
        base_b = V == 5 ? sup[wb >> D.sb_shift] : __ldg(sup + (wb >> D.sb_shift));
        lines_touched += 2;
    }
    const uint32_t cpat = leaf_cpat(c);
    uint32_t ra = leaf_rank<V>(A, cpat, qa);
    uint32_t xb[6], xs[6];
    leaf_match<V>(B, cpat, xb, xs);
    uint32_t rb = leaf_rank_x<V>(B, xb, xs, qb);
    uint32_t rel_a = leaf_rel_count<V>(A, c), rel_b = leaf_rel_count<V>(B, c);
    const uint32_t fl = act ? (A[15] | B[15]) & kFlagAny : 0u;
    const bool any_fl = __any_sync(0xFFFFFFFFu, fl != 0u);      // warp-uniform: some lane sees a variant cluster / the terminator
    if (any_fl) {
        uint32_t sk_a = 0, sk_b = 0;
        coop_cluster_fix<V>(D, A, c, qa, fl && leaf_inside_cluster(A, qa), ra, rel_a, sk_a);
        coop_cluster_fix<V>(D, B, c, qb, fl && leaf_inside_cluster(B, qb), rb, rel_b, sk_b);
        if ((fl & kFlagTerm) && c == 0) {                        // the one TERM window of the index: lane by lane
            term_fix(D, A, l, qa, sk_a, ra);
            term_fix(D, B, h + 1, qb, sk_b, rb);
        }
    }
    const uint64_t new_lo = base_a + rel_a + ra;
    const uint64_t new_end = base_b + rel_b + rb;
    hi_is_c = false;
    if (TOEHOLD) {
        // BWT[hi] == c (LF_w_loc's trivial case) <=> rank_c(hi+1) != rank_c(hi).  When EVERY row of the range holds c
        // (the count grows by the range size: all but ~1 % of the steps of a read on a pangenome index, whose ranges
        // only shrink at variant sites) the answer is yes without looking; the third rank is computed only in warp
        // steps where some lane's range shrank -- about one warp step in six on the BASELINE workload.
        const bool whole = new_end - new_lo == h - l + 1;
        const bool unsure = act && !whole && new_end != new_lo;
        hi_is_c = whole;
        if (__any_sync(0xFFFFFFFFu, unsure)) {
            uint32_t rc = leaf_rank_x<V>(B, xb, xs, qb - 1u), rel_c = leaf_rel_count<V>(B, c);
            if (any_fl) {
                uint32_t sk_c = 0;
                coop_cluster_fix<V>(D, B, c, qb - 1u, fl && leaf_inside_cluster(B, qb - 1u), rc, rel_c, sk_c);
                if ((fl & kFlagTerm) && c == 0) term_fix(D, B, h, qb - 1u, sk_c, rc);
            }
            if (unsure) hi_is_c = (rel_b + rb) != (rel_c + rc);
        }
    }
    if (!act || new_end == new_lo) return false;
    lo = new_lo;
    hi = new_end - 1;
    return true;
}

// ---- two bases per LF step (count search on the pair directory) ----------------------------------
// For a read ...c1 c2 (c2 consumed first) and p = 4 c1 + c2:
//   LF(c1, LF(c2, lo)) = F[c1] + rank_c1(F[c2] + rank_c2(lo))
//                      = F[c1] + rank_c1(F[c2]) + #{i in [F[c2], F[c2] + rank_c2(lo)) : BWT[i] = c1}
//                      = K[p] + #{j < lo : BWT[j] = c2, BWT[LF(j)] = c1} = K[p] + rank_p(lo) over P
// because LF maps the c2-rows below lo, in order, onto the first rank_c2(lo) rows of block c2.  The same holds for hi + 1,
// and the range is empty after both steps exactly when this one is empty.

// A whole warp answers the ranks that fall in CLUSTER windows, one lane's position at a time: lanes 0..31 load the (at most
// 32) words of the window's RAW children, count code p before q in their word, REDUX adds them up.
__device__ __forceinline__ void coop_pair_raw(const DevPairDir& P, const uint32_t (&w)[16], uint32_t p, uint32_t q, bool in, uint32_t& r) {
    uint32_t need = __ballot_sync(0xFFFFFFFFu, in);
    if (!need) return;                                             // warp-uniform
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t child = in ? pair_child_ptr(w) : 0u, qp = q | (p << 16);
    do {
        const int src = __ffs(need) - 1;
        need &= need - 1u;
        const uint32_t sc = __shfl_sync(0xFFFFFFFFu, child, src), sqp = __shfl_sync(0xFFFFFFFFu, qp, src);
        const uint32_t word = lane < 16u * P.n_child ? __ldg(P.lines + (uint64_t) sc * 16 + lane) : 0u;
        const uint32_t cnt = pair_raw_word_count(word, pair_pat(sqp >> 16), 8 * (int) lane, (int) (sqp & 0xFFFFu));
        const uint32_t total = __reduce_add_sync(0xFFFFFFFFu, cnt);
        if ((int) lane == src) r = total;
    } while (need);
}

// TERM window, code 0: the rows stored as code 0 for a pair with the terminator, in [pos_end - q, pos_end)
__device__ __forceinline__ void pair_term_fix(const DevPairDir& P, const uint32_t (&w)[16], uint32_t pos_end, uint32_t q, uint32_t& r) {
    if (!(w[15] & kFlagTerm)) return;
    const uint32_t from = pos_end - q;
#pragma unroll
    for (uint32_t t = 0; t < (uint32_t) kPairMaxBad; ++t)
        r -= (t < P.n_bad && P.bad_pos[t] >= from && P.bad_pos[t] < pos_end) ? 1u : 0u;
}

__device__ __forceinline__ uint32_t pair_line_of(const DevPairDir& P, uint32_t i) {
    return (uint32_t) (((uint64_t) (i >> P.div_k) * P.div_mul) >> P.div_s);
}

// Two LF steps (code p = 4 c1 + c2) for a whole warp; `sup` is the pair superblock table in shared memory.  Every lane calls;
// an inactive lane reads line 0 and keeps its range.  Returns false when the range after both steps is empty.
__device__ __forceinline__ bool lf_pair_warp(const DevPairDir& P, const uint32_t* sup, uint32_t p, uint64_t& lo, uint64_t& hi, bool act,
                                             uint32_t& lines_touched) {
    uint32_t A[16], B[16];
    const uint32_t l = act ? (uint32_t) lo : 0u, h = act ? (uint32_t) hi : 0u;
    const uint32_t wa = pair_line_of(P, l), wb = pair_line_of(P, h);
    const uint32_t qa = l - wa * P.window, qb = h - wb * P.window + 1u;
    load_line(P.lines + (uint64_t) wa * 16, A);
    const uint32_t* sp = sup + p * P.n_super;
    const uint32_t base_a = sp[wa >> P.sb_shift];
    uint32_t base_b = base_a;
    if (wb == wa) {
#pragma unroll
        for (int i = 0; i < 16; ++i) B[i] = A[i];
        lines_touched += act ? 1u : 0u;
    } else {
        load_line(P.lines + (uint64_t) wb * 16, B);
        base_b = sp[wb >> P.sb_shift];
        lines_touched += 2;
    }
    const uint32_t ppat = pair_pat(p);
    uint32_t ra = pair_rank(A, ppat, qa);
    uint32_t rb = pair_rank(B, ppat, qb);
    const uint32_t rel_a = pair_rel_count(A, p), rel_b = pair_rel_count(B, p);
    const uint32_t fl = act ? (A[15] | B[15]) & kFlagAny : 0u;
    if (__any_sync(0xFFFFFFFFu, fl != 0u)) {                       // warp-uniform: some lane sees a CLUSTER / TERM window
        coop_pair_raw(P, A, p, qa, fl && (A[15] & kFlagCluster), ra);
        coop_pair_raw(P, B, p, qb, fl && (B[15] & kFlagCluster), rb);
        if ((fl & kFlagTerm) && p == 0) {
            pair_term_fix(P, A, l, qa, ra);
            pair_term_fix(P, B, h + 1u, qb, rb);
        }
    }
    const uint32_t new_lo = base_a + rel_a + ra, new_end = base_b + rel_b + rb;
    if (!act || new_end == new_lo) return false;
    lo = new_lo;
    hi = new_end - 1u;
    return true;
}

// Same for the terminator (byte 1) as a query symbol: rank over the sorted term_pos list, F[1] = 0.
__device__ __forceinline__ bool lf_step_term(const DevLeafDir& D, uint64_t& lo, uint64_t& hi, bool& hi_is_c) {
    uint64_t before = 0, upto = 0;
    hi_is_c = false;
#pragma unroll
    for (uint32_t t = 0; t < (uint32_t) kDevMaxTerm; ++t) {
        const bool on = t < D.n_term;
        before += on && D.term_pos[t] < lo;
        upto += on && D.term_pos[t] <= hi;
        hi_is_c = hi_is_c || (on && D.term_pos[t] == hi);
    }
    if (upto == before) return false;
    lo = before;
    hi = upto - 1;
    return true;
}

// Toehold after a non-trivial step: `row` is the LF image of a run end (see ToeholdDir): the index of that key
// (#keys < row: bucket table, then a binary search over the ~3 reduced keys of the bucket) selects the sample.
__device__ __forceinline__ uint64_t toehold_at_row(const DevToehold& T, uint64_t row) {
    const uint64_t b = row >> T.shift;
    const uint32_t low = (uint32_t) (row & ((1ull << T.shift) - 1ull));
    uint32_t a = __ldg(T.table + b), z = __ldg(T.table + b + 1);
    while (a < z) {
        const uint32_t mid = (a + z) >> 1;
        uint32_t k;
        if (T.key_bytes == 1) k = __ldg(T.keys + mid);
        else if (T.key_bytes == 2) k = __ldg(reinterpret_cast<const uint16_t*>(T.keys) + mid);
        else k = __ldg(reinterpret_cast<const uint32_t*>(T.keys) + mid);
        if (k < low) a = mid + 1; else z = mid;
    }
    uint64_t v = __ldg(T.sample_lo + a);
    if (T.sample_hi) v |= (uint64_t) __ldg(T.sample_hi + a) << 32;
    return v;
}

__device__ __forceinline__ uint64_t phi_prev_at(const DevPhi& P, uint64_t idx) {
    uint64_t v = __ldg(P.ovf_prev_lo + idx);
    if (P.ovf_prev_hi) v |= (uint64_t) __ldg(P.ovf_prev_hi + idx) << 32;
    return v;
}

// ToeholdSA::phi, include/toehold_sa.hpp:56-72: one L2-resident u64 (which slot), one 32-byte slot (one 256-bit
// load), one more load for the prev value when the bucket of i is a BITMAP bucket and holds a sample below i.
__device__ __forceinline__ uint64_t phi_step(const DevPhi& P, uint64_t i) {
    const uint64_t b = i >> P.shift;
    bool here;
    const uint64_t k = phi_slot_index(__ldg(P.l1 + (b >> 5)), (uint32_t) (b & 31), here);
    uint64_t q[4];
    asm("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
        : "=l"(q[0]), "=l"(q[1]), "=l"(q[2]), "=l"(q[3]) : "l"(P.slots + 4 * k));
    const uint64_t base = b << P.shift;
    uint64_t key = slot_get<0, 40>(q), prev = slot_get<40, 40>(q);          // the carry answers an empty bucket
    if (here) {
        if (!slot_overflow(q)) {
            slot_pred(q, base, (uint32_t) (i - base), key, prev);
        } else if (!slot_search(q)) {
            uint64_t idx;
            if (slot_bitmap_pred(q, base, (uint32_t) (i - base), key, idx)) prev = phi_prev_at(P, idx);
        } else {
            uint64_t lo = slot_ovf_start(q), hi = lo + slot_ovf_count(q);
            const uint64_t first = lo;
            while (lo < hi) {
                const uint64_t mid = (lo + hi) >> 1;
                if (__ldg(P.ovf_keys + mid) < i) lo = mid + 1; else hi = mid;
            }
            if (lo > first) { key = __ldg(P.ovf_keys + lo - 1); prev = phi_prev_at(P, lo - 1); }
        }
    }
    return phi_value(key, prev, i, P.n);
}

__device__ __forceinline__ uint64_t dev_lower_bound(const uint64_t* a, uint64_t m, uint64_t x) {
    uint64_t lo = 0, hi = m;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// rle_window_arr::at_range (pfbwt-f/include/rle_window_array.hpp:130-154) reduced to the index
// range [first,last) of windows it would append, with its clamped rank/select helpers (:202-232).
__device__ __forceinline__ void marker_windows(const DevMarkers& M, uint64_t s, uint64_t e, uint64_t& first, uint64_t& last) {
    first = last = 0;
    // run_starts_rank(e): #starts <= e, clamped at the bit-vector size
    const uint64_t e_rs_rank = e + 1 >= M.size_starts ? M.n_starts : dev_lower_bound(M.starts, M.n_starts, e + 1);
    if (e_rs_rank == 0) return;
    const uint64_t e_rs_pos = e_rs_rank > M.n_starts ? M.size_starts : __ldg(M.starts + e_rs_rank - 1);
    if (e_rs_pos <= s) {
        const uint64_t e_re_pos = e_rs_rank > M.n_ends ? M.size_ends : __ldg(M.ends + e_rs_rank - 1);
        if (e_re_pos >= s) { first = e_rs_rank - 1; last = e_rs_rank; }
        return;
    }
    uint64_t s_rs_rank = s + 1 >= M.size_starts ? M.n_starts : dev_lower_bound(M.starts, M.n_starts, s + 1);
    s_rs_rank = s_rs_rank ? s_rs_rank : 1;
    const uint64_t s_rs_pos = s_rs_rank > M.n_starts ? M.size_starts : __ldg(M.starts + s_rs_rank - 1);
    // run_ends_rank(s): #ends < s, clamped to size-1
    uint64_t s_re_rank = s > M.size_ends - 1 ? dev_lower_bound(M.ends, M.n_ends, M.size_ends - 1)
                                             : dev_lower_bound(M.ends, M.n_ends, s);
    s_re_rank = s_re_rank ? s_re_rank : 1;
    const uint64_t s_re_pos = s_re_rank > M.n_ends ? M.size_ends : __ldg(M.ends + s_re_rank - 1);
    first = s_rs_pos > s_re_pos ? s_rs_rank - 1 : s_rs_rank;
    last = e_rs_rank;
    if (first > last) first = last;
}

// arr_idxs_select (1-based, clamped), rle_window_array.hpp:227-232
__device__ __forceinline__ uint64_t marker_sel(const DevMarkers& M, uint64_t i) {
    return i > M.n_idxs ? M.size_idxs : __ldg(M.idxs + i - 1);
}

#endif  // __CUDACC__

}  // namespace rbg
