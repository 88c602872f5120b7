// The 64-byte rank-directory line ("mixed leaf", layout.hpp) and its decode.  Shared by the
// kernels and by the host-side layout self-check (rbg_selftest_layout), so both read lines
// identically; on the device the helpers below are single sm_100a instructions
// (VIMNMX.U16x2, IDP.2A, SHF, PRMT), on the host plain C.
//
// One line answers rank_c for ALL four symbols over a window of W BWT positions
// (replaces rle_string::rank, include/rle_string.hpp:131-161, ~10 dependent probes):
//   w[0..1]   4 x u16: #c in BWT[superblock_start, window_start), c = A,C,G,T.  The absolute part
//             (F[c] + #c before the superblock) is one u64 per symbol and superblock in a small,
//             L2-resident side array, so that 24 runs fit a line instead of 18.
//   w[2]      heads (2 bits: A,C,G,T) of entries 0..15, TRANSPOSED: entry e sits at bit
//             8*(e&3) + 2*(e>>2), so that (eq >> 2i) & 0x01010101 is the byte vector of
//             entries 4i..4i+3
//   w[3..14]  24 x u16 run starts, entry e in the (e&1) half of w[3 + e/2]: every run that
//             intersects the window, in BWT order, start relative to the window.  Unused
//             entries carry 0xFFFF (they cover nothing).
//   w[15]     heads of entries 16..23 in the same transposed pattern (bits 0-3 of each byte);
//             bits 4-5 of byte 0: mode, bit 6: TERM flag, byte 1 bits 4-7 + byte 2 bit 4: index
//             of the first pseudo-run (CLUSTER), byte 3 bits 4-6: number of pseudo-runs
// rank: run e covers [s_e, s_{e+1}), so with m_e = min(q, s_e) and X_e = [head_e == c]
//   #c in [window_start, window_start + q) = sum_e X_e (m_{e+1} - m_e)
//                                          = sum_e X_{e-1} m_e  -  sum_e X_e m_e      (m_24 = q)
// i.e. 12 packed mins and 24 two-way dot products, no branches, no per-entry extraction.
//
// CLUSTER lines.  A window with more than 24 runs (a variant cluster of a pangenome BWT: dozens of
// runs of length 1-3 within ~65 rows) keeps its regular runs and replaces the densest stretch by
// up to four PSEUDO-RUNS -- the stretch's symbols sorted (all A, then C, G, T).  Rank is then exact
// everywhere except strictly inside the stretch; only those positions (0.5 % of the steps on the
// BASELINE index) read a RAW child line: rel counts at its start + 224 symbols at 2 bits each.
// w[13] of a CLUSTER line holds the stretch bounds [s, e) and w[14] the 30-bit index of the first
// child, each as two 15-bit halves with bit 15 set, so that the uniform decode sees four unused
// entries and the "is q inside the stretch" test is two compares.
// TERM flag: the window covers a terminator (byte 1), which has no 2-bit code: it is stored as
// 'A' and rank_A is corrected from the (<= 8) terminator positions kept in the kernel parameters.
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define RBG_HD __host__ __device__ __forceinline__
#else
#define RBG_HD inline
#endif

// Layout 5 (LeafFmt<5>) trades four entries for ABSOLUTE-enough counts: w[0..3] hold four u32 counts relative to a
// superblock of up to 2^32 positions, whose base (F[c] + #c before it: at most 4 x 256 u64 for n < 2^40) sits in
// shared memory -- the per-step L2 request for the superblock count of layout 4 (one of every three L2 requests of
// search_kernel, ncu r1) disappears.  w[4] = heads of entries 0..15, w[5..14] = 20 starts, w[15] = heads of entries
// 16..19 (bits 0-1 of each byte) + the same flags; RAW children keep u16 counts, relative to their WINDOW start.
namespace rbg {

template <int V> struct LeafFmt;
template <> struct LeafFmt<4> { static constexpr int E = 24, S0 = 3, H0 = 2, NX = 6, CE = 20; };   // entries, first start word, head word, match words, entries of a CLUSTER line
template <> struct LeafFmt<5> { static constexpr int E = 20, S0 = 5, H0 = 4, NX = 5, CE = 16; };
template <> struct LeafFmt<6> { static constexpr int E = 12, S0 = 8, H0 = 14, NX = 3, CE = 0; };    // pair line, below

constexpr int kLeafEntries = 24;                    // layout 4 (the larger of the two)
constexpr int kClusterEntries = 20;                 // w[13], w[14] of a CLUSTER line: stretch bounds, child pointer
constexpr uint32_t kLeafPad = 0xFFFFu;
constexpr uint32_t kRawSymbols = 224;               // 14 words x 16 symbols in a RAW child line
constexpr uint32_t kFlagCluster = 1u << 4, kFlagTerm = 1u << 6, kFlagAny = kFlagCluster | kFlagTerm;

RBG_HD uint32_t rbg_vminu2(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __vminu2(a, b);
#else
    const uint32_t lo = (a & 0xFFFFu) < (b & 0xFFFFu) ? (a & 0xFFFFu) : (b & 0xFFFFu);
    const uint32_t hi = (a >> 16) < (b >> 16) ? (a >> 16) : (b >> 16);
    return lo | (hi << 16);
#endif
}
RBG_HD uint32_t rbg_dp2a_lo(uint32_t a, uint32_t b, uint32_t c) {
#if defined(__CUDA_ARCH__)
    return __dp2a_lo(a, b, c);
#else
    return c + (a & 0xFFFFu) * (b & 0xFFu) + (a >> 16) * ((b >> 8) & 0xFFu);
#endif
}
RBG_HD uint32_t rbg_dp2a_hi(uint32_t a, uint32_t b, uint32_t c) {
#if defined(__CUDA_ARCH__)
    return __dp2a_hi(a, b, c);
#else
    return c + (a & 0xFFFFu) * ((b >> 16) & 0xFFu) + (a >> 16) * (b >> 24);
#endif
}
RBG_HD uint32_t rbg_funnel_l8(uint32_t lo, uint32_t hi) {      // (hi:lo) << 8, upper word
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(lo, hi, 8);
#else
    return (hi << 8) | (lo >> 24);
#endif
}
RBG_HD uint32_t rbg_popc(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return (uint32_t) __popc(x);
#else
    return (uint32_t) __builtin_popcount(x);
#endif
}
RBG_HD uint32_t rbg_popc64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return (uint32_t) __popcll(x);
#else
    return (uint32_t) __builtin_popcountll(x);
#endif
}

// Bit position of entry e's head inside its head word (w[2] for e < 16, w[15] for e >= 16).
RBG_HD uint32_t leaf_head_bit(uint32_t e) { return 8u * (e & 3u) + 2u * ((e & 15u) >> 2); }

// Per-symbol state of one LF step: the pattern that turns head fields equal to c into zero.
RBG_HD uint32_t leaf_cpat(uint32_t c) { return c * 0x55555555u; }

// #c in BWT[superblock_start, window_start)
template <int V = 4>
RBG_HD uint32_t leaf_rel_count(const uint32_t (&w)[16], uint32_t c) {
    if (V == 5) {
        const uint32_t a = (c & 1u) ? w[1] : w[0], b = (c & 1u) ? w[3] : w[2];
        return (c & 2u) ? b : a;
    }
    const uint32_t pair = (c & 2u) ? w[1] : w[0];
    return (c & 1u) ? pair >> 16 : pair & 0xFFFFu;
}

// Byte vectors X (entries 4i..4i+3 -> bytes of xb[i], 1 where the head equals c) and the same
// shifted by one entry (xs byte of entry e = X_{e-1}).
template <int V = 4>
RBG_HD void leaf_match(const uint32_t (&w)[16], uint32_t cpat, uint32_t (&xb)[6], uint32_t (&xs)[6]) {
    const uint32_t x = w[LeafFmt<V>::H0] ^ cpat, y = w[15] ^ cpat;
    const uint32_t eq = ~(x | (x >> 1)), eq2 = ~(y | (y >> 1));
    xb[0] = eq & 0x01010101u;
    xb[1] = (eq >> 2) & 0x01010101u;
    xb[2] = (eq >> 4) & 0x01010101u;
    xb[3] = (eq >> 6) & 0x01010101u;
    xb[4] = eq2 & 0x01010101u;
    xb[5] = V == 4 ? (eq2 >> 2) & 0x01010101u : 0u;
    xs[0] = xb[0] << 8;
#pragma unroll
    for (int i = 1; i < 6; ++i) xs[i] = rbg_funnel_l8(xb[i - 1], xb[i]);
}

// #c in [window_start, window_start + q) given the match vectors, q <= W.
template <int V = 4>
RBG_HD uint32_t leaf_rank_x(const uint32_t (&w)[16], const uint32_t (&xb)[6], const uint32_t (&xs)[6], uint32_t q) {
    const uint32_t qq = q | (q << 16);
    uint32_t plus0 = 0, plus1 = 0, minus0 = 0, minus1 = 0;
#pragma unroll
    for (int j = 0; j < LeafFmt<V>::E / 2; ++j) {
        const uint32_t m = rbg_vminu2(qq, w[LeafFmt<V>::S0 + j]);
        if (j & 1) {
            plus1 = rbg_dp2a_hi(m, xs[j >> 1], plus1);
            minus1 = rbg_dp2a_hi(m, xb[j >> 1], minus1);
        } else {
            plus0 = rbg_dp2a_lo(m, xs[j >> 1], plus0);
            minus0 = rbg_dp2a_lo(m, xb[j >> 1], minus0);
        }
    }
    return plus0 + plus1 + (xb[LeafFmt<V>::NX - 1] >> 24) * q - minus0 - minus1;       // + X_last * m_E, m_E = q
}

template <int V = 4>
RBG_HD uint32_t leaf_rank(const uint32_t (&w)[16], uint32_t cpat, uint32_t q) {
    uint32_t xb[6], xs[6];
    leaf_match<V>(w, cpat, xb, xs);
    return leaf_rank_x<V>(w, xb, xs, q);
}

// ---- rare paths -------------------------------------------------------------------------------
RBG_HD uint32_t leaf_flags_word(uint32_t first, uint32_t count) {     // bookkeeping only: where the pseudo-runs sit
    return ((first & 0xFu) << 12) | (((first >> 4) & 1u) << 20) | ((count & 7u) << 28);
}
// The collapsed stretch [s, e) of a CLUSTER line, window-relative.
RBG_HD uint32_t leaf_cluster_begin(const uint32_t (&w)[16]) { return w[13] & 0x7FFFu; }
RBG_HD uint32_t leaf_cluster_end(const uint32_t (&w)[16]) { return (w[13] >> 16) & 0x7FFFu; }
RBG_HD uint32_t leaf_cluster_word(uint32_t s, uint32_t e) { return 0x80008000u | (s & 0x7FFFu) | ((e & 0x7FFFu) << 16); }
RBG_HD bool leaf_inside_cluster(const uint32_t (&w)[16], uint32_t q) {
    return (w[15] & kFlagCluster) && q > leaf_cluster_begin(w) && q < leaf_cluster_end(w);
}
RBG_HD uint32_t leaf_child_ptr(const uint32_t (&w)[16]) { return (w[14] & 0x7FFFu) | (((w[14] >> 16) & 0x7FFFu) << 15); }
RBG_HD uint32_t leaf_child_word(uint32_t ptr) { return 0x80008000u | (ptr & 0x7FFFu) | (((ptr >> 15) & 0x7FFFu) << 16); }

// RAW child line: cw[0..1] rel counts at its first position, cw[2..15] 224 symbols (2 bits each,
// symbol p at bits 2*(p&15) of cw[2 + p/16]).  #c among its first p symbols.  Reads the line from
// memory word by word: this path runs for ~0.5 % of the ranks.
RBG_HD uint32_t raw_rank(const uint32_t* cw, uint32_t cpat, uint32_t p) {
    uint32_t cnt = 0;
    for (uint32_t j = 0; 16u * j < p; ++j) {
        const uint32_t x = cw[2 + j] ^ cpat;
        uint32_t eq = ~(x | (x >> 1)) & 0x55555555u;
        const uint32_t rem = p - 16u * j;
        if (rem < 16u) eq &= (1u << (2u * rem)) - 1u;
        cnt += rbg_popc(eq);
    }
    return cnt;
}
RBG_HD uint32_t raw_rel_count(const uint32_t* cw, uint32_t c) {
    const uint32_t pair = cw[c >> 1];
    return (c & 1u) ? pair >> 16 : pair & 0xFFFFu;
}

// ---- pair lines (LeafFmt<6>) ------------------------------------------------------------------
// The pair directory (PairDir, layout.hpp) is a rank directory over the sequence P[j] = (BWT[LF(j)], BWT[j]), code
// p = 4 c1 + c2, so that one rank answers two LF steps (derivation beside lf_pair_warp, device_index.cuh).  One line:
//   w[0..7]   16 x u16: #p in P[superblock_start, window_start), code p in the (p&1) half of w[p/2]; the absolute part
//             (K[p] + #p before the superblock) is one u32 per code and superblock, kept in shared memory
//   w[8..13]  12 x u16 run starts, entry e in the (e&1) half of w[8 + e/2], as in the single-base lines
//   w[14]     4-bit heads of entries 0..7, TRANSPOSED: entry e at bit 8*(e&3) + 4*(e>>2), so that (eq >> 4i) & 0x01010101
//             is the byte vector of entries 4i..4i+3
//   w[15]     heads of entries 8..11 at bits 8*(e&3) (low nibble of each byte); byte 0 bit 4: CLUSTER, bit 6: TERM
// The rank is leaf_rank_x<6>: the same mins and dot products as the single-base lines, over 12 entries.
// CLUSTER: a window of more than 12 runs keeps its counts, and w[8] holds the index of its first RAW child: the whole
// window's codes at 4 bits (symbol i at bits 4*(i&7) of word i/8 of child i/128; windows are <= 256, so <= 2 children).
// TERM: rows whose pair has a terminator (BWT[j] or BWT[LF(j)] is '$', at most 16) are stored as code 0 in the heads and
// the children but are not counted anywhere else; a rank of code 0 in such a window subtracts them (pair_bad list).
constexpr uint32_t kPairMaxWindow = 256;
constexpr uint32_t kPairRawSymbols = 128;          // 16 words x 8 codes in a pair RAW child line
constexpr int kPairMaxBad = 16;

RBG_HD uint32_t pair_head_bit(uint32_t e) { return e < 8u ? 8u * (e & 3u) + 4u * (e >> 2) : 8u * (e & 3u); }
RBG_HD uint32_t pair_pat(uint32_t p) { return p * 0x11111111u; }

RBG_HD uint32_t pair_rel_count(const uint32_t (&w)[16], uint32_t p) {
    const bool b1 = p & 2u, b2 = p & 4u, b3 = p & 8u;
    const uint32_t w01 = b1 ? w[1] : w[0], w23 = b1 ? w[3] : w[2], w45 = b1 ? w[5] : w[4], w67 = b1 ? w[7] : w[6];
    const uint32_t w03 = b2 ? w23 : w01, w47 = b2 ? w67 : w45;
    const uint32_t x = b3 ? w47 : w03;
    return (p & 1u) ? x >> 16 : x & 0xFFFFu;
}

// 1 in bit 0 of each nibble of x ^ pat that is zero
RBG_HD uint32_t pair_eq_nibbles(uint32_t x) {
    const uint32_t t = x | (x >> 1);
    return ~(t | (t >> 2));
}

RBG_HD void pair_match(const uint32_t (&w)[16], uint32_t ppat, uint32_t (&xb)[6], uint32_t (&xs)[6]) {
    const uint32_t eq = pair_eq_nibbles(w[14] ^ ppat), eq2 = pair_eq_nibbles(w[15] ^ ppat);
    xb[0] = eq & 0x01010101u;
    xb[1] = (eq >> 4) & 0x01010101u;
    xb[2] = eq2 & 0x01010101u;
    xb[3] = xb[4] = xb[5] = 0u;
    xs[0] = xb[0] << 8;
    xs[1] = rbg_funnel_l8(xb[0], xb[1]);
    xs[2] = rbg_funnel_l8(xb[1], xb[2]);
    xs[3] = xs[4] = xs[5] = 0u;
}

RBG_HD uint32_t pair_rank(const uint32_t (&w)[16], uint32_t ppat, uint32_t q) {
    uint32_t xb[6], xs[6];
    pair_match(w, ppat, xb, xs);
    return leaf_rank_x<6>(w, xb, xs, q);
}

RBG_HD uint32_t pair_child_ptr(const uint32_t (&w)[16]) { return w[8]; }

// #p among the first q codes of one word of a pair RAW child whose first code is code `first` of the window
RBG_HD uint32_t pair_raw_word_count(uint32_t word, uint32_t ppat, int first, int q) {
    const int rem = q - first;
    const uint32_t m = rem >= 8 ? 0xFFFFFFFFu : (rem <= 0 ? 0u : (1u << (4 * rem)) - 1u);
    return rbg_popc(pair_eq_nibbles(word ^ ppat) & 0x11111111u & m);
}

// ---- plain lines (layout 7) -------------------------------------------------------------------
// An index whose BWT is small enough to stay in L2 (n < 2^31, <= kPlainMaxBytes of lines) keeps the BWT itself at 2 bits
// per row, in 32-byte lines of 64 rows: the line of row i is i >> 6, with no division, no superblock table and no run decode.
//   w[0..3]   4 x u32: F[c] + #c in BWT[0, line_start), c = A,C,G,T; bit 31 of w[0] is the TERM flag (free: n < 2^31)
//   w[4..5]   the low bit of each row's code, row line_start + j at bit j of the 64-bit word w[5]:w[4]
//   w[6..7]   the high bit, in the same order
// rank_c(line_start + q) = w[c] + popc(match_c & ((1 << q) - 1)), match_c = the rows whose two bits spell c; the count
// up to and including row q uses the mask (2 << q) - 1, so q never reaches 64, and BWT[line_start + q] == c is bit q of
// match_c.  TERM: a terminator rides as code 0 ('A') in the planes but is not counted in w[0]; rank_A in such a line
// subtracts the terminator rows it counted, from the (<= 8) terminator positions kept in the kernel parameters.
constexpr uint32_t kPlainWords = 8, kPlainRows = 64, kPlainShift = 6;
constexpr uint32_t kPlainTerm = 1u << 31;

// the rows of the line that hold code c, row j at bit j
RBG_HD uint64_t plain_match(const uint32_t (&w)[kPlainWords], uint32_t c) {
    const uint32_t xl = (c & 1u) ? 0u : ~0u, xh = (c & 2u) ? 0u : ~0u;
    const uint32_t m0 = (w[4] ^ xl) & (w[6] ^ xh), m1 = (w[5] ^ xl) & (w[7] ^ xh);
    return (uint64_t) m0 | ((uint64_t) m1 << 32);
}
// F[c] + #c in BWT[0, line_start)
RBG_HD uint32_t plain_count(const uint32_t (&w)[kPlainWords], uint32_t c) {
    const uint32_t a = (c & 1u) ? w[1] : w[0] & ~kPlainTerm, b = (c & 1u) ? w[3] : w[2];
    return (c & 2u) ? b : a;
}
// #c among rows [0, q) of the line, q < 64
RBG_HD uint32_t plain_rank_before(uint64_t match, uint32_t q) { return rbg_popc64(match & ((1ull << q) - 1ull)); }
// #c among rows [0, q] of the line, q < 64
RBG_HD uint32_t plain_rank_upto(uint64_t match, uint32_t q) { return rbg_popc64(match & ((2ull << q) - 1ull)); }

}  // namespace rbg
