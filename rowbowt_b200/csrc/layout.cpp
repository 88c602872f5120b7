// See layout.hpp.
#include "layout.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <thread>

#include "leaf.cuh"
#include "phi_slot.cuh"

namespace rbg {
namespace {

struct Piece { uint32_t start; uint8_t code; };      // one run clipped to a window, window-relative start

// One direct line from `ent` (at most `max_entries`) and the symbol counts relative to the superblock start, in
// layout V (leaf.cuh: 4 = 24 entries + u16 counts, 5 = 20 entries + u32 counts).
template <int V>
void emit_line(uint32_t* w, const std::vector<Piece>& ent, const uint64_t rel[4], uint32_t flags, int max_entries) {
    constexpr int E = LeafFmt<V>::E, S0 = LeafFmt<V>::S0, H0 = LeafFmt<V>::H0;
    if (ent.size() > (size_t) max_entries) throw std::logic_error("leaf overflow");
    memset(w, 0, 64);
    if (V == 5) {
        for (int c = 0; c < 4; ++c) {
            if (rel[c] >> 32) throw std::logic_error("superblock-relative count exceeds 32 bits");
            w[c] = (uint32_t) rel[c];
        }
    } else {
        for (int c = 0; c < 4; ++c)
            if (rel[c] > 0xFFFFu) throw std::logic_error("superblock-relative count exceeds 16 bits");
        w[0] = (uint32_t) rel[0] | ((uint32_t) rel[1] << 16);
        w[1] = (uint32_t) rel[2] | ((uint32_t) rel[3] << 16);
    }
    uint16_t st[E];
    for (int e = 0; e < E; ++e) st[e] = (uint16_t) kLeafPad;
    for (size_t e = 0; e < ent.size(); ++e) {
        uint32_t code = ent[e].code;
        if (code == 4) { code = 0; flags |= kFlagTerm; }      // terminator rides as an 'A' entry, corrected in the kernel
        st[e] = (uint16_t) ent[e].start;
        w[e < 16 ? H0 : 15] |= code << leaf_head_bit((uint32_t) e);
    }
    for (int j = 0; j < E / 2; ++j) w[S0 + j] = (uint32_t) st[2 * j] | ((uint32_t) st[2 * j + 1] << 16);
    w[15] |= flags;
}

// Walks the runs window by window.  out == nullptr: only counts lines.
template <int V>
struct LeafWalker {
    const RunsBwt& bwt;
    const int8_t* code;
    uint32_t W, sb_shift;
    static constexpr int kE = LeafFmt<V>::E, kCE = LeafFmt<V>::CE;
    void run(LeafDir* out, uint64_t& n_children, uint64_t& n_cluster, const uint64_t Fcode[4], uint64_t* stretch_positions = nullptr) const {
        const uint64_t n_direct = (bwt.n + W - 1) / W;
        uint64_t j = 0, jstart = 0;                 // run covering the current window start
        uint64_t cum[4] = {0, 0, 0, 0};             // symbol counts in BWT[0, jstart)
        uint64_t sb_base[4] = {0, 0, 0, 0};         // symbol counts at the current superblock start
        n_children = n_cluster = 0;
        std::vector<Piece> pc, ent;
        std::vector<uint8_t> raw;
        for (uint64_t t = 0; t < n_direct; ++t) {
            const uint64_t P = t * W, Pend = std::min(P + W, bwt.n);
            const uint32_t wend = (uint32_t) (Pend - P);
            while (jstart + bwt.lens[j] <= P) {
                const int8_t c = code[bwt.heads[j]];
                if (c < 4) cum[c] += bwt.lens[j];
                jstart += bwt.lens[j];
                ++j;
            }
            pc.clear();
            uint64_t st = jstart;
            for (uint64_t i = j; i < bwt.R && st < Pend; st += bwt.lens[i], ++i)
                pc.push_back({(uint32_t) (st > P ? st - P : 0), (uint8_t) code[bwt.heads[i]]});
            const size_t np = pc.size();
            uint64_t at[4];                         // counts at the window start
            for (int c = 0; c < 4; ++c) at[c] = cum[c];
            const int8_t c0 = code[bwt.heads[j]];
            if (c0 < 4) at[c0] += P - jstart;
            if ((t & ((1ull << sb_shift) - 1)) == 0) {
                for (int c = 0; c < 4; ++c) sb_base[c] = at[c];
                if (out) for (int c = 0; c < 4; ++c) out->super[(uint64_t) c * out->n_super + (t >> sb_shift)] = Fcode[c] + at[c];
            }
            uint64_t rel[4];
            for (int c = 0; c < 4; ++c) rel[c] = at[c] - sb_base[c];
            if (np <= (size_t) kE) {
                if (out) emit_line<V>(out->lines.data() + t * kLineWords, pc, rel, 0, kE);
                continue;
            }
            // too many runs: collapse the k = np - (CE - 4) consecutive pieces that span the fewest positions
            const size_t k = np - (kCE - 4);
            auto start_of = [&](size_t i) { return i < np ? pc[i].start : wend; };
            size_t best = 0;
            for (size_t i = 1; i + k <= np; ++i)
                if (start_of(i + k) - start_of(i) < start_of(best + k) - start_of(best)) best = i;
            const uint32_t s = start_of(best), e = start_of(best + k);
            const uint64_t nchild = (e - s + kRawSymbols - 1) / kRawSymbols;
            ++n_cluster;
            if (stretch_positions) *stretch_positions += e - s;
            if (out) {
                const uint64_t child0 = n_direct + n_children;
                if ((child0 + nchild) >> 30) throw std::runtime_error("rank directory exceeds 2^30 lines");
                uint64_t in[5] = {0, 0, 0, 0, 0};
                raw.assign(e - s, 0);
                for (size_t i = best; i < best + k; ++i) {
                    const uint32_t a = start_of(i), z = start_of(i + 1);
                    in[pc[i].code] += z - a;
                    for (uint32_t p = a; p < z; ++p) raw[p - s] = pc[i].code;
                }
                uint32_t flags = kFlagCluster;
                if (in[4]) { in[0] += in[4]; flags |= kFlagTerm; }          // terminators count as 'A' inside the stretch too
                ent.assign(pc.begin(), pc.begin() + best);
                uint32_t pos = s, n_pseudo = 0;
                for (uint8_t c = 0; c < 4; ++c)
                    if (in[c]) { ent.push_back({pos, c}); pos += (uint32_t) in[c]; ++n_pseudo; }
                ent.insert(ent.end(), pc.begin() + best + k, pc.end());
                flags |= leaf_flags_word((uint32_t) best, n_pseudo);
                uint32_t* w = out->lines.data() + t * kLineWords;
                emit_line<V>(w, ent, rel, flags, kCE);
                w[13] = leaf_cluster_word(s, e);
                w[14] = leaf_child_word((uint32_t) child0);
                // raw children: counts at each child's first position (layout 4: relative to the superblock like the
                // line's own; layout 5: relative to the WINDOW start, added to the line's u32 counts), then 224 symbols
                uint64_t crel[4];
                for (int c = 0; c < 4; ++c) crel[c] = V == 5 ? 0 : rel[c];
                for (size_t i = 0; i < best; ++i) if (pc[i].code < 4) crel[pc[i].code] += start_of(i + 1) - start_of(i);
                for (uint64_t ch = 0; ch < nchild; ++ch) {
                    uint32_t* cw = out->lines.data() + (child0 + ch) * kLineWords;
                    memset(cw, 0, 64);
                    for (int c = 0; c < 4; ++c) if (crel[c] > 0xFFFFu) throw std::logic_error("raw child count exceeds 16 bits");
                    cw[0] = (uint32_t) crel[0] | ((uint32_t) crel[1] << 16);
                    cw[1] = (uint32_t) crel[2] | ((uint32_t) crel[3] << 16);
                    const uint32_t a = (uint32_t) (ch * kRawSymbols), z = std::min<uint32_t>(a + kRawSymbols, e - s);
                    for (uint32_t p = a; p < z; ++p) {
                        // a terminator is written as 'A' (corrected in the kernel) but is not an 'A' for later counts
                        cw[2 + ((p - a) >> 4)] |= (uint32_t) (raw[p] & 3u) << (2 * ((p - a) & 15));
                        if (raw[p] < 4) crel[raw[p]] += 1;
                    }
                }
            }
            n_children += nchild;
        }
    }
};

// Layout 7 (leaf.cuh, plain lines): the runs expanded into 2-bit planes, 64 rows per line, with the counts in front of each
// line.  O(n / 64 + R), cut into contiguous parts of lines, one per host thread.
void build_plain_lines(const RunsBwt& bwt, const int8_t* code, LeafDir& d) {
    d.version = 7;
    d.window = kPlainRows;
    d.magic = ~0ull / kPlainRows + 1;
    d.n_direct = (bwt.n + kPlainRows - 1) / kPlainRows;
    d.sb_shift = 31 - kPlainShift;                      // one superblock (all zero) covers every line of an index below 2^31 rows
    d.n_super = 1;
    d.super.assign(4, 0);
    d.n_cluster = 0;
    d.lines.assign(d.n_direct * kPlainWords, 0);
    const unsigned n_parts = d.n_direct >= (1u << 16) ? std::max(1u, std::min(16u, std::thread::hardware_concurrency())) : 1u;
    struct Start { uint64_t j, jstart, cum[4]; };         // the run covering a part's first row, its start, counts in front of it
    std::vector<Start> start(n_parts);
    {
        Start s{0, 0, {0, 0, 0, 0}};
        for (unsigned p = 0; p < n_parts; ++p) {
            const uint64_t P0 = d.n_direct * p / n_parts * kPlainRows;
            while (s.jstart + bwt.lens[s.j] <= P0) {
                const int8_t c = code[bwt.heads[s.j]];
                if (c < 4) s.cum[c] += bwt.lens[s.j];
                s.jstart += bwt.lens[s.j];
                ++s.j;
            }
            start[p] = s;
        }
    }
    auto part = [&](unsigned p) {
        Start s = start[p];
        const uint64_t t1 = d.n_direct * (p + 1) / n_parts;
        for (uint64_t t = d.n_direct * p / n_parts; t < t1; ++t) {
            const uint64_t P = t * kPlainRows, Pend = std::min<uint64_t>(P + kPlainRows, bwt.n);
            while (s.jstart + bwt.lens[s.j] <= P) {
                const int8_t c = code[bwt.heads[s.j]];
                if (c < 4) s.cum[c] += bwt.lens[s.j];
                s.jstart += bwt.lens[s.j];
                ++s.j;
            }
            uint32_t* w = d.lines.data() + t * kPlainWords;
            const int8_t c0 = code[bwt.heads[s.j]];
            for (int c = 0; c < 4; ++c) w[c] = (uint32_t) (d.Fcode[c] + s.cum[c] + (c == c0 ? P - s.jstart : 0));
            uint64_t plane[2] = {0, 0};
            for (uint64_t i = s.j, at = s.jstart; i < bwt.R && at < Pend; at += bwt.lens[i], ++i) {
                const uint64_t a = std::max(at, P), z = std::min(at + bwt.lens[i], Pend);
                const uint64_t m = (z - a == kPlainRows ? ~0ull : (1ull << (z - a)) - 1ull) << (a - P);
                uint32_t c = (uint32_t) code[bwt.heads[i]];
                if (c == 4) { c = 0; w[0] |= kPlainTerm; }     // the terminator rides as 'A', uncounted
                if (c & 1u) plane[0] |= m;
                if (c & 2u) plane[1] |= m;
            }
            w[4] = (uint32_t) plane[0];
            w[5] = (uint32_t) (plane[0] >> 32);
            w[6] = (uint32_t) plane[1];
            w[7] = (uint32_t) (plane[1] >> 32);
        }
    };
    if (n_parts == 1) {
        part(0);
    } else {
        std::vector<std::thread> th;
        for (unsigned p = 0; p < n_parts; ++p) th.emplace_back(part, p);
        for (auto& t : th) t.join();
    }
}

}  // namespace

PredTable build_pred_table(std::vector<uint64_t>&& keys, uint64_t universe, double keys_per_bucket) {
    PredTable t;
    t.keys = std::move(keys);
    const double want = std::max(1.0, (double) t.keys.size() / keys_per_bucket);
    uint32_t shift = 0;
    while (shift < 63 && (double) (universe >> shift) > want) ++shift;
    t.shift = shift;
    const uint64_t nb = (universe >> shift) + 2;
    t.table.assign(nb + 1, 0);
    // table[b] = #keys < (b << shift)
    size_t i = 0;
    for (uint64_t b = 0; b <= nb; ++b) {
        const uint64_t lim = b << shift;
        while (i < t.keys.size() && t.keys[i] < lim) ++i;
        t.table[b] = (uint32_t) i;
    }
    if (t.keys.size() >> 32) throw std::runtime_error("more than 2^32 keys in a PredTable");
    return t;
}

LeafDir build_leaf_dir(const RunsBwt& bwt, uint32_t window, int layout) {
    LeafDir d;
    d.n = bwt.n;
    if (bwt.n == 0 || bwt.R == 0) throw format_error("empty BWT");
    static const uint8_t sym[4] = {'A', 'C', 'G', 'T'};
    int8_t code[256];
    memset(code, -1, sizeof code);
    for (int c = 0; c < 4; ++c) code[sym[c]] = (int8_t) c;
    code[1] = 4;
    uint64_t counts256[256] = {0};
    uint64_t pos = 0;
    for (uint64_t j = 0; j < bwt.R; ++j) {
        const uint8_t h = bwt.heads[j];
        if (code[h] < 0)
            throw alphabet_error("BWT contains byte " + std::to_string((int) h) +
                                 ": only {terminator,A,C,G,T} indexes are supported (build with pfbwt-f --non-acgt-to-a)");
        if (bwt.lens[j] == 0) throw format_error("zero-length run");
        if (code[h] == 4)
            for (uint64_t t = 0; t < bwt.lens[j]; ++t) {
                if (d.n_term >= (uint32_t) kMaxTerm) throw alphabet_error("more than 8 terminator symbols in the BWT");
                d.term_pos[d.n_term++] = pos + t;
            }
        counts256[h] += bwt.lens[j];
        pos += bwt.lens[j];
    }
    if (pos != bwt.n) throw format_error("run lengths do not sum to n");
    if (bwt.n >> 40) throw std::runtime_error("BWT longer than 2^40 positions");
    d.F[0] = 0;                                                     // RowBowt::build_f, include/rowbowt.hpp:770-778
    for (int i = 0; i < 255; ++i) d.F[i + 1] = d.F[i] + counts256[i];
    for (int c = 0; c < 4; ++c) { d.Fcode[c] = d.F[sym[c]]; d.count[c] = counts256[sym[c]]; }
    memset(d.code_of, -1, sizeof d.code_of);
    for (int c = 0; c < 4; ++c) if (d.count[c]) d.code_of[sym[c]] = (int8_t) c;
    if (d.n_term) d.code_of[1] = 4;

    // layout 7 while the plain lines stay L2-resident (kPlainMaxBytes); a forced window asks for a run-length layout
    const uint64_t plain_bytes = (bwt.n + kPlainRows - 1) / kPlainRows * kPlainWords * 4;
    if (layout == 7 || (layout == 0 && window == 0 && (bwt.n >> 31) == 0 && plain_bytes <= kPlainMaxBytes)) {
        if (bwt.n >> 31) throw std::runtime_error("layout 7: BWT of 2^31 positions or more");
        build_plain_lines(bwt, code, d);
        return d;
    }

    // layout 4: a superblock is <= 65535 positions (u16 counts); layout 5: <= 2^32 positions (u32 counts)
    auto sb_shift_for = [](int V, uint32_t W) {
        const uint64_t cap = V == 5 ? (1ull << 32) : 65535ull;
        uint32_t s = 0;
        while (((uint64_t) W << (s + 1)) <= cap) ++s;
        return s;
    };
    struct Count { uint64_t children = 0, clusters = 0, stretch = 0; };
    auto count_lines = [&](int V, uint32_t W) {               // read-only walk: safe to run for several W at once
        Count c;
        if (V == 5) LeafWalker<5>{bwt, code, W, sb_shift_for(5, W)}.run(nullptr, c.children, c.clusters, d.Fcode, &c.stretch);
        else LeafWalker<4>{bwt, code, W, sb_shift_for(4, W)}.run(nullptr, c.children, c.clusters, d.Fcode, &c.stretch);
        return c;
    };
    // Which layout: `layout` 4|5 forces one; otherwise 5 (no per-step superblock load) while its directory stays
    // within the reach of the SM TLBs with room for the seed table and the reads (<= 224 MB), else 4 (3.8 instead of
    // 4.6 bytes per run: the gather rate falls 2.5x once the footprint passes 256 MB, profiles/r1_gather_sweep.jsonl).
    uint32_t W = window;
    auto choose_window = [&](int V, uint32_t& Wout, Count& chosen) {
        // aim at ~71 % of the entries used on average; try a ladder of eighths around it.  Cost of a candidate:
        // its lines (footprint decides the gather rate), inflated by the share of positions that fall inside a
        // collapsed stretch (each such rank is a second dependent load that stalls its whole warp).
        const int E = V == 5 ? LeafFmt<5>::E : LeafFmt<4>::E;
        const double target = (17.0 * E / 24.0) * (double) bwt.n / (double) bwt.R;
        const uint32_t unit = std::max<uint32_t>(2, 1u << (uint32_t) std::max(1.0, std::floor(std::log2(target)) - 3.0));
        constexpr int kLadder = 8;
        uint32_t cand[kLadder];
        Count cnt[kLadder];
        for (int k = 0; k < kLadder; ++k) {
            const int64_t cand64 = ((int64_t) (target / unit) + (k - 3)) * (int64_t) unit;
            cand[k] = (uint32_t) std::min<int64_t>(kMaxWindow, std::max<int64_t>(kMinWindow, cand64));
        }
        if (bwt.R > (1u << 20)) {                                // the candidates are independent walks over the runs
            std::vector<std::thread> th;
            for (int k = 0; k < kLadder; ++k) th.emplace_back([&, k] { cnt[k] = count_lines(V, cand[k]); });
            for (auto& t : th) t.join();
        } else {
            for (int k = 0; k < kLadder; ++k) cnt[k] = count_lines(V, cand[k]);
        }
        double best = 1e300;
        for (int k = 0; k < kLadder; ++k) {
            const double lines = (double) ((bwt.n + cand[k] - 1) / cand[k] + cnt[k].children);
            const double cost = lines * (1.0 + 20.0 * (double) cnt[k].stretch / (double) bwt.n);
            if (cost < best) { best = cost; Wout = cand[k]; chosen = cnt[k]; }
        }
        return ((bwt.n + Wout - 1) / Wout + chosen.children) * 64;       // directory bytes
    };
    Count chosen;
    int V = layout ? layout : 5;
    if (W == 0) {
        uint64_t bytes = choose_window(V, W, chosen);
        if (!layout && bytes > (224ull << 20)) {
            V = 4;
            W = 0;
            bytes = choose_window(4, W, chosen);
        }
    } else if (W >= kMinWindow && W <= kMaxWindow) {
        chosen = count_lines(V, W);
    }
    if (W < kMinWindow || W > kMaxWindow) throw std::runtime_error("window out of range [16,32767]");
    d.version = V;
    d.window = W;
    d.magic = ~0ull / W + 1;            // ceil(2^64 / W): umul64hi(i, magic) == i / W while i * W < 2^64
    d.sb_shift = sb_shift_for(V, W);
    d.n_direct = (bwt.n + W - 1) / W;
    d.n_super = (d.n_direct + (1ull << d.sb_shift) - 1) >> d.sb_shift;
    if (V == 5 && d.n_super > (uint64_t) kMaxSuper5) throw std::runtime_error("layout 5: more than 256 superblocks");
    uint64_t children = chosen.children;
    d.lines.assign((d.n_direct + children) * kLineWords, 0);
    d.super.assign(4 * d.n_super, 0);
    if (V == 5) LeafWalker<5>{bwt, code, W, d.sb_shift}.run(&d, children, d.n_cluster, d.Fcode);
    else LeafWalker<4>{bwt, code, W, d.sb_shift}.run(&d, children, d.n_cluster, d.Fcode);
    return d;
}

namespace {
int8_t sym_code(uint8_t h) { return h == 'A' ? 0 : h == 'C' ? 1 : h == 'G' ? 2 : h == 'T' ? 3 : 4; }      // validated by build_leaf_dir
}  // namespace

void pair_runs(const RunsBwt& bwt, const LeafDir& d, std::vector<uint32_t>& lens, std::vector<uint8_t>& codes) {
    if (bwt.n >> 32) throw std::runtime_error("pair directory: n >= 2^32");
    std::vector<uint64_t> start(bwt.R + 1, 0);
    for (uint64_t k = 0; k < bwt.R; ++k) start[k + 1] = start[k] + bwt.lens[k];
    lens.clear();
    codes.clear();
    lens.reserve(2 * bwt.R);
    codes.reserve(2 * bwt.R);
    auto push = [&](uint64_t len, uint8_t code) {
        if (!codes.empty() && codes.back() == code && code != kPairBad) lens.back() += (uint32_t) len;
        else { lens.push_back((uint32_t) len); codes.push_back(code); }
    };
    uint64_t cum[4] = {0, 0, 0, 0};
    for (uint64_t k = 0; k < bwt.R; ++k) {
        const int8_t c = sym_code(bwt.heads[k]);
        if (c == 4) { push(bwt.lens[k], kPairBad); continue; }
        // rows [start[k], start[k+1]) map onto [a, a + len): the first symbols of their pairs are BWT[a, a + len)
        uint64_t a = d.Fcode[c] + cum[c], left = bwt.lens[k];
        cum[c] += left;
        uint64_t m = (uint64_t) (std::upper_bound(start.begin(), start.end(), a) - start.begin()) - 1;
        while (left) {
            const uint64_t take = std::min(left, start[m + 1] - a);
            const int8_t c1 = sym_code(bwt.heads[m]);
            push(take, c1 == 4 ? kPairBad : (uint8_t) (4 * c1 + c));
            a += take;
            left -= take;
            ++m;
        }
    }
}

namespace {

struct PairCount { uint64_t children = 0, clusters = 0, positions = 0; };

// Walks the runs of P window by window (as LeafWalker does for the BWT).  out == nullptr: only counts.
PairCount pair_walk(const std::vector<uint32_t>& lens, const std::vector<uint8_t>& codes, uint64_t n, uint32_t W,
                    uint32_t sb_shift, const uint32_t K[16], PairDir* out) {
    constexpr int E = LeafFmt<6>::E;
    const uint64_t n_direct = (n + W - 1) / W, n_child = (W + kPairRawSymbols - 1) / kPairRawSymbols;
    PairCount pc;
    uint64_t j = 0, jstart = 0, cum[16] = {0}, sb[16] = {0};
    for (uint64_t t = 0; t < n_direct; ++t) {
        const uint64_t P = t * W, Pend = std::min(P + W, n);
        while (jstart + lens[j] <= P) {
            if (codes[j] < kPairBad) cum[codes[j]] += lens[j];
            jstart += lens[j];
            ++j;
        }
        uint64_t at[16];
        for (int p = 0; p < 16; ++p) at[p] = cum[p];
        if (codes[j] < kPairBad) at[codes[j]] += P - jstart;
        if ((t & ((1ull << sb_shift) - 1)) == 0) {
            for (int p = 0; p < 16; ++p) sb[p] = at[p];
            if (out) for (int p = 0; p < 16; ++p) out->super[(uint64_t) p * out->n_super + (t >> sb_shift)] = (uint32_t) (K[p] + at[p]);
        }
        size_t np = 0;
        bool term = false;
        for (uint64_t i = j, st = jstart; i < lens.size() && st < Pend; st += lens[i], ++i) { ++np; term |= codes[i] == kPairBad; }
        const bool cluster = np > (size_t) E;
        if (cluster) { ++pc.clusters; pc.positions += Pend - P; }
        if (out) {
            uint32_t* w = out->lines.data() + t * kLineWords;
            memset(w, 0, 64);
            for (int p = 0; p < 16; ++p) {
                const uint64_t rel = at[p] - sb[p];
                if (rel > 0xFFFFu) throw std::logic_error("pair line: superblock-relative count exceeds 16 bits");
                w[p >> 1] |= (uint32_t) rel << (16 * (p & 1));
            }
            for (int e = 0; e < E / 2; ++e) w[LeafFmt<6>::S0 + e] = 0xFFFFFFFFu;
            if (!cluster) {
                uint64_t st = jstart;
                for (uint64_t i = j, e = 0; e < np; st += lens[i], ++i, ++e) {
                    const uint32_t s = (uint32_t) (st > P ? st - P : 0);
                    uint32_t& sw = w[LeafFmt<6>::S0 + e / 2];
                    sw = (sw & ~(0xFFFFu << (16 * (e & 1)))) | (s << (16 * (e & 1)));
                    w[e < 8 ? 14 : 15] |= (uint32_t) (codes[i] & 15u) << pair_head_bit((uint32_t) e);
                }
            } else {
                const uint64_t child0 = n_direct + pc.children;
                if ((child0 + n_child) >> 32) throw std::runtime_error("pair directory exceeds 2^32 lines");
                w[LeafFmt<6>::S0] = (uint32_t) child0;
                uint32_t* cw = out->lines.data() + child0 * kLineWords;
                memset(cw, 0, 64 * n_child);
                uint64_t st = jstart;
                for (uint64_t i = j; i < lens.size() && st < Pend; st += lens[i], ++i)
                    for (uint64_t r = std::max(st, P); r < std::min(st + lens[i], Pend); ++r)
                        cw[(r - P) >> 3] |= (uint32_t) (codes[i] & 15u) << (4 * ((r - P) & 7));
                w[15] |= kFlagCluster;
            }
            if (term) w[15] |= kFlagTerm;
        }
        if (cluster) pc.children += n_child;
    }
    return pc;
}

uint32_t pair_sb_shift(uint32_t W) {                  // largest s with (2^s - 1) * W <= 65535: the u16 counts of a line
    uint32_t s = 0;
    while (((2ull << s) - 1) * W <= 65535ull) ++s;
    return s;
}

}  // namespace

PairDir build_pair_dir(const RunsBwt& bwt, const LeafDir& d, uint32_t window) {
    PairDir P;
    P.n = bwt.n;
    std::vector<uint32_t> lens;
    std::vector<uint8_t> codes;
    pair_runs(bwt, d, lens, codes);
    P.n_runs = lens.size();
    uint64_t pos = 0;
    for (size_t i = 0; i < lens.size(); ++i) {
        if (codes[i] == kPairBad)
            for (uint32_t t = 0; t < lens[i]; ++t) {
                if (P.n_bad >= (uint32_t) kPairMaxBad) throw std::logic_error("pair directory: more than 16 terminator rows");
                P.bad_pos[P.n_bad++] = (uint32_t) (pos + t);
            }
        pos += lens[i];
    }
    // K[4 c1 + c2] = F[c1] + rank_c1(F[c2]): where the rows of c1 that precede block c2 end
    uint32_t K[16];
    for (int c2 = 0; c2 < 4; ++c2) {
        uint64_t before[4] = {0, 0, 0, 0}, at = 0;
        for (uint64_t k = 0; k < bwt.R && at < d.Fcode[c2]; ++k) {
            const int8_t c = sym_code(bwt.heads[k]);
            const uint64_t take = std::min<uint64_t>(bwt.lens[k], d.Fcode[c2] - at);
            if (c < 4) before[c] += take;
            at += take;
        }
        for (int c1 = 0; c1 < 4; ++c1) K[4 * c1 + c2] = (uint32_t) (d.Fcode[c1] + before[c1]);
    }
    uint32_t W = window;
    if (W == 0) {
        // the ladder of build_leaf_dir with E = 12; a rank in a CLUSTER window is answered by the whole warp from its raw
        // children, so those windows weigh as in the single-base cost model
        const double target = (17.0 * LeafFmt<6>::E / 24.0) * (double) bwt.n / (double) lens.size();
        const uint32_t unit = std::max<uint32_t>(2, 1u << (uint32_t) std::max(1.0, std::floor(std::log2(target)) - 3.0));
        double best = 1e300;
        for (int k = 0; k < 8; ++k) {
            const int64_t c64 = ((int64_t) (target / unit) + (k - 3)) * (int64_t) unit;
            const uint32_t cand = (uint32_t) std::min<int64_t>(kPairMaxWindow, std::max<int64_t>(kMinWindow, c64)) & ~1u;
            const PairCount c = pair_walk(lens, codes, bwt.n, cand, pair_sb_shift(cand), K, nullptr);
            const double cost = (double) ((bwt.n + cand - 1) / cand + c.children) * (1.0 + 20.0 * (double) c.positions / (double) bwt.n);
            if (cost < best) { best = cost; W = cand; }
        }
    }
    if (W < kMinWindow || W > kPairMaxWindow || (W & 1u)) throw std::runtime_error("pair window must be even, in [16,256]");
    P.window = W;
    P.sb_shift = pair_sb_shift(W);
    P.n_direct = (bwt.n + W - 1) / W;
    P.n_super = (P.n_direct + (1ull << P.sb_shift) - 1) >> P.sb_shift;
    const PairCount c = pair_walk(lens, codes, bwt.n, W, P.sb_shift, K, nullptr);
    P.lines.assign((P.n_direct + c.children) * kLineWords, 0);
    P.super.assign(16 * P.n_super, 0);
    P.n_cluster = pair_walk(lens, codes, bwt.n, W, P.sb_shift, K, &P).clusters;
    return P;
}

ToeholdDir build_toehold_dir(const RunsBwt& bwt, const uint64_t (&F)[256], const ToeholdArrays& tsa, uint32_t shift) {
    if (tsa.r != bwt.R || tsa.n != bwt.n) throw format_error("toehold SA does not match the BWT (r/n differ)");
    ToeholdDir t;
    // LF(end of run j) = F[c] + (#c in BWT[0, end_j]) - 1.  Visiting symbols in byte order and runs in
    // BWT order enumerates these rows in increasing order.
    std::vector<uint64_t> rows(bwt.R), sample(bwt.R);
    uint64_t cnt[256] = {0}, fill[256];
    for (uint64_t j = 0; j < bwt.R; ++j) cnt[bwt.heads[j]]++;
    uint64_t acc = 0;
    for (int c = 0; c < 256; ++c) { fill[c] = acc; acc += cnt[c]; }
    uint64_t seen[256] = {0};
    for (uint64_t j = 0; j < bwt.R; ++j) {
        const uint8_t c = bwt.heads[j];
        seen[c] += bwt.lens[j];
        const uint64_t slot = fill[c]++;
        rows[slot] = F[c] + seen[c] - 1;
        sample[slot] = tsa.samples_last[j];
    }
    if (shift == 0) {
        // bucket width: about three keys per bucket, so that the table (4 B per bucket) stays smaller than the keys' samples
        shift = 1;
        while (shift < 32 && (double) (1ull << shift) < 2.0 * (double) bwt.n / (double) bwt.R) ++shift;
    }
    if (shift > 32) throw std::runtime_error("toehold bucket shift out of range [1,32]");
    t.shift = shift;
    t.key_bytes = shift <= 8 ? 1 : shift <= 16 ? 2 : 4;
    t.n_keys = bwt.R;
    if (bwt.R >> 32) throw std::runtime_error("more than 2^32 runs");
    const uint64_t nb = (bwt.n >> shift) + 2;
    t.table.assign(nb + 1, 0);
    t.keys.resize(bwt.R * t.key_bytes);
    t.sample.init(bwt.n, bwt.R);
    const uint64_t mask = shift >= 64 ? ~0ull : (1ull << shift) - 1;
    size_t i = 0;
    for (uint64_t b = 0; b <= nb; ++b) {
        const uint64_t lim = b << shift;
        while (i < rows.size() && rows[i] < lim) ++i;
        t.table[b] = (uint32_t) i;
    }
    for (uint64_t k = 0; k < bwt.R; ++k) {
        if (k && rows[k] <= rows[k - 1]) throw format_error("toehold directory: LF images of run ends not ascending");
        const uint64_t low = rows[k] & mask;
        if (t.key_bytes == 1) t.keys[k] = (uint8_t) low;
        else if (t.key_bytes == 2) { const uint16_t v = (uint16_t) low; memcpy(&t.keys[2 * k], &v, 2); }
        else { const uint32_t v = (uint32_t) low; memcpy(&t.keys[4 * k], &v, 4); }
        t.sample.push(sample[k]);
    }
    t.toehold0 = (tsa.samples_last[tsa.r - 1] + 1) % tsa.n;     // include/toehold_sa.hpp:97-99
    return t;
}

uint64_t toehold_dir_rank(const ToeholdDir& t, uint64_t row) {
    const uint64_t b = row >> t.shift;
    const uint64_t low = row & ((1ull << t.shift) - 1);
    uint64_t a = t.table[b], z = t.table[b + 1];
    while (a < z) {
        const uint64_t mid = (a + z) >> 1;
        uint64_t k;
        if (t.key_bytes == 1) k = t.keys[mid];
        else if (t.key_bytes == 2) { uint16_t v; memcpy(&v, &t.keys[2 * mid], 2); k = v; }
        else { uint32_t v; memcpy(&v, &t.keys[4 * mid], 4); k = v; }
        if (k < low) a = mid + 1; else z = mid;
    }
    return a;
}

PhiDir build_phi_dir(const ToeholdArrays& tsa, uint32_t shift, unsigned n_parts, uint64_t max_slot_bytes) {
    PhiDir p;
    const uint64_t r = tsa.r, n = tsa.n;
    if (r == 0) throw format_error("toehold SA without samples");
    const std::vector<uint64_t>& keys = tsa.pred;               // ascending text positions
    auto prev_of = [&](uint64_t jr) {
        const uint64_t run = tsa.pred_to_run[jr];
        // pred_to_run == 0 only for phi(SA[0]), which locate_range never evaluates (toehold_sa.hpp:65-66)
        return run ? tsa.samples_last[run - 1] : 0;
    };
    if (shift == 0) {
        // 128-position buckets (the largest a BITMAP slot covers); larger ones only when the slots
        // would not fit the budget -- their crowded buckets are binary-searched instead
        shift = kPhiBitmapShift;
        // (slots exist for non-empty buckets only: at most min(r, buckets) + 1 of them)
        while (shift < kPhiMaxShift && (std::min<uint64_t>(r, (n >> shift) + 1) + 1) * 32 + ((n >> shift) / 32 + 2) * 8 > max_slot_bytes) ++shift;
    }
    if (shift < 1 || shift > kPhiMaxShift) throw std::runtime_error("phi bucket shift out of range [1,16]");
    const bool bitmap = shift <= kPhiBitmapShift;
    p.shift = shift;
    p.n_buckets = (n >> shift) + 1;
    p.l1.assign(p.n_buckets / 32 + 1, 0);
    // One slot per NON-EMPTY bucket, plus a sentinel: a position in an empty bucket is answered by the carry of
    // the next slot (no sample lies between the bucket and that slot's own bucket).  The keys are cut into parts at
    // 32-bucket group boundaries (no l1 word is shared) and the parts are built on their own threads -- the work is
    // the random reads of prev_of; indexes into the dense value arrays are part-local until the parts are joined.
    struct Part {
        uint64_t ka = 0, kz = 0, first_bucket = 0, last_bucket = 0, n_over = 0;
        std::vector<uint64_t> slots, ovf_prev, ovf_keys;
        std::string err;
    };
    auto group_of = [&](uint64_t k) { return (keys[k] >> shift) >> 5; };
    if (n_parts == 0) n_parts = r > (1u << 20) ? std::min(8u, std::max(1u, std::thread::hardware_concurrency())) : 1u;
    std::vector<Part> parts(n_parts);
    for (unsigned t = 0; t < n_parts; ++t) {
        uint64_t ka = r * t / n_parts;
        while (ka > 0 && ka < r && group_of(ka) == group_of(ka - 1)) ++ka;
        parts[t].ka = ka;
        if (t) parts[t - 1].kz = ka;
    }
    parts[n_parts - 1].kz = r;
    auto build_part = [&](Part& out) {
        uint64_t a = out.ka;                                     // first key not yet placed
        bool first = true;
        while (a < out.kz) {
            const uint64_t b = keys[a] >> shift;
            if (b >= p.n_buckets) { out.err = "toehold SA: sampled position beyond n"; return; }
            uint64_t z = a;
            while (z < out.kz && (keys[z] >> shift) == b) ++z;
            if (z < out.kz && (keys[z] >> shift) < b) { out.err = "toehold SA: sampled positions not ascending"; return; }
            if (first) { out.first_bucket = b; first = false; }
            out.last_bucket = b;
            const uint64_t cnt = z - a;
            p.l1[b >> 5] |= 1ull << (b & 31);
            uint64_t q[4] = {0, 0, 0, 0};
            const uint64_t carry = a ? a - 1 : r - 1;            // strict predecessor of the bucket start, circular
            slot_put(q, 0, 40, keys[carry]);
            slot_put(q, 40, 40, prev_of(carry));
            if (cnt <= kPhiSlotEntries) {
                for (uint64_t e = 0; e < cnt; ++e) {
                    slot_put(q, 80 + 56 * (uint32_t) e, 16, keys[a + e] - (b << shift));
                    slot_put(q, 96 + 56 * (uint32_t) e, 40, prev_of(a + e));
                }
                slot_put(q, 248, 2, cnt);
            } else {
                if (cnt >> 32) { out.err = "phi overflow bucket too large"; return; }
                slot_put(q, 80, 40, out.ovf_prev.size());        // part-local for now
                slot_put(q, 250, 1, 1);
                if (bitmap) {
                    for (uint64_t e = a; e < z; ++e) slot_put(q, 120 + (uint32_t) (keys[e] - (b << shift)), 1, 1);
                } else {
                    slot_put(q, 120, 32, cnt);
                    slot_put(q, 251, 1, 1);
                    for (uint64_t e = a; e < z; ++e) out.ovf_keys.push_back(keys[e]);
                }
                for (uint64_t e = a; e < z; ++e) out.ovf_prev.push_back(prev_of(e));
                ++out.n_over;
            }
            for (int w = 0; w < 4; ++w) out.slots.push_back(q[w]);
            a = z;
        }
    };
    if (n_parts > 1) {
        std::vector<std::thread> th;
        for (unsigned t = 0; t < n_parts; ++t) th.emplace_back([&, t] { build_part(parts[t]); });
        for (auto& t : th) t.join();
    } else {
        build_part(parts[0]);
    }
    uint64_t n_slot_words = 4, n_ovf = 0;                        // + the sentinel
    for (unsigned t = 0; t < n_parts; ++t) {
        if (!parts[t].err.empty()) throw format_error(parts[t].err);
        if (t && !parts[t].slots.empty() && !parts[t - 1].slots.empty() && parts[t].first_bucket <= parts[t - 1].last_bucket)
            throw format_error("toehold SA: sampled positions not ascending");
        n_slot_words += parts[t].slots.size();
        n_ovf += parts[t].ovf_prev.size();
    }
    if ((n_slot_words / 4) >> 32) throw std::runtime_error("phi directory: more than 2^32 non-empty buckets");
    p.slots.resize(n_slot_words);
    p.ovf_prev.init(n, n_ovf);
    uint64_t at = 0;
    for (Part& part : parts) {
        const uint64_t ovf_base = p.ovf_prev.size();
        for (size_t k = 0; k < part.slots.size(); k += 4) {
            uint64_t q[4] = {part.slots[k], part.slots[k + 1], part.slots[k + 2], part.slots[k + 3]};
            if (slot_overflow(q) && ovf_base) {                  // rebase the index into the dense arrays (bits 80..119)
                const uint64_t idx = slot_get<80, 40>(q) + ovf_base;
                q[1] &= ~(((1ull << 40) - 1) << 16);
                q[1] |= (idx & ((1ull << 40) - 1)) << 16;
            }
            for (int w = 0; w < 4; ++w) p.slots[at + w] = q[w];
            at += 4;
        }
        for (uint64_t v : part.ovf_prev) p.ovf_prev.push(v);
        p.ovf_keys.insert(p.ovf_keys.end(), part.ovf_keys.begin(), part.ovf_keys.end());
        p.n_overflow += part.n_over;
        std::vector<uint64_t>().swap(part.slots);
        std::vector<uint64_t>().swap(part.ovf_prev);
    }
    {                                                            // the sentinel: carry = the last sample
        uint64_t q[4] = {0, 0, 0, 0};
        slot_put(q, 0, 40, keys[r - 1]);
        slot_put(q, 40, 40, prev_of(r - 1));
        for (int w = 0; w < 4; ++w) p.slots[at + w] = q[w];
    }
    uint64_t before = 0;                                         // l1 high halves: non-empty buckets before each group
    for (uint64_t g = 0; g < p.l1.size(); ++g) {
        const uint64_t bm = p.l1[g] & 0xFFFFFFFFull;
        p.l1[g] = bm | (before << 32);
        before += (uint64_t) __builtin_popcountll(bm);
    }
    p.n_slots = p.slots.size() / 4;
    return p;

}

uint64_t phi_dir_eval(const PhiDir& p, uint64_t n, uint64_t i) {
    const uint64_t b = i >> p.shift, base = b << p.shift;
    bool here;
    const uint64_t k = phi_slot_index(p.l1[b >> 5], (uint32_t) (b & 31), here);
    uint64_t q[4];
    for (int w = 0; w < 4; ++w) q[w] = p.slots[k * 4 + w];
    uint64_t key = slot_get<0, 40>(q), prev = slot_get<40, 40>(q);          // the carry answers an empty bucket
    if (here) {
        if (!slot_overflow(q)) {
            slot_pred(q, base, (uint32_t) (i - base), key, prev);
        } else if (!slot_search(q)) {
            uint64_t idx;
            if (slot_bitmap_pred(q, base, (uint32_t) (i - base), key, idx)) prev = p.ovf_prev.get(idx);
        } else {
            uint64_t lo = slot_ovf_start(q), hi = lo + slot_ovf_count(q);
            const uint64_t first = lo;
            while (lo < hi) {                                    // #entries with key < i
                const uint64_t mid = (lo + hi) >> 1;
                if (p.ovf_keys[mid] < i) lo = mid + 1; else hi = mid;
            }
            if (lo > first) { key = p.ovf_keys[lo - 1]; prev = p.ovf_prev.get(lo - 1); }
        }
    }
    return phi_value(key, prev, i, n);
}

}  // namespace rbg
