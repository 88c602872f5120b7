// Host-side consistency check of the load-time re-layout (diagnostic; not on the query path):
// rebuilds the rank directory from <prefix>.rbwt and compares rank_c at p and p+1 (hence
// BWT[p]==c) decoded from the 64-byte lines -- the same leaf.cuh code the kernels run, cluster
// windows with their raw children and the terminator correction included -- with a direct
// count over the runs.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rowbowt_gpu.h"
#include "formats.hpp"
#include "host_pack.hpp"
#include "knobs.hpp"
#include "layout.hpp"
#include "leaf.cuh"
#include "sdsl_writer.hpp"

using namespace rbg;

namespace {
// Layout 7 (plain lines, leaf.cuh): F[c] + rank_c(pos) in both forms the kernel takes it -- from the line of pos counting the
// rows before it (lo) and from the line of pos - 1 counting up to and including that row (hi + 1) -- ~0 when they disagree.
uint64_t plain_dir_rank(const LeafDir& d, uint32_t c, uint64_t pos) {
    uint64_t out = ~0ull;
    for (int upto = 0; upto < 2; ++upto) {
        if (upto ? pos == 0 : pos == d.n) continue;
        const uint64_t at = upto ? pos - 1 : pos, line = at >> kPlainShift;
        const uint32_t q = (uint32_t) (at & (kPlainRows - 1));
        uint32_t w[kPlainWords];
        memcpy(w, d.lines.data() + line * kPlainWords, sizeof w);
        const uint64_t m = plain_match(w, c);
        uint64_t r = plain_count(w, c) + (upto ? plain_rank_upto(m, q) : plain_rank_before(m, q));
        if ((w[0] & kPlainTerm) && c == 0)
            for (uint32_t t = 0; t < d.n_term; ++t) r -= (d.term_pos[t] >= (line << kPlainShift) && d.term_pos[t] < pos) ? 1 : 0;
        if (out != ~0ull && out != r) return ~0ull;
        out = r;
    }
    return out;
}

// Layout 7: BWT[pos] == c as the toehold step reads it, bit q of the match word of c, not at a terminator row.
bool plain_dir_is(const LeafDir& d, uint32_t c, uint64_t pos) {
    uint32_t w[kPlainWords];
    memcpy(w, d.lines.data() + (pos >> kPlainShift) * kPlainWords, sizeof w);
    bool is = (plain_match(w, c) >> (pos & (kPlainRows - 1))) & 1ull;
    if ((w[0] & kPlainTerm) && c == 0)
        for (uint32_t t = 0; t < d.n_term; ++t) is = is && d.term_pos[t] != pos;
    return is;
}

// F[c] + rank_c(pos) through the directory, pos in [0, n]; mirrors lf_step / leaf_rank_slow
// (device_index.cuh): rank at pos is taken in the window of position `at` with offset q.
uint64_t dir_rank(const LeafDir& d, uint32_t c, uint64_t pos) {
    if (d.version == 7) return plain_dir_rank(d, c, pos);
    const bool use_prev = pos == d.n || (pos % d.window == 0 && pos > 0 && (pos & 1));   // also exercise the "hi" form (q = W)
    const uint64_t at = use_prev ? pos - 1 : pos;
    const uint64_t widx = (uint64_t) (((__uint128_t) at * d.magic) >> 64);
    if (widx != at / d.window) return ~0ull;
    const uint32_t q = (uint32_t) (at - widx * d.window) + (use_prev ? 1u : 0u);
    uint32_t w[16];
    memcpy(w, d.lines.data() + widx * 16, 64);
    const bool v5 = d.version == 5;
    uint32_t rel = v5 ? leaf_rel_count<5>(w, c) : leaf_rel_count<4>(w, c);
    uint32_t r = v5 ? leaf_rank<5>(w, leaf_cpat(c), q) : leaf_rank<4>(w, leaf_cpat(c), q);
    uint64_t from = pos - q;
    if (leaf_inside_cluster(w, q)) {
        const uint32_t s = leaf_cluster_begin(w);
        const uint32_t ch = (q - s) / kRawSymbols, p = (q - s) - ch * kRawSymbols;
        const uint32_t* cw = d.lines.data() + ((uint64_t) leaf_child_ptr(w) + ch) * 16;
        rel = (v5 ? rel : 0u) + raw_rel_count(cw, c);             // layout 5: child counts are relative to the window start
        r = raw_rank(cw, leaf_cpat(c), p);
        from += s + ch * kRawSymbols;
    }
    if ((w[15] & kFlagTerm) && c == 0)
        for (uint32_t t = 0; t < d.n_term; ++t) r -= (d.term_pos[t] >= from && d.term_pos[t] < pos) ? 1 : 0;
    return d.super[(uint64_t) c * d.n_super + (widx >> d.sb_shift)] + (uint64_t) rel + r;
}

// The walks below visit every run / sample of a full-size index (10^8 checks): they are cut into contiguous parts, one per
// host thread.  fn(part, begin, end) -> 0 or its failure code; the smallest failure code of any part is returned.
template <class Fn>
int parallel_parts(uint64_t n_items, unsigned n_parts, Fn&& fn) {
    n_parts = (unsigned) std::max<uint64_t>(1, std::min<uint64_t>(n_parts, n_items ? n_items : 1));
    std::vector<int> rc(n_parts, 0);
    std::vector<std::thread> th;
    for (unsigned p = 0; p < n_parts; ++p)
        th.emplace_back([&, p] {
            try { rc[p] = fn(p, n_items * p / n_parts, n_items * (p + 1) / n_parts); } catch (...) { rc[p] = -1; }
        });
    for (auto& t : th) t.join();
    int out = 0;
    for (int r : rc) if (r != 0 && (out == 0 || r < out)) out = r;
    return out;
}
unsigned selftest_threads() { return std::max(1u, std::min(32u, std::thread::hardware_concurrency())); }

// rank_c(p) and rank_c(p + 1) (hence BWT[p] == c) decoded from the directory at the first and last position of every run and
// every stride-th position inside, against a direct count over the runs.  window & 0xFFFF forces the window, window >> 16
// the layout (4, 5 or 7; 0 = the loader's own choice).
int check_layout(const RunsBwt& bwt, uint32_t window, uint64_t stride, uint64_t* checked, uint64_t* n_lines, uint64_t* n_cluster,
                 uint32_t* layout_out) {
    const uint32_t layout = window >> 16;
    LayoutKnobs k = layout_knobs();
    if (window & 0xFFFFu) k.window = window & 0xFFFFu;
    if (layout) k.layout = layout == 5 || layout == 7 ? (int32_t) layout : 4;
    LeafDir d = build_leaf_dir(bwt, k.window, k.leaf_layout());
    if (layout && d.version != (int) k.layout) return 3;
    if (n_lines) *n_lines = d.n_lines();
    if (n_cluster) *n_cluster = d.n_cluster;
    if (layout_out) *layout_out = (uint32_t) d.version;
    static const uint8_t sym[4] = {'A', 'C', 'G', 'T'};
    if (stride == 0) stride = 1;
    int8_t code_of_head[256];
    memset(code_of_head, -1, sizeof code_of_head);
    for (int c = 0; c < 4; ++c) code_of_head[sym[c]] = (int8_t) c;
    // where every part starts: position and per-symbol counts in front of its first run
    const unsigned n_parts = selftest_threads();
    struct Start { uint64_t pos, cum[4]; };
    std::vector<Start> start(n_parts + 1, Start{0, {0, 0, 0, 0}});
    {
        Start cur{0, {0, 0, 0, 0}};
        unsigned p = 0;
        for (uint64_t j = 0; j <= bwt.R; ++j) {
            while (p <= n_parts && j == bwt.R * p / n_parts) start[p++] = cur;
            if (j == bwt.R) break;
            const int hc = code_of_head[bwt.heads[j]];
            if (hc >= 0) cur.cum[hc] += bwt.lens[j];
            cur.pos += bwt.lens[j];
        }
    }
    std::atomic<uint64_t> total{0};
    const int rc = parallel_parts(bwt.R, n_parts, [&](unsigned part, uint64_t j0, uint64_t j1) {
        uint64_t cum[4], pos = start[part].pos, n_checked = 0;
        memcpy(cum, start[part].cum, sizeof cum);
        for (uint64_t j = j0; j < j1; ++j) {
            const int hc = code_of_head[bwt.heads[j]];
            // the first and last position of every run and every stride-th position inside
            for (uint64_t t = 0; t < bwt.lens[j]; t = (t + stride < bwt.lens[j] || t == bwt.lens[j] - 1) ? t + stride : bwt.lens[j] - 1) {
                const uint64_t p = pos + t;
                for (uint32_t c = 0; c < 4; ++c) {
                    if (!d.count[c]) continue;
                    const uint64_t want = d.Fcode[c] + cum[c] + ((int) c == hc ? t : 0);
                    if (dir_rank(d, c, p) != want) return 1;
                    if (dir_rank(d, c, p + 1) != want + ((int) c == hc ? 1 : 0)) return 2;
                    if (d.version == 7 && plain_dir_is(d, c, p) != ((int) c == hc)) return 4;
                    ++n_checked;
                }
            }
            if (hc >= 0) cum[hc] += bwt.lens[j];
            pos += bwt.lens[j];
        }
        total += n_checked;
        return 0;
    });
    if (rc) return rc;
    const uint64_t n_checked = total;
    if (checked) *checked = n_checked;
    return 0;
}
}  // namespace

extern "C" int rbg_selftest_layout(const char* prefix, uint32_t window, uint64_t stride, uint64_t* checked,
                                   uint64_t* n_lines, uint64_t* n_cluster) {
    try {
        return check_layout(read_rbwt(std::string(prefix) + ".rbwt"), window, stride, checked, n_lines, n_cluster, nullptr);
    } catch (const std::exception&) {
        return -1;
    }
}

// The same over caller-supplied runs; *layout receives the line format the directory was built in, which is what an open
// of these runs under the same environment would pick.
extern "C" int rbg_selftest_layout_runs(uint64_t n, const uint8_t* heads, const uint64_t* lens, uint64_t R, uint32_t window,
                                        uint64_t stride, uint64_t* checked, uint64_t* n_lines, uint32_t* layout) {
    try {
        RunsBwt bwt;
        bwt.n = n;
        bwt.R = R;
        bwt.heads.assign(heads, heads + R);
        bwt.lens.assign(lens, lens + R);
        return check_layout(bwt, window, stride, checked, n_lines, nullptr, layout);
    } catch (const std::exception&) {
        return -1;
    }
}

// Same for the phi slots: phi(i) decoded from the 32-byte slots (phi_slot.cuh, the code locate_kernel
// runs) against ToeholdSA::phi restated directly over the .tsa arrays (strict circular predecessor,
// include/toehold_sa.hpp:56-72), for every stride-th text position and both neighbours of every sample.
extern "C" int rbg_selftest_phi(const char* prefix, uint32_t shift, uint64_t stride, uint64_t* checked,
                                uint64_t* n_slots, uint64_t* n_overflow) {
    try {
        ToeholdArrays t = read_tsa(std::string(prefix) + ".tsa");
        LayoutKnobs k = layout_knobs();
        if (shift & 0xFFu) k.phi_shift = shift & 0xFFu;
        PhiDir p = build_phi_dir(t, k.phi_shift, k.phi_parts, (shift >> 8) ? (uint64_t) (shift >> 8) : ~0ull);     // bits 8.. = slot budget in bytes (0 = none)
        if (n_slots) *n_slots = p.n_slots;
        if (n_overflow) *n_overflow = p.n_overflow;
        auto direct = [&](uint64_t i) {
            uint64_t rk = std::lower_bound(t.pred.begin(), t.pred.end(), i) - t.pred.begin();      // #samples < i
            const uint64_t jr = rk == 0 ? t.r - 1 : rk - 1;
            const uint64_t j = t.pred[jr];
            const uint64_t delta = j < i ? i - j : i + 1;
            const uint64_t run = t.pred_to_run[jr];
            return ((run ? t.samples_last[run - 1] : 0) + delta) % t.n;
        };
        if (stride == 0) stride = 1;
        std::atomic<uint64_t> total{0};
        const uint64_t n_strided = (t.n + stride - 1) / stride;
        int rc = parallel_parts(n_strided, selftest_threads(), [&](unsigned, uint64_t a, uint64_t b) {
            for (uint64_t x = a; x < b; ++x)
                if (phi_dir_eval(p, t.n, x * stride) != direct(x * stride)) return 1;
            total += b - a;
            return 0;
        });
        if (rc) return rc;
        rc = parallel_parts(t.r, selftest_threads(), [&](unsigned, uint64_t a, uint64_t b) {
            uint64_t n_checked = 0;
            for (uint64_t k = a; k < b; ++k)
                for (uint64_t i : {t.pred[k], t.pred[k] + 1, t.pred[k] ? t.pred[k] - 1 : 0}) {
                    if (i >= t.n) continue;
                    if (phi_dir_eval(p, t.n, i) != direct(i)) return 2;
                    ++n_checked;
                }
            total += n_checked;
            return 0;
        });
        if (rc) return rc;
        if (checked) *checked = total;
        return 0;
    } catch (const std::exception&) {
        return -1;
    }
}

// The toehold directory (ToeholdDir, layout.hpp): for EVERY run j of the BWT, the row LF(end of run j) looked up
// through the bucket table and the reduced keys -- the host twin of toehold_at_row (device_index.cuh) -- must select
// samples_last[j] (include/rowbowt.hpp:562-566: after a non-trivial step the toehold is that run's sample), and rows
// that are no run-end image must not alias one.  shift = 0: the layout's own choice; else forces the bucket width
// (every key width: 1, 2, 4 bytes).
extern "C" int rbg_selftest_toehold(const char* prefix, uint32_t shift, uint64_t* checked, uint64_t* dir_bytes) {
    try {
        RunsBwt bwt = read_rbwt(std::string(prefix) + ".rbwt");
        ToeholdArrays t = read_tsa(std::string(prefix) + ".tsa");
        LayoutKnobs k = layout_knobs();
        if (shift) k.toehold_shift = shift;
        LeafDir d = build_leaf_dir(bwt, k.window, k.leaf_layout());
        ToeholdDir td = build_toehold_dir(bwt, d.F, t, k.toehold_shift);
        if (shift && td.shift != shift) return 3;
        if (dir_bytes) *dir_bytes = td.bytes();
        // per-symbol counts in front of every part's first run
        const unsigned n_parts = selftest_threads();
        std::vector<std::vector<uint64_t>> seen0(n_parts + 1, std::vector<uint64_t>(256, 0));
        {
            std::vector<uint64_t> cur(256, 0);
            unsigned p = 0;
            for (uint64_t j = 0; j <= bwt.R; ++j) {
                while (p <= n_parts && j == bwt.R * p / n_parts) seen0[p++] = cur;
                if (j == bwt.R) break;
                cur[bwt.heads[j]] += bwt.lens[j];
            }
        }
        std::atomic<uint64_t> total{0};
        const int rc = parallel_parts(bwt.R, n_parts, [&](unsigned part, uint64_t j0, uint64_t j1) {
            std::vector<uint64_t> seen = seen0[part];
            for (uint64_t j = j0; j < j1; ++j) {
                const uint8_t c = bwt.heads[j];
                seen[c] += bwt.lens[j];
                const uint64_t row = d.F[c] + seen[c] - 1;
                const uint64_t k = toehold_dir_rank(td, row);
                if (k >= td.n_keys || td.sample.get(k) != t.samples_last[j]) return 1;
                if (toehold_dir_rank(td, row + 1) != k + 1) return 2;          // #keys < row + 1: this key and no other
            }
            total += j1 - j0;
            return 0;
        });
        if (rc) return rc;
        if (td.toehold0 != (t.samples_last[t.r - 1] + 1) % t.n) return 4;
        if (checked) *checked = total;
        return 0;
    } catch (const std::exception&) {
        return -1;
    }
}

// rbg_pack_bytes without an index handle (CPU-only tests of the host packer): same call with an explicit
// byte -> code table (0..3, 4 = terminator, -1 = no symbol).
extern "C" int rbg_selftest_pack(const int8_t* code_of, const char* bases, const uint64_t* offsets, uint64_t n_reads,
                                 uint64_t x0, uint64_t x1, uint64_t* packed, uint8_t* flags, uint64_t* n_exotic) {
    const uint64_t ex = pack_bytes_host(code_of, (const uint8_t*) bases, offsets, n_reads, x0, x1, packed, flags);
    if (n_exotic) *n_exotic += ex;
    return 0;
}

// Writer check without a GPU: decode <prefix>.rbwt/.tsa/.mab with the readers (formats.cpp) and serialize the
// flat arrays again with sdsl_writer.hpp into <out_prefix>.*; the caller compares the files byte for byte.
// parts: bit 0 .rbwt, bit 1 .tsa, bit 2 .mab; bit 3: <prefix>.rbwt is a wt_fbb (`rb_build --fbb`) -- decoded and
// written as an rle_string .rbwt, which must equal what the reference's plain rb_build writes for the same BWT.
extern "C" int rbg_selftest_rewrite(const char* prefix, const char* out_prefix, uint32_t parts) {
    try {
        const std::string in(prefix), out(out_prefix);
        if (parts & 8) write_rbwt(read_rbwt_fbb(in + ".rbwt"), out + ".rbwt");
        else if (parts & 1) write_rbwt(read_rbwt(in + ".rbwt"), out + ".rbwt");
        if (parts & 2) write_tsa(read_tsa(in + ".tsa"), out + ".tsa");
        if (parts & 4) write_mab(read_mab(in + ".mab"), out + ".mab");
        return 0;
    } catch (const std::exception& e) {
        fprintf(stderr, "rbg_selftest_rewrite: %s\n", e.what());
        return -1;
    }
}

// Pair directory (PairDir, leaf.cuh LeafFmt<6>) over caller-supplied runs: K[p] + rank_p(pos) decoded from the lines -- the
// decode lf_pair_warp runs, CLUSTER children and the terminator correction included -- equals a direct count over the pair
// sequence at every stride-th position (and n) for all 16 codes.  codes_out (n bytes, optional) receives P[j] row by row
// (16 = a pair with the terminator), expanded from the runs the directory was built from.
extern "C" int rbg_selftest_pair(uint64_t n, const uint8_t* heads, const uint64_t* lens, uint64_t R, uint32_t window, uint64_t stride,
                                 uint8_t* codes_out, uint64_t* checked, uint64_t* n_lines, uint64_t* n_cluster) {
    try {
        RunsBwt bwt;
        bwt.n = n;
        bwt.R = R;
        bwt.heads.assign(heads, heads + R);
        bwt.lens.assign(lens, lens + R);
        LayoutKnobs k = layout_knobs();
        k.layout = 5;
        if (window) k.pair_window = window;
        LeafDir d = build_leaf_dir(bwt, k.window, k.layout);
        PairDir P = build_pair_dir(bwt, d, k.pair_window);
        if (n_lines) *n_lines = P.lines.size() / kLineWords;
        if (n_cluster) *n_cluster = P.n_cluster;
        std::vector<uint32_t> rl;
        std::vector<uint8_t> rc;
        pair_runs(bwt, d, rl, rc);
        std::vector<uint8_t> code(n);
        uint64_t at = 0;
        for (size_t i = 0; i < rl.size(); ++i) for (uint32_t t = 0; t < rl[i]; ++t) code[at++] = rc[i];
        if (at != n) return 2;
        if (codes_out) memcpy(codes_out, code.data(), n);
        const uint32_t W = P.window;
        uint64_t cnt[16] = {0}, chk = 0;
        if (stride == 0) stride = 1;
        for (uint64_t pos = 0; pos <= n; ++pos) {
            if (pos % stride == 0 || pos == n) {
                // rank at pos from the window of `a` with offset q; also the "hi" form (q = W) at every other boundary
                const bool prev = pos == n || (pos % W == 0 && pos > 0 && ((pos / W) & 1));
                const uint64_t a = prev ? pos - 1 : pos, widx = a / W;
                const uint32_t q = (uint32_t) (a - widx * W) + (prev ? 1u : 0u);
                uint32_t w[16];
                memcpy(w, P.lines.data() + widx * 16, 64);
                for (uint32_t p = 0; p < 16; ++p) {
                    uint32_t r = pair_rank(w, pair_pat(p), q);
                    if (w[15] & kFlagCluster) {
                        const uint32_t* cw = P.lines.data() + (uint64_t) pair_child_ptr(w) * 16;
                        r = 0;
                        for (uint32_t k = 0; 8 * k < q; ++k) r += pair_raw_word_count(cw[k], pair_pat(p), 8 * (int) k, (int) q);
                    }
                    if ((w[15] & kFlagTerm) && p == 0)
                        for (uint32_t t = 0; t < P.n_bad; ++t) r -= (P.bad_pos[t] >= pos - q && P.bad_pos[t] < pos) ? 1 : 0;
                    const uint64_t got = (uint64_t) P.super[p * P.n_super + (widx >> P.sb_shift)] + pair_rel_count(w, p) + r;
                    if (got != (uint64_t) P.super[p * P.n_super] + cnt[p]) return 1;
                    ++chk;
                }
            }
            if (pos < n && code[pos] < kPairBad) ++cnt[code[pos]];
        }
        if (checked) *checked = chk;
        return 0;
    } catch (...) {
        return -1;
    }
}
