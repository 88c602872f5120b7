// See formats.hpp for the byte layouts and the reference lines they come from.
#include "formats.hpp"

#include <algorithm>
#include <thread>
#include <cstdio>
#include <cstring>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <exception>

namespace rbg {
namespace {

// Read-only view of a whole file (mmap), with a bounds-checked cursor.
class FileView {
  public:
    explicit FileView(const std::string& path) : path_(path) {
        fd_ = ::open(path.c_str(), O_RDONLY);
        if (fd_ < 0) throw io_error("bad file: " + path);
        struct stat st;
        if (fstat(fd_, &st) != 0) { ::close(fd_); throw io_error("bad file: " + path); }
        size_ = (size_t) st.st_size;
        if (size_) {
            void* p = mmap(nullptr, size_, PROT_READ, MAP_PRIVATE, fd_, 0);
            if (p == MAP_FAILED) { ::close(fd_); throw io_error("cannot map: " + path); }
            data_ = (const uint8_t*) p;
            madvise(p, size_, MADV_SEQUENTIAL);
        }
    }
    ~FileView() {
        if (!owner_) return;
        if (data_) munmap((void*) data_, size_);
        if (fd_ >= 0) ::close(fd_);
    }
    FileView(const FileView&) = delete;
    FileView& operator=(const FileView&) = delete;
    // A second cursor over the same mapping (does not own it): components of one file decoded on several threads.
    FileView(const FileView& whole, size_t pos) : path_(whole.path_), data_(whole.data_), size_(whole.size_), pos_(pos), owner_(false) {}
    size_t pos() const { return pos_; }

    const uint8_t* take(size_t nbytes) {
        if (nbytes > size_ - pos_) throw format_error("truncated file: " + path_);
        const uint8_t* p = data_ + pos_;
        pos_ += nbytes;
        return p;
    }
    uint64_t u64() { uint64_t v; memcpy(&v, take(8), 8); return v; }
    uint8_t u8() { return *take(1); }
    int32_t i32() { int32_t v; memcpy(&v, take(4), 4); return v; }
    bool done() const { return pos_ == size_; }
    const std::string& path() const { return path_; }

  private:
    std::string path_;
    int fd_ = -1;
    const uint8_t* data_ = nullptr;
    size_t size_ = 0, pos_ = 0;
    bool owner_ = true;
};

// An sdsl int_vector<>: width, bit length, and a pointer to its (unaligned) u64 words.
struct PackedInts {
    uint8_t width = 0;
    uint64_t bits = 0;
    const uint8_t* words = nullptr;
    uint64_t size() const { return width ? bits / width : 0; }
    uint64_t word(uint64_t i) const { uint64_t w; memcpy(&w, words + 8 * i, 8); return w; }
    uint64_t nwords() const { return (bits + 63) / 64; }
    // element i (LSB-first packing at bit i*width)
    uint64_t get(uint64_t i) const {
        uint64_t bit = i * width, wi = bit >> 6, sh = bit & 63;
        uint64_t v = word(wi) >> sh;
        if (sh + width > 64) v |= word(wi + 1) << (64 - sh);
        return width == 64 ? v : v & ((1ULL << width) - 1);
    }
};

PackedInts read_int_vector(FileView& f) {
    PackedInts v;
    uint64_t h = f.u64();
    v.width = (uint8_t) (h >> 56);
    v.bits = h & ((1ULL << 56) - 1);
    if (v.width > 64) throw format_error("int_vector: element width beyond 64 bits in " + f.path());
    v.words = f.take(8 * v.nwords());
    return v;
}

void skip_select_support(FileView& f) {
    uint64_t arg_cnt = f.u64();
    if (!arg_cnt) return;
    read_int_vector(f);                         // superblock
    read_int_vector(f);                         // mini_or_long
    uint64_t sb = (arg_cnt + 4095) >> 12;
    for (uint64_t i = 0; i < sb; ++i) read_int_vector(f);   // miniblock[i] or longsuperblock[i]
}

// sd_vector -> sorted positions of its ones.  i-th one = ((zeros before it in `high`) << wl) | low[i].
uint64_t read_sd_vector(FileView& f, std::vector<uint64_t>& ones) {
    uint64_t size = f.u64();
    uint8_t wl = f.u8();
    PackedInts low = read_int_vector(f);
    PackedInts high = read_int_vector(f);
    skip_select_support(f);
    skip_select_support(f);
    uint64_t m = low.size();
    ones.clear();
    if (m == 0) return size;
    if (low.width != wl) throw format_error("sd_vector: low width != wl in " + f.path());
    ones.reserve(m);
    uint64_t i = 0;
    for (uint64_t wi = 0, nw = high.nwords(); wi < nw && i < m; ++wi) {
        uint64_t w = high.word(wi);
        if (wi == nw - 1 && (high.bits & 63)) w &= (1ULL << (high.bits & 63)) - 1;
        while (w && i < m) {
            uint64_t p = wi * 64 + (uint64_t) __builtin_ctzll(w);
            ones.push_back(((p - i) << wl) | low.get(i));
            ++i;
            w &= w - 1;
        }
    }
    if (i != m) throw format_error("sd_vector: high/low mismatch in " + f.path());
    return size;
}

// Steps over a sparse_sd_vector without decoding it; returns its universe size u.
uint64_t skip_sparse_sd_vector(FileView& f) {
    const uint64_t u = f.u64();
    if (u == 0) return 0;
    f.u64();                        // size
    f.u8();                         // wl
    read_int_vector(f);             // low
    read_int_vector(f);             // high
    skip_select_support(f);
    skip_select_support(f);
    return u;
}

uint64_t read_sparse_sd_vector(FileView& f, std::vector<uint64_t>& ones) {
    uint64_t u = f.u64();
    ones.clear();
    if (u == 0) return 0;
    uint64_t size = read_sd_vector(f, ones);
    if (size != u) throw format_error("sparse_sd_vector: size mismatch in " + f.path());
    return u;
}

// Huffman-shaped wavelet tree: decode all symbols front to back with one cursor per node.
void read_wt_huff(FileView& f, std::vector<uint8_t>& out) {
    uint64_t size = f.u64();
    f.u64();   // sigma
    PackedInts bv = read_int_vector(f);
    read_int_vector(f);           // rank_support_v
    skip_select_support(f);
    skip_select_support(f);
    uint64_t n_nodes = f.u64();
    if (n_nodes > 1024) throw format_error("wt_huff: implausible node count in " + f.path());
    struct Node { uint64_t bv_pos, sym; uint16_t parent, child[2]; };
    std::vector<Node> nodes(n_nodes);
    for (auto& nd : nodes) {
        nd.bv_pos = f.u64();
        nd.sym = f.u64();
        memcpy(&nd.parent, f.take(2), 2);
        memcpy(nd.child, f.take(4), 4);
    }
    f.take(256 * 2);   // c_to_leaf
    f.take(256 * 8);   // path
    const uint16_t UNDEF = 0xFFFF;
    // every symbol below an inner root spends at least one bit of the tree's bit vector: a size field beyond that is corrupt
    // (and must not size an allocation)
    const bool root_is_leaf = n_nodes == 0 || nodes[0].child[0] == UNDEF;
    if (root_is_leaf ? size > (1ull << 40) : size > bv.bits) throw format_error("wt_huff: size field beyond the tree's bits in " + f.path());
    out.assign(size, 0);
    if (size == 0) return;
    if (n_nodes == 0) throw format_error("wt_huff: no nodes in " + f.path());
    std::vector<uint64_t> cur(n_nodes);
    for (size_t v = 0; v < n_nodes; ++v) cur[v] = nodes[v].bv_pos;
    for (uint64_t i = 0; i < size; ++i) {
        uint16_t v = 0;
        while (nodes[v].child[0] != UNDEF) {
            uint64_t p = cur[v]++;
            if (p >= bv.bits) throw format_error("wt_huff: bit cursor out of range in " + f.path());
            unsigned b = (bv.word(p >> 6) >> (p & 63)) & 1;
            v = nodes[v].child[b];
            if (v >= n_nodes) throw format_error("wt_huff: bad child in " + f.path());
        }
        out[i] = (uint8_t) nodes[v].sym;
    }
}

void unpack_all(const PackedInts& v, std::vector<uint64_t>& out) {
    uint64_t m = v.size();
    out.resize(m);
    for (uint64_t i = 0; i < m; ++i) out[i] = v.get(i);
}

}  // namespace

void validate_runs(const RunsBwt& b, const std::string& what) {
    if (b.heads.size() != b.R || b.lens.size() != b.R) throw format_error("run arrays do not hold R entries in " + what);
    uint64_t pos = 0;
    for (uint64_t j = 0; j < b.R; ++j) {
        if (b.lens[j] == 0 || b.lens[j] > b.n - pos) throw format_error("run length out of range in " + what);      // also a wrapped (negative) length
        pos += b.lens[j];
    }
    if (pos != b.n) throw format_error("run lengths do not sum to n in " + what);
}

void validate_toehold(const ToeholdArrays& t, const std::string& what) {
    if (t.pred.size() != t.r || t.samples_last.size() != t.r || t.pred_to_run.size() != t.r) throw format_error("toehold arrays do not hold r entries in " + what);
    for (uint64_t k = 0; k < t.r; ++k) {
        if (t.pred[k] >= t.n || (k && t.pred[k] <= t.pred[k - 1])) throw format_error("sampled positions not ascending below n in " + what);
        if (t.pred_to_run[k] > t.r) throw format_error("pred_to_run value beyond r in " + what);
        // a sample becomes a toehold and then a phi argument, which indexes the phi directory without a bound
        if (t.samples_last[k] >= t.n) throw format_error("run-end sample beyond n in " + what);
    }
}

void validate_markers(const MarkerArrays& m, const std::string& what) {
    auto ascending_below = [&](const std::vector<uint64_t>& v, uint64_t universe, const char* name) {
        for (size_t i = 0; i < v.size(); ++i)
            if (v[i] >= universe || (i && v[i] <= v[i - 1])) throw format_error(std::string("marker array: ") + name + " not ascending inside its universe in " + what);
    };
    ascending_below(m.starts, m.size_starts, "window starts");
    ascending_below(m.ends, m.size_ends, "window ends");
    ascending_below(m.idxs, m.size_idxs, "window indexes");
    if (!m.idxs.empty() && m.idxs.back() > m.arr.size()) throw format_error("marker array: window index beyond the marker words in " + what);
    // the select past the last window returns size_idxs: it ends the last window's gather
    if (m.size_idxs > m.arr.size()) throw format_error("marker array: index universe beyond the marker words in " + what);
}

RunsBwt read_rbwt(const std::string& path) {
    FileView f(path);
    RunsBwt b;
    b.n = f.u64();
    b.R = f.u64();
    uint64_t B = f.u64();
    (void) B;
    if (b.n == 0) return b;
    skip_sparse_sd_vector(f);                             // sampled run ends: redundant with the per-letter vectors
    // The per-letter vectors and the run heads are independent components: find where each starts (headers only),
    // then decode them on their own threads (41 M runs: 1.8 s -> 0.6 s on the BASELINE index).
    std::vector<std::vector<uint64_t>> per_letter(256);
    size_t start[256];
    uint64_t total = 0;
    std::vector<int> present;
    for (int c = 0; c < 256; ++c) {
        start[c] = f.pos();
        const uint64_t u = skip_sparse_sd_vector(f);
        total += u;
        if (u) present.push_back(c);
    }
    if (total != b.n) throw format_error("rbwt: per-letter lengths do not sum to n in " + path);
    std::vector<std::string> errors(present.size());
    std::vector<std::thread> th;
    for (size_t k = 0; k < present.size(); ++k)
        th.emplace_back([&, k] {
            try {
                FileView part(f, start[present[k]]);
                read_sparse_sd_vector(part, per_letter[present[k]]);
            } catch (const std::exception& e) {
                errors[k] = e.what();
            }
        });
    std::string head_error;
    try {
        read_wt_huff(f, b.heads);
    } catch (const std::exception& e) {
        head_error = e.what();
    }
    for (auto& t : th) t.join();
    for (const std::string& e : errors)
        if (!e.empty()) throw format_error(e);
    if (!head_error.empty()) throw format_error(head_error);
    if (b.heads.size() != b.R) throw format_error("rbwt: run_heads size != R in " + path);
    if (!f.done()) throw format_error("rbwt: trailing bytes in " + path);
    // run j with head c is the k-th c-run: its length is the gap between the (k-1)-th and k-th
    // one of runs_per_letter[c] (rle_string::run_at, include/rle_string.hpp:238-242)
    b.lens.resize(b.R);
    uint64_t cursor[256] = {0};
    uint64_t sum = 0;
    for (uint64_t j = 0; j < b.R; ++j) {
        uint8_t c = b.heads[j];
        uint64_t k = cursor[c]++;
        const auto& ones = per_letter[c];
        if (k >= ones.size()) throw format_error("rbwt: more runs than lengths for a letter in " + path);
        uint64_t len = k == 0 ? ones[0] + 1 : ones[k] - ones[k - 1];
        if (len == 0) throw format_error("rbwt: zero-length run in " + path);
        b.lens[j] = len;
        sum += len;
    }
    if (sum != b.n) throw format_error("rbwt: run lengths do not sum to n in " + path);
    validate_runs(b, path);                     // a wrapped length can still sum to n modulo 2^64
    return b;
}

// ---- wt_fbb ------------------------------------------------------------------------------------
namespace {

// std::vector<X> of PODs as sdsl::serialize writes it (sdsl/io.hpp:145-152,358-377): u64 count, raw elements.
struct PodVec {
    const uint8_t* p = nullptr;
    uint64_t n = 0;
};
PodVec read_pod_vec(FileView& f, size_t elem_bytes) {
    PodVec v;
    v.n = f.u64();
    if (v.n > (1ull << 48)) throw format_error("wt_fbb: implausible vector length in " + f.path());
    v.p = f.take(v.n * elem_bytes);
    return v;
}

// sdsl::hyb_vector<16> -> one byte per bit.  Blocks of 256 bits; the u16 header of block b sits at byte
// (b/16)*40 + 8 + 2*(b%16) of sblock_header: ones = h & 0x1ff, special = bit 9, encoded bytes = h >> 10
// (hyb_vector.hpp:256-265).  0 bytes: at most two runs (first run = `special`); 32: the plain 256 bits;
// min(ones, zeros): positions of the minority bit (= special); otherwise: end positions of all runs but the
// last two, first bit = special, and the popcount fixes where the last two meet (:267-357, access0 :372-510).
void decode_hyb_vector(FileView& f, std::vector<uint8_t>& bits) {
    const uint64_t size = f.u64();
    PackedInts trunk = read_int_vector(f), sbh = read_int_vector(f);
    read_int_vector(f);                                              // hblock headers: not needed sequentially
    if (size > (1ull << 40)) throw format_error("wt_fbb: implausible bitvector size in " + f.path());
    const uint64_t n_blocks = (size + 255) / 256, trunk_bytes = trunk.bits / 8;
    if (sbh.bits / 8 < ((n_blocks + 15) / 16) * 40) throw format_error("wt_fbb: short hyb_vector header in " + f.path());
    bits.assign(n_blocks * 256, 0);
    uint64_t tp = 0;
    for (uint64_t b = 0; b < n_blocks; ++b) {
        const uint8_t* hp = sbh.words + (b / 16) * 40 + 8 + (b % 16) * 2;
        const uint32_t h = (uint32_t) hp[0] | ((uint32_t) hp[1] << 8);
        const uint32_t ones = h & 0x1FFu, special = (h >> 9) & 1u, enc = h >> 10, zeros = 256 - ones;
        if (ones > 256 || tp + enc > trunk_bytes) throw format_error("wt_fbb: bad hyb_vector block in " + f.path());
        uint8_t* blk = bits.data() + b * 256;
        const uint8_t* t = trunk.words + tp;
        if (enc == 0) {
            const uint32_t first = special ? ones : zeros;
            memset(blk, (int) special, first);
            memset(blk + first, (int) (1 - special), 256 - first);
        } else if (enc >= 32) {
            for (uint32_t i = 0; i < 256; ++i) blk[i] = (t[i >> 3] >> (i & 7)) & 1;
        } else if (enc == (ones < zeros ? ones : zeros)) {
            memset(blk, (int) (1 - special), 256);
            for (uint32_t k = 0; k < enc; ++k) blk[t[k]] = (uint8_t) special;
        } else {
            uint32_t bit = special, pos = 0, cnt[2] = {0, 0};
            for (uint32_t k = 0; k < enc; ++k) {
                const uint32_t e = t[k];
                if (e < pos) throw format_error("wt_fbb: run ends out of order in " + f.path());
                memset(blk + pos, (int) bit, e + 1 - pos);
                cnt[bit] += e + 1 - pos;
                pos = e + 1;
                bit ^= 1u;
            }
            const uint32_t total = bit ? ones : zeros;
            if (total < cnt[bit] || pos + (total - cnt[bit]) > 256) throw format_error("wt_fbb: bad run encoding in " + f.path());
            const uint32_t first = total - cnt[bit];
            memset(blk + pos, (int) bit, first);
            memset(blk + pos + first, (int) (bit ^ 1u), 256 - pos - first);
        }
        tp += enc;
    }
    if (tp != trunk_bytes) throw format_error("wt_fbb: hyb_vector trunk not consumed in " + f.path());
    bits.resize(size);
}

struct RunSink {
    RunsBwt& b;
    uint64_t total = 0;
    void put(uint8_t c, uint64_t len) {
        if (!len) return;
        if (c == 1) throw format_error("wt_fbb: byte 1 in the text collides with the terminator code");
        if (c == 0) c = 1;                                           // rle_string's TERMINATOR (include/rle_string.hpp:59-62)
        if (!b.heads.empty() && b.heads.back() == c) b.lens.back() += len;
        else { b.heads.push_back(c); b.lens.push_back(len); }
        total += len;
    }
};

}  // namespace

RunsBwt read_rbwt_fbb(const std::string& path) {
    FileView whole(path);
    FileView& f = whole;
    RunsBwt out;
    out.n = f.u64();
    read_pod_vec(f, 8);                                              // m_count
    read_pod_vec(f, 8);                                              // m_hyperblock_rank
    read_pod_vec(f, 4);                                              // m_superblock_rank
    read_pod_vec(f, 1);                                              // m_global_mapping
    const uint64_t n_sb = f.u64();
    constexpr uint64_t kSuper = 1ull << 20;                          // t_sbs_log = 20 (wt_fbb.hpp:78)
    if (n_sb != (out.n + kSuper - 1) / kSuper) throw format_error("wt_fbb: superblock count does not match the size in " + path);
    // Superblocks are independent: find where each starts (headers only), then decode contiguous groups of them on
    // their own threads into run lists that are joined afterwards (a run may continue across a group boundary).
    std::vector<size_t> sb_at(n_sb + 1);
    for (uint64_t sb = 0; sb < n_sb; ++sb) {
        sb_at[sb] = f.pos();
        f.u8();
        f.u8();
        f.u64();                                                     // hyb_vector: size, trunk, sblock headers, hblock headers
        read_int_vector(f);
        read_int_vector(f);
        read_int_vector(f);
        read_pod_vec(f, 1);
        read_pod_vec(f, 14);
        read_pod_vec(f, 1);
    }
    sb_at[n_sb] = f.pos();
    auto decode_range = [&](uint64_t sb0, uint64_t sb1, RunsBwt& part) {
        FileView f(whole, sb_at[sb0]);
        RunSink sink{part};
        std::vector<uint8_t> bv;
        // per level of a block's tree: where each internal node's bits start, and how many were consumed
        std::vector<std::vector<uint64_t>> off, cur;
        std::vector<uint64_t> sizes, next_sizes, level_end;
        for (uint64_t sb = sb0; sb < sb1; ++sb) {
            f.u8();                                                      // superblock alphabet size - 1
            const uint32_t bs_log = f.u8();
            if (bs_log > 16) throw format_error("wt_fbb: bad block size in " + path);      // 2-byte level sizes limit blocks to 2^16 (:452-455)
            decode_hyb_vector(f, bv);
            PodVec var = read_pod_vec(f, 1);
            PodVec bh = read_pod_vec(f, 14);                             // {u32 bv_rank, u32 bv_offset, u32 var_offset, u8 sigma-1, u8 height} packed
            read_pod_vec(f, 1);                                          // superblock -> block alphabet mapping
            const uint64_t sb_beg = sb * kSuper, sb_len = std::min(kSuper, out.n - sb_beg);
            if (bh.n != (sb_len + (1ull << bs_log) - 1) >> bs_log) throw format_error("wt_fbb: block count mismatch in " + path);
            for (uint64_t blk = 0; blk < bh.n; ++blk) {
                uint32_t bv_off, var_off;
                memcpy(&bv_off, bh.p + 14 * blk + 4, 4);
                memcpy(&var_off, bh.p + 14 * blk + 8, 4);
                const uint32_t sigma = (uint32_t) bh.p[14 * blk + 12] + 1, height = bh.p[14 * blk + 13];
                const uint64_t beg = blk << bs_log, bsz = std::min<uint64_t>(1ull << bs_log, sb_len - beg);
                if (height == 0) {                                       // one distinct symbol: no bits (:1117-1120)
                    if ((uint64_t) var_off + 4 > var.n) throw format_error("wt_fbb: block header out of range in " + path);
                    sink.put(var.p[var_off], bsz);
                    continue;
                }
                if (height > 64 || (uint64_t) var_off + 3ull * (height - 1) + 4ull * sigma > var.n)
                    throw format_error("wt_fbb: block header out of range in " + path);
                // leaves per depth (depth 0 has none); the deepest level takes the rest (:443-455)
                uint32_t leaves_at[66] = {0}, leaf_base[67] = {0}, acc = 0;
                for (uint32_t d = 1; d < height; ++d) { leaves_at[d] = var.p[var_off + 3 * (d - 1)]; acc += leaves_at[d]; }
                if (acc > sigma) throw format_error("wt_fbb: leaf counts exceed sigma in " + path);
                leaves_at[height] = sigma - acc;
                for (uint32_t d = 0; d <= height; ++d) leaf_base[d + 1] = leaf_base[d] + leaves_at[d];
                const uint8_t* leaf = var.p + var_off + 3 * (height - 1);                     // u32 (symbol | rank << 8) per leaf, canonical order
                // Canonical codes, shortest first (:245-267): the nodes of depth d are the children of depth d-1's
                // internal nodes, leaves leftmost; node bit vectors are concatenated level by level, left to right.
                off.assign(height, {});
                cur.assign(height, {});
                level_end.assign(height, 0);
                sizes.assign(1, bsz);
                uint64_t p = bv_off;
                for (uint32_t d = 0; d < height; ++d) {
                    next_sizes.clear();
                    for (uint64_t sz : sizes) {
                        if (p + sz > bv.size()) throw format_error("wt_fbb: block bits out of range in " + path);
                        off[d].push_back(p);
                        cur[d].push_back(0);
                        uint64_t o = 0;
                        for (uint64_t i = 0; i < sz; ++i) o += bv[p + i];
                        next_sizes.push_back(sz - o);
                        next_sizes.push_back(o);
                        p += sz;
                    }
                    level_end[d] = p;
                    if (next_sizes.size() < leaves_at[d + 1]) throw format_error("wt_fbb: more leaves than nodes in " + path);
                    sizes.assign(next_sizes.begin() + leaves_at[d + 1], next_sizes.end());
                }
                if (!sizes.empty()) throw format_error("wt_fbb: internal nodes below the tree height in " + path);
                for (uint64_t i = 0; i < bsz; ++i) {
                    uint32_t d = 0;
                    uint64_t t = 0;
                    for (;;) {
                        // a consistent block consumes exactly the bits of each node; anything else is a malformed file
                        const uint64_t at = off[d][t] + cur[d][t]++;
                        if (at >= (t + 1 < off[d].size() ? off[d][t + 1] : level_end[d])) throw format_error("wt_fbb: node bits overrun in " + path);
                        const uint64_t idx = 2 * t + bv[at];
                        if (idx < leaves_at[d + 1]) {
                            sink.put(leaf[4 * (leaf_base[d + 1] + idx)], 1);
                            break;
                        }
                        t = idx - leaves_at[d + 1];
                        ++d;
                    }
                }
            }

        }
        part.n = sink.total;
    };
    unsigned n_thr = n_sb >= 16 ? std::min<unsigned>(8, std::max(1u, std::thread::hardware_concurrency())) : 1;
    if (const char* e = getenv("RBG_FBB_THREADS")) n_thr = (unsigned) std::max(1, std::min(64, atoi(e)));       // tests
    n_thr = (unsigned) std::min<uint64_t>(n_thr, std::max<uint64_t>(1, n_sb));
    std::vector<RunsBwt> parts(n_thr);
    std::vector<std::string> errors(n_thr);
    std::vector<std::thread> th;
    for (unsigned t = 0; t < n_thr; ++t)
        th.emplace_back([&, t] {
            try {
                decode_range(n_sb * t / n_thr, n_sb * (t + 1) / n_thr, parts[t]);
            } catch (const std::exception& e) {
                errors[t] = e.what();
            }
        });
    for (auto& t : th) t.join();
    for (const std::string& e : errors)
        if (!e.empty()) throw format_error(e);
    RunSink sink{out};
    for (RunsBwt& part : parts) {
        for (size_t j = 0; j < part.heads.size(); ++j) {
            // (parts already hold rle_string codes: the terminator is 1 here, which RunSink::put would refuse)
            if (!out.heads.empty() && out.heads.back() == part.heads[j]) out.lens.back() += part.lens[j];
            else { out.heads.push_back(part.heads[j]); out.lens.push_back(part.lens[j]); }
            sink.total += part.lens[j];
        }
        RunsBwt().heads.swap(part.heads);
    }
    if (!f.done()) throw format_error("wt_fbb: trailing bytes in " + path);
    if (sink.total != out.n) throw format_error("wt_fbb: decoded length != size in " + path);
    out.R = out.heads.size();
    validate_runs(out, path);
    return out;
}

ToeholdArrays read_tsa(const std::string& path) {
    FileView f(path);
    ToeholdArrays t;
    t.r = f.u64();
    t.n = f.u64();
    const size_t pred_at = f.pos();
    const uint64_t u = skip_sparse_sd_vector(f);
    PackedInts sl = read_int_vector(f);
    PackedInts pr = read_int_vector(f);
    if (!f.done()) throw format_error("tsa: trailing bytes in " + path);
    if (u != t.n || sl.size() != t.r || pr.size() != t.r) throw format_error("tsa: inconsistent sizes in " + path);
    // three independent components, three threads (the packed arrays only need unpacking)
    std::exception_ptr ea, eb;                                    // a bad_alloc on a worker must reach the C ABI as a code
    std::thread a([&] { try { unpack_all(sl, t.samples_last); } catch (...) { ea = std::current_exception(); } });
    std::thread b([&] { try { unpack_all(pr, t.pred_to_run); } catch (...) { eb = std::current_exception(); } });
    std::string pred_error;
    try {
        FileView part(f, pred_at);
        read_sparse_sd_vector(part, t.pred);
    } catch (const std::exception& e) {
        pred_error = e.what();
    }
    a.join();
    b.join();
    if (ea) std::rethrow_exception(ea);
    if (eb) std::rethrow_exception(eb);
    if (!pred_error.empty()) throw format_error(pred_error);
    if (t.pred.size() != t.r) throw format_error("tsa: inconsistent sizes in " + path);
    validate_toehold(t, path);
    return t;
}

MarkerArrays read_mab(const std::string& path) {
    FileView f(path);
    MarkerArrays m;
    m.size_starts = read_sd_vector(f, m.starts);
    m.size_ends = read_sd_vector(f, m.ends);
    m.size_idxs = read_sd_vector(f, m.idxs);
    uint64_t arr_size = f.u64();
    if (arr_size >> 60) throw format_error("mab: implausible number of marker words in " + path);       // 8 * arr_size must not wrap
    const uint8_t* p = f.take(8 * arr_size);
    m.arr.resize(arr_size);
    if (arr_size) memcpy(m.arr.data(), p, 8 * arr_size);
    m.wsize = f.i32();
    if (!f.done()) throw format_error("mab: trailing bytes in " + path);
    validate_markers(m, path);
    return m;
}

}  // namespace rbg
