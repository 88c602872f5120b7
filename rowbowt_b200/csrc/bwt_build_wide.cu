// BWT construction on the GPU with u64 positions and ranks: the files of bwt_build.cu for texts of 2^32 positions and more
// (and, with RBG_BWT_WIDE=1, for any text).
//
// The algorithm is bwt_build.cu's (prefix doubling over the suffixes still unsorted, the rank of a suffix being the first
// row of its group), with the suffix array cut into parts: contiguous ranges of rows, each sorted with buffers of one part.
//   bwt_prefix_hist_kernel      histogram of the first 11 symbols of every suffix (the leading digits of the 27-symbol key);
//                               the rows are cut greedily at bucket boundaries into parts of at most M rows, so no group
//                               of equal 27-symbol keys crosses a part
//   per part, rows [R0, R0 + m):
//     cub::DeviceSelect         the positions of the part's buckets (one pass over the text)
//     bwt_wide_init_keys_kernel key = first 27 symbols, value = item index (its position is pos[item])
//     radix sort, bwt_wide_heads_kernel + max-scan, bwt_wide_scatter_kernel: SA[R0 + row], rank[p] = R0 + head row
//     cub::DeviceSelect         the part's active local rows, kept in act[R0, R0 + m)
//   rounds h = 27, 54, 108, ...: the parts one after another; bwt_wide_round_keys_kernel keys an active row by
//     (rank[p] - R0) << shift | rank[p + h], shift = max(33, bits of n - 1), and sorts end_bit = shift + bits(m - 1).
//     Ranks change in place across parts within a round: rank[p + h] only has to be refined to h symbols, and a part
//     already done this round holds 2h-refined ranks, which are still consistent with the final order.  Within a part,
//     every key is built before any of its ranks change.
//   bwt_check_kernel            certificate (Burkhardt-Kaerkkaeinen) before anything is written: rank[SA[i]] == i and
//                               (T[SA[i]], rank[SA[i] + 1]) < (T[SA[i + 1]], rank[SA[i + 1] + 1]) for every row
//   bwt_gather_kernel<u64>, then run starts and bwt_samples_kernel<u64, u64> in chunks of at most M runs, in the part
//   buffers (r may be close to n).
//
// Device memory: 21 bytes per text position (text 1, SA 8, rank 8, active local rows 4), 32 per part row (two u64 key
// buffers, two u32 item buffers, u64 positions), 5^11 u64 prefix counts (391 MB) and CUB's scratch.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <cstdio>
#include <string>
#include <vector>

#include "bwt_build.cuh"
#include "bwt_build.hpp"
#include "cuda_host.hpp"

namespace rbg {

constexpr int kBwtPrefixK = 11;
constexpr uint64_t kBwtBuckets = 48828125ull;              // 5^11
constexpr uint32_t kWideSorted = 0xFFFFFFFFu;              // item whose group is a singleton (local rows stay below 2^31)
constexpr uint64_t kWideBytesPerPos = 21;
constexpr uint64_t kWideBytesPerPartRow = 32;
constexpr uint64_t kWideMaxPartRows = (1ull << 31) - 1;    // u32 items and local rows; CUB item counts are int
constexpr uint64_t kWidePiece = 1ull << 30;                // items of one cub::DeviceSelect call over text positions or rows
constexpr int kWideMinShift = 33;

// The first k symbols of the suffix at p in base 5 (terminator and past the end 0).
__device__ __forceinline__ uint64_t bwt_prefix(const uint8_t* __restrict__ text, uint64_t n, uint64_t p, int k) {
    uint64_t key = 0;
    for (int j = 0; j < k; ++j) key = key * 5 + (p + j < n ? bwt_code(text[p + j]) : 0);
    return key;
}

__global__ void __launch_bounds__(kBwtBlock) bwt_prefix_hist_kernel(const uint8_t* __restrict__ text, uint64_t n,
                                                                    unsigned long long* __restrict__ hist) {
    const uint64_t p = bwt_item();
    if (p >= n) return;
    atomicAdd(&hist[bwt_prefix(text, n, p, kBwtPrefixK)], 1ull);
}

__global__ void __launch_bounds__(kBwtBlock) bwt_wide_init_keys_kernel(const uint8_t* __restrict__ text, uint64_t n,
                                                                       const uint64_t* __restrict__ pos, uint64_t m,
                                                                       uint64_t* __restrict__ keys, uint32_t* __restrict__ items) {
    const uint64_t k = bwt_item();
    if (k >= m) return;
    keys[k] = bwt_prefix(text, n, pos[k], kBwtK);
    items[k] = (uint32_t) k;
}

__global__ void __launch_bounds__(kBwtBlock) bwt_wide_round_keys_kernel(const uint32_t* __restrict__ rows, const uint64_t* __restrict__ sa,
                                                                        const uint64_t* __restrict__ rank, uint64_t r0, uint64_t h,
                                                                        uint64_t n, uint64_t n_act, int shift, uint64_t* __restrict__ keys,
                                                                        uint32_t* __restrict__ items, uint64_t* __restrict__ pos) {
    const uint64_t k = bwt_item();
    if (k >= n_act) return;
    const uint64_t p = sa[r0 + rows[k]], q = p + h;
    keys[k] = (rank[p] - r0) << shift | (q < n ? rank[q] : 0ull);
    items[k] = (uint32_t) k;
    pos[k] = p;
}

// rows == nullptr: item k is local row k (the initial sort covers every row of the part); likewise in the scatter.
__global__ void __launch_bounds__(kBwtBlock) bwt_wide_heads_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ rows,
                                                                   uint64_t n_act, uint32_t* __restrict__ hd) {
    const uint64_t k = bwt_item();
    if (k >= n_act) return;
    hd[k] = bwt_is_head(keys, k) ? (rows ? rows[k] : (uint32_t) k) : 0u;
}

// hd[k] holds the item's new local group rank on entry; on exit its local row, or kWideSorted when its group is a singleton.
__global__ void __launch_bounds__(kBwtBlock) bwt_wide_scatter_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ items,
                                                                     const uint64_t* __restrict__ pos, const uint32_t* __restrict__ rows,
                                                                     uint64_t r0, uint64_t n_act, uint32_t* __restrict__ hd,
                                                                     uint64_t* __restrict__ sa, uint64_t* __restrict__ rank) {
    const uint64_t k = bwt_item();
    if (k >= n_act) return;
    const uint32_t row = rows ? rows[k] : (uint32_t) k;
    const uint64_t p = pos[items[k]];
    sa[r0 + row] = p;
    rank[p] = r0 + hd[k];
    const bool single = bwt_is_head(keys, k) && (k + 1 == n_act || keys[k + 1] != keys[k]);
    hd[k] = single ? kWideSorted : row;
}

// rank[v] = the first row i with sa[i] = v (rank starts all ones): the inverse of a caller's suffix array.
__global__ void __launch_bounds__(kBwtBlock) bwt_rank_of_kernel(const uint64_t* __restrict__ sa, uint64_t n,
                                                                unsigned long long* __restrict__ rank) {
    const uint64_t i = bwt_item();
    if (i >= n) return;
    const uint64_t p = sa[i];
    if (p < n) atomicMin(&rank[p], (unsigned long long) i);
}

// *first_bad = min(*first_bad, every row i where sa[i] >= n, rank[sa[i]] != i, or (T[sa[i]], rank[sa[i] + 1]) is not below
// (T[sa[i + 1]], rank[sa[i + 1] + 1]).  Only the terminator (T[n - 1]) has code 0, so equal codes other than 0 have both
// successors inside the text, and equal codes 0 are the same position twice.
__global__ void __launch_bounds__(kBwtBlock) bwt_check_kernel(const uint8_t* __restrict__ text, const uint64_t* __restrict__ sa,
                                                              const uint64_t* __restrict__ rank, uint64_t n,
                                                              unsigned long long* __restrict__ first_bad) {
    const uint64_t i = bwt_item();
    if (i >= n) return;
    const uint64_t p = sa[i];
    bool bad = p >= n || rank[p] != i;
    if (!bad && i + 1 < n) {
        const uint64_t q = sa[i + 1];
        if (q < n) {
            const uint64_t cp = bwt_code(text[p]), cq = bwt_code(text[q]);
            bad = cp > cq || (cp == cq && (cp == 0 || rank[p + 1] >= rank[q + 1]));
        }
    }
    if (bad) atomicMin(first_bad, (unsigned long long) i);
}

namespace {

struct MaxU32 {
    __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};
struct Unsorted {
    __device__ __forceinline__ bool operator()(uint32_t v) const { return v != kWideSorted; }
};
struct InBuckets {
    const uint8_t* text;
    uint64_t n, b0, b1;
    __device__ __forceinline__ bool operator()(uint64_t p) const {
        const uint64_t b = bwt_prefix(text, n, p, kBwtPrefixK);
        return b >= b0 && b < b1;
    }
};
struct RunStart64 {
    const uint8_t* bwt;
    __device__ __forceinline__ bool operator()(uint64_t i) const { return i == 0 || bwt[i] != bwt[i - 1]; }
};

unsigned grid(uint64_t items) { return (unsigned) ((items + kBwtBlock - 1) / kBwtBlock); }

int bits_of(uint64_t x) {
    int b = 0;
    while (b < 64 && (x >> b)) ++b;
    return b;
}

std::string prefix_name(uint64_t b) {
    std::string s(kBwtPrefixK, '?');
    for (int j = kBwtPrefixK - 1; j >= 0; --j, b /= 5) s[j] = "$ACGT"[b % 5];
    return s;
}

struct Part {
    uint64_t r0 = 0, rows = 0, b0 = 0, b1 = 0, active = 0;
};

// The device side of one build: buffers, stream, CUB scratch.
struct WideDev {
    cudaStream_t s = nullptr;
    DevBuf tmp, cnt;
    size_t tmp_bytes = 0;

    // Items i of [a, b) with pred(i), in order, to out; cub::DeviceSelect in pieces of kWidePiece.  Returns how many.
    template <class Pred>
    uint64_t select_range(Pred pred, uint64_t a, uint64_t b, uint64_t* out) {
        uint64_t got = 0;
        for (uint64_t c = a; c < b; c += kWidePiece) {
            const uint64_t m = std::min(kWidePiece, b - c);
            size_t tb = tmp_bytes;
            CU(cub::DeviceSelect::If(tmp.p, tb, thrust::counting_iterator<uint64_t>(c), out + got, cnt.as<uint64_t>(), (int64_t) m, pred, s));
            uint64_t k = 0;
            CU(cudaMemcpyAsync(&k, cnt.p, 8, cudaMemcpyDeviceToHost, s));
            CU(cudaStreamSynchronize(s));
            got += k;
        }
        return got;
    }
};

}  // namespace

void build_bwt_files_wide(const uint8_t* text, uint64_t len, int device, uint64_t part_rows, const std::string& out_prefix,
                          rbg_bwt_stats& st) {
    const uint64_t n = len + 1;
    check_bwt_length(n, "the text", kBwtWideMaxN);
    const double t_sort = wall_s();
    st.n = n;
    st.wide = 1;
    int shift = kWideMinShift;
    while (shift < 64 && ((n - 1) >> shift)) ++shift;           // bits of a rank, at least 33: the key layout of c5w
    uint64_t cap = std::min<uint64_t>(std::min(n, kWideMaxPartRows), 1ull << (64 - shift));
    if (part_rows) cap = std::min(cap, part_rows);

    // scratch of every CUB call, for the largest part and select piece, before anything is allocated
    WideDev dv;
    {
        size_t t[5] = {0, 0, 0, 0, 0};
        cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
        cub::DoubleBuffer<uint32_t> di(nullptr, nullptr);
        CU(cub::DeviceRadixSort::SortPairs(nullptr, t[0], dk, di, (uint32_t) cap, 0, 64));
        CU(cub::DeviceScan::InclusiveScan(nullptr, t[1], (uint32_t*) nullptr, (uint32_t*) nullptr, MaxU32(), (int64_t) cap));
        CU(cub::DeviceSelect::If(nullptr, t[2], (uint32_t*) nullptr, (uint32_t*) nullptr, (uint64_t*) nullptr, (int64_t) cap, Unsorted()));
        CU(cub::DeviceSelect::If(nullptr, t[3], thrust::counting_iterator<uint64_t>(0), (uint64_t*) nullptr, (uint64_t*) nullptr,
                                 (int64_t) kWidePiece, InBuckets{}));
        CU(cub::DeviceSelect::If(nullptr, t[4], thrust::counting_iterator<uint64_t>(0), (uint64_t*) nullptr, (uint64_t*) nullptr,
                                 (int64_t) kWidePiece, RunStart64{}));
        dv.tmp_bytes = *std::max_element(t, t + 5);
    }
    const uint64_t fixed = kWideBytesPerPos * n + 16 + kBwtBuckets * 8 + dv.tmp_bytes + 64;
    const uint64_t reserve = 256ull << 20;                       // allocation granularity and fragmentation
    const uint64_t min_rows = std::min<uint64_t>(cap, 1ull << 20);
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    if (fixed + kWideBytesPerPartRow * min_rows + reserve > free_b)
        throw nomem_error("the BWT of n = " + std::to_string(n) + " positions needs at least " +
                          std::to_string(fixed + kWideBytesPerPartRow * min_rows + reserve) + " bytes of device memory (" +
                          std::to_string(kWideBytesPerPos) + " per position + " + std::to_string(kWideBytesPerPartRow) + " per part row for " +
                          std::to_string(min_rows) + " rows + " + std::to_string(kBwtBuckets * 8 + dv.tmp_bytes + reserve) +
                          " of prefix histogram, sort scratch and headroom); " + std::to_string(free_b) + " are free on device " +
                          std::to_string(device));
    const uint64_t M = std::min(cap, (free_b - fixed - reserve) / kWideBytesPerPartRow);
    st.peak_bytes = fixed + kWideBytesPerPartRow * M;

    DevBuf d_text(n + 16), d_sa(8 * n), d_rank(8 * n), d_act(4 * n), d_hist(kBwtBuckets * 8), d_k[2] = {DevBuf(8 * M), DevBuf(8 * M)},
        d_i[2] = {DevBuf(4 * M), DevBuf(4 * M)}, d_pos(8 * M);
    dv.tmp = DevBuf(std::max<size_t>(dv.tmp_bytes, 16));
    dv.cnt = DevBuf(64);
    uint8_t* text_d = d_text.as<uint8_t>();
    uint64_t *sa = d_sa.as<uint64_t>(), *rank = d_rank.as<uint64_t>(), *pos = d_pos.as<uint64_t>();
    uint32_t* act = d_act.as<uint32_t>();
    CU(cudaStreamCreateWithFlags(&dv.s, cudaStreamNonBlocking));
    cudaStream_t s = dv.s;
    cudaEvent_t ev[2];
    for (auto& e : ev) CU(cudaEventCreate(&e));
    struct Cleanup {
        cudaStream_t s;
        cudaEvent_t* ev;
        ~Cleanup() { for (int i = 0; i < 2; ++i) cudaEventDestroy(ev[i]); cudaStreamDestroy(s); }
    } cleanup{s, ev};
    auto elapsed = [&]() {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, ev[0], ev[1]));
        return ms;
    };

    CU(cudaMemcpyAsync(text_d, text, len, cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(text_d + len, 0, 16, s));

    // the parts: buckets of equal 11-symbol prefixes, cut greedily into at most M rows
    CU(cudaEventRecord(ev[0], s));
    CU(cudaMemsetAsync(d_hist.p, 0, kBwtBuckets * 8, s));
    bwt_prefix_hist_kernel<<<grid(n), kBwtBlock, 0, s>>>(text_d, n, d_hist.as<unsigned long long>());
    CU(cudaGetLastError());
    std::vector<uint64_t> hist(kBwtBuckets);
    CU(cudaMemcpyAsync(hist.data(), d_hist.p, kBwtBuckets * 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    std::vector<Part> parts(1);
    for (uint64_t b = 0, row = 0; b < kBwtBuckets; ++b) {
        const uint64_t c = hist[b];
        if (!c) continue;
        if (c > M)
            throw nomem_error("the 11-symbol prefix " + prefix_name(b) + " starts " + std::to_string(c) + " suffixes, more than the " +
                              std::to_string(M) + " rows of one part on device " + std::to_string(device) +
                              " (a part must hold every suffix of its prefix)");
        if (parts.back().rows + c > M) {
            parts.back().b1 = b;
            parts.push_back(Part{row, 0, b, 0, 0});
        }
        parts.back().rows += c;
        row += c;
    }
    parts.back().b1 = kBwtBuckets;
    hist = std::vector<uint64_t>();
    st.parts = (uint32_t) parts.size();
    for (const Part& P : parts) st.part_rows = std::max(st.part_rows, P.rows);

    // the initial sort of every part by the first 27 symbols
    auto sort_part = [&](Part& P, const uint32_t* rows, uint64_t items, int end_bit) {
        cub::DoubleBuffer<uint64_t> dk(d_k[0].as<uint64_t>(), d_k[1].as<uint64_t>());
        cub::DoubleBuffer<uint32_t> di(d_i[0].as<uint32_t>(), d_i[1].as<uint32_t>());
        size_t tb = dv.tmp_bytes;
        CU(cub::DeviceRadixSort::SortPairs(dv.tmp.p, tb, dk, di, (uint32_t) items, 0, end_bit, s));
        uint32_t* hd = (uint32_t*) dk.Alternate();               // free after the sort: 8 bytes per item
        bwt_wide_heads_kernel<<<grid(items), kBwtBlock, 0, s>>>(dk.Current(), rows, items, hd);
        CU(cudaGetLastError());
        tb = dv.tmp_bytes;
        CU(cub::DeviceScan::InclusiveScan(dv.tmp.p, tb, hd, hd, MaxU32(), (int64_t) items, s));        // in place
        bwt_wide_scatter_kernel<<<grid(items), kBwtBlock, 0, s>>>(dk.Current(), di.Current(), pos, rows, P.r0, items, hd, sa, rank);
        CU(cudaGetLastError());
        tb = dv.tmp_bytes;
        CU(cub::DeviceSelect::If(dv.tmp.p, tb, hd, act + P.r0, dv.cnt.as<uint64_t>(), (int64_t) items, Unsorted(), s));
        CU(cudaMemcpyAsync(&P.active, dv.cnt.p, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    };
    uint64_t total = 0;
    for (Part& P : parts) {
        const uint64_t got = dv.select_range(InBuckets{text_d, n, P.b0, P.b1}, 0, n, pos);
        if (got != P.rows)
            throw internal_error("part at row " + std::to_string(P.r0) + " selected " + std::to_string(got) + " suffixes for " +
                                 std::to_string(P.rows) + " rows");
        bwt_wide_init_keys_kernel<<<grid(P.rows), kBwtBlock, 0, s>>>(text_d, n, pos, P.rows, d_k[0].as<uint64_t>(), d_i[0].as<uint32_t>());
        CU(cudaGetLastError());
        sort_part(P, nullptr, P.rows, 63);
        total += P.active;
    }

    // the rounds over the active rows, part by part
    for (uint64_t h = kBwtK; total; h *= 2) {
        if (st.rounds < RBG_BWT_MAX_ROUNDS) st.active[st.rounds] = total;
        st.max_active = std::max(st.max_active, total);
        ++st.rounds;
        total = 0;
        for (Part& P : parts) {
            if (!P.active) continue;
            const uint32_t* rows = act + P.r0;
            bwt_wide_round_keys_kernel<<<grid(P.active), kBwtBlock, 0, s>>>(rows, sa, rank, P.r0, h, n, P.active, shift,
                                                                          d_k[0].as<uint64_t>(), d_i[0].as<uint32_t>(), pos);
            CU(cudaGetLastError());
            sort_part(P, rows, P.active, shift + bits_of(P.rows - 1));
            total += P.active;
        }
    }
    CU(cudaEventRecord(ev[1], s));
    CU(cudaStreamSynchronize(s));
    st.ms_sort = elapsed();

    // the certificate: rank is the inverse of SA now
    CU(cudaEventRecord(ev[0], s));
    unsigned long long bad = n;
    CU(cudaMemcpyAsync(dv.cnt.p, &bad, 8, cudaMemcpyHostToDevice, s));
    bwt_check_kernel<<<grid(n), kBwtBlock, 0, s>>>(text_d, sa, rank, n, dv.cnt.as<unsigned long long>());
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(&bad, dv.cnt.p, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(ev[1], s));
    CU(cudaStreamSynchronize(s));
    st.ms_verify = elapsed();
    if (bad != n)
        throw internal_error("the suffix array of n = " + std::to_string(n) + " positions failed its check at row " + std::to_string(bad) +
                             "; nothing was written");

    // BWT into the rank buffer; run starts and samples in chunks that start at a run start and hold at most M runs
    CU(cudaEventRecord(ev[0], s));
    uint8_t* bwt = d_rank.as<uint8_t>();
    bwt_gather_kernel<uint64_t><<<grid(n), kBwtBlock, 0, s>>>(text_d, sa, n, bwt);
    CU(cudaGetLastError());
    std::vector<uint8_t> h_bwt(n);
    CU(cudaMemcpyAsync(h_bwt.data(), bwt, n, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    uint64_t *starts = d_k[0].as<uint64_t>(), *sa_first = d_k[1].as<uint64_t>(), *sa_last = pos;
    std::vector<uint64_t> ssa, esa, h_starts, h_first, h_last;
    for (uint64_t c0 = 0; c0 < n;) {
        uint64_t c1 = std::min(n, c0 + M);
        while (c1 < n && h_bwt[c1] == h_bwt[c1 - 1]) ++c1;     // no run starts in (c0 + M, c1)
        const uint64_t rc = dv.select_range(RunStart64{bwt}, c0, c1, starts);
        bwt_samples_kernel<uint64_t, uint64_t><<<grid(rc), kBwtBlock, 0, s>>>(starts, rc, c1, sa, sa_first, sa_last);
        CU(cudaGetLastError());
        if (h_starts.size() < rc) {
            h_starts.resize(rc);
            h_first.resize(rc);
            h_last.resize(rc);
        }
        CU(cudaMemcpyAsync(h_starts.data(), starts, rc * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(h_first.data(), sa_first, rc * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(h_last.data(), sa_last, rc * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        for (uint64_t j = 0; j < rc; ++j) {
            ssa.push_back(h_starts[j]);
            ssa.push_back(h_first[j]);
            esa.push_back((j + 1 < rc ? h_starts[j + 1] : c1) - 1);
            esa.push_back(h_last[j]);
        }
        c0 = c1;
    }
    CU(cudaEventRecord(ev[1], s));
    CU(cudaStreamSynchronize(s));
    st.ms_gather = elapsed();
    st.r = ssa.size() / 2;
    st.s_sort = wall_s() - t_sort;

    const double t_write = wall_s();
    write_file(out_prefix + ".bwt", h_bwt.data(), n);
    write_file(out_prefix + ".ssa", ssa.data(), ssa.size() * 8);
    write_file(out_prefix + ".esa", esa.data(), esa.size() * 8);
    st.s_write = wall_s() - t_write;
}

uint64_t check_suffix_array(const uint8_t* text, uint64_t len, const uint64_t* sa, int device) {
    (void) device;                                               // selected by the caller
    const uint64_t n = len + 1;
    DevBuf d_text(n + 16), d_sa(8 * n), d_rank(8 * n), d_bad(64);
    cudaStream_t s;
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    struct Cleanup {
        cudaStream_t s;
        ~Cleanup() { cudaStreamDestroy(s); }
    } cleanup{s};
    unsigned long long bad = n;
    CU(cudaMemcpyAsync(d_text.p, text, len, cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(d_text.as<uint8_t>() + len, 0, 16, s));
    CU(cudaMemcpyAsync(d_sa.p, sa, 8 * n, cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(d_rank.p, 0xFF, 8 * n, s));
    CU(cudaMemcpyAsync(d_bad.p, &bad, 8, cudaMemcpyHostToDevice, s));
    bwt_rank_of_kernel<<<grid(n), kBwtBlock, 0, s>>>(d_sa.as<uint64_t>(), n, d_rank.as<unsigned long long>());
    CU(cudaGetLastError());
    bwt_check_kernel<<<grid(n), kBwtBlock, 0, s>>>(d_text.as<uint8_t>(), d_sa.as<uint64_t>(), d_rank.as<uint64_t>(), n,
                                                   d_bad.as<unsigned long long>());
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(&bad, d_bad.p, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return bad;
}

}  // namespace rbg
