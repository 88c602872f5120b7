// BWT construction on the GPU for texts below 2^32 positions: the raw files pfbwt-f64 --non-acgt-to-a --print-docs -r writes
// (.bwt, .ssa, .esa, .docs), from a FASTA.
//
// Suffix sorting by prefix doubling over the suffixes that are still unsorted (Manber-Myers with Larsson-Sadakane's active
// set), u32 positions and ranks.  The rank of a suffix is the first row of its group: the suffixes sharing its first h symbols.
//   bwt_init_keys_kernel   key = the first 27 symbols in base 5 (terminator 0, A..T 1..4: 63 bits), value = the position
//   (radix sort of the pairs)
//   bwt_heads_kernel       per sorted item: its row where its key differs from the one before, else 0; a max-scan turns that
//                          into the group rank of every item
//   bwt_scatter_kernel     SA[row] = position, rank[position] = group rank; the rows of groups larger than one stay active
//                          (cub::DeviceSelect)
//   bwt_round_keys_kernel  round h = 27, 54, 108, ...: over the active rows only, key = (rank[p], rank[p + h]), then the same
//                          sort / heads / scatter.  Every key of a round is built before any rank of that round changes.
// A suffix whose group is larger than one is longer than h (the terminator is unique), so p + h < n for every active p.
// Then bwt_gather_kernel (BWT[i] = T[SA[i] - 1]), cub::DeviceSelect of the rows that start a run, and bwt_samples_kernel
// (SA at the first and last row of every run).  The BWT and the r samples come back to the host; the suffix array does not.
//
// Device memory: 37 bytes per text position (text 1, SA 4, rank 4, three u32 item buffers 12, two u64 key buffers 16) plus
// CUB's scratch; the BWT stage reuses the rank and key buffers.
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <unistd.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "bwt_build.cuh"
#include "bwt_build.hpp"
#include "cuda_host.hpp"
#include "formats.hpp"
#include "host_io.hpp"
#include "layout.hpp"

namespace rbg {

// Kernels outside the anonymous namespace: their names stay the same from build to build (traces, profiles).
constexpr uint32_t kBwtSorted = 0xFFFFFFFFu;      // item whose group is a singleton (no row reaches 2^32 - 1)
constexpr uint64_t kBwtBytesPerPos = 37;

__global__ void __launch_bounds__(kBwtBlock) bwt_init_keys_kernel(const uint8_t* __restrict__ text, uint64_t n, uint64_t* __restrict__ keys,
                                                                  uint32_t* __restrict__ pos) {
    const uint64_t i = bwt_item();
    if (i >= n) return;
    uint64_t key = 0;
#pragma unroll
    for (int j = 0; j < kBwtK; ++j) key = key * 5 + (i + j < n ? bwt_code(text[i + j]) : 0);
    keys[i] = key;
    pos[i] = (uint32_t) i;
}

__global__ void __launch_bounds__(kBwtBlock) bwt_round_keys_kernel(const uint32_t* __restrict__ rows, const uint32_t* __restrict__ sa,
                                                                   const uint32_t* __restrict__ rank, uint64_t h, uint64_t n,
                                                                   uint64_t n_act, int shift, uint64_t* __restrict__ keys,
                                                                   uint32_t* __restrict__ pos) {
    const uint64_t k = bwt_item();
    if (k >= n_act) return;
    const uint32_t p = sa[rows[k]];
    const uint64_t q = p + h;
    keys[k] = (uint64_t) rank[p] << shift | (q < n ? rank[q] : 0u);
    pos[k] = p;
}

// rows == nullptr: item k is row k (the pass after the initial sort covers every row); likewise in bwt_scatter_kernel.
__global__ void __launch_bounds__(kBwtBlock) bwt_heads_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ rows,
                                                              uint64_t n_act, uint32_t* __restrict__ hd) {
    const uint64_t k = bwt_item();
    if (k >= n_act) return;
    hd[k] = bwt_is_head(keys, k) ? (rows ? rows[k] : (uint32_t) k) : 0u;
}

// hd[k] holds the item's new group rank on entry; on exit its row, or kBwtSorted when its group is a singleton.
__global__ void __launch_bounds__(kBwtBlock) bwt_scatter_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ pos,
                                                                const uint32_t* __restrict__ rows, uint64_t n_act, uint32_t* __restrict__ hd,
                                                                uint32_t* __restrict__ sa, uint32_t* __restrict__ rank) {
    const uint64_t k = bwt_item();
    if (k >= n_act) return;
    const uint32_t row = rows ? rows[k] : (uint32_t) k, p = pos[k];
    sa[row] = p;
    rank[p] = hd[k];
    const bool single = bwt_is_head(keys, k) && (k + 1 == n_act || keys[k + 1] != keys[k]);
    hd[k] = single ? kBwtSorted : row;
}

namespace {

struct MaxU32 {
    __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};
struct Unsorted {
    __device__ __forceinline__ bool operator()(uint32_t v) const { return v != kBwtSorted; }
};
struct RunStart {
    const uint8_t* bwt;
    __device__ __forceinline__ bool operator()(uint32_t i) const { return i == 0 || bwt[i] != bwt[i - 1]; }
};

unsigned grid(uint64_t items) { return (unsigned) ((items + kBwtBlock - 1) / kBwtBlock); }

std::string printable(uint8_t c) {
    char buf[16];
    if (c >= 0x20 && c < 0x7f) snprintf(buf, sizeof buf, "'%c'", c);
    else snprintf(buf, sizeof buf, "0x%02x", c);
    return buf;
}

}  // namespace

void write_file(const std::string& path, const void* data, size_t bytes) {
    const std::string tmp = path + ".tmp." + std::to_string((long) getpid());
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) throw io_error("cannot write " + tmp);
    bool ok = bytes == 0 || fwrite(data, 1, bytes, f) == bytes;
    ok = fclose(f) == 0 && ok;
    if (ok) ok = rename(tmp.c_str(), path.c_str()) == 0;
    if (!ok) {
        remove(tmp.c_str());
        throw io_error("cannot write " + path);
    }
}

void check_bwt_length(uint64_t n, const std::string& what, uint64_t max_n) {
    if (n > max_n) {
        int bits = 0;
        while (bits < 64 && (max_n >> bits)) ++bits;
        throw std::invalid_argument(what + " would have n >= 2^" + std::to_string(bits) + " positions (terminator included); this "
                                    "BWT builder takes n <= " + std::to_string(max_n));
    }
}

void check_acgt(const uint8_t* text, uint64_t len) {
    for (uint64_t i = 0; i < len; ++i) {
        const uint8_t c = text[i];
        if (c != 'A' && c != 'C' && c != 'G' && c != 'T')
            throw alphabet_error("byte " + printable(c) + " at offset " + std::to_string(i) + " of the text is not one of A, C, G, T");
    }
}

FastaText read_fasta_text(const std::string& path, uint64_t max_n) {
    struct stat sb;
    if (stat(path.c_str(), &sb) != 0) throw io_error("bad file: " + path);
    rbhost::FastxReader rd(path.c_str());
    if (!rd.ok()) throw io_error("bad file: " + path);
    // ACGT kept, other uppercase letters -> 'A' (--non-acgt-to-a), everything else 0 = refused
    uint8_t map[256] = {};
    for (int c = 'A'; c <= 'Z'; ++c) map[c] = 'A';
    map['C'] = 'C';
    map['G'] = 'G';
    map['T'] = 'T';
    FastaText ft;
    if (S_ISREG(sb.st_mode)) ft.text.reserve(std::min<uint64_t>((uint64_t) sb.st_size + 1024, max_n));
    std::string name, seq;
    for (;;) {
        seq.clear();
        const int rc = rd.next(name, seq);
        if (rc == -1 && seq.empty()) break;
        if (rc == -2) throw format_error("truncated FASTQ record after '" + name + "' in " + path + " (a FASTA is expected)");
        if (rc == -3) throw io_error("cannot read " + path);
        if (seq.empty()) throw format_error("record '" + name + "' of " + path + " has no bases");
        const uint64_t start = ft.text.size();
        check_bwt_length(start + seq.size() + kBwtPad + 1, "the text of " + path, max_n);
        ft.text.resize(start + seq.size() + kBwtPad, 'A');
        uint8_t* out = ft.text.data() + start;
        uint8_t bad = 0xff;
        for (size_t i = 0; i < seq.size(); ++i) {
            out[i] = map[(uint8_t) seq[i]];
            bad &= out[i];
        }
        if (!bad) {
            size_t i = 0;
            while (map[(uint8_t) seq[i]]) ++i;
            throw alphabet_error("record '" + name + "' of " + path + ": byte " + printable((uint8_t) seq[i]) + " at offset " +
                                 std::to_string(i) + " is not an uppercase letter.  Lowercase (soft-masked) bases are not "
                                 "accepted: uppercase the sequence lines first");
        }
        ft.names.push_back(name);
        ft.starts.push_back(start);
    }
    if (ft.names.empty()) throw format_error("no FASTA records in " + path);
    return ft;
}

void write_docs(const FastaText& ft, const std::string& path) {
    std::string s;
    for (size_t i = 0; i < ft.names.size(); ++i) s += ft.names[i] + " " + std::to_string(ft.starts[i]) + "\n";
    write_file(path, s.data(), s.size());
}

void build_bwt_files(const uint8_t* text, uint64_t len, int device, const std::string& out_prefix, rbg_bwt_stats& st) {
    const uint64_t n = len + 1;
    check_bwt_length(n, "the text", kBwtMaxN);
    const double t_sort = wall_s();
    st.n = n;
    st.parts = 1;
    st.part_rows = n;

    // scratch of every CUB call, for the largest item count, before anything is allocated
    size_t tmp_sort = 0, tmp_scan = 0, tmp_sel = 0, tmp_runs = 0;
    {
        cub::DoubleBuffer<uint64_t> dk(nullptr, nullptr);
        cub::DoubleBuffer<uint32_t> dv(nullptr, nullptr);
        CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, dk, dv, (uint32_t) n, 0, 64));
        CU(cub::DeviceScan::InclusiveScan(nullptr, tmp_scan, (uint32_t*) nullptr, (uint32_t*) nullptr, MaxU32(), (int64_t) n));
        CU(cub::DeviceSelect::If(nullptr, tmp_sel, (uint32_t*) nullptr, (uint32_t*) nullptr, (uint64_t*) nullptr, (int64_t) n, Unsorted()));
        CU(cub::DeviceSelect::If(nullptr, tmp_runs, thrust::counting_iterator<uint32_t>(0), (uint32_t*) nullptr, (uint64_t*) nullptr,
                                 (int64_t) n, RunStart{nullptr}));
    }
    const size_t tmp_bytes = std::max(std::max(tmp_sort, tmp_scan), std::max(tmp_sel, tmp_runs));
    const uint64_t need = kBwtBytesPerPos * n + 16 + tmp_bytes + 64;
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    if (need > free_b)
        throw nomem_error("the BWT of n = " + std::to_string(n) + " positions needs " + std::to_string(need) + " bytes of device memory (" +
                          std::to_string(kBwtBytesPerPos) + " per position + " + std::to_string(tmp_bytes) + " of sort scratch); " +
                          std::to_string(free_b) + " are free on device " + std::to_string(device));
    st.peak_bytes = need;

    DevBuf d_text(n + 16), d_sa(4 * n), d_rank(4 * n), d_u[3] = {DevBuf(4 * n), DevBuf(4 * n), DevBuf(4 * n)},
                                                        d_k[2] = {DevBuf(8 * n), DevBuf(8 * n)}, d_tmp(std::max<size_t>(tmp_bytes, 16)), d_cnt(64);
    uint8_t* text_d = d_text.as<uint8_t>();
    uint32_t *sa = d_sa.as<uint32_t>(), *rank = d_rank.as<uint32_t>();
    uint64_t* cnt = d_cnt.as<uint64_t>();
    cudaStream_t s;
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
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

    // the initial sort by the first 27 symbols, then the rounds over the active rows
    int shift = 1;
    while ((n - 1) >> shift) ++shift;                         // bits of a rank
    uint32_t *rows = nullptr, *spare = d_u[2].as<uint32_t>();
    uint32_t* pos_buf[2] = {d_u[0].as<uint32_t>(), d_u[1].as<uint32_t>()};
    uint64_t n_act = n, h = kBwtK;
    for (int round = 0;; ++round) {
        CU(cudaEventRecord(ev[0], s));
        cub::DoubleBuffer<uint64_t> dk(d_k[0].as<uint64_t>(), d_k[1].as<uint64_t>());
        cub::DoubleBuffer<uint32_t> dv(pos_buf[0], pos_buf[1]);
        int end_bit = 63;
        if (round == 0) {
            bwt_init_keys_kernel<<<grid(n), kBwtBlock, 0, s>>>(text_d, n, dk.Current(), dv.Current());
        } else {
            bwt_round_keys_kernel<<<grid(n_act), kBwtBlock, 0, s>>>(rows, sa, rank, h, n, n_act, shift, dk.Current(), dv.Current());
            end_bit = 2 * shift;
        }
        CU(cudaGetLastError());
        size_t tb = tmp_bytes;
        CU(cub::DeviceRadixSort::SortPairs(d_tmp.p, tb, dk, dv, (uint32_t) n_act, 0, end_bit, s));
        uint32_t* hd = (uint32_t*) dk.Alternate();             // free after the sort: 8 bytes per item
        bwt_heads_kernel<<<grid(n_act), kBwtBlock, 0, s>>>(dk.Current(), rows, n_act, hd);
        CU(cudaGetLastError());
        tb = tmp_bytes;
        CU(cub::DeviceScan::InclusiveScan(d_tmp.p, tb, hd, hd, MaxU32(), (int64_t) n_act, s));          // in place
        bwt_scatter_kernel<<<grid(n_act), kBwtBlock, 0, s>>>(dk.Current(), dv.Current(), rows, n_act, hd, sa, rank);
        CU(cudaGetLastError());
        uint32_t* next_rows = dv.Alternate();                  // free after the sort
        tb = tmp_bytes;
        CU(cub::DeviceSelect::If(d_tmp.p, tb, hd, next_rows, cnt, (int64_t) n_act, Unsorted(), s));
        CU(cudaEventRecord(ev[1], s));
        uint64_t left = 0;
        CU(cudaMemcpyAsync(&left, cnt, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        st.ms_sort += elapsed();
        // the buffers of the next round: the old rows (or the spare) and the sorted positions hold positions next
        uint32_t* freed = rows ? rows : spare;
        pos_buf[0] = freed;
        pos_buf[1] = dv.Current();
        rows = next_rows;
        n_act = left;
        if (!n_act) break;
        if (round > 0) h *= 2;
        if (st.rounds < RBG_BWT_MAX_ROUNDS) st.active[st.rounds] = n_act;
        st.max_active = std::max(st.max_active, n_act);
        ++st.rounds;
    }

    // BWT, run starts, SA at both ends of every run; the rank and key buffers are free now
    CU(cudaEventRecord(ev[0], s));
    uint8_t* bwt = d_rank.as<uint8_t>();
    uint32_t* starts = d_k[0].as<uint32_t>();
    uint32_t *sa_first = d_k[1].as<uint32_t>(), *sa_last = sa_first + n;
    bwt_gather_kernel<uint32_t><<<grid(n), kBwtBlock, 0, s>>>(text_d, sa, n, bwt);
    CU(cudaGetLastError());
    size_t tb = tmp_bytes;
    CU(cub::DeviceSelect::If(d_tmp.p, tb, thrust::counting_iterator<uint32_t>(0), starts, cnt, (int64_t) n, RunStart{bwt}, s));
    uint64_t r = 0;
    CU(cudaMemcpyAsync(&r, cnt, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    bwt_samples_kernel<uint32_t, uint32_t><<<grid(r), kBwtBlock, 0, s>>>(starts, r, n, sa, sa_first, sa_last);
    CU(cudaGetLastError());
    CU(cudaEventRecord(ev[1], s));
    std::vector<uint8_t> h_bwt(n);
    std::vector<uint32_t> h_starts(r), h_first(r), h_last(r);
    CU(cudaMemcpyAsync(h_bwt.data(), bwt, n, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(h_starts.data(), starts, r * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(h_first.data(), sa_first, r * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(h_last.data(), sa_last, r * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    st.ms_gather = elapsed();
    st.r = r;
    st.s_sort = wall_s() - t_sort;

    const double t_write = wall_s();
    std::vector<uint64_t> ssa(2 * r), esa(2 * r);
    for (uint64_t j = 0; j < r; ++j) {
        ssa[2 * j] = h_starts[j];
        ssa[2 * j + 1] = h_first[j];
        esa[2 * j] = (j + 1 < r ? (uint64_t) h_starts[j + 1] : n) - 1;
        esa[2 * j + 1] = h_last[j];
    }
    write_file(out_prefix + ".bwt", h_bwt.data(), n);
    write_file(out_prefix + ".ssa", ssa.data(), ssa.size() * 8);
    write_file(out_prefix + ".esa", esa.data(), esa.size() * 8);
    st.s_write = wall_s() - t_write;
}

}  // namespace rbg
