// mps_to_ma (pfbwt-f/src/mps_to_ma.cpp) on the GPU, with SA taken from the index's own phi instead of a suffix-array stream.
//
// The reference reads SA[0..n) as a stream (`pfbwt-f64 --stdout sa | mps_to_ma`, 8n bytes) on one thread.  Here SA comes
// from the toehold samples: inside BWT run j, SA[last row of j] = (samples_last[j] + 1) mod n (a stored sample is sa - 1,
// SURVEY.md A.1), and each phi step gives SA[i] -> SA[i - 1] down to the run's first row: n - R phi steps cover all n rows.
//
//   ma_rows_kernel    each lane draws a whole run (runs differ greatly in length), walks it from its last row with the
//                     shared phi_step and writes, for every row of the window, the list id of the .mps record holding SA[row]
//                     (or kNoList) into the chunk's id array, in row order.  The record of a text position is found through a
//                     directory over text positions: one load, then a short forward scan over the records' first / last.
//   ma_blocks_kernel  after cub::DeviceRunLengthEncode (+ an exclusive scan of the lengths) over the id array: one
//                     (offset, length, id) block per run; cub::DeviceSelect drops the kNoList blocks.
// A chunk is a range of whole runs; the host joins the last block of a chunk to the first of the next when they touch and
// carry the same list.
#include <cub/cub.cuh>

#include <unistd.h>

#include <algorithm>
#include <cstdio>
#include <string>
#include <vector>

#include "ma_build.hpp"
#include "cuda_host.hpp"
#include "device_index.cuh"
#include "knobs.hpp"
#include "raw_build.hpp"
#include "sdsl_writer.hpp"

namespace rbg {

// Kernels outside the anonymous namespace: their names stay the same from build to build (traces, profiles).
constexpr int kMaBlock = 256;
constexpr uint64_t kMaxChunkRows = 1ull << 28;     // <= 12.9 GB of chunk buffers; cub item counts are int, row offsets in a chunk u32

// The .mps records on the device: dir[p >> shift] = first record with last >= (p >> shift) << shift.
struct DevRecords {
    const uint64_t* first;
    const uint64_t* last;
    const uint32_t* list;
    const uint64_t* dir;
    uint64_t m;
    uint32_t shift;
};

__device__ __forceinline__ uint32_t list_at(const DevRecords& R, uint64_t p) {
    uint64_t k = __ldg(R.dir + (p >> R.shift));
    while (k < R.m && __ldg(R.last + k) < p) ++k;
    return k < R.m && __ldg(R.first + k) <= p ? __ldg(R.list + k) : kNoList;
}

// Runs [0, n_runs) of the chunk: run k ends at row run_last[k] with SA run_sa[k] and starts after run_last[k - 1] (run 0 at
// first_row).  Rows [row0, row_end) are written to ids[row - row0]; a run cut by row_end is still walked from its end.
__global__ void __launch_bounds__(kMaBlock) ma_rows_kernel(DevPhi P, DevRecords R, const uint64_t* __restrict__ run_last,
                                                           const uint64_t* __restrict__ run_sa, uint64_t n_runs, uint64_t first_row,
                                                           uint64_t row0, uint64_t row_end, uint32_t* __restrict__ ids,
                                                           unsigned long long* cursor, unsigned long long* phi_steps) {
    unsigned long long steps = 0;
    for (;;) {
        const uint64_t j = atomicAdd(cursor, 1ull);
        if (j >= n_runs) break;
        const uint64_t hi = __ldg(run_last + j);
        const uint64_t lo = max(j ? __ldg(run_last + j - 1) + 1 : first_row, row0);
        uint64_t sa = __ldg(run_sa + j);
        for (uint64_t row = hi;; --row) {
            if (row < row_end) ids[row - row0] = list_at(R, sa);
            if (row == lo) break;
            sa = phi_step(P, sa);
            ++steps;
        }
    }
    if (steps) atomicAdd(phi_steps, steps);
}

struct MaBlock {
    uint32_t off, len, id, pad;
};

struct HasList {
    __device__ __forceinline__ bool operator()(const MaBlock& b) const { return b.id != kNoList; }
};

__global__ void __launch_bounds__(kMaBlock) ma_blocks_kernel(const uint32_t* __restrict__ unique, const uint32_t* __restrict__ lens,
                                                             const uint32_t* __restrict__ offs, uint32_t n, MaBlock* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = MaBlock{offs[i], lens[i], unique[i], 0u};
}

namespace {

DevBuf dev_mem(size_t bytes) { return DevBuf(std::max<size_t>(bytes, 64)); }

struct Block {
    uint64_t first, last;
    uint32_t id;
};

// `first last word* ~0` per block, written to a temporary file renamed into place.
void write_ma(const std::vector<Block>& blocks, const MpsRecords& mps, const std::string& path, uint64_t& words) {
    const std::string tmp = path + ".tmp." + std::to_string((long) getpid());
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) throw io_error("cannot write " + tmp);
    std::vector<uint64_t> buf;
    bool ok = true;
    words = 0;
    for (size_t b = 0; b < blocks.size() && ok; ++b) {
        const Block& k = blocks[b];
        buf.push_back(k.first);
        buf.push_back(k.last);
        buf.insert(buf.end(), mps.words.begin() + mps.list_off[k.id], mps.words.begin() + mps.list_off[k.id + 1]);
        words += mps.list_off[k.id + 1] - mps.list_off[k.id];
        buf.push_back(~0ull);
        if (buf.size() >= (1u << 20) || b + 1 == blocks.size()) {
            ok = fwrite(buf.data(), 8, buf.size(), f) == buf.size();
            buf.clear();
        }
    }
    ok = fclose(f) == 0 && ok;
    if (ok) ok = rename(tmp.c_str(), path.c_str()) == 0;
    if (!ok) {
        remove(tmp.c_str());
        throw io_error("cannot write " + path);
    }
}

}  // namespace

void build_marker_array(const RunsBwt& bwt, const ToeholdArrays& tsa, const MpsRecords& mps, uint64_t row_begin, uint64_t row_end,
                        int device, const std::string& ma_path, const std::string& mab_path, rbg_ma_stats& st) {
    const uint64_t n = bwt.n, R = bwt.R;
    const double t_layout = wall_s();
    CU(cudaSetDevice(device));
    // run starts, and the runs the window [row_begin, row_end) overlaps: [j0, j1]
    std::vector<uint64_t> start(R + 1, 0);
    for (uint64_t j = 0; j < R; ++j) start[j + 1] = start[j] + bwt.lens[j];
    const uint64_t j0 = (uint64_t) (std::upper_bound(start.begin(), start.end(), row_begin) - start.begin()) - 1;
    const uint64_t j1 = (uint64_t) (std::upper_bound(start.begin(), start.end(), row_end - 1) - start.begin()) - 1;

    std::vector<Upload> owned;
    const LayoutKnobs knobs = layout_knobs();
    const DevPhi P = upload_phi(build_phi_dir(tsa, knobs.phi_shift, knobs.phi_parts, phi_slot_budget()), n, owned);

    // directory over text positions: about one record per bucket, so it costs no more than the records themselves
    const uint64_t m = mps.first.size();
    uint32_t shift = 0;
    while ((n >> shift) > std::max<uint64_t>(m, 1)) ++shift;
    std::vector<uint64_t> dir(((n - 1) >> shift) + 2);
    for (uint64_t b = 0, k = 0; b < dir.size(); ++b) {
        while (k < m && mps.last[k] < (b << shift)) ++k;
        dir[b] = k;
    }
    DevRecords D{upload(mps.first, owned), upload(mps.last, owned), upload(mps.list, owned), upload(dir, owned), m, shift};

    // chunk buffers: the id array plus, per row at worst, one run of the encoder, its scan and two blocks
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    const uint64_t per_row = 4 * 4 + 2 * sizeof(MaBlock);
    uint64_t cap = std::min<uint64_t>(kMaxChunkRows, (uint64_t) free_b / 2 / per_row);
    if (const uint64_t rows = knob_ma_chunk_rows()) cap = std::max<uint64_t>(1, std::min(cap, rows));
    uint64_t max_run = 0;
    for (uint64_t j = j0; j <= j1; ++j) max_run = std::max(max_run, bwt.lens[j]);
    const uint64_t rows_alloc = std::max(cap, std::min(max_run, row_end - row_begin));      // a chunk holds at least one run
    if (rows_alloc > kMaxChunkRows) throw std::invalid_argument("a BWT run longer than 2^28 rows (one device pass)");
    uint64_t runs_alloc = 0;                                                                 // most runs in one chunk
    for (uint64_t a = j0; a <= j1;) {
        const uint64_t base = std::max(start[a], row_begin);
        uint64_t e = (uint64_t) (std::upper_bound(start.begin() + a + 1, start.begin() + j1 + 2, base + cap) - start.begin()) - 1;
        e = std::max(e, a + 1);
        runs_alloc = std::max(runs_alloc, e - a);
        a = e;
    }
    DevBuf d_ids = dev_mem(rows_alloc * 4), d_unique = dev_mem(rows_alloc * 4), d_lens = dev_mem(rows_alloc * 4),
           d_offs = dev_mem(rows_alloc * 4);
    DevBuf d_blocks = dev_mem(rows_alloc * sizeof(MaBlock)), d_sel = dev_mem(rows_alloc * sizeof(MaBlock));
    DevBuf d_run_last = dev_mem(runs_alloc * 8), d_run_sa = dev_mem(runs_alloc * 8), d_ctr = dev_mem(4 * 8);
    size_t tmp_a = 0, tmp_b = 0, tmp_c = 0;
    const int items = (int) rows_alloc;
    CU(cub::DeviceRunLengthEncode::Encode(nullptr, tmp_a, d_ids.as<uint32_t>(), d_unique.as<uint32_t>(), d_lens.as<uint32_t>(),
                                          d_ctr.as<int>(), items));
    CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp_b, d_lens.as<uint32_t>(), d_offs.as<uint32_t>(), items));
    CU(cub::DeviceSelect::If(nullptr, tmp_c, d_blocks.as<MaBlock>(), d_sel.as<MaBlock>(), d_ctr.as<int>() + 1, items, HasList()));
    const size_t tmp_bytes = std::max(tmp_a, std::max(tmp_b, tmp_c));
    DevBuf d_tmp = dev_mem(tmp_bytes);
    cudaStream_t s;
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    cudaEvent_t ev[3];
    for (auto& e : ev) CU(cudaEventCreate(&e));
    struct Cleanup {
        cudaStream_t s;
        cudaEvent_t* ev;
        ~Cleanup() { for (int i = 0; i < 3; ++i) cudaEventDestroy(ev[i]); cudaStreamDestroy(s); }
    } cleanup{s, ev};
    std::vector<uint64_t> h_last(runs_alloc), h_sa(runs_alloc);
    std::vector<MaBlock> h_sel;
    std::vector<Block> blocks;
    unsigned long long* ctr = d_ctr.as<unsigned long long>();     // [0] run cursor, [1] phi steps; [2..3] the encoder / select counts
    int* counts = (int*) (ctr + 2);
    CU(cudaMemsetAsync(ctr + 1, 0, 8, s));
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    st.s_layout = wall_s() - t_layout;

    // chunks of whole runs, at most `cap` window rows each (or one run)
    for (uint64_t a = j0; a <= j1;) {
        const uint64_t row0 = std::max(start[a], row_begin);
        uint64_t e = (uint64_t) (std::upper_bound(start.begin() + a + 1, start.begin() + j1 + 2, row0 + cap) - start.begin()) - 1;
        e = std::max(e, a + 1);                                                   // runs [a, e)
        const uint64_t rows = std::min(start[e], row_end) - row0;
        for (uint64_t j = a; j < e; ++j) {
            h_last[j - a] = start[j + 1] - 1;
            h_sa[j - a] = tsa.samples_last[j] + 1 == n ? 0 : tsa.samples_last[j] + 1;
        }
        CU(cudaMemcpyAsync(d_run_last.p, h_last.data(), (e - a) * 8, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(d_run_sa.p, h_sa.data(), (e - a) * 8, cudaMemcpyHostToDevice, s));
        CU(cudaMemsetAsync(ctr, 0, 8, s));
        CU(cudaEventRecord(ev[0], s));
        const uint64_t want = (e - a + kMaBlock - 1) / kMaBlock;
        const int grid = (int) std::min<uint64_t>(want, (uint64_t) sms * 8);
        ma_rows_kernel<<<grid, kMaBlock, 0, s>>>(P, D, d_run_last.as<uint64_t>(), d_run_sa.as<uint64_t>(), e - a, start[a], row0, row_end,
                                                 d_ids.as<uint32_t>(), ctr, ctr + 1);
        CU(cudaGetLastError());
        CU(cudaEventRecord(ev[1], s));
        size_t tb = tmp_bytes;
        CU(cub::DeviceRunLengthEncode::Encode(d_tmp.p, tb, d_ids.as<uint32_t>(), d_unique.as<uint32_t>(), d_lens.as<uint32_t>(), counts,
                                              (int) rows, s));
        int n_runs = 0;
        CU(cudaMemcpyAsync(&n_runs, counts, 4, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        tb = tmp_bytes;
        CU(cub::DeviceScan::ExclusiveSum(d_tmp.p, tb, d_lens.as<uint32_t>(), d_offs.as<uint32_t>(), n_runs, s));
        ma_blocks_kernel<<<(n_runs + kMaBlock - 1) / kMaBlock, kMaBlock, 0, s>>>(d_unique.as<uint32_t>(), d_lens.as<uint32_t>(),
                                                                                 d_offs.as<uint32_t>(), (uint32_t) n_runs, d_blocks.as<MaBlock>());
        CU(cudaGetLastError());
        tb = tmp_bytes;
        CU(cub::DeviceSelect::If(d_tmp.p, tb, d_blocks.as<MaBlock>(), d_sel.as<MaBlock>(), counts + 1, n_runs, HasList(), s));
        CU(cudaEventRecord(ev[2], s));
        int n_sel = 0;
        CU(cudaMemcpyAsync(&n_sel, counts + 1, 4, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        h_sel.resize(n_sel);
        if (n_sel) CU(cudaMemcpyAsync(h_sel.data(), d_sel.p, (size_t) n_sel * sizeof(MaBlock), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, ev[0], ev[1]));
        st.ms_rows_kernel += ms;
        CU(cudaEventElapsedTime(&ms, ev[1], ev[2]));
        st.ms_blocks += ms;
        for (int i = 0; i < n_sel; ++i) {
            const MaBlock& b = h_sel[i];
            const uint64_t f = row0 + b.off, l = f + b.len - 1;
            if (i == 0 && !blocks.empty() && blocks.back().last + 1 == f && blocks.back().id == b.id) blocks.back().last = l;   // the seam
            else blocks.push_back(Block{f, l, b.id});
        }
        st.rows += rows;
        a = e;
    }
    unsigned long long steps = 0;
    CU(cudaMemcpy(&steps, ctr + 1, 8, cudaMemcpyDeviceToHost));
    st.phi_steps = steps;
    st.ma_records = blocks.size();

    const double t_write = wall_s();
    write_ma(blocks, mps, ma_path, st.ma_words);
    if (!mab_path.empty()) {             // rb_build -m over the .ma just written (the .ma stays even when this refuses it)
        MarkerArrays ma = markers_from_ma(ma_path);
        const std::string tmp = mab_path + ".tmp." + std::to_string((long) getpid());
        try {
            write_mab(ma, tmp);
        } catch (...) {
            remove(tmp.c_str());
            throw;
        }
        if (rename(tmp.c_str(), mab_path.c_str()) != 0) {
            remove(tmp.c_str());
            throw io_error("cannot write " + mab_path);
        }
    }
    st.s_write = wall_s() - t_write;
}

}  // namespace rbg
