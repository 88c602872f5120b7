// rb_build's job on the GPU (SURVEY.md §8(f) row 4): from the builder's raw outputs
// (.bwt one byte per row, .ssa/.esa run-boundary suffix-array samples, .ma marker records) to the
// flat arrays of formats.hpp -- from which either the device layout is built directly
// (rbg_index_open_raw) or the reference's .rbwt/.tsa/.mab files are written byte for byte
// (rbg_build_index, sdsl_writer.hpp).
//
// Reference code replaced:
//   rle_string(std::string fname, B)   include/rle_string.hpp:44-97   char-at-a-time `ifs >> c` over n bytes,
//                                       three vector<bool> of n bits, then sd_vector / wt_huff construction
//   ToeholdSA(n, r, ssa, esa)          include/toehold_sa.hpp:28-36,105-156   std::sort of r pairs
//   rle_window_arr(fname)              pfbwt-f/include/rle_window_array.hpp:15-50
//
// Kernels (HBM-streaming, 16 bytes per thread per load, contiguous tiles so run order is preserved):
//   rle_count_kernel   per-tile number of run starts (+ number of whitespace bytes, see below)
//   rle_emit_kernel    tile offsets from an exclusive scan of those counts; writes (start row, head) per run
// The .bwt streams through two pinned buffers: fread of chunk k+1 overlaps H2D + kernels of chunk k.
#include <cub/cub.cuh>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "cuda_host.hpp"
#include "formats.hpp"
#include "layout.hpp"
#include "raw_build.hpp"

namespace rbg {

namespace {

constexpr int kThreads = 256;
constexpr int kVecPerThread = 8;                                   // 16-byte vectors per thread
constexpr uint64_t kTileBytes = (uint64_t) kThreads * 16 * kVecPerThread;   // 32 KB per CTA

// `ifs >> c` maps nothing, the ctor maps 0 -> TERMINATOR(1): c = c > 1 ? c : 1 (rle_string.hpp:59,62)
__device__ __forceinline__ uint32_t norm4(uint32_t w) {
    // per byte: 0 -> 1 (bytes equal to 1 stay 1)
    const uint32_t zero = ~(((w & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w | 0x7f7f7f7fu);     // 0x80 where the byte is 0
    return w | (zero >> 7);
}

// bit i set iff byte i of (w0..w3) differs from the byte before it (prev = byte before byte 0)
__device__ __forceinline__ uint32_t boundary_mask(const uint4& v, uint32_t prev) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t mask = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t shifted = (w[k] << 8) | prev;              // byte i-1 aligned under byte i
        const uint32_t x = w[k] ^ shifted;                         // non-zero byte = boundary
        const uint32_t nz = ((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x; // bit 7 of each byte set iff byte != 0
        mask |= (((nz >> 7) & 1u) | ((nz >> 14) & 2u) | ((nz >> 21) & 4u) | ((nz >> 28) & 8u)) << (4 * k);
        prev = w[k] >> 24;
    }
    return mask;
}

__device__ __forceinline__ uint32_t whitespace_count(const uint4& v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t n = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const uint32_t c = (w[k] >> (8 * b)) & 0xff;
            n += (c == 32u) | (c - 9u <= 4u);
        }
    return n;
}

// One CTA per tile of kTileBytes; `bytes` is padded to a multiple of 16 with copies of its last byte.
// carry = normalised byte before byte 0 of this chunk, or 0x100 for the first chunk (row 0 starts a run).
template <bool kEmit>
__global__ void __launch_bounds__(kThreads) rle_kernel(const uint4* __restrict__ bytes, uint64_t n_vec, uint32_t carry,
                                                       uint64_t row0, uint32_t* __restrict__ tile_count,
                                                       const uint64_t* __restrict__ tile_off, uint64_t* __restrict__ starts,
                                                       uint8_t* __restrict__ heads, unsigned long long* __restrict__ n_space) {
    __shared__ uint32_t warp_sum[kThreads / 32];
    __shared__ uint64_t tile_base;
    const uint64_t vec0 = (uint64_t) blockIdx.x * kThreads * kVecPerThread;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t total = 0, spaces = 0;
    uint64_t base = kEmit ? tile_off[blockIdx.x] : 0;
    for (int it = 0; it < kVecPerThread; ++it) {
        const uint64_t vi = vec0 + (uint64_t) it * kThreads + threadIdx.x;
        uint32_t mask = 0;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (vi < n_vec) {
            v = bytes[vi];
            if (!kEmit) spaces += whitespace_count(v);
            v.x = norm4(v.x); v.y = norm4(v.y); v.z = norm4(v.z); v.w = norm4(v.w);
            uint32_t prev;
            if (vi == 0) prev = carry;
            else prev = norm4((uint32_t) reinterpret_cast<const uint8_t*>(bytes)[vi * 16 - 1]) & 0xff;
            mask = boundary_mask(v, prev & 0xff);
            if (vi == 0 && carry > 0xff) mask |= 1u;
        }
        const uint32_t cnt = __popc(mask);
        if (!kEmit) {
            total += cnt;
        } else {
            // CTA-wide exclusive scan of cnt
            uint32_t incl = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += t;
            }
            if (lane == 31) warp_sum[warp] = incl;
            __syncthreads();
            uint32_t wbase = 0, all = 0;
#pragma unroll
            for (int w = 0; w < kThreads / 32; ++w) {
                const uint32_t s = warp_sum[w];
                if (w < warp) wbase += s;
                all += s;
            }
            uint64_t o = base + wbase + incl - cnt;
            const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
            while (mask) {
                const int b = __ffs(mask) - 1;
                mask &= mask - 1;
                starts[o] = row0 + vi * 16 + b;
                heads[o] = (uint8_t) (w4[b >> 2] >> (8 * (b & 3)));
                ++o;
            }
            base += all;
            __syncthreads();
        }
    }
    if (!kEmit) {
#pragma unroll
        for (int d = 16; d; d >>= 1) {
            total += __shfl_xor_sync(0xffffffffu, total, d);
            spaces += __shfl_xor_sync(0xffffffffu, spaces, d);
        }
        if (lane == 0) warp_sum[warp] = total;
        if (lane == 0 && spaces) atomicAdd(n_space, (unsigned long long) spaces);
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t s = 0;
            for (int w = 0; w < kThreads / 32; ++w) s += warp_sum[w];
            tile_count[blockIdx.x] = s;
        }
    }
    (void) tile_base;
}

__global__ void widen_kernel(const uint32_t* __restrict__ in, uint64_t* __restrict__ out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}

// Room for n items of T, growing by at least half of what `b` holds.
template <class T>
T* grow(DevBuf& b, size_t n) {
    const size_t held = b.cap / sizeof(T);
    b.reserve(n * sizeof(T), std::max(n, held + held / 2) * sizeof(T));
    return b.as<T>();
}

std::vector<uint64_t> read_u64_file(const std::string& path) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) throw io_error("bad file: " + path);
    fseek(f, 0, SEEK_END);
    const long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<uint64_t> v((size_t) sz / 8);
    if (!v.empty() && fread(v.data(), 8, v.size(), f) != v.size()) { fclose(f); throw io_error("short read: " + path); }
    fclose(f);
    return v;
}

}  // namespace

// rle_string(fname): run heads and lengths of the BWT file.
RunsBwt rle_bwt_gpu(const std::string& path, int device, RawBuildStats* st) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) throw io_error("bad file: " + path);
    CU(cudaSetDevice(device));
    const size_t chunk = (size_t) 64 << 20;
    PinnedBuf hb_mem[2] = {PinnedBuf(chunk + 16), PinnedBuf(chunk + 16)};
    uint8_t* hb[2] = {hb_mem[0].as<uint8_t>(), hb_mem[1].as<uint8_t>()};
    DevBuf d_bytes_mem[2], d_cnt_mem, d_cnt64_mem, d_off_mem, d_space_mem, d_tmp_mem, d_starts, d_heads;
    uint8_t* d_bytes[2] = {grow<uint8_t>(d_bytes_mem[0], chunk + 16), grow<uint8_t>(d_bytes_mem[1], chunk + 16)};
    const uint32_t max_tiles = (uint32_t) ((chunk + kTileBytes - 1) / kTileBytes);
    uint32_t* d_cnt = grow<uint32_t>(d_cnt_mem, max_tiles);
    uint64_t* d_cnt64 = grow<uint64_t>(d_cnt64_mem, max_tiles + 1);
    uint64_t* d_off = grow<uint64_t>(d_off_mem, max_tiles + 1);
    unsigned long long* d_space = grow<unsigned long long>(d_space_mem, 1);
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_cnt64, d_off, max_tiles + 1);
    uint8_t* d_tmp = grow<uint8_t>(d_tmp_mem, tmp_bytes);
    cudaStream_t s;
    CU(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    CU(cudaMemsetAsync(d_space, 0, 8, s));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));

    RunsBwt out;
    std::vector<uint64_t> starts;
    double t_read = 0, t_gpu_wait = 0;
    float ms_kernels = 0;
    uint64_t row0 = 0;
    uint32_t carry = 0x100;
    int cur = 0;
    double t0 = wall_s();
    size_t got = fread(hb[0], 1, chunk, f);
    t_read += wall_s() - t0;
    std::vector<uint64_t> h_starts;
    std::vector<uint8_t> h_heads;
    while (got) {
        const uint64_t n_vec = (got + 15) / 16;
        memset(hb[cur] + got, hb[cur][got - 1], n_vec * 16 - got);           // pad: no new run starts
        const uint32_t tiles = (uint32_t) ((n_vec * 16 + kTileBytes - 1) / kTileBytes);
        CU(cudaMemcpyAsync(d_bytes[cur], hb[cur], n_vec * 16, cudaMemcpyHostToDevice, s));
        CU(cudaEventRecord(e0, s));
        rle_kernel<false><<<tiles, kThreads, 0, s>>>((const uint4*) d_bytes[cur], n_vec, carry, row0, d_cnt, nullptr, nullptr,
                                                     nullptr, d_space);
        widen_kernel<<<(tiles + 1 + 255) / 256, 256, 0, s>>>(d_cnt, d_cnt64, tiles);
        cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_cnt64, d_off, tiles + 1, s);
        uint64_t n_runs = 0;
        CU(cudaMemcpyAsync(&n_runs, d_off + tiles, 8, cudaMemcpyDeviceToHost, s));
        // overlap: read the next chunk while the GPU counts
        t0 = wall_s();
        const size_t got_next = fread(hb[cur ^ 1], 1, chunk, f);
        t_read += wall_s() - t0;
        t0 = wall_s();
        CU(cudaStreamSynchronize(s));
        t_gpu_wait += wall_s() - t0;
        uint64_t* d_starts_p = grow<uint64_t>(d_starts, n_runs + 1);
        uint8_t* d_heads_p = grow<uint8_t>(d_heads, n_runs + 1);
        rle_kernel<true><<<tiles, kThreads, 0, s>>>((const uint4*) d_bytes[cur], n_vec, carry, row0, nullptr, d_off, d_starts_p,
                                                    d_heads_p, nullptr);
        CU(cudaEventRecord(e1, s));
        h_starts.resize(n_runs);
        h_heads.resize(n_runs);
        if (n_runs) {
            CU(cudaMemcpyAsync(h_starts.data(), d_starts_p, n_runs * 8, cudaMemcpyDeviceToHost, s));
            CU(cudaMemcpyAsync(h_heads.data(), d_heads_p, n_runs, cudaMemcpyDeviceToHost, s));
        }
        t0 = wall_s();
        CU(cudaStreamSynchronize(s));
        t_gpu_wait += wall_s() - t0;
        CU(cudaGetLastError());
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        ms_kernels += ms;
        starts.insert(starts.end(), h_starts.begin(), h_starts.end());
        out.heads.insert(out.heads.end(), h_heads.begin(), h_heads.end());
        const uint8_t last = hb[cur][got - 1];
        carry = last > 1 ? last : 1;
        row0 += got;
        cur ^= 1;
        got = got_next;
    }
    fclose(f);
    unsigned long long n_space = 0;
    CU(cudaMemcpy(&n_space, d_space, 8, cudaMemcpyDeviceToHost));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaStreamDestroy(s);
    if (n_space)      // formatted extraction skips whitespace bytes; no BWT of the documented pipeline contains any
        throw alphabet_error("the .bwt contains whitespace bytes, which the reference's reader (ifs >> c) would drop");
    out.n = row0;
    out.R = starts.size();
    out.lens.resize(out.R);
    for (uint64_t j = 0; j < out.R; ++j) out.lens[j] = (j + 1 < out.R ? starts[j + 1] : out.n) - starts[j];
    if (st) {
        st->bwt_bytes = out.n;
        st->runs = out.R;
        st->s_read = t_read;
        st->s_gpu_wait = t_gpu_wait;
        st->ms_kernels = ms_kernels;
        st->launches += 0;
    }
    return out;
}

// ToeholdSA(n, r, ssa, esa): samples of the first / last row of every run.  The (text position, run) pairs
// of the run starts are sorted by position on the GPU (stable radix sort = std::sort on pairs here, the
// second members being increasing).
ToeholdArrays toehold_from_raw(const std::string& ssa_path, const std::string& esa_path, uint64_t n, uint64_t r, int device) {
    std::vector<uint64_t> ssa = read_u64_file(ssa_path), esa = read_u64_file(esa_path);
    if (ssa.size() / 2 != r || esa.size() / 2 != r)
        throw format_error(".ssa/.esa do not hold one sample per BWT run (" + std::to_string(ssa.size() / 2) + ", " +
                           std::to_string(esa.size() / 2) + " vs " + std::to_string(r) + " runs)");
    ToeholdArrays t;
    t.r = r;
    t.n = n;
    t.samples_last.resize(r);
    std::vector<uint64_t> keys(r), vals(r);
    for (uint64_t i = 0; i < r; ++i) {
        const uint64_t y = ssa[2 * i + 1], z = esa[2 * i + 1];
        keys[i] = y ? y - 1 : n - 1;                                  // toehold_sa.hpp:140
        vals[i] = i;
        t.samples_last[i] = z ? z - 1 : n - 1;                        // :152
        if (keys[i] >= n || t.samples_last[i] >= n) throw format_error("suffix-array sample beyond the text length");
    }
    CU(cudaSetDevice(device));
    DevBuf k_mem[2], v_mem[2], tmp_mem;
    uint64_t *k_in = grow<uint64_t>(k_mem[0], r), *k_out = grow<uint64_t>(k_mem[1], r);
    uint64_t *v_in = grow<uint64_t>(v_mem[0], r), *v_out = grow<uint64_t>(v_mem[1], r);
    CU(cudaMemcpy(k_in, keys.data(), r * 8, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(v_in, vals.data(), r * 8, cudaMemcpyHostToDevice));
    size_t tb = 0;
    const int end_bit = 64 - __builtin_clzll(n | 1);
    cub::DeviceRadixSort::SortPairs(nullptr, tb, k_in, k_out, v_in, v_out, (int64_t) r, 0, end_bit);
    cub::DeviceRadixSort::SortPairs(grow<uint8_t>(tmp_mem, tb), tb, k_in, k_out, v_in, v_out, (int64_t) r, 0, end_bit);
    t.pred_to_run.resize(r);
    CU(cudaMemcpy(keys.data(), k_out, r * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t.pred_to_run.data(), v_out, r * 8, cudaMemcpyDeviceToHost));
    CU(cudaGetLastError());
    keys.erase(std::unique(keys.begin(), keys.end()), keys.end());   // pred_ is a bit vector: duplicates collapse
    t.pred = std::move(keys);
    return t;
}

// rle_window_arr(fname): records `first_row last_row marker* 0xFFFF...F`.
MarkerArrays markers_from_ma(const std::string& path) {
    std::vector<uint64_t> in = read_u64_file(path);
    const uint64_t delim = ~0ull;
    MarkerArrays m;
    m.wsize = 10;                                                     // rle_window_array.hpp:264 (never set from the file)
    if (in.size() < 2) throw format_error(".ma: no records in " + path);
    // get_last_position_ (:244-250): keys[1] of the record after the second-to-last delimiter
    size_t i = in.size() - 2;
    while (in[i] != delim) {
        if (i == 0) throw format_error(".ma: fewer than two records (the reference reads out of bounds here)");
        --i;
    }
    if (i + 2 >= in.size()) throw format_error(".ma: malformed last record");
    const uint64_t size = in[i + 2] + 2;
    m.size_starts = m.size_ends = size;
    uint64_t keys[2] = {0, 0};
    int state = 0;
    std::vector<uint64_t> values;
    for (size_t k = 0; k < in.size(); ++k) {
        if (in[k] == delim) {
            if (keys[0] == 0 || keys[1] == 0) throw format_error(".ma: window starting or ending at row 0 (the reference exits)");
            if (keys[0] >= size || keys[1] >= size) throw format_error(".ma: window beyond the last record's end");
            m.starts.push_back(keys[0]);
            m.ends.push_back(keys[1]);
            m.idxs.push_back(m.arr.size());
            m.arr.insert(m.arr.end(), values.begin(), values.end());
            values.clear();
            state = 0;
        } else if (state < 2) {
            keys[state++] = in[k];
        } else {
            values.push_back(in[k]);
        }
    }
    m.size_idxs = m.arr.size();
    auto as_bits = [](std::vector<uint64_t>& v) {
        std::sort(v.begin(), v.end());
        v.erase(std::unique(v.begin(), v.end()), v.end());
    };
    as_bits(m.starts);
    as_bits(m.ends);
    as_bits(m.idxs);
    while (!m.idxs.empty() && m.idxs.back() >= m.size_idxs) m.idxs.pop_back();      // arr_idxs.resize(arr_.size()) drops them
    return m;
}

}  // namespace rbg
