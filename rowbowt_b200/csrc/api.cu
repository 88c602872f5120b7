// C ABI of librowbowt_gpu.so (include/rowbowt_gpu.h): index residency on one GPU and the
// batched query call.  No CPU fallback: without a CUDA device every entry point that needs
// one returns RBG_E_CUDA.
#include "../../include/rowbowt_gpu.h"

#include <cuda_runtime.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <future>
#include <memory>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "cuda_host.hpp"
#include "bwt_build.hpp"
#include "formats.hpp"
#include "host_pack.hpp"
#include "raw_build.hpp"
#include "sdsl_writer.hpp"
#include "kernels.cuh"
#include "knobs.hpp"
#include "layout.hpp"
#include "ma_build.hpp"

using namespace rbg;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

// Reserves with headroom: the next slightly larger batch reuses the buffer.
template <class B>
void reserve(B& b, size_t bytes) { b.reserve(bytes, bytes + bytes / 8 + 256); }

struct HostSeedResult {  // pinned buffers behind one rbg_seed_result
    PinnedBuf seed_off, seeds, markers;
    rbg_index* ix = nullptr;
};

struct GreedyScratch {   // device buffers of rbg_markers_greedy
    DevBuf bad, item_seeds, item_words, seed_off, word_off, seeds, words;
};

static_assert(sizeof(DevSeed) == sizeof(rbg_seed) && sizeof(rbg_seed) == 40, "rbg_seed layout");

struct HostResult {      // pinned buffers behind one rbg_result
    PinnedBuf lo, hi, toehold, loc_off, locs, locs_hi, mk_off, markers;      // lo / hi hold u32 planes with RBG_NARROW_RANGES
    rbg_index* ix = nullptr;
};

// Results handed to callers through `_owner`; up to 4 given back are kept for the next call.
template <class H>
class ResultPool {
    std::mutex mu;
    std::vector<std::unique_ptr<H>> kept;
  public:
    H* take(rbg_index* ix) {
        {
            std::lock_guard<std::mutex> lock(mu);
            if (!kept.empty()) {
                H* h = kept.back().release();
                kept.pop_back();
                return h;
            }
        }
        H* h = new H;
        h->ix = ix;
        return h;
    }
    void give_back(H* h) {
        std::lock_guard<std::mutex> lock(mu);
        if (kept.size() < 4) kept.emplace_back(h);
        else delete h;
    }
};

}  // namespace

struct rbg_reads {
    rbg_index* ix = nullptr;
    uint64_t n_reads = 0, n_bytes = 0;
    bool prepacked = false;              // `packed` / `flags` came from the host (rbg_reads_upload_packed): no pack_kernel
    bool has_bases = false;
    DevBuf bases, offs, packed, flags;
    DevBuf lo, hi, toehold, loc_cnt, loc_off, locs, locs_hi, mk_cnt, mk_off, mk_first, markers, scan_tmp;
    DevBuf lo32, hi32;                   // RBG_NARROW_RANGES: what leaves the device instead of lo / hi
    uint64_t n_locs = 0, n_markers = 0;
    uint32_t last_mode = 0;
    bool ran = false;
};

namespace {

// Everything ONE call in flight needs: its own streams, events, counters and device scratch.  rbg_query and friends
// take a lane for the duration of the call, so calls on one handle run concurrently (SURVEY.md 8(b) threading row).
struct Lane {
    static constexpr int kMaxChunks = 64;
    cudaStream_t stream = nullptr;                   // kernels
    cudaStream_t s_in = nullptr, s_out = nullptr;    // H2D / D2H of the pipelined rbg_query
    cudaStream_t s_srch[2] = {nullptr, nullptr};     // pack + search of even / odd chunks: chunk c+1 fills the SMs chunk c's tail leaves idle
    cudaEvent_t ev[8] = {nullptr};
    cudaEvent_t ev_in[kMaxChunks] = {nullptr}, ev_cmp[kMaxChunks] = {nullptr}, ev_span[6] = {nullptr};
    cudaEvent_t ev_tot[kMaxChunks] = {nullptr}, ev_loc[kMaxChunks] = {nullptr};   // pipelined locate: chunk total known / chunk located
    cudaEvent_t ev_pack[kMaxChunks] = {nullptr};     // pack_kernel of chunk c done (orders the packs of neighbouring chunks across s_srch)
    uint64_t* h_tot = nullptr;           // pinned [kMaxChunks]: running number of locations after each chunk
    uint64_t* d_base = nullptr;          // device scalar: where the next chunk's offsets start
    DevCounters* d_ctr = nullptr;
    DevCounters* h_ctr = nullptr;        // pinned
    rbg_reads scratch;                   // reused by rbg_query
    GreedyScratch greedy;                // reused by rbg_markers_greedy
    bool busy = false;
    // RBG_BLOCKING_SYNC=1 (the host drivers set it): the calling thread SLEEPS while it waits for the GPU instead of spinning.
    // A driver runs parser and formatter threads on every core beside its GPU worker; a spinning waiter competes with them
    // for a core and, descheduled, adds milliseconds to a 0.4 ms call (profiles/r2_call_latency_and_search_variants.jsonl
    // against the 6.3 ms per call RBG_HOST_STATS showed inside rb_align).  Costs ~20-50 us of wake-up latency per wait.
    bool blocking = false;
    cudaEvent_t ev_done[3] = {nullptr, nullptr, nullptr};
    void wait_stream(cudaStream_t st, int slot) {
        if (!blocking) { CU(cudaStreamSynchronize(st)); return; }
        CU(cudaEventRecord(ev_done[slot], st));
        CU(cudaEventSynchronize(ev_done[slot]));
    }
    void create() {
        blocking = knob_blocking_sync();
        const unsigned wait_flags = cudaEventDisableTiming | (blocking ? cudaEventBlockingSync : 0u);
        for (auto& ev1 : ev_done) CU(cudaEventCreateWithFlags(&ev1, wait_flags));
        CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
        for (auto& st : s_srch) CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        for (auto& e : ev) CU(cudaEventCreate(&e));
        for (auto& e : ev_span) CU(cudaEventCreate(&e));
        for (auto& e : ev_in) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : ev_cmp) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : ev_tot) CU(cudaEventCreateWithFlags(&e, wait_flags));
        for (auto& e : ev_loc) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : ev_pack) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CU(cudaHostAlloc(&h_tot, sizeof(uint64_t) * kMaxChunks, cudaHostAllocDefault));
        CU(cudaMalloc(&d_base, sizeof(uint64_t)));
        CU(cudaMalloc(&d_ctr, sizeof(DevCounters)));
        CU(cudaHostAlloc(&h_ctr, sizeof(DevCounters), cudaHostAllocDefault));
    }
    ~Lane() {
        if (d_ctr) cudaFree(d_ctr);
        if (h_ctr) cudaFreeHost(h_ctr);
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        for (auto& e : ev_in) if (e) cudaEventDestroy(e);
        for (auto& e : ev_cmp) if (e) cudaEventDestroy(e);
        for (auto& e : ev_tot) if (e) cudaEventDestroy(e);
        for (auto& e : ev_loc) if (e) cudaEventDestroy(e);
        for (auto& e : ev_pack) if (e) cudaEventDestroy(e);
        for (auto& e : ev_span) if (e) cudaEventDestroy(e);
        for (auto& e : ev_done) if (e) cudaEventDestroy(e);
        if (h_tot) cudaFreeHost(h_tot);
        if (d_base) cudaFree(d_base);
        if (stream) cudaStreamDestroy(stream);
        if (s_in) cudaStreamDestroy(s_in);
        if (s_out) cudaStreamDestroy(s_out);
        for (auto& st : s_srch) if (st) cudaStreamDestroy(st);
    }
};

}  // namespace

struct rbg_index {
    int device = 0;
    std::vector<Upload> owned;
    DevLeafDir dir{};
    DevPairDir pair{};                   // lines == nullptr: the count search takes one base per step
    std::vector<Upload> pair_owned;      // kept out of `owned`: a layout cache does not carry the pair directory
    DevToehold toe{};
    DevPhi phi{};
    DevMarkers mk{};
    CodeTable codes{};
    DevFtab ft{};                        // k-mer seed table (k == 0: none)
    std::vector<ulonglong2> ft_host;     // host copy of ft.range (rbg_ftab_save / rbg_ftab_lookup)
    void* hot = nullptr;                 // one allocation: superblock counts + ftab
    size_t hot_bytes = 0;
    rbg_info info{};
    rbg_stats stats{};                   // of the call that finished last
    std::mutex mu;                       // lanes, stats
    std::condition_variable cv;
    std::vector<std::unique_ptr<Lane>> lanes;
    int max_lanes = 2;
    int n_busy = 0;
    bool exclusive = false;              // an ftab rebuild owns the handle
    ResultPool<HostResult> results;
    ResultPool<HostSeedResult> seed_results;
    // One free lane (creating it on first use); with `all`, waits until no call is in flight and keeps others out.
    Lane* acquire(bool all = false) {
        std::unique_lock<std::mutex> lock(mu);
        for (;;) {
            if (!exclusive && (all ? n_busy == 0 : n_busy < max_lanes)) break;
            cv.wait(lock);
        }
        Lane* l = nullptr;
        for (auto& c : lanes) if (!c->busy) { l = c.get(); break; }
        if (!l) {
            std::unique_ptr<Lane> fresh(new Lane);
            CU(cudaSetDevice(device));
            fresh->create();
            l = fresh.get();
            lanes.push_back(std::move(fresh));
        }
        l->busy = true;
        ++n_busy;
        exclusive = all;
        return l;
    }
    void release(Lane* l, const rbg_stats* st = nullptr) {
        {
            std::lock_guard<std::mutex> lock(mu);
            l->busy = false;
            --n_busy;
            exclusive = false;
            if (st) stats = *st;
        }
        cv.notify_all();
    }
    ~rbg_index() {
        cudaSetDevice(device);
        lanes.clear();
        if (hot) cudaFree(hot);
    }
};

namespace rbg {
DevPhi upload_phi(const PhiDir& pd, uint64_t n, std::vector<Upload>& owned, size_t* acc) {
    DevPhi P{};
    P.l1 = upload(pd.l1, owned, acc);
    P.slots = upload(pd.slots, owned, acc);
    P.ovf_keys = upload(pd.ovf_keys, owned, acc);
    P.ovf_prev_lo = upload(pd.ovf_prev.lo, owned, acc);
    P.ovf_prev_hi = pd.ovf_prev.wide ? upload(pd.ovf_prev.hi, owned, acc) : nullptr;
    P.n = n;
    P.shift = pd.shift;
    return P;
}
}  // namespace rbg

namespace {

// A lane held for the scope of one C-ABI call; stats are published when the call succeeds.
struct LaneHold {
    rbg_index* ix;
    Lane* lane;
    rbg_stats stats{};
    bool publish = false;
    LaneHold(rbg_index* i, bool all = false) : ix(i), lane(i->acquire(all)) {}
    ~LaneHold() { ix->release(lane, publish ? &stats : nullptr); }
    LaneHold(const LaneHold&) = delete;
    LaneHold& operator=(const LaneHold&) = delete;
};

// The small, hot arrays -- superblock counts (read by every LF step) and the k-mer seed table (read
// once per read) -- live in ONE allocation, (re)built whenever the ftab changes.  No L2 access-policy window is set:
// measured on the BASELINE batch with the final 158 MB directory, a window marking this region persisting LOST 4 %
// (22.9 vs 21.9 ms: both arrays are hot enough to stay under plain LRU, and the carve-out is taken from the lines), and
// a window over the directory itself (83 MB persisting) lost 6 % and starved the phi slots (locate 12.7 -> 51 ms).
void rebuild_hot_region(rbg_index* ix, uint32_t k, bool with_toe) {
    const size_t super_bytes = (size_t) ix->dir.n_super * 4 * sizeof(uint64_t);
    const size_t entries = k ? (size_t) 1 << (2 * k) : 0;
    const size_t off_range = (super_bytes + 255) & ~(size_t) 255;
    const size_t off_toe = off_range + entries * sizeof(ulonglong2);
    const size_t total = std::max<size_t>(off_toe + (with_toe ? entries * sizeof(uint64_t) : 0), 256);
    void* region = nullptr;
    CU(cudaMalloc(&region, total));
    CU(cudaMemcpy(region, ix->dir.super, super_bytes, cudaMemcpyDeviceToDevice));
    if (ix->hot) cudaFree(ix->hot);      // the previous region (dir.super pointed into it)
    ix->hot = region;
    ix->hot_bytes = total;
    ix->dir.super = (const uint64_t*) region;
    ix->ft = DevFtab{};
    ix->ft_host.clear();
    if (k) {
        ix->ft.range = (const ulonglong2*) ((char*) region + off_range);
        ix->ft.toe = with_toe ? (const uint64_t*) ((char*) region + off_toe) : nullptr;
        // ft.k is set by the caller once the table is filled
    }
    ix->info.ftab_k = 0;
    ix->info.ftab_bytes = 0;
    ix->info.hot_bytes = total;
    ix->info.l2_pinned_bytes = 0;
}

// RowBowt::build_ftab(k), include/rowbowt.hpp:726-743, as one kernel over all 4^k k-mers; with the
// toehold SA loaded the table also carries the toehold state after the k steps, so that
// find_range_w_toehold can be seeded the same way.
void build_ftab(rbg_index* ix, cudaStream_t st, uint32_t k) {
    if (k == 0) { rebuild_hot_region(ix, 0, false); return; }
    if (k > kFtabMaxK) throw std::invalid_argument("ftab k must be in [1, 13]");
    const bool with_toe = ix->info.has_sa;
    rebuild_hot_region(ix, k, with_toe);
    launch_ftab_build(ix->dir, k, with_toe, const_cast<ulonglong2*>(ix->ft.range), const_cast<uint64_t*>(ix->ft.toe), st);
    ix->ft_host.resize((size_t) 1 << (2 * k));
    CU(cudaMemcpyAsync(ix->ft_host.data(), ix->ft.range, ix->ft_host.size() * sizeof(ulonglong2), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    ix->ft.k = k;
    ix->info.ftab_k = k;
    ix->info.ftab_bytes = ix->ft_host.size() * (sizeof(ulonglong2) + (with_toe ? sizeof(uint64_t) : 0));
}

inline int base_code(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }

// key of a k-mer string in the table: base i -> bits 2i (the enumeration of build_ftab)
bool kmer_key(const char* s, uint32_t k, uint64_t& key) {
    key = 0;
    for (uint32_t i = 0; i < k; ++i) {
        const int c = base_code(s[i]);
        if (c < 0) return false;
        key |= (uint64_t) c << (2 * i);
    }
    return true;
}

// FTab::load, include/ftab.hpp:15-28: "<kmer> <lo> <hi>" per line; k = length of the last k-mer.
// The table is then REBUILT on the GPU for that k (the file has no toehold state) and every entry
// of the file is checked against it: an ftab that belongs to another index is an error here,
// where the reference would silently return wrong ranges.
void load_ftab(rbg_index* ix, cudaStream_t st, const std::string& path) {
    FILE* f = fopen(path.c_str(), "r");
    if (!f) throw io_error("bad file: " + path);
    struct Ent { std::string kmer; uint64_t lo, hi; };
    std::vector<Ent> ents;
    char buf[256];
    unsigned long long lo, hi;
    char km[64];
    while (fgets(buf, sizeof buf, f)) {
        if (sscanf(buf, "%63s %llu %llu", km, &lo, &hi) != 3) { fclose(f); throw format_error("ftab: malformed line in " + path); }
        ents.push_back({km, lo, hi});
    }
    fclose(f);
    const uint32_t k = ents.empty() ? 10u : (uint32_t) ents.back().kmer.size();      // FTab::k defaults to 10
    if (k == 0 || k > kFtabMaxK) throw format_error("ftab: unsupported k in " + path);
    build_ftab(ix, st, k);
    for (const Ent& e : ents) {
        uint64_t key;
        if (e.kmer.size() != k || !kmer_key(e.kmer.c_str(), k, key)) throw format_error("ftab: bad k-mer '" + e.kmer + "' in " + path);
        if (ix->ft_host[key].x != e.lo || ix->ft_host[key].y != e.hi)
            throw format_error("ftab: entry " + e.kmer + " does not match this index (" + path + ")");
    }
}

// FTab::serialize, include/ftab.hpp:30-34: std::map order (k-mers ascending as strings), present
// k-mers only, "<kmer> <lo> <hi>\n".
void save_ftab(const rbg_index* ix, const std::string& path) {
    if (!ix->ft.k) throw std::invalid_argument("no ftab to save");
    FILE* f = fopen(path.c_str(), "w");
    if (!f) throw io_error("cannot write " + path);
    const uint32_t k = ix->ft.k;
    const uint64_t total = 1ull << (2 * k);
    std::string kmer(k, 'A');
    for (uint64_t y = 0; y < total; ++y) {          // y = rank of the k-mer in string order: first base most significant
        uint64_t key = 0;
        for (uint32_t i = 0; i < k; ++i) {
            const uint32_t c = (uint32_t) (y >> (2 * (k - 1 - i))) & 3u;
            kmer[i] = "ACGT"[c];
            key |= (uint64_t) c << (2 * i);
        }
        const ulonglong2 e = ix->ft_host[key];
        if (e.x <= e.y) fprintf(f, "%s %llu %llu\n", kmer.c_str(), e.x, e.y);
    }
    if (fclose(f) != 0) throw io_error("cannot write " + path);
}

// ---- layout cache (RBG_LOAD_CACHE) --------------------------------------------------------------------------------
// Opening an index decodes the reference's serializations and re-lays them out for the GPU: ~1.3-2.2 s for the BASELINE
// index where the reference maps its files in 0.05-0.5 s.  With RBG_LOAD_CACHE the device arrays of the finished layout are
// written once to <prefix>.rbgcache and later opens upload them as they are.  The cache is valid only for exactly
// these index files (size + mtime of each part), these load flags, this library's layout version and the layout knobs the
// open read; anything else rebuilds and rewrites it.  The index files stay the source of truth.
constexpr uint64_t kCacheMagic = 0x3145484341434752ull;       // "RGCACHE1"
constexpr uint32_t kCacheVersion = 5;                         // bump when a device structure or its meaning changes

struct CacheHeader {
    uint64_t magic;
    uint32_t version, flags;
    uint64_t file_size[3], file_mtime_ns[3];                  // .rbwt, .tsa, .mab (0 when not loaded)
    uint32_t sizeof_dir, sizeof_toe, sizeof_phi, sizeof_mk, sizeof_info, sizeof_codes, sizeof_knobs;
    LayoutKnobs knobs;                                         // what the layout was built with
    uint32_t n_blobs;
    int32_t field_blob[15];                                    // which blob each device pointer of the structs refers to, -1 = null
};
static_assert(std::has_unique_object_representations_v<CacheHeader>, "headers are compared with memcmp: no padding");

CacheHeader cache_stamp(const std::string& pre, uint32_t flags, const LayoutKnobs& knobs) {
    CacheHeader h{};
    h.magic = kCacheMagic;
    h.version = kCacheVersion;
    h.flags = flags & (RBG_LOAD_SA | RBG_LOAD_MA | RBG_LOAD_FBB);
    const char* suf[3] = {".rbwt", ".tsa", ".mab"};
    const bool need[3] = {true, (flags & RBG_LOAD_SA) != 0, (flags & RBG_LOAD_MA) != 0};
    for (int i = 0; i < 3; ++i) {
        struct stat st;
        if (need[i] && stat((pre + suf[i]).c_str(), &st) == 0) {
            h.file_size[i] = (uint64_t) st.st_size;
            h.file_mtime_ns[i] = (uint64_t) st.st_mtim.tv_sec * 1000000000ull + (uint64_t) st.st_mtim.tv_nsec;
        }
    }
    h.sizeof_dir = sizeof(DevLeafDir); h.sizeof_toe = sizeof(DevToehold); h.sizeof_phi = sizeof(DevPhi);
    h.sizeof_mk = sizeof(DevMarkers); h.sizeof_info = sizeof(rbg_info); h.sizeof_codes = sizeof(CodeTable);
    h.sizeof_knobs = sizeof(LayoutKnobs);
    h.knobs = knobs;
    return h;
}

// the device pointers of the structs, in a fixed order
void cache_fields(rbg_index* ix, const void*** f) {
    int i = 0;
    f[i++] = (const void**) &ix->dir.lines;      f[i++] = (const void**) &ix->dir.super;
    f[i++] = (const void**) &ix->toe.table;      f[i++] = (const void**) &ix->toe.keys;
    f[i++] = (const void**) &ix->toe.sample_lo;  f[i++] = (const void**) &ix->toe.sample_hi;
    f[i++] = (const void**) &ix->phi.l1;         f[i++] = (const void**) &ix->phi.slots;
    f[i++] = (const void**) &ix->phi.ovf_keys;   f[i++] = (const void**) &ix->phi.ovf_prev_lo;
    f[i++] = (const void**) &ix->phi.ovf_prev_hi;
    f[i++] = (const void**) &ix->mk.starts;      f[i++] = (const void**) &ix->mk.ends;
    f[i++] = (const void**) &ix->mk.idxs;        f[i++] = (const void**) &ix->mk.arr;
}

// After open_from_arrays: dir.super already points into the hot region; its blob is the second upload (owned[1]).
void write_layout_cache(rbg_index* ix, const std::string& pre, uint32_t flags, const LayoutKnobs& knobs) {
    CacheHeader h = cache_stamp(pre, flags, knobs);
    if (ix->owned.size() < 2) return;
    const void** f[15];
    cache_fields(ix, f);
    for (int i = 0; i < 15; ++i) {
        h.field_blob[i] = -1;
        for (size_t b = 0; b < ix->owned.size(); ++b) if (*f[i] == ix->owned[b].mem.p) h.field_blob[i] = (int32_t) b;
    }
    h.field_blob[1] = 1;                                       // dir.super: the blob behind the hot region's copy
    h.n_blobs = (uint32_t) ix->owned.size();
    // rb_align --gpus N opens N handles of one prefix at the same time: one writer per process at a time, own temp file each
    static std::mutex write_mu;
    std::lock_guard<std::mutex> write_lock(write_mu);
    const std::string path = pre + ".rbgcache", tmp = path + ".tmp." + std::to_string((long) getpid()) + "." + std::to_string(ix->device);
    FILE* fp = fopen(tmp.c_str(), "wb");
    if (!fp) return;                                            // read-only index directory: no cache, no error
    bool ok = fwrite(&h, sizeof h, 1, fp) == 1;
    ok = ok && fwrite(&ix->dir, sizeof ix->dir, 1, fp) == 1 && fwrite(&ix->toe, sizeof ix->toe, 1, fp) == 1 &&
         fwrite(&ix->phi, sizeof ix->phi, 1, fp) == 1 && fwrite(&ix->mk, sizeof ix->mk, 1, fp) == 1 &&
         fwrite(&ix->codes, sizeof ix->codes, 1, fp) == 1 && fwrite(&ix->info, sizeof ix->info, 1, fp) == 1;
    try {
        std::vector<char> buf;
        for (size_t b = 0; ok && b < ix->owned.size(); ++b) {
            const uint64_t bytes = ix->owned[b].bytes;
            ok = fwrite(&bytes, 8, 1, fp) == 1;
            if (!bytes) continue;
            buf.resize(bytes);
            CU(cudaMemcpy(buf.data(), ix->owned[b].mem.p, bytes, cudaMemcpyDeviceToHost));
            ok = ok && fwrite(buf.data(), 1, bytes, fp) == bytes;
        }
    } catch (...) {
        fclose(fp);
        remove(tmp.c_str());
        throw;
    }
    ok = (fclose(fp) == 0) && ok;
    if (ok) ok = rename(tmp.c_str(), path.c_str()) == 0;
    if (!ok) remove(tmp.c_str());
}

// A handle on `device` (after the device checks) that answers queries with RBG_LANES lanes at most.
std::unique_ptr<rbg_index> new_index(int device) {
    select_device(device);
    std::unique_ptr<rbg_index> ix(new rbg_index);
    ix->device = device;
    ix->max_lanes = knob_lanes();
    return ix;
}

// nullptr when there is no valid cache for (prefix, flags)
std::unique_ptr<rbg_index> open_layout_cache(const std::string& pre, uint32_t flags, int device, const LayoutKnobs& knobs) {
    const std::string path = pre + ".rbgcache";
    const int fd = open(path.c_str(), O_RDONLY);
    if (fd < 0) return nullptr;
    struct stat st;
    if (fstat(fd, &st) != 0 || (size_t) st.st_size < sizeof(CacheHeader)) { close(fd); return nullptr; }
    const size_t size = (size_t) st.st_size;
    const char* m = (const char*) mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
    close(fd);
    if (m == MAP_FAILED) return nullptr;
    struct Unmap { const char* p; size_t n; ~Unmap() { munmap((void*) p, n); } } unmap{m, size};
    CacheHeader h;
    memcpy(&h, m, sizeof h);
    CacheHeader want = cache_stamp(pre, flags, knobs);
    want.n_blobs = h.n_blobs;
    memcpy(want.field_blob, h.field_blob, sizeof want.field_blob);
    if (memcmp(&h, &want, sizeof h) != 0) return nullptr;      // other files, flags, library version or knobs
    size_t at = sizeof h;
    const size_t pods = sizeof(DevLeafDir) + sizeof(DevToehold) + sizeof(DevPhi) + sizeof(DevMarkers) + sizeof(CodeTable) + sizeof(rbg_info);
    if (at + pods > size || h.n_blobs < 2 || h.n_blobs > 64) return nullptr;
    std::unique_ptr<rbg_index> ix = new_index(device);
    memcpy(&ix->dir, m + at, sizeof ix->dir); at += sizeof ix->dir;
    memcpy(&ix->toe, m + at, sizeof ix->toe); at += sizeof ix->toe;
    memcpy(&ix->phi, m + at, sizeof ix->phi); at += sizeof ix->phi;
    memcpy(&ix->mk, m + at, sizeof ix->mk); at += sizeof ix->mk;
    memcpy(&ix->codes, m + at, sizeof ix->codes); at += sizeof ix->codes;
    memcpy(&ix->info, m + at, sizeof ix->info); at += sizeof ix->info;
    for (uint32_t b = 0; b < h.n_blobs; ++b) {
        if (at + 8 > size) return nullptr;
        uint64_t bytes;
        memcpy(&bytes, m + at, 8);
        at += 8;
        if (bytes > size - at) return nullptr;                 // truncated file
        ix->owned.push_back(Upload{DevBuf(std::max<size_t>(bytes, 64)), bytes});
        if (bytes) CU(cudaMemcpy(ix->owned.back().mem.p, m + at, bytes, cudaMemcpyHostToDevice));
        at += bytes;
    }
    const void** f[15];
    cache_fields(ix.get(), f);
    for (int i = 0; i < 15; ++i) {
        if (h.field_blob[i] >= (int32_t) h.n_blobs) return nullptr;
        *f[i] = h.field_blob[i] < 0 ? nullptr : ix->owned[h.field_blob[i]].mem.p;
    }
    ix->hot = nullptr;
    CU(cudaDeviceSynchronize());
    rebuild_hot_region(ix.get(), 0, false);                    // superblock counts into the hot region, no seed table yet
    ix->info.from_cache = 1;
    ix->info.pair_bytes = 0;                                   // not rebuilt from a cache: the count search steps base by base
    ix->info.pair_window = 0;
    return ix;
}

// The pair directory, when the count search gains from it: a layout-5 index with n < 2^32 whose pair directory stays
// within kPairBudget -- small enough to stay resident in L2 beside the single-base directory, where the search is bound by
// instructions and two bases per step take fewer of them than two steps -- and whose superblock table fits shared memory.
// Larger indexes are bound by their line gathers, which the pair directory would only multiply.  knobs.pair = 0|1 (tests)
// forces either form; 1 still needs layout 5, n < 2^32 and the shared-memory table.  Every index small enough for it opens
// in layout 7 unless a layout is forced (RBG_PAIR=1 asks for layout 5, LayoutKnobs::leaf_layout), so automatically it is
// built only under RBG_LAYOUT=5.
constexpr uint64_t kPairBudget = 64ull << 20;
void build_pair(rbg_index* ix, const RunsBwt& bwt, const LeafDir& ld, const LayoutKnobs& knobs) {
    const int force = knobs.pair;
    if (force == 0 || ld.version != 5 || (bwt.n >> 32)) return;
    // a line holds at most 12 runs of P, and P has at least as many runs as the BWT: skip what cannot fit without building it
    if (force != 1 && bwt.R * 64 / LeafFmt<6>::E > kPairBudget) return;
    PairDir pd = build_pair_dir(bwt, ld, knobs.pair_window);
    if (64 * pd.n_super > kPairMaxShared || (force != 1 && pd.bytes() > kPairBudget)) return;
    size_t acc = 0;
    DevPairDir& P = ix->pair;
    P.lines = upload(pd.lines, ix->pair_owned, &acc);
    P.super = upload(pd.super, ix->pair_owned, &acc);
    P.n_super = (uint32_t) pd.n_super;
    P.window = pd.window;
    P.sb_shift = pd.sb_shift;
    DevLeafDir div{};
    div.window = pd.window;
    div.n = pd.n;
    set_fast_div(div);
    if (!div.div_fast) throw std::logic_error("pair directory: no 32-bit division");
    P.div_k = div.div_k;
    P.div_mul = div.div_mul;
    P.div_s = div.div_s;
    P.n_child = (pd.window + kPairRawSymbols - 1) / kPairRawSymbols;
    P.n_bad = pd.n_bad;
    for (int t = 0; t < kPairMaxBad; ++t) P.bad_pos[t] = pd.bad_pos[t];
    ix->info.pair_bytes = acc;
    ix->info.pair_window = pd.window;
}

std::unique_ptr<rbg_index> open_from_arrays(const RunsBwt& bwt, const ToeholdArrays* tsa, const MarkerArrays* ma, int device,
                                            const LayoutKnobs& knobs) {
    std::unique_ptr<rbg_index> ix = new_index(device);

    // caller-supplied arrays (rbg_index_open_arrays) and raw builds come here without passing a file reader
    validate_runs(bwt, "the BWT runs");
    if (tsa) validate_toehold(*tsa, "the toehold arrays");
    if (ma) validate_markers(*ma, "the marker arrays");
    rbg_info& info = ix->info;
    info.n = bwt.n;
    info.r = bwt.R;
    uint64_t F[256];
    size_t acc = 0;
    // the phi directory depends on the toehold arrays only: built on another host thread while this one lays out the BWT
    std::future<PhiDir> phi_job;
    if (tsa) {
        const uint64_t budget = phi_slot_budget();
        phi_job = std::async(std::launch::async, [tsa, budget, knobs] { return build_phi_dir(*tsa, knobs.phi_shift, knobs.phi_parts, budget); });
    }
    {
        LeafDir ld = build_leaf_dir(bwt, knobs.window, knobs.leaf_layout());
        memcpy(F, ld.F, sizeof F);
        info.window = ld.window;
        info.layout = (uint32_t) ld.version;
        info.n_lines = ld.n_lines();
        info.n_cluster = ld.n_cluster;
        ix->dir.lines = upload(ld.lines, ix->owned, &acc);
        ix->dir.super = upload(ld.super, ix->owned, &acc);
        info.dir_bytes = acc;
        ix->dir.n = ld.n;
        ix->dir.magic = ld.magic;
        ix->dir.n_super = ld.n_super;
        ix->dir.window = ld.window;
        ix->dir.sb_shift = ld.sb_shift;
        ix->dir.version = (uint32_t) ld.version;
        ix->dir.n_term = ld.n_term;
        set_fast_div(ix->dir);
        for (int t = 0; t < kMaxTerm; ++t) ix->dir.term_pos[t] = ld.term_pos[t];
        memcpy(ix->codes.code_of, ld.code_of, 256);
        build_pair(ix.get(), bwt, ld, knobs);
    }
    memcpy(info.F, F, sizeof info.F);

    if (tsa) {
        ToeholdDir td = build_toehold_dir(bwt, F, *tsa, knobs.toehold_shift);
        acc = 0;
        ix->toe.table = upload(td.table, ix->owned, &acc);
        ix->toe.keys = upload(td.keys, ix->owned, &acc);
        ix->toe.sample_lo = upload(td.sample.lo, ix->owned, &acc);
        ix->toe.sample_hi = td.sample.wide ? upload(td.sample.hi, ix->owned, &acc) : nullptr;
        ix->toe.shift = td.shift;
        ix->toe.key_bytes = td.key_bytes;
        ix->toe.toehold0 = td.toehold0;
        info.toehold_bytes = acc;
        info.toehold0 = td.toehold0;
        PhiDir pd = phi_job.get();
        acc = 0;
        ix->phi = upload_phi(pd, tsa->n, ix->owned, &acc);
        info.phi_shift = pd.shift;
        info.phi_overflow = pd.n_overflow;
        info.phi_bytes = acc;
        info.has_sa = 1;
    }
    if (ma) {
        acc = 0;
        ix->mk.starts = upload(ma->starts, ix->owned, &acc);
        ix->mk.ends = upload(ma->ends, ix->owned, &acc);
        ix->mk.idxs = upload(ma->idxs, ix->owned, &acc);
        ix->mk.arr = upload(ma->arr, ix->owned, &acc);
        ix->mk.n_starts = ma->starts.size();
        ix->mk.n_ends = ma->ends.size();
        ix->mk.n_idxs = ma->idxs.size();
        ix->mk.size_starts = ma->size_starts;
        ix->mk.size_ends = ma->size_ends;
        ix->mk.size_idxs = ma->size_idxs;
        info.marker_bytes = acc;
        info.has_ma = 1;
        info.wsize = ma->wsize;
    }
    CU(cudaDeviceSynchronize());
    rebuild_hot_region(ix.get(), 0, false);
    return ix;
}

template <class Fn>
int guarded(Fn&& fn) {
    try {
        return fn();
    } catch (const io_error& e) { return fail(RBG_E_IO, e.what());
    } catch (const format_error& e) { return fail(RBG_E_FORMAT, e.what());
    } catch (const alphabet_error& e) { return fail(RBG_E_ALPHABET, e.what());
    } catch (const cuda_error& e) { cudaGetLastError(); return fail(RBG_E_CUDA, e.what());
    } catch (const nomem_error& e) { return fail(RBG_E_NOMEM, e.what());
    } catch (const internal_error& e) { return fail(RBG_E_INTERNAL, e.what());
    } catch (const std::bad_alloc&) { return fail(RBG_E_NOMEM, "out of host memory");
    } catch (const std::exception& e) { return fail(RBG_E_ARG, e.what()); }
}

// What a query call was handed: raw bytes (rbg_batch) or the 2-bit stream packed on the host (rbg_packed_batch).
struct BatchIn {
    uint64_t n = 0;
    const uint64_t* offsets = nullptr;
    const char* bases = nullptr;
    const uint64_t* packed = nullptr;    // non-null: packed input
    const uint8_t* flags = nullptr;
    uint64_t n_exotic = 0;
    bool is_packed() const { return packed != nullptr; }
    static BatchIn raw(const rbg_batch* in) {
        BatchIn b;
        b.n = in->n_reads;
        b.offsets = in->offsets;
        b.bases = in->bases;
        return b;
    }
    static BatchIn from_packed(const rbg_packed_batch* in) {
        BatchIn b;
        b.n = in->n_reads;
        b.offsets = in->offsets;
        b.bases = in->bases;
        b.packed = in->packed;
        b.flags = in->flags;
        b.n_exotic = in->flags ? in->n_exotic : 0;
        return b;
    }
};

int check_packed(const rbg_packed_batch* in) {
    if (in->n_reads && (!in->offsets || !in->packed)) return fail(RBG_E_ARG, "packed batch without packed/offsets");
    if (in->n_reads && in->offsets[0] != 0) return fail(RBG_E_ARG, "packed batch: offsets[0] must be 0");
    if (in->flags && in->n_exotic && !in->bases) return fail(RBG_E_ARG, "packed batch: reads flagged RBG_READ_EXOTIC need `bases`");
    return RBG_OK;
}

// Device buffers for a batch of n reads / n_bytes bases.
void reserve_input(rbg_reads* rd, rbg_index* ix, uint64_t n, uint64_t n_bytes, bool with_bases) {
    rd->ix = ix;
    rd->n_reads = n;
    rd->n_bytes = n_bytes;
    rd->ran = false;
    rd->prepacked = false;
    rd->has_bases = with_bases;
    if (with_bases) reserve(rd->bases, n_bytes + 64);
    reserve(rd->offs, (n + 1) * 8);
    reserve(rd->packed, ((n_bytes + 31) / 32 + 1) * 8);
    reserve(rd->flags, n + 8);
}

// Raw bytes of the reads flagged RBG_READ_EXOTIC among [r0, r1) of a packed batch (normally none).
void copy_exotic_bases(const BatchIn& in, rbg_reads* rd, uint64_t r0, uint64_t r1, cudaStream_t st) {
    if (!in.n_exotic) return;
    for (uint64_t i = r0; i < r1; ++i)
        if (in.flags[i] & RBG_READ_EXOTIC) {
            const uint64_t a = in.offsets[i], z = in.offsets[i + 1];
            if (z > a) CU(cudaMemcpyAsync(rd->bases.as<uint8_t>() + a, in.bases + a, z - a, cudaMemcpyHostToDevice, st));
        }
}

// The batch's offsets re-based so that offs[0] == 0: the caller's own array when they already are, else a copy in `tmp`.
const uint64_t* rebased_offsets(const BatchIn& in, std::vector<uint64_t>& tmp) {
    const uint64_t base = in.n ? in.offsets[0] : 0;
    if (base == 0) return in.offsets;
    tmp.resize(in.n + 1);
    for (uint64_t i = 0; i <= in.n; ++i) tmp[i] = in.offsets[i] - base;
    return tmp.data();
}

// H2D of one whole batch into `rd` (raw: bases re-based so that offs[0] == 0; packed: words + flags as given).
void stage_batch(rbg_index* ix, cudaStream_t st, const BatchIn& in, rbg_reads* rd) {
    const uint64_t n = in.n;
    const uint64_t base = n ? in.offsets[0] : 0;
    const uint64_t n_bytes = n ? in.offsets[n] - base : 0;
    reserve_input(rd, ix, n, n_bytes, !in.is_packed() || in.n_exotic);
    if (in.is_packed()) {
        rd->prepacked = true;
        if (n) CU(cudaMemcpyAsync(rd->offs.p, in.offsets, (n + 1) * 8, cudaMemcpyHostToDevice, st));
        if (n_bytes) CU(cudaMemcpyAsync(rd->packed.p, in.packed, ((n_bytes + 31) / 32) * 8, cudaMemcpyHostToDevice, st));
        if (in.flags && n) CU(cudaMemcpyAsync(rd->flags.p, in.flags, n, cudaMemcpyHostToDevice, st));
        else CU(cudaMemsetAsync(rd->flags.p, 0, n + 4, st));
        copy_exotic_bases(in, rd, 0, n, st);
        return;
    }
    if (n_bytes) CU(cudaMemcpyAsync(rd->bases.p, in.bases + base, n_bytes, cudaMemcpyHostToDevice, st));
    std::vector<uint64_t> tmp;
    CU(cudaMemcpyAsync(rd->offs.p, rebased_offsets(in, tmp), (n + 1) * 8, cudaMemcpyHostToDevice, st));
    if (!tmp.empty()) CU(cudaStreamSynchronize(st));      // the copy reads `tmp`
}

float ev_ms(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

struct Views { DevBatch b; DevResult r; };

// Result buffers of the fixed-size part and the kernel-side views of `rd`.
Views prepare(rbg_index* ix, rbg_reads* rd, uint32_t mode) {
    const bool locate = mode & RBG_LOCATE, markers = mode & RBG_MARKERS;
    if (locate && !ix->info.has_sa) throw std::invalid_argument("RBG_LOCATE needs an index opened with RBG_LOAD_SA");
    if (markers && !ix->info.has_ma) throw std::invalid_argument("RBG_MARKERS needs an index opened with RBG_LOAD_MA");
    const uint64_t n = rd->n_reads;
    reserve(rd->lo, (n + 1) * 8);
    reserve(rd->hi, (n + 1) * 8);
    if (locate) {
        reserve(rd->toehold, (n + 1) * 8);
        reserve(rd->loc_cnt, (n + 2) * 8);
        reserve(rd->loc_off, (n + 2) * 8);
    }
    if (markers) {
        reserve(rd->mk_cnt, (n + 2) * 8);
        reserve(rd->mk_off, (n + 2) * 8);
        reserve(rd->mk_first, (n + 1) * 8);
    }
    if (locate || markers) reserve(rd->scan_tmp, std::max(scan_tmp_bytes(n + 1), scan_from_tmp_bytes(n + 1)));
    Views v{};
    v.b = DevBatch{rd->bases.as<uint8_t>(), rd->offs.as<uint64_t>(), n, rd->n_bytes, 0, n, rd->packed.as<uint64_t>(), rd->flags.as<uint8_t>()};
    v.r.lo = rd->lo.as<uint64_t>();
    v.r.hi = rd->hi.as<uint64_t>();
    v.r.toehold = rd->toehold.as<uint64_t>();
    v.r.loc_cnt = rd->loc_cnt.as<uint64_t>();
    v.r.loc_off = rd->loc_off.as<uint64_t>();
    v.r.mk_cnt = rd->mk_cnt.as<uint64_t>();
    v.r.mk_off = rd->mk_off.as<uint64_t>();
    v.r.mk_first = rd->mk_first.as<uint64_t>();
    v.r.markers = rd->markers.as<uint64_t>();
    return v;
}

// How locations leave the device: u64 each, or with RBG_NARROW_LOCS a u32 plane plus, when n > 2^32, a u8 plane.
struct LocForm {
    bool narrow, hi_plane;
    LocForm(uint32_t mode, uint64_t n) : narrow((mode & RBG_LOCATE) && (mode & RBG_NARROW_LOCS)), hi_plane(narrow && (n >> 32)) {}
    size_t item() const { return narrow ? 4 : 8; }
};

// Location planes of `rd` into the kernel view.
void point_locs(const rbg_reads* rd, DevResult& r, LocForm f) {
    r.locs = f.narrow ? nullptr : rd->locs.as<uint64_t>();
    r.locs_lo = f.narrow ? rd->locs.as<uint32_t>() : nullptr;
    r.locs_hi = f.hi_plane ? rd->locs_hi.as<uint8_t>() : nullptr;
}

// Location planes of `h` into the caller's result.
void point_locs(const HostResult* h, rbg_result* out, LocForm f) {
    out->locs = f.narrow ? nullptr : h->locs.as<uint64_t>();
    out->locs_lo32 = f.narrow ? h->locs.as<uint32_t>() : nullptr;
    out->locs_hi8 = f.hi_plane ? h->locs_hi.as<uint8_t>() : nullptr;
}

// Occurrence / marker-word counts of every read -> offsets; returns the total (one host sync).
uint64_t scan_counts(Lane& L, rbg_reads* rd, uint64_t* cnt, uint64_t* off, uint64_t n, cudaStream_t st) {
    CU(cudaMemsetAsync(cnt + n, 0, 8, st));
    launch_scan(cnt, off, n, rd->scan_tmp.p, rd->scan_tmp.cap, st);
    CU(cudaMemcpyAsync(&L.h_ctr->checksum, off + n, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return L.h_ctr->checksum;
}

void collect_counters(Lane& L, rbg_stats& s, rbg_reads* rd, uint32_t launches) {
    s.reads = rd->n_reads;
    s.bases = rd->n_bytes;
    s.lf_steps = L.h_ctr->lf_steps;
    s.lf_lines = L.h_ctr->lf_lines;
    s.phi_steps = L.h_ctr->phi_steps;
    s.marker_words = L.h_ctr->marker_words;
    s.launches = launches;
}

// All kernels of one query over a staged batch, one launch per stage (the kernel-only measurement
// path).  Leaves results on the device.
void run_staged(rbg_index* ix, Lane& L, rbg_stats& s, rbg_reads* rd, uint32_t mode, uint64_t max_hits, bool want_checksum) {
    const bool locate = mode & RBG_LOCATE, markers = mode & RBG_MARKERS;
    const QueryKnobs knobs = query_knobs(Lane::kMaxChunks);
    const LocForm lf(mode, ix->info.n);
    Views v = prepare(ix, rd, mode);
    DevBatch& b = v.b;
    DevResult& r = v.r;
    const uint64_t n = rd->n_reads;
    cudaStream_t st = L.stream;
    uint32_t launches = 0;
    CU(cudaMemsetAsync(L.d_ctr, 0, sizeof(DevCounters), st));
    CU(cudaEventRecord(L.ev[0], st));
    if (!rd->prepacked) {
        CU(cudaMemsetAsync(b.flags, 0, n + 4, st));
        launches += launch_pack(b, ix->codes, rd->n_bytes, st);
    }
    CU(cudaEventRecord(L.ev[1], st));
    launches += launch_search(ix->dir, ix->pair, locate ? &ix->toe : nullptr, ix->ft, b, r, L.d_ctr, &L.d_ctr->cursor[0], st);
    if (rd->has_bases) launches += launch_search_bytes(ix->dir, locate ? &ix->toe : nullptr, b, r, ix->codes, L.d_ctr, st);
    CU(cudaEventRecord(L.ev[2], st));
    rd->n_locs = rd->n_markers = 0;
    if (locate) {
        launches += launch_locate_counts(r, 0, n, max_hits, st);
        rd->n_locs = scan_counts(L, rd, r.loc_cnt, r.loc_off, n, st);
        launches += 1;
        reserve(rd->locs, (rd->n_locs + 1) * lf.item());
        if (lf.hi_plane) reserve(rd->locs_hi, rd->n_locs + 8);
        point_locs(rd, r, lf);
        CU(cudaEventRecord(L.ev[6], st));
        launches += launch_locate(ix->phi, r, 0, n, rd->n_locs, knobs.loc_draw, L.d_ctr, &L.d_ctr->loc_cursor[0], st);
    }
    CU(cudaEventRecord(L.ev[3], st));
    if (markers) {
        launches += launch_marker_counts(ix->mk, r, 0, n, st);
        rd->n_markers = scan_counts(L, rd, r.mk_cnt, r.mk_off, n, st);
        launches += 1;
        reserve(rd->markers, (rd->n_markers + 1) * 8);
        r.markers = rd->markers.as<uint64_t>();
        launches += launch_marker_gather(ix->mk, r, 0, n, L.d_ctr, st);
    }
    CU(cudaEventRecord(L.ev[4], st));
    if (want_checksum) launches += launch_checksum(r, n, locate, locate, markers, L.d_ctr, st);
    CU(cudaMemcpyAsync(L.h_ctr, L.d_ctr, sizeof(DevCounters), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(L.ev[5], st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    collect_counters(L, s, rd, launches);
    s.ms_pack = ev_ms(L.ev[0], L.ev[1]);
    s.ms_search = ev_ms(L.ev[1], L.ev[2]);
    s.ms_toehold = 0;
    s.ms_locate = ev_ms(L.ev[2], L.ev[3]);
    s.ms_phi = locate ? ev_ms(L.ev[6], L.ev[3]) : 0;
    s.ms_markers = ev_ms(L.ev[3], L.ev[4]);
    s.ms_h2d = s.ms_d2h = 0;
    s.ms_total = ev_ms(L.ev[0], L.ev[5]);
    rd->last_mode = mode;
    rd->ran = true;
}

// D2H of a staged run's results into pinned buffers.
void fetch_staged(rbg_index* ix, Lane& L, rbg_reads* rd, uint32_t mode, rbg_result* out) {
    if (!rd->ran) throw std::invalid_argument("no staged run to fetch");
    const LocForm lf(rd->last_mode, ix->info.n);
    mode = rd->last_mode & mode;
    const uint64_t n = rd->n_reads;
    cudaStream_t st = L.stream;
    HostResult* h = ix->results.take(ix);
    memset(out, 0, sizeof *out);
    out->_owner = h;
    out->n_reads = n;
    reserve(h->lo, (n + 1) * 8);
    reserve(h->hi, (n + 1) * 8);
    CU(cudaMemcpyAsync(h->lo.p, rd->lo.p, n * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h->hi.p, rd->hi.p, n * 8, cudaMemcpyDeviceToHost, st));
    out->lo = (uint64_t*) h->lo.p;
    out->hi = (uint64_t*) h->hi.p;
    if (mode & RBG_LOCATE) {
        reserve(h->toehold, (n + 1) * 8);
        reserve(h->loc_off, (n + 2) * 8);
        reserve(h->locs, (rd->n_locs + 1) * lf.item());
        if (lf.hi_plane) reserve(h->locs_hi, rd->n_locs + 8);
        CU(cudaMemcpyAsync(h->toehold.p, rd->toehold.p, n * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(h->loc_off.p, rd->loc_off.p, (n + 1) * 8, cudaMemcpyDeviceToHost, st));
        if (rd->n_locs) CU(cudaMemcpyAsync(h->locs.p, rd->locs.p, rd->n_locs * lf.item(), cudaMemcpyDeviceToHost, st));
        if (lf.hi_plane && rd->n_locs) CU(cudaMemcpyAsync(h->locs_hi.p, rd->locs_hi.p, rd->n_locs, cudaMemcpyDeviceToHost, st));
        out->toehold = (uint64_t*) h->toehold.p;
        out->loc_off = (uint64_t*) h->loc_off.p;
        point_locs(h, out, lf);
    }
    if (mode & RBG_MARKERS) {
        reserve(h->mk_off, (n + 2) * 8);
        reserve(h->markers, (rd->n_markers + 1) * 8);
        CU(cudaMemcpyAsync(h->mk_off.p, rd->mk_off.p, (n + 1) * 8, cudaMemcpyDeviceToHost, st));
        if (rd->n_markers) CU(cudaMemcpyAsync(h->markers.p, rd->markers.p, rd->n_markers * 8, cudaMemcpyDeviceToHost, st));
        out->mk_off = (uint64_t*) h->mk_off.p;
        out->markers = (uint64_t*) h->markers.p;
    }
    CU(cudaStreamSynchronize(st));
}


// rbg_query / rbg_query_packed: the batch is cut into chunks of reads and the three engines are kept busy at once --
// H2D of chunk c+1 (s_in), pack + search of chunk c (stream), D2H of chunk c-1's ranges (s_out).  A packed batch
// skips pack_kernel: its words and flags are copied as they are.
// Locate / marker output sizes are data dependent: see the comments at the locate and marker stages below.
void run_pipelined(rbg_index* ix, Lane& L, rbg_stats& s, const BatchIn& in, uint32_t mode, uint64_t max_hits, rbg_result* out) {
    const bool locate = mode & RBG_LOCATE, markers = mode & RBG_MARKERS;
    const QueryKnobs knobs = query_knobs(Lane::kMaxChunks);
    const LocForm lf(mode, ix->info.n);
    const size_t loc_item = lf.item();
    const bool narrow_rg = (mode & RBG_NARROW_RANGES) && !(ix->info.n >> 32);       // u32 planes of lo / hi on the wire
    rbg_reads* rd = &L.scratch;
    const uint64_t n = in.n;
    const uint64_t base = n ? in.offsets[0] : 0;
    const uint64_t n_bytes = n ? in.offsets[n] - base : 0;
    const bool packed_in = in.is_packed();
    reserve_input(rd, ix, n, n_bytes, !packed_in || in.n_exotic);
    rd->prepacked = packed_in;
    Views v = prepare(ix, rd, mode);
    DevBatch b = v.b;
    DevResult r = v.r;
    cudaStream_t sc = L.stream, si = L.s_in, so = L.s_out;

    HostResult* h = ix->results.take(ix);
    memset(out, 0, sizeof *out);
    out->_owner = h;
    out->n_reads = n;
    reserve(h->lo, (n + 1) * 8);
    reserve(h->hi, (n + 1) * 8);
    if (narrow_rg) {
        out->lo32 = (uint32_t*) h->lo.p;
        out->hi32 = (uint32_t*) h->hi.p;
        reserve(rd->lo32, (n + 1) * 4);
        reserve(rd->hi32, (n + 1) * 4);
    } else {
        out->lo = (uint64_t*) h->lo.p;
        out->hi = (uint64_t*) h->hi.p;
    }
    if (locate) {
        reserve(h->toehold, (n + 1) * 8);
        reserve(h->loc_off, (n + 2) * 8);
        out->toehold = (uint64_t*) h->toehold.p;
        out->loc_off = (uint64_t*) h->loc_off.p;
    }
    if (markers) {
        reserve(h->mk_off, (n + 2) * 8);
        out->mk_off = (uint64_t*) h->mk_off.p;
    }

    // chunking: about 16 chunks, at least 64 K reads each
    int n_chunks = knobs.chunks ? knobs.chunks : (int) std::min<uint64_t>(16, std::max<uint64_t>(1, n >> 16));
    if ((uint64_t) n_chunks > n) n_chunks = n ? (int) n : 1;
    auto cut = [&](int c) { return (uint64_t) ((__uint128_t) n * (uint64_t) c / (uint64_t) n_chunks); };

    uint32_t launches = 0;
    CU(cudaEventRecord(L.ev_span[0], si));
    // offsets first (pack's flagging searches them), re-based to 0 when the caller's are not
    std::vector<uint64_t> rebased;
    const uint64_t* offs_h = rebased_offsets(in, rebased);
    if (n) CU(cudaMemcpyAsync(rd->offs.p, offs_h, (n + 1) * 8, cudaMemcpyHostToDevice, si));
    CU(cudaMemsetAsync(L.d_ctr, 0, sizeof(DevCounters), sc));
    if (!packed_in || !in.flags) CU(cudaMemsetAsync(b.flags, 0, n + 4, sc));
    CU(cudaEventRecord(L.ev_span[2], sc));
    // Locations (-s) flow through the same pipeline: chunk c's counts are scanned on the device right after its
    // search, continuing from the running total chunk c-1 left in loc_off[r0] (no host round trip), and only the
    // 8-byte total comes back.  Once the host knows it (one chunk later, so the GPU queue never drains) it sizes the
    // buffers, launches the phi kernel of that chunk and queues the D2H of its locations behind it -- the locations
    // of the BASELINE batch (565 M: 2.3 GB narrow, 4.5 GB as u64) leave the device while later chunks are searched.
    PinnedBuf& loc_h = h->locs;
    PinnedBuf& loc_hi_h = h->locs_hi;
    DevBuf& loc_d = rd->locs;
    DevBuf& loc_hi_d = rd->locs_hi;
    uint64_t loc_done = 0;                                        // locations whose D2H has been queued
    auto grow_dev = [&](DevBuf& d, size_t want, size_t keep) {
        if (want <= d.cap) return;
        CU(cudaStreamSynchronize(sc));                             // phi kernels write the old buffer
        CU(cudaStreamSynchronize(so));                             // ... and copies read it
        DevBuf bigger;
        reserve(bigger, want + want / 4);
        if (keep) CU(cudaMemcpy(bigger.p, d.p, keep, cudaMemcpyDeviceToDevice));
        d = std::move(bigger);
    };
    auto grow_host = [&](PinnedBuf& hb, size_t want, size_t keep) {
        if (want <= hb.cap) return;
        CU(cudaStreamSynchronize(so));                             // copies in flight target the old buffer
        PinnedBuf bigger;
        reserve(bigger, want + want / 4);
        if (keep) memcpy(bigger.p, hb.p, keep);
        hb = std::move(bigger);
    };
    auto grow_locs = [&](uint64_t want_items) {                    // keeps [0, loc_done) on both sides
        grow_dev(loc_d, (size_t) (want_items + 1) * loc_item, loc_done * loc_item);
        grow_host(loc_h, (size_t) (want_items + 1) * loc_item, loc_done * loc_item);
        if (lf.hi_plane) {
            grow_dev(loc_hi_d, (size_t) want_items + 8, loc_done);
            grow_host(loc_hi_h, (size_t) want_items + 8, loc_done);
        }
        point_locs(rd, r, lf);
        point_locs(h, out, lf);
    };
    auto locate_chunk = [&](int c) {
        const uint64_t r0 = cut(c), r1 = cut(c + 1);
        CU(cudaEventSynchronize(L.ev_tot[c]));
        const uint64_t begin = c ? L.h_tot[c - 1] : 0, end = L.h_tot[c];
        // first sizing: extrapolate from the chunks seen so far; later chunks only grow it when the guess was short
        uint64_t want = end;
        if (r1 < n && end > 0) want = std::max<uint64_t>(end, (uint64_t) ((double) end / (double) r1 * (double) n * 1.08) + 4096);
        if (knobs.loc_est >= 0) want = std::max<uint64_t>(end, (uint64_t) knobs.loc_est);      // tests: force regrowth
        grow_locs(want);
        launches += launch_locate(ix->phi, r, r0, r1, end - begin, knobs.loc_draw, L.d_ctr, &L.d_ctr->loc_cursor[c], sc);
        CU(cudaEventRecord(L.ev_loc[c], sc));
        CU(cudaStreamWaitEvent(so, L.ev_loc[c], 0));
        CU(cudaMemcpyAsync(out->loc_off + r0, r.loc_off + r0, (r1 - r0 + 1) * 8, cudaMemcpyDeviceToHost, so));
        if (end > begin) {
            CU(cudaMemcpyAsync((char*) loc_h.p + begin * loc_item, (const char*) loc_d.p + begin * loc_item, (end - begin) * loc_item,
                               cudaMemcpyDeviceToHost, so));
            if (lf.hi_plane) CU(cudaMemcpyAsync((char*) loc_hi_h.p + begin, (const char*) loc_hi_d.p + begin, end - begin, cudaMemcpyDeviceToHost, so));
        }
        loc_done = end;
    };
    if (locate && n) CU(cudaMemsetAsync(r.loc_off, 0, 8, sc));
    for (int c = 0; c < n_chunks && n; ++c) {
        const uint64_t r0 = cut(c), r1 = cut(c + 1);
        const uint64_t b0 = offs_h[r0], b1 = offs_h[r1];
        if (packed_in) {
            // whole words; the word a chunk boundary falls into travels with the earlier chunk
            const uint64_t w0 = c ? (b0 + 31) >> 5 : 0, w1 = (b1 + 31) >> 5;
            if (w1 > w0) CU(cudaMemcpyAsync(rd->packed.as<uint64_t>() + w0, in.packed + w0, (w1 - w0) * 8, cudaMemcpyHostToDevice, si));
            if (in.flags) CU(cudaMemcpyAsync(rd->flags.as<uint8_t>() + r0, in.flags + r0, r1 - r0, cudaMemcpyHostToDevice, si));
            copy_exotic_bases(in, rd, r0, r1, si);
        } else if (b1 > b0) {
            CU(cudaMemcpyAsync(rd->bases.as<uint8_t>() + b0, in.bases + base + b0, b1 - b0, cudaMemcpyHostToDevice, si));
        }
        CU(cudaEventRecord(L.ev_in[c], si));
        // pack + search of consecutive chunks alternate between two streams, so that the next chunk's CTAs take the SMs
        // the tail of this one leaves idle (16 launches per batch: their tails were ~8 % of the end-to-end step)
        cudaStream_t ss = L.s_srch[c & 1];
        if (c < 2) CU(cudaStreamWaitEvent(ss, L.ev_span[2], 0));                     // counters and flags are zeroed on sc
        CU(cudaStreamWaitEvent(ss, L.ev_in[c], 0));
        b.r0 = r0;
        b.r1 = r1;
        if (!packed_in) {
            // The 2-bit word a chunk boundary falls into is written by BOTH chunks' pack kernels: incomplete by the earlier chunk
            // (the later chunk's bytes may not have arrived), complete by the later one.  The packs must therefore run in chunk
            // order even though consecutive chunks sit on different streams -- otherwise the earlier chunk's incomplete word
            // can land on top of the complete one while the later chunk is still searching (found by a parity failure under
            // compute-sanitizer's timing; RBG_TEST_STALL reproduces the order).  A search reading the word while the next
            // chunk's pack rewrites it sees the same bits for its own bases either way.
            if (knobs.stall_ns[0] && !(c & 1)) launch_stall(knobs.stall_ns[0], ss);
            if (c > 0) CU(cudaStreamWaitEvent(ss, L.ev_pack[c - 1], 0));
            launches += launch_pack(b, ix->codes, b1 - b0, ss);
            CU(cudaEventRecord(L.ev_pack[c], ss));
            if (knobs.stall_ns[1] && (c & 1)) launch_stall(knobs.stall_ns[1], ss);
        }
        launches += launch_search(ix->dir, ix->pair, locate ? &ix->toe : nullptr, ix->ft, b, r, L.d_ctr, &L.d_ctr->cursor[c], ss);
        if (rd->has_bases) launches += launch_search_bytes(ix->dir, locate ? &ix->toe : nullptr, b, r, ix->codes, L.d_ctr, ss);
        if (narrow_rg) launches += launch_narrow_ranges(r.lo, r.hi, rd->lo32.as<uint32_t>(), rd->hi32.as<uint32_t>(), r0, r1, ss);
        CU(cudaEventRecord(L.ev_cmp[c], ss));
        CU(cudaStreamWaitEvent(so, L.ev_cmp[c], 0));
        CU(cudaStreamWaitEvent(sc, L.ev_cmp[c], 0));                                  // what follows on sc (counts, scans, phi, markers) needs this chunk's ranges
        if (c == 0) CU(cudaEventRecord(L.ev_span[4], so));
        if (narrow_rg) {
            CU(cudaMemcpyAsync(out->lo32 + r0, rd->lo32.as<uint32_t>() + r0, (r1 - r0) * 4, cudaMemcpyDeviceToHost, so));
            CU(cudaMemcpyAsync(out->hi32 + r0, rd->hi32.as<uint32_t>() + r0, (r1 - r0) * 4, cudaMemcpyDeviceToHost, so));
        } else {
            CU(cudaMemcpyAsync(out->lo + r0, r.lo + r0, (r1 - r0) * 8, cudaMemcpyDeviceToHost, so));
            CU(cudaMemcpyAsync(out->hi + r0, r.hi + r0, (r1 - r0) * 8, cudaMemcpyDeviceToHost, so));
        }
        if (locate) {
            CU(cudaMemcpyAsync(out->toehold + r0, r.toehold + r0, (r1 - r0) * 8, cudaMemcpyDeviceToHost, so));
            launches += launch_locate_counts(r, r0, r1, max_hits, sc);
            CU(cudaMemcpyAsync(L.d_base, r.loc_off + r0, 8, cudaMemcpyDeviceToDevice, sc));
            launches += launch_scan_from(r.loc_cnt + r0, r.loc_off + r0, r1 - r0, L.d_base, rd->scan_tmp.p, rd->scan_tmp.cap, sc);
            CU(cudaMemcpyAsync(L.h_tot + c, r.loc_off + r1, 8, cudaMemcpyDeviceToHost, sc));
            CU(cudaEventRecord(L.ev_tot[c], sc));
            if (c > 0) locate_chunk(c - 1);
        }
    }
    if (locate && n) locate_chunk(n_chunks - 1);
    CU(cudaEventRecord(L.ev_span[1], si));
    rd->n_locs = locate && n ? L.h_tot[n_chunks - 1] : 0;
    rd->n_markers = 0;
    if (locate && !n) { grow_locs(0); out->loc_off[0] = 0; }
    // markers: whole-batch scan, then chunked gathers overlapped with their D2H (they are few)
    if (markers) {
        uint64_t* cnt = r.mk_cnt;
        uint64_t* off = r.mk_off;
        uint64_t* off_h = out->mk_off;
        launches += launch_marker_counts(ix->mk, r, 0, n, sc);
        const uint64_t total = scan_counts(L, rd, cnt, off, n, sc);           // syncs sc
        launches += 1;
        CU(cudaMemcpyAsync(off_h, off, (n + 1) * 8, cudaMemcpyDeviceToHost, sc));
        reserve(rd->markers, (total + 1) * 8);
        reserve(h->markers, (total + 1) * 8);
        rd->n_markers = total;
        r.markers = rd->markers.as<uint64_t>();
        out->markers = (uint64_t*) h->markers.p;
        CU(cudaStreamSynchronize(sc));                                        // boundaries of the segments below
        for (int c = 0; c < n_chunks && n; ++c) {
            const uint64_t r0 = cut(c), r1 = cut(c + 1);
            launches += launch_marker_gather(ix->mk, r, r0, r1, L.d_ctr, sc);
            CU(cudaEventRecord(L.ev_cmp[c], sc));
            CU(cudaStreamWaitEvent(so, L.ev_cmp[c], 0));
            const uint64_t a = off_h[r0], z = off_h[r1];
            if (z > a) CU(cudaMemcpyAsync((uint64_t*) h->markers.p + a, rd->markers.as<uint64_t>() + a, (z - a) * 8, cudaMemcpyDeviceToHost, so));
        }
    }
    CU(cudaMemcpyAsync(L.h_ctr, L.d_ctr, sizeof(DevCounters), cudaMemcpyDeviceToHost, sc));
    CU(cudaEventRecord(L.ev_span[3], sc));
    L.wait_stream(sc, 0);
    CU(cudaEventRecord(L.ev_span[5], so));
    L.wait_stream(so, 1);
    L.wait_stream(si, 2);
    CU(cudaGetLastError());
    collect_counters(L, s, rd, launches);
    s.ms_h2d = ev_ms(L.ev_span[0], L.ev_span[1]);          // busy spans of the three streams (they overlap)
    s.ms_search = ev_ms(L.ev_span[2], L.ev_span[3]);
    s.ms_d2h = n ? ev_ms(L.ev_span[4], L.ev_span[5]) : 0;
    s.ms_pack = s.ms_toehold = s.ms_locate = s.ms_markers = 0;
    rd->last_mode = mode;
    rd->ran = true;
}

// seq_ntoa_table, src/rb_markers.cpp:135-152: acgtACGT -> ACGT, n/N -> A, everything else -> 'N' (never in the index)
inline uint8_t seq_ntoa(uint8_t c) {
    switch (c) {
        case 'A': case 'a': case 'N': case 'n': return 'A';
        case 'C': case 'c': return 'C';
        case 'G': case 'g': return 'G';
        case 'T': case 't': return 'T';
        default: return 'N';
    }
}

// The rb_markers worker over one batch (src/rb_markers.cpp:375-404): H2D, pack with the seq_ntoa_table code
// map (+ the bad-base plane), counting walk, two scans, emitting walk, per-seed sort + unique, D2H.
void run_greedy(rbg_index* ix, Lane& L, rbg_stats& s, const rbg_batch* in, const rbg_greedy_params* gp, rbg_seed_result* out) {
    if (!ix->info.has_ma) throw std::invalid_argument("rbg_markers_greedy needs an index opened with RBG_LOAD_MA");
    GreedyParams P{gp->wsize, gp->max_range, gp->min_range, 0};
    const uint64_t n = in->n_reads;
    if (gp->use_ftab) {
        if (!ix->ft.k) throw std::invalid_argument("use_ftab without a resident seed table (rbg_ftab_build / RBG_LOAD_FT)");
        P.k = ix->ft.k;
        // the reference exits here (include/rowbowt.hpp:423-426) ...
        if ((uint64_t) P.k - 1 > gp->wsize) throw std::invalid_argument("wsize cannot be smaller than ftab k - 1");
        // ... and std::string::substr throws for a read shorter than k (:431)
        for (uint64_t i = 0; i < n; ++i)
            if (in->offsets[i + 1] - in->offsets[i] < P.k) throw std::invalid_argument("read shorter than the ftab k");
    }
    rbg_reads* rd = &L.scratch;
    GreedyScratch& g = L.greedy;
    cudaStream_t st = L.stream;
    CU(cudaEventRecord(L.ev[0], st));
    stage_batch(ix, st, BatchIn::raw(in), rd);
    const uint64_t n_words = (rd->n_bytes + 31) / 32 + 1;
    reserve(g.bad, n_words * 4);
    const uint64_t n_items = 2 * n;
    for (DevBuf* d : {&g.item_seeds, &g.item_words, &g.seed_off, &g.word_off}) reserve(*d, (n_items + 2) * 8);
    reserve(rd->scan_tmp, scan_tmp_bytes(n_items + 1));
    // Every A/C/G/T gets its code even when the index lacks that base: the minus strand complements the code, so a base
    // the index lacks may stand for one it has.  A code the index lacks ends its seed through LF (an empty range), as
    // in the reference; only 'N' after seq_ntoa has no code.
    CodeTable ct;
    for (int c = 0; c < 256; ++c) {
        const uint8_t a = seq_ntoa((uint8_t) c);
        ct.code_of[c] = a == 'A' ? 0 : a == 'C' ? 1 : a == 'G' ? 2 : a == 'T' ? 3 : (int8_t) -1;
    }
    DevBatch b{rd->bases.as<uint8_t>(), rd->offs.as<uint64_t>(), n, rd->n_bytes, 0, n, rd->packed.as<uint64_t>(),
               rd->flags.as<uint8_t>(), g.bad.as<uint32_t>()};
    DevSeedOut o{g.item_seeds.as<uint64_t>(), g.item_words.as<uint64_t>(), g.seed_off.as<uint64_t>(), g.word_off.as<uint64_t>(),
                 nullptr, nullptr};
    uint32_t launches = 0;
    CU(cudaMemsetAsync(L.d_ctr, 0, sizeof(DevCounters), st));
    CU(cudaMemsetAsync(g.bad.p, 0xFF, n_words * 4, st));          // words no launch packs count as bad bases
    CU(cudaEventRecord(L.ev[1], st));
    launches += launch_pack(b, ct, rd->n_bytes, st);
    CU(cudaEventRecord(L.ev[2], st));
    launches += launch_greedy(ix->dir, ix->ft, ix->mk, b, P, o, false, L.d_ctr, st);
    const uint64_t total_seeds = scan_counts(L, rd, o.item_seeds, o.seed_off, n_items, st);
    const uint64_t total_words = scan_counts(L, rd, o.item_words, o.word_off, n_items, st);
    launches += 2;
    reserve(g.seeds, (total_seeds + 1) * sizeof(DevSeed));
    reserve(g.words, (total_words + 1) * 8);
    o.seeds = g.seeds.as<DevSeed>();
    o.words = g.words.as<uint64_t>();
    launches += launch_greedy(ix->dir, ix->ft, ix->mk, b, P, o, true, L.d_ctr, st);
    CU(cudaEventRecord(L.ev[3], st));
    launches += launch_seed_sort(o, total_seeds, st);
    CU(cudaEventRecord(L.ev[4], st));

    HostSeedResult* h = ix->seed_results.take(ix);
    memset(out, 0, sizeof *out);
    out->_owner = h;
    out->n_reads = n;
    out->n_seeds = total_seeds;
    out->n_marker_words = total_words;
    reserve(h->seed_off, (n_items + 1) * 8);
    reserve(h->seeds, (total_seeds + 1) * sizeof(rbg_seed));
    reserve(h->markers, (total_words + 1) * 8);
    out->seed_off = (uint64_t*) h->seed_off.p;
    out->seeds = (rbg_seed*) h->seeds.p;
    out->markers = (uint64_t*) h->markers.p;
    CU(cudaMemcpyAsync(out->seed_off, o.seed_off, (n_items + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (total_seeds) CU(cudaMemcpyAsync(out->seeds, o.seeds, total_seeds * sizeof(rbg_seed), cudaMemcpyDeviceToHost, st));
    if (total_words) CU(cudaMemcpyAsync(out->markers, o.words, total_words * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(L.h_ctr, L.d_ctr, sizeof(DevCounters), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(L.ev[5], st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    collect_counters(L, s, rd, launches);
    s.ms_h2d = ev_ms(L.ev[0], L.ev[1]);
    s.ms_pack = ev_ms(L.ev[1], L.ev[2]);
    s.ms_search = ev_ms(L.ev[2], L.ev[3]);          // both walks + the scans
    s.ms_markers = ev_ms(L.ev[3], L.ev[4]);         // sort + unique
    s.ms_d2h = ev_ms(L.ev[4], L.ev[5]);
    s.ms_toehold = s.ms_locate = 0;
    rd->ran = false;
}

}  // namespace

extern "C" {

const char* rbg_last_error(void) { return g_err.c_str(); }

int rbg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int rbg_index_open(const char* prefix, uint32_t flags, int device, rbg_index** out) {
    if (!prefix || !out) return fail(RBG_E_ARG, "null argument");
    *out = nullptr;
    return guarded([&] {
        const std::string pre(prefix);
        if ((flags & RBG_LOAD_FBB) && (flags & RBG_LOAD_SA))
            return fail(RBG_E_ARG, "fbb_string does not support loading toehold suffix array");     // include/rowbowt_io.hpp:107
        const LayoutKnobs knobs = layout_knobs();
        std::unique_ptr<rbg_index> ix;
        if (flags & RBG_LOAD_CACHE) ix = open_layout_cache(pre, flags, device, knobs);
        if (!ix) {
            // the three files are decoded at the same time (each reader is itself multi-threaded over its components)
            std::future<ToeholdArrays> tsa_job;
            std::future<MarkerArrays> ma_job;
            if (flags & RBG_LOAD_SA) tsa_job = std::async(std::launch::async, [&pre] { return read_tsa(pre + ".tsa"); });   // tsa_suffix :18
            if (flags & RBG_LOAD_MA) ma_job = std::async(std::launch::async, [&pre] { return read_mab(pre + ".mab"); });    // ma_suffix  :19
            RunsBwt bwt = (flags & RBG_LOAD_FBB) ? read_rbwt_fbb(pre + ".rbwt") : read_rbwt(pre + ".rbwt");   // rbwt_suffix, include/rowbowt_io.hpp:17
            ToeholdArrays tsa;
            MarkerArrays ma;
            if (flags & RBG_LOAD_SA) tsa = tsa_job.get();
            if (flags & RBG_LOAD_MA) ma = ma_job.get();
            ix = open_from_arrays(bwt, (flags & RBG_LOAD_SA) ? &tsa : nullptr, (flags & RBG_LOAD_MA) ? &ma : nullptr, device, knobs);
            if (flags & RBG_LOAD_FBB) ix->codes.code_of[1] = -1;   // wt_fbb: terminator is byte 0, byte 1 is no symbol
            if (flags & RBG_LOAD_CACHE) {
                try { write_layout_cache(ix.get(), pre, flags, knobs); } catch (...) { cudaGetLastError(); }      // best effort: the index is open either way
            }
        }
        if (flags & RBG_LOAD_FT) {                  // ft_suffix :21, LoadRbwtFlag::FT :151
            LaneHold hold(ix.get(), true);
            load_ftab(ix.get(), hold.lane->stream, pre + ".ftab");
        }
        *out = ix.release();
        return (int) RBG_OK;
    });
}

namespace {
// The arrays an index is laid out from; the toehold / marker arrays only with has_sa / has_ma.
struct IndexArrays {
    RunsBwt bwt;
    ToeholdArrays tsa;
    MarkerArrays ma;
    bool has_sa = false, has_ma = false;
};

// The arrays of a caller's rbg_index_desc: toehold arrays when all four of their pointers are set, marker arrays when all
// three are.  With `tsa_only` (the marker-array build) the toehold arrays are required and marker arrays are not read.
IndexArrays index_arrays_from_desc(const rbg_index_desc* d, bool tsa_only) {
    if (!d->run_heads || !d->run_lens) throw std::invalid_argument("run_heads/run_lens missing");
    IndexArrays p;
    p.has_sa = d->r && d->pred && d->samples_last && d->pred_to_run;
    if (tsa_only && !p.has_sa) throw std::invalid_argument("toehold arrays missing");
    p.bwt.n = d->n;
    p.bwt.R = d->R;
    p.bwt.heads.assign(d->run_heads, d->run_heads + d->R);
    p.bwt.lens.assign(d->run_lens, d->run_lens + d->R);
    if (p.has_sa) {
        p.tsa.r = d->r;
        p.tsa.n = d->n;
        p.tsa.pred.assign(d->pred, d->pred + d->r);
        p.tsa.samples_last.assign(d->samples_last, d->samples_last + d->r);
        p.tsa.pred_to_run.assign(d->pred_to_run, d->pred_to_run + d->r);
    }
    p.has_ma = !tsa_only && d->win_starts && d->win_ends && d->win_idxs;
    if (p.has_ma) {
        p.ma.starts.assign(d->win_starts, d->win_starts + d->n_windows);
        p.ma.ends.assign(d->win_ends, d->win_ends + d->n_windows);
        p.ma.idxs.assign(d->win_idxs, d->win_idxs + d->n_windows);
        if (d->arr_size) p.ma.arr.assign(d->arr, d->arr + d->arr_size);
        p.ma.size_starts = d->size_starts;
        p.ma.size_ends = d->size_ends;
        p.ma.size_idxs = d->size_idxs;
    }
    return p;
}

std::unique_ptr<rbg_index> open_from_arrays(const IndexArrays& p, int device) {
    return open_from_arrays(p.bwt, p.has_sa ? &p.tsa : nullptr, p.has_ma ? &p.ma : nullptr, device, layout_knobs());
}

// rb_build's inputs (src/rb_build.cpp:76-87): <prefix>.bwt, .ssa/.esa, .ma
void load_raw(const std::string& pre, uint32_t flags, int device, IndexArrays& p, rbg_build_stats* st) {
    select_device(device);
    RawBuildStats rs;
    double t0 = wall_s();
    p.bwt = rle_bwt_gpu(pre + ".bwt", device, &rs);
    if (st) {
        st->n = p.bwt.n;
        st->r = p.bwt.R;
        st->s_bwt_read = rs.s_read;
        st->ms_rle_kernels = rs.ms_kernels;
        st->s_rle = wall_s() - t0;
    }
    p.has_sa = flags & RBG_LOAD_SA;
    if (p.has_sa) {
        t0 = wall_s();
        p.tsa = toehold_from_raw(pre + ".ssa", pre + ".esa", p.bwt.n, p.bwt.R, device);
        if (st) st->s_samples = wall_s() - t0;
    }
    p.has_ma = flags & RBG_LOAD_MA;
    if (p.has_ma) {
        t0 = wall_s();
        p.ma = markers_from_ma(pre + ".ma");
        if (st) st->s_markers = wall_s() - t0;
    }
}
}  // namespace

int rbg_index_open_arrays(const rbg_index_desc* d, int device, rbg_index** out) {
    if (!d || !out) return fail(RBG_E_ARG, "null argument");
    *out = nullptr;
    return guarded([&] {
        *out = open_from_arrays(index_arrays_from_desc(d, false), device).release();
        return (int) RBG_OK;
    });
}

int rbg_index_open_raw(const char* prefix, uint32_t flags, int device, rbg_index** out) {
    if (!prefix || !out) return fail(RBG_E_ARG, "null argument");
    *out = nullptr;
    return guarded([&] {
        IndexArrays p;
        load_raw(prefix, flags, device, p, nullptr);
        *out = open_from_arrays(p, device).release();
        return (int) RBG_OK;
    });
}

int rbg_build_index(const char* in_prefix, const char* out_prefix, uint32_t flags, uint32_t ftab_k, int device, rbg_build_stats* stats) {
    if (!in_prefix || !out_prefix) return fail(RBG_E_ARG, "null argument");
    return guarded([&] {
        rbg_build_stats st;
        memset(&st, 0, sizeof st);
        const double t_begin = wall_s();
        IndexArrays p;
        load_raw(in_prefix, flags, device, p, &st);
        const std::string out(out_prefix);
        double t0 = wall_s();
        write_rbwt(p.bwt, out + ".rbwt");                                  // rowbowt_io.hpp:54-57
        if (flags & RBG_LOAD_MA) write_mab(p.ma, out + ".mab");            // :58-64
        if (flags & RBG_LOAD_SA) write_tsa(p.tsa, out + ".tsa");           // :65-72
        st.s_write = wall_s() - t0;
        if (flags & RBG_LOAD_FT) {                                         // :82-88 (rb_build -f): build_ftab(k) + FTab::serialize
            std::unique_ptr<rbg_index> ix = open_from_arrays(p.bwt, nullptr, nullptr, device, layout_knobs());
            {
                LaneHold hold(ix.get(), true);
                build_ftab(ix.get(), hold.lane->stream, ftab_k ? ftab_k : 10);
            }
            save_ftab(ix.get(), out + ".ftab");
        }
        st.s_total = wall_s() - t_begin;
        if (stats) *stats = st;
        return (int) RBG_OK;
    });
}

namespace {
// What the two rbg_build_marker_array entries share once the index arrays are in hand: the device check, then the build.
// `mps` was read and checked against n (read_mps_window) before any CUDA call.
int build_ma_from(const IndexArrays& p, const MpsRecords& mps, uint64_t row_begin, uint64_t row_end, int device, const char* ma_path,
                  const char* mab_path, rbg_ma_stats& st, double t_begin, rbg_ma_stats* out) {
    select_device(device);
    st.n = p.bwt.n;
    st.r = p.bwt.R;
    st.mps_records = mps.first.size();
    st.lists = mps.list_off.size() - 1;
    build_marker_array(p.bwt, p.tsa, mps, row_begin, row_end, device, ma_path, mab_path ? mab_path : "", st);
    st.s_total = wall_s() - t_begin;
    if (out) *out = st;
    return (int) RBG_OK;
}

void check_sample_count(uint64_t r, uint64_t R) {
    if (r != R) throw std::invalid_argument("the toehold arrays hold " + std::to_string(r) + " samples for " + std::to_string(R) + " runs");
}

// The window [row_begin, min(row_end, n)) must hold a row; then the .mps is read against n.
MpsRecords read_mps_window(const char* mps_path, uint64_t n, uint64_t row_begin, uint64_t& row_end) {
    row_end = std::min(row_end, n);
    if (row_begin >= row_end) throw std::invalid_argument("empty row window");
    return read_mps(mps_path, n);
}
}  // namespace

int rbg_build_marker_array(const char* index_prefix, const char* mps_path, const char* ma_path, const char* mab_path,
                           uint64_t row_begin, uint64_t row_end, int device, rbg_ma_stats* stats) {
    if (!index_prefix || !mps_path || !ma_path) return fail(RBG_E_ARG, "null argument");
    return guarded([&] {
        rbg_ma_stats st;
        memset(&st, 0, sizeof st);
        const double t_begin = wall_s();
        const std::string pre(index_prefix);
        struct stat sb;
        IndexArrays p;
        uint64_t n;
        const bool raw = stat((pre + ".rbwt").c_str(), &sb) != 0;
        if (!raw) {
            if (stat((pre + ".tsa").c_str(), &sb) != 0) return fail(RBG_E_IO, "no toehold samples: " + pre + ".tsa");
            p.bwt = read_rbwt(pre + ".rbwt");
            p.tsa = read_tsa(pre + ".tsa");
            check_sample_count(p.tsa.r, p.bwt.R);
            n = p.bwt.n;
        } else {           // the raw inputs: n is the size of the .bwt (one byte per row); decoded on the GPU afterwards
            if (stat((pre + ".bwt").c_str(), &sb) != 0) return fail(RBG_E_IO, "no index: neither " + pre + ".rbwt nor " + pre + ".bwt");
            n = (uint64_t) sb.st_size;
            for (const char* suf : {".ssa", ".esa"})
                if (stat((pre + suf).c_str(), &sb) != 0) return fail(RBG_E_IO, "no toehold samples: " + pre + suf);
        }
        const MpsRecords mps = read_mps_window(mps_path, n, row_begin, row_end);
        if (raw) load_raw(pre, RBG_LOAD_SA, device, p, nullptr);
        st.s_read = wall_s() - t_begin;
        return build_ma_from(p, mps, row_begin, row_end, device, ma_path, mab_path, st, t_begin, stats);
    });
}

int rbg_build_marker_array_arrays(const rbg_index_desc* d, const char* mps_path, const char* ma_path, const char* mab_path,
                                  uint64_t row_begin, uint64_t row_end, int device, rbg_ma_stats* stats) {
    if (!d || !mps_path || !ma_path) return fail(RBG_E_ARG, "null argument");
    return guarded([&] {
        rbg_ma_stats st;
        memset(&st, 0, sizeof st);
        const double t_begin = wall_s();
        const IndexArrays p = index_arrays_from_desc(d, true);
        check_sample_count(p.tsa.r, p.bwt.R);
        const MpsRecords mps = read_mps_window(mps_path, p.bwt.n, row_begin, row_end);
        validate_runs(p.bwt, "the BWT runs");
        validate_toehold(p.tsa, "the toehold arrays");
        st.s_read = wall_s() - t_begin;
        return build_ma_from(p, mps, row_begin, row_end, device, ma_path, mab_path, st, t_begin, stats);
    });
}

int rbg_build_bwt(const char* fasta_path, const char* out_prefix, int device, rbg_bwt_stats* stats) {
    if (!fasta_path || !out_prefix) return fail(RBG_E_ARG, "null argument");
    return guarded([&] {
        rbg_bwt_stats st;
        memset(&st, 0, sizeof st);
        const double t_begin = wall_s();
        const BwtKnobs knobs = bwt_knobs();
        const FastaText ft = read_fasta_text(fasta_path, kBwtWideMaxN);
        st.records = ft.names.size();
        st.s_parse = wall_s() - t_begin;
        select_device(device);
        if (knobs.wide || ft.text.size() + 1 > kBwtMaxN) build_bwt_files_wide(ft.text.data(), ft.text.size(), device, knobs.part_rows, out_prefix, st);
        else build_bwt_files(ft.text.data(), ft.text.size(), device, out_prefix, st);
        const double t_docs = wall_s();
        write_docs(ft, std::string(out_prefix) + ".docs");
        st.s_write += wall_s() - t_docs;
        st.s_total = wall_s() - t_begin;
        if (stats) *stats = st;
        return (int) RBG_OK;
    });
}

int rbg_build_bwt_text(const uint8_t* text, uint64_t len, const char* out_prefix, int device, rbg_bwt_stats* stats) {
    if (!text || !out_prefix) return fail(RBG_E_ARG, "null argument");
    if (len == 0) return fail(RBG_E_ARG, "empty text");
    return guarded([&] {
        rbg_bwt_stats st;
        memset(&st, 0, sizeof st);
        const double t_begin = wall_s();
        check_bwt_length(std::min(len, kBwtMaxN) + 1, "a text of " + std::to_string(len) + " bases", kBwtMaxN);   // before the buffer is read
        const BwtKnobs knobs = bwt_knobs();
        check_acgt(text, len);
        st.s_parse = wall_s() - t_begin;
        select_device(device);
        if (knobs.wide) build_bwt_files_wide(text, len, device, knobs.part_rows, out_prefix, st);
        else build_bwt_files(text, len, device, out_prefix, st);
        st.s_total = wall_s() - t_begin;
        if (stats) *stats = st;
        return (int) RBG_OK;
    });
}

void rbg_index_close(rbg_index* ix) {
    if (ix) cudaSetDevice(ix->device);
    delete ix;
}

int rbg_ftab_build(rbg_index* ix, uint32_t k) {
    if (!ix) return fail(RBG_E_ARG, "null argument");
    return guarded([&] {
        CU(cudaSetDevice(ix->device));
        LaneHold hold(ix, true);             // no query in flight while the table (and the counts next to it) move
        build_ftab(ix, hold.lane->stream, k);
        return (int) RBG_OK;
    });
}

int rbg_ftab_load(rbg_index* ix, const char* path) {
    if (!ix || !path) return fail(RBG_E_ARG, "null argument");
    return guarded([&] {
        CU(cudaSetDevice(ix->device));
        LaneHold hold(ix, true);
        try {
            load_ftab(ix, hold.lane->stream, path);
        } catch (...) {
            build_ftab(ix, hold.lane->stream, 0);           // never keep a table that failed its check
            throw;
        }
        return (int) RBG_OK;
    });
}

int rbg_ftab_save(const rbg_index* ix, const char* path) {
    if (!ix || !path) return fail(RBG_E_ARG, "null argument");
    return guarded([&] {
        save_ftab(ix, path);
        return (int) RBG_OK;
    });
}

int rbg_ftab_lookup(const rbg_index* ix, const char* kmers, uint64_t n_kmers, uint64_t* lo, uint64_t* hi, uint64_t* consumed) {
    if (!ix || !kmers || !lo || !hi) return fail(RBG_E_ARG, "null argument");
    if (!ix->ft.k) return fail(RBG_E_ARG, "no ftab loaded");
    const uint32_t k = ix->ft.k;
    for (uint64_t i = 0; i < n_kmers; ++i) {
        uint64_t key;
        const bool ok = kmer_key(kmers + i * k, k, key) && ix->ft_host[key].x <= ix->ft_host[key].y;
        lo[i] = ok ? ix->ft_host[key].x : 0;                  // miss: (full_range(), 0), rowbowt.hpp:757
        hi[i] = ok ? ix->ft_host[key].y : ix->info.n - 1;
        if (consumed) consumed[i] = ok ? k : 0;
    }
    return RBG_OK;
}

int rbg_index_info(const rbg_index* ix, rbg_info* info) {
    if (!ix || !info) return fail(RBG_E_ARG, "null argument");
    *info = ix->info;
    return RBG_OK;
}

int rbg_last_stats(const rbg_index* ix, rbg_stats* st) {
    if (!ix || !st) return fail(RBG_E_ARG, "null argument");
    std::lock_guard<std::mutex> lock(const_cast<rbg_index*>(ix)->mu);
    *st = ix->stats;
    return RBG_OK;
}

namespace {
int query_any(rbg_index* ix, const BatchIn& in, uint32_t mode, uint64_t max_hits, rbg_result* out) {
    return guarded([&] {
        CU(cudaSetDevice(ix->device));
        LaneHold hold(ix);
        auto t0 = std::chrono::steady_clock::now();
        memset(out, 0, sizeof *out);
        try {
            run_pipelined(ix, *hold.lane, hold.stats, in, mode, max_hits, out);
        } catch (...) {
            cudaStreamSynchronize(hold.lane->s_in);
            for (auto& st : hold.lane->s_srch) cudaStreamSynchronize(st);
            cudaStreamSynchronize(hold.lane->stream);
            cudaStreamSynchronize(hold.lane->s_out);
            if (out->_owner) { ix->results.give_back((HostResult*) out->_owner); memset(out, 0, sizeof *out); }
            throw;
        }
        hold.stats.ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        hold.publish = true;
        return (int) RBG_OK;
    });
}
}  // namespace

int rbg_query(rbg_index* ix, const rbg_batch* in, uint32_t mode, uint64_t max_hits, rbg_result* out) {
    if (!ix || !in || !out) return fail(RBG_E_ARG, "null argument");
    if (in->n_reads && (!in->offsets || !in->bases)) return fail(RBG_E_ARG, "batch without bases/offsets");
    return query_any(ix, BatchIn::raw(in), mode, max_hits, out);
}

int rbg_query_packed(rbg_index* ix, const rbg_packed_batch* in, uint32_t mode, uint64_t max_hits, rbg_result* out) {
    if (!ix || !in || !out) return fail(RBG_E_ARG, "null argument");
    if (int rc = check_packed(in)) return rc;
    return query_any(ix, BatchIn::from_packed(in), mode, max_hits, out);
}

void rbg_result_free(rbg_result* res) {
    if (!res || !res->_owner) return;
    HostResult* h = (HostResult*) res->_owner;
    h->ix->results.give_back(h);
    memset(res, 0, sizeof *res);
}

int rbg_markers_greedy(rbg_index* ix, const rbg_batch* in, const rbg_greedy_params* params, rbg_seed_result* out) {
    if (!ix || !in || !params || !out) return fail(RBG_E_ARG, "null argument");
    if (in->n_reads && (!in->offsets || !in->bases)) return fail(RBG_E_ARG, "batch without bases/offsets");
    return guarded([&] {
        CU(cudaSetDevice(ix->device));
        LaneHold hold(ix);
        auto t0 = std::chrono::steady_clock::now();
        memset(out, 0, sizeof *out);
        try {
            run_greedy(ix, *hold.lane, hold.stats, in, params, out);
        } catch (...) {
            cudaStreamSynchronize(hold.lane->stream);
            if (out->_owner) { ix->seed_results.give_back((HostSeedResult*) out->_owner); memset(out, 0, sizeof *out); }
            throw;
        }
        hold.stats.ms_total = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        hold.publish = true;
        return (int) RBG_OK;
    });
}

void rbg_seed_result_free(rbg_seed_result* res) {
    if (!res || !res->_owner) return;
    HostSeedResult* h = (HostSeedResult*) res->_owner;
    h->ix->seed_results.give_back(h);
    memset(res, 0, sizeof *res);
}

namespace {
int upload_any(rbg_index* ix, const BatchIn& in, rbg_reads** out) {
    *out = nullptr;
    return guarded([&] {
        CU(cudaSetDevice(ix->device));
        LaneHold hold(ix);
        std::unique_ptr<rbg_reads> rd(new rbg_reads);
        stage_batch(ix, hold.lane->stream, in, rd.get());
        CU(cudaStreamSynchronize(hold.lane->stream));
        *out = rd.release();
        return (int) RBG_OK;
    });
}
}  // namespace

int rbg_reads_upload(rbg_index* ix, const rbg_batch* in, rbg_reads** out) {
    if (!ix || !in || !out) return fail(RBG_E_ARG, "null argument");
    if (in->n_reads && (!in->offsets || !in->bases)) return fail(RBG_E_ARG, "batch without bases/offsets");
    return upload_any(ix, BatchIn::raw(in), out);
}

int rbg_reads_upload_packed(rbg_index* ix, const rbg_packed_batch* in, rbg_reads** out) {
    if (!ix || !in || !out) return fail(RBG_E_ARG, "null argument");
    if (int rc = check_packed(in)) return rc;
    return upload_any(ix, BatchIn::from_packed(in), out);
}

int rbg_query_staged(rbg_index* ix, rbg_reads* reads, uint32_t mode, uint64_t max_hits, uint64_t* checksum) {
    if (!ix || !reads || reads->ix != ix) return fail(RBG_E_ARG, "bad staged batch");
    return guarded([&] {
        CU(cudaSetDevice(ix->device));
        LaneHold hold(ix);
        run_staged(ix, *hold.lane, hold.stats, reads, mode, max_hits, checksum != nullptr);
        if (checksum) *checksum = hold.lane->h_ctr->checksum;
        hold.publish = true;
        return (int) RBG_OK;
    });
}

int rbg_reads_fetch(rbg_index* ix, rbg_reads* reads, uint32_t mode, rbg_result* out) {
    if (!ix || !reads || !out || reads->ix != ix) return fail(RBG_E_ARG, "bad staged batch");
    return guarded([&] {
        CU(cudaSetDevice(ix->device));
        LaneHold hold(ix);
        fetch_staged(ix, *hold.lane, reads, mode, out);
        return (int) RBG_OK;
    });
}

void rbg_reads_free(rbg_reads* reads) {
    if (!reads) return;
    if (reads->ix) cudaSetDevice(reads->ix->device);
    delete reads;
}

int rbg_pack_bytes(const rbg_index* ix, const char* bases, const uint64_t* offsets, uint64_t n_reads,
                   uint64_t x0, uint64_t x1, uint64_t* packed, uint8_t* flags, uint64_t* n_exotic) {
    if (!ix || !offsets || !packed || !flags || (!bases && x1 > x0)) return fail(RBG_E_ARG, "null argument");
    if (x0 & 31) return fail(RBG_E_ARG, "rbg_pack_bytes: x0 must be a multiple of 32");
    if (n_reads && offsets[0] != 0) return fail(RBG_E_ARG, "rbg_pack_bytes: offsets[0] must be 0");
    if (n_reads == 0 || x1 > offsets[n_reads]) x1 = n_reads ? offsets[n_reads] : 0;
    const uint64_t ex = pack_bytes_host(ix->codes.code_of, (const uint8_t*) bases, offsets, n_reads, x0, x1, packed, flags);
    if (n_exotic && ex) __atomic_fetch_add(n_exotic, ex, __ATOMIC_RELAXED);
    return RBG_OK;
}

void* rbg_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        g_err = "cudaHostAlloc failed";
        return nullptr;
    }
    return p;
}

void rbg_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int rbg_check_suffix_array(const uint8_t* text, uint64_t len, const uint64_t* sa, int device, uint64_t* first_bad) {
    if (!text || !sa || !first_bad) return fail(RBG_E_ARG, "null argument");
    if (len == 0) return fail(RBG_E_ARG, "empty text");
    return guarded([&] {
        check_acgt(text, len);
        select_device(device);
        *first_bad = check_suffix_array(text, len, sa, device);
        return (int) RBG_OK;
    });
}

double rbg_gather_roofline(int device, size_t footprint_bytes, int line_bytes, int iters) {
    int dependent = 0;
    if (iters < 0) { dependent = 1; iters = -iters; }
    if (line_bytes == -64) { dependent = 2; line_bytes = 64; }          // 64-byte lines read by lane pairs: one request per line
    if (line_bytes != 32 && line_bytes != 64 && line_bytes != 128) { g_err = "line_bytes must be 32, 64 or 128"; return -1.0; }
    double gbs = -1.0;
    int rc = guarded([&] {
        select_device(device);
        void* buf = nullptr;
        CU(cudaMalloc(&buf, footprint_bytes));
        CU(cudaMemset(buf, 0x5A, footprint_bytes));
        cudaStream_t st;
        CU(cudaStreamCreate(&st));
        uint64_t lines = 0;
        float ms = run_gather((const uint32_t*) buf, footprint_bytes / line_bytes, line_bytes, iters, dependent, &lines, st);
        cudaError_t e = cudaGetLastError();
        cudaStreamDestroy(st);
        cudaFree(buf);
        if (e != cudaSuccess) throw cuda_error(cudaGetErrorString(e));
        gbs = (double) lines * line_bytes / (ms * 1e-3) / 1e9;
        return (int) RBG_OK;
    });
    return rc == RBG_OK ? gbs : -1.0;
}

}  // extern "C"
