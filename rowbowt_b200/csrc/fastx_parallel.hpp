// Parallel FASTQ front end of the host drivers (SURVEY.md §8(f) row 2).
//
// The reference parses one record at a time with klib's kseq (include/kseq.h:178-218) on the
// thread that also searches and prints (src/rb_align.cpp:176-178).  Once the search runs on the
// GPU the parser is the bottleneck, so an uncompressed input is mmap'ed, cut into byte chunks and
// parsed by several threads straight into pinned batch buffers -- with NO change in what the
// query sees:
//
//   * a chunk parser only accepts the strict four-line form (`@name...`, one sequence line, `+...`,
//     one quality line of the same length, no '\r', no blank lines, next record starts with '@').
//     On that form it yields exactly kseq's (name, sequence).  Anything else makes it stop ("bail")
//     at the start of the offending record, where kseq's state is simply "between records".
//   * where a chunk starts is a GUESS (first line starting with '@' whose line after next starts
//     with '+').  The guess is never trusted: chunk k+1 is accepted only if its start equals the
//     position where chunk k's parse really ended.  Chunk 0 starts at byte 0, so by induction the
//     accepted records are those of a sequential parse.
//   * after a bail or a wrong guess everything from the last verified position is re-read by the
//     sequential kseq-compatible reader (FastxReader), which also serves .gz inputs.
//
//
// BGZF (bgzip) inputs take the same road: the block headers give every block's place in the inflated stream, so a
// parser thread inflates the blocks under ITS chunk (plus a margin behind it for the record that straddles the chunk end)
// into a private buffer and parses that.  The end of such a view is never taken for the end of the input: a record
// that runs into it is a bail.  Files that are not blocks from the first byte to the last keep the sequential reader.
//
// Batches come out of next() in input order with dense ids.
#pragma once
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/resource.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <atomic>
#include <functional>
#include <map>
#include <memory>
#include <thread>

#include "host_io.hpp"
#include "report_format.hpp"

namespace rbhost {

struct HostAlloc {              // pinned (rbg_host_alloc) in the drivers, malloc in --parse-only
    void* (*alloc)(size_t);
    void (*release)(void*);
};

template <class T>
struct GrowBuf {
    T* p = nullptr;
    size_t cap = 0;
    HostAlloc a{nullptr, nullptr};
    ~GrowBuf() { if (p) a.release(p); }
    void reserve(size_t want, size_t keep) {
        if (want <= cap) return;
        size_t ncap = std::max(want, cap + cap / 2);
        T* q = (T*) a.alloc(ncap * sizeof(T));
        if (!q) { fprintf(stderr, "host allocation of %zu bytes failed\n", ncap * sizeof(T)); exit(1); }
        if (keep) memcpy(q, p, keep * sizeof(T));
        if (p) a.release(p);
        p = q;
        cap = ncap;
    }
};

// What one rbg_query / rbg_markers_greedy call consumes, plus the names for the report.
struct ReadBatch {
    uint64_t id = 0;
    uint64_t n = 0;                     // reads
    GrowBuf<char> bases;                // concatenated sequences (C-string semantics already applied)
    GrowBuf<uint64_t> offs;             // n + 1
    std::vector<char> names;            // concatenated names
    std::vector<uint64_t> name_off{0};  // n + 1
    std::vector<OutBuf> text;           // formatted text, one buffer per formatter slice; keeps its pages across recycles
    size_t n_text = 0;                  // slices of `text` in use
    std::vector<uint8_t> aux;           // one driver-defined byte per read (rb_markers --heuristic: strand tried first)
    // 2-bit form of `bases` for rbg_query_packed, filled by the driver's on_batch hook (on the parser thread that built the batch)
    GrowBuf<uint64_t> packed;
    GrowBuf<uint8_t> flags;
    uint64_t n_exotic = 0;
    // chunk bookkeeping of the parallel parser
    size_t begin = 0, end = 0;
    bool bailed = false;

    void clear() {
        n = 0;
        names.clear();
        name_off.assign(1, 0);
        n_text = 0;
        aux.clear();
        n_exotic = 0;
        bailed = false;
        offs.reserve(1, 0);
        offs.p[0] = 0;
    }
    uint64_t n_bases() const { return offs.p[n]; }
    void add(const char* name, size_t name_len, const char* seq, size_t seq_len) {
        const uint64_t at = offs.p[n];
        bases.reserve(at + seq_len + 1, at);
        memcpy(bases.p + at, seq, seq_len);
        offs.reserve(n + 2, n + 1);
        offs.p[n + 1] = at + seq_len;
        names.insert(names.end(), name, name + name_len);
        name_off.push_back(names.size());
        ++n;
    }
    const char* name(uint64_t i, size_t& len) const {
        len = name_off[i + 1] - name_off[i];
        return names.data() + name_off[i];
    }
};

class FastxBatchSource {
  public:
    // chunk_bytes = 0: chosen from the file size.  threads <= 1, a pipe or a .gz input that is not BGZF: sequential reader.
    // on_batch (optional) runs on the thread that completed a batch, before it is handed out: the drivers pack the bases there.
    // `alloc`: what the GPU call reads (offsets, packed bases, flags; the raw bases too unless bases_alloc is given) -- pinned in
    // the drivers.  bases_alloc (optional): where the raw bases go when the driver ships the packed form (plain malloc: pinning
    // costs ~0.3 ms per MB and holds the CUDA context lock the GPU worker needs).  start = false: the parser threads wait for start().
    FastxBatchSource(const char* path, int threads, size_t chunk_bytes, size_t batch_reads, HostAlloc alloc, size_t pool_size,
                     std::function<void(ReadBatch&)> on_batch = nullptr, bool start = true, const HostAlloc* bases_alloc = nullptr)
        : path_(path), alloc_(alloc), batch_reads_(std::max<size_t>(1, batch_reads)), on_batch_(std::move(on_batch)) {
        for (size_t i = 0; i < std::max<size_t>(pool_size, 2); ++i) {
            std::unique_ptr<ReadBatch> b(new ReadBatch);
            b->bases.a = bases_alloc ? *bases_alloc : alloc_;
            b->offs.a = alloc_;
            b->packed.a = alloc_;
            b->flags.a = alloc_;
            b->clear();
            pool_.push_back(std::move(b));
        }
        // stat first: a FIFO / /dev/stdin / <(...) must be opened exactly once, by the sequential reader's gzopen
        // (an open + close here would eat the head of the stream or SIGPIPE its writer)
        struct stat st;
        if (stat(path, &st) != 0) return;
        const bool regular = S_ISREG(st.st_mode);
        if (regular && threads > 1 && st.st_size > 0) {
            int fd = open(path, O_RDONLY);
            if (fd < 0) return;
            unsigned char magic[2] = {0, 0};
            const bool gz = pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
            void* m = mmap(nullptr, (size_t) st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
            close(fd);
            if (m != MAP_FAILED && !gz) {
                data_ = (const char*) m;
                size_ = (size_t) st.st_size;
                madvise(m, size_, MADV_SEQUENTIAL);
            } else if (m != MAP_FAILED) {
                // BGZF from the first byte to the last: block table -> chunks of the inflated stream
                const unsigned char* z = (const unsigned char*) m;
                if (BgzfSource::index(z, (size_t) st.st_size, bz_coff_, bz_uoff_) && bz_uoff_.back() > 0) {
                    if (const char* e = getenv("RBG_VIEW_MARGIN")) { view_margin_ = (size_t) std::max(0l, atol(e)); margin_forced_ = true; }
                    zdata_ = z;
                    zsize_ = (size_t) st.st_size;
                    size_ = (size_t) bz_uoff_.back();
                } else {
                    munmap(m, (size_t) st.st_size);
                }
            }
        }
        ok_ = true;
        threads_ = threads;
        if (data_ || zdata_) {
            // a chunk is a GPU batch and a pinned buffer: 16 MB (~50 k reads) keeps the pinned pool small (pinning costs ~0.3 ms/MB)
            // while one rbg_query per chunk is still far from launch-bound
            if (!chunk_bytes) chunk_bytes = std::min<size_t>(16u << 20, std::max<size_t>(1u << 20, size_ / (4 * (size_t) threads)));
            chunk_bytes_ = chunk_bytes;
            n_chunks_ = (size_ + chunk_bytes_ - 1) / chunk_bytes_;
            // the margin is inflated twice (by this chunk's thread and the next one's): a quarter of a chunk at most
            if (!margin_forced_) view_margin_ = std::min<size_t>(1u << 20, std::max<size_t>(64u << 10, chunk_bytes_ / 4));
            if (start) this->start();
        } else {
            seq_.reset(new FastxReader(path, threads));          // --threads 1: plain gzread, no inflate workers
            ok_ = seq_->ok();
        }
    }
    ~FastxBatchSource() {
        stop_parsers();
        if (data_) munmap((void*) data_, size_);
        if (zdata_) munmap((void*) zdata_, zsize_);
    }
    // Launches the parser threads (parallel mode); a no-op when they run already or the input is read sequentially.
    void start() {
        if (!parallel() || !workers_.empty() || sequential_) return;
        for (int t = 0; t < threads_; ++t) workers_.emplace_back([this] { parse_loop(); });
    }
    // Allocates every pooled batch's buffers at the size a parser chunk needs (what parse_loop would reserve on first use),
    // so that no pinned allocation happens while the pipeline runs: the drivers call it while the index is being opened.
    void prewarm(bool packed) {
        if (!parallel()) return;
        std::lock_guard<std::mutex> l(m_);
        for (auto& b : pool_) reserve_for(*b, chunk_bytes_ + 4096, packed);
    }
    bool ok() const { return ok_; }
    int err() const { return err_; }            // kseq_read's final code: -1 end of input, -2, -3
    bool parallel() const { return data_ != nullptr || zdata_ != nullptr; }
    uint64_t fallbacks() const { return fallbacks_; }

    // Next batch in input order; nullptr at the end of input (then see err()).
    std::unique_ptr<ReadBatch> next() {
        while (parallel() && !sequential_) {
            if (want_ >= n_chunks_) {
                if (verified_ < size_) { start_sequential(verified_); break; }     // trailing bytes no chunk claimed
                err_ = -1;
                return nullptr;
            }
            std::unique_ptr<ReadBatch> b;
            {
                std::unique_lock<std::mutex> l(m_);
                done_cv_.wait(l, [&] { return done_.count(want_) != 0; });
                b = std::move(done_[want_]);
                done_.erase(want_);
            }
            ++want_;
            if (b->begin == b->end && !b->bailed && b->n == 0) {     // chunk without a record start
                recycle(std::move(b));
                continue;
            }
            if (b->begin != verified_) {                              // the guess was wrong
                recycle(std::move(b));
                start_sequential(verified_);
                break;
            }
            verified_ = b->end;
            const bool bailed = b->bailed;
            if (bailed) start_sequential(verified_);
            if (b->n == 0) { recycle(std::move(b)); if (bailed) break; continue; }
            b->id = next_id_++;
            return b;
        }
        // sequential kseq-compatible reader
        if (finished_) return nullptr;
        std::unique_ptr<ReadBatch> b = acquire();
        int r = 0;
        while (b->n < batch_reads_ && b->n_bases() < (256u << 20) && (r = seq_->next(name_, seqbuf_)) >= 0)
            b->add(name_.data(), strlen(name_.c_str()), seqbuf_.data(), strlen(seqbuf_.c_str()));     // both are printed / searched as C strings
        if (r < 0) { err_ = r; finished_ = true; }
        if (b->n == 0) { recycle(std::move(b)); return nullptr; }
        if (on_batch_) on_batch_(*b);
        b->id = next_id_++;
        return b;
    }

    void recycle(std::unique_ptr<ReadBatch> b) {
        b->clear();
        std::lock_guard<std::mutex> l(m_);
        pool_.push_back(std::move(b));
        pool_cv_.notify_one();
    }

  private:
    std::unique_ptr<ReadBatch> acquire() {
        std::unique_lock<std::mutex> l(m_);
        pool_cv_.wait(l, [&] { return !pool_.empty() || stop_; });
        if (pool_.empty()) return nullptr;
        std::unique_ptr<ReadBatch> b = std::move(pool_.back());
        pool_.pop_back();
        return b;
    }

    static bool is_space(unsigned char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }

    // What a chunk parser reads: bytes [lo, hi) of the input, addressed by their position in the input (d + p is byte p).  The
    // mmap'ed plain file is one view of everything; a BGZF chunk's view is the thread's private buffer of inflated blocks.
    struct View {
        const char* d;
        size_t lo, hi;
        bool to_end;                    // hi is the end of the input (a last record may end without a newline)
    };

    // First position >= from that looks like the start of a four-line record; v.hi when the view holds none.
    size_t guess_start(const View& v, size_t from) const {
        if (from == 0) return 0;
        if (from >= v.hi) return v.hi;
        const char* data = v.d;
        const size_t size = v.hi;
        const char* p = (const char*) memchr(data + from - 1, '\n', size - (from - 1));
        size_t pos = p ? (size_t) (p - data) + 1 : size;
        while (pos < size && !stop_.load(std::memory_order_relaxed)) {
            const char* e1 = (const char*) memchr(data + pos, '\n', size - pos);
            if (!e1) return size;
            if (data[pos] == '@') {
                const size_t l1 = (size_t) (e1 - data) + 1;
                const char* e2 = l1 < size ? (const char*) memchr(data + l1, '\n', size - l1) : nullptr;
                if (!e2) return size;
                const size_t l2 = (size_t) (e2 - data) + 1;
                if (l2 < size && data[l2] == '+' && data[l1] != '@') return pos;
            }
            pos = (size_t) (e1 - data) + 1;
        }
        return size;
    }

    // Strict four-line records starting at b.begin while they start before `limit`.
    void parse_strict(ReadBatch& b, const View& view, size_t limit) const {
        size_t p = b.begin;
        const char* d = view.d;
        const size_t size = view.hi;
        while (p < limit) {
            if (d[p] != '@') break;
            const char* h = (const char*) memchr(d + p + 1, '\n', size - p - 1);
            if (!h) break;
            size_t nm = p + 1;
            while (!is_space((unsigned char) d[nm])) ++nm;           // stops at the '\n' at the latest
            const size_t s = (size_t) (h - d) + 1;
            if (s >= size) break;
            const char* e = (const char*) memchr(d + s, '\n', size - s);
            if (!e) break;
            const size_t len = (size_t) (e - d) - s;
            if (len == 0 || d[s] == '>' || d[s] == '+' || d[s] == '@' || e[-1] == '\r') break;
            const size_t t = (size_t) (e - d) + 1;
            if (t >= size || d[t] != '+') break;
            const char* u = (const char*) memchr(d + t, '\n', size - t);
            if (!u) break;
            const size_t v = (size_t) (u - d) + 1;
            if (v + len > size) break;
            const char* w = (const char*) memchr(d + v, '\n', size - v);
            if (!w && !view.to_end) break;                            // the view ends inside the record, the input does not
            const size_t qend = w ? (size_t) (w - d) : size;
            if (qend - v != len) break;
            const size_t nxt = w ? qend + 1 : size;
            if (nxt >= size && !view.to_end) break;                   // what follows the record lies outside the view
            if (nxt < size && d[nxt] != '@') {
                // kseq would skip ahead to the next '@' or '>': leave that to the sequential reader,
                // but this record is complete and unambiguous
                const void* z = memchr(d + s, 0, len);
                b.add(d + p + 1, strnlen(d + p + 1, nm - p - 1), d + s, z ? (size_t) ((const char*) z - (d + s)) : len);
                p = nxt;
                b.end = p;
                b.bailed = true;
                return;
            }
            const void* z = memchr(d + s, 0, len);                   // seq->seq.s is used as a C string
            b.add(d + p + 1, strnlen(d + p + 1, nm - p - 1), d + s, z ? (size_t) ((const char*) z - (d + s)) : len);
            p = nxt;
        }
        b.end = p;
        b.bailed = p < limit;
    }

    // BGZF: inflates the blocks under bytes [want_lo, want_hi) of the inflated stream into buf; the view covers whole blocks.
    // false: a block does not inflate to what its header and CRC say (the sequential reader will report it in its place).
    bool inflate_view(size_t want_lo, size_t want_hi, std::vector<char>& buf, View& v) const {
        const size_t nb = bz_coff_.size() - 1;
        size_t first = (size_t) (std::upper_bound(bz_uoff_.begin(), bz_uoff_.end(), (uint64_t) want_lo) - bz_uoff_.begin()) - 1;
        if (first >= nb) first = nb - 1;
        size_t last = first;                                          // one past the last block needed
        while (last < nb && bz_uoff_[last] < want_hi) ++last;
        v.lo = (size_t) bz_uoff_[first];
        v.hi = (size_t) bz_uoff_[last];
        v.to_end = v.hi == size_;
        if (buf.size() < v.hi - v.lo + 1) buf.resize(v.hi - v.lo + 1);
        for (size_t j = first; j < last; ++j) {
            if (stop_.load(std::memory_order_relaxed)) return false;
            if (!BgzfSource::inflate_block(zdata_ + bz_coff_[j], (size_t) (bz_coff_[j + 1] - bz_coff_[j]), buf.data() + (bz_uoff_[j] - v.lo),
                                           (uint32_t) (bz_uoff_[j + 1] - bz_uoff_[j])))
                return false;
        }
        v.d = buf.data() - v.lo;                                     // only ever dereferenced at positions in [lo, hi)
        return true;
    }

    // one allocation per buffer for typical records (150 bp reads: ~half of the bytes are bases, >= 96 bytes per record), not a growth ladder
    static void reserve_for(ReadBatch& b, size_t est, bool packed) {
        b.bases.reserve(est / 2 + 64, 0);
        b.offs.reserve(est / 96 + 1024, 1);
        if (packed) {
            b.packed.reserve((est / 2 + 64) / 32 + 2, 0);
            b.flags.reserve(est / 96 + 1024 + 8, 0);
        }
    }

    void parse_loop() {
        // parsing is the stage that can wait: the formatter threads and the GPU worker of the same process share the cores
        // with these threads, and a batch parsed early only sits in the queue (per-thread nice on Linux)
        setpriority(PRIO_PROCESS, (id_t) syscall(SYS_gettid), 10);
        std::vector<char> inflated;                              // BGZF: this thread's view of the inflated stream
        for (;;) {
            std::unique_ptr<ReadBatch> b = acquire();            // buffer first, then the lowest free chunk: no deadlock
            if (!b) return;
            const size_t k = claim_.fetch_add(1);
            if (k >= n_chunks_ || stop_) { recycle(std::move(b)); return; }
            View v{data_, 0, size_, true};
            bool readable = true;
            if (zdata_) {
                // the byte in front of the chunk (guess_start looks at it) up to a margin behind it: the record that starts
                // before the chunk's end, the three lines guess_start reads behind the next chunk's start
                const size_t lo = k ? k * chunk_bytes_ - 1 : 0;
                readable = inflate_view(lo, std::min(size_, (k + 1) * chunk_bytes_ + view_margin_), inflated, v);
            }
            if (readable) {
                b->begin = guess_start(v, k * chunk_bytes_);
                const size_t limit = k + 1 < n_chunks_ ? guess_start(v, (k + 1) * chunk_bytes_) : size_;
                b->end = b->begin;
                reserve_for(*b, limit > b->begin ? limit - b->begin : 0, false);
                if (b->begin < limit) parse_strict(*b, v, limit);
            } else {
                b->begin = b->end = size_ + 1;                       // never equals a verified position: next() falls back from there
                b->bailed = true;
            }
            if (on_batch_ && b->n) on_batch_(*b);
            {
                std::lock_guard<std::mutex> l(m_);
                done_[k] = std::move(b);
            }
            done_cv_.notify_all();
        }
    }

    void stop_parsers() {
        {
            std::lock_guard<std::mutex> l(m_);
            stop_ = true;
        }
        pool_cv_.notify_all();
        for (auto& t : workers_) t.join();
        workers_.clear();
        std::lock_guard<std::mutex> l(m_);
        for (auto& kv : done_) { kv.second->clear(); pool_.push_back(std::move(kv.second)); }
        done_.clear();
        stop_ = false;
    }

    void start_sequential(size_t pos) {
        stop_parsers();
        sequential_ = true;
        ++fallbacks_;
        seq_.reset(new FastxReader(path_.c_str(), threads_));
        if (!seq_->ok() || !seq_->seek(pos)) { err_ = -3; finished_ = true; }
    }

    std::string path_;
    HostAlloc alloc_;
    size_t batch_reads_;
    int threads_ = 0;
    std::function<void(ReadBatch&)> on_batch_;
    bool ok_ = false;
    int err_ = -1;
    // parallel mode
    size_t view_margin_ = 1u << 20;              // BGZF views: bytes inflated behind the chunk's end (RBG_VIEW_MARGIN: tests)
    bool margin_forced_ = false;
    const char* data_ = nullptr;                 // plain file
    const unsigned char* zdata_ = nullptr;       // BGZF file (compressed bytes) + its block table; size_ = inflated size
    size_t zsize_ = 0;
    std::vector<uint64_t> bz_coff_, bz_uoff_;
    size_t size_ = 0, chunk_bytes_ = 0, n_chunks_ = 0;
    std::vector<std::thread> workers_;
    std::atomic<size_t> claim_{0};
    std::mutex m_;
    std::condition_variable pool_cv_, done_cv_;
    std::vector<std::unique_ptr<ReadBatch>> pool_;
    std::map<size_t, std::unique_ptr<ReadBatch>> done_;
    std::atomic<bool> stop_{false};
    size_t want_ = 0, verified_ = 0;
    uint64_t next_id_ = 0, fallbacks_ = 0;
    // sequential mode
    bool sequential_ = false, finished_ = false;
    std::unique_ptr<FastxReader> seq_;
    std::string name_, seqbuf_;
};

}  // namespace rbhost
