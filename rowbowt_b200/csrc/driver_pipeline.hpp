// The host pipeline of the query drivers (rb_align, rb_markers):
//
//   parser threads (fastx_parallel.hpp) ──► GPU workers ──► formatter pool ──► ordered writer
//
// Each driver supplies its query call, its result type and its formatter.  No collective: batches are independent
// (SURVEY.md §8(e)).
#pragma once
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rowbowt_gpu.h"
#include "fastx_parallel.hpp"
#include "host_io.hpp"

namespace rbhost {

// RBG_HOST_STATS=1: busy seconds of every stage of the host pipeline on stderr (before the driver's timing line)
struct StageClock {
    std::atomic<uint64_t> ns{0};
    struct Scope {
        StageClock& c;
        std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
        ~Scope() { c.ns += (uint64_t) std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count(); }
    };
    double s() const { return (double) ns.load() * 1e-9; }
};

// Result: what one query call fills (rbg_result, rbg_seed_result); the pipeline frees it after its last slice is formatted.
template <class Result>
class QueryPipeline {
  public:
    struct Options {
        std::string fastq;
        int threads = 1;                // parser threads, and as many formatter threads
        size_t chunk_bytes = 0;         // FASTQ bytes per parser chunk = GPU batch (0: from the file size)
        size_t batch_reads = 1;         // reads per batch of the sequential reader
        int gpus = 1;                   // devices asked for
        int workers_per_gpu = 1;        // the driver's default; RBG_WORKERS_PER_GPU overrides
        int slice_shift = 12;           // a formatter slice holds at least 2^slice_shift reads
        // Runs on the parser thread that completed a batch, with device 0's handle: rb_align packs the bases to 2 bits
        // there.  When it is set only the packed form crosses PCIe, so the raw bases go to pageable memory.
        std::function<void(rbg_index*, ReadBatch&)> pack;
    };
    using Query = std::function<void(rbg_index*, ReadBatch&, Result&)>;
    using Format = std::function<void(const Result&, const ReadBatch&, uint64_t i0, uint64_t i1, OutBuf&)>;

    explicit QueryPipeline(Options o) : o_(std::move(o)) {}
    ~QueryPipeline() {
        if (prewarm_.joinable()) prewarm_.join();
        close_handles();
    }

    // Sets the batch source up and opens one handle per device, in parallel; after_open (optional) runs on the thread that
    // opened a handle.  The source parses nothing before run(): only its pinned buffers are allocated meanwhile, on a thread
    // of their own -- pinning is ~0.3 ms per MB under the CUDA context lock, which must not happen while a GPU worker is
    // issuing copies and launches.  Returns 0, or the code of the first handle that failed with its rbg_last_error(), which
    // is thread-local and so read on the thread that opened the handle.
    int open(const char* prefix, uint32_t flags, const std::function<int(rbg_index*)>& after_open, std::string& msg) {
        const int ndev = rbg_device_count();
        if (ndev <= 0) {
            msg = "no CUDA device available (this build has no CPU path)";
            return RBG_E_CUDA;
        }
        // RBG_GPU_MODULO=1 (tests on a box with fewer devices): worker g shares the handle of device g % ndev -- calls on one
        // handle run concurrently -- so that the ordered reassembly of a multi-worker run is exercised anywhere; otherwise the
        // request is clamped to the visible devices.
        const bool modulo = getenv("RBG_GPU_MODULO") && atoi(getenv("RBG_GPU_MODULO")) > 0;
        const int n_gpus = modulo ? o_.gpus : std::min(o_.gpus, ndev);
        const char* wpg = getenv("RBG_WORKERS_PER_GPU");
        workers_ = n_gpus * (wpg ? std::max(1, std::min(4, atoi(wpg))) : o_.workers_per_gpu);
        idx_.assign(std::min(n_gpus, ndev), nullptr);
        pool_ = 2 * (size_t) o_.threads + 6 * (size_t) workers_ + 4;
        const HostAlloc pinned{rbg_host_alloc, rbg_host_free}, pageable{malloc, free};
        std::function<void(ReadBatch&)> on_batch;
        if (o_.pack)
            on_batch = [this](ReadBatch& b) {
                StageClock::Scope sc{clk_pack_};
                o_.pack(idx_[0], b);
            };
        src_.reset(new FastxBatchSource(o_.fastq.c_str(), o_.threads, o_.chunk_bytes, o_.batch_reads, pinned, pool_, on_batch,
                                        /*start=*/false, o_.pack ? &pageable : nullptr));
        prewarm_ = std::thread([this] { if (src_->ok()) src_->prewarm((bool) o_.pack); });
        const int n = (int) idx_.size();
        std::vector<std::thread> th;
        std::vector<int> rc(n, 0);
        std::vector<std::string> err(n);
        for (int g = 0; g < n; ++g)
            th.emplace_back([&, g] {
                rc[g] = rbg_index_open(prefix, flags, g, &idx_[g]);
                if (!rc[g] && after_open) rc[g] = after_open(idx_[g]);
                if (rc[g]) err[g] = rbg_last_error();
            });
        for (auto& t : th) t.join();
        for (int g = 0; g < n; ++g)
            if (rc[g]) {
                msg = err[g];
                return rc[g];
            }
        return 0;
    }

    // Waits for the prewarmed buffers.  false: the FASTQ cannot be read (the drivers report it after the load, as the
    // reference does).
    bool finish_load() {
        prewarm_.join();
        return src_->ok();
    }

    // Queries, formats and writes the whole input in input order; feed (optional) runs on the calling thread on every batch,
    // in input order, before the batch goes to a GPU worker.  Ends with the reference's exits on a truncated or unreadable
    // input, after the handles are closed.  Returns the seconds from the first parsed byte to the last written one.
    double run(const Query& query, void (*free_result)(Result*), const Format& format,
               const std::function<void(ReadBatch&)>& feed = nullptr) {
        using clk = std::chrono::high_resolution_clock;
        const auto q0 = clk::now();
        FastxBatchSource& src = *src_;
        src.start();
        StageClock clk_query, clk_format, clk_write, clk_wait_gpu, clk_next;
        uint64_t n_batches = 0, n_reads_total = 0;

        struct Job {                                   // one batch between its query and its last formatted slice
            std::unique_ptr<ReadBatch> b;
            Result res{};
            std::atomic<int> left{0};
            int gpu = 0;
        };
        struct Slice { Job* job; int s; uint64_t i0, i1; };
        Channel<std::unique_ptr<ReadBatch>> to_gpu(2 * (size_t) workers_), to_writer(pool_);
        Channel<Slice> to_format(64 * (size_t) o_.threads);
        std::mutex inflight_m;
        std::condition_variable inflight_cv;
        std::vector<int> inflight(workers_, 0);        // results of worker g not yet freed (the library pools 4)

        std::vector<std::thread> workers, formatters;
        for (int g = 0; g < workers_; ++g)
            workers.emplace_back([&, g] {
                std::unique_ptr<ReadBatch> b;
                while (to_gpu.pop(b)) {
                    {
                        std::unique_lock<std::mutex> l(inflight_m);
                        inflight_cv.wait(l, [&] { return inflight[g] < 3; });
                        ++inflight[g];
                    }
                    Job* job = new Job;
                    StageClock::Scope sq{clk_query};
                    query(idx_[g % idx_.size()], *b, job->res);
                    job->gpu = g;
                    const uint64_t n = b->n;
                    const int slices = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) o_.threads, n >> o_.slice_shift));
                    if (b->text.size() < (size_t) slices) b->text.resize(slices);
                    b->n_text = (size_t) slices;
                    job->b = std::move(b);
                    job->left = slices;
                    for (int s = 0; s < slices; ++s)
                        to_format.push(Slice{job, s, n * (uint64_t) s / slices, n * (uint64_t) (s + 1) / slices});
                }
            });
        for (int t = 0; t < o_.threads; ++t)
            formatters.emplace_back([&] {
                Slice sl;
                while (to_format.pop(sl)) {
                    Job* job = sl.job;
                    {
                        StageClock::Scope sf{clk_format};
                        format(job->res, *job->b, sl.i0, sl.i1, job->b->text[sl.s]);
                    }
                    if (job->left.fetch_sub(1) == 1) {
                        const int g = job->gpu;
                        free_result(&job->res);
                        {
                            std::lock_guard<std::mutex> l(inflight_m);
                            --inflight[g];
                        }
                        inflight_cv.notify_all();
                        to_writer.push(std::move(job->b));
                        delete job;
                    }
                }
            });
        // Ordered output.  A pipe / terminal / O_APPEND stdout gets one write(2) after the other from this thread.  When stdout is
        // a regular file (the usual `rb_align ... > report.txt`; with -s that is 1.4 KB per read) the order is only a matter of
        // OFFSETS: this thread hands every slice of the next batch its place in the file and a few writer threads pwrite(2) them
        // concurrently -- one thread copying into the page cache moved 2.3 GB/s, a third of what the formatters produce.
        struct WriteTask { ReadBatch* b; size_t k; off_t at; };
        struct stat out_st;
        const int out_fl = fcntl(1, F_GETFL);
        const off_t out_pos = lseek(1, 0, SEEK_CUR);
        const bool positional = !(getenv("RBG_SEQ_WRITE") && atoi(getenv("RBG_SEQ_WRITE")) > 0) && fstat(1, &out_st) == 0 &&
                                S_ISREG(out_st.st_mode) && out_fl >= 0 && !(out_fl & O_APPEND) && out_pos >= 0;
        const int n_writers = positional ? std::max(1, std::min(4, o_.threads / 2)) : 0;
        Channel<WriteTask> to_pwrite(256);
        std::mutex left_m;
        std::map<ReadBatch*, std::pair<size_t, std::unique_ptr<ReadBatch>>> writing;      // batch -> (slices not yet written, owner)
        std::vector<std::thread> pwriters;
        for (int t = 0; t < n_writers; ++t)
            pwriters.emplace_back([&] {
                WriteTask w;
                while (to_pwrite.pop(w)) {
                    {
                        StageClock::Scope sw{clk_write};
                        const char* p = w.b->text[w.k].p;
                        size_t left = w.b->text[w.k].len;
                        off_t at = w.at;
                        while (left) {
                            const ssize_t n = pwrite(1, p, left, at);
                            if (n < 0) { if (errno == EINTR) continue; perror("pwrite"); exit(1); }
                            p += n; at += n; left -= (size_t) n;
                        }
                    }
                    std::unique_ptr<ReadBatch> done;
                    {
                        std::lock_guard<std::mutex> l(left_m);
                        auto it = writing.find(w.b);
                        if (--it->second.first == 0) { done = std::move(it->second.second); writing.erase(it); }
                    }
                    if (done) src.recycle(std::move(done));
                }
            });
        std::thread writer([&] {
            std::map<uint64_t, std::unique_ptr<ReadBatch>> pending;
            uint64_t next = 0;
            off_t at = out_pos;
            std::unique_ptr<ReadBatch> b;
            while (to_writer.pop(b)) {
                pending[b->id] = std::move(b);
                for (auto it = pending.find(next); it != pending.end(); it = pending.find(next)) {
                    if (positional) {
                        ReadBatch* rbp = it->second.get();
                        std::vector<WriteTask> tasks;
                        for (size_t k = 0; k < rbp->n_text; ++k) {
                            if (rbp->text[k].len) tasks.push_back(WriteTask{rbp, k, at});
                            at += (off_t) rbp->text[k].len;
                        }
                        if (tasks.empty()) {
                            src.recycle(std::move(it->second));
                        } else {
                            {
                                std::lock_guard<std::mutex> l(left_m);
                                writing[rbp] = std::make_pair(tasks.size(), std::move(it->second));
                            }
                            for (const WriteTask& w : tasks) to_pwrite.push(w);
                        }
                    } else {
                        {
                            StageClock::Scope sw{clk_write};
                            for (size_t k = 0; k < it->second->n_text; ++k) write_all(1, it->second->text[k].p, it->second->text[k].len);
                        }
                        src.recycle(std::move(it->second));
                    }
                    pending.erase(it);
                    ++next;
                }
            }
            to_pwrite.close();
            for (auto& t : pwriters) t.join();
            if (positional && lseek(1, at, SEEK_SET) < 0) { perror("lseek"); exit(1); }       // whatever is written next continues behind the report
        });

        for (;;) {
            std::unique_ptr<ReadBatch> b;
            {
                StageClock::Scope sn{clk_next};
                b = src.next();
            }
            if (!b) break;
            ++n_batches;
            n_reads_total += b->n;
            if (feed) feed(*b);
            StageClock::Scope sg{clk_wait_gpu};
            to_gpu.push(std::move(b));
        }
        const int err = src.err();
        to_gpu.close();
        for (auto& w : workers) w.join();
        to_format.close();
        for (auto& f : formatters) f.join();
        to_writer.close();
        writer.join();
        const std::chrono::duration<double> query_time = clk::now() - q0;
        if (getenv("RBG_HOST_STATS"))
            fprintf(stderr, "host stages (busy seconds, summed over threads): pack %.3f  rbg_query %.3f  format %.3f  write %.3f | main thread: "
                    "waiting for parsed batches %.3f, waiting for a GPU worker %.3f | %llu batches, %llu reads, %d parser/formatter threads, %d GPU workers\n",
                    clk_pack_.s(), clk_query.s(), clk_format.s(), clk_write.s(), clk_next.s(), clk_wait_gpu.s(),
                    (unsigned long long) n_batches, (unsigned long long) n_reads_total, o_.threads, workers_);
        close_handles();
        switch (err) {           // src/rb_align.cpp:181-191, src/rb_markers.cpp:584-593
            case -2: fprintf(stderr, "ERROR: truncated quality string\n"); exit(1);
            case -3: fprintf(stderr, "ERROR: error reading stream\n"); exit(1);
            default: break;
        }
        return query_time.count();
    }

  private:
    void close_handles() {
        for (auto*& ix : idx_)
            if (ix) { rbg_index_close(ix); ix = nullptr; }
    }

    Options o_;
    std::vector<rbg_index*> idx_;
    int workers_ = 0;                   // GPU workers; worker g calls on the handle of device g % idx_.size()
    size_t pool_ = 0;                   // batches in flight between the parsers and the writer
    std::unique_ptr<FastxBatchSource> src_;
    std::thread prewarm_;
    StageClock clk_pack_;
};

}  // namespace rbhost
