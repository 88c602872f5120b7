// rb_markers — drop-in host driver of the greedy-seeding marker genotyping over librowbowt_gpu
// (C ABI).  Same command line, index files (.rbwt/.mab[/.ftab]) and stdout grammar as the
// reference driver (src/rb_markers.cpp); the per-read worker body (:375-404) runs on the GPU a
// batch at a time through rbg_markers_greedy, both strands of every read.
//
// Output order: the reference prints each worker thread's buffer whenever it exceeds 4 KB, so its
// line order depends on thread scheduling; this driver always prints reads in input order, which
// is the reference's order at --threads 1.
//
// Not offered: --lmem (experimental O(m^2) path that logs every step to stderr), --overlap (the
// reference itself exits with "overlapped seeds currently broken").
#include <getopt.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <memory>
#include <random>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rowbowt_gpu.h"
#include "driver_pipeline.hpp"

namespace {

struct Args {                       // RbAlignArgs, src/rb_markers.cpp:21-39
    std::string inpre, fastq;
    int ftab = 0, fbb = 0, overlap = 0, lmem = 0;
    int layout_cache = 0;           // keep / use <index_prefix>.rbgcache (RBG_LOAD_CACHE)
    size_t wsize = 19, max_range = 1000, min_range = 0, threads = 1, max_tasks = 1024, read_len = 101, min_seed_len = 0;
    int clear_conflicting = 0, clear_identical = 0, best_strand = 0, heuristic = 0;
    int gpus = 1;
    size_t batch_reads = 1u << 18;
};

void print_help() {
    fprintf(stderr, "rb_markers\n");
    fprintf(stderr, "Usage: rb_markers_only [options] <index_prefix> <input_fastq_name>\n");
    fprintf(stderr, "    --wsize            <int>         window size for performing marker queries along read\n");
    fprintf(stderr, "    --max-range        <int>         range-size upper threshold for performing marker queries\n");
    fprintf(stderr, "    --min-range        <int>         range-size upper threshold for performing marker queries\n");
    fprintf(stderr, "    --ftab                           seed through <index_prefix>.ftab\n");
    fprintf(stderr, "    --layout-cache                   keep the GPU layout in <index_prefix>.rbgcache and open from it when it is current\n");
    fprintf(stderr, "    --heuristic [--best-strand-only --min-seed-length <int> --clear-conflicting --clear-identical --read-len <int>]\n");
    fprintf(stderr, "    --gpus <N> --batch <reads>       GPUs to use (index replicated), reads per batch\n");
    fprintf(stderr, "    <input_prefix>                   index prefix\n");
    fprintf(stderr, "    <input_fastq>                    input fastq\n");
}

Args parse_args(int argc, char** argv) {
    Args a;
    static struct option lopts[] = {{"wsize", required_argument, 0, 'w'},
                                    {"max-range", required_argument, 0, 'r'},
                                    {"min-range", required_argument, 0, 'm'},
                                    {"threads", required_argument, 0, 't'},
                                    {"max-tasks", required_argument, 0, 'u'},
                                    {"read-len", required_argument, 0, 'l'},
                                    {"fbb", no_argument, &a.fbb, 1},
                                    {"ftab", no_argument, &a.ftab, 1},
                                    {"layout-cache", no_argument, &a.layout_cache, 1},
                                    {"overlap", no_argument, &a.overlap, 1},
                                    {"lmem", no_argument, &a.lmem, 1},
                                    {"heuristic", no_argument, &a.heuristic, 1},
                                    {"best-strand-only", no_argument, &a.best_strand, 1},
                                    {"min-seed-length", required_argument, 0, 'y'},
                                    {"clear-conflicting", no_argument, &a.clear_conflicting, 1},
                                    {"clear-identical", no_argument, &a.clear_identical, 1},
                                    {"gpus", required_argument, 0, 'g'},
                                    {"batch", required_argument, 0, 'b'},
                                    {0, 0, 0, 0}};
    int c, li = 0;
    while ((c = getopt_long(argc, argv, "o:w:r:hft:m:u:xl:y:g:b:", lopts, &li)) != -1) {
        switch (c) {
            case 0: break;
            case 'y': a.min_seed_len = std::atol(optarg); break;
            case 'l': a.read_len = std::atol(optarg); break;
            case 't': a.threads = std::atol(optarg); break;         // here: host parser + formatter threads (the GPU replaces the worker pool)
            case 'u': a.max_tasks = std::atol(optarg); break;
            case 'f': a.ftab = 1; break;
            case 'r': a.max_range = std::atol(optarg); break;
            case 'm': a.min_range = std::atol(optarg); break;
            case 'w': a.wsize = std::atol(optarg); break;
            case 'o': break;
            case 'h': print_help(); exit(0);
            case 'x': a.fbb = 1; break;
            case 'g': a.gpus = std::max(1, atoi(optarg)); break;
            case 'b': a.batch_reads = (size_t) std::max(1ll, atoll(optarg)); break;
            default: print_help(); exit(1);
        }
    }
    if (a.overlap) {                        // src/rb_markers.cpp:119-122
        fprintf(stderr, "overlapped seeds currently broken\n");
        exit(1);
    }
    if (a.lmem) {
        fprintf(stderr, "--lmem is not offered by the GPU driver\n");
        exit(1);
    }
    if (argc - optind < 2) {
        fprintf(stderr, "no argument provided\n");
        exit(1);
    }
    a.inpre = argv[optind++];
    a.fastq = argv[optind++];
    return a;
}

// MarkerT accessors, pfbwt-f/include/marker.hpp:7-37
inline uint64_t m_seq(uint64_t m) { return (m & 0x0FFFF00000000000ull) >> 46; }
inline uint64_t m_pos(uint64_t m) { return m & 0x00000FFFFFFFFFFFull; }
inline uint64_t m_allele(uint64_t m) { return (m & 0xF000000000000000ull) >> 60; }

using rbhost::ReadBatch;

struct Seed {                           // MarkerSeed, src/rb_markers.cpp:255-300
    int strand;                         // 0 = '+', 1 = '-'
    uint64_t range_size, query_start, query_len;
    std::vector<uint64_t> markers;
};

// MarkerSeed::print_buf :262-272
void print_seed(std::string& o, const char* name, size_t name_len, uint64_t range_size, int strand, uint64_t query_start,
                uint64_t query_len, const uint64_t* mk, size_t n_mk) {
    o.append(name, name_len);
    o += ' ';
    rbhost::put_u64(o, range_size);
    o += strand ? " - " : " + ";
    rbhost::put_u64(o, query_start);
    o += ' ';
    rbhost::put_u64(o, query_len);
    for (size_t k = 0; k < n_mk; ++k) {
        o += ' ';
        rbhost::put_u64(o, m_seq(mk[k]));
        o += '/';
        rbhost::put_u64(o, m_pos(mk[k]));
        o += '/';
        rbhost::put_u64(o, m_allele(mk[k]));
    }
    if (!n_mk) o += " .";
    o += '\n';
}

uint64_t seed_query_start(const rbg_seed& g) { return g.query_start == 0xFFFFFFFFu ? ~0ull : g.query_start; }      // the reference's size_t(-1)

Seed make_seed(const rbg_seed_result& r, uint64_t j, int strand) {
    const rbg_seed& g = r.seeds[j];
    Seed s;
    s.strand = strand;
    s.range_size = g.hi - g.lo + 1;
    s.query_start = seed_query_start(g);
    s.query_len = g.query_len;
    s.markers.assign(r.markers + g.mk_off, r.markers + g.mk_off + g.mk_cnt);
    return s;
}

// MarkerSeed::filter_identical_pos, src/rb_markers.cpp:276-288 (markers sorted)
void filter_identical_pos(std::vector<uint64_t>& mk) {
    if (mk.empty()) return;
    uint64_t pm = 0;
    std::vector<uint64_t> keep;
    for (size_t i = 0; i < mk.size(); ++i) {
        const uint64_t m = mk[i];
        if (m_seq(m) == m_seq(pm) && m_pos(m) == m_pos(pm)) continue;
        pm = m;
        if (i + 1 < mk.size() && m_seq(mk[i + 1]) == m_seq(m) && m_pos(mk[i + 1]) == m_pos(m)) continue;
        keep.push_back(m);
    }
    mk.swap(keep);
}

// MarkerSeed::clear_if_conflicting, :291-296
void clear_if_conflicting(std::vector<uint64_t>& mk, size_t read_len) {
    if (mk.empty()) return;
    if (m_seq(mk.back()) != m_seq(mk.front()) || m_pos(mk.back()) - m_pos(mk.front()) >= read_len) mk.clear();
}

// The report of reads [i0, i1) of one batch, built in a string of the formatter thread (it keeps its capacity from slice
// to slice) and copied into the slice's buffer.
void format_slice(const Args& a, const rbg_seed_result& r, const ReadBatch& b, uint64_t i0, uint64_t i1, rbhost::OutBuf& out) {
    thread_local std::string o;
    o.clear();
    o.reserve((size_t) ((r.seed_off[2 * i1] - r.seed_off[2 * i0]) * 40 + (i1 - i0) * 16));
    std::vector<Seed> seeds;
    for (uint64_t i = i0; i < i1; ++i) {
        size_t nl;
        const char* nm = b.name(i, nl);
        if (!a.heuristic) {                                     // worker, :347-415
            for (int s = 0; s < 2; ++s)                         // straight from the result arrays: ~10 seeds per read
                for (uint64_t j = r.seed_off[2 * i + s]; j < r.seed_off[2 * i + s + 1]; ++j) {
                    const rbg_seed& g = r.seeds[j];
                    print_seed(o, nm, nl, g.hi - g.lo + 1, s, seed_query_start(g), g.query_len, r.markers + g.mk_off, g.mk_cnt);
                }
            continue;
        }
        // worker_heuristic, :416-507: a random strand first, the other one only if no seed of the first asked to stop
        seeds.clear();
        bool stop = false;
        const int first = b.aux[i] ? 1 : 0;
        for (int pass = 0; pass < 2 && !(pass == 1 && stop); ++pass) {
            const int s = pass == 0 ? first : 1 - first;
            for (uint64_t j = r.seed_off[2 * i + s]; j < r.seed_off[2 * i + s + 1]; ++j) {
                Seed ms = make_seed(r, j, s);
                if (ms.query_len < a.min_seed_len) continue;
                if (a.clear_conflicting) clear_if_conflicting(ms.markers, a.read_len);
                if (a.clear_identical) filter_identical_pos(ms.markers);
                const uint64_t used = ms.query_start + ms.query_len;
                seeds.push_back(std::move(ms));
                if (a.best_strand && (uint64_t) a.read_len - used < a.min_seed_len) stop = true;
            }
        }
        if (a.best_strand && !seeds.empty()) {                  // SeedVec::keep_seeds_best_strand, :306-325
            size_t best = 0;
            for (size_t k = 1; k < seeds.size(); ++k)
                if (seeds[best].query_len < seeds[k].query_len) best = k;
            const int strand = seeds[best].strand;
            std::vector<Seed> kept;
            for (auto& s : seeds)
                if (s.strand == strand) kept.push_back(std::move(s));
            seeds.swap(kept);
        }
        for (const Seed& s : seeds) print_seed(o, nm, nl, s.range_size, s.strand, s.query_start, s.query_len, s.markers.data(), s.markers.size());
    }
    out.reserve(o.size());
    if (!o.empty()) memcpy(out.p, o.data(), o.size());
    out.len = o.size();
}

}  // namespace

int main(int argc, char** argv) {
    Args args = parse_args(argc, argv);
    using clk = std::chrono::high_resolution_clock;
    auto t0 = clk::now();
    std::cerr << "(gpu) loading rowbowt + markers";
    if (args.ftab) std::cerr << " and ftab";
    std::cerr << std::endl;
    const uint32_t flags = RBG_LOAD_MA | (args.ftab ? RBG_LOAD_FT : 0) | (args.fbb ? RBG_LOAD_FBB : 0) | (args.layout_cache ? RBG_LOAD_CACHE : 0);       // load_rbwt, src/rb_markers.cpp:534-542
    rbhost::QueryPipeline<rbg_seed_result>::Options po;
    po.fastq = args.fastq;
    po.threads = args.threads > 1 ? (int) args.threads : (int) std::max(1u, std::thread::hardware_concurrency());
    po.batch_reads = args.batch_reads;
    po.gpus = args.gpus;
    po.workers_per_gpu = 1;
    po.slice_shift = 11;
    rbhost::QueryPipeline<rbg_seed_result> pipe(std::move(po));
    std::string msg;
    if (pipe.open(args.inpre.c_str(), flags, nullptr, msg)) {
        std::cerr << msg << std::endl;
        return 1;
    }
    const bool input_ok = pipe.finish_load();
    std::chrono::duration<double> diff = clk::now() - t0;
    std::cerr << "loading rowbowt + markers took: " << diff.count() << " seconds\n";
    if (!input_ok) {
        fprintf(stderr, "invalid file\n");
        return 1;
    }
    const rbg_greedy_params gp{args.wsize, args.max_range, args.min_range, (uint32_t) args.ftab, 0};
    // RandomBoolGenerator, src/rb_markers.cpp:225-240: one bit per read IN INPUT ORDER, 32 per draw of a default-seeded
    // mt19937 -- batches leave the source in input order, so the bits are dealt on the one thread that sees them all
    std::mt19937 rng;
    uint32_t bits = 0;
    int bit_count = 0;
    const double counting = pipe.run(
        [&](rbg_index* ix, ReadBatch& b, rbg_seed_result& res) {
            rbg_batch in{b.n, b.bases.p, b.offs.p};
            if (rbg_markers_greedy(ix, &in, &gp, &res) != RBG_OK) {
                // the reference exits (k - 1 > wsize) or dies on an uncaught std::out_of_range (read shorter than k) here
                fprintf(stderr, "ERROR: %s\n", rbg_last_error());
                exit(1);
            }
        },
        rbg_seed_result_free,
        [&](const rbg_seed_result& res, const ReadBatch& b, uint64_t i0, uint64_t i1, rbhost::OutBuf& out) { format_slice(args, res, b, i0, i1, out); },
        [&](ReadBatch& b) {
            if (!args.heuristic) return;
            b.aux.resize(b.n);
            for (uint64_t i = 0; i < b.n; ++i) {
                if (bit_count == 0) { bits = (uint32_t) rng(); bit_count = 32; }
                b.aux[i] = (bits & 1u) ? 0 : 1;                // get_bool() ? FWD : REV
                bits >>= 1;
                --bit_count;
            }
        });
    std::cerr << "counting markers took: " << counting << " seconds" << std::endl;
    return 0;
}
