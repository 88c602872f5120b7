// rb_align — drop-in host driver over librowbowt_gpu (C ABI).  Same command line, same
// index files (.rbwt/.tsa/.mab/.docs), same stdout grammar and stderr timing line as the
// reference driver (src/rb_align.cpp), but the per-read loop (src/rb_align.cpp:176-178) is
// batched: reads are parsed on the host, queried on the GPU(s) a batch at a time, and
// printed in FASTQ order.
//
//   rb_align [-s] [-m] [-o prefix] [--gpus N] [--threads T] [--batch READS] [--ftab | --ftab-k K] <index_prefix> <fastq>
//
// Pipeline (driver_pipeline.hpp): parser threads, which also pack the bases to 2 bits -> GPU
// workers calling rbg_query_packed -> formatter pool (report_format.hpp) -> ordered writer.
#include <getopt.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rowbowt_gpu.h"
#include "driver_pipeline.hpp"

namespace {

using rbhost::ReadBatch;

struct Args {
    std::string inpre, fastq, outpre;
    int sam = 0, markers = 0, fbb = 0;
    int gpus = 1;
    size_t batch_reads = 1u << 20;
    int ftab_file = 0;          // load <prefix>.ftab (LoadRbwtFlag::FT) instead of building the seed table
    int ftab_k = 10;            // k of the seed table built on the GPU at load (RowBowt::build_ftab default); 0 = none
    int layout_cache = 0;       // keep / use <index_prefix>.rbgcache (RBG_LOAD_CACHE): the finished GPU layout, uploaded as it is
    int parse_only = 0;         // diagnostic: dump "name<TAB>sequence" per record, no GPU needed
    long format_selftest = 0;   // diagnostic: N random reads through both report writers, compared byte for byte; no GPU needed
    int threads = 0;            // host parser / formatter threads (0 = all cores)
    size_t chunk_bytes = 0;     // bytes of FASTQ per parser chunk = per GPU batch (0 = from the file size)
};

void print_help() {
    fprintf(stderr, "rb_align");
    fprintf(stderr, "Usage: rb_align [options] <index_prefix> <input_fastq_name>\n");
    fprintf(stderr, "    --output_prefix/-o <basename>    output prefix\n");
    fprintf(stderr, "    --markers/-m                     print markers\n");
    fprintf(stderr, "    --sam/-s                         print locations\n");
    fprintf(stderr, "    --fbb                            index is based on wt-fbb\n");
    fprintf(stderr, "    --gpus/-g <N>                    number of GPUs (index replicated, batches sharded)\n");
    fprintf(stderr, "    --batch/-b <reads>               reads per GPU batch of a .gz / irregular input (default 1048576)\n");
    fprintf(stderr, "    --threads/-t <N>                 host parser + formatter threads (default: all cores)\n");
    fprintf(stderr, "    --chunk-bytes/-c <bytes>         FASTQ bytes per parser chunk = GPU batch (default: from the file size)\n");
    fprintf(stderr, "    --ftab                           load the k-mer seed table from <index_prefix>.ftab\n");
    fprintf(stderr, "    --ftab-k/-k <k>                  build the k-mer seed table on the GPU (default 10, 0 = none)\n");
    fprintf(stderr, "    --layout-cache                   keep the GPU layout in <index_prefix>.rbgcache and open from it when it is current\n");
    fprintf(stderr, "    <input_prefix>                   index prefix\n");
    fprintf(stderr, "    <input_fastq>                    input fastq\n");
}

Args parse_args(int argc, char** argv) {
    Args a;
    static struct option lopts[] = {{"output_prefix", required_argument, 0, 'o'},
                                    {"markers", no_argument, 0, 'm'},
                                    {"sam", no_argument, 0, 's'},
                                    {"fbb", no_argument, 0, 'f'},
                                    {"gpus", required_argument, 0, 'g'},
                                    {"batch", required_argument, 0, 'b'},
                                    {"parse-only", no_argument, 0, 'P'},
                                    {"format-selftest", required_argument, 0, 'S'},
                                    {"layout-cache", no_argument, 0, 'L'},
                                    {"ftab", no_argument, 0, 'F'},
                                    {"ftab-k", required_argument, 0, 'k'},
                                    {"threads", required_argument, 0, 't'},
                                    {"chunk-bytes", required_argument, 0, 'c'},
                                    {"help", no_argument, 0, 'h'},
                                    {0, 0, 0, 0}};
    int c, li = 0;
    while ((c = getopt_long(argc, argv, "o:smhg:b:k:t:c:", lopts, &li)) != -1) {
        switch (c) {
            case 'f': a.fbb = 1; break;
            case 'o': a.outpre = optarg; break;
            case 'h': print_help(); exit(0);
            case 's': a.sam = 1; break;
            case 'm': a.markers = 1; break;
            case 'P': a.parse_only += 1; break;      // given twice: totals only
            case 'S': a.format_selftest = std::max(1l, atol(optarg)); break;
            case 'L': a.layout_cache = 1; break;
            case 'F': a.ftab_file = 1; break;
            case 'k': a.ftab_k = std::max(0, atoi(optarg)); break;
            case 'g': a.gpus = std::max(1, atoi(optarg)); break;
            case 't': a.threads = std::max(1, atoi(optarg)); break;
            case 'c': a.chunk_bytes = (size_t) std::max(64ll, atoll(optarg)); break;
            case 'b': a.batch_reads = (size_t) std::max(1ll, atoll(optarg)); break;
            default: print_help(); exit(1);
        }
    }
    if (a.format_selftest) return a;
    if (argc - optind < (a.parse_only ? 1 : 2)) {
        fprintf(stderr, "no argument provided\n");
        exit(1);
    }
    if (!a.parse_only) a.inpre = argv[optind++];
    a.fastq = argv[optind++];
    if (a.outpre.empty()) a.outpre = a.inpre;
    if (a.threads <= 0) a.threads = (int) std::max(1u, std::thread::hardware_concurrency());
    return a;
}

// MarkerT accessors, pfbwt-f/include/marker.hpp:19-21,35-37
inline uint64_t marker_pos(uint64_t m) { return m & 0x00000FFFFFFFFFFFull; }
inline uint64_t marker_allele(uint64_t m) { return (m & 0xF000000000000000ull) >> 60; }

// rb_report's text for reads [i0, i1) of one batch, src/rb_align.cpp:118-145 -- the plain writer.  The driver uses
// rbhost::format_report (report_format.hpp: same bytes, ~10x faster); this one is what --format-selftest compares it with.
void format_slice_plain(const Args& args, const rbhost::DocList& docs, const rbg_result& r, const ReadBatch& b,
                        uint64_t i0, uint64_t i1, std::string& o) {
    o.clear();
    size_t want = (i1 - i0) * 48;
    if (args.sam) want += (r.loc_off[i1] - r.loc_off[i0]) * 28 + (i1 - i0) * 8;
    if (args.markers) want += (r.mk_off[i1] - r.mk_off[i0]) * 12 + (i1 - i0) * 12;
    o.reserve(want);
    for (uint64_t i = i0; i < i1; ++i) {
        size_t nl;
        const char* nm = b.name(i, nl);
        o.append(nm, nl);                               // (already cut at a NUL: printed as a C string)
        const uint64_t lo = r.lo ? r.lo[i] : r.lo32[i], hi = r.hi ? r.hi[i] : r.hi32[i];
        o += " (";
        rbhost::put_u64(o, lo);
        o += ',';
        rbhost::put_u64(o, hi);
        o += "), count=";
        rbhost::put_u64(o, hi - lo + 1);               // 64-bit wraparound, as printed by the reference
        o += '\n';
        if (args.sam) {
            o += "\tlocs: ";
            for (uint64_t j = r.loc_off[i]; j < r.loc_off[i + 1]; ++j) {
                const std::string* dn;
                uint64_t off;
                // RBG_NARROW_LOCS: a u32 plane plus, for an index with n > 2^32, a u8 plane
                const uint64_t loc = r.locs_lo32 ? (uint64_t) r.locs_lo32[j] | (r.locs_hi8 ? (uint64_t) r.locs_hi8[j] << 32 : 0ull) : r.locs[j];
                docs.resolve(loc, dn, off);
                rbhost::put_u64(o, loc);
                o += '/';
                o += *dn;
                o += ':';
                rbhost::put_u64(o, off);
                o += ' ';
            }
            o += '\n';
        }
        if (args.markers) {
            o += "\tmarkers: ";
            if (r.mk_off[i] == r.mk_off[i + 1]) o += "no markers (consider building the marker array with a larger window size)";
            for (uint64_t j = r.mk_off[i]; j < r.mk_off[i + 1]; ++j) {
                rbhost::put_u64(o, marker_pos(r.markers[j]));
                o += '/';
                rbhost::put_u64(o, marker_allele(r.markers[j]));
                o += ' ';
            }
            o += '\n';
        }
    }
}


// --format-selftest N: N random reads (names, ranges, locations in all three encodings, markers) through the plain
// writer and through rbhost::format_report, every flag set; the texts must be identical.  Prints the two rates.
int format_selftest(long n_reads) {
    uint64_t st = 88172645463325252ull;
    auto rnd = [&] { st ^= st << 13; st ^= st >> 7; st ^= st << 17; return st; };
    for (uint64_t v : {0ull, 1ull, 9ull, 10ull, 99ull, 100ull, 999ull, 1000ull, 4294967295ull, 4294967296ull, 9999999999ull, 10000000000ull,
                       999999999999999999ull, 1000000000000000000ull, 9999999999999999999ull, 10000000000000000000ull, ~0ull}) {
        char a[32], b[32];
        *rbhost::put_dec(a, v) = 0;
        snprintf(b, sizeof b, "%llu", (unsigned long long) v);
        if (strcmp(a, b)) { fprintf(stderr, "put_dec(%s) wrote %s\n", b, a); return 1; }
    }
    for (int it = 0; it < 2000000; ++it) {
        const uint64_t v = rnd() >> (rnd() & 63);
        char a[32], b[32];
        *rbhost::put_dec(a, v) = 0;
        snprintf(b, sizeof b, "%llu", (unsigned long long) v);
        if (strcmp(a, b)) { fprintf(stderr, "put_dec(%s) wrote %s\n", b, a); return 1; }
    }
    // documents: unevenly spaced, with a duplicate start (DocList::load sorts + uniques the starts but keeps the names)
    rbhost::DocList docs;
    std::vector<std::string> names;
    std::vector<uint64_t> starts;
    uint64_t at = 0;
    for (int d = 0; d < 65; ++d) {
        names.push_back(d % 7 ? "h" + std::to_string(d) : "a_rather_long_document_name_" + std::to_string(d));
        starts.push_back(at);
        at += 1000 + rnd() % 90000000;
    }
    names.push_back("dup");
    const uint64_t n_text = at;
    docs.set(names, starts);
    rbhost::DocResolver resolver;
    resolver.init(docs.names(), docs.starts());
    ReadBatch b;
    b.bases.a = b.offs.a = b.packed.a = b.flags.a = rbhost::HostAlloc{malloc, free};
    b.clear();
    const uint64_t n = (uint64_t) n_reads;
    std::vector<uint64_t> lo(n), hi(n), loc_off(n + 1, 0), mk_off(n + 1, 0), locs, markers;
    for (uint64_t i = 0; i < n; ++i) {
        const std::string nm = "read" + std::to_string(rnd() % 1000000007);
        b.add(nm.data(), nm.size(), "ACGT", 4);
        const int kind = (int) (rnd() % 10);
        lo[i] = kind == 0 ? 1 : rnd() % n_text;
        hi[i] = kind == 0 ? 0 : (kind == 1 ? lo[i] - 2 - rnd() % 5 : lo[i] + rnd() % 70);        // empty, wrapped, ordinary
        const uint64_t cnt = kind <= 1 ? 0 : hi[i] - lo[i] + 1;
        for (uint64_t j = 0; j < cnt; ++j) locs.push_back(rnd() % (n_text + 5000));
        loc_off[i + 1] = locs.size();
        for (uint64_t j = 0, m = rnd() % 4 ? 0 : rnd() % 5; j < m; ++j) markers.push_back((rnd() & 0xF00003FFFFFFFFFFull));
        mk_off[i + 1] = markers.size();
    }
    std::vector<uint32_t> lo32(locs.size());
    std::vector<uint8_t> hi8(locs.size());
    for (size_t j = 0; j < locs.size(); ++j) { lo32[j] = (uint32_t) locs[j]; hi8[j] = (uint8_t) (locs[j] >> 32); }
    const bool wide = (n_text >> 32) != 0;
    double t_plain = 0, t_fast = 0, t_warm = 0;
    uint64_t bytes = 0;
    for (int enc = 0; enc < 2; ++enc)
        for (int flags = 0; flags < 4; ++flags) {
            Args a;
            a.sam = flags & 1;
            a.markers = (flags >> 1) & 1;
            rbg_result r{};
            r.n_reads = n;
            r.lo = lo.data(); r.hi = hi.data(); r.loc_off = loc_off.data(); r.mk_off = mk_off.data(); r.markers = markers.data();
            if (enc == 0) r.locs = locs.data();
            else { r.locs_lo32 = lo32.data(); r.locs_hi8 = wide ? hi8.data() : nullptr; }
            if (enc == 1 && !wide) for (size_t j = 0; j < locs.size(); ++j) locs[j] = lo32[j];      // what the narrow planes can carry
            std::vector<uint32_t> rlo32(n), rhi32(n);
            if (enc == 1 && !wide) {                           // RBG_NARROW_RANGES: u32 planes (the wrapped ranges of the u64 case do not occur on the wire)
                for (uint64_t i = 0; i < n; ++i) { rlo32[i] = (uint32_t) lo[i]; rhi32[i] = (uint32_t) hi[i]; lo[i] = rlo32[i]; hi[i] = rhi32[i]; }
            }
            std::string plain;
            rbhost::OutBuf fast;
            auto c0 = std::chrono::steady_clock::now();
            format_slice_plain(a, docs, r, b, 0, n, plain);
            auto c1 = std::chrono::steady_clock::now();
            rbg_result rf = r;                                  // the fast writer reads the narrow planes when they are given
            if (enc == 1 && !wide) { rf.lo = rf.hi = nullptr; rf.lo32 = rlo32.data(); rf.hi32 = rhi32.data(); }
            rbhost::format_report(a.sam != 0, a.markers != 0, resolver, rf, [&b](uint64_t i, size_t& nl) { return b.name(i, nl); }, 0, n, fast);
            auto c2 = std::chrono::steady_clock::now();
            if (flags == 1 && enc == 1) {                      // once more into the now mapped buffer: the steady state of a recycled batch
                rbhost::format_report(a.sam != 0, a.markers != 0, resolver, r, [&b](uint64_t i, size_t& nl) { return b.name(i, nl); }, 0, n, fast);
                t_warm = std::chrono::duration<double>(std::chrono::steady_clock::now() - c2).count();
            }
            if (plain.size() != fast.len || memcmp(plain.data(), fast.p, fast.len)) {
                fprintf(stderr, "format-selftest: texts differ (encoding %d, flags %d: %zu vs %zu bytes)\n", enc, flags, plain.size(), fast.len);
                return 1;
            }
            if (flags == 1 && enc == 1) {
                t_plain = std::chrono::duration<double>(c1 - c0).count();
                t_fast = std::chrono::duration<double>(c2 - c1).count();
                bytes = fast.len;
            }
        }
    printf("format-selftest ok: %ld reads, %zu locations, -s text %llu bytes: plain writer %.3f GB/s, format_report %.3f GB/s (%.3f GB/s into a mapped buffer)\n",
           n_reads, locs.size(), (unsigned long long) bytes, (double) bytes / t_plain * 1e-9, (double) bytes / t_fast * 1e-9, (double) bytes / t_warm * 1e-9);
    return 0;
}

[[noreturn]] void die_rbg(const char* what) {
    fprintf(stderr, "%s: %s\n", what, rbg_last_error());
    exit(1);
}

}  // namespace

int main(int argc, char** argv) {
    Args args = parse_args(argc, argv);
    if (args.format_selftest) return format_selftest(args.format_selftest);
    setenv("RBG_BLOCKING_SYNC", "1", 0);         // the GPU worker sleeps while it waits: every core is busy parsing / formatting (api.cu, Lane)
    if (args.parse_only) {                       // diagnostic of the FASTX front end; no GPU needed
        rbhost::FastxBatchSource src(args.fastq.c_str(), args.threads, args.chunk_bytes, args.batch_reads,
                                     rbhost::HostAlloc{malloc, free}, 2 * (size_t) args.threads + 4);
        if (!src.ok()) { fprintf(stderr, "invalid file\n"); return 1; }
        uint64_t n_batches = 0, n_reads = 0, n_bases = 0;
        while (std::unique_ptr<ReadBatch> b = src.next()) {
            n_reads += b->n;
            n_bases += b->n_bases();
            for (uint64_t i = 0; i < b->n && args.parse_only == 1; ++i) {
                size_t nl;
                const char* nm = b->name(i, nl);
                fwrite(nm, 1, nl, stdout);
                fputc('\t', stdout);
                fwrite(b->bases.p + b->offs.p[i], 1, b->offs.p[i + 1] - b->offs.p[i], stdout);
                fputc('\n', stdout);
            }
            ++n_batches;
            src.recycle(std::move(b));
        }
        fprintf(stderr, "parse-only: %s, %llu reads, %llu bases, %llu batches, %llu fallbacks\n", src.parallel() ? "parallel" : "sequential",
                (unsigned long long) n_reads, (unsigned long long) n_bases, (unsigned long long) n_batches, (unsigned long long) src.fallbacks());
        if (src.err() == -2) { fprintf(stderr, "ERROR: truncated quality string\n"); return 1; }
        if (src.err() == -3) { fprintf(stderr, "ERROR: error reading stream\n"); return 1; }
        return 0;
    }
    if (args.fbb && args.sam) {
        // the reference accepts this and prints locations walked from an uninitialised toehold
        // (src/rb_align.cpp:110-116,125): there is no defined output to reproduce
        fprintf(stderr, "--fbb: fbb_string does not support the toehold suffix array (-s)\n");
        return 1;
    }
    using clk = std::chrono::high_resolution_clock;
    auto t0 = clk::now();

    // load_rbwt, src/rb_align.cpp:147-160
    uint32_t flags = 0;
    rbhost::DocList docs;
    if (args.sam) {
        std::cerr << "will load SA and DA" << std::endl;
        flags |= RBG_LOAD_SA | RBG_LOAD_DL;
    }
    if (args.markers) {
        std::cerr << "will load SA and DA" << std::endl;
        flags |= RBG_LOAD_MA;
    }
    if (args.ftab_file) flags |= RBG_LOAD_FT;
    if (args.fbb) flags |= RBG_LOAD_FBB;
    if (args.layout_cache) flags |= RBG_LOAD_CACHE;
    rbhost::QueryPipeline<rbg_result>::Options po;
    po.fastq = args.fastq;
    po.threads = args.threads;
    po.chunk_bytes = args.chunk_bytes;
    po.batch_reads = args.batch_reads;
    po.gpus = args.gpus;
    // A parser chunk is ~50 k reads: 0.4 ms on an idle GPU (0.12 ms of it kernel time, the rest the latency of 140 dependent
    // LF steps and three copies), so ONE caller per device leaves the GPU mostly idle and, at 10^7 reads, was the slowest
    // stage of the count / -m pipeline.  Two workers per device overlap their calls (the library runs concurrent calls on one
    // handle in separate lanes).  With -s the report writer is the bound and concurrent locate calls contend for the device
    // allocator: one worker.
    po.workers_per_gpu = args.sam ? 1 : 2;
    po.slice_shift = 12;
    // the thread that parsed a batch also packs its bases to 2 bits (rbg_pack_bytes): 46 instead of 158 bytes per
    // 150 bp read cross PCIe, and the GPU skips pack_kernel (RBG_HOST_PACK=0: ship the bytes, pack on the device)
    const bool host_pack = !(getenv("RBG_HOST_PACK") && atoi(getenv("RBG_HOST_PACK")) == 0);
    if (host_pack)
        po.pack = [](rbg_index* ix, ReadBatch& b) {
            const uint64_t nb = b.n_bases();
            b.packed.reserve(nb / 32 + 2, 0);
            b.flags.reserve(b.n + 8, 0);
            memset(b.flags.p, 0, b.n);
            b.n_exotic = 0;
            uint64_t ex = 0;
            if (rbg_pack_bytes(ix, b.bases.p, b.offs.p, b.n, 0, nb, b.packed.p, b.flags.p, &ex) != RBG_OK) die_rbg("rbg_pack_bytes");
            if (ex)
                for (uint64_t i = 0; i < b.n; ++i) b.n_exotic += (b.flags.p[i] & RBG_READ_EXOTIC) ? 1 : 0;
        };
    rbhost::QueryPipeline<rbg_result> pipe(std::move(po));
    std::string msg;
    const int rc = pipe.open(args.inpre.c_str(), flags, [&](rbg_index* ix) {
        return !args.ftab_file && args.ftab_k ? rbg_ftab_build(ix, (uint32_t) args.ftab_k) : RBG_OK;
    }, msg);
    if (rc) {
        // the reference prints "bad file" and exits for a missing part (rowbowt_io.hpp:166-169)
        std::cerr << (rc == RBG_E_IO ? "bad file" : msg) << std::endl;
        return 1;
    }
    if (args.sam) {
        std::cerr << "loading: " << args.inpre + ".docs" << std::endl;
        if (!docs.load(args.inpre + ".docs")) {
            std::cerr << "bad file" << std::endl;
            return 1;
        }
    }
    rbhost::DocResolver resolver;
    resolver.init(docs.names(), docs.starts());
    const bool input_ok = pipe.finish_load();
    std::chrono::duration<double> load_time = clk::now() - t0;
    if (!input_ok) {                                  // src/rb_align.cpp:170-173 (after the index is loaded, as there)
        fprintf(stderr, "invalid file\n");
        return 1;
    }

    // narrow wire forms (u32 ranges / locations when n <= 2^32): half the D2H bytes, widened while formatting
    const uint32_t mode = (args.sam ? RBG_LOCATE | RBG_NARROW_LOCS : 0) | (args.markers ? RBG_MARKERS : 0) | RBG_NARROW_RANGES;
    const double query_time = pipe.run(
        [&](rbg_index* ix, ReadBatch& b, rbg_result& res) {
            if (host_pack) {
                rbg_packed_batch in{b.n, b.packed.p, b.offs.p, b.flags.p, b.n_exotic, b.bases.p};
                if (rbg_query_packed(ix, &in, mode, UINT64_MAX, &res) != RBG_OK) die_rbg("rbg_query_packed");
            } else {
                rbg_batch in{b.n, b.bases.p, b.offs.p};
                if (rbg_query(ix, &in, mode, UINT64_MAX, &res) != RBG_OK) die_rbg("rbg_query");
            }
        },
        rbg_result_free,
        [&](const rbg_result& res, const ReadBatch& b, uint64_t i0, uint64_t i1, rbhost::OutBuf& out) {
            rbhost::format_report(args.sam != 0, args.markers != 0, resolver, res, [&b](uint64_t i, size_t& nl) { return b.name(i, nl); }, i0, i1, out);
        });
    std::cerr << load_time.count() << " " << query_time << std::endl;
    return 0;
}
