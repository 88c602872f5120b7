// fa_to_bwt — the first step of the reference's scripts/fa_to_rowbowt.sh (`pfbwt-f64 --non-acgt-to-a --print-docs -r -o P P.fa`)
// over librowbowt_gpu (C ABI): the BWT of a FASTA on the GPU, with its run-boundary samples and document list.
//
//   fa_to_bwt [-o out_prefix] [--device D] <in.fa[.gz]>
#include <getopt.h>

#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../include/rowbowt_gpu.h"

namespace {

void print_help() {
    fprintf(stderr, "fa_to_bwt\n");
    fprintf(stderr, "Usage: fa_to_bwt [options] <in.fa[.gz]>\n");
    fprintf(stderr, "    -o <out_prefix>      writes <out_prefix>.bwt/.ssa/.esa/.docs (default <in.fa[.gz]>)\n");
    fprintf(stderr, "    --device <D>         CUDA device to build on (default 0)\n");
    fprintf(stderr, "    Uppercase A C G T are kept and other uppercase letters become A; lowercase input is refused.\n");
}

}  // namespace

int main(int argc, char** argv) {
    std::string out;
    int device = 0;
    static struct option lopts[] = {{"device", required_argument, 0, 'd'}, {0, 0, 0, 0}};
    int c, li = 0;
    while ((c = getopt_long(argc, argv, "o:h", lopts, &li)) != -1) {
        switch (c) {
            case 'o': out = optarg; break;
            case 'd': device = atoi(optarg); break;
            case 'h': print_help(); return 0;
            default: print_help(); return 1;
        }
    }
    if (argc - optind != 1) {
        print_help();
        return 1;
    }
    const std::string fa = argv[optind];
    if (out.empty()) out = fa;
    rbg_bwt_stats st;
    if (rbg_build_bwt(fa.c_str(), out.c_str(), device, &st) != RBG_OK) {
        fprintf(stderr, "rbg_build_bwt: %s\n", rbg_last_error());
        return 1;
    }
    fprintf(stderr,
            "n=%llu r=%llu  records %llu  wide %u  parts %u  rounds %u (largest active set %llu)  parse %.3fs  sort %.3fs (kernels %.1f ms, "
            "verify %.1f ms, gather %.1f ms)  write %.3fs  total %.3fs  device memory %.2f GB\n",
            (unsigned long long) st.n, (unsigned long long) st.r, (unsigned long long) st.records, st.wide, st.parts, st.rounds,
            (unsigned long long) st.max_active, st.s_parse, st.s_sort, st.ms_sort, st.ms_verify, st.ms_gather, st.s_write, st.s_total,
            st.peak_bytes / 1e9);
    return 0;
}
