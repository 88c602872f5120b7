// mps_to_ma — the reference's marker-array builder (pfbwt-f/src/mps_to_ma.cpp) over librowbowt_gpu (C ABI).  The same
// .mps input and .ma output, but SA comes from the index's own phi on the GPU instead of a suffix-array stream, so the
// last argument is the index prefix (<prefix>.rbwt + .tsa, else the raw <prefix>.bwt/.ssa/.esa).
//
//   mps_to_ma [-o out.ma] [--mab out.mab] [--device D] <in.mps> <index_prefix>
#include <getopt.h>

#include <cstdio>
#include <cstdlib>
#include <string>

#include "../../include/rowbowt_gpu.h"

namespace {

void print_help() {
    fprintf(stderr, "mps_to_ma\n");
    fprintf(stderr, "Usage: mps_to_ma [options] <in.mps> <index_prefix>\n");
    fprintf(stderr, "    -o <out.ma>          output marker array (default <index_prefix>.ma)\n");
    fprintf(stderr, "    --mab <out.mab>      also write the .mab rb_build -m makes from it\n");
    fprintf(stderr, "    --device <D>         CUDA device to build on (default 0)\n");
    fprintf(stderr, "    <index_prefix>       <prefix>.rbwt + .tsa, else the raw <prefix>.bwt/.ssa/.esa\n");
}

}  // namespace

int main(int argc, char** argv) {
    std::string out, mab;
    int device = 0;
    static struct option lopts[] = {{"mab", required_argument, 0, 'b'}, {"device", required_argument, 0, 'd'}, {0, 0, 0, 0}};
    int c, li = 0;
    while ((c = getopt_long(argc, argv, "o:h", lopts, &li)) != -1) {
        switch (c) {
            case 'o': out = optarg; break;
            case 'b': mab = optarg; break;
            case 'd': device = atoi(optarg); break;
            case 'h': print_help(); return 0;
            default: print_help(); return 1;
        }
    }
    if (argc - optind != 2) {
        print_help();
        return 1;
    }
    const std::string mps = argv[optind], prefix = argv[optind + 1];
    if (prefix == "-") {
        fprintf(stderr, "mps_to_ma: the suffix-array stream is not read; give the index prefix (SA comes from its .tsa)\n");
        return 1;
    }
    if (out.empty()) out = prefix + ".ma";
    rbg_ma_stats st;
    if (rbg_build_marker_array(prefix.c_str(), mps.c_str(), out.c_str(), mab.empty() ? nullptr : mab.c_str(), 0, UINT64_MAX, device,
                               &st) != RBG_OK) {
        fprintf(stderr, "rbg_build_marker_array: %s\n", rbg_last_error());
        return 1;
    }
    fprintf(stderr,
            "n=%llu r=%llu  records %llu (%llu lists) -> .ma %llu records, %llu words  phi steps %llu  read %.3fs  layout %.3fs  "
            "rows kernel %.1f ms  blocks %.1f ms  write %.3fs  total %.3fs\n",
            (unsigned long long) st.n, (unsigned long long) st.r, (unsigned long long) st.mps_records, (unsigned long long) st.lists,
            (unsigned long long) st.ma_records, (unsigned long long) st.ma_words, (unsigned long long) st.phi_steps, st.s_read,
            st.s_layout, st.ms_rows_kernel, st.ms_blocks, st.s_write, st.s_total);
    return 0;
}
