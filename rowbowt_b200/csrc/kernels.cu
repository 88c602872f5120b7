// sm_100a kernels of the rb_align query path.  Integer-only, random-access: bounded by
// HBM random-sector bandwidth, not tensor cores (SURVEY.md §0, §8(d)).
//
//   pack_kernel      raw read bytes -> 2-bit codes (+ per-read dead/exotic flags)
//   search_kernel    backward search, one read per thread, one 64-byte mixed leaf per rank
//                    (RowBowt::find_range / find_range_w_toehold, include/rowbowt.hpp:121-131,169-184)
//   search_bytes_kernel  same, byte-wise, for the rare reads that contain the terminator byte
//   locate_kernel    phi iteration (ToeholdSA::locate_range, include/toehold_sa.hpp:37-72)
//   marker_*_kernel  rle_window_arr::at_range (pfbwt-f/include/rle_window_array.hpp:130-154)
#include "kernels.cuh"

#include <stdexcept>

#include <cub/device/device_scan.cuh>

namespace rbg {

int grid_for(uint64_t work_items, int block, int per_sm) {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    uint64_t want = (work_items + block - 1) / block;
    uint64_t cap = (uint64_t) sms * per_sm;
    return (int) (want < cap ? (want ? want : 1) : cap);
}

namespace {

constexpr int kBlock = 256;
// Resident CTAs per SM search_kernel is built and launched for: 4 x 256 threads at 64 registers.  5 x 256 at 48 registers
// and 9 x 128 at 56 registers spill and measured 26.8 / 22.7 ms against 21.2 ms (profiles/r2_search_occupancy_variants.jsonl).
// Layout 7 is not bound by its L2-resident lines (DESIGN.md 2.1b) and its step needs fewer registers, so more resident warps
// hide more of each step's dependent latency.  Count: 6 x 256 at 40 registers (no spill), toehold: 5 x 256 at 46 (at 6 it
// spills and is slower); on `small` (B200) search_kernel 7.19 -> 6.69 ms and the toehold search 7.83 -> 7.52 ms
// (profiles/plain_occupancy_small.jsonl).
constexpr int kSearchCtas = 4;
constexpr int search_ctas(int V, bool toehold) { return V == 7 ? (toehold ? 5 : 6) : kSearchCtas; }

__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ uint64_t digest(uint64_t tag, uint64_t idx, uint64_t val) {
    return mix64(mix64(val) ^ (idx * 0x9E3779B97F4A7C15ull + tag));
}

// per-read flags are bytes; set one through the aligned word that holds it
__device__ __forceinline__ void flag_read(uint8_t* flags, uint64_t i, uint32_t f) {
    atomicOr(reinterpret_cast<uint32_t*>(flags) + (i >> 2), f << (8u * (uint32_t) (i & 3)));
}

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// pack: group t = bytes [32t, 32t+32) becomes one u64 of 2-bit codes.  One coalesced 32-byte load
// per group, no dependence on read boundaries.  A byte that is not A/C/G/T marks its read through a
// binary search over the offsets (rare path).  One launch covers the words that hold reads
// [r0, r1); bytes at or beyond offs[r1] may not have arrived yet (chunked H2D) and are ignored --
// the word that straddles the chunk boundary is packed again, complete, by the next chunk.
// A group's eight words stay in registers: every index into them is a compile-time constant, the tail group's too (writing
// them through a byte pointer would put them in local memory for every group).

// The bytes of group t; past `limit` they read as 0.
__device__ __forceinline__ void pack_load(const DevBatch& b, uint64_t t, uint64_t limit, uint32_t (&vw)[8]) {
    const uint64_t x0 = t << 5;
    if (x0 + 32 <= limit) {
        load_nc_32B(b.bases + x0, vw);
        return;
    }
#pragma unroll
    for (int wd = 0; wd < 8; ++wd) {
        uint32_t x = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x0 + 4 * wd + k < limit) x |= (uint32_t) b.bases[x0 + 4 * wd + k] << (8 * k);
        vw[wd] = x;
    }
}

__device__ __forceinline__ void pack_group(const DevBatch& b, const CodeTable& ct, const int8_t* lut, uint64_t t, uint64_t limit,
                                           const uint32_t (&vw)[8]) {
    const uint64_t x0 = t << 5;
    uint64_t out = 0;
    uint32_t bad = 0;
    // fast path (every index built by the documented pipeline maps A,C,G,T -> 0..3): four bytes at a time, SIMD-in-register.
    // A=0x41 C=0x43 G=0x47 T=0x54: ((c >> 1) ^ (c >> 2)) & 3 = 0,1,2,3; the four 2-bit fields of a word are gathered
    // into one byte by a multiply (fields land at bits 24..31, nothing else does).
    uint32_t all_ok = 0xFFFFFFFFu;
    if (ct.plain) {
#pragma unroll
        for (int wd = 0; wd < 8; ++wd) {
            const uint32_t x = vw[wd];
            all_ok &= __vcmpeq4(x, 0x41414141u) | __vcmpeq4(x, 0x43434343u) | __vcmpeq4(x, 0x47474747u) | __vcmpeq4(x, 0x54545454u);
            const uint32_t f = ((x >> 1) ^ (x >> 2)) & 0x03030303u;
            out |= (uint64_t) ((f * 0x01041040u) >> 24) << (8 * wd);
        }
    }
    if (!ct.plain || all_ok != 0xFFFFFFFFu || x0 + 32 > limit) {        // byte by byte through the table: flags / bad bits
        out = 0;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const uint32_t byte = (vw[i >> 2] >> (8 * (i & 3))) & 0xFFu;
            const int code = lut[byte];
            if (code >= 0 && code < 4) {
                out |= (uint64_t) code << (2 * i);
            } else if (b.bad) {
                bad |= 1u << i;                       // greedy seeding: such a base fails its seed, not its read
            } else if (x0 + i < limit) {
                // which read owns byte x0+i: last offset <= x
                const uint64_t x = x0 + i;
                uint64_t lo = 0, hi = b.n_reads;      // invariant offs[lo] <= x < offs[hi]
                while (hi - lo > 1) {
                    const uint64_t mid = (lo + hi) >> 1;
                    if (b.offs[mid] <= x) lo = mid; else hi = mid;
                }
                flag_read(b.flags, lo, code == 4 ? kReadExotic : kReadDead);
            }
        }
    }
    b.packed[t] = out;
    if (b.bad) b.bad[t] = bad;
}

// One group per thread and iteration: two per iteration, both loads issued before either group is converted, measured
// 0.586 against 0.574 ms for the 1.5 GB of the `small` batch (B200, profiles/pack_bench_small.jsonl).
__global__ void __launch_bounds__(kBlock) pack_kernel(DevBatch b, CodeTable ct) {
    __shared__ int8_t lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = ct.code_of[i];
    __syncthreads();
    const uint64_t limit = b.offs[b.r1];
    const uint64_t w0 = b.offs[b.r0] >> 5, w1 = (limit + 31) >> 5;
    for (uint64_t t = w0 + (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; t < w1; t += (uint64_t) gridDim.x * blockDim.x) {
        uint32_t vw[8];
        pack_load(b, t, limit, vw);
        pack_group(b, ct, lut, t, limit, vw);
    }
}

// ---------------------------------------------------------------------------------------------
// Toehold bookkeeping shared by both search kernels.  Invariant of the reference: k == SA[hi]
// (SURVEY Appendix B.4).  A trivial step decrements k; a non-trivial one replaces it by the
// sample of the run end whose LF image is the new hi.  Only the LAST non-trivial step matters,
// so the row is remembered and resolved once per read.
struct ToeholdTrack {
    uint64_t row;           // new hi after the last non-trivial step
    uint32_t since;         // trivial steps since then (or since the start)
    bool pending;
    __device__ __forceinline__ void init() { row = 0; since = 0; pending = false; }
    __device__ __forceinline__ void step(bool trivial, uint64_t new_hi) {
        if (trivial) ++since;
        else { row = new_hi; since = 0; pending = true; }
    }
    // ftab entry form: row (40 bits) | since << 40 | pending << 63
    __device__ __forceinline__ uint64_t pack() const { return row | ((uint64_t) since << 40) | ((uint64_t) pending << 63); }
    __device__ __forceinline__ void unpack(uint64_t v) {
        row = v & ((1ull << 40) - 1);
        since = (uint32_t) (v >> 40) & 0xFFu;
        pending = v >> 63;
    }
    __device__ __forceinline__ uint64_t finish(const DevToehold& T) const {
        const uint64_t base = pending ? toehold_at_row(T, row) : T.toehold0;
        return base - since;        // plain u64 arithmetic, as k-1 repeated (rowbowt.hpp:560)
    }
};

// One read per lane, and a lane whose read is over -- searched to its first base, or its range became empty (a
// mismatching or N-bearing read stops early, include/rowbowt.hpp:127) -- draws the next read of the launch from a
// device counter, so that lanes never idle behind the longest read of their warp: on the noisy read set of SURVEY 8(d)
// (1 % substitutions, 0.1 % N) the one-read-per-lane-per-round form ran every warp for the full 140 steps with half of
// its lanes dead.  Refills are batched (when a quarter of the warp is idle, or nothing is left to step) because the
// set-up of a read (seed-table lookup) is paid by the whole warp.
// The step loop is WARP-UNIFORM (every lane calls lf_step_warp) so that the rare rank positions can be answered by the
// whole warp (device_index.cuh).
// Layout 5 (V == 5): the superblock bases (<= 4 x 256 u64) are copied to shared memory once per CTA, so an LF step
// issues no load besides its one or two directory lines.
// Layout 7 (V == 7): the plain 2-bit lines of an L2-resident index (lf_step_plain); nothing to stage in shared memory.
// PAIR (count search only): two bases per step from the pair directory (lf_pair_warp), whose superblock table (16 x n_super
// u32, <= kPairMaxShared bytes) is the kernel's dynamic shared memory.  A lane whose read has an odd number of bases left
// first takes one step on the single-base directory, which then reads its superblock bases from global memory.
template <bool TOEHOLD, int V, bool PAIR>
__global__ void __launch_bounds__(kBlock, search_ctas(V, TOEHOLD)) search_kernel(DevLeafDir D, DevPairDir PD, DevToehold T, DevFtab ft, DevBatch b,
                                                                     DevResult r, DevCounters* ctr, unsigned long long* cursor) {
    constexpr uint32_t kFull = 0xFFFFFFFFu;
    __shared__ uint64_t s_base[V == 5 && !PAIR ? 4 * kMaxSuper5Dev : 1];
    extern __shared__ uint32_t s_pair[];
    const uint64_t* sup = D.super;
    if (PAIR) {
        for (uint32_t i = threadIdx.x; i < 16u * PD.n_super; i += blockDim.x) s_pair[i] = __ldg(PD.super + i);
        __syncthreads();
    } else if (V == 5) {
        for (uint32_t i = threadIdx.x; i < 4u * (uint32_t) D.n_super; i += blockDim.x) s_base[i] = __ldg(D.super + i);
        __syncthreads();
        sup = s_base;
    }
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t steps = 0, lines = 0;                          // per lane: far below 2^32
    bool have = false;                                      // this lane owns a read that is not finished
    uint64_t i = 0, lo = 0, hi = 0, x = 0, word = 0;
    uint32_t left = 0;
    ToeholdTrack tt;
    tt.init();
    bool exhausted = false;                                 // warp-uniform: the launch has handed out its last read
    constexpr int kRefillAt = 8;
    for (;;) {
        const uint32_t idle = __ballot_sync(kFull, !have);
        if (!exhausted && (idle == kFull || __popc(idle) >= kRefillAt)) {
            // idle lanes take the next reads of the launch, in order
            unsigned long long base = 0;
            const int leader = __ffs(idle) - 1;
            if ((int) lane == leader) base = atomicAdd(cursor, (unsigned long long) __popc(idle));
            base = __shfl_sync(kFull, base, leader);
            exhausted = b.r0 + base + (unsigned long long) __popc(idle) >= b.r1;
            if (!have) {
                i = b.r0 + base + (uint64_t) __popc(idle & ((1u << lane) - 1u));
                const uint32_t fl = i < b.r1 ? (uint32_t) b.flags[i] : (uint32_t) kReadExotic;
                if (!(fl & kReadExotic)) {                  // search_bytes_kernel owns exotic reads
                    have = true;
                    lo = 0;
                    hi = D.n - 1;                           // full_range, rowbowt.hpp:115-118
                    bool alive = !(fl & kReadDead);
                    tt.init();
                    left = 0;
                    if (alive) {
                        const uint64_t beg = b.offs[i], end = b.offs[i + 1];
                        x = end;
                        if (ft.k && end - beg >= ft.k) {
                            // seed: the last k bases through the k-mer table instead of k LF steps (search_ftab,
                            // rowbowt.hpp:745-758; an absent k-mer ends the search exactly as the k steps would)
                            x = end - ft.k;
                            const uint32_t sh = 2u * (uint32_t) (x & 31);
                            uint64_t key = __ldg(b.packed + (x >> 5)) >> sh;
                            if (sh + 2u * ft.k > 64u) key |= __ldg(b.packed + (x >> 5) + 1) << (64u - sh);
                            key &= (1ull << (2u * ft.k)) - 1;
                            const ulonglong2 seed = __ldg(ft.range + key);
                            lo = seed.x;
                            hi = seed.y;
                            alive = lo <= hi;
                            if (TOEHOLD && alive) tt.unpack(__ldg(ft.toe + key));
                        }
                        left = alive ? (uint32_t) (x - beg) : 0u;
                        if (left) word = __ldg(b.packed + ((x - 1) >> 5));
                    }
                    if (!alive) { lo = 1; hi = 0; }         // the empty range is exactly (1,0)
                }
            }
        }
        if (!__any_sync(kFull, have)) {
            if (exhausted) break;                           // no reads left and none in flight
            continue;                                       // only exotic reads were drawn: draw again
        }
        // one LF step for every lane with bases left; an empty range has left == 0
        const bool act = have && left != 0u;
        const bool single = PAIR ? act && (left & 1u) : act;
        if (!PAIR || __any_sync(kFull, single)) {
            uint32_t c = 0;
            if (single) {
                --x;
                if ((x & 31) == 31) word = __ldg(b.packed + (x >> 5));
                c = (uint32_t) (word >> (2 * (x & 31))) & 3u;
            }
            bool hi_is_c;
            const bool ok = lf_step_warp<TOEHOLD, V>(D, sup, c, lo, hi, single, hi_is_c, lines);
            if (single) {
                --left;
                ++steps;                                    // the failing step is counted, the rest of the read is not searched
                if (!ok) {
                    left = 0;
                    lo = 1;
                    hi = 0;
                } else if (TOEHOLD) {
                    tt.step(hi_is_c, hi);
                }
            }
        } else {
            uint32_t c1 = 0, c2 = 0;
            if (act) {
                --x;
                if ((x & 31) == 31) word = __ldg(b.packed + (x >> 5));
                c2 = (uint32_t) (word >> (2 * (x & 31))) & 3u;
                --x;
                if ((x & 31) == 31) word = __ldg(b.packed + (x >> 5));
                c1 = (uint32_t) (word >> (2 * (x & 31))) & 3u;
            }
            const bool ok = lf_pair_warp(PD, s_pair, 4u * c1 + c2, lo, hi, act, lines);     // leaves lo, hi as they were when it fails
            const bool failed = act && !ok;
            if (act) {
                left -= 2;
                steps += 2;
            }
            if (__any_sync(kFull, failed)) {
                // lf_steps counts the step that emptied the range and none after it: when the range was already empty after
                // c2 that is one step, not two (statistics only: the result is (1,0) either way)
                bool unused;
                const bool ok2 = lf_step_warp<false, V>(D, sup, c2, lo, hi, failed, unused, lines);
                if (failed && !ok2) --steps;
            }
            if (failed) {
                left = 0;
                lo = 1;
                hi = 0;
            }
        }
        if (have && left == 0u) {                           // finished: report and free the lane
            r.lo[i] = lo;
            r.hi[i] = hi;
            if (TOEHOLD) r.toehold[i] = hi >= lo ? tt.finish(T) : 0;   // cleared LFData on failure, rowbowt.hpp:176-179
            have = false;
        }
    }
    const unsigned long long st = warp_sum((unsigned long long) steps), ln = warp_sum((unsigned long long) lines);
    if (lane == 0 && st) {
        atomicAdd(&ctr->lf_steps, st);
        atomicAdd(&ctr->lf_lines, ln);
    }
}

// RowBowt::build_ftab (include/rowbowt.hpp:726-743): find_range of every k-mer, one k-mer per thread.
// k-mer x spells base i as code (x >> 2i) & 3; the search runs right to left, i = k-1 first.
template <bool TOEHOLD>
__global__ void __launch_bounds__(kBlock) ftab_build_kernel(DevLeafDir D, uint32_t k, ulonglong2* range, uint64_t* toe) {
    const uint64_t total = 1ull << (2 * k);
    for (uint64_t x = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (uint64_t) gridDim.x * blockDim.x) {
        uint64_t lo = 0, hi = D.n - 1;
        bool alive = true;
        ToeholdTrack tt;
        tt.init();
        uint32_t touched = 0;
        for (int i = (int) k - 1; i >= 0 && alive; --i) {
            bool hi_is_c;
            alive = lf_step<TOEHOLD>(D, (uint32_t) (x >> (2 * i)) & 3u, lo, hi, hi_is_c, touched);
            if (alive && TOEHOLD) tt.step(hi_is_c, hi);
        }
        range[x] = alive ? make_ulonglong2(lo, hi) : make_ulonglong2(1, 0);
        if (TOEHOLD) toe[x] = alive ? tt.pack() : 0;
    }
}

// Byte-wise search for reads flagged exotic (they contain the terminator byte 1, a legal BWT
// symbol with F[1] = 0).  One read per thread; these reads are vanishingly rare.
template <bool TOEHOLD>
__global__ void __launch_bounds__(kBlock) search_bytes_kernel(DevLeafDir D, DevToehold T, DevBatch b, DevResult r,
                                                               CodeTable ct, DevCounters* ctr) {
    for (uint64_t i = b.r0 + (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < b.r1;
         i += (uint64_t) gridDim.x * blockDim.x) {
        const uint32_t fl = b.flags[i];
        if (!(fl & kReadExotic)) continue;
        uint64_t lo = 0, hi = D.n - 1;
        bool alive = true;
        ToeholdTrack tt;
        tt.init();
        unsigned long long steps = 0, lines = 0;
        const uint64_t beg = b.offs[i], end = b.offs[i + 1];
        for (uint64_t x = end; x > beg && alive;) {
            --x;
            const int code = ct.code_of[b.bases[x]];
            bool hi_is_c = false;
            uint32_t touched = 0;
            ++steps;
            if (code < 0) alive = false;
            else if (code == 4) alive = lf_step_term(D, lo, hi, hi_is_c);
            else alive = lf_step<TOEHOLD>(D, (uint32_t) code, lo, hi, hi_is_c, touched);
            lines += touched;
            if (alive && TOEHOLD) tt.step(hi_is_c, hi);
        }
        if (!alive) { lo = 1; hi = 0; }
        r.lo[i] = lo;
        r.hi[i] = hi;
        if (TOEHOLD) r.toehold[i] = alive ? tt.finish(T) : 0;
        atomicAdd(&ctr->lf_steps, steps);
        atomicAdd(&ctr->lf_lines, lines);
    }
}

// ---------------------------------------------------------------------------------------------
// locate: n_occ = min(hi-lo+1, max_hits) values k, phi(k), phi(phi(k)), ... per read
__global__ void __launch_bounds__(kBlock) locate_count_kernel(DevResult r, uint64_t r0, uint64_t r1, uint64_t max_hits) {
    for (uint64_t i = r0 + (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < r1; i += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t lo = r.lo[i], hi = r.hi[i];
        uint64_t c = hi >= lo ? (hi - lo) + 1 : 0;
        r.loc_cnt[i] = c > max_hits ? max_hits : c;
    }
}

// One dependent phi chain per lane: what bounds the kernel is how many chains are in flight, so (1) a warp's 32
// chains must be equally long -- each CTA takes a tile of consecutive reads, counting-sorts it by chain length in
// shared memory (longest first) and its warps draw 32 sorted reads at a time -- and (2) the kernel fits 8 CTAs per SM
// (32 registers).  The ncu capture of the unsorted one-read-per-lane form showed 20.1 of 32 lanes active, 14 % issue
// slots and 30 % DRAM: nothing saturated, only latency.  Locations leave as a u32 plane (+ a u8 plane for bits
// 32..39 when n > 2^32) with NARROW, 8 bytes otherwise; streaming stores keep them from evicting the slots.
// Narrow locations leave the SM eight at a time: a lane collects the low words of consecutive locations in registers
// and writes them with ONE 256-bit streaming store once it reaches a 32-byte boundary of its output range (the head and
// the tail of a range go out word by word).  One L2 write request per eight phi steps instead of one per step: the
// kernel is bound by the number of memory requests per step (l1 word, slot, 10 % value, store), not by bytes.
__device__ __forceinline__ void st_cs_v8(uint32_t* p, const uint32_t (&v)[8]) {
    asm volatile("st.global.cs.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]),
                 "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}

// NARROW: u32 plane (HI: + the u8 plane of an index with n > 2^32) instead of u64 locations
template <bool NARROW, bool HI>
__device__ __forceinline__ uint64_t locate_chain(const DevPhi& P, const DevResult& r, uint64_t i) {
    const uint64_t off = r.loc_off[i], cnt = r.loc_off[i + 1] - off;
    if (!cnt) return 0;
    uint64_t k = r.toehold[i];
    if (!NARROW) {
        __stcs(r.locs + off, k);                    // streaming stores: the output must not push the slots out of L2
        for (uint64_t t = 1; t < cnt; ++t) {
            k = phi_step(P, k);
            __stcs(r.locs + off + t, k);
        }
        return cnt - 1;
    }
    uint32_t buf[8];
    unsigned long long hib = 0;                     // bits 32..39 of the same eight locations (index with n > 2^32)
    uint64_t at = off;                              // where location t goes
    const uint64_t end = off + cnt;
    for (;;) {
        const uint32_t slot = (uint32_t) at & 7u;
        // inside a full aligned group of eight: collect; otherwise (head before the first boundary, tail after the last) store now
        const uint64_t group = at & ~7ull;
        if (group >= off && group + 8 <= end) {
#pragma unroll
            for (int j = 0; j < 8; ++j) if (slot == (uint32_t) j) buf[j] = (uint32_t) k;
            if (HI) hib |= (unsigned long long) ((k >> 32) & 0xFFull) << (8u * slot);
            if (slot == 7u) {
                st_cs_v8(r.locs_lo + group, buf);
                if (HI) {                           // one 8-byte store instead of eight byte stores
                    __stcs(reinterpret_cast<unsigned long long*>(r.locs_hi + group), hib);
                    hib = 0;
                }
            }
        } else {
            __stcs(r.locs_lo + at, (uint32_t) k);
            if (HI) r.locs_hi[at] = (uint8_t) (k >> 32);
        }
        if (++at == end) break;
        k = phi_step(P, k);
    }
    return cnt - 1;
}

// One dependent phi chain per lane, one read per thread at a time, grid-stride in read order.  What bounds this
// kernel is the memory system's request rate, not latency: measured on the BASELINE batch (565 M phi steps,
// profiles/r2_locate_sweep.jsonl) FEWER resident CTAs are faster (8 per SM: 10.5 ms, 6: 9.5 ms, 4: 8.6 ms) and
// counting-sorting tiles of reads by chain length so that a warp's 32 chains are equally long (20 -> 32 active lanes)
// changes nothing (tiles of 256..2048 reads: 8.8..9.6 ms at 4 CTAs per SM) -- so the kernel stays unsorted and the grid is
// sized for 4 CTAs per SM.
template <bool NARROW, bool HI, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) locate_kernel(DevPhi P, DevResult r, uint64_t r0, uint64_t r1, DevCounters* ctr) {
    unsigned long long steps = 0;
    for (uint64_t i = r0 + (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < r1; i += (uint64_t) gridDim.x * blockDim.x)
        steps += locate_chain<NARROW, HI>(P, r, i);
    steps = warp_sum(steps);
    if ((threadIdx.x & 31) == 0 && steps) atomicAdd(&ctr->phi_steps, steps);
}

// Same with every lane DRAWING its next read from a device counter.  For the short chains of the BASELINE batch (56 steps
// on average, up to 65) the static grid-stride order above is faster (the draw costs an atomic per chain and measured
// 13.4 against 12.7 ms in round 1).  On the config-5 family an exact read occurs ~2200 times: 500 k chains of thousands
// of dependent steps over 151 k resident lanes are 3.3 chains per lane, and statically assigned the lanes holding four
// finish a third later than those holding three.  launch_locate picks this form when a chain averages >= 256 steps.
template <bool NARROW, bool HI, int MINB>
__global__ void __launch_bounds__(kBlock, MINB) locate_draw_kernel(DevPhi P, DevResult r, uint64_t r0, uint64_t r1, DevCounters* ctr,
                                                                   unsigned long long* cursor) {
    unsigned long long steps = 0;
    for (;;) {
        const uint64_t i = r0 + atomicAdd(cursor, 1ull);
        if (i >= r1) break;
        steps += locate_chain<NARROW, HI>(P, r, i);
    }
    steps = warp_sum(steps);
    if ((threadIdx.x & 31) == 0 && steps) atomicAdd(&ctr->phi_steps, steps);
}

// ---------------------------------------------------------------------------------------------
// markers: count pass (window range -> word count), scan, gather pass
__global__ void __launch_bounds__(kBlock) marker_count_kernel(DevMarkers M, DevResult r, uint64_t r0, uint64_t r1) {
    for (uint64_t i = r0 + (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < r1; i += (uint64_t) gridDim.x * blockDim.x) {
        uint64_t first, last;
        marker_windows(M, r.lo[i], r.hi[i], first, last);
        uint64_t words = 0;
        if (last > first) {
            const uint64_t a = marker_sel(M, first + 1), z = marker_sel(M, last + 1);
            words = z > a ? z - a : 0;
        }
        r.mk_first[i] = first;
        r.mk_cnt[i] = words;
    }
}

__global__ void __launch_bounds__(kBlock) marker_gather_kernel(DevMarkers M, DevResult r, uint64_t r0, uint64_t r1, DevCounters* ctr) {
    unsigned long long words = 0;
    for (uint64_t i = r0 + (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < r1; i += (uint64_t) gridDim.x * blockDim.x) {
        const uint64_t off = r.mk_off[i], cnt = r.mk_off[i + 1] - off;
        if (!cnt) continue;
        const uint64_t a = marker_sel(M, r.mk_first[i] + 1);
        for (uint64_t t = 0; t < cnt; ++t) r.markers[off + t] = __ldg(M.arr + a + t);
        words += cnt;
    }
    words = warp_sum(words);
    if ((threadIdx.x & 31) == 0 && words) atomicAdd(&ctr->marker_words, words);
}

// ---------------------------------------------------------------------------------------------
// order-independent digest of a result (parity at full size without moving it to the host)
__global__ void __launch_bounds__(kBlock) checksum_kernel(DevResult r, uint64_t n_reads, bool toehold, bool locs, bool markers,
                                                           DevCounters* ctr) {
    unsigned long long acc = 0;
    const uint64_t stride = (uint64_t) gridDim.x * blockDim.x, t0 = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    for (uint64_t i = t0; i < n_reads; i += stride) {
        acc += digest(1, i, r.lo[i]) + digest(2, i, r.hi[i]);
        if (toehold) acc += digest(3, i, r.toehold[i]);
        if (locs) acc += digest(4, i, r.loc_off[i + 1] - r.loc_off[i]);
        if (markers) acc += digest(7, i, r.mk_off[i + 1] - r.mk_off[i]);
    }
    if (locs) {
        const uint64_t tot = r.loc_off[n_reads];
        for (uint64_t j = t0; j < tot; j += stride) {
            uint64_t v;
            if (r.locs_lo) v = (uint64_t) r.locs_lo[j] | (r.locs_hi ? (uint64_t) r.locs_hi[j] << 32 : 0ull);
            else v = r.locs[j];
            acc += digest(5, j, v);
        }
    }
    if (markers) {
        const uint64_t tot = r.mk_off[n_reads];
        for (uint64_t j = t0; j < tot; j += stride) acc += digest(6, j, r.markers[j]);
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) atomicAdd(&ctr->checksum, acc);
}

// ---------------------------------------------------------------------------------------------
// random-gather microbenchmark: the roofline denominator for this path (SURVEY §8(d)).
// Each thread reads `iters` pseudo-random lines of LINE bytes; with `dependent` the next index
// is derived from the data just read (an LF-like chain), otherwise loads are independent.
// 64-byte lines fetched by lane PAIRS: lanes 2j and 2j+1 read the two 32-byte halves of the same random line in one
// warp instruction, so the line is ONE 64-byte L2 request (and one L1 tag look-up) instead of two 32-byte ones.
// Answers whether search_kernel's two LDG.256 per line are bound by requests or by bytes.
__global__ void __launch_bounds__(kBlock) gather_pair_kernel(const uint32_t* buf, uint64_t n_lines, int iters, unsigned long long* sink) {
    constexpr int U = 4;
    const uint32_t pair = (blockIdx.x * blockDim.x + threadIdx.x) >> 1, half = threadIdx.x & 1u;
    uint64_t state = mix64((uint64_t) pair * 2654435761ull + 12345);
    uint32_t acc = 0;
    for (int it = 0; it < iters; it += U) {
        uint32_t w[U][8];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t line = __umul64hi(mix64(state + u), n_lines);
            const uint32_t* p = buf + line * 16 + half * 8;
            asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(w[u][0]), "=r"(w[u][1]), "=r"(w[u][2]), "=r"(w[u][3]), "=r"(w[u][4]), "=r"(w[u][5]), "=r"(w[u][6]), "=r"(w[u][7])
                         : "l"(p));
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int i = 0; i < 8; ++i) acc ^= w[u][i];
        state = mix64(state + U);
    }
    if (acc == 0x12345678u) atomicAdd(sink, 1ull);
}

template <int LINE>
__global__ void __launch_bounds__(kBlock) gather_kernel(const uint32_t* buf, uint64_t n_lines, int iters, int dependent,
                                                        unsigned long long* sink) {
    constexpr int U = 4;        // independent lines in flight per thread
    uint64_t state = mix64(((uint64_t) blockIdx.x * blockDim.x + threadIdx.x) * 2654435761ull + 12345);
    uint32_t acc = 0;
    for (int it = 0; it < iters; it += U) {
        uint32_t w[U][LINE / 4];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t line = __umul64hi(mix64(state + u), n_lines);
            const uint32_t* p = buf + line * (LINE / 4);
#pragma unroll
            for (int h = 0; h < LINE / 32; ++h)
                asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                             : "=r"(w[u][8 * h + 0]), "=r"(w[u][8 * h + 1]), "=r"(w[u][8 * h + 2]), "=r"(w[u][8 * h + 3]),
                               "=r"(w[u][8 * h + 4]), "=r"(w[u][8 * h + 5]), "=r"(w[u][8 * h + 6]), "=r"(w[u][8 * h + 7])
                             : "l"(p + 8 * h));
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int i = 0; i < LINE / 4; ++i) acc ^= w[u][i];
        state = mix64(state + U + (dependent ? acc : 0u));
    }
    if (acc == 0x12345678u) atomicAdd(sink, 1ull);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// b.flags must have been zeroed for the whole batch before the first chunk is packed.
int launch_pack(const DevBatch& b, const CodeTable& ct, uint64_t approx_bytes, cudaStream_t st) {
    if (b.r1 <= b.r0) return 0;
    CodeTable c2 = ct;
    c2.plain = ct.code_of[(uint8_t) 'A'] == 0 && ct.code_of[(uint8_t) 'C'] == 1 && ct.code_of[(uint8_t) 'G'] == 2 && ct.code_of[(uint8_t) 'T'] == 3;
    pack_kernel<<<grid_for((approx_bytes >> 5) + 1, kBlock, 16), kBlock, 0, st>>>(b, c2);
    return 1;
}

int launch_search(const DevLeafDir& D, const DevPairDir& PD, const DevToehold* T, const DevFtab& ft, const DevBatch& b, const DevResult& r,
                  DevCounters* ctr, unsigned long long* cursor, cudaStream_t st) {
    if (b.r1 <= b.r0) return 0;
    DevToehold t0{};
    // reads are handed out by the device cursor, so ONE wave of CTAs is the whole grid: resident CTAs per SM x SMs.
    const int grid = grid_for(b.r1 - b.r0, kBlock, search_ctas((int) D.version, T != nullptr));
    if (!T && PD.lines) {                                   // the pair directory is built only over a layout-5 directory
        if (D.version != 5 || 64ull * PD.n_super > kPairMaxShared) throw std::logic_error("pair directory without its layout");
        search_kernel<false, 5, true><<<grid, kBlock, 64 * PD.n_super, st>>>(D, PD, t0, ft, b, r, ctr, cursor);
    } else if (D.version == 7) {
        if (T) search_kernel<true, 7, false><<<grid, kBlock, 0, st>>>(D, PD, *T, ft, b, r, ctr, cursor);
        else search_kernel<false, 7, false><<<grid, kBlock, 0, st>>>(D, PD, t0, ft, b, r, ctr, cursor);
    } else if (D.version == 5) {
        if (T) search_kernel<true, 5, false><<<grid, kBlock, 0, st>>>(D, PD, *T, ft, b, r, ctr, cursor);
        else search_kernel<false, 5, false><<<grid, kBlock, 0, st>>>(D, PD, t0, ft, b, r, ctr, cursor);
    } else {
        if (T) search_kernel<true, 4, false><<<grid, kBlock, 0, st>>>(D, PD, *T, ft, b, r, ctr, cursor);
        else search_kernel<false, 4, false><<<grid, kBlock, 0, st>>>(D, PD, t0, ft, b, r, ctr, cursor);
    }
    return 1;
}

int launch_ftab_build(const DevLeafDir& D, uint32_t k, bool toehold, ulonglong2* range, uint64_t* toe, cudaStream_t st) {
    const int grid = grid_for(1ull << (2 * k), kBlock, 8);
    if (toehold) ftab_build_kernel<true><<<grid, kBlock, 0, st>>>(D, k, range, toe);
    else ftab_build_kernel<false><<<grid, kBlock, 0, st>>>(D, k, range, toe);
    return 1;
}

int launch_search_bytes(const DevLeafDir& D, const DevToehold* T, const DevBatch& b, const DevResult& r,
                        const CodeTable& ct, DevCounters* ctr, cudaStream_t st) {
    if (b.r1 <= b.r0) return 0;
    const int grid = grid_for(b.r1 - b.r0, kBlock, 8);
    DevToehold t0{};
    if (T) search_bytes_kernel<true><<<grid, kBlock, 0, st>>>(D, *T, b, r, ct, ctr);
    else search_bytes_kernel<false><<<grid, kBlock, 0, st>>>(D, t0, b, r, ct, ctr);
    return 1;
}

int launch_locate_counts(const DevResult& r, uint64_t r0, uint64_t r1, uint64_t max_hits, cudaStream_t st) {
    if (r1 <= r0) return 0;
    locate_count_kernel<<<grid_for(r1 - r0, kBlock, 8), kBlock, 0, st>>>(r, r0, r1, max_hits);
    return 1;
}

// Resident CTAs per SM of the locate kernels, measured after the narrow stores went out eight at a time
// (profiles/r2_locate_ctas.jsonl; BASELINE batch / c5w): u64 locations are bound by their store requests and want FEWER warps
// (4: 10.7 ms, 6: 12.7 ms); narrow locations are latency-bound and want more -- the static kernel 6 (6.5 -> 6.0 ms; 40 registers,
// no spills without the high plane), the drawing kernel and the high-plane builds 5 (c5w: 14.3 -> 12.4 ms; 6 would spill).
constexpr int default_loc_ctas(bool narrow, bool hi_plane, bool draw) { return !narrow ? 4 : (draw || hi_plane) ? 5 : 6; }
// The build whose register budget lets that many CTAs of 256 threads be resident: 64 registers for 4 (and for 5, where the
// kernel needs <= 48), 40 for 6.  Each form is instantiated for its own count only.
constexpr int loc_minb(int ctas) { return ctas == 6 ? 6 : 4; }

template <bool NARROW, bool HI>
static void launch_locate_form(bool draw, const DevPhi& P, const DevResult& r, uint64_t r0, uint64_t r1, DevCounters* ctr,
                               unsigned long long* cursor, cudaStream_t st) {
    if (draw) {
        constexpr int ctas = default_loc_ctas(NARROW, HI, true);
        locate_draw_kernel<NARROW, HI, loc_minb(ctas)><<<grid_for(r1 - r0, kBlock, ctas), kBlock, 0, st>>>(P, r, r0, r1, ctr, cursor);
    } else {
        constexpr int ctas = default_loc_ctas(NARROW, HI, false);
        locate_kernel<NARROW, HI, loc_minb(ctas)><<<grid_for(r1 - r0, kBlock, ctas), kBlock, 0, st>>>(P, r, r0, r1, ctr);
    }
}

int launch_locate(const DevPhi& P, const DevResult& r, uint64_t r0, uint64_t r1, uint64_t n_locs, int force_draw, DevCounters* ctr,
                  unsigned long long* cursor, cudaStream_t st) {
    if (r1 <= r0) return 0;
    const bool draw = force_draw >= 0 ? force_draw != 0 : n_locs / (r1 - r0) >= 256;
    if (r.locs_lo && r.locs_hi) launch_locate_form<true, true>(draw, P, r, r0, r1, ctr, cursor, st);
    else if (r.locs_lo) launch_locate_form<true, false>(draw, P, r, r0, r1, ctr, cursor, st);
    else launch_locate_form<false, false>(draw, P, r, r0, r1, ctr, cursor, st);
    return 1;
}

int launch_marker_counts(const DevMarkers& M, const DevResult& r, uint64_t r0, uint64_t r1, cudaStream_t st) {
    if (r1 <= r0) return 0;
    marker_count_kernel<<<grid_for(r1 - r0, kBlock, 8), kBlock, 0, st>>>(M, r, r0, r1);
    return 1;
}

int launch_marker_gather(const DevMarkers& M, const DevResult& r, uint64_t r0, uint64_t r1, DevCounters* ctr, cudaStream_t st) {
    if (r1 <= r0) return 0;
    marker_gather_kernel<<<grid_for(r1 - r0, kBlock, 8), kBlock, 0, st>>>(M, r, r0, r1, ctr);
    return 1;
}

size_t scan_tmp_bytes(uint64_t n) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const uint64_t*) nullptr, (uint64_t*) nullptr, (int64_t) (n + 1));
    return bytes;
}

// cnt must have n+1 readable elements (cnt[n] ignored by construction: we scan n+1 items so
// that off[n] receives the total).
int launch_scan(const uint64_t* cnt, uint64_t* off, uint64_t n, void* tmp, size_t tmp_bytes, cudaStream_t st) {
    cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, cnt, off, (int64_t) (n + 1), st);
    return 1;
}

// Same scan continued from a running total that lives on the device (*init): chunk c of a pipelined batch starts
// where chunk c-1 ended without the host knowing the value.  n + 1 outputs, off[n] = *init + sum.
size_t scan_from_tmp_bytes(uint64_t n) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveScan(nullptr, bytes, (const uint64_t*) nullptr, (uint64_t*) nullptr, cub::Sum(),
                                   cub::FutureValue<uint64_t>((uint64_t*) nullptr), (int64_t) (n + 1));
    return bytes;
}
int launch_scan_from(const uint64_t* cnt, uint64_t* off, uint64_t n, const uint64_t* init, void* tmp, size_t tmp_bytes, cudaStream_t st) {
    cub::DeviceScan::ExclusiveScan(tmp, tmp_bytes, cnt, off, cub::Sum(), cub::FutureValue<uint64_t>(const_cast<uint64_t*>(init)),
                                   (int64_t) (n + 1), st);
    return 1;
}

int launch_checksum(const DevResult& r, uint64_t n_reads, bool toehold, bool locs, bool markers,
                    DevCounters* ctr, cudaStream_t st) {
    checksum_kernel<<<grid_for(n_reads ? n_reads : 1, kBlock, 8), kBlock, 0, st>>>(r, n_reads, toehold, locs, markers, ctr);
    return 1;
}

float run_gather(const uint32_t* buf, uint64_t n_lines, int line_bytes, int iters, int dependent, uint64_t* lines_done,
                 cudaStream_t st) {
    unsigned long long* sink = nullptr;
    cudaMalloc(&sink, 8);
    cudaMemsetAsync(sink, 0, 8, st);
    const int grid = grid_for(~0ull >> 8, kBlock, 8);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const bool paired = dependent == 2;                       // lane pairs share a 64-byte line (gather_pair_kernel)
    auto launch = [&](int n_it) {
        if (paired) gather_pair_kernel<<<grid, kBlock, 0, st>>>(buf, n_lines, n_it, sink);
        else if (line_bytes == 32) gather_kernel<32><<<grid, kBlock, 0, st>>>(buf, n_lines, n_it, dependent, sink);
        else if (line_bytes == 128) gather_kernel<128><<<grid, kBlock, 0, st>>>(buf, n_lines, n_it, dependent, sink);
        else gather_kernel<64><<<grid, kBlock, 0, st>>>(buf, n_lines, n_it, dependent, sink);
    };
    iters = (iters + 3) & ~3;
    launch(4);   // warm-up
    cudaEventRecord(e0, st);
    launch(iters);
    cudaEventRecord(e1, st);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *lines_done = (uint64_t) grid * kBlock * (uint64_t) iters / (paired ? 2 : 1);
    return ms;
}

}  // namespace rbg
