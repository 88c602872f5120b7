// Host-side CUDA plumbing shared by the C ABI (api.cu) and the builders (raw_build.cu, ma_build.cu): the one CUDA error
// type the ABI maps to RBG_E_CUDA, owning device / pinned buffers, uploads, device selection and the phi upload.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <stdexcept>
#include <string>
#include <vector>

#include "layout.hpp"

namespace rbg {

struct cuda_error : std::runtime_error { using std::runtime_error::runtime_error; };

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            throw ::rbg::cuda_error(std::string(#call) + ": " + cudaGetErrorString(e_));           \
    } while (0)

struct DeviceAlloc {
    static cudaError_t alloc(void** p, size_t bytes) { return cudaMalloc(p, bytes); }
    static void free(void* p) { cudaFree(p); }
};
struct PinnedAlloc {
    static cudaError_t alloc(void** p, size_t bytes) { return cudaHostAlloc(p, bytes, cudaHostAllocDefault); }
    static void free(void* p) { cudaFreeHost(p); }
};

// An owning, growable buffer.  It frees itself on the device that is current when it is destroyed.
template <class A>
struct Buf {
    void* p = nullptr;
    size_t cap = 0;
    Buf() = default;
    explicit Buf(size_t bytes) { reserve(bytes, bytes); }
    Buf(Buf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    Buf& operator=(Buf&& o) noexcept {
        std::swap(p, o.p);
        std::swap(cap, o.cap);
        return *this;
    }
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    ~Buf() { if (p) A::free(p); }
    // Nothing when `need` bytes fit; else the old contents are dropped and `alloc` (>= need) bytes taken.
    void reserve(size_t need, size_t alloc) {
        if (need <= cap) return;
        if (p) A::free(p);
        p = nullptr;
        cap = 0;
        CU(A::alloc(&p, alloc));
        cap = alloc;
    }
    template <class T> T* as() const { return (T*) p; }
};
using DevBuf = Buf<DeviceAlloc>;
using PinnedBuf = Buf<PinnedAlloc>;

// One device copy of a host array and its payload bytes (the layout cache writes exactly those).
struct Upload {
    DevBuf mem;
    size_t bytes;
};

// At least 64 bytes are allocated, so that an empty array still has an address; `acc` adds the allocated bytes.
template <class T>
T* upload(const std::vector<T>& v, std::vector<Upload>& owned, size_t* acc = nullptr) {
    const size_t bytes = v.size() * sizeof(T);
    owned.push_back(Upload{DevBuf(std::max<size_t>(bytes, 64)), bytes});
    const DevBuf& m = owned.back().mem;
    if (bytes) CU(cudaMemcpy(m.p, v.data(), bytes, cudaMemcpyHostToDevice));
    if (acc) *acc += m.cap;
    return m.as<T>();
}

inline void select_device(int device) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) throw cuda_error("no CUDA device: librowbowt_gpu has no CPU fallback");
    if (device < 0 || device >= n) throw std::invalid_argument("device ordinal out of range");
    CU(cudaSetDevice(device));
}

inline double wall_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// The phi slots may take a quarter of the device memory free right now.
inline uint64_t phi_slot_budget() {
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    return (uint64_t) free_b / 4;
}

struct DevPhi;
// `pd` on the device, for text length n; the high plane only when the directory has one.  Defined in api.cu, so that this
// header keeps the device structures (device_index.cuh) out of the files that do not use them.
DevPhi upload_phi(const PhiDir& pd, uint64_t n, std::vector<Upload>& owned, size_t* acc = nullptr);

}  // namespace rbg
