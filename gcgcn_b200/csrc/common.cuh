// Shared helpers for the gcgcn_b200 kernels (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>

#include "../../include/gcgcn_b200.h"

namespace gcgcn {

constexpr int D = GCGCN_HIDDEN;  // hidden width, G:234
constexpr int WARP = 32;

// ---- per-thread error text + process-wide launch counter --------------------------------
char* error_buffer();
int fail(int code, const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
// optional per-kernel timing (gcgcn_timing_begin/end): one CUDA event after every launch and at
// every API entry; a kernel's time is the gap to the previous event on the same stream.
extern std::atomic<bool> g_timing;
void timing_mark(const char* name, cudaStream_t st);
// floating-point operations (or bytes) the NEXT marked launch performs; summed per kernel name by timing_end
void timing_set_work(double work);

inline int cuda_ok(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return GCGCN_OK;
    return fail(GCGCN_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

#define GCGCN_CHECK_LAUNCH(name)                                        \
    do {                                                                \
        ::gcgcn::g_launches.fetch_add(1, std::memory_order_relaxed);    \
        if (::gcgcn::g_timing.load(std::memory_order_relaxed)) ::gcgcn::timing_mark(name, st); \
        int rc__ = ::gcgcn::cuda_ok(cudaPeekAtLastError(), name);       \
        if (rc__ != GCGCN_OK) return rc__;                              \
    } while (0)

// Every entry point launches on the device that owns `stream`, whatever the calling thread's current device is
// (a stream of cuda:1 handed in while cuda:0 is current used to launch into the wrong context); the previous
// device is restored when the entry point returns.  The legacy default stream (NULL) keeps the current device.
struct StreamDeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit StreamDeviceGuard(cudaStream_t st) {
        int dev = -1;
        if (st == nullptr) return;
        // a capturing stream must not be queried (the query would invalidate the capture); whoever captures has
        // made the stream's device current already
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { cudaGetLastError(); return; }
        if (cap != cudaStreamCaptureStatusNone) return;
        if (cudaStreamGetDevice(st, &dev) != cudaSuccess) { cudaGetLastError(); return; }
        if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); return; }
        if (prev != dev && cudaSetDevice(dev) == cudaSuccess) switched = true;
    }
    ~StreamDeviceGuard() { if (switched) cudaSetDevice(prev); }
    StreamDeviceGuard(const StreamDeviceGuard&) = delete;
    StreamDeviceGuard& operator=(const StreamDeviceGuard&) = delete;
};

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a PER-DEVICE setting: one bit per device ordinal records
// where a kernel has been prepared (a process that touches a second GPU prepares it there on first use).
inline bool device_prepared(const std::atomic<unsigned long long>& mask) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return false;
    return (mask.load(std::memory_order_acquire) >> dev) & 1ULL;
}
inline void device_mark_prepared(std::atomic<unsigned long long>& mask) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return;
    mask.fetch_or(1ULL << dev, std::memory_order_release);
}

// Dynamic shared memory above the default 48 KB must be enabled per kernel; more than an SM has (227 KB) is refused.
template <typename K>
inline int set_smem(K kernel, size_t bytes, const char* name) {
    if (bytes > 227 * 1024)
        return fail(GCGCN_ERR_UNSUPPORTED, "%s needs %zu bytes of shared memory (> 227 KB): documents "
                    "this large are not supported", name, bytes);
    if (bytes > 48 * 1024)
        return cuda_ok(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            static_cast<int>(bytes)), name);
    return GCGCN_OK;
}
// set_smem for a kernel that always launches with the same size, once per device; `mask` is a static of the caller,
// one per kernel instantiation
template <typename K>
inline int set_smem_once(std::atomic<unsigned long long>& mask, K kernel, size_t bytes, const char* name) {
    if (device_prepared(mask)) return GCGCN_OK;
    const int rc = set_smem(kernel, bytes, name);
    if (rc == GCGCN_OK) device_mark_prepared(mask);
    return rc;
}

#define GCGCN_API_ENTER(stream)                                                          \
    ::gcgcn::StreamDeviceGuard device_guard__(static_cast<cudaStream_t>(stream));        \
    do {                                                                                 \
        if (::gcgcn::g_timing.load(std::memory_order_relaxed))                           \
            ::gcgcn::timing_mark("(between calls)", static_cast<cudaStream_t>(stream));  \
    } while (0)

#define GCGCN_TRY(expr)                    \
    do {                                   \
        int rc__ = (expr);                 \
        if (rc__ != GCGCN_OK) return rc__; \
    } while (0)

#define GCGCN_REQUIRE(cond, ...)                                        \
    do {                                                                \
        if (!(cond)) return ::gcgcn::fail(GCGCN_ERR_INVALID_ARG, __VA_ARGS__); \
    } while (0)

int sm_count();
int check_batch(const gcgcn_batch* bt);
int check_device_ptr(const void* p, const char* name);

// bump allocator over a caller-owned workspace
struct Arena {
    char* base;
    size_t cap;
    size_t off = 0;
    Arena(void* p, size_t bytes) : base(static_cast<char*>(p)), cap(bytes) {}
    template <typename T>
    T* take(size_t count) {
        size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
        if (base == nullptr || off + bytes > cap) return nullptr;
        T* p = reinterpret_cast<T*>(base + off);
        off += bytes;
        return p;
    }
};

static inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

// One launch per size class (padded n = 64, 48, 32, 16) when the batch carries the doc_order hint, so that small
// documents do not reserve the shared memory of the largest one: fn(count, first, nmax, order).
template <class LaunchFn>
inline int for_each_size_class(const gcgcn_batch* bt, LaunchFn fn) {
    if (bt->doc_order == nullptr) return fn(bt->num_docs, 0, bt->max_nodes, static_cast<const int*>(nullptr));
    static const int cap[4] = {64, 48, 32, 16};
    int first = 0;
    for (int c = 0; c < 4; ++c) {
        const int count = bt->class_end[c] - first;
        if (count > 0) GCGCN_TRY(fn(count, first, cap[c] < bt->max_nodes ? cap[c] : bt->max_nodes, bt->doc_order));
        first = bt->class_end[c] > first ? bt->class_end[c] : first;
    }
    return GCGCN_OK;
}

// ---- device helpers ------------------------------------------------------------------------
// sigmoid of a logit (C:355), within 1 ulp of torch.sigmoid: one definition for the loss kernels and the evaluation
__device__ __forceinline__ float logit_sigmoid(float z) { return 1.0f / (1.0f + expf(-z)); }
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- counter-based dropout (train mode of the block kernels) -------------------------------------
// keep-scale factor of element `idx` of dropout stream `stream` under `seed`: 0 with probability p, else 1/(1-p).
// One SplitMix64 hash serves the two elements of an even/odd index pair; forward and backward (and
// gcgcn_dropout_mask, which materialises a stream for the tests) regenerate the same values, so no mask is stored.
struct BlockDrop {
    unsigned long long seed;
    uint32_t thr_att, thr_gcn;      // p * 2^32 of the attention / GraphConv-output dropout (0 = off)
    float inv_att, inv_gcn;         // 1 / (1 - p)
    uint32_t s_att, s_gcn;          // stream ids
};
__host__ __device__ __forceinline__ unsigned long long drop_hash(unsigned long long seed, uint32_t stream,
                                                                  unsigned long long pair_idx) {
    unsigned long long z = seed + 0x9E3779B97F4A7C15ULL * (pair_idx + (static_cast<unsigned long long>(stream) << 56) + 1ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ float drop_keep(unsigned long long seed, uint32_t stream, unsigned long long idx,
                                                    uint32_t thr, float inv) {
    const unsigned long long h = drop_hash(seed, stream, idx >> 1);
    const uint32_t r = (idx & 1ULL) ? static_cast<uint32_t>(h >> 32) : static_cast<uint32_t>(h);
    return r >= thr ? inv : 0.f;
}
// idx even: the factors of idx and idx + 1 from one hash
__host__ __device__ __forceinline__ float2 drop_keep2(unsigned long long seed, uint32_t stream, unsigned long long idx,
                                                      uint32_t thr, float inv) {
    const unsigned long long h = drop_hash(seed, stream, idx >> 1);
    return make_float2(static_cast<uint32_t>(h) >= thr ? inv : 0.f, static_cast<uint32_t>(h >> 32) >= thr ? inv : 0.f);
}

// Streaming 4-element loads/stores of an edge vector slice, fp32 or bf16 storage, fp32 math.
// The n^2 x 128 tensors are read/written exactly once per pass: bypass L1 allocation.
template <typename T>
struct Vec4;

template <>
struct Vec4<float> {
    static __device__ __forceinline__ float4 load(const float* p) {
        float4 r;
        asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                     : "l"(p));
        return r;
    }
    static __device__ __forceinline__ void store(float* p, float4 v) {
        asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x),
                     "f"(v.y), "f"(v.z), "f"(v.w)
                     : "memory");
    }
};

template <>
struct Vec4<__nv_bfloat16> {
    static __device__ __forceinline__ float4 load(const __nv_bfloat16* p) {
        uint32_t a, b;
        asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
        float4 r;
        r.x = __uint_as_float(a << 16);
        r.y = __uint_as_float(a & 0xffff0000u);
        r.z = __uint_as_float(b << 16);
        r.w = __uint_as_float(b & 0xffff0000u);
        return r;
    }
    static __device__ __forceinline__ void store(__nv_bfloat16* p, float4 v) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y);
        __nv_bfloat162 hi = __floats2bfloat162_rn(v.z, v.w);
        uint32_t a = *reinterpret_cast<uint32_t*>(&lo);
        uint32_t b = *reinterpret_cast<uint32_t*>(&hi);
        asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(a), "r"(b)
                     : "memory");
    }
};

}  // namespace gcgcn
