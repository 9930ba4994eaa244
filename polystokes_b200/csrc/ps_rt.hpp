// ps_rt.hpp -- thin runtime layer under the kernels.
//
// Product build (nvcc, sm_100a): ps_for() launches a grid-stride CUDA kernel, memory is cudaMalloc'd,
// atomics are the hardware ones.  There is NO CPU fallback in the product library.
//
// Test-only build (-DPS_EMULATE, g++): the *same* per-thread bodies are executed serially on the
// host so the index/stencil logic can be checked against the oracle on a machine without a GPU
// (tests/test_emulated_kernels.py).  That build produces a differently named library
// (libpolystokes_emul.so) which the python package never loads.
#pragma once
#include <cstdint>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <stdexcept>
#include <vector>
#include <algorithm>

#ifndef PS_EMULATE
#include <cuda_runtime.h>
#define PS_HD __host__ __device__ __forceinline__
#define PS_D __device__ __forceinline__
#define PS_LAMBDA [=] __device__
#else
#define PS_HD inline
#define PS_D inline
#define PS_LAMBDA [=]
typedef void* cudaStream_t;
#endif

namespace ps {

struct Error : std::runtime_error { using std::runtime_error::runtime_error; };
extern thread_local int64_t g_launches;   // kernels launched since the step began (ps_stats::gpu_launches)
#define PS_COUNT_LAUNCH(n) (::ps::g_launches += (n))
// Rank threads of a ps_create_multi handle (several GPUs, ONE process): cudaFree waits for the work of every device that maps the
// allocation (peer access is on), so a free issued while another rank's kernel spins on a flag THIS rank has yet to raise would
// never return.  Such threads park their frees here; the caller releases them once every rank has finished the collective call.
extern thread_local std::vector<void*>* g_deferredFree;
// where a rank thread currently is (a string literal), for the watchdog of the multi handle
extern thread_local const char* volatile* g_where;
#define PS_WHERE(s) do { if (::ps::g_where) *::ps::g_where = (s); } while (0)

#ifndef PS_EMULATE
inline void check(cudaError_t e, const char* what, const char* file, int line) {
    if (e != cudaSuccess) {
        char buf[512];
        snprintf(buf, sizeof buf, "CUDA error %s (%s) at %s:%d", cudaGetErrorString(e), what, file, line);
        throw Error(buf);
    }
}
#define PS_CUDA(x) ::ps::check((x), #x, __FILE__, __LINE__)

// SM count of the CURRENT device (grids are sized in multiples of it); cached per host thread and device
inline int sm_count() {
    static thread_local int cachedDev = -1, cachedSms = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return cachedSms;
    if (dev != cachedDev) { int sms = 0; if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) { cachedSms = sms; cachedDev = dev; } }
    return cachedSms;
}
template <class F>
__global__ void __launch_bounds__(256) ps_for_kernel(int64_t n, F f) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) f(i);
}
// one thread per item, grid capped at a multiple of the SM count (16 CTAs of 256 threads per SM)
template <class F>
inline void ps_for(cudaStream_t s, int64_t n, F f) {
    if (n <= 0) return;
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    ps_for_kernel<<<(unsigned)blocks, 256, 0, s>>>(n, f);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
// the same over the index range [lo, hi)
template <class F>
__global__ void __launch_bounds__(256) ps_for_range_kernel(int64_t lo, int64_t n, F f) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) f(lo + i);
}
template <class F>
inline void ps_for_range(cudaStream_t s, int64_t lo, int64_t hi, F f) {
    const int64_t n = hi - lo;
    if (n <= 0) return;
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    ps_for_range_kernel<<<(unsigned)blocks, 256, 0, s>>>(lo, n, f);
    PS_COUNT_LAUNCH(1);
    PS_CUDA(cudaGetLastError());
}
inline void* dev_alloc_bytes(size_t bytes) { void* p = nullptr; if (bytes == 0) bytes = 16; PS_CUDA(cudaMalloc(&p, bytes)); return p; }
inline void dev_free(void* p) { if (!p) return; if (g_deferredFree) g_deferredFree->push_back(p); else cudaFree(p); }
inline void dev_memset(void* p, int v, size_t bytes, cudaStream_t s) { if (bytes) PS_CUDA(cudaMemsetAsync(p, v, bytes, s)); }
inline void copy_h2d(void* d, const void* h, size_t bytes, cudaStream_t s) { if (bytes) PS_CUDA(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s)); }
inline void copy_d2h(void* h, const void* d, size_t bytes, cudaStream_t s) { if (bytes) { PS_CUDA(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, s)); PS_CUDA(cudaStreamSynchronize(s)); } }
inline void copy_d2d(void* d, const void* s_, size_t bytes, cudaStream_t s) { if (bytes) PS_CUDA(cudaMemcpyAsync(d, s_, bytes, cudaMemcpyDeviceToDevice, s)); }
// input pointers may be host or device (ps_fields_in::memory)
inline void copy_any2d(void* d, const void* src, size_t bytes, bool srcOnDevice, cudaStream_t s) { if (bytes) PS_CUDA(cudaMemcpyAsync(d, src, bytes, srcOnDevice ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s)); }
inline void copy_d2any(void* dst, const void* d, size_t bytes, bool dstOnDevice, cudaStream_t s) { if (bytes) PS_CUDA(cudaMemcpyAsync(dst, d, bytes, dstOnDevice ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s)); }
inline void stream_sync(cudaStream_t s) { PS_CUDA(cudaStreamSynchronize(s)); }

// never-contracted arithmetic for values that must match the reference's separately rounded ops
PS_D double mul_rn(double a, double b) { return __dmul_rn(a, b); }
PS_D double add_rn(double a, double b) { return __dadd_rn(a, b); }
PS_D double sub_rn(double a, double b) { return __dsub_rn(a, b); }
PS_D float fmul_rn(float a, float b) { return __fmul_rn(a, b); }
PS_D float fadd_rn(float a, float b) { return __fadd_rn(a, b); }
PS_D float fsub_rn(float a, float b) { return __fsub_rn(a, b); }
PS_D int atomic_min(int* a, int v) { return atomicMin(a, v); }
PS_D int atomic_max(int* a, int v) { return atomicMax(a, v); }
PS_D int atomic_add(int* a, int v) { return atomicAdd(a, v); }
PS_D unsigned long long atomic_add(unsigned long long* a, unsigned long long v) { return atomicAdd(a, v); }
PS_D int atomic_or(int* a, int v) { return atomicOr(a, v); }
#else
template <class F>
inline void ps_for(cudaStream_t, int64_t n, F f) { for (int64_t i = 0; i < n; ++i) f(i); }
template <class F>
inline void ps_for_range(cudaStream_t, int64_t lo, int64_t hi, F f) { for (int64_t i = lo; i < hi; ++i) f(i); }
inline void* dev_alloc_bytes(size_t bytes) { if (bytes == 0) bytes = 16; void* p = calloc(1, bytes); if (!p) throw Error("calloc failed"); return p; }
inline void dev_free(void* p) { free(p); }
inline void dev_memset(void* p, int v, size_t bytes, cudaStream_t) { if (bytes) memset(p, v, bytes); }
inline void copy_h2d(void* d, const void* h, size_t bytes, cudaStream_t) { if (bytes) memcpy(d, h, bytes); }
inline void copy_d2h(void* h, const void* d, size_t bytes, cudaStream_t) { if (bytes) memcpy(h, d, bytes); }
inline void copy_d2d(void* d, const void* s_, size_t bytes, cudaStream_t) { if (bytes) memcpy(d, s_, bytes); }
inline void copy_any2d(void* d, const void* src, size_t bytes, bool, cudaStream_t) { if (bytes) memcpy(d, src, bytes); }
inline void copy_d2any(void* dst, const void* d, size_t bytes, bool, cudaStream_t) { if (bytes) memcpy(dst, d, bytes); }
inline void stream_sync(cudaStream_t) {}
using std::min; using std::max;
inline double mul_rn(double a, double b) { return a * b; }   // built with -ffp-contract=off
inline double add_rn(double a, double b) { return a + b; }
inline double sub_rn(double a, double b) { return a - b; }
inline float fmul_rn(float a, float b) { return a * b; }
inline float fadd_rn(float a, float b) { return a + b; }
inline float fsub_rn(float a, float b) { return a - b; }
inline int atomic_min(int* a, int v) { int o = *a; if (v < o) *a = v; return o; }
inline int atomic_max(int* a, int v) { int o = *a; if (v > o) *a = v; return o; }
inline int atomic_add(int* a, int v) { int o = *a; *a += v; return o; }
inline unsigned long long atomic_add(unsigned long long* a, unsigned long long v) { unsigned long long o = *a; *a += v; return o; }
inline int atomic_or(int* a, int v) { int o = *a; *a |= v; return o; }
#endif

// owning device buffer
template <class T>
struct DBuf {
    T* p = nullptr;
    size_t n = 0;
    bool view = false;                   // p points into somebody else's allocation (adopt)
    DBuf() = default;
    DBuf(const DBuf&) = delete;
    DBuf& operator=(const DBuf&) = delete;
    ~DBuf() { if (!view) dev_free(p); }
    void alloc(size_t count) {
        if (count <= n && p) return;     // grow-only: buffers persist across steps (no per-step cudaMalloc)
        if (!view) dev_free(p);
        p = nullptr; n = 0; view = false;
        p = (T*)dev_alloc_bytes(count * sizeof(T)); n = count;
    }
    // non-owning window of `count` elements at q
    void adopt(T* q, size_t count) { if (!view) dev_free(p); p = q; n = count; view = true; }
    // hands the allocation over (the caller frees it with dev_free)
    T* release() { T* q = view ? nullptr : p; p = nullptr; n = 0; view = false; return q; }
    void zero(cudaStream_t s, size_t count) { dev_memset(p, 0, count * sizeof(T), s); }
    void fill_byte(cudaStream_t s, int v, size_t count) { dev_memset(p, v, count * sizeof(T), s); }
    std::vector<T> to_host(cudaStream_t s, size_t count) const { std::vector<T> h(count); copy_d2h(h.data(), p, count * sizeof(T), s); return h; }
    void from_host(cudaStream_t s, const T* h, size_t count) { alloc(count); copy_h2d(p, h, count * sizeof(T), s); }
};

// Grow-only scratch buffers of the setup stages.  They belong to ONE solver (its device, its stream): every C-ABI entry point
// points `g_scratch` at the handle's instance for the duration of the call (ps_api.cu), so two handles on different devices
// driven from one host thread never share device memory, and a handle called from many host threads does not leak a copy per thread.
struct Scratch {
    DBuf<uint8_t> selTmp, sortTmp, scanTmp, haloFlag;
    DBuf<int32_t> selCnt, selStaging, dremap, keys, kt, vt;
    DBuf<int> bb, rc;
    DBuf<unsigned long long> sums;
    DBuf<float> planes;
    DBuf<double> applyX, applyY;
    DBuf<uint8_t> gather;                // staging of the pieces sent to rank 0 (ps_api.cu, gather_bytes)
};
extern thread_local Scratch* g_scratch;
inline Scratch& scratch() { static thread_local Scratch fallback; return g_scratch ? *g_scratch : fallback; }

}  // namespace ps
