// KERNEL-LOGIC EMULATOR (development / test infrastructure only; NOT a product path and NOT a
// fallback: the python package refuses to load a library built with it, see
// halo2_scaffold_b200/_lib.py).
//
// The build container has nvcc but no GPU, and GPU time is rationed.  To unit-test the *same
// kernel sources* that ship in libh2b200.so, `make emu` compiles csrc/*.cu with g++ and
// -DH2B_EMU against this header, which provides just enough of the CUDA execution model on the
// CPU: every CUDA thread of a block is a ucontext fiber, __syncthreads()/warp shuffles are fiber
// barriers, blocks are distributed over a few OS threads, `__shared__` becomes
// `static thread_local`.  Device-side inline PTX is replaced by portable C (the PTX itself is
// verified separately by tools/gen_field_ptx.py's interpreter).
#pragma once
#include <ucontext.h>

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
#define __restrict__
#define __launch_bounds__(...)
#define __align__(x) alignas(x)
#define __shared__ static thread_local
#define __constant__ static

struct uint2 { uint32_t x, y; };
struct alignas(16) uint4 { uint32_t x, y, z, w; };
struct alignas(16) ulonglong2 { unsigned long long x, y; };
static inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { return uint4{x, y, z, w}; }
static inline uint2 make_uint2(uint32_t x, uint32_t y) { return uint2{x, y}; }
struct uint3 { unsigned x, y, z; };
struct dim3 {
    unsigned x, y, z;
    dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};

typedef int cudaError_t;
typedef void* cudaStream_t;
typedef void* cudaEvent_t;
enum { cudaSuccess = 0, cudaErrorMemoryAllocation = 2, cudaErrorInvalidValue = 1 };
enum cudaMemcpyKind { cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };
enum { cudaFuncAttributeMaxDynamicSharedMemorySize = 8, cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2 };
struct cudaDeviceProp { int multiProcessorCount; size_t totalGlobalMem; char name[64]; int major, minor; size_t sharedMemPerBlockOptin; };

namespace emu {

struct Barrier { unsigned expected = 0, arrived = 0; unsigned long gen = 0; };

struct Fiber {
    ucontext_t ctx;
    uint3 tid;
    bool done = false;
};

struct BlockCtx {
    ucontext_t sched;
    std::vector<Fiber> fibers;
    char* stacks = nullptr;
    size_t stacks_size = 0;
    Fiber* cur = nullptr;
    Barrier block_bar;
    std::vector<Barrier> warp_bar;
    std::vector<uint64_t> warp_scratch;   // 32 x u64 per warp
    std::function<void()> body;
    std::vector<char> dyn_smem;
};

extern thread_local BlockCtx* g_blk;
extern thread_local uint3 threadIdx, blockIdx;
extern thread_local dim3 blockDim, gridDim;
extern thread_local char* dyn_smem_ptr;

void yield_();
void barrier_wait(Barrier& b);
void launch(dim3 grid, dim3 block, size_t smem, const std::function<void()>& body);

inline unsigned linear_tid() { return threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z); }
inline unsigned lane_id() { return linear_tid() & 31; }
inline unsigned warp_id() { return linear_tid() >> 5; }

template <class T>
inline T shfl_generic(T v, unsigned src_lane) {
    static_assert(sizeof(T) <= 8, "shfl width");
    unsigned w = warp_id();
    uint64_t* sc = &g_blk->warp_scratch[w * 32];
    uint64_t raw = 0;
    memcpy(&raw, &v, sizeof(T));
    sc[lane_id()] = raw;
    barrier_wait(g_blk->warp_bar[w]);
    uint64_t got = sc[src_lane & 31];
    barrier_wait(g_blk->warp_bar[w]);
    T out;
    memcpy(&out, &got, sizeof(T));
    return out;
}

}  // namespace emu

using emu::blockDim;
using emu::blockIdx;
using emu::gridDim;
using emu::threadIdx;

static inline void __syncthreads() { emu::barrier_wait(emu::g_blk->block_bar); }
static inline void __syncwarp(unsigned = 0xffffffffu) { emu::barrier_wait(emu::g_blk->warp_bar[emu::warp_id()]); }
template <class T> static inline T __shfl_sync(unsigned, T v, int src, int width = 32) {
    unsigned base = emu::lane_id() & ~(unsigned)(width - 1);
    return emu::shfl_generic(v, base + ((unsigned)src & (width - 1)));
}
template <class T> static inline T __shfl_xor_sync(unsigned, T v, int m, int = 32) { return emu::shfl_generic(v, emu::lane_id() ^ (unsigned)m); }
template <class T> static inline T __shfl_down_sync(unsigned, T v, unsigned d, int = 32) {
    unsigned s = emu::lane_id() + d;
    return emu::shfl_generic(v, s < 32 ? s : emu::lane_id());
}
template <class T> static inline T __shfl_up_sync(unsigned, T v, unsigned d, int = 32) {
    unsigned l = emu::lane_id();
    return emu::shfl_generic(v, l >= d ? l - d : l);
}
static inline unsigned __ballot_sync(unsigned, int pred) {
    unsigned r = 0;
    for (int i = 0; i < 32; ++i) r |= (emu::shfl_generic<unsigned>(pred ? 1u : 0u, i) & 1u) << i;
    return r;
}
static inline unsigned __match_any_sync(unsigned, unsigned key) {
    unsigned r = 0;
    for (int i = 0; i < 32; ++i) r |= (emu::shfl_generic<unsigned>(key, i) == key ? 1u : 0u) << i;
    return r;
}
static inline int __any_sync(unsigned m, int pred) { return __ballot_sync(m, pred) != 0; }
static inline int __all_sync(unsigned m, int pred) { return __ballot_sync(m, pred) == 0xffffffffu; }
static inline int __popc(unsigned x) { return __builtin_popcount(x); }
static inline int __clz(int x) { return x == 0 ? 32 : __builtin_clz((unsigned)x); }
static inline int __ffs(int x) { return __builtin_ffs(x); }
static inline unsigned __brev(unsigned x) {
    unsigned r = 0;
    for (int i = 0; i < 32; ++i) { r = (r << 1) | (x & 1); x >>= 1; }
    return r;
}
static inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned)(((uint64_t)a * b) >> 32); }
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned s) {
    uint64_t v = ((uint64_t)hi << 32) | lo;
    return (unsigned)(v >> (s & 31));
}
static inline unsigned __funnelshift_l(unsigned lo, unsigned hi, unsigned s) {
    uint64_t v = ((uint64_t)hi << 32) | lo;
    return (unsigned)((v << (s & 31)) >> 32);
}

// atomics: blocks may run on different OS threads
static inline unsigned atomicAdd(unsigned* p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline int atomicAdd(int* p, int v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline unsigned atomicMax(unsigned* p, unsigned v) {
    unsigned old = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (old < v && !__atomic_compare_exchange_n(p, &old, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
    return old;
}
static inline unsigned atomicOr(unsigned* p, unsigned v) { return __atomic_fetch_or(p, v, __ATOMIC_RELAXED); }
static inline unsigned atomicExch(unsigned* p, unsigned v) { return __atomic_exchange_n(p, v, __ATOMIC_RELAXED); }
static inline void __threadfence() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
template <class T> static inline T __ldg(const T* p) { return *p; }

// ---- runtime API subset -------------------------------------------------------------------
// the runtime's per-thread last error: a failed cudaMalloc leaves it set until cudaGetLastError reads it, so a caller that does
// not clear it sees its next launch check fail
namespace emu { inline thread_local cudaError_t last_error = cudaSuccess; }
static inline cudaError_t cudaMalloc(void** p, size_t n) {
    *p = aligned_alloc(256, ((n + 255) / 256) * 256 + 256);
    if (*p) return cudaSuccess;
    emu::last_error = cudaErrorMemoryAllocation;
    return cudaErrorMemoryAllocation;
}
template <class T> static inline cudaError_t cudaMalloc(T** p, size_t n) { return cudaMalloc((void**)p, n); }
static inline cudaError_t cudaFree(void* p) { free(p); return cudaSuccess; }
static inline cudaError_t cudaMallocHost(void** p, size_t n) { return cudaMalloc(p, n); }
static inline cudaError_t cudaFreeHost(void* p) { free(p); return cudaSuccess; }
template <class T> static inline cudaError_t cudaMallocHost(T** p, size_t n) { return cudaMalloc((void**)p, n); }
static inline cudaError_t cudaHostRegister(void*, size_t, unsigned) { return cudaSuccess; }
static inline cudaError_t cudaHostUnregister(void*) { return cudaSuccess; }
static inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t = 0) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpy2DAsync(void* d, size_t dpitch, const void* s, size_t spitch, size_t width, size_t height, cudaMemcpyKind, cudaStream_t = 0) {
    for (size_t r = 0; r < height; ++r) memcpy((char*)d + r * dpitch, (const char*)s + r * spitch, width);
    return cudaSuccess;
}
static inline cudaError_t cudaMemcpyPeer(void* d, int, const void* s, int, size_t n) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpyPeerAsync(void* d, int, const void* s, int, size_t n, cudaStream_t = 0) { memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaDeviceCanAccessPeer(int* can, int, int) { *can = 1; return cudaSuccess; }
static inline cudaError_t cudaDeviceEnablePeerAccess(int, unsigned) { return cudaSuccess; }
static inline cudaError_t cudaMemset(void* d, int v, size_t n) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t = 0) { memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemset2DAsync(void* d, size_t pitch, int v, size_t width, size_t height, cudaStream_t = 0) {
    for (size_t r = 0; r < height; ++r) memset((char*)d + r * pitch, v, width);
    return cudaSuccess;
}
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = nullptr; return cudaSuccess; }
static inline cudaError_t cudaStreamCreate(cudaStream_t* s) { *s = nullptr; return cudaSuccess; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
static inline cudaError_t cudaGetLastError() { const cudaError_t e = emu::last_error; emu::last_error = cudaSuccess; return e; }
static inline cudaError_t cudaPeekAtLastError() { return emu::last_error; }
static inline const char* cudaGetErrorString(cudaError_t) { return "emu"; }
static inline cudaError_t cudaSetDevice(int) { return cudaSuccess; }
static inline cudaError_t cudaGetDevice(int* d) { *d = 0; return cudaSuccess; }
// H2B_EMU_DEVICES=D makes the emulator report D devices (they share the host heap): the multi-device host logic -- point-range
// sharding, sharded base sets, round-robin columns -- runs under the CPU suite
static inline cudaError_t cudaGetDeviceCount(int* n) { const char* e = getenv("H2B_EMU_DEVICES"); *n = (e && atoi(e) >= 1 && atoi(e) <= 16) ? atoi(e) : 1; return cudaSuccess; }
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp* p, int) {
    memset(p, 0, sizeof(*p)); p->multiProcessorCount = 148; p->totalGlobalMem = (size_t)180 << 30; strcpy(p->name, "emu"); p->major = 10;
    p->sharedMemPerBlockOptin = 227 * 1024; return cudaSuccess;
}
template <class F> static inline cudaError_t cudaFuncSetAttribute(F, int, int) { return cudaSuccess; }
static inline cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = nullptr; return cudaSuccess; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = nullptr; return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t = 0) { return cudaSuccess; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0.f; return cudaSuccess; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned = 0) { return cudaSuccess; }
static inline cudaError_t cudaMemGetInfo(size_t* f, size_t* t) { *f = (size_t)8 << 30; *t = (size_t)8 << 30; return cudaSuccess; }

// kernel launch: H2B_LAUNCH(kernel, grid, block, smem, stream, args...)
namespace h2b { inline void count_launch(); }
#define H2B_LAUNCH(kern, grid, block, smem, stream, ...) \
    (h2b::count_launch(), emu::launch(dim3(grid), dim3(block), (size_t)(smem), [&]() { kern(__VA_ARGS__); }))
#define H2B_DYN_SMEM(T, name) T* name = reinterpret_cast<T*>(emu::dyn_smem_ptr)
