// Shared helpers for the s2d_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/s2d_b200.h"

namespace s2d {

void set_error(const char* fmt, ...);

#define S2D_CHECK_ARG(cond, ...)            \
    do {                                    \
        if (!(cond)) {                      \
            s2d::set_error(__VA_ARGS__);    \
            return -1;                      \
        }                                   \
    } while (0)

#define S2D_CHECK_LAUNCH(name)                                                       \
    do {                                                                             \
        cudaError_t e_ = cudaGetLastError();                                         \
        if (e_ != cudaSuccess) {                                                     \
            s2d::set_error("%s: launch failed: %s", name, cudaGetErrorString(e_));   \
            return -2;                                                               \
        }                                                                            \
    } while (0)

// Device of the caller's stream made current for the duration of a C-ABI call (and restored afterwards): launches,
// memsets, occupancy queries and the SM count then all refer to the device the stream lives on, whatever device
// the calling thread had current. The legacy / per-thread default stream handles keep the current device.
struct StreamDeviceGuard {
    int dev = 0, prev = 0;
    explicit StreamDeviceGuard(void* stream) {
        cudaGetDevice(&prev);
        dev = prev;
        cudaStream_t st = (cudaStream_t)stream;
        if (st == nullptr || st == cudaStreamLegacy || st == cudaStreamPerThread) return;
        // a capturing stream must not be queried (it invalidates the capture); whoever captures has the stream's
        // device current already (CUDA requires it for the launches being recorded)
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { cudaGetLastError(); return; }
        if (cap != cudaStreamCaptureStatusNone) return;
        int d = -1;
        if (cudaStreamGetDevice(st, &d) == cudaSuccess && d >= 0) dev = d;
        else cudaGetLastError();
        if (dev != prev) cudaSetDevice(dev);
    }
    ~StreamDeviceGuard() { if (dev != prev) cudaSetDevice(prev); }
    StreamDeviceGuard(const StreamDeviceGuard&) = delete;
    StreamDeviceGuard& operator=(const StreamDeviceGuard&) = delete;
};
#define S2D_ENTER(stream) s2d::StreamDeviceGuard s2d_dev_guard_(stream)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: set it once per (kernel, device).
constexpr int S2D_MAX_DEVICES = 64;
template <typename K>
inline cudaError_t opt_in_smem(K kfn, int smem, bool (&done)[S2D_MAX_DEVICES]) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < S2D_MAX_DEVICES && done[dev]) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess && dev >= 0 && dev < S2D_MAX_DEVICES) done[dev] = true;
    return e;
}

// Device-side bounds checks of the debug build (make check): trap on an out-of-range index. Compiles to nothing
// in the product library.
#ifdef S2D_BOUNDS_CHECK
#define S2D_DEV_ASSERT(cond) do { if (!(cond)) { printf("S2D_DEV_ASSERT failed: %s (%s:%d) block (%d,%d,%d) thread %d\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, (int)blockIdx.y, (int)blockIdx.z, (int)threadIdx.x); __trap(); } } while (0)
#define S2D_PV_BOUNDS_CHECK 1
#else
#define S2D_DEV_ASSERT(cond) do { } while (0)
#endif

// streaming 128-bit load that does not pollute L1 (read-once data: tracks, flags, labels)
__device__ __forceinline__ int4 ld_stream(const int4* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(0xffffffffu, v); }

// inclusive sum of x over the 32 lanes of a full warp (1-D blocks: lane = threadIdx.x & 31)
template <typename T>
__device__ __forceinline__ T warp_incl_scan(T x) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const T u = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += u; }
    return x;
}

// exclusive prefix of x over a block of THREADS threads (every thread calls it); total = the block sum. wsum: THREADS / 32
// shared slots. Ends with a barrier, so the caller may reuse wsum at once. The warp sums are read eight at a time: a full
// unroll keeps all 32 of a 1024-thread block in flight, which costs up to 64 registers per thread.
template <int THREADS, typename T>
__device__ __forceinline__ T block_excl_scan(T x, T* wsum, T& total) {
    S2D_DEV_ASSERT(blockDim.x == THREADS);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const T incl = warp_incl_scan(x);
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    T before = 0;
    total = 0;
#pragma unroll 8
    for (int w = 0; w < THREADS / 32; ++w) { const T s = wsum[w]; if (w < warp) before += s; total += s; }
    __syncthreads();
    return before + incl - x;
}

// out[0, n] = exclusive prefix of in[0, n) as int64 (out[n] = the sum), *total = the sum: one 1024-thread CTA on st.
// Returns 0, or -2 with the error set when the launch fails. Defined in label_rle.cu.
int launch_offsets(const int32_t* in, int64_t n, int64_t* out, int64_t* total, cudaStream_t st);

__device__ __forceinline__ int cdiv(int a, int b) { return (a + b - 1) / b; }

}  // namespace s2d
