// common.cuh -- shared device helpers for libtrtx_hot (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "trtx_hot.h"

namespace trtx {

constexpr int kWarp = 32;
constexpr size_t kAlign = 256;  // workspace sub-buffer alignment (rcnn/cuda_utils.h:7 uses the same)

__host__ __device__ inline size_t align_up(size_t v, size_t a = kAlign) { return (v + a - 1) / a * a; }

// ---- step timeline (probe build only: build(probe=True) / -DTRTX_NMS_PROBE; release builds carry no stamps) ----
// Every launch of the scan, NMS and letterbox kernels takes the next record of the buffer registered with
// trtx_probe_set_timeline (this host thread's launches, in launch order; null once the buffer is full) through its
// argument block.  Record: [kind, CTAs, then per CTA (first %globaltimer stamp at entry, last stamp at exit)], in ns.
// The caller zeroes the buffer before each run (exit stamps are atomic maxima).
#ifdef TRTX_NMS_PROBE
enum TlKind { kTlScan = 1, kTlNms = 2, kTlLetterbox = 3 };
constexpr int kTlMaxCtas = 8192;
constexpr size_t kTlRecordWords = 2 + 2 * (size_t)kTlMaxCtas;
unsigned long long* tl_take();  // nms.cu
__device__ __forceinline__ unsigned long long tl_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
struct TlStamp {
    unsigned long long* r;
    __device__ __forceinline__ TlStamp(unsigned long long* rec, int kind) : r(nullptr) {
        const unsigned ncta = gridDim.x * gridDim.y * gridDim.z;
        if (!rec || ncta > (unsigned)kTlMaxCtas) return;
        const unsigned cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        r = rec + 2 + 2 * (size_t)cta;
        if (threadIdx.x + threadIdx.y + threadIdx.z == 0) {
            r[0] = tl_now();
            if (cta == 0) {
                rec[0] = (unsigned long long)kind;
                rec[1] = ncta;
            }
        }
    }
    __device__ __forceinline__ ~TlStamp() {  // runs at every return: one atomic max per (warp, exit point)
        if (r && (threadIdx.x & 31) == (unsigned)(__ffs(__activemask()) - 1)) atomicMax(r + 1, tl_now());
    }
};
#define TRTX_TL_FIELD unsigned long long* tl;
#define TRTX_TL(args, kind) TlStamp tl_stamp_((args).tl, (kind))
#define TRTX_TL_TAKE(args) ((args).tl = tl_take())
#else
#define TRTX_TL_FIELD
#define TRTX_TL(args, kind) do { } while (0)
#define TRTX_TL_TAKE(args) do { } while (0)
#endif

// thread-local last CUDA error (trtx_last_cuda_error)
extern thread_local int g_last_cuda_error;
inline int check_launch() {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        g_last_cuda_error = (int)e;
        return TRTX_ERR_CUDA;
    }
    return TRTX_OK;
}

// ---- streaming loads: read-once data bypasses L1 allocation (guide: Guideline 13/14) ----
__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float ldg_stream_f1(const float* p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
// 4 halfs (8 bytes) -> 4 floats
__device__ __forceinline__ float4 ldg_stream_h4(const __half* p) {
    uint32_t a, b;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
    __half2 h0 = *reinterpret_cast<__half2*>(&a);
    __half2 h1 = *reinterpret_cast<__half2*>(&b);
    float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
    return make_float4(f0.x, f0.y, f1.x, f1.y);
}
// 8 halfs (16 bytes), raw
__device__ __forceinline__ uint4 ldg_stream_h8(const __half* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ float ldg_stream_h1(const __half* p) {
    unsigned short r;
    asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(r) : "l"(p));
    return __half2float(__ushort_as_half(r));
}

template <typename T>
struct Elem;
template <>
struct Elem<float> {
    static __device__ __forceinline__ float4 ld4(const float* p) { return ldg_stream_f4(p); }
    static __device__ __forceinline__ float ld1(const float* p) { return ldg_stream_f1(p); }
    static __device__ __forceinline__ float ld1_cached(const float* p) { return __ldg(p); }
};
template <>
struct Elem<__half> {
    static __device__ __forceinline__ float4 ld4(const __half* p) { return ldg_stream_h4(p); }
    static __device__ __forceinline__ float ld1(const __half* p) { return ldg_stream_h1(p); }
    static __device__ __forceinline__ float ld1_cached(const __half* p) { return __half2float(__ldg(p)); }
};

// The reference's Logist(): 1.0f / (1.0f + expf(-x)), IEEE division, CUDA expf
// (yolov8/plugin/yololayer.cu:174-176).  No fast-math anywhere in this library.
__device__ __forceinline__ float logist(float x) { return 1.0f / (1.0f + expf(-x)); }

// order-preserving float -> uint32 (larger float => larger key); -0.0 < +0.0 like cub's radix twiddle
__device__ __forceinline__ uint32_t float_key(float f) {
    uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ int warp_excl_scan(int v, int lane, int* total) {
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    *total = __shfl_sync(0xffffffffu, x, 31);
    return x - v;
}

}  // namespace trtx
