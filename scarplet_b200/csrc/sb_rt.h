// Thin device-runtime layer used by every kernel in this library.
//
// Product build (nvcc, sm_100a): the macros below are the CUDA built-ins.
// Test build (-DSB_EMU, g++): the same kernel source is compiled against
// tests/emu/sb_emu.h, a fiber-per-CUDA-thread emulator, so that index logic can
// be checked on a machine without a GPU.  The emulator is test infrastructure:
// the product package never loads it (scarplet_b200/_lib.py only opens the
// CUDA library and raises if it is missing).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cmath>

#ifdef SB_EMU
#include "sb_emu.h"
#else
#include <cuda_runtime.h>

#define SB_GLOBAL __global__ void
#define SB_DEVICE __device__ __forceinline__
#define SB_HOSTDEV __host__ __device__ __forceinline__
#define SB_CONSTEXPR __host__ __device__ constexpr
#define SB_LAUNCH_BOUNDS(t, b) __launch_bounds__(t, b)
#define SB_RESTRICT __restrict__

SB_DEVICE int sb_tid() { return threadIdx.x; }
SB_DEVICE int sb_bx() { return blockIdx.x; }
SB_DEVICE int sb_by() { return blockIdx.y; }
SB_DEVICE int sb_bz() { return blockIdx.z; }
SB_DEVICE int sb_nbx() { return gridDim.x; }
SB_DEVICE int sb_nby() { return gridDim.y; }
SB_DEVICE void sb_sync() { __syncthreads(); }
// named barrier: `count` threads (a multiple of 32) of the block meet at barrier `id` (1..15)
SB_DEVICE void sb_bar(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
// signal named barrier `id` without waiting (the `count` includes the threads that will wait)
SB_DEVICE void sb_bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }
SB_DEVICE void* sb_shared() {
    extern __shared__ __align__(16) unsigned char sb_smem_raw[];
    return sb_smem_raw;
}
template <typename T> SB_DEVICE T sb_ldg(const T* p) { return __ldg(p); }
// read-once data (spectra, intermediate planes): do not let it evict the twiddle tables from L1
SB_DEVICE float2 sb_ld_stream(const float2* p) {
    float2 r;
    asm("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
SB_DEVICE float4 sb_ld_stream(const float4* p) {
    float4 r;
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
// read-twice-soon data (the sibling row group of the same CTA wants the other half of every
// sector): keep it in L1, but first in line for eviction
SB_DEVICE float4 sb_ld_shared_soon(const float4* p) {
    float4 r;
    asm("ld.global.nc.L1::evict_first.v4.f32 {%0, %1, %2, %3}, [%4];"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
// write-once data (the planes handed to the next kernel)
SB_DEVICE void sb_st_stream(float4* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// two adjacent values as one full-sector (float) / two-sector (double) store
SB_DEVICE void sb_st_pair(float4* p, float4 a, float4 b) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(a.x), "f"(a.y), "f"(a.z),
                 "f"(a.w), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w) : "memory");
}
SB_DEVICE void sb_st_pair(double4* p, double4 a, double4 b) { p[0] = a; p[1] = b; }
// one whole 32-byte sector (two adjacent float4) in one request; kept in L1 until its second
// reader (the thread that needs the mirrored element) has had it, first in line for eviction
SB_DEVICE void sb_ld_sector(const float4* p, float4& a, float4& b) {
    asm("ld.global.nc.L1::evict_first.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(p));
}
// hint: pull one 128-byte line towards L2 ahead of the loads that will need it
SB_DEVICE void sb_prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// a / b to ~2 ulp (MUFU.RCP + multiply); used where the tolerance is 1e-4
SB_DEVICE float sb_fdiv_fast(float a, float b) { return __fdividef(a, b); }

// IEEE operations that must not be contracted into FMAs (bit-exact float64
// parity with NumPy for the curvature stencil and the template window).
SB_DEVICE double sb_mul(double a, double b) { return __dmul_rn(a, b); }
SB_DEVICE double sb_add(double a, double b) { return __dadd_rn(a, b); }
SB_DEVICE double sb_sub(double a, double b) { return __dsub_rn(a, b); }
SB_DEVICE double sb_div(double a, double b) { return __ddiv_rn(a, b); }

typedef cudaStream_t sb_stream_t;

#define SB_LAUNCH(kern, grid, block, smem, stream, ...) \
    kern<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)

inline int sb_rt_malloc(void** p, size_t n) { return (int)cudaMalloc(p, n); }
inline int sb_rt_free(void* p) { return (int)cudaFree(p); }
inline int sb_rt_h2d(void* d, const void* h, size_t n, sb_stream_t s) {
    return (int)cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, s);
}
inline int sb_rt_d2h(void* h, const void* d, size_t n, sb_stream_t s) {
    return (int)cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, s);
}
inline int sb_rt_d2d(void* d, const void* s0, size_t n, sb_stream_t s) {
    return (int)cudaMemcpyAsync(d, s0, n, cudaMemcpyDeviceToDevice, s);
}
inline int sb_rt_memset(void* d, int v, size_t n, sb_stream_t s) {
    return (int)cudaMemsetAsync(d, v, n, s);
}
inline int sb_rt_sync(sb_stream_t s) { return (int)cudaStreamSynchronize(s); }
inline int sb_rt_mem_info(size_t* free_b, size_t* total_b) { return (int)cudaMemGetInfo(free_b, total_b); }
inline int sb_rt_last_error() { return (int)cudaGetLastError(); }
typedef cudaEvent_t sb_event_t;
inline int sb_rt_event_create(sb_event_t* e) { return (int)cudaEventCreate(e); }
inline int sb_rt_event_destroy(sb_event_t e) { return (int)cudaEventDestroy(e); }
inline int sb_rt_event_record(sb_event_t e, sb_stream_t s) { return (int)cudaEventRecord(e, s); }
inline float sb_rt_event_ms(sb_event_t a, sb_event_t b) { float ms = 0.f; cudaEventElapsedTime(&ms, a, b); return ms; }
inline const char* sb_rt_error_string(int e) { return cudaGetErrorString((cudaError_t)e); }
#endif

// bit casts
SB_DEVICE unsigned sb_float_bits(float v) { unsigned u; memcpy(&u, &v, 4); return u; }
SB_DEVICE float sb_bits_float(unsigned u) { float v; memcpy(&v, &u, 4); return v; }

// ---- precision-generic vector types ------------------------------------------
template <typename R> struct Vec;
template <> struct Vec<float> { typedef float2 v2; typedef float4 v4; };
template <> struct Vec<double> { typedef double2 v2; typedef double4 v4; };

template <typename R> SB_DEVICE typename Vec<R>::v2 mk2(R x, R y);
template <> SB_DEVICE float2 mk2<float>(float x, float y) { return make_float2(x, y); }
template <> SB_DEVICE double2 mk2<double>(double x, double y) { return make_double2(x, y); }
template <typename R> SB_DEVICE typename Vec<R>::v4 mk4(R x, R y, R z, R w);
template <> SB_DEVICE float4 mk4<float>(float x, float y, float z, float w) { return make_float4(x, y, z, w); }
template <> SB_DEVICE double4 mk4<double>(double x, double y, double z, double w) { return make_double4(x, y, z, w); }

// read-only loads of the vector types (double4 goes as two 16-byte loads)
SB_DEVICE float2 ld2(const float2* p) { return sb_ldg(p); }
SB_DEVICE double2 ld2(const double2* p) { return sb_ldg(p); }
SB_DEVICE float4 ld4(const float4* p) { return sb_ldg(p); }
SB_DEVICE double4 ld4(const double4* p) {
    const double2 a = sb_ldg(reinterpret_cast<const double2*>(p));
    const double2 b = sb_ldg(reinterpret_cast<const double2*>(p) + 1);
    return make_double4(a.x, a.y, b.x, b.y);
}
