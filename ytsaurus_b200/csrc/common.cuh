// common.cuh — shared device/host helpers for the ytgpu kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ytgpu.h"

namespace ytgpu {

using u8 = uint8_t;
using u16 = uint16_t;
using u32 = uint32_t;
using u64 = uint64_t;
using i32 = int32_t;
using i64 = int64_t;

constexpr int kNumSms = 148;  // B200: 2 dies x 74 SMs

// Kernel classes for the per-context CUDA-event timers (ytgpu_context_kernel_ms).
enum KernelClass { KC_RADIX_PASS = 0, KC_GATHER = 1, KC_EXTRACT = 2, KC_HISTOGRAM = 3, KC_PARTITION = 4,
                   KC_GROUPBY = 5, KC_DECODE = 6, KC_PASS_SKIPPED = 7, KC_SCATTER = 8, KC_SHUFFLE_SYNC = 9,
                   KC_REDUCE = 10, KC_COUNT = 11 };

struct Status {
    int code = YTGPU_OK;
    int cuda = 0;
    char msg[248] = {0};
    bool ok() const { return code == YTGPU_OK; }
};

Status make_status(int code, const char* fmt, ...);
Status cuda_status(cudaError_t e, const char* what);

#define YTGPU_CUDA_TRY(expr)                                   \
    do {                                                        \
        cudaError_t _e = (expr);                                \
        if (_e != cudaSuccess) return ::ytgpu::cuda_status(_e, #expr); \
    } while (0)

#define YTGPU_TRY(expr)                    \
    do {                                   \
        ::ytgpu::Status _s = (expr);       \
        if (!_s.ok()) return _s;           \
    } while (0)

// Device error flag bits written by kernels, checked by the host after the call.
enum DevErr : u32 {
    DE_UNSUPPORTED_TYPE = 1u << 0,   // Any / Composite / unknown type in a key column
    DE_SCHEMA_VIOLATION = 1u << 1,   // value type != declared type (or Null in a required column)
    DE_STRING_TOO_LONG = 1u << 2,    // string longer than the declared key width
    DE_PART_BAD_TYPE = 1u << 3,
    DE_PART_NEGATIVE = 1u << 4,
    DE_PART_OUT_OF_BOUNDS = 1u << 5,
    DE_PART_NO_COLUMN = 1u << 6,
    DE_TABLE_FULL = 1u << 7,
    DE_PEER_TIMEOUT = 1u << 8,       // a peer GPU did not reach the in-box shuffle's barrier in time
    DE_BAD_PARTITION_INDEX = 1u << 9,  // caller-supplied partition index outside [0, partition_count)
};

struct Context;  // context.cu

// Streaming loads/stores that do not pollute L1 (data touched once per pass).
__device__ __forceinline__ u64 ld_stream_u64(const u64* p) {
    u64 v;
    asm volatile("ld.global.nc.L1::no_allocate.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ u32 ld_stream_u32(const u32* p) {
    u32 v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_stream_u128(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream_u128(uint4* p, const uint4& v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w));
}
__device__ __forceinline__ u32 ld_volatile_u32(const u32* p) {
    u32 v;
    asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_volatile_u32(u32* p, u32 v) {
    asm volatile("st.volatile.global.u32 [%0], %1;" :: "l"(p), "r"(v));
}
__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ u32 lanemask_lt() {
    u32 m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

}  // namespace ytgpu
