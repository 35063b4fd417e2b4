// common.cuh -- error plumbing and small device helpers shared by all kernels of
// libmnf_b200.so.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/mnf_b200.h"

namespace mnf {

// thread-local error string behind mnf_last_error()
char *err_buf();
int fail(int code, const char *fmt, ...);

#define MNF_REQUIRE(cond, code, ...)                       \
    do {                                                   \
        if (!(cond)) return ::mnf::fail((code), __VA_ARGS__); \
    } while (0)

#define MNF_CUDA(expr)                                                                     \
    do {                                                                                   \
        cudaError_t e__ = (expr);                                                          \
        if (e__ != cudaSuccess)                                                            \
            return ::mnf::fail((int)e__, "%s failed: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

// process-wide count of kernel launches made by this library (mnf_launch_count(); bench.py reports it)
unsigned long long &launch_counter();

// per-launch-site tally behind mnf_launch_stats() (diagnostics: which kernels a timed region really ran)
void note_launch(const char *what);

inline int launch_status(const char *what) {
    ++launch_counter();
    note_launch(what);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail((int)e, "%s launch failed: %s", what, cudaGetErrorString(e));
    return 0;
}

struct DeviceProps {
    int sm_count;
    int smem_optin;
    int cc_major, cc_minor;
};
// cached per device, thread-safe (function-local statics); returns nullptr on error
const DeviceProps *device_props();

// output size of a zero-padded, strided, dilated convolution along one axis; 0 when the padded input is narrower than
// the dilated filter, whose extent is dil * (ks - 1) + 1
__host__ __device__ inline int conv_out_size(int in, int ks, int pad, int stride, int dil = 1) {
    const int ext = dil * (ks - 1) + 1;
    return in + 2 * pad >= ext ? (in + 2 * pad - ext) / stride + 1 : 0;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// streaming (read-once / write-once) global accesses: keep L1 for weights
__device__ __forceinline__ float2 ld_stream2(const float2 *p) {
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ float4 ld_stream4(const float4 *p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream2(float2 *p, float2 v) {
    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream4(float4 *p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w)
                 : "memory");
}

}  // namespace mnf
