// 128-bit bf16 vectors of the memory-bound kernels (elementwise.cu, elementwise_bwd.cu, cmix.cu, ddlerp_tma.cu).
#pragma once
#include <cuda_bf16.h>
#include <stddef.h>
#include <stdint.h>

namespace wkv6 {

struct alignas(16) bf16x8 { __nv_bfloat162 v[4]; };
// ONE 128-bit access each way, global or shared (copying the struct itself is compiled to four 32-bit accesses:
// __nv_bfloat162 has its own copy operations)
__device__ __forceinline__ bf16x8 ld8(const void *p) {
    const uint4 u = *reinterpret_cast<const uint4 *>(p);
    bf16x8 r;
    r.v[0] = *reinterpret_cast<const __nv_bfloat162 *>(&u.x);
    r.v[1] = *reinterpret_cast<const __nv_bfloat162 *>(&u.y);
    r.v[2] = *reinterpret_cast<const __nv_bfloat162 *>(&u.z);
    r.v[3] = *reinterpret_cast<const __nv_bfloat162 *>(&u.w);
    return r;
}
__device__ __forceinline__ void st8(void *p, const bf16x8 &x) {
    *reinterpret_cast<uint4 *>(p) = make_uint4(*reinterpret_cast<const uint32_t *>(&x.v[0]), *reinterpret_cast<const uint32_t *>(&x.v[1]),
                                                *reinterpret_cast<const uint32_t *>(&x.v[2]), *reinterpret_cast<const uint32_t *>(&x.v[3]));
}
__device__ __forceinline__ void unpack8(const bf16x8 &x, float *f) {
#pragma unroll
    for (int i = 0; i < 4; i++) { float2 t = __bfloat1622float2(x.v[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}
__device__ __forceinline__ bf16x8 pack8(const float *f) {
    bf16x8 x;
#pragma unroll
    for (int i = 0; i < 4; i++) x.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    return x;
}
// round-trip through bf16: what a bf16 eager op in the reference does to its fp32 result
__device__ __forceinline__ float rb(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// blocks of a grid-stride loop over `items`: enough to oversubscribe the 148 SMs, capped at 16 blocks per SM
inline int grid_for(size_t items, int block) {
    size_t g = (items + block - 1) / block;
    const size_t cap = 148 * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace wkv6
