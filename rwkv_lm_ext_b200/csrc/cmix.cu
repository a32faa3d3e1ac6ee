// Channel-mix elementwise pieces (RWKV_CMix_x060.forward, src/model.py:635-644; infctx :804-812) around
// its two cuBLAS GEMMs:
//     xk, xr = x + (shift(x) - x) * time_maa_{k,r}          one pass over x, two outputs
//     k      = relu(key(xk)) ** 2                            one pass over [B,T,dim_ffn]
//     out    = sigmoid(receptance(xr)) * value(k)            one pass
// All HBM-bound; 128-bit accesses; arithmetic in packed bf16 with the non-contracting intrinsics, i.e. with
// exactly the op-by-op rounding of the eager bf16 chain (results are bit-identical to it).  The gradient of
// the two-output shift-lerp is the TMA-fed kernel of ddlerp_tma.cu (nout = 2).
#include "bf16x8.cuh"
#include "common.cuh"

namespace wkv6 {
namespace {

typedef __nv_bfloat16 bf16;
typedef __nv_bfloat162 bf162;
// out_n = x + bf16(bf16(prev - x) * maa_n),  n = 0..NOUT-1
template <int NOUT>
__global__ void __launch_bounds__(256) shift_lerp_n_kernel(int B, int T, int C, const bf16 *__restrict__ x,
                                                           const bf16 *__restrict__ shift, const bf16 *__restrict__ maa,
                                                           bf16 *__restrict__ out) {
    const size_t nvec = (size_t)B * T * C / 8, plane = (size_t)B * T * C;
    const int cv = C / 8;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
        const size_t row = i / cv;
        const int c = (int)(i % cv) * 8, t = (int)(row % T), b = (int)(row / T);
        const bf16x8 xv = ld8(x + i * 8);
        bf16x8 pv;
        if (t > 0) pv = ld8(x + i * 8 - C);
        else if (shift) pv = ld8(shift + (size_t)b * C + c);
        else {
#pragma unroll
            for (int e = 0; e < 4; e++) pv.v[e] = __floats2bfloat162_rn(0.f, 0.f);
        }
        bf16x8 xx;
#pragma unroll
        for (int e = 0; e < 4; e++) xx.v[e] = __hsub2_rn(pv.v[e], xv.v[e]);
#pragma unroll
        for (int n = 0; n < NOUT; n++) {
            const bf16x8 a = ld8(maa + (size_t)n * C + c);
            bf16x8 o;
#pragma unroll
            for (int e = 0; e < 4; e++) o.v[e] = __hadd2_rn(xv.v[e], __hmul2_rn(xx.v[e], a.v[e]));
            st8(out + n * plane + i * 8, o);
        }
    }
}

// y = relu(x)^2   (torch.relu(k) ** 2)
__global__ void __launch_bounds__(256) relu_sq_kernel(size_t nvec, const bf16 *__restrict__ x, bf16 *__restrict__ y) {
    const bf162 zero = __floats2bfloat162_rn(0.f, 0.f);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
        const bf16x8 v = ld8(x + i * 8);
        bf16x8 o;
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const bf162 r = __hmax2(v.v[e], zero);
            o.v[e] = __hmul2_rn(r, r);
        }
        st8(y + i * 8, o);
    }
}
// gx = gy * 2 * relu(x)
__global__ void __launch_bounds__(256) relu_sq_bwd_kernel(size_t nvec, const bf16 *__restrict__ x, const bf16 *__restrict__ gy,
                                                          bf16 *__restrict__ gx) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
        const bf16x8 v = ld8(x + i * 8), g = ld8(gy + i * 8);
        bf16x8 o;
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const float2 xf = __bfloat1622float2(v.v[e]), gf = __bfloat1622float2(g.v[e]);
            o.v[e] = __floats2bfloat162_rn(2.f * fmaxf(xf.x, 0.f) * gf.x, 2.f * fmaxf(xf.y, 0.f) * gf.y);
        }
        st8(gx + i * 8, o);
    }
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }

// out = bf16(sigmoid(r)) * kv
__global__ void __launch_bounds__(256) sigmoid_mul_kernel(size_t nvec, const bf16 *__restrict__ r, const bf16 *__restrict__ kv,
                                                          bf16 *__restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
        const bf16x8 rv = ld8(r + i * 8), kk = ld8(kv + i * 8);
        bf16x8 o;
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const float2 rf = __bfloat1622float2(rv.v[e]);
            o.v[e] = __hmul2_rn(__floats2bfloat162_rn(sigmoidf_(rf.x), sigmoidf_(rf.y)), kk.v[e]);
        }
        st8(out + i * 8, o);
    }
}
// gr = gout * kv * s (1 - s),  gkv = gout * s
__global__ void __launch_bounds__(256) sigmoid_mul_bwd_kernel(size_t nvec, const bf16 *__restrict__ r, const bf16 *__restrict__ kv,
                                                              const bf16 *__restrict__ gout, bf16 *__restrict__ gr,
                                                              bf16 *__restrict__ gkv) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
        const bf16x8 rv = ld8(r + i * 8), kk = ld8(kv + i * 8), go = ld8(gout + i * 8);
        bf16x8 o1, o2;
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const float2 rf = __bfloat1622float2(rv.v[e]), kf = __bfloat1622float2(kk.v[e]), gf = __bfloat1622float2(go.v[e]);
            const float s0 = sigmoidf_(rf.x), s1 = sigmoidf_(rf.y);
            o1.v[e] = __floats2bfloat162_rn(gf.x * kf.x * s0 * (1.f - s0), gf.y * kf.y * s1 * (1.f - s1));
            o2.v[e] = __floats2bfloat162_rn(gf.x * s0, gf.y * s1);
        }
        st8(gr + i * 8, o1);
        st8(gkv + i * 8, o2);
    }
}

}  // namespace
}  // namespace wkv6

using namespace wkv6;

extern "C" {

int cmix_shift_lerp2_bf16(int B, int T, int C, const void *x, const void *shift_state, const void *maa_kr, void *out,
                          void *stream) {
    if (B < 0 || T < 0 || C <= 0 || (C & 7)) { set_error("cmix_shift_lerp2_bf16: need C %% 8 == 0"); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    if (!x || !maa_kr || !out) { set_error("cmix_shift_lerp2_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("cmix_shift_lerp2_bf16", {{"x", x}, {"shift_state", shift_state}, {"maa_kr", maa_kr}, {"out", out}})) return WKV6_EINVAL;
    shift_lerp_n_kernel<2><<<grid_for((size_t)B * T * C / 8, 256), 256, 0, (cudaStream_t)stream>>>(
        B, T, C, (const bf16 *)x, (const bf16 *)shift_state, (const bf16 *)maa_kr, (bf16 *)out);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int relu_sq_bf16(size_t n, const void *x, void *y, void *stream) {
    if (n == 0) return WKV6_OK;
    if (!x || !y || (n & 7)) { set_error("relu_sq_bf16: need n %% 8 == 0 and non-null pointers"); return WKV6_EINVAL; }
    if (!check_aligned16("relu_sq_bf16", {{"x", x}, {"y", y}})) return WKV6_EINVAL;
    relu_sq_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(n / 8, (const bf16 *)x, (bf16 *)y);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int relu_sq_backward_bf16(size_t n, const void *x, const void *gy, void *gx, void *stream) {
    if (n == 0) return WKV6_OK;
    if (!x || !gy || !gx || (n & 7)) { set_error("relu_sq_backward_bf16: need n %% 8 == 0 and non-null pointers"); return WKV6_EINVAL; }
    if (!check_aligned16("relu_sq_backward_bf16", {{"x", x}, {"gy", gy}, {"gx", gx}})) return WKV6_EINVAL;
    relu_sq_bwd_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(n / 8, (const bf16 *)x, (const bf16 *)gy, (bf16 *)gx);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int sigmoid_mul_bf16(size_t n, const void *r, const void *kv, void *out, void *stream) {
    if (n == 0) return WKV6_OK;
    if (!r || !kv || !out || (n & 7)) { set_error("sigmoid_mul_bf16: need n %% 8 == 0 and non-null pointers"); return WKV6_EINVAL; }
    if (!check_aligned16("sigmoid_mul_bf16", {{"r", r}, {"kv", kv}, {"out", out}})) return WKV6_EINVAL;
    sigmoid_mul_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(n / 8, (const bf16 *)r, (const bf16 *)kv, (bf16 *)out);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int sigmoid_mul_backward_bf16(size_t n, const void *r, const void *kv, const void *gout, void *gr, void *gkv, void *stream) {
    if (n == 0) return WKV6_OK;
    if (!r || !kv || !gout || !gr || !gkv || (n & 7)) { set_error("sigmoid_mul_backward_bf16: need n %% 8 == 0 and non-null pointers"); return WKV6_EINVAL; }
    if (!check_aligned16("sigmoid_mul_backward_bf16", {{"r", r}, {"kv", kv}, {"gout", gout}, {"gr", gr}, {"gkv", gkv}})) return WKV6_EINVAL;
    sigmoid_mul_bwd_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>(n / 8, (const bf16 *)r, (const bf16 *)kv,
                                                                                  (const bf16 *)gout, (bf16 *)gr, (bf16 *)gkv);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

}  // extern "C"
