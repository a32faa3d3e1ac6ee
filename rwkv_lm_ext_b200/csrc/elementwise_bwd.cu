// Gradients of the memory-bound neighbours (token-shift ddlerp, GroupNorm*gate, pooling, the two
// gathers), so the fused forwards of elementwise.cu can sit inside a training graph in place of the
// reference's eager chains (src/model.py:434-468, src/model_ext.py:1708-1738).
//
// Layout of the two "column reduce" kernels: grid (ceil(C/256), S), block 256 = 32 column lanes
// (8 channels each, so a warp reads 512 contiguous bytes of a token row) x 8 token lanes (one warp
// each).  A block owns rows [split*R, split*R+R) of the flattened [B*T, C] tensor, a warp a contiguous
// run of them walked backwards (the token-shift gradient needs the value of row t+1 when it is at
// row t).  Parameter gradients (sums over all rows) are accumulated per thread, reduced over the 8
// token lanes in shared memory and written as fp32 partials [S][n][C]; a second, tiny kernel sums
// the S partials in a fixed order -> deterministic, no atomics.
#include "common.cuh"
#include <algorithm>

namespace wkv6 {
namespace {

typedef __nv_bfloat16 bf16;
struct alignas(16) bf16x8 { __nv_bfloat162 v[4]; };
// ONE 128-bit access each way (copying the struct itself is compiled to four 32-bit accesses: __nv_bfloat162 has its own
// copy operations)
__device__ __forceinline__ bf16x8 ld8(const bf16 *p) {
    const uint4 u = *reinterpret_cast<const uint4 *>(p);
    bf16x8 r;
    r.v[0] = *reinterpret_cast<const __nv_bfloat162 *>(&u.x);
    r.v[1] = *reinterpret_cast<const __nv_bfloat162 *>(&u.y);
    r.v[2] = *reinterpret_cast<const __nv_bfloat162 *>(&u.z);
    r.v[3] = *reinterpret_cast<const __nv_bfloat162 *>(&u.w);
    return r;
}
__device__ __forceinline__ void st8(bf16 *p, const bf16x8 &x) {
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
__device__ __forceinline__ float rb(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

constexpr int TL = 8;  // token lanes (warps) per block
// register-fed ddlerp gradient (the "simt" route of the one- and five-output forms; ddlerp_tma.cu otherwise): 8 channels per thread,
// one 256-thread block per SM.  Measured alternatives: 4 channels per thread 1.07 ms, two blocks per SM 0.93 ms,
// a block spanning 2048 channels 0.73 ms, against 0.59 ms for this layout (1B6 shape).
constexpr int DD_V = 8;

struct Split { int rows_per_split, rows_per_lane; };
struct Ptr5 { const bf16 *p[5]; };   // the five incoming gradients (xw,xk,xv,xr,xg) are separate tensors

// ------------------------------------------------------------------------------------------------
// out_n = x + xx * coef_n,  xx = bf16(prev - x),  coef_n = bf16(maa_n + m_n)   (HAS_M)  or  maa_n
//   gm_n   = gout_n * xx                                   (HAS_M only)
//   gmaa_n = sum_rows gout_n * xx
//   gxx    = sum_n gout_n * coef_n
//   gx[t]  = sum_n gout_n[t] - gxx[t] + gxx[t+1]           (gxx[T] = 0)
//   gshift[b] = gxx[b, 0]                                  (when a shift state was given)
// ------------------------------------------------------------------------------------------------
// V channels per thread
template <int V> struct VecIO;
template <> struct VecIO<8> {
    static __device__ __forceinline__ void ld(const bf16 *p, float *f) { unpack8(ld8(p), f); }
    static __device__ __forceinline__ void st(bf16 *p, const float *f) { st8(p, pack8(f)); }
};

template <int NOUT, bool HAS_M, int V>
__global__ void __launch_bounds__(256) ddlerp_bwd_kernel(int B, int T, int C, Split sp, const bf16 *__restrict__ x,
                                                         const bf16 *__restrict__ shift, const bf16 *__restrict__ maa,
                                                         const bf16 *__restrict__ m, const Ptr5 gout,
                                                         bf16 *__restrict__ gx, bf16 *__restrict__ gm,
                                                         bf16 *__restrict__ gshift, float *__restrict__ partial) {
    typedef VecIO<V> IO;
    constexpr int COLS = 32 * V;                       // channels per block
    const int lane = threadIdx.x & 31, tl = threadIdx.x >> 5;
    const int c = (blockIdx.x * 32 + lane) * V;
    const bool live = c < C;
    const long long BT = (long long)B * T;
    const size_t plane = (size_t)BT * C;
    const long long s0 = (long long)blockIdx.y * sp.rows_per_split;
    long long r0 = s0 + (long long)tl * sp.rows_per_lane;
    long long r1 = r0 + sp.rows_per_lane;
    const long long send = s0 + sp.rows_per_split < BT ? s0 + sp.rows_per_split : BT;
    if (r1 > send) r1 = send;

    float acc[NOUT][V];
#pragma unroll
    for (int n = 0; n < NOUT; n++)
#pragma unroll
        for (int e = 0; e < V; e++) acc[n][e] = 0.f;

    if (live && r0 < r1) {
        float af[NOUT][V];
#pragma unroll
        for (int n = 0; n < NOUT; n++) IO::ld(maa + (size_t)n * C + c, af[n]);

        // gxx of one row (needed for the row after this run, if it belongs to the same sequence)
        auto row_gxx = [&](long long row, const float *xx, float *gxx, float *gsum, bool write) {
#pragma unroll
            for (int e = 0; e < V; e++) { gxx[e] = 0.f; gsum[e] = 0.f; }
#pragma unroll
            for (int n = 0; n < NOUT; n++) {
                float gf[V], cf[V];
                IO::ld(gout.p[n] + (size_t)row * C + c, gf);
                if (HAS_M) {
                    IO::ld(m + n * plane + (size_t)row * C + c, cf);
#pragma unroll
                    for (int e = 0; e < V; e++) cf[e] = rb(af[n][e] + cf[e]);
                } else {
#pragma unroll
                    for (int e = 0; e < V; e++) cf[e] = af[n][e];
                }
                float gmv[V];
#pragma unroll
                for (int e = 0; e < V; e++) {
                    gxx[e] = fmaf(gf[e], cf[e], gxx[e]);
                    gsum[e] += gf[e];
                    gmv[e] = gf[e] * xx[e];
                    if (write) acc[n][e] += gmv[e];
                }
                if (HAS_M && write) IO::st(gm + n * plane + (size_t)row * C + c, gmv);
            }
        };

        float carry[V], xf[V], pf[V], xx[V], gxx[V], gsum[V];
        // carry = gxx[r1] when row r1 continues the sequence of row r1-1
        if (r1 < BT && (r1 % T) != 0) {
#pragma unroll
            for (int e = 0; e < V; e++) xf[e] = 0.f;
            row_gxx(r1, xf, carry, gsum, false);
        } else {
#pragma unroll
            for (int e = 0; e < V; e++) carry[e] = 0.f;
        }
        IO::ld(x + (size_t)(r1 - 1) * C + c, xf);
        for (long long row = r1 - 1; row >= r0; row--) {
            const int t = (int)(row % T);
            if (t > 0) IO::ld(x + (size_t)(row - 1) * C + c, pf);
            else if (shift) IO::ld(shift + (size_t)(row / T) * C + c, pf);
            else {
#pragma unroll
                for (int e = 0; e < V; e++) pf[e] = 0.f;
            }
#pragma unroll
            for (int e = 0; e < V; e++) xx[e] = rb(pf[e] - xf[e]);
            row_gxx(row, xx, gxx, gsum, true);
            float o[V];
#pragma unroll
            for (int e = 0; e < V; e++) o[e] = gsum[e] - gxx[e] + carry[e];
            IO::st(gx + (size_t)row * C + c, o);
            if (t == 0) {
                if (gshift) IO::st(gshift + (size_t)(row / T) * C + c, gxx);
#pragma unroll
                for (int e = 0; e < V; e++) carry[e] = 0.f;   // previous row ends another sequence
            } else {
#pragma unroll
                for (int e = 0; e < V; e++) carry[e] = gxx[e];
            }
#pragma unroll
            for (int e = 0; e < V; e++) xf[e] = pf[e];         // x[row-1] (only used when t > 0)
            if (t == 0 && row > r0) IO::ld(x + (size_t)(row - 1) * C + c, xf);
        }
    }

    // reduce the parameter gradient over the 8 token lanes
    __shared__ float red[TL][NOUT][COLS + V];
#pragma unroll
    for (int n = 0; n < NOUT; n++)
#pragma unroll
        for (int e = 0; e < V; e++) red[tl][n][lane * V + e] = acc[n][e];
    __syncthreads();
    for (int i = threadIdx.x; i < NOUT * COLS; i += 256) {
        const int n = i / COLS, cc = i % COLS;
        float s = 0.f;
#pragma unroll
        for (int l = 0; l < TL; l++) s += red[l][n][cc];
        const int col = blockIdx.x * COLS + cc;
        if (col < C) partial[((size_t)blockIdx.y * NOUT + n) * C + col] = s;
    }
}

// out[i] = sum_s partial[s][i]
__global__ void sum_partials_kernel(int S, int n, size_t stride, const float *__restrict__ partial,
                                    float *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = 0.f;
    for (int k = 0; k < S; k++) s += partial[(size_t)k * stride + i];
    out[i] = s;
}

// ------------------------------------------------------------------------------------------------
// out = z * g,  z = bf16(n * w + b),  n = (y - mean) * rstd  over each 64-channel group
//   gg = gout * z ;  gz = gout * g ;  glw = sum_rows gz * n ;  glb = sum_rows gz
//   gn = gz * w ;  gy = rstd * (gn - mean(gn) - n * mean(gn * n))
// 8 consecutive lanes = one group.
// ------------------------------------------------------------------------------------------------
template <bool SILU>
__global__ void __launch_bounds__(256) gn_gate_bwd_kernel(long long BT, int C, float eps, Split sp,
                                                          const bf16 *__restrict__ y, const bf16 *__restrict__ g,
                                                          const bf16 *__restrict__ lw, const bf16 *__restrict__ lb,
                                                          const bf16 *__restrict__ gout, bf16 *__restrict__ gy,
                                                          bf16 *__restrict__ gg, float *__restrict__ partial) {
    const int lane = threadIdx.x & 31, tl = threadIdx.x >> 5;
    const int c_raw = (blockIdx.x * 32 + lane) * 8;
    const bool live = c_raw < C;
    const int c = live ? c_raw : 0;
    const long long s0 = (long long)blockIdx.y * sp.rows_per_split;
    const long long r0 = s0 + (long long)tl * sp.rows_per_lane;
    long long r1 = r0 + sp.rows_per_lane;
    const long long send = s0 + sp.rows_per_split < BT ? s0 + sp.rows_per_split : BT;
    if (r1 > send) r1 = send;

    float aw[8], ab[8], wf[8], bfv[8];
#pragma unroll
    for (int e = 0; e < 8; e++) aw[e] = ab[e] = 0.f;
    unpack8(ld8(lw + c), wf);
    unpack8(ld8(lb + c), bfv);

    // one row ahead: the three 16-byte loads of row + 1 are in flight while row is reduced (a row is 12 shuffles deep)
    bf16x8 ny, ng, ngo;
    if (r0 < r1) {
        const size_t off0 = (size_t)r0 * C + c;
        ny = ld8(y + off0); ng = ld8(g + off0); ngo = ld8(gout + off0);
    }
    for (long long row = r0; row < r1; row++) {          // warp-uniform bounds: shuffles are safe
        const size_t off = (size_t)row * C + c;
        float f[8], gf[8], go[8];
        unpack8(ny, f);
        unpack8(ng, gf);
        unpack8(ngo, go);
        if (row + 1 < r1) {
            const size_t offn = off + C;
            ny = ld8(y + offn); ng = ld8(g + offn); ngo = ld8(gout + offn);
        }
        float s = 0.f;
#pragma unroll
        for (int e = 0; e < 8; e++) s += f[e];
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        const float mean = s * (1.0f / 64.0f);
        float q = 0.f;
#pragma unroll
        for (int e = 0; e < 8; e++) { f[e] -= mean; q += f[e] * f[e]; }
        q += __shfl_xor_sync(0xffffffffu, q, 1);
        q += __shfl_xor_sync(0xffffffffu, q, 2);
        q += __shfl_xor_sync(0xffffffffu, q, 4);
        const float rstd = rsqrtf(q * (1.0f / 64.0f) + eps);
        float gn[8], ggv[8], m1 = 0.f, m2 = 0.f;
#pragma unroll
        for (int e = 0; e < 8; e++) {
            f[e] *= rstd;                                  // n
            const float z = rb(fmaf(f[e], wf[e], bfv[e]));
            float gate = gf[e], dgate = 1.f;
            if (SILU) {                                    // gate = silu(graw), as bf16 like the eager op
                const float sg = 1.f / (1.f + __expf(-gf[e]));
                gate = rb(gf[e] * sg);
                dgate = sg * (1.f + gf[e] * (1.f - sg));
            }
            ggv[e] = go[e] * z * dgate;
            const float gz = go[e] * gate;
            aw[e] = fmaf(gz, f[e], aw[e]);
            ab[e] += gz;
            gn[e] = gz * wf[e];
            m1 += gn[e];
            m2 = fmaf(gn[e], f[e], m2);
        }
        m1 += __shfl_xor_sync(0xffffffffu, m1, 1);
        m2 += __shfl_xor_sync(0xffffffffu, m2, 1);
        m1 += __shfl_xor_sync(0xffffffffu, m1, 2);
        m2 += __shfl_xor_sync(0xffffffffu, m2, 2);
        m1 += __shfl_xor_sync(0xffffffffu, m1, 4);
        m2 += __shfl_xor_sync(0xffffffffu, m2, 4);
        m1 *= (1.0f / 64.0f);
        m2 *= (1.0f / 64.0f);
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; e++) o[e] = rstd * (gn[e] - m1 - f[e] * m2);
        if (live) {
            st8(gy + off, pack8(o));
            st8(gg + off, pack8(ggv));
        }
    }

    __shared__ float red[TL][2][256 + 8];
#pragma unroll
    for (int e = 0; e < 8; e++) {
        red[tl][0][lane * 8 + e] = live ? aw[e] : 0.f;
        red[tl][1][lane * 8 + e] = live ? ab[e] : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * 256; i += 256) {
        const int n = i >> 8, cc = i & 255;
        float s = 0.f;
#pragma unroll
        for (int l = 0; l < TL; l++) s += red[l][n][cc];
        const int col = blockIdx.x * 256 + cc;
        if (col < C) partial[((size_t)blockIdx.y * 2 + n) * C + col] = s;
    }
}

// ------------------------------------------------------------------------------------------------
// pooling backward: gx[b,t,:] = gout[b,:] * wgt(t) / L  inside the pooled range, 0 outside.
// ------------------------------------------------------------------------------------------------
// Write-only: gx[b,t,:] = gout[b,:] * weight(t).  One block per (b, 16 token rows): a thread keeps its 8 channels of gout[b] in registers
// and walks 16 token rows, so there is no index arithmetic per store and the weight is one value per row.
constexpr int POOL_ROWS = 16;
__global__ void __launch_bounds__(256) pooling_bwd_kernel(int kind, int B, int T, int D,
                                                          const int64_t *__restrict__ alen, int add_one,
                                                          const float *__restrict__ gout, bf16 *__restrict__ gx) {
    const int nt = (T + POOL_ROWS - 1) / POOL_ROWS;
    const int b = blockIdx.x / nt, t0 = (blockIdx.x % nt) * POOL_ROWS, t1 = min(T, t0 + POOL_ROWS);
    const long long L64 = alen[b] + add_one;
    const float Lf = (float)L64, inv = 1.0f / Lf;
    const long long tend = (kind == 0) ? L64 + 1 : L64;
    for (int d = threadIdx.x * 8; d < D; d += blockDim.x * 8) {
        const float4 a = *reinterpret_cast<const float4 *>(gout + (size_t)b * D + d);
        const float4 c = *reinterpret_cast<const float4 *>(gout + (size_t)b * D + d + 4);
        bf16 *dst = gx + ((size_t)b * T + t0) * D + d;
        for (int t = t0; t < t1; t++, dst += D) {
            const float wgt = t < tend ? ((kind == 0) ? (float)(t + 1) / Lf : 1.0f) / Lf : 0.f;
            float o[8] = {a.x * wgt, a.y * wgt, a.z * wgt, a.w * wgt, c.x * wgt, c.y * wgt, c.z * wgt, c.w * wgt};
            st8(dst, pack8(o));
        }
    }
    (void)inv; (void)B;
}

// gx[b,t,:] = (t == pos[b]) ? gout[b,:] : 0      (gradient of gather_rows)
__global__ void __launch_bounds__(256) scatter_rows_kernel(int B, int T, int D, const bf16 *__restrict__ gout,
                                                           const int64_t *__restrict__ pos, bf16 *__restrict__ gx) {
    const int dv = D / 8;
    const size_t nvec = (size_t)B * T * dv;
    bf16x8 zero;
#pragma unroll
    for (int i = 0; i < 4; i++) zero.v[i] = __floats2bfloat162_rn(0.f, 0.f);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
        const size_t row = i / dv;
        const int d = (int)(i % dv) * 8, t = (int)(row % T), b = (int)(row / T);
        int64_t p = pos[b];
        p = p < 0 ? p + T : p;
        st8(gx + i * 8, t == p ? ld8(gout + (size_t)b * D + d) : zero);
    }
}

// gx[b,rev[b,t],:] = gout[b,t,:]   (gradient of gather_tokens when rev is a per-row permutation)
__global__ void scatter_tokens_kernel(int BT, int T, int D, const bf16 *__restrict__ gout,
                                      const int64_t *__restrict__ rev, bf16 *__restrict__ gx) {
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < BT; row += warps) {
        const int b = row / T;
        bf16 *dst = gx + ((size_t)b * T + (size_t)rev[row]) * D;
        const bf16 *src = gout + (size_t)row * D;
        for (int d = lane * 8; d < D; d += 256) st8(dst + d, ld8(src + d));
    }
}

int grid_for(size_t items, int block) {
    size_t g = (items + block - 1) / block;
    const size_t cap = 148 * 16;
    return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

// number of row splits: enough blocks to fill 148 SMs a few times over, at least 8 rows per lane
int splits_for(long long BT, int C, int cols = 256, int lanes = TL) {
    const int colblocks = (C + cols - 1) / cols;
    long long S = (148 * 6 + colblocks - 1) / colblocks;
    const long long maxS = (BT + lanes * 8 - 1) / (lanes * 8);
    if (S > maxS) S = maxS;
    if (S < 1) S = 1;
    return (int)S;
}
Split split_of(long long BT, int S, int lanes = TL) {
    Split sp;
    sp.rows_per_split = (int)((BT + S - 1) / S);
    sp.rows_per_lane = (sp.rows_per_split + lanes - 1) / lanes;
    return sp;
}
constexpr int DD_COLS = 32 * DD_V, DD_LANES = TL;

}  // namespace
}  // namespace wkv6

using namespace wkv6;

extern "C" {

size_t elementwise_backward_workspace_bytes(int B, int T, int C, int nparam) {
    if (B <= 0 || T <= 0 || C <= 0 || nparam <= 0) return 0;
    const long long BT = (long long)B * T;
    // nparam: 5 ddlerp, 1 shift-lerp, 2 GroupNorm*gate, 3 = the two-output channel-mix shift-lerp (2 rows)
    size_t slots = nparam == 2 ? splits_for(BT, C) : splits_for(BT, C, DD_COLS, DD_LANES);
    if (nparam != 2) slots = std::max(slots, ddlerp_tma_partial_slots(nparam == 3 ? 2 : nparam, B, T, C));
    return slots * (nparam == 3 ? 2 : nparam) * C * sizeof(float);
}

int tmix_ddlerp_mix_backward_bf16(int B, int T, int C, const void *x, const void *shift_state, const void *maa,
                                  const void *m, const void *gxw, const void *gxk, const void *gxv,
                                  const void *gxr, const void *gxg, void *gx, void *gm, float *gmaa,
                                  void *gshift, void *ws, size_t ws_bytes, void *stream) {
    if (B < 0 || T < 0 || C <= 0 || (C & 7)) { set_error("tmix_ddlerp_mix_backward_bf16: need C %% 8 == 0"); return WKV6_EINVAL; }
    const long long BT = (long long)B * T;
    if (BT == 0) return WKV6_OK;
    if (!x || !maa || !m || !gxw || !gxk || !gxv || !gxr || !gxg || !gx || !gm || !ws) {
        set_error("tmix_ddlerp_mix_backward_bf16: null pointer");
        return WKV6_EINVAL;
    }
    Ptr5 gout;
    gout.p[0] = (const bf16 *)gxw; gout.p[1] = (const bf16 *)gxk; gout.p[2] = (const bf16 *)gxv;
    gout.p[3] = (const bf16 *)gxr; gout.p[4] = (const bf16 *)gxg;
    if (ws_bytes < elementwise_backward_workspace_bytes(B, T, C, 5)) { set_error("tmix_ddlerp_mix_backward_bf16: workspace too small"); return WKV6_EINVAL; }
    if (!check_aligned16("tmix_ddlerp_mix_backward_bf16", {{"x", x}, {"shift_state", shift_state}, {"maa", maa}, {"m", m}, {"gxw", gxw},
                                                            {"gxk", gxk}, {"gxv", gxv}, {"gxr", gxr}, {"gxg", gxg}, {"gx", gx}, {"gm", gm},
                                                            {"gshift", shift_state ? gshift : nullptr}}))
        return WKV6_EINVAL;
    if (wkv6b200_get_impl() != WKV6_IMPL_SIMT) {
        const void *gs[5] = {gxw, gxk, gxv, gxr, gxg};
        int slots = 0;
        const int rc = ddlerp_backward_tma(5, B, T, C, x, shift_state, maa, m, gs, gx, gm, shift_state ? gshift : nullptr,
                                           (float *)ws, &slots, (cudaStream_t)stream);
        if (rc <= 0) {
            if (rc < 0) return rc;
            if (gmaa) sum_partials_kernel<<<(5 * C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(slots, 5 * C, (size_t)5 * C, (const float *)ws, gmaa);
            if (gmaa) count_launch();
            WKV6_CUDA_CHECK(cudaGetLastError());
            return WKV6_OK;
        }
    }
    const int S = splits_for(BT, C, DD_COLS, DD_LANES);
    dim3 grid((C + DD_COLS - 1) / DD_COLS, S);
    ddlerp_bwd_kernel<5, true, DD_V><<<grid, 256, 0, (cudaStream_t)stream>>>(
        B, T, C, split_of(BT, S, DD_LANES), (const bf16 *)x, (const bf16 *)shift_state, (const bf16 *)maa, (const bf16 *)m,
        gout, (bf16 *)gx, (bf16 *)gm, shift_state ? (bf16 *)gshift : nullptr, (float *)ws);
    if (gmaa) sum_partials_kernel<<<(5 * C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(S, 5 * C, (size_t)5 * C, (const float *)ws, gmaa);
    count_launch(gmaa ? 2 : 1);
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int tmix_shift_lerp_backward_bf16(int B, int T, int C, const void *x, const void *shift_state, const void *maa_x,
                                  const void *gout, void *gx, float *gmaa_x, void *gshift, void *ws,
                                  size_t ws_bytes, void *stream) {
    if (B < 0 || T < 0 || C <= 0 || (C & 7)) { set_error("tmix_shift_lerp_backward_bf16: need C %% 8 == 0"); return WKV6_EINVAL; }
    const long long BT = (long long)B * T;
    if (BT == 0) return WKV6_OK;
    if (!x || !maa_x || !gout || !gx || !ws) { set_error("tmix_shift_lerp_backward_bf16: null pointer"); return WKV6_EINVAL; }
    Ptr5 g1;
    for (int i = 0; i < 5; i++) g1.p[i] = (const bf16 *)gout;
    if (ws_bytes < elementwise_backward_workspace_bytes(B, T, C, 1)) { set_error("tmix_shift_lerp_backward_bf16: workspace too small"); return WKV6_EINVAL; }
    if (!check_aligned16("tmix_shift_lerp_backward_bf16", {{"x", x}, {"shift_state", shift_state}, {"maa_x", maa_x}, {"gout", gout}, {"gx", gx},
                                                            {"gshift", shift_state ? gshift : nullptr}}))
        return WKV6_EINVAL;
    if (wkv6b200_get_impl() != WKV6_IMPL_SIMT) {
        const void *gs[1] = {gout};
        int slots = 0;
        const int rc = ddlerp_backward_tma(1, B, T, C, x, shift_state, maa_x, nullptr, gs, gx, nullptr,
                                           shift_state ? gshift : nullptr, (float *)ws, &slots, (cudaStream_t)stream);
        if (rc <= 0) {
            if (rc < 0) return rc;
            if (gmaa_x) sum_partials_kernel<<<(C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(slots, C, (size_t)C, (const float *)ws, gmaa_x);
            if (gmaa_x) count_launch();
            WKV6_CUDA_CHECK(cudaGetLastError());
            return WKV6_OK;
        }
    }
    const int S = splits_for(BT, C, DD_COLS, DD_LANES);
    dim3 grid((C + DD_COLS - 1) / DD_COLS, S);
    ddlerp_bwd_kernel<1, false, DD_V><<<grid, 256, 0, (cudaStream_t)stream>>>(
        B, T, C, split_of(BT, S, DD_LANES), (const bf16 *)x, (const bf16 *)shift_state, (const bf16 *)maa_x, nullptr,
        g1, (bf16 *)gx, nullptr, shift_state ? (bf16 *)gshift : nullptr, (float *)ws);
    if (gmaa_x) sum_partials_kernel<<<(C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(S, C, (size_t)C, (const float *)ws, gmaa_x);
    count_launch(gmaa_x ? 2 : 1);
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int groupnorm_gate_backward_bf16(int BT, int C, int H, float eps, int gate_act, const void *y, const void *g,
                                 const void *ln_w, const void *ln_b, const void *gout, void *gy, void *gg,
                                 float *gln_w, float *gln_b, void *ws, size_t ws_bytes, void *stream) {
    if (BT < 0 || H <= 0 || C != H * 64) { set_error("groupnorm_gate_backward_bf16: need C == H*64"); return WKV6_EINVAL; }
    if (BT == 0) return WKV6_OK;
    if (!y || !g || !ln_w || !ln_b || !gout || !gy || !gg || (!gln_w != !gln_b) || !ws) {
        set_error("groupnorm_gate_backward_bf16: null pointer");
        return WKV6_EINVAL;
    }
    if (!check_aligned16("groupnorm_gate_backward_bf16", {{"y", y}, {"g", g}, {"ln_w", ln_w}, {"ln_b", ln_b}, {"gout", gout}, {"gy", gy}, {"gg", gg}}))
        return WKV6_EINVAL;
    const int S = splits_for(BT, C);
    if (ws_bytes < (size_t)S * 2 * C * sizeof(float)) {
        set_error("groupnorm_gate_backward_bf16: workspace too small");
        return WKV6_EINVAL;
    }
    dim3 grid((C + 255) / 256, S);
    float *partial = (float *)ws;
    if (gate_act)
        gn_gate_bwd_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(
            BT, C, eps, split_of(BT, S), (const bf16 *)y, (const bf16 *)g, (const bf16 *)ln_w, (const bf16 *)ln_b,
            (const bf16 *)gout, (bf16 *)gy, (bf16 *)gg, partial);
    else
        gn_gate_bwd_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(
            BT, C, eps, split_of(BT, S), (const bf16 *)y, (const bf16 *)g, (const bf16 *)ln_w, (const bf16 *)ln_b,
            (const bf16 *)gout, (bf16 *)gy, (bf16 *)gg, partial);
    if (gln_w) sum_partials_kernel<<<(C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(S, C, (size_t)2 * C, partial, gln_w);
    if (gln_b) sum_partials_kernel<<<(C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(S, C, (size_t)2 * C, partial + C, gln_b);
    count_launch(gln_w ? 3 : 1);
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int pooling_backward_bf16(int kind, int variant, int B, int T, int D, const int64_t *actual_len,
                          const float *gout_f32, void *gx, void *stream) {
    if (B < 0 || T <= 0 || D <= 0 || (D & 7) || (kind != 0 && kind != 2)) { set_error("pooling_backward_bf16: bad arguments (D %% 8 == 0, kind 0 or 2)"); return WKV6_EINVAL; }
    if (B == 0) return WKV6_OK;
    if (!actual_len || !gout_f32 || !gx) { set_error("pooling_backward_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("pooling_backward_bf16", {{"gout_f32", gout_f32}, {"gx", gx}})) return WKV6_EINVAL;
    pooling_bwd_kernel<<<(unsigned)((size_t)B * ((T + POOL_ROWS - 1) / POOL_ROWS)), 256, 0, (cudaStream_t)stream>>>(
        kind, B, T, D, actual_len, (kind == 0 && variant == 1) ? 1 : 0, gout_f32, (bf16 *)gx);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int scatter_rows_bf16(int B, int T, int D, const void *gout, const int64_t *pos, void *gx, void *stream) {
    if (B < 0 || T <= 0 || D <= 0 || (D & 7)) { set_error("scatter_rows_bf16: need D %% 8 == 0"); return WKV6_EINVAL; }
    if (B == 0) return WKV6_OK;
    if (!gout || !pos || !gx) { set_error("scatter_rows_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("scatter_rows_bf16", {{"gout", gout}, {"gx", gx}})) return WKV6_EINVAL;
    scatter_rows_kernel<<<grid_for((size_t)B * T * D / 8, 256), 256, 0, (cudaStream_t)stream>>>(
        B, T, D, (const bf16 *)gout, pos, (bf16 *)gx);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int scatter_tokens_bf16(int B, int T, int D, const void *gout, const int64_t *rev_idx, void *gx, void *stream) {
    if (B < 0 || T < 0 || D <= 0 || (D & 7)) { set_error("scatter_tokens_bf16: need D %% 8 == 0"); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    if (!gout || !rev_idx || !gx) { set_error("scatter_tokens_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("scatter_tokens_bf16", {{"gout", gout}, {"gx", gx}})) return WKV6_EINVAL;
    const int BT = B * T;
    scatter_tokens_kernel<<<grid_for((size_t)BT * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        BT, T, D, (const bf16 *)gout, rev_idx, (bf16 *)gx);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

// gradient of cmix_shift_lerp2_bf16: gx [B,T,C], gmaa_kr fp32 [2,C] from gxk, gxr
int cmix_shift_lerp2_backward_bf16(int B, int T, int C, const void *x, const void *shift_state, const void *maa_kr,
                                   const void *gxk, const void *gxr, void *gx, float *gmaa_kr, void *gshift, void *ws,
                                   size_t ws_bytes, void *stream) {
    if (B < 0 || T < 0 || C <= 0 || (C & 7)) { set_error("cmix_shift_lerp2_backward_bf16: need C %% 8 == 0"); return WKV6_EINVAL; }
    const long long BT = (long long)B * T;
    if (BT == 0) return WKV6_OK;
    if (!x || !maa_kr || !gxk || !gxr || !gx || !ws) { set_error("cmix_shift_lerp2_backward_bf16: null pointer"); return WKV6_EINVAL; }
    if (ws_bytes < elementwise_backward_workspace_bytes(B, T, C, 3)) { set_error("cmix_shift_lerp2_backward_bf16: workspace too small"); return WKV6_EINVAL; }
    if (!check_aligned16("cmix_shift_lerp2_backward_bf16", {{"x", x}, {"shift_state", shift_state}, {"gxk", gxk}, {"gxr", gxr}, {"gx", gx},
                                                             {"gshift", shift_state ? gshift : nullptr}}))
        return WKV6_EINVAL;
    const void *gs[2] = {gxk, gxr};
    int slots = 0;
    const int rc = ddlerp_backward_tma(2, B, T, C, x, shift_state, maa_kr, nullptr, gs, gx, nullptr, shift_state ? gshift : nullptr,
                                       (float *)ws, &slots, (cudaStream_t)stream);
    if (rc != WKV6_OK) return rc;      // (the TMA kernel declines only the five-output form)
    if (gmaa_kr) sum_partials_kernel<<<(2 * C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(slots, 2 * C, (size_t)2 * C, (const float *)ws, gmaa_kr);
    if (gmaa_kr) count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

}  // extern "C"
