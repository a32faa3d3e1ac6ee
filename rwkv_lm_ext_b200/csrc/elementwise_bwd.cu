// Gradients of the memory-bound neighbours (token-shift ddlerp, GroupNorm*gate, pooling, the two
// gathers), so the fused forwards of elementwise.cu can sit inside a training graph in place of the
// reference's eager chains (src/model.py:434-468, src/model_ext.py:1708-1738).  The token-shift
// gradients are the TMA-fed kernel of ddlerp_tma.cu; this file sums its partials.
//
// Layout of the GroupNorm*gate "column reduce" kernel: grid (ceil(C/256), S), block 256 = 32 column
// lanes (8 channels each, so a warp reads 512 contiguous bytes of a token row) x 8 token lanes (one
// warp each).  A block owns rows [split*R, split*R+R) of the flattened [B*T, C] tensor, a warp a
// contiguous run of them.  The parameter gradients (sums over all rows) are accumulated per thread,
// reduced over the 8 token lanes in shared memory and written as fp32 partials [S][2][C]; a second,
// tiny kernel sums the S partials in a fixed order -> deterministic, no atomics.
#include "bf16x8.cuh"
#include "common.cuh"

#include <climits>

namespace wkv6 {
namespace {

typedef __nv_bfloat16 bf16;

constexpr int TL = 8;  // token lanes (warps) per block

struct Split { int rows_per_split, rows_per_lane; };

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

// number of row splits: enough blocks to fill 148 SMs a few times over, at least 8 rows per lane
int splits_for(long long BT, int C) {
    const int colblocks = (C + 255) / 256;
    long long S = (148 * 6 + colblocks - 1) / colblocks;
    const long long maxS = (BT + TL * 8 - 1) / (TL * 8);
    if (S > maxS) S = maxS;
    if (S < 1) S = 1;
    return (int)S;
}
Split split_of(long long BT, int S) {
    Split sp;
    sp.rows_per_split = (int)((BT + S - 1) / S);
    sp.rows_per_lane = (sp.rows_per_split + TL - 1) / TL;
    return sp;
}

// the shift-lerp backward entries (nout = 5 with m, 1 and 2 without): the TMA-fed kernel, then the fixed-order sum of
// its partials when the parameter gradient is wanted.  The caller has checked the arguments.
int shift_lerp_backward(int nout, int B, int T, int C, const void *x, const void *shift_state, const void *maa, const void *m,
                        const void *const *gouts, void *gx, void *gm, float *gmaa, void *gshift, void *ws, void *stream) {
    int slots = 0;
    const int rc = ddlerp_backward_tma(nout, B, T, C, x, shift_state, maa, m, gouts, gx, gm, shift_state ? gshift : nullptr,
                                       (float *)ws, &slots, (cudaStream_t)stream);
    if (rc != WKV6_OK) return rc;
    if (gmaa) {
        sum_partials_kernel<<<(nout * C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(slots, nout * C, (size_t)nout * C,
                                                                                      (const float *)ws, gmaa);
        count_launch();
    }
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

}  // namespace
}  // namespace wkv6

using namespace wkv6;

extern "C" {

size_t elementwise_backward_workspace_bytes(int B, int T, int C, int nparam) {
    if (B <= 0 || T <= 0 || C <= 0 || nparam <= 0) return 0;
    // nparam: 5 ddlerp, 1 shift-lerp, 2 GroupNorm*gate, 3 = the two-output channel-mix shift-lerp (2 rows)
    if (nparam == 2) return (size_t)splits_for((long long)B * T, C) * 2 * C * sizeof(float);
    const int nout = nparam == 3 ? 2 : nparam;
    return ddlerp_tma_partial_slots(nout, B, T, C) * nout * C * sizeof(float);
}

int tmix_ddlerp_mix_backward_bf16(int B, int T, int C, const void *x, const void *shift_state, const void *maa,
                                  const void *m, const void *gxw, const void *gxk, const void *gxv,
                                  const void *gxr, const void *gxg, void *gx, void *gm, float *gmaa,
                                  void *gshift, void *ws, size_t ws_bytes, void *stream) {
    if (B < 0 || T < 0 || C <= 0 || (C & 7)) { set_error("tmix_ddlerp_mix_backward_bf16: need C %% 8 == 0"); return WKV6_EINVAL; }
    if (B > INT_MAX / 5) { set_error("tmix_ddlerp_mix_backward_bf16: need 5*B <= INT_MAX"); return WKV6_EINVAL; }
    if ((long long)B * T == 0) return WKV6_OK;
    if (!x || !maa || !m || !gxw || !gxk || !gxv || !gxr || !gxg || !gx || !gm || !ws) {
        set_error("tmix_ddlerp_mix_backward_bf16: null pointer");
        return WKV6_EINVAL;
    }
    if (ws_bytes < elementwise_backward_workspace_bytes(B, T, C, 5)) { set_error("tmix_ddlerp_mix_backward_bf16: workspace too small"); return WKV6_EINVAL; }
    if (!check_aligned16("tmix_ddlerp_mix_backward_bf16", {{"x", x}, {"shift_state", shift_state}, {"maa", maa}, {"m", m}, {"gxw", gxw},
                                                            {"gxk", gxk}, {"gxv", gxv}, {"gxr", gxr}, {"gxg", gxg}, {"gx", gx}, {"gm", gm},
                                                            {"gshift", shift_state ? gshift : nullptr}}))
        return WKV6_EINVAL;
    const void *gouts[5] = {gxw, gxk, gxv, gxr, gxg};
    return shift_lerp_backward(5, B, T, C, x, shift_state, maa, m, gouts, gx, gm, gmaa, gshift, ws, stream);
}

int tmix_shift_lerp_backward_bf16(int B, int T, int C, const void *x, const void *shift_state, const void *maa_x,
                                  const void *gout, void *gx, float *gmaa_x, void *gshift, void *ws,
                                  size_t ws_bytes, void *stream) {
    if (B < 0 || T < 0 || C <= 0 || (C & 7)) { set_error("tmix_shift_lerp_backward_bf16: need C %% 8 == 0"); return WKV6_EINVAL; }
    if ((long long)B * T == 0) return WKV6_OK;
    if (!x || !maa_x || !gout || !gx || !ws) { set_error("tmix_shift_lerp_backward_bf16: null pointer"); return WKV6_EINVAL; }
    if (ws_bytes < elementwise_backward_workspace_bytes(B, T, C, 1)) { set_error("tmix_shift_lerp_backward_bf16: workspace too small"); return WKV6_EINVAL; }
    if (!check_aligned16("tmix_shift_lerp_backward_bf16", {{"x", x}, {"shift_state", shift_state}, {"maa_x", maa_x}, {"gout", gout}, {"gx", gx},
                                                            {"gshift", shift_state ? gshift : nullptr}}))
        return WKV6_EINVAL;
    return shift_lerp_backward(1, B, T, C, x, shift_state, maa_x, nullptr, &gout, gx, nullptr, gmaa_x, gshift, ws, stream);
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
    const void *gouts[2] = {gxk, gxr};
    return shift_lerp_backward(2, B, T, C, x, shift_state, maa_kr, nullptr, gouts, gx, nullptr, gmaa_kr, gshift, ws, stream);
}

}  // extern "C"
