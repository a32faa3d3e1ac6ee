// Memory-bound neighbours of the WKV6 recurrence: eos gather, pooling, mask / reverse index,
// token-shift ddlerp mixing, GroupNorm*gate.  All HBM-bound: 128-bit accesses, one pass over the
// big tensor each, grids sized to oversubscribe the 148 SMs.
#include "bf16x8.cuh"
#include "common.cuh"

namespace wkv6 {
namespace {

typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------------------------------------
// eos index: first t with idx[b,t] == id, 0 if absent.  One block per row.
// ------------------------------------------------------------------------------------------------
__global__ void eos_index_kernel(int T, const int64_t *__restrict__ idx, int64_t id, int64_t *__restrict__ pos) {
    const int b = blockIdx.x;
    const int64_t *row = idx + (size_t)b * T;
    __shared__ int best;
    if (threadIdx.x == 0) best = T;
    __syncthreads();
    int mine = T;
    for (int t = threadIdx.x; t < T; t += blockDim.x)
        if (row[t] == id) { mine = t; break; }
    // warp min then one shared atomic per warp
    for (int o = 16; o > 0; o >>= 1) mine = min(mine, __shfl_xor_sync(0xffffffffu, mine, o));
    if ((threadIdx.x & 31) == 0 && mine < T) atomicMin(&best, mine);
    __syncthreads();
    if (threadIdx.x == 0) pos[b] = best >= T ? 0 : best;
}

// out[b,:] = x[b,pos[b],:]
__global__ void gather_rows_kernel(int T, int D, const bf16 *__restrict__ x, const int64_t *__restrict__ pos,
                                   bf16 *__restrict__ out) {
    const int b = blockIdx.x;
    int64_t p = pos[b];
    p = p < 0 ? p + T : p;  // python-style negative index, like torch advanced indexing
    if (p < 0 || p >= T) __trap();   // torch raises an IndexError here; never read out of bounds
    const bf16 *src = x + ((size_t)b * T + (size_t)p) * D;
    bf16 *dst = out + (size_t)b * D;
    if ((D & 7) == 0) {
        for (int d = threadIdx.x * 8; d < D; d += blockDim.x * 8) st8(dst + d, ld8(src + d));
    } else {
        for (int d = threadIdx.x; d < D; d += blockDim.x) dst[d] = src[d];
    }
}

// out[b,t,:] = x[b,rev[b,t],:]   one warp per token row
__global__ void gather_tokens_kernel(int BT, int T, int D, const bf16 *__restrict__ x,
                                     const int64_t *__restrict__ rev, bf16 *__restrict__ out) {
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < BT; row += warps) {
        const int b = row / T;
        const bf16 *src = x + ((size_t)b * T + (size_t)rev[row]) * D;
        bf16 *dst = out + (size_t)row * D;
        if ((D & 7) == 0) for (int d = lane * 8; d < D; d += 256) st8(dst + d, ld8(src + d));
        else for (int d = lane; d < D; d += 32) dst[d] = src[d];
    }
}

// out[b,t,:] = x[b,t,:] and out[B + b,t,:] = x[b,rev[b,t],:]: the plain and the reversed sequences stacked as one batch of
// 2B rows (what the bidirectional encoders feed their projections), one read of x
__global__ void stack_reversed_kernel(int BT, int T, int D, const bf16 *__restrict__ x, const int64_t *__restrict__ rev,
                                      bf16 *__restrict__ out) {
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < BT; row += warps) {
        const int b = row / T;
        const bf16 *src = x + (size_t)row * D, *srcr = x + ((size_t)b * T + (size_t)rev[row]) * D;
        bf16 *dst = out + (size_t)row * D, *dstr = dst + (size_t)BT * D;
        for (int d = lane * 8; d < D; d += 256) {
            st8(dst + d, ld8(src + d));
            st8(dstr + d, ld8(srcr + d));
        }
    }
}

// mask + reverse index, one block per row
__global__ void mask_rev_kernel(int T, const int64_t *__restrict__ idx, int64_t emb, int64_t pad,
                                int32_t *__restrict__ mask, int64_t *__restrict__ rev) {
    const int b = blockIdx.x;
    const int64_t *row = idx + (size_t)b * T;
    __shared__ int len;
    if (threadIdx.x == 0) len = 0;
    __syncthreads();
    int cnt = 0;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        const int m = (row[t] != pad) && (row[t] != emb);
        if (mask) mask[(size_t)b * T + t] = m;
        cnt += m;
    }
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&len, cnt);
    __syncthreads();
    const int L = len;
    if (rev)
        for (int t = threadIdx.x; t < T; t += blockDim.x) rev[(size_t)b * T + t] = t < L ? L - 1 - t : t;
}

// ------------------------------------------------------------------------------------------------
// pooling.  grid (D/64 column tiles, B); block 256 = 8 column threads (8 channels each) x 32 row
// groups; deterministic in-block reduction.  fp32 accumulate, weights exactly as the reference
// writes them: w_t = float(t+1) / float(L) * [t <= L], result / float(L).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pooling_kernel(int kind, int T, int D, const bf16 *__restrict__ x,
                                                      const int64_t *__restrict__ alen, int add_one,
                                                      float *__restrict__ out) {
    const int b = blockIdx.y;
    const int cg = threadIdx.x & 7, rg = threadIdx.x >> 3;
    const int d0 = blockIdx.x * 64 + cg * 8;
    const int64_t L64 = alen[b] + add_one;
    const float Lf = (float)L64;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    __shared__ float red[32][64 + 1];
    // weightedmean: t <= L ; avg: t < L
    long long tend = (kind == 0) ? L64 + 1 : L64;
    if (tend > T) tend = T;
    if (d0 < D) {
        const bf16 *base = x + (size_t)b * T * D + d0;
        for (int t = rg; t < tend; t += 32) {
            float f[8];
            if (d0 + 8 <= D && (D & 7) == 0) unpack8(ld8(base + (size_t)t * D), f);
            else
                for (int e = 0; e < 8; e++) f[e] = d0 + e < D ? __bfloat162float(base[(size_t)t * D + e]) : 0.f;
            // reference: x(bf16) * weights(fp32) -> fp32 product, summed in fp32
            const float wgt = (kind == 0) ? (float)(t + 1) / Lf : 1.0f;
#pragma unroll
            for (int e = 0; e < 8; e++) acc[e] += f[e] * wgt;
        }
    }
#pragma unroll
    for (int e = 0; e < 8; e++) red[rg][cg * 8 + e] = acc[e];
    __syncthreads();
    if (threadIdx.x < 64) {
        float s = 0.f;
#pragma unroll 8
        for (int r = 0; r < 32; r++) s += red[r][threadIdx.x];
        const int d = blockIdx.x * 64 + threadIdx.x;
        if (d < D) out[(size_t)b * D + d] = s / Lf;
    }
}

// ------------------------------------------------------------------------------------------------
// token-shift ddlerp, mixing stage: out[n] = x + (shift(x) - x) * (maa[n] + m[n]),  n = 0..4
// bf16 op-by-op rounding like the reference's eager chain (src/model.py:437-449).
// One thread = 8 channels of one token; grid-stride.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ddlerp_mix_kernel(int B, int T, int C, const bf16 *__restrict__ x,
                                                         const bf16 *__restrict__ shift, const bf16 *__restrict__ maa,
                                                         const bf16 *__restrict__ m, bf16 *__restrict__ out) {
    const size_t nvec = (size_t)B * T * C / 8, plane = (size_t)B * T * C;
    const int cv = C / 8;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (size_t)gridDim.x * blockDim.x) {
        const size_t row = i / cv;
        const int c = (int)(i % cv) * 8, t = (int)(row % T), b = (int)(row / T);
        float xf[8], pf[8], xx[8];
        unpack8(ld8(x + i * 8), xf);
        if (t > 0) unpack8(ld8(x + i * 8 - C), pf);
        else if (shift) unpack8(ld8(shift + (size_t)b * C + c), pf);
        else
            for (int e = 0; e < 8; e++) pf[e] = 0.f;
#pragma unroll
        for (int e = 0; e < 8; e++) xx[e] = rb(pf[e] - xf[e]);
#pragma unroll
        for (int n = 0; n < 5; n++) {
            float mf[8], af[8], o[8];
            unpack8(ld8(m + n * plane + i * 8), mf);
            unpack8(ld8(maa + (size_t)n * C + c), af);
#pragma unroll
            for (int e = 0; e < 8; e++) o[e] = xf[e] + rb(xx[e] * rb(af[e] + mf[e]));
            st8(out + n * plane + i * 8, pack8(o));
        }
    }
}

// xxx = x + (shift(x) - x) * maa_x.  One block per (b, 16 token rows): a thread keeps its 8 channels of maa_x and of the previous token in
// registers and walks 16 token rows -- every x element is read once (plus one row per 16), no index arithmetic per vector.
constexpr int SHIFT_ROWS = 16;
__global__ void __launch_bounds__(256) shift_lerp_kernel(int B, int T, int C, const bf16 *__restrict__ x,
                                                         const bf16 *__restrict__ shift, const bf16 *__restrict__ maa_x,
                                                         bf16 *__restrict__ out) {
    const int nt = (T + SHIFT_ROWS - 1) / SHIFT_ROWS;
    const int b = blockIdx.x / nt, t0 = (blockIdx.x % nt) * SHIFT_ROWS, t1 = min(T, t0 + SHIFT_ROWS);
    for (int c = threadIdx.x * 8; c < C; c += blockDim.x * 8) {
        float pf[8], af[8];
        unpack8(ld8(maa_x + c), af);
        if (t0 > 0) unpack8(ld8(x + ((size_t)b * T + t0 - 1) * C + c), pf);
        else if (shift) unpack8(ld8(shift + (size_t)b * C + c), pf);
        else
            for (int e = 0; e < 8; e++) pf[e] = 0.f;
        const bf16 *src = x + ((size_t)b * T + t0) * C + c;
        bf16 *dst = out + ((size_t)b * T + t0) * C + c;
        for (int t = t0; t < t1; t++, src += C, dst += C) {
            float xf[8], o[8];
            unpack8(ld8(src), xf);
#pragma unroll
            for (int e = 0; e < 8; e++) { o[e] = xf[e] + rb(rb(pf[e] - xf[e]) * af[e]); pf[e] = xf[e]; }
            st8(dst, pack8(o));
        }
    }
    (void)B;
}

// GroupNorm over 64-channel groups, then * g.  8 lanes (8 channels each) per group.
// PAIR: the normalised input is (y + y2[b, rev[b,t]]) / 2 -- the two directions of the bi-directional
// encoders (src/model_encoder_run.py:72-74) -- so the reverse gather and the average cost no pass of their own
template <bool SILU, bool PAIR>
__global__ void __launch_bounds__(256) gn_gate_kernel(size_t ngroups, int C, float eps, const bf16 *__restrict__ y,
                                                      const bf16 *__restrict__ g, const bf16 *__restrict__ lw,
                                                      const bf16 *__restrict__ lb, bf16 *__restrict__ out,
                                                      const bf16 *__restrict__ y2, const int64_t *__restrict__ rev, int T) {
    const size_t nvec = ngroups * 8;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    // all 32 lanes of a warp iterate together (nvec is a multiple of 8, pad the loop to warps)
    for (size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i0 - (threadIdx.x & 31) < nvec; i0 += stride) {
        const bool live = i0 < nvec;
        const size_t i = live ? i0 : nvec - 1;
        float f[8];
        unpack8(ld8(y + i * 8), f);
        if (PAIR) {
            const size_t row = (i * 8) / C;                      // b*T + t
            const size_t src = (row / T) * T + (size_t)rev[row];
            float f2[8];
            unpack8(ld8(y2 + src * C + (i * 8) % C), f2);
#pragma unroll
            for (int e = 0; e < 8; e++) f[e] = rb(f[e] + f2[e]) * 0.5f;
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
        for (int e = 0; e < 8; e++) { const float d = f[e] - mean; q += d * d; }
        q += __shfl_xor_sync(0xffffffffu, q, 1);
        q += __shfl_xor_sync(0xffffffffu, q, 2);
        q += __shfl_xor_sync(0xffffffffu, q, 4);
        const float rstd = rsqrtf(q * (1.0f / 64.0f) + eps);
        const int c = (int)((i * 8) % C);
        float wf[8], bfv[8], gf[8], o[8];
        unpack8(ld8(lw + c), wf);
        unpack8(ld8(lb + c), bfv);
        unpack8(ld8(g + i * 8), gf);
        if (SILU) {                                        // g = F.silu(gate(xg)) of jit_func, as a bf16 tensor
#pragma unroll
            for (int e = 0; e < 8; e++) gf[e] = rb(gf[e] / (1.f + __expf(-gf[e])));
        }
#pragma unroll
        for (int e = 0; e < 8; e++) o[e] = rb((f[e] - mean) * rstd * wf[e] + bfv[e]) * gf[e];
        if (live) st8(out + i * 8, pack8(o));
    }
}

// ------------------------------------------------------------------------------------------------
// fp32 log-decay ew = -exp(w) (what the reference's wkv6 / wkv6_bi pybind entries receive,
// src/model.py:210) -> the raw bf16 logits w the tensor-core kernels read.  The reference builds ew
// from a bf16 w, so bf16(log(-ew)) recovers that w exactly; a stream in which some element does not
// survive the round trip (ew was not made from bf16 logits) gets its flag raised and is computed by
// the exact SIMT kernels from the original fp32 values.
// ------------------------------------------------------------------------------------------------
// mode 0: in = ew = -exp(w);  mode 1: in = decay = exp(-exp(w)) (the rwkv6 inference entry, src/model_run.py:64)
__global__ void __launch_bounds__(256) ew_to_raw_kernel(size_t n8, int T, int H, int mode, const float *__restrict__ in,
                                                        bf16 *__restrict__ w, int *__restrict__ flags) {
    const size_t C = (size_t)H * 64;
    const float tol = mode ? 2e-4f : 1e-5f;               // log(decay) of a slow channel carries fewer exact bits
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
        const float4 a = reinterpret_cast<const float4 *>(in)[2 * i], b = reinterpret_cast<const float4 *>(in)[2 * i + 1];
        float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        float f[8];
        bool bad = false;
#pragma unroll
        for (int e = 0; e < 8; e++) {
            x[e] = mode ? -logf(x[e]) : -x[e];              // exp(w)
            const float lw = logf(x[e]);                    // x = 0 -> -inf (no decay), x < 0 -> NaN (flagged)
            f[e] = lw;
            const float back = expf(rb(lw));
            bad |= !(fabsf(back - x[e]) <= tol * x[e]);
        }
        st8(w + 8 * i, pack8(f));
        if (bad) {
            const size_t e0 = 8 * i, bt = e0 / C, c = e0 % C;
            flags[(bt / T) * H + c / 64] = 1;
        }
    }
}

}  // namespace
}  // namespace wkv6

// internal (not part of the C ABI)
namespace wkv6 {
int ew_to_raw_bf16(int B, int T, int H, const float *ew, void *w_raw, int *flags, cudaStream_t stream, int from_decay) {
    const size_t n8 = (size_t)B * T * H * 64 / 8;
    if (n8 == 0) return WKV6_OK;
    ew_to_raw_kernel<<<grid_for(n8, 256), 256, 0, stream>>>(n8, T, H, from_decay, ew, (bf16 *)w_raw, flags);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}
}  // namespace wkv6

using namespace wkv6;

extern "C" {

int eos_index_i64(int B, int T, const int64_t *idx, int64_t token_id, int64_t *pos, void *stream) {
    if (B < 0 || T < 0) { set_error("eos_index_i64: bad shape"); return WKV6_EINVAL; }
    if (B == 0) return WKV6_OK;
    if (!idx || !pos) { set_error("eos_index_i64: null pointer"); return WKV6_EINVAL; }
    eos_index_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(T, idx, token_id, pos);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int gather_rows_bf16(int B, int T, int D, const void *x, const int64_t *pos, void *out, void *stream) {
    if (B < 0 || T <= 0 || D <= 0) { set_error("gather_rows_bf16: bad shape"); return WKV6_EINVAL; }
    if (B == 0) return WKV6_OK;
    if (!x || !pos || !out) { set_error("gather_rows_bf16: null pointer"); return WKV6_EINVAL; }
    if ((D & 7) == 0 && !check_aligned16("gather_rows_bf16", {{"x", x}, {"out", out}})) return WKV6_EINVAL;
    gather_rows_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(T, D, (const bf16 *)x, pos, (bf16 *)out);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int pooling_bf16(int kind, int variant, int B, int T, int D, const void *x, const int64_t *actual_len,
                 float *out_f32, void *stream) {
    if (B < 0 || T <= 0 || D <= 0 || kind < 0 || kind > 2) { set_error("pooling_bf16: bad arguments"); return WKV6_EINVAL; }
    if (B == 0) return WKV6_OK;
    if (!x || !actual_len || !out_f32) { set_error("pooling_bf16: null pointer"); return WKV6_EINVAL; }
    if ((D & 7) == 0 && !check_aligned16("pooling_bf16", {{"x", x}})) return WKV6_EINVAL;
    if (kind == 1) { set_error("pooling_bf16: lasttoken is gather_rows_bf16"); return WKV6_EINVAL; }
    dim3 grid((D + 63) / 64, B);
    pooling_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(kind, T, D, (const bf16 *)x, actual_len,
                                                           (kind == 0 && variant == 1) ? 1 : 0, out_f32);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int create_mask_rev_idx(int B, int T, const int64_t *idx, int64_t emb_id, int64_t pad_id, int32_t *mask,
                        int64_t *rev_idx, void *stream) {
    if (B < 0 || T < 0) { set_error("create_mask_rev_idx: bad shape"); return WKV6_EINVAL; }
    if (B == 0 || T == 0) return WKV6_OK;
    if (!idx) { set_error("create_mask_rev_idx: null pointer"); return WKV6_EINVAL; }
    mask_rev_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(T, idx, emb_id, pad_id, mask, rev_idx);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int gather_tokens_bf16(int B, int T, int D, const void *x, const int64_t *rev_idx, void *out, void *stream) {
    if (B < 0 || T < 0 || D <= 0) { set_error("gather_tokens_bf16: bad shape"); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    if (!x || !rev_idx || !out) { set_error("gather_tokens_bf16: null pointer"); return WKV6_EINVAL; }
    if ((D & 7) == 0 && !check_aligned16("gather_tokens_bf16", {{"x", x}, {"out", out}})) return WKV6_EINVAL;
    const int BT = B * T;
    gather_tokens_kernel<<<grid_for((size_t)BT * 32, 256), 256, 0, (cudaStream_t)stream>>>(
        BT, T, D, (const bf16 *)x, rev_idx, (bf16 *)out);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int stack_reversed_bf16(int B, int T, int D, const void *x, const int64_t *rev_idx, void *out, void *stream) {
    if (B < 0 || T < 0 || D <= 0 || (D & 7)) { set_error("stack_reversed_bf16: need D %% 8 == 0"); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    if (!x || !rev_idx || !out) { set_error("stack_reversed_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("stack_reversed_bf16", {{"x", x}, {"out", out}})) return WKV6_EINVAL;
    const int BT = B * T;
    stack_reversed_kernel<<<grid_for((size_t)BT * 32, 256), 256, 0, (cudaStream_t)stream>>>(BT, T, D, (const bf16 *)x, rev_idx, (bf16 *)out);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int tmix_ddlerp_mix_bf16(int B, int T, int C, const void *x, const void *shift_state, const void *maa,
                         const void *m, void *out, void *stream) {
    if (B < 0 || T < 0 || C <= 0 || (C & 7)) { set_error("tmix_ddlerp_mix_bf16: need C %% 8 == 0"); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    if (!x || !maa || !m || !out) { set_error("tmix_ddlerp_mix_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("tmix_ddlerp_mix_bf16", {{"x", x}, {"shift_state", shift_state}, {"maa", maa}, {"m", m}, {"out", out}}))
        return WKV6_EINVAL;
    ddlerp_mix_kernel<<<grid_for((size_t)B * T * C / 8, 256), 256, 0, (cudaStream_t)stream>>>(
        B, T, C, (const bf16 *)x, (const bf16 *)shift_state, (const bf16 *)maa, (const bf16 *)m, (bf16 *)out);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int tmix_shift_lerp_bf16(int B, int T, int C, const void *x, const void *shift_state, const void *maa_x,
                         void *out, void *stream) {
    if (B < 0 || T < 0 || C <= 0 || (C & 7)) { set_error("tmix_shift_lerp_bf16: need C %% 8 == 0"); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    if (!x || !maa_x || !out) { set_error("tmix_shift_lerp_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("tmix_shift_lerp_bf16", {{"x", x}, {"shift_state", shift_state}, {"maa_x", maa_x}, {"out", out}})) return WKV6_EINVAL;
    shift_lerp_kernel<<<(unsigned)((size_t)B * ((T + SHIFT_ROWS - 1) / SHIFT_ROWS)), 256, 0, (cudaStream_t)stream>>>(
        B, T, C, (const bf16 *)x, (const bf16 *)shift_state, (const bf16 *)maa_x, (bf16 *)out);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int groupnorm_gate_bf16(int BT, int C, int H, float eps, int gate_act, const void *y, const void *g,
                        const void *ln_w, const void *ln_b, void *out, void *stream) {
    if (BT < 0 || H <= 0 || C != H * 64) { set_error("groupnorm_gate_bf16: need C == H*64"); return WKV6_EINVAL; }
    if (BT == 0) return WKV6_OK;
    if (!y || !g || !ln_w || !ln_b || !out) { set_error("groupnorm_gate_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("groupnorm_gate_bf16", {{"y", y}, {"g", g}, {"ln_w", ln_w}, {"ln_b", ln_b}, {"out", out}})) return WKV6_EINVAL;
    const size_t ngroups = (size_t)BT * H;
    if (gate_act)
        gn_gate_kernel<true, false><<<grid_for(ngroups * 8, 256), 256, 0, (cudaStream_t)stream>>>(
            ngroups, C, eps, (const bf16 *)y, (const bf16 *)g, (const bf16 *)ln_w, (const bf16 *)ln_b, (bf16 *)out, nullptr, nullptr, 1);
    else
        gn_gate_kernel<false, false><<<grid_for(ngroups * 8, 256), 256, 0, (cudaStream_t)stream>>>(
            ngroups, C, eps, (const bf16 *)y, (const bf16 *)g, (const bf16 *)ln_w, (const bf16 *)ln_b, (bf16 *)out, nullptr, nullptr, 1);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int groupnorm_gate_pair_bf16(int B, int T, int C, int H, float eps, int gate_act, const void *y, const void *y_rev,
                             const int64_t *rev_idx, const void *g, const void *ln_w, const void *ln_b, void *out,
                             void *stream) {
    if (B < 0 || T < 0 || H <= 0 || C != H * 64) { set_error("groupnorm_gate_pair_bf16: need C == H*64"); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    if (!y || !y_rev || !rev_idx || !g || !ln_w || !ln_b || !out) { set_error("groupnorm_gate_pair_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("groupnorm_gate_pair_bf16", {{"y", y}, {"y_rev", y_rev}, {"g", g}, {"ln_w", ln_w}, {"ln_b", ln_b}, {"out", out}}))
        return WKV6_EINVAL;
    const size_t ngroups = (size_t)B * T * H;
    if (gate_act)
        gn_gate_kernel<true, true><<<grid_for(ngroups * 8, 256), 256, 0, (cudaStream_t)stream>>>(
            ngroups, C, eps, (const bf16 *)y, (const bf16 *)g, (const bf16 *)ln_w, (const bf16 *)ln_b, (bf16 *)out,
            (const bf16 *)y_rev, rev_idx, T);
    else
        gn_gate_kernel<false, true><<<grid_for(ngroups * 8, 256), 256, 0, (cudaStream_t)stream>>>(
            ngroups, C, eps, (const bf16 *)y, (const bf16 *)g, (const bf16 *)ln_w, (const bf16 *)ln_b, (bf16 *)out,
            (const bf16 *)y_rev, rev_idx, T);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

}  // extern "C"
