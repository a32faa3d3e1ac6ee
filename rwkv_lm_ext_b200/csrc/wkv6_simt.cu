// WKV6 on CUDA cores: exact fp32 step recurrence, every shape, every variant.
//
// This is the always-available GPU path (tiny T, odd shapes, cross-check for the tensor-core
// kernels).  Unlike the reference (one 64-thread block per (b,h), 2 barriers per time step,
// cuda/wkv6_cuda.cu:23-60) a 256-thread block owns one (b,h) stream, splits the 64x64 state into
// 4 slices of 16 contraction indices held in registers, stages TT time steps of r,k,v,decay in
// shared memory at a time and needs barriers only per tile: the per-thread state recurrences are
// independent, only the partial dot products are reduced across the 4 slices at the end of a tile.
//
// Logical time: step tau in [0, Teff) maps to physical t = tau (causal) or Teff-1-tau (the
// reverse pass of wkv6_bi); Teff = T, or p+1 with p the first masked position (wkv6_bi).
#include "common.cuh"

namespace wkv6 {

namespace {

constexpr int TT = 16;        // time steps per shared-memory tile
constexpr int NT = 256;       // threads per block
constexpr int NG = NT / N;    // 4 slices
constexpr int SL = N / NG;    // 16 contraction indices per slice
constexpr int TR = 8;         // tile of the reverse sweep (more shared arrays per step)
constexpr int PER = TR * N / NT;

__device__ __forceinline__ int bi_last_index(const int *mask_row, int T, int *sh) {
    // p = first t with mask == 0, or T-1 (SURVEY.md 8c; cuda/wkv6_bi_cuda.cu:25-69)
    int best = T;
    for (int t = threadIdx.x; t < T; t += blockDim.x)
        if (mask_row[t] == 0) { best = t; break; }
    if (threadIdx.x == 0) *sh = T;
    __syncthreads();
    atomicMin(sh, best);
    __syncthreads();
    int p = *sh;
    __syncthreads();
    return p >= T ? T - 1 : p;
}

template <typename IO>
__device__ __forceinline__ float load_state(const void *s, int f32, size_t idx) {
    return f32 ? ((const float *)s)[idx] : __bfloat162float(((const __nv_bfloat16 *)s)[idx]);
}
__device__ __forceinline__ void store_state(void *s, int f32, size_t idx, float x) {
    if (f32) ((float *)s)[idx] = x;
    else ((__nv_bfloat16 *)s)[idx] = __float2bfloat16_rn(x);
}

// ---------------------------------------------------------------------------------------------
// forward:  y_t[j] = sum_i r_t[i] (u[i] k_t[i] v_t[j] + S[i][j]);  S[i][j] = d_t[i] S[i][j] + k_t[i] v_t[j]
// thread (x = j, g): S[i in 16g..16g+15][j = x]
// mode: 0 causal; 1 = reverse pass of wkv6_bi (reversed time, u = 0, accumulate into y)
// ---------------------------------------------------------------------------------------------
template <typename IO, int WK>
__global__ void __launch_bounds__(NT) fwd_kernel(Args a, int mode) {
    if (a.stream_flags && a.stream_flags[blockIdx.x] == 0) return;
    const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
    const int x = threadIdx.x & (N - 1), g = threadIdx.x >> 6;
    const int T = a.T, C = a.H * N;
    __shared__ float sr[TT][N], sk[TT][N], sd[TT][N], sv[TT][N];
    __shared__ float part[TT][NG][N];
    __shared__ int sh_p;

    int Teff = T;
    if (a.mask) Teff = bi_last_index(a.mask + (size_t)b * T, T, &sh_p) + 1;
    const bool rev = (mode == 1);

    float S[SL], uu[SL];
#pragma unroll
    for (int ii = 0; ii < SL; ii++) {
        const int i = g * SL + ii;
        uu[ii] = rev ? 0.f : to_f32(((const IO *)a.u)[h * N + i]);
        S[ii] = 0.f;
        if (a.s0 && !rev)
            S[ii] = load_state<IO>(a.s0, a.s0_f32, (size_t)b * a.s0_bstride + ((size_t)h * N + x) * N + i);
    }
    const IO *R = (const IO *)a.r, *K = (const IO *)a.k, *V = (const IO *)a.v;
    IO *Y = (IO *)a.y;
    const size_t base = (size_t)b * T * C + (size_t)h * N;

    const int ntiles = (Teff + TT - 1) / TT;
    // register prefetch of the next tile: TT*N = 1024 elements per tensor, 4 per thread
    float pr[4], pk[4], pd[4], pv[4];
    auto prefetch = [&](int tile) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = threadIdx.x + q * NT, tau = tile * TT + e / N, c = e % N;
            if (tau < Teff) {
                const int t = rev ? (Teff - 1 - tau) : tau;
                const size_t o = base + (size_t)t * C + c;
                pr[q] = to_f32(R[o]); pk[q] = to_f32(K[o]); pv[q] = to_f32(V[o]);
                pd[q] = __expf(load_logdecay<WK>(a.w, o, a.lmin));
            } else { pr[q] = 0.f; pk[q] = 0.f; pv[q] = 0.f; pd[q] = 1.f; }
        }
    };
    if (ntiles > 0) prefetch(0);
    for (int tile = 0; tile < ntiles; tile++) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = threadIdx.x + q * NT, tt = e / N, c = e % N;
            sr[tt][c] = pr[q]; sk[tt][c] = pk[q]; sd[tt][c] = pd[q]; sv[tt][c] = pv[q];
        }
        __syncthreads();
        if (tile + 1 < ntiles) prefetch(tile + 1);
#pragma unroll 4
        for (int tt = 0; tt < TT; tt++) {
            const float vj = sv[tt][x];
            float acc = 0.f;
#pragma unroll
            for (int ii = 0; ii < SL; ii++) {
                const int i = g * SL + ii;
                const float kv = sk[tt][i] * vj;
                acc = fmaf(sr[tt][i], fmaf(uu[ii], kv, S[ii]), acc);
                S[ii] = fmaf(S[ii], sd[tt][i], kv);
            }
            part[tt][g][x] = acc;
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = threadIdx.x + q * NT, tt = e / N, c = e % N, tau = tile * TT + tt;
            if (tau < Teff) {
                const int t = rev ? (Teff - 1 - tau) : tau;
                const size_t o = base + (size_t)t * C + c;
                float yv = part[tt][0][c] + part[tt][1][c] + part[tt][2][c] + part[tt][3][c];
                if (rev) yv += to_f32(Y[o]);
                Y[o] = from_f32<IO>(yv);
            }
        }
        // next iteration's smem writes are fenced by the barrier after the tile stores above:
        __syncthreads();
    }
    // positions past the masked end are defined as zero (reference leaves them unwritten)
    if (a.mask && !rev)
        for (int e = threadIdx.x; e < (T - Teff) * N; e += NT)
            Y[base + (size_t)(Teff + e / N) * C + (e % N)] = from_f32<IO>(0.f);
    if (a.sT && !rev) {
#pragma unroll
        for (int ii = 0; ii < SL; ii++)
            store_state(a.sT, a.sT_f32, ((size_t)b * a.H + h) * N * N + (size_t)x * N + g * SL + ii, S[ii]);
    }
}

// ---------------------------------------------------------------------------------------------
// backward, forward-time sweep: gr, gu partials, A_t[i] = r_t[i] * sum_j S_t[i][j] gy_t[j];
// with a final-state gradient also Q0[b,h,i] = sum_j S_T[i][j] gT[i][j], where the reverse sweep's Q starts
// thread (x = i, g): S[i = x][j in 16g..16g+15]
// ---------------------------------------------------------------------------------------------
template <typename IO, int WK>
__global__ void __launch_bounds__(NT) bwd_f_kernel(Args a, int mode, float *Abuf, float *Q0) {
    if (a.stream_flags && a.stream_flags[blockIdx.x] == 0) return;
    const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
    const int x = threadIdx.x & (N - 1), g = threadIdx.x >> 6;
    const int T = a.T, C = a.H * N;
    __shared__ float sr[TT][N], sk[TT][N], sd[TT][N], sv[TT][N], sgy[TT][N];
    __shared__ float part[TT][NG][N];
    __shared__ float pvg[TT][NG];
    __shared__ float sgu[NG][N];
    __shared__ int sh_p;

    int Teff = T;
    if (a.mask) Teff = bi_last_index(a.mask + (size_t)b * T, T, &sh_p) + 1;
    const bool rev = (mode == 1);

    float S[SL];
#pragma unroll
    for (int jj = 0; jj < SL; jj++) {
        const int j = g * SL + jj;
        S[jj] = 0.f;
        if (a.s0 && !rev)
            S[jj] = load_state<IO>(a.s0, a.s0_f32, (size_t)b * a.s0_bstride + ((size_t)h * N + j) * N + x);
    }
    const float ui = rev ? 0.f : to_f32(((const IO *)a.u)[h * N + x]);
    const IO *R = (const IO *)a.r, *K = (const IO *)a.k, *V = (const IO *)a.v, *GY = (const IO *)a.gy;
    IO *GR = (IO *)a.gr;
    const size_t base = (size_t)b * T * C + (size_t)h * N;
    float gu_acc = 0.f;

    const int ntiles = (Teff + TT - 1) / TT;
    float pr[4], pk[4], pd[4], pv[4], pg[4];
    auto prefetch = [&](int tile) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = threadIdx.x + q * NT, tau = tile * TT + e / N, c = e % N;
            if (tau < Teff) {
                const int t = rev ? (Teff - 1 - tau) : tau;
                const size_t o = base + (size_t)t * C + c;
                pr[q] = to_f32(R[o]); pk[q] = to_f32(K[o]); pv[q] = to_f32(V[o]); pg[q] = to_f32(GY[o]);
                pd[q] = __expf(load_logdecay<WK>(a.w, o, a.lmin));
            } else { pr[q] = 0.f; pk[q] = 0.f; pv[q] = 0.f; pg[q] = 0.f; pd[q] = 1.f; }
        }
    };
    if (ntiles > 0) prefetch(0);
    for (int tile = 0; tile < ntiles; tile++) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int e = threadIdx.x + q * NT, tt = e / N, c = e % N;
            sr[tt][c] = pr[q]; sk[tt][c] = pk[q]; sd[tt][c] = pd[q]; sv[tt][c] = pv[q]; sgy[tt][c] = pg[q];
        }
        __syncthreads();
        if (tile + 1 < ntiles) prefetch(tile + 1);
#pragma unroll 2
        for (int tt = 0; tt < TT; tt++) {
            const float ki = sk[tt][x], di = sd[tt][x];
            float sg = 0.f, vg = 0.f;
#pragma unroll
            for (int jj = 0; jj < SL; jj++) {
                const int j = g * SL + jj;
                const float gyj = sgy[tt][j], vj = sv[tt][j];
                sg = fmaf(S[jj], gyj, sg);
                vg = fmaf(vj, gyj, vg);
                S[jj] = fmaf(S[jj], di, ki * vj);
            }
            part[tt][g][x] = sg;
            if (x == 0) pvg[tt][g] = vg;
        }
        __syncthreads();
        // thread (x = i, g) finishes steps tt = g, g+4, g+8, g+12
#pragma unroll
        for (int q = 0; q < TT / NG; q++) {
            const int tt = g + q * NG, tau = tile * TT + tt;
            if (tau < Teff) {
                const int t = rev ? (Teff - 1 - tau) : tau;
                const size_t o = base + (size_t)t * C + x;
                const float sg = part[tt][0][x] + part[tt][1][x] + part[tt][2][x] + part[tt][3][x];
                const float vg = pvg[tt][0] + pvg[tt][1] + pvg[tt][2] + pvg[tt][3];
                const float ri = sr[tt][x], ki = sk[tt][x];
                float grv = fmaf(ui * ki, vg, sg);
                if (rev) grv += to_f32(GR[o]);
                GR[o] = from_f32<IO>(grv);
                // A is indexed by LOGICAL time for the reverse sweep
                Abuf[((size_t)blockIdx.x * T + tau) * N + x] = ri * sg;
                gu_acc = fmaf(ri * ki, vg, gu_acc);
            }
        }
        __syncthreads();
    }
    if (!rev) {
        // zero-fill gr past the masked end (wkv6_bi) so the op's outputs are fully defined
        if (a.mask)
            for (int e = threadIdx.x; e < (T - Teff) * N; e += NT)
                GR[base + (size_t)(Teff + e / N) * C + (e % N)] = from_f32<IO>(0.f);
        sgu[g][x] = gu_acc;
        __syncthreads();
        if (g == 0)
            ((IO *)a.gu)[(size_t)b * C + h * N + x] = from_f32<IO>(sgu[0][x] + sgu[1][x] + sgu[2][x] + sgu[3][x]);
        if (a.gT) {
            float q = 0.f;
#pragma unroll
            for (int jj = 0; jj < SL; jj++)
                q = fmaf(S[jj], load_state<IO>(a.gT, a.gT_f32, ((size_t)blockIdx.x * N + g * SL + jj) * N + x), q);
            __syncthreads();
            sgu[g][x] = q;
            __syncthreads();
            if (g == 0) Q0[(size_t)blockIdx.x * N + x] = sgu[0][x] + sgu[1][x] + sgu[2][x] + sgu[3][x];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// backward, reverse-time sweep: gk, gv, gw, gs.  G = dL/dS_{t+1}, starting from gT (or 0).
//   G1: thread (x = i, g) holds G[i][j in slice]  -> gk_t[i], B_t[i] = k_t[i] sum_j G[i][j] v_t[j]
//   G2: thread (x = j, g) holds G[i in slice][j]  -> gv_t[j]
//   gl_t = Q - B_t ;  Q += A_t - B_t   (Q = Q0 + sum_{s>t}(A_s - B_s));  gw_t = l_t * gl_t
// ---------------------------------------------------------------------------------------------
template <typename IO, int WK>
__global__ void __launch_bounds__(NT, 2) bwd_r_kernel(Args a, int mode, const float *Abuf, const float *Q0) {   // 2 blocks per SM: at most 128 registers
    if (a.stream_flags && a.stream_flags[blockIdx.x] == 0) return;
    const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
    const int x = threadIdx.x & (N - 1), g = threadIdx.x >> 6;
    const int T = a.T, C = a.H * N;
    __shared__ float sr[TR][N], sk[TR][N], sl[TR][N], sv[TR][N], sgy[TR][N], sA[TR][N], sd[TR][N];
    __shared__ float part1[TR][NG][N], part2[TR][NG][N];
    __shared__ float pvg[TR][NG];
    __shared__ int sh_p;

    int Teff = T;
    if (a.mask) Teff = bi_last_index(a.mask + (size_t)b * T, T, &sh_p) + 1;
    const bool rev = (mode == 1);

    float G1[SL], G2[SL], uu[SL];
#pragma unroll
    for (int q = 0; q < SL; q++) {
        G1[q] = 0.f; G2[q] = 0.f;
        if (a.gT && !rev) {
            G1[q] = load_state<IO>(a.gT, a.gT_f32, ((size_t)blockIdx.x * N + g * SL + q) * N + x);
            G2[q] = load_state<IO>(a.gT, a.gT_f32, ((size_t)blockIdx.x * N + x) * N + g * SL + q);
        }
        uu[q] = rev ? 0.f : to_f32(((const IO *)a.u)[h * N + g * SL + q]);
    }
    const float ui = rev ? 0.f : to_f32(((const IO *)a.u)[h * N + x]);
    const IO *R = (const IO *)a.r, *K = (const IO *)a.k, *V = (const IO *)a.v, *GY = (const IO *)a.gy;
    IO *GK = (IO *)a.gk, *GV = (IO *)a.gv, *GW = (IO *)a.gw;
    const size_t base = (size_t)b * T * C + (size_t)h * N;
    const bool zero_gw0 = (a.s0 == nullptr) || rev;
    float Q = a.gT && !rev ? Q0[(size_t)blockIdx.x * N + x] : 0.f;  // meaningful in threads with g == 0 (x = i)
    const bool zero_gw_last = a.gT == nullptr || rev;   // the last decay feeds nothing but the final state

    const int ntiles = (Teff + TR - 1) / TR;
    float pr[PER], pk[PER], pl[PER], pv[PER], pg[PER], pa[PER];
    // tile index counts DOWN; inside a tile tt still counts up in logical time
    auto prefetch = [&](int tile) {
#pragma unroll
        for (int q = 0; q < PER; q++) {
            const int e = threadIdx.x + q * NT, tau = tile * TR + e / N, c = e % N;
            if (tau < Teff) {
                const int t = rev ? (Teff - 1 - tau) : tau;
                const size_t o = base + (size_t)t * C + c;
                pr[q] = to_f32(R[o]); pk[q] = to_f32(K[o]); pv[q] = to_f32(V[o]); pg[q] = to_f32(GY[o]);
                pl[q] = load_logdecay<WK>(a.w, o, a.lmin);
                pa[q] = Abuf[((size_t)blockIdx.x * T + tau) * N + c];
            } else { pr[q] = 0.f; pk[q] = 0.f; pv[q] = 0.f; pg[q] = 0.f; pl[q] = 0.f; pa[q] = 0.f; }
        }
    };
    if (ntiles > 0) prefetch(ntiles - 1);
    for (int tile = ntiles - 1; tile >= 0; tile--) {
#pragma unroll
        for (int q = 0; q < PER; q++) {
            const int e = threadIdx.x + q * NT, tt = e / N, c = e % N;
            sr[tt][c] = pr[q]; sk[tt][c] = pk[q]; sl[tt][c] = pl[q]; sv[tt][c] = pv[q]; sgy[tt][c] = pg[q];
            sA[tt][c] = pa[q]; sd[tt][c] = __expf(pl[q]);
        }
        __syncthreads();
        if (tile > 0) prefetch(tile - 1);
#pragma unroll 2
        for (int tt = TR - 1; tt >= 0; tt--) {
            // layout 1: i = x, j in slice
            const float ri = sr[tt][x], di = sd[tt][x];
            // layout 2: j = x, i in slice
            const float gyx = sgy[tt][x];
            float gvd = 0.f, vg = 0.f, gvp = 0.f, kur = 0.f;
#pragma unroll
            for (int q = 0; q < SL; q++) {
                const int c = g * SL + q;
                const float gyc = sgy[tt][c], vc = sv[tt][c];
                gvd = fmaf(G1[q], vc, gvd);
                vg = fmaf(vc, gyc, vg);
                G1[q] = fmaf(di, G1[q], ri * gyc);
                const float kc = sk[tt][c], rc = sr[tt][c], dc = sd[tt][c];
                gvp = fmaf(kc, G2[q], gvp);
                kur = fmaf(kc * uu[q], rc, kur);
                G2[q] = fmaf(dc, G2[q], rc * gyx);
            }
            part1[tt][g][x] = gvd;
            part2[tt][g][x] = fmaf(kur, gyx, gvp);
            if (x == 0) pvg[tt][g] = vg;
        }
        __syncthreads();
        // gv: 4 outputs per thread
#pragma unroll
        for (int q = 0; q < PER; q++) {
            const int e = threadIdx.x + q * NT, tt = e / N, c = e % N, tau = tile * TR + tt;
            if (tau < Teff) {
                const int t = rev ? (Teff - 1 - tau) : tau;
                const size_t o = base + (size_t)t * C + c;
                float val = part2[tt][0][c] + part2[tt][1][c] + part2[tt][2][c] + part2[tt][3][c];
                if (rev) val += to_f32(GV[o]);
                GV[o] = from_f32<IO>(val);
            }
        }
        // gk and gw: serial in time per key channel (threads g == 0)
        if (g == 0) {
            for (int tt = TR - 1; tt >= 0; tt--) {
                const int tau = tile * TR + tt;
                if (tau >= Teff) continue;
                const int t = rev ? (Teff - 1 - tau) : tau;
                const size_t o = base + (size_t)t * C + x;
                const float gvd = part1[tt][0][x] + part1[tt][1][x] + part1[tt][2][x] + part1[tt][3][x];
                const float vg = pvg[tt][0] + pvg[tt][1] + pvg[tt][2] + pvg[tt][3];
                float gkv = fmaf(ui * sr[tt][x], vg, gvd);
                const float Bt = sk[tt][x] * gvd;
                float gwv = sl[tt][x] > a.lmin ? sl[tt][x] * (Q - Bt) : 0.f;   // a clamped decay no longer depends on w
                if ((tau == Teff - 1 && zero_gw_last) || (tau == 0 && zero_gw0)) gwv = 0.f;
                Q += sA[tt][x] - Bt;
                if (rev) { gkv += to_f32(GK[o]); gwv += to_f32(GW[o]); }
                GK[o] = from_f32<IO>(gkv);
                GW[o] = from_f32<IO>(gwv);
            }
        }
        __syncthreads();
    }
    if (!rev) {
        if (a.mask)
            for (int e = threadIdx.x; e < (T - Teff) * N; e += NT) {
                const size_t o = base + (size_t)(Teff + e / N) * C + (e % N);
                GK[o] = from_f32<IO>(0.f); GV[o] = from_f32<IO>(0.f); GW[o] = from_f32<IO>(0.f);
            }
        if (a.gs) {
            // gs[b,h,j,i] = dL/dS_0[i][j]; thread (x = j, g) holds i in slice
#pragma unroll
            for (int q = 0; q < SL; q++)
                ((IO *)a.gs)[((size_t)b * a.H + h) * N * N + (size_t)x * N + g * SL + q] = from_f32<IO>(G2[q]);
        }
    }
}

template <typename IO>
int launch_fwd(const Args &a, int mode) {
    const dim3 grid(a.B * a.H), block(NT);
    switch (a.w_kind) {
        case W_RAW_BF16: fwd_kernel<IO, W_RAW_BF16><<<grid, block, 0, a.stream>>>(a, mode); break;
        case W_LOG_F32: fwd_kernel<IO, W_LOG_F32><<<grid, block, 0, a.stream>>>(a, mode); break;
        default: fwd_kernel<IO, W_DECAY_F32><<<grid, block, 0, a.stream>>>(a, mode); break;
    }
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

// Q0: nullptr, or fp32 [B*H][64] that carries <S_T, gT>_i from the forward-time sweep to the reverse one
int launch_bwd(const Args &a, int mode, float *Q0) {
    using IO = __nv_bfloat16;
    const dim3 grid(a.B * a.H), block(NT);
    float *A = (float *)a.workspace;
    if (a.w_kind == W_RAW_BF16) {
        bwd_f_kernel<IO, W_RAW_BF16><<<grid, block, 0, a.stream>>>(a, mode, A, Q0);
        bwd_r_kernel<IO, W_RAW_BF16><<<grid, block, 0, a.stream>>>(a, mode, A, Q0);
    } else {
        bwd_f_kernel<IO, W_LOG_F32><<<grid, block, 0, a.stream>>>(a, mode, A, Q0);
        bwd_r_kernel<IO, W_LOG_F32><<<grid, block, 0, a.stream>>>(a, mode, A, Q0);
    }
    count_launch(2);
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

}  // namespace

size_t simt_backward_workspace_bytes(int B, int T, int H) {
    return (size_t)B * T * H * N * sizeof(float);
}

int simt_forward(const Args &a) {
    if (a.B * a.H == 0 || a.T == 0) return WKV6_OK;
    int rc;
    if (a.io_dtype == WKV6_BF16) rc = launch_fwd<__nv_bfloat16>(a, 0);
    else if (a.io_dtype == WKV6_FP16) rc = launch_fwd<__half>(a, 0);
    else rc = launch_fwd<float>(a, 0);
    if (rc != WKV6_OK || !a.mask) return rc;
    return launch_fwd<__nv_bfloat16>(a, 1);   // reverse pass of wkv6_bi, accumulates into y
}

int simt_backward(const Args &a) {
    if (a.B * a.H == 0 || a.T == 0) return WKV6_OK;
    if (a.io_dtype != WKV6_BF16) { set_error("backward is bf16 only"); return WKV6_EINVAL; }
    if (a.workspace_bytes < simt_backward_workspace_bytes(a.B, a.T, a.H) || !a.workspace) {
        set_error("workspace too small: need %zu bytes", simt_backward_workspace_bytes(a.B, a.T, a.H));
        return WKV6_EWORKSPACE;
    }
    if (a.gT) {
        // the final-state gradient (training pair only, never with a mask): <S_T, gT> in stream-ordered scratch, so the
        // workspace of a call without one stays what it was
        ensure_pool_keeps_memory();
        float *Q0 = nullptr;
        WKV6_CUDA_CHECK(cudaMallocAsync((void **)&Q0, (size_t)a.B * a.H * N * sizeof(float), a.stream));
        const int rc = launch_bwd(a, 0, Q0);
        cudaFreeAsync(Q0, a.stream);
        return rc;
    }
    int rc = launch_bwd(a, 0, nullptr);
    if (rc != WKV6_OK || !a.mask) return rc;
    return launch_bwd(a, 1, nullptr);
}

}  // namespace wkv6
