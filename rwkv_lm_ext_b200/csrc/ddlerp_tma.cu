// Token-shift ddlerp backward as a TMA-fed streaming kernel.
//
// The gradient of  out_n = x + xx * coef_n  reads 11 tensors of [B,T,C] (x, five incoming gradients,
// five LoRA coefficients m_n) and writes 6 (gx, five gm_n): 34 B per element, nothing but HBM
// traffic.  A register-fed kernel keeps only ~45 KB per SM in flight and stalls on every cold miss
// (DESIGN.md §4.4); here one elected thread streams [8 tokens x 256 channels] boxes of all 11
// inputs into a 3-stage shared-memory ring with cp.async.bulk.tensor (~90 KB in flight per SM while
// a tile is being consumed) and the 8 warps read the tile with conflict-free 16-byte loads.
//
// CTA = (256-channel column block, sequence b, split k of the T axis); tiles are walked from the
// last token of the split to the first, because gx[t] needs gxx[t+1]:
//     gxx[t] = sum_n gout_n[t] * coef_n[t]          gx[t] = sum_n gout_n[t] - gxx[t] + gxx[t+1]
// Inside a tile every warp owns one token row; rows exchange gxx through shared memory.  Rows past
// the end of the sequence and the row before its start arrive zero-filled from TMA, which is exactly
// gxx[T] = 0 and the zero padding of nn.ZeroPad2d((0,0,1,-1)) (src/model.py:428).
// Parameter gradients: per-thread accumulators, reduced over the 8 rows in shared memory, written as
// fp32 partials [B*splits][n][C]; sum_partials (elementwise_bwd.cu) adds them in a fixed order.
#include "bf16x8.cuh"
#include "common.cuh"
#include "tc_common.cuh"

namespace wkv6 {
namespace {

using namespace tc;
typedef __nv_bfloat16 bf16;

constexpr int ROWS = 8, COLS = 256, NS = 3;

struct Maps5 { CUtensorMap m[5]; };
struct Ptr5 { const bf16 *p[5]; };

template <int NOUT, bool HAS_M>
struct Smem {
    static constexpr int X_BYTES = (ROWS + 1) * COLS * 2;                  // 9 rows: t0-1 .. t0+7
    static constexpr int T_BYTES = ROWS * COLS * 2;                        // one [8][256] bf16 box
    static constexpr int STAGE = X_BYTES + NOUT * T_BYTES * (HAS_M ? 2 : 1);
    static constexpr int OFF_GXX = NS * STAGE;                             // float [9][256]
    static constexpr int OFF_MAA = OFF_GXX + (ROWS + 1) * COLS * 4;        // float [NOUT][256]
    static constexpr int OFF_BAR = OFF_MAA + NOUT * COLS * 4;
    static constexpr int TOTAL = OFF_BAR + NS * 8;
    static constexpr int RED = ROWS * NOUT * (COLS + 8) * 4;               // aliases the stages at the end
    static_assert(RED <= NS * STAGE, "reduction scratch must fit in the stage ring");
};

template <int NOUT, bool HAS_M>
__global__ void __launch_bounds__(256, 1)
ddlerp_bwd_tma_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_m,
                      const __grid_constant__ Maps5 map_g, int B, int T, int C, int splits, int rows_per_split,
                      const bf16 *__restrict__ shift, const bf16 *__restrict__ maa, const bf16 *__restrict__ m,
                      const Ptr5 gout, bf16 *__restrict__ gx, bf16 *__restrict__ gm, bf16 *__restrict__ gshift,
                      float *__restrict__ partial) {
    typedef Smem<NOUT, HAS_M> S;
    extern __shared__ __align__(128) uint8_t smem[];
    float *gxs = reinterpret_cast<float *>(smem + S::OFF_GXX);
    float *maas = reinterpret_cast<float *>(smem + S::OFF_MAA);
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + S::OFF_BAR);

    const int lane = threadIdx.x & 31, row = threadIdx.x >> 5;
    const int c0 = blockIdx.x * COLS, c = c0 + lane * 8;
    const bool clive = c < C;
    const int b = blockIdx.y / splits, k = blockIdx.y % splits;
    const int ta = k * rows_per_split;
    const int tb = min(T, ta + rows_per_split);
    const int ntiles = (tb - ta + ROWS - 1) / ROWS;
    const size_t plane = (size_t)B * T * C;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NS; s++) mbar_init(&full[s], 1);
        fence_barrier_init();
        tma_prefetch_desc(&map_x);
        if (HAS_M) tma_prefetch_desc(&map_m);
    }
    for (int i = threadIdx.x; i < NOUT * COLS; i += 256) {
        const int n = i / COLS, cc = c0 + i % COLS;
        maas[i] = cc < C ? __bfloat162float(maa[(size_t)n * C + cc]) : 0.f;
    }
    __syncthreads();

    auto issue = [&](int i) {          // tile i counts down from the end of the split
        const int s = i % NS, t0 = ta + (ntiles - 1 - i) * ROWS;
        uint8_t *st = smem + s * S::STAGE;
        mbar_arrive_expect_tx(&full[s], S::STAGE);
        tma_load_3d(st, &map_x, &full[s], c0, t0 - 1, b);
#pragma unroll
        for (int n = 0; n < NOUT; n++) {
            tma_load_3d(st + S::X_BYTES + n * S::T_BYTES, &map_g.m[n], &full[s], c0, t0, b);
            if (HAS_M) tma_load_3d(st + S::X_BYTES + (NOUT + n) * S::T_BYTES, &map_m, &full[s], c0, t0, n * B + b);
        }
    };
    if (threadIdx.x == 0)
        for (int i = 0; i < NS && i < ntiles; i++) issue(i);

    // carry-in: gxx of the first row after this split (0 at the end of the sequence)
    if (row == 0) {
        float cg[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (tb < T && clive) {
            const size_t off = ((size_t)b * T + tb) * C + c;
#pragma unroll
            for (int n = 0; n < NOUT; n++) {
                float gf[8], cf[8];
                unpack8(ld8(gout.p[n] + off), gf);
                if (HAS_M) unpack8(ld8(m + n * plane + off), cf);
#pragma unroll
                for (int e = 0; e < 8; e++) {
                    const float a = maas[n * COLS + lane * 8 + e];
                    cg[e] = fmaf(gf[e], HAS_M ? rb(a + cf[e]) : a, cg[e]);
                }
            }
        }
#pragma unroll
        for (int e = 0; e < 8; e++) gxs[ROWS * COLS + lane * 8 + e] = cg[e];
    }
    __syncthreads();

    float acc[NOUT][8];
#pragma unroll
    for (int n = 0; n < NOUT; n++)
#pragma unroll
        for (int e = 0; e < 8; e++) acc[n][e] = 0.f;

    for (int i = 0; i < ntiles; i++) {
        const int s = i % NS, t0 = ta + (ntiles - 1 - i) * ROWS, t = t0 + row;
        const bool live = clive && t < tb;
        const uint8_t *st = smem + s * S::STAGE;
        mbar_wait(&full[s], (i / NS) & 1);

        float xf[8], pf[8], xx[8], gxx[8], gsum[8];
        unpack8(ld8(st + ((row + 1) * COLS + lane * 8) * 2), xf);
        if (t == 0 && shift != nullptr && clive) unpack8(ld8(shift + (size_t)b * C + c), pf);
        else unpack8(ld8(st + (row * COLS + lane * 8) * 2), pf);
#pragma unroll
        for (int e = 0; e < 8; e++) { xx[e] = rb(pf[e] - xf[e]); gxx[e] = 0.f; gsum[e] = 0.f; }
        const size_t off = ((size_t)b * T + t) * C + c;
#pragma unroll
        for (int n = 0; n < NOUT; n++) {
            float gf[8], cf[8], gmv[8];
            unpack8(ld8(st + S::X_BYTES + n * S::T_BYTES + (row * COLS + lane * 8) * 2), gf);
            if (HAS_M)
                unpack8(ld8(st + S::X_BYTES + (NOUT + n) * S::T_BYTES + (row * COLS + lane * 8) * 2), cf);
            const float4 a0 = *reinterpret_cast<const float4 *>(maas + n * COLS + lane * 8);
            const float4 a1 = *reinterpret_cast<const float4 *>(maas + n * COLS + lane * 8 + 4);
            const float af[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const float co = HAS_M ? rb(af[e] + cf[e]) : af[e];
                gxx[e] = fmaf(gf[e], co, gxx[e]);
                gsum[e] += gf[e];
                gmv[e] = gf[e] * xx[e];
                acc[n][e] += gmv[e];                       // rows past the split arrive as zeros
            }
            if (HAS_M && live) st8(gm + n * plane + off, pack8(gmv));
        }
        *reinterpret_cast<float4 *>(gxs + row * COLS + lane * 8) = make_float4(gxx[0], gxx[1], gxx[2], gxx[3]);
        *reinterpret_cast<float4 *>(gxs + row * COLS + lane * 8 + 4) = make_float4(gxx[4], gxx[5], gxx[6], gxx[7]);
        __syncthreads();
        const float4 n0 = *reinterpret_cast<const float4 *>(gxs + (row + 1) * COLS + lane * 8);
        const float4 n1 = *reinterpret_cast<const float4 *>(gxs + (row + 1) * COLS + lane * 8 + 4);
        if (live) {
            const float o[8] = {gsum[0] - gxx[0] + n0.x, gsum[1] - gxx[1] + n0.y, gsum[2] - gxx[2] + n0.z,
                                gsum[3] - gxx[3] + n0.w, gsum[4] - gxx[4] + n1.x, gsum[5] - gxx[5] + n1.y,
                                gsum[6] - gxx[6] + n1.z, gsum[7] - gxx[7] + n1.w};
            st8(gx + off, pack8(o));
            if (t == 0 && gshift != nullptr) st8(gshift + (size_t)b * C + c, pack8(gxx));
        }
        __syncthreads();                                   // gxs and stage s are free again
        if (row == 0) {
            *reinterpret_cast<float4 *>(gxs + ROWS * COLS + lane * 8) = make_float4(gxx[0], gxx[1], gxx[2], gxx[3]);
            *reinterpret_cast<float4 *>(gxs + ROWS * COLS + lane * 8 + 4) = make_float4(gxx[4], gxx[5], gxx[6], gxx[7]);
        }
        if (threadIdx.x == 0 && i + NS < ntiles) issue(i + NS);
    }

    // parameter gradient: reduce over the 8 rows (the stage ring is idle now)
    float *red = reinterpret_cast<float *>(smem);
#pragma unroll
    for (int n = 0; n < NOUT; n++)
#pragma unroll
        for (int e = 0; e < 8; e++) red[(row * NOUT + n) * (COLS + 8) + lane * 8 + e] = acc[n][e];
    __syncthreads();
    for (int i = threadIdx.x; i < NOUT * COLS; i += 256) {
        const int n = i / COLS, cc = i % COLS;
        float sum = 0.f;
#pragma unroll
        for (int r = 0; r < ROWS; r++) sum += red[(r * NOUT + n) * (COLS + 8) + cc];
        if (c0 + cc < C) partial[((size_t)blockIdx.y * NOUT + n) * C + c0 + cc] = sum;
    }
}

// split the T axis so that the grid has about three waves of CTAs (the light shift-lerp variant fits
// several CTAs per SM: eight waves' worth) and every CTA at least 8 tiles
void geometry(int nout, int B, int T, int C, int *splits, int *rows_per_split) {
    const int colblocks = (C + COLS - 1) / COLS;
    int want = (148 * (nout == 5 ? 3 : 8) + B * colblocks - 1) / (B * colblocks);
    const int max_splits = (T + ROWS * 8 - 1) / (ROWS * 8);
    if (want > max_splits) want = max_splits;
    if (want < 1) want = 1;
    int rps = (T + want - 1) / want;
    rps = (rps + ROWS - 1) / ROWS * ROWS;
    *rows_per_split = rps;
    *splits = (T + rps - 1) / rps;
}

}  // namespace

size_t ddlerp_tma_partial_slots(int nout, int B, int T, int C) {
    int splits, rps;
    geometry(nout, B, T, C, &splits, &rps);
    return (size_t)B * splits;
}

int ddlerp_backward_tma(int nout, int B, int T, int C, const void *x, const void *shift, const void *maa, const void *m,
                        const void *const *gouts, void *gx, void *gm, void *gshift, float *partial, int *slots,
                        cudaStream_t stream) {
    int splits, rps;
    geometry(nout, B, T, C, &splits, &rps);
    *slots = B * splits;
    CUtensorMap mx, mm;
    Maps5 mg;
    const CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    bool ok = make_btc_map(&mx, x, B, T, C, ROWS + 1, dt, 2, COLS, false);
    ok = ok && make_btc_map(&mm, m ? m : x, m ? 5 * B : B, T, C, ROWS, dt, 2, COLS, false);
    for (int n = 0; n < 5; n++) ok = ok && make_btc_map(&mg.m[n], gouts[n < nout ? n : 0], B, T, C, ROWS, dt, 2, COLS, false);
    if (!ok) { set_error("ddlerp backward: cuTensorMapEncodeTiled failed"); return WKV6_ECUDA; }
    Ptr5 gp;
    for (int n = 0; n < 5; n++) gp.p[n] = (const bf16 *)gouts[n < nout ? n : 0];
    dim3 grid((C + COLS - 1) / COLS, B * splits);
    static thread_local int attr_done[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (nout == 5) {
        auto kern = ddlerp_bwd_tma_kernel<5, true>;
        if (dev < 64 && !(attr_done[dev] & 1)) {
            WKV6_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Smem<5, true>::TOTAL));
            attr_done[dev] |= 1;
        }
        kern<<<grid, 256, Smem<5, true>::TOTAL, stream>>>(mx, mm, mg, B, T, C, splits, rps, (const bf16 *)shift,
                                                          (const bf16 *)maa, (const bf16 *)m, gp, (bf16 *)gx, (bf16 *)gm,
                                                          (bf16 *)gshift, partial);
    } else if (nout == 2) {
        auto kern = ddlerp_bwd_tma_kernel<2, false>;
        if (dev < 64 && !(attr_done[dev] & 4)) {
            WKV6_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Smem<2, false>::TOTAL));
            attr_done[dev] |= 4;
        }
        kern<<<grid, 256, Smem<2, false>::TOTAL, stream>>>(mx, mm, mg, B, T, C, splits, rps, (const bf16 *)shift,
                                                           (const bf16 *)maa, nullptr, gp, (bf16 *)gx, nullptr,
                                                           (bf16 *)gshift, partial);
    } else {
        auto kern = ddlerp_bwd_tma_kernel<1, false>;
        if (dev < 64 && !(attr_done[dev] & 2)) {
            WKV6_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Smem<1, false>::TOTAL));
            attr_done[dev] |= 2;
        }
        kern<<<grid, 256, Smem<1, false>::TOTAL, stream>>>(mx, mm, mg, B, T, C, splits, rps, (const bf16 *)shift,
                                                           (const bf16 *)maa, nullptr, gp, (bf16 *)gx, nullptr,
                                                           (bf16 *)gshift, partial);
    }
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

}  // namespace wkv6
