// Token-shift ddlerp with the rank-32 LoRA product fused in (RWKV_Tmix_x060.jit_func, src/model.py:441-448):
//
//     m_n   = h_n @ W2_n                      h = tanh(xxx @ W1) viewed [B*T, 5, 32],  W2 [5, 32, C]
//     out_n = x + xx * (maa_n + m_n)          n = w,k,v,r,g          xx = shift(x) - x
//
// The eager chain (and tmix_ddlerp_mix_bf16) materialises m [5,B,T,C]: 10 B/element written by the bmm
// and 10 B/element read back.  Here the five K=32 products run on the tensor cores inside the kernel and
// m only ever exists in TMEM: HBM traffic drops from 32 to 12 B/element (x in, five outputs out).
//
// CTA = 128 token rows x a range of 64-channel groups; work item = (group g, output n):
//   issuer warp : TMA loads (h tile once; x tile per group, double-buffered; W2_n tile per item, ring
//                 of 3), two tcgen05.mma (M=128, N=64, K=16) per item into one of two TMEM accumulators
//   8 epilogue warps (256 threads): thread = (token row, 32 of the 64 channels): tcgen05.ld of its
//                 accumulator slice, the mixing arithmetic with the reference's bf16 op-by-op rounding,
//                 swizzled shared-memory staging, TMA store of the [128 x 64] output tile
// The MMA of item i+1 runs under the epilogue of item i.
#include "common.cuh"
#include "tc_common.cuh"

namespace wkv6 {
namespace {

using namespace tc;
typedef __nv_bfloat16 bf16;

constexpr int TM = 128, NC = 64, RANK = 32, NOUT = 5;
constexpr int EPI_THREADS = 256, THREADS = 288;
constexpr int H_BOX = TM * 128;                       // one [128 rows][64 cols] bf16 box, 128-byte rows
constexpr int OFF_H = 0;                              // 3 boxes: columns 0-63, 64-127, 128-191 of h
constexpr int X_BYTES = 17408;                        // [129 rows][128 B] of x + [5 rows][128 B] of maa, rounded up to 1024
constexpr int OFF_X = OFF_H + 3 * H_BOX;              // 2 buffers
constexpr int W_BYTES = RANK * 128;                   // [32 k][64 c] bf16
constexpr int OFF_W = OFF_X + 2 * X_BYTES;            // ring of 3
constexpr int OFF_STG = OFF_W + 3 * W_BYTES;          // [128][64] bf16 output staging
constexpr int OFF_BAR = OFF_STG + TM * 128;
constexpr int SMEM_BYTES = OFF_BAR + 128 + 1024;      // + slack for the 1024-byte alignment of the base
constexpr int TM_COLS = 128;                          // two fp32 accumulators of 64 columns

struct Bars {
    uint64_t h, x_full[2], x_free[2], w_full[3], mma[2], acc_free[2];
    uint32_t tmem_base;
};


struct Params {
    int BT, T, C, groups_per_cta;
    const bf16 *shift;      // nullptr or [B, C]
    const bf16 *maa;        // [5, C]
};

__global__ void __launch_bounds__(THREADS, 2)
ddlerp_lora_kernel(const __grid_constant__ CUtensorMap map_h, const __grid_constant__ CUtensorMap map_w2,
                   const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_o,
                   const __grid_constant__ CUtensorMap map_a, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *sm = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    Bars &bar = *reinterpret_cast<Bars *>(sm + OFF_BAR);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r0 = blockIdx.x * TM;
    const int g0 = blockIdx.y * p.groups_per_cta;
    const int ngroups = min(p.groups_per_cta, p.C / NC - g0);
    const int nitems = ngroups * NOUT;

    if (threadIdx.x == 0) {
        mbar_init(&bar.h, 1);
        for (int i = 0; i < 2; i++) {
            mbar_init(&bar.x_full[i], 1);
            mbar_init(&bar.x_free[i], EPI_THREADS);
            mbar_init(&bar.mma[i], 1);
            mbar_init(&bar.acc_free[i], EPI_THREADS);
        }
        for (int i = 0; i < 3; i++) mbar_init(&bar.w_full[i], 1);
        fence_barrier_init();
    }
    if (warp == 8) {
        tmem_alloc(&bar.tmem_base, TM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bar.tmem_base;
    const uint32_t sbase = smem_u32(sm);

    if (warp == 8) {
        // ------------------------------------------------------------------ issuer
        if (elect_one()) {
            tma_prefetch_desc(&map_h); tma_prefetch_desc(&map_w2); tma_prefetch_desc(&map_x); tma_prefetch_desc(&map_o);
            mbar_arrive_expect_tx(&bar.h, 3 * H_BOX);
            for (int j = 0; j < 3; j++) tma_load_3d(sm + OFF_H + j * H_BOX, &map_h, &bar.h, j * 64, r0, 0);
            auto load_x = [&](int gi) {          // group index inside this CTA
                const int s = gi & 1;
                mbar_arrive_expect_tx(&bar.x_full[s], (TM + 1 + NOUT) * 128);
                tma_load_3d(sm + OFF_X + s * X_BYTES, &map_x, &bar.x_full[s], (g0 + gi) * NC, r0 - 1, 0);
                // the group's 5 x 64 time_maa values ride along as rows 129..133 of the same swizzled tile
                tma_load_3d(sm + OFF_X + s * X_BYTES + (TM + 1) * 128, &map_a, &bar.x_full[s], (g0 + gi) * NC, 0, 0);
            };
            auto load_w = [&](int item) {
                const int s = item % 3, gi = item / NOUT, n = item % NOUT;
                mbar_arrive_expect_tx(&bar.w_full[s], W_BYTES);
                tma_load_3d(sm + OFF_W + s * W_BYTES, &map_w2, &bar.w_full[s], (g0 + gi) * NC, 0, n);
            };
            load_x(0);
            if (ngroups > 1) load_x(1);
            for (int i = 0; i < 3 && i < nitems; i++) load_w(i);
            mbar_wait(&bar.h, 0);
            const uint32_t idesc = idesc_bf16(TM, NC, 0, 1);
            for (int i = 0; i < nitems; i++) {
                const int n = i % NOUT, gi = i / NOUT, a = i & 1;
                mbar_wait(&bar.w_full[i % 3], (i / 3) & 1);
                if (i >= 2) mbar_wait(&bar.acc_free[a], ((i - 2) >> 1) & 1);      // epilogue of item i-2 has read the accumulator
                tc_fence_after();
                const uint32_t abase = sbase + OFF_H + (n >> 1) * H_BOX + (n & 1) * 64;
                const uint32_t bbase = sbase + OFF_W + (i % 3) * W_BYTES;
#pragma unroll
                for (int k = 0; k < RANK / 16; k++)
                    mma_bf16_ss(tmem + a * NC, smem_desc_sw128(abase + 32 * k, 8192, 1024),
                                smem_desc_sw128(bbase + 2048 * k, 8192, 1024), idesc, k > 0);
                mma_commit(&bar.mma[a]);
                // refill: the W2 slot of item i-1 is free once its MMA has completed; the x buffer of group
                // gi-1 once the epilogue has finished that group
                if (i >= 1 && i + 2 < nitems) {
                    mbar_wait(&bar.mma[(i - 1) & 1], ((i - 1) >> 1) & 1);
                    load_w(i + 2);
                }
                if (n == 0 && gi >= 1 && gi + 1 < ngroups) {
                    mbar_wait(&bar.x_free[(gi - 1) & 1], ((gi - 1) >> 1) & 1);
                    load_x(gi + 1);
                }
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------------ epilogue: row = token, 32 channels
        const int row = (warp & 3) * 32 + lane;               // TMEM lane == token row of the tile
        const int half = warp >> 2;                           // which 32 of the 64 channels
        const long long rg = (long long)r0 + row;             // flattened (b,t) row
        const bool rlive = rg < p.BT;
        const int t = rlive ? (int)(rg % p.T) : 1;
        const int b = rlive ? (int)(rg / p.T) : 0;
        // packed bf16 arithmetic: every op of the eager chain rounds to bf16, which is what HADD2 / HMUL2.BF16 do
        __nv_bfloat162 xxp[16];                               // xx = shift(x) - x of this thread's 32 channels (per group)
        for (int i = 0; i < nitems; i++) {
            const int n = i % NOUT, gi = i / NOUT, a = i & 1;
            const int c = (g0 + gi) * NC + half * 32;
            const uint8_t *xs = sm + OFF_X + (gi & 1) * X_BYTES;
            if (n == 0) {
                mbar_wait(&bar.x_full[gi & 1], (gi >> 1) & 1);
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const uint32_t byte = (half * 4 + q) * 16;
                    const uint4 xv = *reinterpret_cast<const uint4 *>(xs + sw128(row + 1, byte));
                    uint4 pv = *reinterpret_cast<const uint4 *>(xs + sw128(row, byte));
                    if (t == 0) {
                        if (p.shift) pv = *reinterpret_cast<const uint4 *>(p.shift + (size_t)b * p.C + c + q * 8);
                        else pv = make_uint4(0, 0, 0, 0);
                    }
                    const __nv_bfloat162 *x2 = reinterpret_cast<const __nv_bfloat162 *>(&xv);
                    const __nv_bfloat162 *p2 = reinterpret_cast<const __nv_bfloat162 *>(&pv);
#pragma unroll
                    for (int e = 0; e < 4; e++) xxp[q * 4 + e] = __hsub2_rn(p2[e], x2[e]);
                }
            }
            mbar_wait(&bar.mma[a], (i >> 1) & 1);
            tc_fence_after();
            uint32_t acc[32];
            tmem_ld32(tmem_addr(tmem, (warp & 3) * 32, a * NC + half * 32), acc);
            tmem_wait_ld();
            tc_fence_before();
            mbar_arrive(&bar.acc_free[a]);
            uint32_t outp[16];
#pragma unroll
            for (int q = 0; q < 4; q++) {                     // 4 chunks of 8 channels
                const uint4 xv = *reinterpret_cast<const uint4 *>(xs + sw128(row + 1, (half * 4 + q) * 16));
                const uint4 av = *reinterpret_cast<const uint4 *>(xs + sw128(TM + 1 + n, (half * 4 + q) * 16));
                const __nv_bfloat162 *x2 = reinterpret_cast<const __nv_bfloat162 *>(&xv);
                const __nv_bfloat162 *a2 = reinterpret_cast<const __nv_bfloat162 *>(&av);
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const __nv_bfloat162 m2 = __floats2bfloat162_rn(__uint_as_float(acc[q * 8 + 2 * e]), __uint_as_float(acc[q * 8 + 2 * e + 1]));
                    const __nv_bfloat162 o2 = __hadd2_rn(x2[e], __hmul2_rn(xxp[q * 4 + e], __hadd2_rn(a2[e], m2)));
                    outp[q * 4 + e] = *reinterpret_cast<const uint32_t *>(&o2);
                }
            }
            // staging buffer free?  (thread 0 issued the previous store)
            if (threadIdx.x == 0) tma_store_wait_read<0>();
            named_bar_sync<1, EPI_THREADS>();
#pragma unroll
            for (int q = 0; q < 4; q++)
                *reinterpret_cast<uint4 *>(sm + OFF_STG + sw128(row, (half * 4 + q) * 16)) =
                    make_uint4(outp[q * 4], outp[q * 4 + 1], outp[q * 4 + 2], outp[q * 4 + 3]);
            // The x buffer is released only after stores that consume every value read from it: the arrive does not wait
            // for loads still in flight, and an arrive ahead of them lets the refill of group gi+2 land under the reads
            // of this item.
            if (n == NOUT - 1) mbar_arrive(&bar.x_free[gi & 1]);
            fence_proxy_async();
            named_bar_sync<2, EPI_THREADS>();
            if (threadIdx.x == 0) {
                tma_store_3d(&map_o, sm + OFF_STG, (g0 + gi) * NC, r0, n);
                tma_store_commit();
            }
        }
        if (threadIdx.x == 0) tma_store_wait_all<0>();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

bool ddlerp_lora_supported(int B, int T, int C, int R) {
    return R == RANK && C % NC == 0 && (long long)B * T > 0 && (long long)B * T < (1ll << 31) - TM;
}

int ddlerp_lora_forward(int B, int T, int C, const void *x, const void *shift, const void *maa, const void *h,
                        const void *w2, void *out, cudaStream_t stream) {
    const long long BT = (long long)B * T;
    CUtensorMap mh, mw, mx, mo, ma;
    const auto dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    if (!make_btc_map(&mh, h, 1, (int)BT, NOUT * RANK, TM, dt, 2, 64) || !make_btc_map(&mw, w2, NOUT, RANK, C, RANK, dt, 2, 64) ||
        !make_btc_map(&mx, x, 1, (int)BT, C, TM + 1, dt, 2, 64) || !make_btc_map(&mo, out, NOUT, (int)BT, C, TM, dt, 2, 64) ||
        !make_btc_map(&ma, maa, 1, NOUT, C, NOUT, dt, 2, 64)) {
        set_error("ddlerp_lora: cuTensorMapEncodeTiled failed");
        return WKV6_ECUDA;
    }
    const int tiles = (int)((BT + TM - 1) / TM), groups = C / NC;
    // channel split: about four waves of CTAs (2 resident per SM), at least 2 groups per CTA
    int split = (148 * 2 * 4 + tiles - 1) / tiles;
    if (split > groups / 2) split = groups / 2;
    if (split < 1) split = 1;
    const int gpc = (groups + split - 1) / split;
    split = (groups + gpc - 1) / gpc;
    Params p;
    p.BT = (int)BT; p.T = T; p.C = C; p.groups_per_cta = gpc;
    p.shift = (const bf16 *)shift; p.maa = (const bf16 *)maa;
    static thread_local bool attr_done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !attr_done[dev]) {
        WKV6_CUDA_CHECK(cudaFuncSetAttribute(ddlerp_lora_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
    ddlerp_lora_kernel<<<dim3(tiles, split), THREADS, SMEM_BYTES, stream>>>(mh, mw, mx, mo, ma, p);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

}  // namespace wkv6

using namespace wkv6;

extern "C" int tmix_ddlerp_lora_bf16(int B, int T, int C, int R, const void *x, const void *shift_state, const void *maa,
                                     const void *h, const void *w2, void *out, void *stream) {
    if (B < 0 || T < 0 || C <= 0 || R <= 0) { set_error("tmix_ddlerp_lora_bf16: bad shape"); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    if (!x || !maa || !h || !w2 || !out) { set_error("tmix_ddlerp_lora_bf16: null pointer"); return WKV6_EINVAL; }
    if (!check_aligned16("tmix_ddlerp_lora_bf16", {{"x", x}, {"shift_state", shift_state}, {"maa", maa}, {"h", h}, {"w2", w2}, {"out", out}}))
        return WKV6_EINVAL;
    if (!ddlerp_lora_supported(B, T, C, R)) {
        set_error("tmix_ddlerp_lora_bf16: needs R == 32 and C %% 64 == 0 (use bmm + tmix_ddlerp_mix_bf16)");
        return WKV6_EUNSUPPORTED;
    }
    return ddlerp_lora_forward(B, T, C, x, shift_state, maa, h, w2, out, (cudaStream_t)stream);
}
