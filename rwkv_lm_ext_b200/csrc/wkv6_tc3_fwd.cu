// WKV6 forward, chunked, on tcgen05 tensor cores fed by TMA -- role-uniform, software-pipelined.
//
// One CTA owns one (batch, head) stream and walks its T tokens in chunks of L = 64; 2 CTAs per SM.
// Per chunk (SURVEY.md Appendix A; i = key channel, j = value channel, l_t = -exp(w_t), cum =
// inclusive prefix sum of l inside the chunk, exc = cum - l, Lam = cum at the chunk end), with FOUR
// 16-token blocks q (reference rho_q = exc at the block middle rounded to the INTEGER log2 grid).  The
// per-token log2-decay is floored at -13 (a factor 2^-13 is below bf16 resolution), so every scaled
// operand stays within 8 x 13 binary orders of 1: nothing overflows whatever the decays are, and no
// stream ever needs an exact fallback.  The versions of Kt are exact power-of-two multiples (<= 1) of
// one another -- bf16 mul.rn, no second exp:
//
//   A    A^T[s,t] = sum_i Kt_q[s,i] * Rt[t,i]        4 x (64 x 16 x 64), one per target block q
//         Rt[t] = r_t * 2^(exc_t - rho_q),   Kt_q[s] = k_s * 2^(rho_q - cum_s)   (s in blocks <= q)
//   T1   P = strict-lower(A) + diag(sum_i r u k)  (bf16),   S[i,j] *= 2^Lam_i  (fp32, in TMEM)
//   M2   Y[t,j]  = sum_i Rh[t,i] * S_in[i,j] + sum_s P[t,s] * V[s,j]          Rh = r * 2^exc
//        S[i,j] += sum_s Kh[s,i] * V[s,j]     Kh = k * 2^(Lam - cum), split into bf16 hi + lo so that the
//         fp32 master state keeps ~16 mantissa bits per update
//   T2   y tile -> TMA store;  bf16 copy of S for the next chunk (and, for training, TMA-stored as the
//         chunk-start checkpoint the backward kernel reads)
//
// 8 compute warps do EVERY stage in the fragment mapping of tc3_common.cuh (a thread keeps its two
// channels from the decay scan to the state rows it rescales); warp 8 issues TMA and tcgen05.mma.
// The operand preparation of chunk c+1 runs while the tensor cores work on M2 of chunk c (only the
// tiles M2 still reads -- Rh, Kh -- are written after it), and A of chunk c+1 is queued behind M2, so
// the compute warps never wait for a full MMA round trip; the co-resident CTA fills what is left.
// The per-stream flags only mark streams the CALLER routed to the exact SIMT kernels (fp32 decay
// entries whose values are not bf16 logits); this kernel never raises one.
#include "common.cuh"
#include "tc3_common.cuh"

namespace wkv6 {
namespace {

using namespace tc3;

constexpr uint32_t OFF_R = 0, OFF_K = 8192, OFF_W = 16384, OFF_V = 24576;
// Kt versions: version q holds rows s = 0 .. 16q+15 (reference rho_q); 64 + 48 + 32 + 16 rows, 1024-byte aligned
constexpr uint32_t OFF_KT = 32768;
__host__ __device__ constexpr uint32_t kt_ver(int q) { return q == 3 ? 0u : q == 2 ? 8192u : q == 1 ? 14336u : 18432u; }
constexpr uint32_t OFF_RT = 53248, OFF_P = 61440, OFF_RH = 69632, OFF_KH = 77824, OFF_KL = 86016, OFF_SB = 94208, OFF_YT = 102400;
constexpr uint32_t OFF_TILES_END = 110592;
struct Extra {
    float gtot[64][8];        // decay total of every 8-token group, per channel (log2 units): one 32-byte row per channel
    float pdu[4][64];         // per channel-quarter partial sums of r u k, per token
    uint64_t bar_rkw, bar_v, bar_a, bar_m2;
    uint32_t tmem_base;
};
constexpr uint32_t SMEM_BYTES = OFF_TILES_END + sizeof(Extra);
constexpr uint32_t TM_A = 0, TM_Y = 64, TM_S = 128, TM_COLS = 256;
// named barriers (288 threads): B_RAW raw r,k,w landed; B_PA Kt / Rt written; B_PB Rh / Kh written;
// B_A A^T done; B_T1 P written, S decayed; B_M2 Y and S done; B_T2 y tile and bf16 S written
enum : int { B_PA = B_PREP, B_PB = B_M3, B_A = B_M1 };

struct Params {
    int B, T, H;
    const bf16 *u;
    const void *s0;
    int s0_f32;
    long long s0_bstride;
    void *sT;
    int sT_f32;
    int has_y, has_ckpt;
    int *hz_flags;            // nullptr, or [rows*H]: 1 = this stream needs the exact route
    // time-axis segmentation (seg_scan.cu): the grid has B*nseg rows; row = b*nseg + seg covers tokens
    // [seg*seg_chunks*64, min(T, (seg+1)*seg_chunks*64)) of sequence b.  States (s0, sT), flags and the
    // checkpoints are indexed by row; nseg = 1 and seg_chunks = ceil(T/64) for an ordinary call.
    int nseg, seg_chunks;
    float lmin;               // floor of the per-token log2-decay (opt-in clamp; -inf = off)
    const int *row_len;       // BI modes: tokens of every batch row (p + 1 of wkv6_bi), device int [B]
    const int *row_order;     // BI modes: batch rows sorted by length, longest first (CTAs of long rows start first), device int [B]
};

// 9 warps x 2 CTAs = 5 warps on the fullest SM sub-partition (16384 registers): at most 96 per thread
// SEG = false is the ordinary call (one row per (b,h), the whole sequence): kept as its own instantiation so
// that the segment arithmetic costs it nothing (with run-time descriptors ptxas scheduled the forward 7 % slower)
// SO = true: a state-only pass known at compile time (the two extra passes of the segmented routes): no r tile,
// no Rt / Kt versions, no diag(u) term, no A / Y products -- about half of the operand preparation.
// BI: direction of the bidirectional op (tc3_common.cuh); BI_NONE for every other call.
// KLO: split Kh into bf16 hi + lo for the state update.  Needed where the fp32 state leaves the kernel (sT: infctx /
// inference / the segment passes): without it the final state drifts by 1.5e-3 rel-RMS over 64 chunks.  Where only y and
// the bf16 chunk-start states are produced it changes y by 1.4 % of its own bf16 error (3.25e-3 -> 3.29e-3 against the fp64
// recurrence at T = 4096, tests/tc_emulation.py) and costs 5 % of the forward: those calls run without it.
template <bool SEG, bool SO = false, int BI = BI_NONE, bool KLO = true>
__global__ void __launch_bounds__(NTHREADS, 2)
wkv6_tc3_fwd_kernel(const __grid_constant__ CUtensorMap map_r, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_w,
                    const __grid_constant__ CUtensorMap map_y, const __grid_constant__ CUtensorMap map_ck, Params p) {
    const int h = blockIdx.x % p.H;
    const int row = BI ? p.row_order[blockIdx.x / p.H] : blockIdx.x / p.H;
    const int rid = BI ? row * p.H + h : blockIdx.x;     // row id: flags, checkpoints
    if (p.hz_flags && p.hz_flags[rid] != 0) return; // flagged before launch (inexact logit conversion): exact route
    extern __shared__ __align__(1024) uint8_t sm[];
    Extra &ex = *reinterpret_cast<Extra *>(sm + OFF_TILES_END);
    if ((smem_u32(sm) & 1023u) != 0) __trap();
    const int b = SEG ? row / p.nseg : row;                                  // batch index inside the [B,T,C] tensors
    const int t_base = SEG ? (row % p.nseg) * p.seg_chunks * L : 0;          // first token of this row's segment
    const int T = BI ? p.row_len[b] : SEG ? min(p.T - t_base, p.seg_chunks * L) : p.T;   // tokens of the segment / row
    const int NC = (T + L - 1) / L;
    const int ck_stride = SEG ? p.seg_chunks : BI ? (p.T + L - 1) / L : NC;  // checkpoint slots per row
    // first token of chunk c's tile (BI_REV: the tile that ends at token T-1-64c, read backwards; see tc3_common.cuh)
    auto tok0 = [&](int c) { return BI == BI_REV ? max(T - (c + 1) * L, 0) : t_base + c * L; };
    Frag F;
    F.init();
    const int warp = F.warp, lane = F.lane;

    if (threadIdx.x == 0) {
        mbar_init(&ex.bar_rkw, 1);
        mbar_init(&ex.bar_v, 1);
        mbar_init(&ex.bar_a, 1);
        mbar_init(&ex.bar_m2, 1);
        fence_barrier_init();
    }
    if (warp == 0) {
        tmem_alloc(&ex.tmem_base, TM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = ex.tmem_base;
    const uint32_t sbase = smem_u32(sm);

    if (warp == CWARPS) {
        // =====================================================================================
        // issuer: TMA loads / stores and every tcgen05.mma (lane 0); all 32 lanes take part in the
        // named barriers
        // =====================================================================================
        auto issue_rkw = [&](int c) {
            mbar_arrive_expect_tx(&ex.bar_rkw, (SO ? 2 : 3) * 8192);
            if constexpr (!SO) tma_load_3d(sm + OFF_R, &map_r, &ex.bar_rkw, h * 64, tok0(c), b);
            tma_load_3d(sm + OFF_K, &map_k, &ex.bar_rkw, h * 64, tok0(c), b);
            tma_load_3d(sm + OFF_W, &map_w, &ex.bar_rkw, h * 64, tok0(c), b);
        };
        auto issue_v = [&](int c) {
            mbar_arrive_expect_tx(&ex.bar_v, 8192);
            tma_load_3d(sm + OFF_V, &map_v, &ex.bar_v, h * 64, tok0(c), b);
        };
        const uint32_t kt = sbase + OFF_KT, rt = sbase + OFF_RT, rh = sbase + OFF_RH, kh = sbase + OFF_KH;
        const uint32_t kl = sbase + OFF_KL, pp = sbase + OFF_P, sb = sbase + OFF_SB, vv = sbase + OFF_V;
        constexpr uint32_t ID16_KK = idesc_bf16(64, 16, 0, 0);
        constexpr uint32_t ID_KM = idesc_bf16(64, 64, 0, 1);
        constexpr uint32_t ID_MM = idesc_bf16(64, 64, 1, 1);
        auto issue_A = [&]() {                               // A^T[s, t in q] = Kt_q Rt_own^T   (not in a state-only pass)
            if (!SO && p.has_y)
#pragma unroll
            for (int qq = 0; qq < 4; qq++)                   // rows s past block qq are never read (strictly lower part only)
#pragma unroll
                for (int k = 0; k < 4; k++)
                    mma_bf16_ss(tmem + TM_A + 16 * qq, smem_desc_sw128(kt + kt_ver(qq) + 32 * k, 8192, 1024),
                                smem_desc_sw128(rt + 2048 * qq + 32 * k, 8192, 1024), ID16_KK, k > 0);
            mma_commit(&ex.bar_a);
        };
        if (lane == 0) {
            tma_prefetch_desc(&map_r);
            tma_prefetch_desc(&map_k);
            tma_prefetch_desc(&map_v);
            tma_prefetch_desc(&map_w);
            issue_rkw(0);
            issue_v(0);
            mbar_wait(&ex.bar_rkw, 0);
        }
        __syncwarp();
        bar_arrive_all<B_RAW>();
        bar_sync_all<B_PA>();
        if (elect_one()) {
            tc_fence_after();
            issue_A();
            if (NC > 1) issue_rkw(1);
        }
        __syncwarp();
        bar_sync_all<B_PB>();
        bar_sync_all<B_T2>();                                    // initial state in TMEM / shared
        if (lane == 0) {
            if (p.has_ckpt) tma_store_3d(&map_ck, sm + OFF_SB, 0, (rid * ck_stride) * 64, 0);
            tma_store_commit();
        }
        if (lane == 0) mbar_wait(&ex.bar_a, 0);
        __syncwarp();
        bar_arrive_all<B_A>();
        for (int c = 0; c < NC; c++) {
            const uint32_t par = c & 1;
            const bool more = c + 1 < NC;
            if (more) {
                if (lane == 0) mbar_wait(&ex.bar_rkw, par ^ 1);
                __syncwarp();
                bar_arrive_all<B_RAW>();
            }
            bar_sync_all<B_T1>();                                // P written, S decayed
            if (elect_one()) {
                tc_fence_after();
                if (!SO && p.has_y)
#pragma unroll
                for (int k = 0; k < 4; k++)                      // Y = Rh * S_in      (S tile is [i][j]: MN-major B)
                    mma_bf16_ss(tmem + TM_Y, smem_desc_sw128(rh + 32 * k, 8192, 1024),
                                smem_desc_sw128(sb + 2048 * k, 8192, 1024), ID_KM, k > 0);
                mbar_wait(&ex.bar_v, par);
                if (!SO && p.has_y)
#pragma unroll
                for (int k = 0; k < 4; k++)                      // Y += P * V
                    mma_bf16_ss(tmem + TM_Y, smem_desc_sw128(pp + 32 * k, 8192, 1024),
                                smem_desc_sw128(vv + 2048 * k, 8192, 1024), ID_KM, 1);
#pragma unroll
                for (int k = 0; k < 4; k++)                      // S[i,j] += Kh^T V  (hi, then lo)
                    mma_bf16_ss(tmem + TM_S, smem_desc_sw128(kh + 2048 * k, 8192, 1024),
                                smem_desc_sw128(vv + 2048 * k, 8192, 1024), ID_MM, 1);
                if constexpr (KLO)
#pragma unroll
                for (int k = 0; k < 4; k++)
                    mma_bf16_ss(tmem + TM_S, smem_desc_sw128(kl + 2048 * k, 8192, 1024),
                                smem_desc_sw128(vv + 2048 * k, 8192, 1024), ID_MM, 1);
                mma_commit(&ex.bar_m2);
            }
            __syncwarp();
            if (more) {
                bar_sync_all<B_PA>();                            // Kt / Rt of chunk c+1 written, its raw tiles consumed
                if (lane == 0 && c + 2 < NC) issue_rkw(c + 2);
            }
            // M2 ran under the preparation of chunk c+1: release the compute warps (deferred stores, T2) BEFORE spending
            // a few hundred cycles on issuing A of chunk c+1 -- they wait for nothing else at this point
            if (lane == 0) {
                mbar_wait(&ex.bar_m2, par);
                tma_store_wait_read<0>();                        // SB / YT of the previous stores may be rewritten now
            }
            __syncwarp();
            bar_arrive_all<B_M2>();
            if (lane == 0 && more) issue_v(c + 1);               // V is free again
            if (more) {
                if (elect_one()) {
                    tc_fence_after();
                    issue_A();                                   // reads only Kt / Rt, writes only the A columns T1 has consumed
                }
                __syncwarp();
            }
            if (more) {
                bar_sync_all<B_PB>();
                if (lane == 0) mbar_wait(&ex.bar_a, par ^ 1);    // A^T of chunk c+1 ran right behind M2
                __syncwarp();
                bar_arrive_all<B_A>();
            }
            bar_sync_all<B_T2>();                                // y tile and the new bf16 S written
            if (lane == 0) {
                if (!SO && p.has_y) {
                    if (BI == BI_REV) tma_reduce_add_3d(&map_y, sm + OFF_YT, h * 64, tok0(c), b);
                    else tma_store_3d(&map_y, sm + OFF_YT, h * 64, tok0(c), b);
                }
                if (more && p.has_ckpt) tma_store_3d(&map_ck, sm + OFF_SB, 0, (rid * ck_stride + c + 1) * 64, 0);
                tma_store_commit();
            }
        }
        if (BI == BI_CAUSAL && !SO && p.has_y && NC * L < p.T) {      // y = 0 behind the row's last chunk
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 16; k++) *reinterpret_cast<uint4 *>(sm + OFF_YT + (lane + 32 * k) * 16) = make_uint4(0, 0, 0, 0);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                for (int c = NC; c * L < p.T; c++) tma_store_3d(&map_y, sm + OFF_YT, h * 64, c * L, b);
                tma_store_commit();
            }
        }
        if (lane == 0) tma_store_wait_read<0>();          // shared memory has been read; the writes complete with the grid
    } else {
        // =====================================================================================
        // compute warps
        // =====================================================================================
        const int sp = F.sp, ch = F.ch, q = F.q;
        const float u_h[2] = {__bfloat162float(p.u[h * 64 + F.row(0)]), __bfloat162float(p.u[h * 64 + F.row(1)])};
        // the warp's TMEM window (sub-partition sp, column half ch), kept in a register: re-derived from SR_TID in front of
        // every TMEM access it cost an S2R round trip + 6 instructions at the start of each stage
        uint32_t twin = tmem_addr(tmem, 32 * sp, 32 * ch);
        asm volatile("" : "+r"(twin));
        const uint32_t tS = twin + TM_S;
        int dcol = (32 * ch + 2 * q) - (16 * sp + F.ri);           // column(g, e = 0) - row(hh) at g = hh
        asm volatile("" : "+r"(dcol));
        // where the warp's part of a 64 x 64 (row, column) tile lies: 1 = entirely above the diagonal (column > row), 2 =
        // entirely below it, 0 = the diagonal runs through it
        const int tri = 32 * ch - 16 * sp - 15 > 0 ? 1 : 32 * ch + 31 - 16 * sp < 0 ? 2 : 0;
        uint32_t v[16];

        // ---- initial state -> TMEM (fp32 master, [i][j]) and shared (bf16 operand copy)
#pragma unroll
        for (int g = 0; g < 4; g++)
#pragma unroll
            for (int hh = 0; hh < 2; hh++)
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    float x = 0.f;
                    if (p.s0) {   // caller layout [.,H,64(value j),64(key i)]
                        const size_t idx = (size_t)row * p.s0_bstride + ((size_t)h * 64 + F.col(g, e)) * 64 + F.row(hh);
                        x = p.s0_f32 ? ((const float *)p.s0)[idx] : __bfloat162float(((const bf16 *)p.s0)[idx]);
                    }
                    v[4 * g + 2 * hh + e] = __float_as_uint(x);
                }
        tmem_st_frag(tS, v);
#pragma unroll
        for (int hh = 0; hh < 2; hh++)
            stsm_x4(sbase + OFF_SB + F.rc(hh), pack2(__uint_as_float(v[0 + 2 * hh]), __uint_as_float(v[1 + 2 * hh])),
                    pack2(__uint_as_float(v[4 + 2 * hh]), __uint_as_float(v[5 + 2 * hh])),
                    pack2(__uint_as_float(v[8 + 2 * hh]), __uint_as_float(v[9 + 2 * hh])),
                    pack2(__uint_as_float(v[12 + 2 * hh]), __uint_as_float(v[13 + 2 * hh])));
        tmem_wait_st();
        fence_proxy_async();
        tc_fence_before();
        bar_arrive_all<B_T2>();

        // Operand preparation of chunk c: Kt (both versions) and Rt go to shared memory at once; Rh, Kh (hi,
        // lo) and 2^Lam stay in registers until the MMAs of the previous chunk no longer read those tiles.
        uint32_t rhp[2][4], khp[2][4], klp[KLO ? 2 : 1][4];
        float elam_nx[2];
        // Token groups of the operand preparation: thread (ch, lane) owns the 8-token groups 2g + ch, g = 0..3, i.e.
        // ONE group of each 16-token reference block (block g = groups 2g and 2g + 1).  With the natural mapping
        // (groups 4ch + g) the warps of ch = 0 would scale and store ten Kt group-versions and those of ch = 1 three.
        // ldmatrix / stmatrix take one row address per lane, so any group assignment costs the same there.
        const uint32_t tg_off = sw128(16 * (lane >> 3) + 8 * ch + (lane & 7), 32 * sp);    // .x4: matrix m = group 2m + ch
        const uint32_t tg1_off = sw128(8 * ch + (lane & 7), 32 * sp);                       // .x1 of group 2m + ch: + 2048 m
        auto tg = [&](int hh) { return tg_off ^ (hh ? 16u : 0u); };
        auto prepare = [&](int c) {
            const int nv = min(L, T - c * L);
            // where the RAW r, k, w tiles are read: the same rows, or (BI_REV) row (nv - 1 - x) mod 64
            const uint32_t tgr_off = BI == BI_REV ? flip_rows(tg_off, nv - 1) : tg_off;
            auto tgr = [&](int hh) { return tgr_off ^ (hh ? 16u : 0u); };
            float l[2][4][2], exq[2][4];
            {
                uint32_t wp[2][4];
                ldsm_x4_t(sbase + OFF_W + tgr(0), wp[0][0], wp[0][1], wp[0][2], wp[0][3]);
                ldsm_x4_t(sbase + OFF_W + tgr(1), wp[1][0], wp[1][1], wp[1][2], wp[1][3]);
#pragma unroll
                for (int hh = 0; hh < 2; hh++)
#pragma unroll
                    for (int g = 0; g < 4; g++) {
                        float l0 = -fast_ex2(fmaf(bf_lo(wp[hh][g]), LOG2E, LOG2_LOG2E));   // -exp(w) * log2(e)
                        float l1 = -fast_ex2(fmaf(bf_hi(wp[hh][g]), LOG2E, LOG2_LOG2E));
                        l0 = fmaxf(l0, p.lmin);
                        l1 = fmaxf(l1, p.lmin);
                        if (nv < L) {                                   // ragged last chunk: no decay on the padded rows
                            const int t0 = 8 * (2 * g + ch) + 2 * q;
                            if (t0 >= nv) l0 = 0.f;
                            if (t0 + 1 >= nv) l1 = 0.f;
                        }
                        l[hh][g][0] = l0;
                        l[hh][g][1] = l1;
                        const float ps = l0 + l1;
                        float x = ps, y;
                        y = __shfl_up_sync(0xffffffffu, x, 1, 4);
                        if (q >= 1) x += y;
                        y = __shfl_up_sync(0xffffffffu, x, 2, 4);
                        if (q >= 2) x += y;
                        exq[hh][g] = x - ps;
                        if (q == 3) ex.gtot[F.row(hh)][2 * g + ch] = x;
                    }
            }
            named_bar_sync<B_SCAN, CTHREADS>();

            uint32_t rr[2][4] = {}, kk[2][4];
            if constexpr (!SO) {
                ldsm_x4_t(sbase + OFF_R + tgr(0), rr[0][0], rr[0][1], rr[0][2], rr[0][3]);
                ldsm_x4_t(sbase + OFF_R + tgr(1), rr[1][0], rr[1][1], rr[1][2], rr[1][3]);
            }
            ldsm_x4_t(sbase + OFF_K + tgr(0), kk[0][0], kk[0][1], kk[0][2], kk[0][3]);
            ldsm_x4_t(sbase + OFF_K + tgr(1), kk[1][0], kk[1][1], kk[1][2], kk[1][3]);
            if (BI && nv < L) {              // what lies behind the chunk's nv tokens is real data here, not TMA's zero fill
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    const uint32_t m = pair_mask(8 * (2 * g + ch) + 2 * q, nv);
                    rr[0][g] &= m; rr[1][g] &= m;
                    kk[0][g] &= m; kk[1][g] &= m;
                }
            }
            f2 du2[4];
#pragma unroll
            for (int g = 0; g < 4; g++) du2[g] = 0ull;
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                // prefix over the 8 groups of this channel: start of my groups, the four block references, total
                float run = 0.f, gb[4];
                int ir[4];
                const float4 gt0 = *reinterpret_cast<const float4 *>(&ex.gtot[F.row(hh)][0]), gt1 = *reinterpret_cast<const float4 *>(&ex.gtot[F.row(hh)][4]);
                const float gt[8] = {gt0.x, gt0.y, gt0.z, gt0.w, gt1.x, gt1.y, gt1.z, gt1.w};
#pragma unroll
                for (int x8 = 0; x8 < 8; x8++) {
                    if (x8 & 1) ir[x8 >> 1] = __float2int_rn(run);        // middle of block x8/2, integer log2 grid
                    if ((x8 & 1) == ch) gb[x8 >> 1] = run;
                    run += gt[x8];
                }
                const float lam = run;
                elam_nx[hh] = fast_ex2(lam);
                uint32_t rto[4], kto[4];
                const f2 uu = f2bcast(u_h[hh]);
#pragma unroll
                for (int g = 0; g < 4; g++) {                             // my group g lies in block g
                    const float rq = (float)ir[g];
                    const f2 el = f2bcast(fast_ex2(lam - rq));
                    // a0 = exc_0 - rho, a1 = cum_0 - rho = exc_1 - rho, a2 = cum_1 - rho
                    const float a0 = (gb[g] - rq) + exq[hh][g], a1 = a0 + l[hh][g][0], a2 = a1 + l[hh][g][1];
                    const f2 k2 = bf2f2(kk[hh][g]);
                    const f2 kf = f2mul(k2, f2pack(fast_ex2(-a1), fast_ex2(-a2)));
                    if constexpr (!SO) {
                        const f2 r2 = bf2f2(rr[hh][g]);
                        rto[g] = f2tobf(f2mul(r2, f2pack(fast_ex2(a0), fast_ex2(a1))));
                        kto[g] = f2tobf(kf);
                        rhp[hh][g] = hmul2(rto[g], bfpow2pair(ir[g]));    // Rh = Rt * 2^rho (exact)
                        du2[g] = f2fma(f2mul(r2, uu), k2, du2[g]);
                    }
                    const f2 kh = f2mul(kf, el);                          // Kh = k * 2^(Lam - cum)
                    khp[hh][g] = f2tobf(kh);
                    if constexpr (KLO) klp[hh][g] = f2tobf(f2sub(kh, bf2f2(khp[hh][g])));
                }
                if constexpr (!SO) {
                const uint32_t ti = tg(hh), t1 = tg1_off ^ (hh ? 16u : 0u);
                stsm_x4_t(sbase + OFF_RT + ti, rto[0], rto[1], rto[2], rto[3]);
                // Kt versions: version q holds the groups of blocks <= q in the reference of block q.  My group g
                // enters version g as it is and is then scaled down (exactly, by powers of two <= 1) for every later
                // version.  2^(rho_q - rho_(q-1)) spans 16 tokens and may leave the bf16 range although the products
                // it is meant for do not: two exact factors.
                stsm_x1_t(sbase + OFF_KT + kt_ver(0) + t1, kto[0]);
                scale1(kto[0], ir[1] - ir[0]);
                stsm_x2_t(sbase + OFF_KT + kt_ver(1) + ti, kto[0], kto[1]);
                scale2(kto[0], kto[1], ir[2] - ir[1]);
                stsm_x2_t(sbase + OFF_KT + kt_ver(2) + ti, kto[0], kto[1]);
                stsm_x1_t(sbase + OFF_KT + kt_ver(2) + t1 + 4096u, kto[2]);
                scale2(kto[0], kto[1], ir[3] - ir[2]);
                scale1(kto[2], ir[3] - ir[2]);
                stsm_x4_t(sbase + OFF_KT + kt_ver(3) + ti, kto[0], kto[1], kto[2], kto[3]);
                }
            }
            // ---- diag(u) term: sum over channels of r u k per token; reduce-scatter over the 8 lanes ri
            if constexpr (!SO) {
                const bool b2 = lane & 16, b1 = lane & 8, b0 = lane & 4;
                float du[4][2];
#pragma unroll
                for (int g = 0; g < 4; g++) f2unpack(du2[g], du[g][0], du[g][1]);
                float a4[2][2], a2[2], a1;
#pragma unroll
                for (int gg = 0; gg < 2; gg++)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const float keep = b2 ? du[2 + gg][e] : du[gg][e], send = b2 ? du[gg][e] : du[2 + gg][e];
                        a4[gg][e] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
                    }
#pragma unroll
                for (int e = 0; e < 2; e++) {
                    const float keep = b1 ? a4[1][e] : a4[0][e], send = b1 ? a4[0][e] : a4[1][e];
                    a2[e] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
                }
                {
                    const float keep = b0 ? a2[1] : a2[0], send = b0 ? a2[0] : a2[1];
                    a1 = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                }
                // the partial of my group gsel = (b2 ? 2 : 0) + (b1 ? 1 : 0), token 8 (2 gsel + ch) + 2q + e
                ex.pdu[sp][8 * (2 * ((b2 ? 2 : 0) + (b1 ? 1 : 0)) + ch) + 2 * q + (b0 ? 1 : 0)] = a1;
            }
            fence_proxy_async();
            bar_arrive_all<B_PA>();
        };
        auto store_deferred = [&]() {
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                const uint32_t ti = tg(hh);
                if constexpr (!SO) stsm_x4_t(sbase + OFF_RH + ti, rhp[hh][0], rhp[hh][1], rhp[hh][2], rhp[hh][3]);
                stsm_x4_t(sbase + OFF_KH + ti, khp[hh][0], khp[hh][1], khp[hh][2], khp[hh][3]);
                if constexpr (KLO) stsm_x4_t(sbase + OFF_KL + ti, klp[hh][0], klp[hh][1], klp[hh][2], klp[hh][3]);
            }
            fence_proxy_async();
            bar_arrive_all<B_PB>();
        };

        bar_sync_all<B_RAW>();
        prepare(0);
        store_deferred();
        float elam[2] = {elam_nx[0], elam_nx[1]};

        for (int c = 0; c < NC; c++) {
            const bool more = c + 1 < NC;
            // ================================================================== T1: A^T -> P, decay S
            bar_sync_all<B_A>();
            tc_fence_after();
            if (!SO && p.has_y) {
            // The warp's 16 x 32 part of A^T (rows s = 16sp.., columns t = 32ch..) lies entirely above the diagonal for
            // (sp 0,1; ch 1): kept as it is; entirely below for (sp 2,3; ch 0): zeros, no TMEM load; the other four warps mask
            if (tri == 2) {
#pragma unroll
                for (int hh = 0; hh < 2; hh++) stsm_x4_t(sbase + OFF_P + F.ti(hh), 0u, 0u, 0u, 0u);
            } else {
            tmem_ld_frag(twin + TM_A, v);
            tmem_wait_ld();
            // branch-free: dcol = (t of e = 0) - s at g = hh; 8 more per column group
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                uint32_t pk[4];
                if (tri == 1) {
#pragma unroll
                    for (int g = 0; g < 4; g++) pk[g] = pack2(__uint_as_float(v[4 * g + 2 * hh]), __uint_as_float(v[4 * g + 2 * hh + 1]));
                } else {
                const int sr = F.row(hh);
                const float dg = (ex.pdu[0][sr] + ex.pdu[1][sr]) + (ex.pdu[2][sr] + ex.pdu[3][sr]);
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    const int d = dcol + 8 * (g - hh);                    // (t - s) for e = 0
                    const float a0 = __uint_as_float(v[4 * g + 2 * hh]), a1 = __uint_as_float(v[4 * g + 2 * hh + 1]);
                    pk[g] = pack2(d > 0 ? a0 : (d == 0 ? dg : 0.f), d > -1 ? a1 : (d == -1 ? dg : 0.f));
                }
                }
                stsm_x4_t(sbase + OFF_P + F.ti(hh), pk[0], pk[1], pk[2], pk[3]);       // P[t][s]
            }
            }
            }
            if (c == 0) {              // S *= 2^Lam of the first chunk (every later chunk: T2 of the chunk before it, below)
            tmem_ld_frag(tS, v);
            tmem_wait_ld();
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                const f2 el2 = f2bcast(elam[hh]);
#pragma unroll
                for (int g = 0; g < 4; g++)
                    f2unpacku(f2mul(f2packu(v[4 * g + 2 * hh], v[4 * g + 2 * hh + 1]), el2), v[4 * g + 2 * hh], v[4 * g + 2 * hh + 1]);
            }
            tmem_st_frag(tS, v);
            }
            if (BI == BI_REV) {        // the V tile goes to the tensor cores as it lies in shared memory: reverse its rows
                mbar_wait(&ex.bar_v, c & 1);                            // (issued a whole chunk ago: landed long since)
                const int nvc = min(L, T - c * L);
                const uint32_t vt[1] = {sbase + OFF_V};
                if (nvc == L) flip_tiles_full(vt, warp, lane);
                else flip_tiles_short(vt, nvc, warp, lane);
            }
            tmem_wait_st();
            fence_proxy_async();
            tc_fence_before();
            bar_arrive_all<B_T1>();

            // ================================================================== P of the next chunk, under M2
            if (more) {
                bar_sync_all<B_RAW>();
                prepare(c + 1);
            }
            bar_sync_all<B_M2>();
            tc_fence_after();
            if (more) {
                store_deferred();
                elam[0] = elam_nx[0];
                elam[1] = elam_nx[1];
            }
            // ================================================================== T2: y tile, new bf16 S
            if (!SO && p.has_y) {
                tmem_ld_frag(twin + TM_Y, v);
                tmem_wait_ld();
#pragma unroll
                for (int hh = 0; hh < 2; hh++)
                    stsm_x4(sbase + OFF_YT + (BI == BI_REV ? flip_rows(F.rc(hh), min(L, T - c * L) - 1) : F.rc(hh)), pack2(__uint_as_float(v[0 + 2 * hh]), __uint_as_float(v[1 + 2 * hh])),
                            pack2(__uint_as_float(v[4 + 2 * hh]), __uint_as_float(v[5 + 2 * hh])),
                            pack2(__uint_as_float(v[8 + 2 * hh]), __uint_as_float(v[9 + 2 * hh])),
                            pack2(__uint_as_float(v[12 + 2 * hh]), __uint_as_float(v[13 + 2 * hh])));
            }
            tmem_ld_frag(tS, v);
            tmem_wait_ld();
#pragma unroll
            for (int hh = 0; hh < 2; hh++)
                stsm_x4(sbase + OFF_SB + F.rc(hh), pack2(__uint_as_float(v[0 + 2 * hh]), __uint_as_float(v[1 + 2 * hh])),
                        pack2(__uint_as_float(v[4 + 2 * hh]), __uint_as_float(v[5 + 2 * hh])),
                        pack2(__uint_as_float(v[8 + 2 * hh]), __uint_as_float(v[9 + 2 * hh])),
                        pack2(__uint_as_float(v[12 + 2 * hh]), __uint_as_float(v[13 + 2 * hh])));
            if (c == NC - 1 && p.sT) {
#pragma unroll
                for (int g = 0; g < 4; g++)
#pragma unroll
                    for (int hh = 0; hh < 2; hh++)
#pragma unroll
                        for (int e = 0; e < 2; e++) {
                            const size_t idx = (((size_t)row * p.H + h) * 64 + F.col(g, e)) * 64 + F.row(hh);
                            const float x = __uint_as_float(v[4 * g + 2 * hh + e]);
                            if (p.sT_f32) ((float *)p.sT)[idx] = x;
                            else ((bf16 *)p.sT)[idx] = __float2bfloat16_rn(x);
                        }
            }
            if (more) {                // the state is in registers anyway: decay it for the next chunk here (elam is already
#pragma unroll                 // the next chunk's), so T1 no longer loads, scales and stores it
                for (int hh = 0; hh < 2; hh++) {
                    const f2 el2 = f2bcast(elam[hh]);
#pragma unroll
                    for (int g = 0; g < 4; g++)
                        f2unpacku(f2mul(f2packu(v[4 * g + 2 * hh], v[4 * g + 2 * hh + 1]), el2), v[4 * g + 2 * hh], v[4 * g + 2 * hh + 1]);
                }
                tmem_st_frag(tS, v);
                tmem_wait_st();
            }
            fence_proxy_async();
            tc_fence_before();
            bar_arrive_all<B_T2>();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

bool tc3_forward_supported(const Args &a) {
    return a.io_dtype == WKV6_BF16 && a.w_kind == W_RAW_BF16 && a.mask == nullptr && a.T >= 1 &&
           tc::get_encode_fn() != nullptr;
}

// ckpt: nullptr or bf16 [B*H][ceil(T/64)][64 i][64 j] receiving the state at the start of every chunk;
// hz_flags: nullptr or device int [B*H] (see common.cuh); a.y may be nullptr (state-only pass).
// bi / row_len: direction of the bidirectional op (tc3_common.cuh) and the device int [B] row lengths it needs.
template <bool SEG, bool SO, int BI, bool KLO>
static int launch_fwd(dim3 grid, cudaStream_t stream, const CUtensorMap &mr, const CUtensorMap &mk, const CUtensorMap &mv,
                      const CUtensorMap &mw, const CUtensorMap &my, const CUtensorMap &mc, const Params &p) {
    static bool attr_done[64] = {};          // function attributes are per device (and per instantiation)
    int dev = 0;
    WKV6_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_done[dev]) {
        WKV6_CUDA_CHECK(cudaFuncSetAttribute(wkv6_tc3_fwd_kernel<SEG, SO, BI, KLO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        WKV6_CUDA_CHECK(cudaFuncSetAttribute(wkv6_tc3_fwd_kernel<SEG, SO, BI, KLO>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                             cudaSharedmemCarveoutMaxShared));
        if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
    wkv6_tc3_fwd_kernel<SEG, SO, BI, KLO><<<grid, NTHREADS, SMEM_BYTES, stream>>>(mr, mk, mv, mw, my, mc, p);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

int tc3_forward(const Args &a, void *ckpt, int *hz_flags, int nseg, int seg_chunks, int bi, const int *row_len,
                const int *row_order) {
    if (a.B * a.H == 0 || a.T == 0) return WKV6_OK;
    const int C = a.H * 64;
    if (nseg <= 1) { nseg = 1; seg_chunks = (a.T + L - 1) / L; }
    if (bi != BI_NONE && (nseg > 1 || !row_len || !row_order)) { set_error("bidirectional pass: one segment and row lengths required"); return WKV6_EINVAL; }
    const size_t NC = (size_t)nseg * seg_chunks;                 // checkpoint slots per (b,h)
    CUtensorMap mr, mk, mv, mw, my, mc;
    const auto dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const void *yy = a.y ? a.y : a.r, *cc = ckpt ? ckpt : a.r;    // unused maps still have to encode
    const int ck_rows = ckpt ? (int)((size_t)a.B * a.H * NC * 64) : 64, ck_cols = ckpt ? 64 : C;
    if (!tc::make_btc_map(&mr, a.r, a.B, a.T, C, L, dt, 2, 64) || !tc::make_btc_map(&mk, a.k, a.B, a.T, C, L, dt, 2, 64) ||
        !tc::make_btc_map(&mv, a.v, a.B, a.T, C, L, dt, 2, 64) || !tc::make_btc_map(&mw, a.w, a.B, a.T, C, L, dt, 2, 64) ||
        !tc::make_btc_map(&my, yy, a.B, a.T, C, L, dt, 2, 64) || !tc::make_btc_map(&mc, cc, 1, ck_rows, ck_cols, 64, dt, 2, 64)) {
        set_error("cuTensorMapEncodeTiled failed (pointers must be 16-byte aligned)");
        return WKV6_ECUDA;
    }
    Params p;
    p.B = a.B; p.T = a.T; p.H = a.H;
    p.u = (const bf16 *)a.u;
    p.s0 = a.s0; p.s0_f32 = a.s0_f32; p.s0_bstride = a.s0_bstride;
    p.sT = a.sT; p.sT_f32 = a.sT_f32;
    p.has_y = a.y != nullptr;
    p.has_ckpt = ckpt != nullptr;
    p.hz_flags = hz_flags;
    p.nseg = nseg; p.seg_chunks = seg_chunks;
    p.lmin = tc_lmin_log2(a);
    p.row_len = row_len; p.row_order = row_order;
    const dim3 grid(a.B * nseg * a.H);
    const bool so = !p.has_y;
    // the fp32 state leaves the kernel: keep the hi + lo split of Kh.  (A state-only pass that only recomputes the bf16
    // chunk-start states -- the backward without a training pair -- runs without it, like the forward whose states it
    // reproduces bit for bit.)
    const bool klo = a.hi_lo >= 0 ? a.hi_lo != 0 : a.sT != nullptr;
#define FWD(SEG_, BI_) (so ? (klo ? launch_fwd<SEG_, true, BI_, true>(grid, a.stream, mr, mk, mv, mw, my, mc, p) \
                                  : launch_fwd<SEG_, true, BI_, false>(grid, a.stream, mr, mk, mv, mw, my, mc, p)) \
                        : (klo ? launch_fwd<SEG_, false, BI_, true>(grid, a.stream, mr, mk, mv, mw, my, mc, p) \
                               : launch_fwd<SEG_, false, BI_, false>(grid, a.stream, mr, mk, mv, mw, my, mc, p)))
    if (bi == BI_CAUSAL) return FWD(false, BI_CAUSAL);
    if (bi == BI_REV) return FWD(false, BI_REV);
    if (nseg > 1) return FWD(true, BI_NONE);
    return FWD(false, BI_NONE);
#undef FWD
}

}  // namespace wkv6
