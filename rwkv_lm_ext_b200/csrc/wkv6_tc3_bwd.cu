// WKV6 backward, chunked, on tcgen05 tensor cores fed by TMA -- role-uniform version (reverse sweep
// over 64-token chunks; 2 CTAs per SM; thread <-> data mapping of tc3_common.cuh).
//
// Notation as in wkv6_tc3_fwd.cu, with FOUR 16-token blocks per chunk (block b = tokens 16b..16b+15,
// reference rho_b = exc at the block middle on the integer log2 grid; the per-token log2-decay is floored
// at -13, so every scaled operand stays within 8 x 13 binary orders of 1 and no stream needs an exact
// fallback).  Inputs per chunk: r,k,v,w,gy tiles, S_in = bf16 state at the chunk start ([i][j], saved by
// the forward), G = dL/dS at the chunk end, fp32 in TMEM as [key i][value j].
//
//   E = 2^(exc - rho_b(t)), F = 2^(rho_b(s) - cum);  Rt = r E, Kt_own = k F  (bf16)
//   Kt_q[s] = Kt_own[s] 2^(rho_q - rho_b(s)), q >= b(s);   Rp_p[t] = Rt[t] 2^(rho_b(t) - rho_p), p <= b(t)
//       exact power-of-two multiples (<= 1): every pair product r k 2^(exc_t - cum_s) has ONE bf16 value
//
//   M1  Bm[t,s]  = gy_t . v_s                               -> dA = strict-lower(Bm), bd[t] = Bm[t,t]
//       A^T[s,t] = sum_i Kt_q[s,i] Rt[t,i]   (q = b(t))      -> P^T = strict-upper + diag(sum_i r u k)
//       Drs[i,t] = sum_j S_in[i,j] gy_t[j]
//   T1  dA, P^T tiles (bf16);  q0_i = <S_in, G>_i;  Gb = bf16(G 2^(Lam - rho_3));  G <- G 2^(Lam - rho_0)
//   M2  gv[s,j]  = sum_t P^T[s,t] gy_t[j] + sum_i Kt_3[s,i] Gb[i,j]       (Kt_3 2^(Lam - rho_3) = k 2^(Lam - cum))
//       Dr[i,t]  = sum_{s<t} Kt_q[s,i] dA[t,s]              (q = b(t))
//       G[i,j]  += sum_t Rp_0[t,i] gy_t[j]                  (G is carried as G_true 2^(-rho_0): Rp_0 2^rho_0 = r 2^exc)
//   T2  Z = Dr + 2^rho_q Drs;   gr_t[i] = E Z + u_i k_t[i] bd[t];   XA = Rt Z        (XA parked in TMEM)
//   M3  Dk[i,s]  = sum_{t>s} Rp_p[t,i] dA[t,s]  (p = b(s));   Dks[i,s] = sum_j Gb[i,j] v_s[j]
//   T3  Zk = Dk + 2^(rho_3 - rho_p) Dks;   gk_s[i] = F Zk + u_i r_s[i] bd[s];
//       X = XA - Kt_own Dk,  D = Kt_own Zk - XA
//       gl_t[i] = 2^Lam_i q0_i + sum_all X + sum_{s<t} D_s - XA_t,   gw = l * gl
//       This is d_t <S_t, G_t>_i (SURVEY.md Appendix A) expanded so that no two large quantities are
//       subtracted: the intra-chunk pair terms Rt Dr and Kt_own Dk are sums of bit-identical pair products
//       r k dA, so their difference telescopes like the reference's fp32 suffix trick
//       (cuda/wkv6_cuda.cu:161-227).
//   gr, gk, gw, gv leave through swizzled tiles + TMA stores.
//
// What the output stages need per element (Rt, Kt_own, E, F as bf16, the raw r, k, and l) is parked by the
// operand preparation in the unused half of TMEM (see PARK_* below) instead of being recomputed.
//
// The per-stream flags only mark streams the CALLER routed to the exact SIMT kernels (fp32 decay entries
// whose values are not bf16 logits); the kernels never raise one.
#include <cmath>
#include "common.cuh"
#include "tc3_common.cuh"

namespace wkv6 {
namespace {

using namespace tc3;

constexpr uint32_t OFF_R = 0, OFF_K = 8192, OFF_V = 16384, OFF_GY = 24576, OFF_W = 32768, OFF_PT = OFF_W;
constexpr uint32_t OFF_SIN = 40960, OFF_GB = 49152;
// Kt versions: version q = rows s 0..16q+15 in reference rho_q (64 + 48 + 32 + 16 rows)
constexpr uint32_t OFF_KT = 57344;
// Rp versions: version p = rows t 16p..63 (stored from row 0) in reference rho_p (64 + 48 + 32 + 16 rows)
constexpr uint32_t OFF_RP = 77824;
constexpr uint32_t OFF_DA = 98304, OFF_TILES_END = 106496;
__host__ __device__ constexpr uint32_t kt_ver(int q) { return q == 3 ? 0u : q == 2 ? 8192u : q == 1 ? 14336u : 18432u; }
__host__ __device__ constexpr uint32_t rp_ver(int p) { return p == 0 ? 0u : p == 1 ? 8192u : p == 2 ? 14336u : 18432u; }
// output tiles reuse operand tiles that are dead by the time they are written: gr the Kt versions 0-2 (dead
// once Dr is done), gv Kt_3 (dead once gv is done), gk the dA tile, gw the Rp versions (dead once M3 is done)
constexpr uint32_t OFF_GRT = OFF_KT + 8192, OFF_GVT = OFF_KT, OFF_GKT = OFF_DA, OFF_GWT = OFF_RP;

struct Extra {
    float gtot[64][8];        // decay total of every 8-token group, per channel (log2 units): one 32-byte row per channel
    float pdu[4][64];         // per channel-quarter partial sums of r u k, per token
    float bd[64];             // Bm[t,t]
    float q0p[2][64];         // <S_in, G>_i, partial over each half of j
    float htY[2][64], htX[2][64];   // per token-half totals of D and of X, per channel
    float gu_s[64];
    int gu_last;
    uint64_t bar_rk, bar_w, bar_vg, bar_sin, bar_bm, bar_m1, bar_dr, bar_m2, bar_m3;
    uint32_t tmem_base;
};
constexpr uint32_t SMEM_BYTES = OFF_TILES_END + sizeof(Extra);
constexpr uint32_t TM_G = 0, TM_X0 = 64, TM_X1 = 128, TM_X2 = 192, TM_COLS = 256;
// An M = 64 accumulator only occupies lanes 0-15 of each 32-lane TMEM sub-partition; lanes 16-31 of the
// same columns are per-thread scratch ("parking"): 4 regions x 2 registers per token pair.
//   PARK_A: Rt (packed bf16 pair), E of e = 0 (fp32; E_1 = E_0 2^l_0)   -> T2 replaces them by XA (fp32, e = 0,1),
//           T3 by its part of gl
//   PARK_B: (r, k) raw packed bf16 pairs
//   PARK_C: Kt_own (packed bf16 pair), F of e = 0 (fp32; F_1 = F_0 2^-l_1)
//   PARK_L: l (fp32, e = 0,1)
// (E and F stay fp32: as bf16 they put 2^-9 of relative error on whole output elements, which showed in the max-abs
// bound of gk at the full benchmark shape)
constexpr uint32_t PARK_A = 0, PARK_B = 64, PARK_C = 128, PARK_L = 192;

struct Params {
    int B, T, H;
    const bf16 *u;
    int has_s0;
    // time-axis segmentation (seg_scan.cu): the grid has B*nseg rows; row = b*nseg + seg covers tokens
    // [seg*seg_chunks*64, min(T, (seg+1)*seg_chunks*64)) of sequence b; g_init = dL/dS behind the last token of
    // each row, [rows,H,64(value),64(key)], fp32 or (g_init_f32 = 0) bf16; gu, gs, flags and checkpoints are indexed
    // by row.  nseg = 1, seg_chunks = ceil(T/64), g_init = nullptr for an ordinary call; the SEG instantiation with
    // nseg = 1 and g_init = the caller's final-state gradient for an ordinary call that has one.
    const void *g_init;
    int nseg, seg_chunks;
    float lmin;               // floor of the per-token log2-decay (>= -LCLAMP2)
    bf16 *gu, *gs;
    bf16 *gu_total;           // nullptr, or bf16 [C]: sum of gu over the grid's rows, added up by the last CTA of every head
    int *gu_count;            // its arrival counters, int [H], zero before the launch (left zero again)
    const int *hz_flags;      // nullptr, or [rows*H]: 1 = this stream needs the exact route
    const int *row_len;       // BI modes: tokens of every batch row (p + 1 of wkv6_bi), device int [B]
    const int *row_order;     // BI modes: batch rows sorted by length, longest first, device int [B]
    long long *dbg;           // nullptr, or [gridDim][NC][8 (32 in the profiling build)] clock64 stamps of warp 0 at the stage boundaries (profiling aid)
    int g_init_f32;           // (last: the fields above keep their offsets, and SEG = false reads none of the new ones)
    int gs_f32;               // SEG only: gs is fp32 (reinterpreted), else bf16
};

// true when `x` holds in any of the 256 compute threads (named barrier B_SCAN, which they all reach)
__device__ __forceinline__ bool compute_any(bool x) {
    uint32_t r;
    asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %1, 0;\n\tbar.red.or.pred q, %2, %3, p;\n\tselp.u32 %0, 1, 0, q;\n\t}"
                 : "=r"(r) : "r"((uint32_t)x), "n"(B_SCAN_ID), "n"(CTHREADS) : "memory");
    return r != 0;
}

__device__ __forceinline__ uint32_t pack_frag(const uint32_t *v, int g, int hh) {
    return pack2(__uint_as_float(v[4 * g + 2 * hh]), __uint_as_float(v[4 * g + 2 * hh + 1]));
}

// SEG = false: the ordinary call, its own instantiation (see the forward kernel).
// BI: direction of the bidirectional op (tc3_common.cuh); BI_NONE for every other call.
template <bool SEG, int BI = BI_NONE>
__global__ void __launch_bounds__(NTHREADS, 2)
wkv6_tc3_bwd_kernel(const __grid_constant__ CUtensorMap map_r, const __grid_constant__ CUtensorMap map_k,
                    const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_w,
                    const __grid_constant__ CUtensorMap map_gy, const __grid_constant__ CUtensorMap map_ck,
                    const __grid_constant__ CUtensorMap map_gr, const __grid_constant__ CUtensorMap map_gk,
                    const __grid_constant__ CUtensorMap map_gv, const __grid_constant__ CUtensorMap map_gw, Params p) {
    const int h = blockIdx.x % p.H;
    const int row = BI ? p.row_order[blockIdx.x / p.H] : blockIdx.x / p.H;
    const int rid = BI ? row * p.H + h : blockIdx.x;     // row id: flags, checkpoints
    if (p.hz_flags && p.hz_flags[rid] != 0) return; // the exact (SIMT) route handles this stream
    extern __shared__ __align__(1024) uint8_t sm[];
    Extra &ex = *reinterpret_cast<Extra *>(sm + OFF_TILES_END);
    if ((smem_u32(sm) & 1023u) != 0) __trap();
    const int b = SEG ? row / p.nseg : row;                                  // batch index inside the [B,T,C] tensors
    const int t_base = SEG ? (row % p.nseg) * p.seg_chunks * L : 0;          // first token of this row's segment
    const int T = BI ? p.row_len[b] : SEG ? min(p.T - t_base, p.seg_chunks * L) : p.T, C = p.H * 64;
    const int NC = (T + L - 1) / L;
    const int ck_stride = SEG ? p.seg_chunks : BI ? (p.T + L - 1) / L : NC;  // checkpoint slots per row
    // first token of chunk c's tile (BI_REV: the tile that ends at token T-1-64c, read backwards; see tc3_common.cuh)
    auto tok0 = [&](int c) { return BI == BI_REV ? max(T - (c + 1) * L, 0) : t_base + c * L; };
    Frag F;
    F.init();
    const int warp = F.warp, lane = F.lane;

    if (threadIdx.x == 0) {
        mbar_init(&ex.bar_rk, 1);
        mbar_init(&ex.bar_w, 1);
        mbar_init(&ex.bar_vg, 1);
        mbar_init(&ex.bar_sin, 1);
        mbar_init(&ex.bar_bm, 1);
        mbar_init(&ex.bar_m1, 1);
        mbar_init(&ex.bar_dr, 1);
        mbar_init(&ex.bar_m2, 1);
        mbar_init(&ex.bar_m3, 1);
        fence_barrier_init();
    }
    if (threadIdx.x < 64) ex.gu_s[threadIdx.x] = 0.f;
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
        // issuer
        // =====================================================================================
        auto issue_rk = [&](int c) {
            mbar_arrive_expect_tx(&ex.bar_rk, 2 * 8192);
            tma_load_3d(sm + OFF_R, &map_r, &ex.bar_rk, h * 64, tok0(c), b);
            tma_load_3d(sm + OFF_K, &map_k, &ex.bar_rk, h * 64, tok0(c), b);
        };
        auto issue_w = [&](int c) {
            mbar_arrive_expect_tx(&ex.bar_w, 8192);
            tma_load_3d(sm + OFF_W, &map_w, &ex.bar_w, h * 64, tok0(c), b);
        };
        auto issue_vg = [&](int c) {
            mbar_arrive_expect_tx(&ex.bar_vg, 2 * 8192);
            tma_load_3d(sm + OFF_V, &map_v, &ex.bar_vg, h * 64, tok0(c), b);
            tma_load_3d(sm + OFF_GY, &map_gy, &ex.bar_vg, h * 64, tok0(c), b);
        };
        auto issue_sin = [&](int c) {
            mbar_arrive_expect_tx(&ex.bar_sin, 8192);
            tma_load_3d(sm + OFF_SIN, &map_ck, &ex.bar_sin, 0, (rid * ck_stride + c) * 64, 0);
        };
        if (lane == 0) {
            tma_prefetch_desc(&map_r); tma_prefetch_desc(&map_k); tma_prefetch_desc(&map_v);
            tma_prefetch_desc(&map_w); tma_prefetch_desc(&map_gy); tma_prefetch_desc(&map_ck);
            issue_rk(NC - 1);
            issue_w(NC - 1);
            issue_vg(NC - 1);
            issue_sin(NC - 1);
        }
        const uint32_t kt = sbase + OFF_KT, rp = sbase + OFF_RP;
        const uint32_t da = sbase + OFF_DA, pt = sbase + OFF_PT, gb = sbase + OFF_GB, sin = sbase + OFF_SIN;
        const uint32_t vv = sbase + OFF_V, gy = sbase + OFF_GY;
        constexpr uint32_t ID_KK = idesc_bf16(64, 64, 0, 0), ID_KM = idesc_bf16(64, 64, 0, 1), ID_MM = idesc_bf16(64, 64, 1, 1);
        constexpr uint32_t ID16_KK = idesc_bf16(64, 16, 0, 0), ID16_MK = idesc_bf16(64, 16, 1, 0), ID16_MM = idesc_bf16(64, 16, 1, 1);
        bar_sync_all<B_T3>();                                    // G = 0 written (TMEM)
        if (lane == 0) {
            mbar_wait(&ex.bar_rk, 0);
            mbar_wait(&ex.bar_w, 0);
            if (BI) mbar_wait(&ex.bar_vg, 0);                    // the compute warps reverse / mask the V and GY tiles first
        }
        __syncwarp();
        bar_arrive_all<B_RAW>();
        for (int it = 0; it < NC; it++) {
            const int c = NC - 1 - it;
            const uint32_t par = it & 1;
            if (lane == 0 && it > 0) tma_store_wait_read<0>();   // every output tile of the previous chunk has left shared memory
            __syncwarp();
            bar_arrive_all<B_FREE>();                            // ... so the preparation may overwrite KT, RP (and T1 DA)
            if (BI) bar_sync_all<B_VG>();                        // V, GY reversed (BI_REV) / masked behind the row's end (BI_CAUSAL)
            // ---- products that need nothing from the operand preparation run under it
            if (elect_one()) {
                mbar_wait(&ex.bar_vg, par);
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < 4; k++)   // Bm[t,s] = GY V^T
                    mma_bf16_ss(tmem + TM_X0, smem_desc_sw128(gy + 32 * k, 8192, 1024), smem_desc_sw128(vv + 32 * k, 8192, 1024), ID_KK, k > 0);
                mbar_wait(&ex.bar_sin, par);
#pragma unroll
                for (int k = 0; k < 4; k++)   // Drs[i,t] = S_in GY^T
                    mma_bf16_ss(tmem + TM_X2, smem_desc_sw128(sin + 32 * k, 8192, 1024), smem_desc_sw128(gy + 32 * k, 8192, 1024), ID_KK, k > 0);
                mma_commit(&ex.bar_bm);
                mbar_wait(&ex.bar_bm, par);
            }
            __syncwarp();
            bar_arrive_all<B_BM>();
            bar_sync_all<B_PREP>();                              // operands written, raw r,k,w consumed
            if (elect_one()) {
                tc_fence_after();
#pragma unroll
                for (int q = 0; q < 4; q++)   // A^T[s, t in q] = Kt_q Rt_own^T            (runs under T1a)
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        mma_bf16_ss(tmem + TM_X1 + 16 * q, smem_desc_sw128(kt + kt_ver(q) + 32 * k, 8192, 1024),
                                    smem_desc_sw128(rp + rp_ver(q) + 32 * k, 8192, 1024), ID16_KK, k > 0);
                mma_commit(&ex.bar_m1);
                mbar_wait(&ex.bar_m1, par);
            }
            __syncwarp();
            bar_arrive_all<B_M1>();
            if (lane == 0 && c > 0) issue_rk(c - 1);             // raw r,k of this chunk were consumed by the preparation
            bar_sync_all<B_T1A>();                               // dA written, Bm consumed
            if (elect_one()) {
                tc_fence_after();
#pragma unroll
                for (int q = 0; q < 4; q++)   // Dr[i, t in q] = sum_{s in blocks <= q} Kt_q[s,i] dA[t,s]     (runs under T1b)
#pragma unroll
                    for (int ks = 0; ks < 4; ks++)
                        if (ks <= q)
                            mma_bf16_ss(tmem + TM_X0 + 16 * q, smem_desc_sw128(kt + kt_ver(q) + 2048 * ks, 8192, 1024),
                                        smem_desc_sw128(da + 2048 * q + 32 * ks, 8192, 1024), ID16_MK, ks > 0);
                mma_commit(&ex.bar_dr);
                mbar_wait(&ex.bar_dr, par);
            }
            __syncwarp();
            bar_arrive_all<B_DR>();
            bar_sync_all<B_T1>();                                // P^T, Gb written; <S_in,G> taken; G decayed
            if (elect_one()) {
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < 4; k++)   // gv[s,j] = P^T GY ...                               (runs under T2a)
                    mma_bf16_ss(tmem + TM_X1, smem_desc_sw128(pt + 32 * k, 8192, 1024), smem_desc_sw128(gy + 2048 * k, 8192, 1024), ID_KM, k > 0);
#pragma unroll
                for (int k = 0; k < 4; k++)   // ... + Kt_3 Gb
                    mma_bf16_ss(tmem + TM_X1, smem_desc_sw128(kt + kt_ver(3) + 32 * k, 8192, 1024), smem_desc_sw128(gb + 2048 * k, 8192, 1024), ID_KM, 1);
                mma_commit(&ex.bar_m2);
#pragma unroll
                for (int k = 0; k < 4; k++)   // G[i,j] += Rp_0^T GY                  (first read in the next T1: covered by the M3 commit)
                    mma_bf16_ss(tmem + TM_G, smem_desc_sw128(rp + rp_ver(0) + 2048 * k, 8192, 1024), smem_desc_sw128(gy + 2048 * k, 8192, 1024), ID_MM, 1);
                mbar_wait(&ex.bar_m2, par);
            }
            __syncwarp();
            bar_arrive_all<B_M2>();
            if (lane == 0 && c > 0) {
                issue_sin(c - 1);                                // S_in of this chunk: read by Drs and T1 only
                issue_w(c - 1);                                  // the P^T tile (= W space) is dead
            }
            bar_sync_all<B_T2A>();                               // Dr, Drs consumed (gr tile written, XA parked)
            if (elect_one()) {
                tc_fence_after();
#pragma unroll
                for (int pb = 0; pb < 4; pb++)   // Dk[i, s in p] = sum_{t >= 16p} Rp_p[t,i] dA[t,s]   (dA read MN-major; under T2b)
#pragma unroll
                    for (int kk = 0; kk < 4; kk++)
                        if (kk < 4 - pb)
                            mma_bf16_ss(tmem + TM_X0 + 16 * pb, smem_desc_sw128(rp + rp_ver(pb) + 2048 * kk, 8192, 1024),
                                        smem_desc_sw128(da + 2048 * (pb + kk) + 32 * pb, 8192, 1024), ID16_MM, kk > 0);
#pragma unroll
                for (int k = 0; k < 4; k++)   // Dks[i,s] = Gb V^T
                    mma_bf16_ss(tmem + TM_X2, smem_desc_sw128(gb + 32 * k, 8192, 1024), smem_desc_sw128(vv + 32 * k, 8192, 1024), ID_KK, k > 0);
                mma_commit(&ex.bar_m3);
                mbar_wait(&ex.bar_m3, par);
                if (c > 0) issue_vg(c - 1);                      // V, GY are dead: the loads have T3 and a whole preparation to land
            }
            __syncwarp();
            bar_arrive_all<B_M3>();
            bar_sync_all<B_T2>();                                // gv tile written (under M3)
            if (lane == 0) {
                if (BI == BI_REV) {                              // added to what the causal pass stored
                    tma_reduce_add_3d(&map_gv, sm + OFF_GVT, h * 64, tok0(c), b);
                    tma_reduce_add_3d(&map_gr, sm + OFF_GRT, h * 64, tok0(c), b);
                } else {
                    tma_store_3d(&map_gv, sm + OFF_GVT, h * 64, tok0(c), b);
                    tma_store_3d(&map_gr, sm + OFF_GRT, h * 64, tok0(c), b);
                }
                tma_store_commit();
                if (c > 0) {                                     // the raw tiles of the next chunk, while T3 runs
                    mbar_wait(&ex.bar_rk, par ^ 1);
                    mbar_wait(&ex.bar_w, par ^ 1);
                    if (BI) mbar_wait(&ex.bar_vg, par ^ 1);
                }
            }
            __syncwarp();
            if (c > 0) bar_arrive_all<B_RAW>();                  // ... have landed: the compute warps go from T3 straight into the next preparation
            bar_sync_all<B_T3>();                                // gk, gw tiles written
            if (lane == 0) {
                if (BI == BI_REV) {
                    tma_reduce_add_3d(&map_gk, sm + OFF_GKT, h * 64, tok0(c), b);
                    tma_reduce_add_3d(&map_gw, sm + OFF_GWT, h * 64, tok0(c), b);
                } else {
                    tma_store_3d(&map_gk, sm + OFF_GKT, h * 64, tok0(c), b);
                    tma_store_3d(&map_gw, sm + OFF_GWT, h * 64, tok0(c), b);
                }
                tma_store_commit();
            }
            __syncwarp();
        }
        if (BI == BI_CAUSAL && NC * L < p.T) {                    // all four gradients are 0 behind the row's last chunk
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 16; k++) *reinterpret_cast<uint4 *>(sm + OFF_R + (lane + 32 * k) * 16) = make_uint4(0, 0, 0, 0);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                for (int c = NC; c * L < p.T; c++) {
                    tma_store_3d(&map_gr, sm + OFF_R, h * 64, c * L, b);
                    tma_store_3d(&map_gk, sm + OFF_R, h * 64, c * L, b);
                    tma_store_3d(&map_gv, sm + OFF_R, h * 64, c * L, b);
                    tma_store_3d(&map_gw, sm + OFF_R, h * 64, c * L, b);
                }
                tma_store_commit();
            }
        }
        if (lane == 0) tma_store_wait_read<0>();          // shared memory has been read; the writes complete with the grid
    } else {
        // =====================================================================================
        // compute warps
        // =====================================================================================
        const int sp = F.sp, ch = F.ch, q = F.q, ri = F.ri;
        const float u_h[2] = {__bfloat162float(p.u[h * 64 + F.row(0)]), __bfloat162float(p.u[h * 64 + F.row(1)])};
        // (The forward pins its TMEM window address in a register, which removes the S2R + 6 instructions the compiler
        // otherwise re-derives in front of every TMEM access: forward 0.2193 -> 0.2167 ms.  Here, at the 96-register limit, one
        // more live register spills 48 bytes and gains nothing.  More registers for the compute warps through setmaxnreg were
        // tried both ways: the issuer warp alone down to 32 / compute warps up to 104 deadlocks in USETMAXREG.TRY_ALLOC (the
        // pool is per sub-partition: only a whole warpgroup, one warp on each, can feed it); with three full warpgroups (384
        // threads, launch at 80 registers, warps 9-11 idle) it runs and is exact, but slower -- forward 0.2166 -> 0.2192 ms,
        // backward 0.3825 -> 0.411 ms: the 32-register issuer path spills.)
        const uint32_t tG = tmem_addr(tmem, 32 * sp, TM_G + 32 * ch);
        const uint32_t tPark = tmem_addr(tmem, 32 * sp + 16, 32 * ch);
        // x2 transposing stores of one 8-token group: lanes 0-7 address the rows of channel half 0, lanes 8-15 of half 1
        uint32_t ti2_off = F.ti1_off ^ ((lane & 8) ? 16u : 0u);
        int dcol = (32 * ch + 2 * q) - (16 * sp + ri);           // column(g, e = 0) - row(hh) at g = hh
        asm volatile("" : "+r"(dcol), "+r"(ti2_off));
        // where the warp's part of a 64 x 64 (row, column) tile lies: 1 = entirely above the diagonal (column > row), 2 =
        // entirely below it, 0 = the diagonal runs through it
        const int tri = 32 * ch - 16 * sp - 15 > 0 ? 1 : 32 * ch + 31 - 16 * sp < 0 ? 2 : 0;
        bool diag_hit[2];                                        // this thread holds the diagonal element of row(hh)
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
            diag_hit[hh] = false;
#pragma unroll
            for (int g = 0; g < 4; g++) diag_hit[hh] |= (dcol + 8 * (g - hh) == 0) | (dcol + 8 * (g - hh) == -1);
        }
        f2 gu2[2] = {0ull, 0ull};
        int sig[2] = {0, 0};              // G in TMEM = G_true 2^(-sig) per key row: rho_0 of the chunk processed last
        uint32_t v[16];

        // G = dL/dS behind the last token (0, or handed in: a segment's scanned G, or the caller's final-state gradient)
        const int seg = SEG ? row % p.nseg : 0;
        const bool first_has_s0 = p.has_s0 || seg > 0;          // a later segment starts from a non-zero state
        bool g_is_zero = !SEG || p.g_init == nullptr;
#pragma unroll
        for (int x = 0; x < 16; x++) v[x] = 0u;
        if (!g_is_zero) {
            bool nz = false;
#pragma unroll
            for (int g = 0; g < 4; g++)
#pragma unroll
                for (int hh = 0; hh < 2; hh++)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const size_t gi = (((size_t)row * p.H + h) * 64 + F.col(g, e)) * 64 + F.row(hh);
                        const float gv = p.g_init_f32 ? static_cast<const float *>(p.g_init)[gi]
                                                      : __bfloat162float(static_cast<const bf16 *>(p.g_init)[gi]);
                        v[4 * g + 2 * hh + e] = __float_as_uint(gv);
                        nz |= gv != 0.f;
                    }
            // the stream's last segment: its G is the final-state gradient, and where that is 0 the last decay feeds
            // nothing, so its gw stays an exact 0 (what the call without a final-state gradient computes)
            if (seg == p.nseg - 1) g_is_zero = !compute_any(nz);
        }
        tmem_st_frag(tG, v);
        tmem_wait_st();
        tc_fence_before();
        bar_arrive_all<B_T3>();

#ifdef WKV6_FINE_STAMPS      // profiling build only (profiles/stage_times.py): 32 clock64 stamps per chunk; the product has none
#define STAMP_N 32
#define STAMP(k) do { if (p.dbg && threadIdx.x == 0) p.dbg[((size_t)blockIdx.x * ck_stride + it) * STAMP_N + (k)] = clock64(); } while (0)
#else
#define STAMP(k) do { } while (0)
#endif
#define STAMPX(k) STAMP(k)
        for (int it = 0; it < NC; it++) {
            const int c = NC - 1 - it;
            const int nv = min(L, T - c * L);
            // ================================================================== P: operand preparation
            bar_sync_all<B_RAW>();
            asm volatile("fence.acq_rel.cta;" ::: "memory");     // (measured: free -- 0.598 ms with and without it)
            STAMP(0);
#ifdef WKV6_FINE_STAMPS
            if (p.dbg && threadIdx.x == 0) {          // slots 30 / 31: global timer (ns) and the SM this CTA runs on
                unsigned long long gt; unsigned smid;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
                asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
                p.dbg[((size_t)blockIdx.x * ck_stride + it) * STAMP_N + 30] = (long long)gt;
                p.dbg[((size_t)blockIdx.x * ck_stride + it) * STAMP_N + 31] = smid;
            }
#endif
            if (BI) {      // the V and GY tiles go to the tensor cores as they lie in shared memory
                if (BI == BI_REV) {
                    const uint32_t vt[2] = {sbase + OFF_V, sbase + OFF_GY};
                    if (nv == L) flip_tiles_full(vt, warp, lane);
                    else flip_tiles_short(vt, nv, warp, lane);
                } else if (nv < L) {
                    zero_tile_rows(sm + OFF_V, nv, threadIdx.x);
                    zero_tile_rows(sm + OFF_GY, nv, threadIdx.x);
                }
                fence_proxy_async();
                bar_arrive_all<B_VG>();
            }
            const int r0 = nv - 1;                  // BI_REV: row x of a tile holds reversed position (r0 - x) mod 64
            const auto raw = [&](int hh) { return BI == BI_REV ? flip_rows(F.ti(hh), r0) : F.ti(hh); };   // where the raw r, k, w tiles are read
            float lamf[2];                    // Lam (log2 units)
            int irb[2][2], ir0[2], ir3[2];    // block references (integers, log2 units): my two blocks, block 0, block 3
            {   // ---- everything per element lives only inside this block
            float l[2][4][2], exq[2][4];
            {
                uint32_t wp[2][4];
                ldsm_x4_t(sbase + OFF_W + raw(0), wp[0][0], wp[0][1], wp[0][2], wp[0][3]);
                ldsm_x4_t(sbase + OFF_W + raw(1), wp[1][0], wp[1][1], wp[1][2], wp[1][3]);
#pragma unroll
                for (int hh = 0; hh < 2; hh++)
#pragma unroll
                    for (int g = 0; g < 4; g++) {
                        float l0 = -fast_ex2(fmaf(bf_lo(wp[hh][g]), LOG2E, LOG2_LOG2E));   // -exp(w) * log2(e)
                        float l1 = -fast_ex2(fmaf(bf_hi(wp[hh][g]), LOG2E, LOG2_LOG2E));
                        l0 = fmaxf(l0, p.lmin);
                        l1 = fmaxf(l1, p.lmin);
                        if (nv < L) {                                   // ragged last chunk: no decay on the padded rows
                            const int t0 = F.col(g, 0);
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
                        if (q == 3) ex.gtot[F.row(hh)][4 * ch + g] = x;
                    }
            }
            {   // park l in the shadow lanes (fragment order [4g + 2h + e])
                uint32_t pk[16];
#pragma unroll
                for (int g = 0; g < 4; g++)
#pragma unroll
                    for (int hh = 0; hh < 2; hh++) {
                        pk[4 * g + 2 * hh] = __float_as_uint(l[hh][g][0]);
                        pk[4 * g + 2 * hh + 1] = __float_as_uint(l[hh][g][1]);
                    }
                tmem_st_frag(tPark + PARK_L, pk);
            }
            STAMPX(8);
            named_bar_sync<B_SCAN, CTHREADS>();
            STAMPX(9);
            bar_sync_all<B_FREE>();              // the output tiles of the previous chunk (KT, RP, DA space) have been stored
            STAMPX(10);

            uint32_t rr[2][4], kk[2][4];
            ldsm_x4_t(sbase + OFF_R + raw(0), rr[0][0], rr[0][1], rr[0][2], rr[0][3]);
            ldsm_x4_t(sbase + OFF_R + raw(1), rr[1][0], rr[1][1], rr[1][2], rr[1][3]);
            ldsm_x4_t(sbase + OFF_K + raw(0), kk[0][0], kk[0][1], kk[0][2], kk[0][3]);
            ldsm_x4_t(sbase + OFF_K + raw(1), kk[1][0], kk[1][1], kk[1][2], kk[1][3]);
            if (BI && nv < L) {              // what lies behind the chunk's nv tokens is real data here, not TMA's zero fill
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    const uint32_t m = pair_mask(F.col(g, 0), nv);
                    rr[0][g] &= m; rr[1][g] &= m;
                    kk[0][g] &= m; kk[1][g] &= m;
                }
            }
            {
                uint32_t pk[16];
#pragma unroll
                for (int g = 0; g < 4; g++)
#pragma unroll
                    for (int hh = 0; hh < 2; hh++) {
                        pk[4 * g + 2 * hh] = rr[hh][g];
                        pk[4 * g + 2 * hh + 1] = kk[hh][g];
                    }
                tmem_st_frag(tPark + PARK_B, pk);
            }
            STAMPX(24);
            uint32_t pa[16], pc[16];                // (Rt, E_0) and (Kt_own, F_0) in fragment order
            f2 du2[4];
#pragma unroll
            for (int g = 0; g < 4; g++) du2[g] = 0ull;
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                float run = 0.f, gb[4];
                int ir[4];
                const float4 gt0 = *reinterpret_cast<const float4 *>(&ex.gtot[F.row(hh)][0]), gt1 = *reinterpret_cast<const float4 *>(&ex.gtot[F.row(hh)][4]);
                const float gt[8] = {gt0.x, gt0.y, gt0.z, gt0.w, gt1.x, gt1.y, gt1.z, gt1.w};
#pragma unroll
                for (int x8 = 0; x8 < 8; x8++) {
                    if (x8 & 1) ir[x8 >> 1] = __float2int_rn(run);        // middle of block x8/2, integer log2 grid
                    if ((x8 >> 2) == ch) gb[x8 & 3] = run;
                    run += gt[x8];
                }
                lamf[hh] = run;
                irb[hh][0] = ch ? ir[2] : ir[0];                           // my groups 0,1 are block 2ch, groups 2,3 block 2ch+1
                irb[hh][1] = ch ? ir[3] : ir[1];
                ir0[hh] = ir[0];
                ir3[hh] = ir[3];
                uint32_t rto[4], kto[4];
                const f2 uu = f2bcast(u_h[hh]);
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    // a0 = exc_0 - rho, a1 = cum_0 - rho = exc_1 - rho, a2 = cum_1 - rho
                    const float a0 = (gb[g] - (float)irb[hh][g >> 1]) + exq[hh][g], a1 = a0 + l[hh][g][0], a2 = a1 + l[hh][g][1];
                    const float E0 = fast_ex2(a0), F0 = fast_ex2(-a1);
                    const f2 E2 = f2pack(E0, fast_ex2(a1)), F2 = f2pack(F0, fast_ex2(-a2));
                    const f2 r2 = bf2f2(rr[hh][g]), k2 = bf2f2(kk[hh][g]);
                    rto[g] = f2tobf(f2mul(r2, E2));
                    kto[g] = f2tobf(f2mul(k2, F2));
                    pa[4 * g + 2 * hh] = rto[g];
                    pa[4 * g + 2 * hh + 1] = __float_as_uint(E0);
                    pc[4 * g + 2 * hh] = kto[g];
                    pc[4 * g + 2 * hh + 1] = __float_as_uint(F0);
                    du2[g] = f2fma(f2mul(r2, uu), k2, du2[g]);
                }
                // versions: my rows in their own reference, then scaled (exactly, by powers of two <= 1) to the
                // reference of every later block (Kt) / earlier block (Rp)
                const uint32_t ti = F.ti(hh);
                if (ch == 0) {
                    stsm_x2_t(sbase + OFF_RP + rp_ver(1) + ti, rto[2], rto[3]);                    // t 16..31 -> rows 0..15
                    scale2(rto[2], rto[3], ir[1] - ir[0]);
                    stsm_x4_t(sbase + OFF_RP + rp_ver(0) + ti, rto[0], rto[1], rto[2], rto[3]);
                    stsm_x2_t(sbase + OFF_KT + kt_ver(0) + ti, kto[0], kto[1]);
                    scale2(kto[0], kto[1], ir[1] - ir[0]);
                    stsm_x4_t(sbase + OFF_KT + kt_ver(1) + ti, kto[0], kto[1], kto[2], kto[3]);
                    scale4(kto, ir[2] - ir[1]);
                    stsm_x4_t(sbase + OFF_KT + kt_ver(2) + ti, kto[0], kto[1], kto[2], kto[3]);
                    scale4(kto, ir[3] - ir[2]);
                    stsm_x4_t(sbase + OFF_KT + kt_ver(3) + ti, kto[0], kto[1], kto[2], kto[3]);
                } else {
                    stsm_x2_t(sbase + OFF_KT + kt_ver(2) + ti, kto[0], kto[1]);                    // s 32..47
                    scale2(kto[0], kto[1], ir[3] - ir[2]);
                    stsm_x4_t(sbase + OFF_KT + kt_ver(3) + ti, kto[0], kto[1], kto[2], kto[3]);
                    stsm_x2_t(sbase + OFF_RP + rp_ver(3) + ti - 4096u, rto[2], rto[3]);            // t 48..63 -> rows 0..15
                    scale2(rto[2], rto[3], ir[3] - ir[2]);
                    stsm_x4_t(sbase + OFF_RP + rp_ver(2) + ti - 4096u, rto[0], rto[1], rto[2], rto[3]);   // t 32..63 -> rows 0..31
                    scale4(rto, ir[2] - ir[1]);
                    stsm_x4_t(sbase + OFF_RP + rp_ver(1) + ti - 2048u, rto[0], rto[1], rto[2], rto[3]);   // rows 16..47
                    scale4(rto, ir[1] - ir[0]);
                    stsm_x4_t(sbase + OFF_RP + rp_ver(0) + ti, rto[0], rto[1], rto[2], rto[3]);
                }
            }
            STAMPX(11);
            tmem_st_frag(tPark + PARK_A, pa);
            tmem_st_frag(tPark + PARK_C, pc);
            {   // diag(u) term: reduce-scatter over the 8 lanes ri, then one partial per channel quarter
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
                ex.pdu[sp][32 * ch + 8 * ((b2 ? 2 : 0) + (b1 ? 1 : 0)) + 2 * q + (b0 ? 1 : 0)] = a1;
            }
            STAMPX(12);
            tmem_wait_st();
            }
            STAMPX(13);
            fence_proxy_async();
            STAMP(1);
            bar_arrive_all<B_PREP>();

            // ================================================================== T1
            bar_sync_all<B_BM>();                        // Bm and Drs were issued before the preparation started
            tc_fence_after();
            STAMP(2);
            // ---- Bm[t rows][s cols] -> dA[t][s] = Bm for s < t; bd[t] = Bm[t,t]   (G is fetched along with it)
            uint32_t vg[16];
            tmem_ld_frag(tmem_addr(tmem, 32 * sp, TM_X0 + 32 * ch), v);
            tmem_ld_frag(tG, vg);
            tmem_wait_ld();
            STAMPX(14);
            // branch-free: dcol = (column of e = 0) - row for g = hh; 8 more per group.  The diagonal element (if this
            // thread holds it) is picked with selects and stored once per row half (divergent stores per element were
            // 700 cycles of this stage)
            // (the warp's part of the tile lies entirely below the diagonal -- kept as it is --, entirely above -- zeros --, or
            // on it: `tri`)
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                uint32_t pk[4];
                if (tri == 2) {
#pragma unroll
                    for (int g = 0; g < 4; g++) pk[g] = pack2(__uint_as_float(v[4 * g + 2 * hh]), __uint_as_float(v[4 * g + 2 * hh + 1]));
                } else if (tri == 1) {
                    pk[0] = pk[1] = pk[2] = pk[3] = 0u;
                } else {
                float dv = 0.f;
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    const int d = dcol + 8 * (g - hh);                    // (s - t) for e = 0
                    const float a0 = __uint_as_float(v[4 * g + 2 * hh]), a1 = __uint_as_float(v[4 * g + 2 * hh + 1]);
                    pk[g] = pack2(d < 0 ? a0 : 0.f, d < -1 ? a1 : 0.f);
                    dv = sel_eq(d, 0, a0, sel_eq(d, -1, a1, dv));
                }
                if (diag_hit[hh]) ex.bd[F.row(hh)] = dv;
                }
                stsm_x4(sbase + OFF_DA + F.rc(hh), pk[0], pk[1], pk[2], pk[3]);
            }
            STAMPX(25);
            fence_proxy_async();
            STAMPX(26);
            tc_fence_before();
            STAMPX(15);
            bar_arrive_all<B_T1A>();                     // Dr (into the Bm columns) can start while G and P^T are handled
            // ---- G rows (key channel i): G_old = G' 2^sig;  q0_i = <S_in, G_old>_i (partial over my half of j);
            //      Gb = bf16(G_old 2^(Lam - rho_3)) (operand of gv and Dks);  G' <- G_old 2^(Lam - rho_0)
            //      (factors applied one after the other: their product may leave the fp32 range although the result does not)
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                const f2 es = f2bcast(pow2i(sig[hh]));
                const f2 f3 = f2bcast(fast_ex2(lamf[hh] - (float)ir3[hh])), f0 = f2bcast(fast_ex2(lamf[hh] - (float)ir0[hh]));
                uint32_t s4[4], gbp[4];
                ldsm_x4(sbase + OFF_SIN + F.rc(hh), s4[0], s4[1], s4[2], s4[3]);
                f2 qs2 = 0ull;
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    const f2 gold = f2mul(f2packu(vg[4 * g + 2 * hh], vg[4 * g + 2 * hh + 1]), es);
                    qs2 = f2fma(bf2f2(s4[g]), gold, qs2);
                    gbp[g] = f2tobf(f2mul(gold, f3));
                    f2unpacku(f2mul(gold, f0), vg[4 * g + 2 * hh], vg[4 * g + 2 * hh + 1]);
                }
                stsm_x4(sbase + OFF_GB + F.rc(hh), gbp[0], gbp[1], gbp[2], gbp[3]);
                float qa, qb;
                f2unpack(qs2, qa, qb);
                float qs = qa + qb;
                qs += __shfl_xor_sync(0xffffffffu, qs, 1);
                qs += __shfl_xor_sync(0xffffffffu, qs, 2);
                if (q == 0) ex.q0p[ch][F.row(hh)] = qs;
                sig[hh] = ir0[hh];
            }
            tmem_st_frag(tG, vg);
            STAMPX(16);
            bar_sync_all<B_M1>();                        // A^T ran under the conversions above
            tc_fence_after();
            STAMPX(17);
            // ---- A^T[s rows][t cols] -> P^T[s][t] = A^T for t > s, diag = sum_i r u k
            tmem_ld_frag(tmem_addr(tmem, 32 * sp, TM_X1 + 32 * ch), v);
            tmem_wait_ld();
            STAMPX(18);
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                uint32_t pk[4];
                if (tri == 1) {
#pragma unroll
                    for (int g = 0; g < 4; g++) pk[g] = pack2(__uint_as_float(v[4 * g + 2 * hh]), __uint_as_float(v[4 * g + 2 * hh + 1]));
                } else if (tri == 2) {
                    pk[0] = pk[1] = pk[2] = pk[3] = 0u;
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
                stsm_x4(sbase + OFF_PT + F.rc(hh), pk[0], pk[1], pk[2], pk[3]);
            }
            STAMPX(19);
            tmem_wait_st();
            fence_proxy_async();
            tc_fence_before();
            STAMP(3);
            bar_arrive_all<B_T1>();

            // ================================================================== T2: gr tile, XA
            bar_sync_all<B_DR>();                        // Dr ran under T1b; gv is not needed yet
            tc_fence_after();
            STAMP(4);
            // per 8-token group: Dr, Drs -> gr (tile) and XA, which replaces (Rt, E) in the shadow lanes until T3.
            // The TMEM loads of group g+1 are in flight while group g is computed (tcgen05.wait::ld waits for ALL
            // outstanding loads, so they are issued right after the wait).
            {
            uint32_t tb[2][5][4];
            auto t2_load = [&](int g, uint32_t (&b)[5][4]) {
                tmem_ld_frag1(tmem_addr(tmem, 32 * sp, TM_X0 + 32 * ch + 8 * g), b[0]);
                tmem_ld_frag1(tmem_addr(tmem, 32 * sp, TM_X2 + 32 * ch + 8 * g), b[1]);
                tmem_ld_frag1(tPark + PARK_A + 8 * g, b[2]);
                tmem_ld_frag1(tPark + PARK_B + 8 * g, b[3]);
                tmem_ld_frag1(tPark + PARK_L + 8 * g, b[4]);
            };
            t2_load(0, tb[0]);
#pragma unroll
            for (int g = 0; g < 4; g++) {
                uint32_t (&d4)[4] = tb[g & 1][0], (&s4)[4] = tb[g & 1][1], (&a4)[4] = tb[g & 1][2], (&b4)[4] = tb[g & 1][3], (&l4)[4] = tb[g & 1][4];
                tmem_wait_ld();
                if (g < 3) t2_load(g + 1, tb[(g + 1) & 1]);
                const f2 bd2 = *reinterpret_cast<const f2 *>(&ex.bd[F.col(g, 0)]);
                uint32_t grp[2];
#pragma unroll
                for (int hh = 0; hh < 2; hh++) {
                    const f2 erho = f2bcast(pow2i(irb[hh][g >> 1]));                       // 2^rho of this block (0 when out of range)
                    const f2 z = f2fma(erho, f2packu(s4[2 * hh], s4[2 * hh + 1]), f2packu(d4[2 * hh], d4[2 * hh + 1]));
                    const f2 ubk = f2mul(f2mul(bd2, f2bcast(u_h[hh])), bf2f2(b4[2 * hh + 1]));
                    const float E0 = __uint_as_float(a4[2 * hh + 1]);
                    grp[hh] = f2tobf(f2fma(f2pack(E0, E0 * fast_ex2(__uint_as_float(l4[2 * hh]))), z, ubk));     // E Z + u bd k
                    f2unpacku(f2mul(bf2f2(a4[2 * hh]), z), a4[2 * hh], a4[2 * hh + 1]);    // XA = Rt Z, Rt exactly as the MMAs saw it
                }
                stsm_x2_t(sbase + OFF_GRT + (BI == BI_REV ? flip_rows(ti2_off + 1024u * g, r0) : ti2_off + 1024u * g), grp[0], grp[1]);
                tmem_st_frag1(tPark + PARK_A + 8 * g, a4);
            }
            }
            tmem_wait_st();
            fence_proxy_async();
            tc_fence_before();
            STAMP(5);
            bar_arrive_all<B_T2A>();                     // Dk / Dks may overwrite the Dr / Drs columns
            // ---- gv rows -> tile (runs while the tensor cores work on M3)
            bar_sync_all<B_M2>();
            tc_fence_after();
            tmem_ld_frag(tmem_addr(tmem, 32 * sp, TM_X1 + 32 * ch), v);
            tmem_wait_ld();
            stsm_x4(sbase + OFF_GVT + (BI == BI_REV ? flip_rows(F.rc(0), r0) : F.rc(0)), pack_frag(v, 0, 0), pack_frag(v, 1, 0), pack_frag(v, 2, 0), pack_frag(v, 3, 0));
            stsm_x4(sbase + OFF_GVT + (BI == BI_REV ? flip_rows(F.rc(1), r0) : F.rc(1)), pack_frag(v, 0, 1), pack_frag(v, 1, 1), pack_frag(v, 2, 1), pack_frag(v, 3, 1));
            fence_proxy_async();
            tc_fence_before();
            bar_arrive_all<B_T2>();

            // ================================================================== T3: gk tile, gw tile
            bar_sync_all<B_M3>();
            tc_fence_after();
            STAMP(6);
            // per 8-token group: Dk, Dks, XA -> gk (tile), running scans; the part of gl that does not need the
            // other token half replaces (XA, Kt_own) in the shadow lanes.
            // With X = XA - Kt_own Dk and D = Kt_own Zk - XA:  gl_t = 2^Lam q0 + sum_all X + sum_{s<t} D_s - XA_t,
            // so one exclusive prefix scan of D plus the totals of X are enough (the scan runs on -D).
            float runD[2] = {0.f, 0.f}, runX[2] = {0.f, 0.f};
            {
            uint32_t tb[2][6][4];
            auto t3_load = [&](int g, uint32_t (&b)[6][4]) {
                tmem_ld_frag1(tmem_addr(tmem, 32 * sp, TM_X0 + 32 * ch + 8 * g), b[0]);
                tmem_ld_frag1(tmem_addr(tmem, 32 * sp, TM_X2 + 32 * ch + 8 * g), b[1]);
                tmem_ld_frag1(tPark + PARK_A + 8 * g, b[2]);
                tmem_ld_frag1(tPark + PARK_B + 8 * g, b[3]);
                tmem_ld_frag1(tPark + PARK_C + 8 * g, b[4]);
                tmem_ld_frag1(tPark + PARK_L + 8 * g, b[5]);
            };
            t3_load(0, tb[0]);
#pragma unroll
            for (int g = 0; g < 4; g++) {
                uint32_t (&d4)[4] = tb[g & 1][0], (&s4)[4] = tb[g & 1][1], (&a4)[4] = tb[g & 1][2], (&b4)[4] = tb[g & 1][3];
                uint32_t (&c4)[4] = tb[g & 1][4], (&l4)[4] = tb[g & 1][5];
                tmem_wait_ld();
                if (g < 3) t3_load(g + 1, tb[(g + 1) & 1]);
                const f2 bd2 = *reinterpret_cast<const f2 *>(&ex.bd[F.col(g, 0)]);
                uint32_t gkp[2];
#pragma unroll
                for (int hh = 0; hh < 2; hh++) {
                    const f2 elr = f2bcast(pow2i(ir3[hh] - irb[hh][g >> 1]));              // 2^(rho_3 - rho_p)
                    const f2 dk = f2packu(d4[2 * hh], d4[2 * hh + 1]), xa = f2packu(a4[2 * hh], a4[2 * hh + 1]);
                    const f2 z = f2fma(elr, f2packu(s4[2 * hh], s4[2 * hh + 1]), dk);
                    const f2 nkt = bf2f2(c4[2 * hh] ^ 0x80008000u);          // -Kt_own, exactly as the MMAs saw it
                    const f2 x2 = f2fma(nkt, dk, xa);                          // X = XA - Bi
                    const f2 nd2 = f2fma(nkt, z, xa);                          // -D = XA - Kt_own Zk
                    const f2 br = f2mul(bd2, bf2f2(b4[2 * hh]));
                    const float F0 = __uint_as_float(c4[2 * hh + 1]);
                    gkp[hh] = f2tobf(f2fma(f2pack(F0, F0 * fast_ex2(-__uint_as_float(l4[2 * hh + 1]))), z, f2mul(br, f2bcast(u_h[hh]))));   // F Zk + u bd r
                    gu2[hh] = f2fma(br, bf2f2(b4[2 * hh + 1]), gu2[hh]);
                    float x0, x1, nd0, nd1, xa0, xa1;
                    f2unpack(x2, x0, x1);
                    f2unpack(nd2, nd0, nd1);
                    f2unpack(xa, xa0, xa1);
                    // exclusive prefix of -D over the 4 lanes of the group; X is only needed as a total: per-lane sums
                    // here, one reduction over the 4 lanes behind the loop
                    const float pd = nd0 + nd1;
                    float y = pd, tmp;
                    tmp = __shfl_up_sync(0xffffffffu, y, 1, 4);
                    if (q >= 1) y += tmp;
                    tmp = __shfl_up_sync(0xffffffffu, y, 2, 4);
                    if (q >= 2) y += tmp;
                    const float ex0 = runD[hh] + (y - pd);                     // sum_{s<t} (-D_s) for e = 0
                    a4[2 * hh] = __float_as_uint(ex0 + xa0);                   // gl_t = base - (this)
                    a4[2 * hh + 1] = __float_as_uint(ex0 + nd0 + xa1);
                    runD[hh] += __shfl_sync(0xffffffffu, y, 3, 4);
                    runX[hh] += x0 + x1;
                }
                stsm_x2_t(sbase + OFF_GKT + (BI == BI_REV ? flip_rows(ti2_off + 1024u * g, r0) : ti2_off + 1024u * g), gkp[0], gkp[1]);
                tmem_st_frag1(tPark + PARK_A + 8 * g, a4);
            }
            }
            STAMPX(20);
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                runX[hh] += __shfl_xor_sync(0xffffffffu, runX[hh], 1);
                runX[hh] += __shfl_xor_sync(0xffffffffu, runX[hh], 2);
            }
            if (q == 0) {
#pragma unroll
                for (int hh = 0; hh < 2; hh++) {
                    ex.htY[ch][F.row(hh)] = runD[hh];
                    ex.htX[ch][F.row(hh)] = runX[hh];
                }
            }
            if (c == 0 && p.gs) {        // after chunk 0, G' 2^rho_0 is dL/dS_0 (the G update of M2 is covered by the M3 commit)
                tmem_ld_frag(tG, v);
                tmem_wait_ld();
#pragma unroll
                for (int hh = 0; hh < 2; hh++) {
                    const float es = pow2i(sig[hh]);
#pragma unroll
                    for (int g = 0; g < 4; g++)
#pragma unroll
                        for (int e = 0; e < 2; e++) {   // gs[b,h,j,i] = dL/dS_0[i][j]
                            const size_t gi = (((size_t)row * p.H + h) * 64 + F.col(g, e)) * 64 + F.row(hh);
                            const float gsv = __uint_as_float(v[4 * g + 2 * hh + e]) * es;
                            if (SEG && p.gs_f32) reinterpret_cast<float *>(p.gs)[gi] = gsv;
                            else p.gs[gi] = __float2bfloat16_rn(gsv);
                        }
                }
            }
            tmem_wait_st();
            STAMPX(21);
            named_bar_sync<B_SCAN, CTHREADS>();          // token-half totals of both scans are in shared memory
            STAMPX(22);
            uint32_t lp[16];
            tmem_ld_frag(tPark + PARK_A, v);
            tmem_ld_frag(tPark + PARK_L, lp);
            tmem_wait_ld();
            STAMPX(23);
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                const int i = F.row(hh);
                // 2^Lam <S_in,G> + total X of both halves + D of the earlier half (runD / htY hold sums of -D)
                const float base = (ex.q0p[0][i] + ex.q0p[1][i]) * fast_ex2(lamf[hh]) + runX[hh] + (ch ? ex.htX[0][i] - ex.htY[0][i] : ex.htX[1][i]);
                const f2 base2 = f2bcast(base), ln2 = f2bcast(LN2);
                uint32_t gwp[4];
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    const f2 gl = f2sub(base2, f2packu(v[4 * g + 2 * hh], v[4 * g + 2 * hh + 1]));
                    float gw0, gw1;
                    f2unpack(f2mul(f2mul(f2packu(lp[4 * g + 2 * hh], lp[4 * g + 2 * hh + 1]), ln2), gl), gw0, gw1);
                    if (c == 0 && !first_has_s0 && ch == 0 && g == 0 && q == 0) gw0 = 0.f;   // t = 0 with S_0 = 0
                    if (c == NC - 1 && g_is_zero) {      // the last decay feeds no output: exactly 0 like cuda/wkv6_cuda.cu:226
                        if (F.col(g, 0) == nv - 1) gw0 = 0.f;
                        if (F.col(g, 1) == nv - 1) gw1 = 0.f;
                    }
                    gwp[g] = pack2(gw0, gw1);
                }
                stsm_x4_t(sbase + OFF_GWT + (BI == BI_REV ? flip_rows(F.ti(hh), r0) : F.ti(hh)), gwp[0], gwp[1], gwp[2], gwp[3]);
            }
            fence_proxy_async();
            tc_fence_before();
            STAMP(7);
            bar_arrive_all<B_T3>();
        }
        // gu[b, i] = sum_t r k bd: reduce over the 4 lanes q and the two token halves
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
            float xa_, xb_;
            f2unpack(gu2[hh], xa_, xb_);
            float x = xa_ + xb_;
            x += __shfl_xor_sync(0xffffffffu, x, 1);
            x += __shfl_xor_sync(0xffffffffu, x, 2);
            if (q == 0) atomicAdd(&ex.gu_s[F.row(hh)], x);
        }
        named_bar_sync<B_SCAN, CTHREADS>();
        if (BI != BI_REV && threadIdx.x < 64) p.gu[(size_t)row * C + h * 64 + threadIdx.x] = __float2bfloat16_rn(ex.gu_s[threadIdx.x]);   // (the reverse pass has u = 0)
        if (!SEG && BI == BI_NONE && p.gu_total) {
            // sum over the batch rows (src/model.py:232 does it with torch.sum): the last CTA of this head to get here adds
            // the bf16 rows in fp32, in row order
            const int rows = gridDim.x / p.H;
            if (threadIdx.x < 64) __threadfence();
            named_bar_sync<B_SCAN, CTHREADS>();
            if (threadIdx.x == 0) ex.gu_last = atomicAdd(&p.gu_count[h], 1) == rows - 1;
            named_bar_sync<B_SCAN, CTHREADS>();
            if (ex.gu_last && threadIdx.x < 64) {
                __threadfence();
                float acc = 0.f;
                for (int rb = 0; rb < rows; rb++) acc += __bfloat162float(__ldcg(&p.gu[(size_t)rb * C + h * 64 + threadIdx.x]));
                p.gu_total[h * 64 + threadIdx.x] = __float2bfloat16_rn(acc);
                if (threadIdx.x == 0) p.gu_count[h] = 0;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

#ifdef WKV6_FINE_STAMPS
void *g_tc3_bwd_stamps = nullptr;   // profiling build: set through wkv6b200_debug_stamps()
#endif

size_t tc3_saved_bytes(int B, int T, int H) {
    size_t NC = (size_t)(T + L - 1) / L;
    int nseg = 1, seg_chunks = 0;
    seg_plan_train(B, T, H, &nseg, &seg_chunks);           // uneven segments leave a few checkpoint slots unused
    if (nseg > 1) NC = (size_t)nseg * seg_chunks;
    return TC3_SAVED_HEADER + (size_t)B * H * NC * 8192;
}
// scratch of the time-segmented backward (seg_scan.cu): r, gy, w reversed inside the segments, the segments'
// own and scanned state gradients, decay sums, per-row gs and gu
static size_t seg_backward_scratch_bytes(int B, int T, int H) {
    int nseg = 1, seg_chunks = 0;
    seg_plan_train(B, T, H, &nseg, &seg_chunks);
    if (nseg <= 1) return 0;
    const size_t C = (size_t)H * 64, Bs = (size_t)B * nseg, n_el = (size_t)B * T * C, st = Bs * H * 4096;
    return 3 * n_el * 2 + 2 * st * 4 + Bs * C * 4 + st * 2 + Bs * C * 2 + 1024;
}
size_t tc3_backward_workspace_bytes(int B, int T, int H, bool has_saved) {
    return simt_backward_workspace_bytes(B, T, H) + (has_saved ? seg_backward_scratch_bytes(B, T, H) : tc3_saved_bytes(B, T, H));
}
bool tc3_backward_supported(const Args &a) {
    return a.io_dtype == WKV6_BF16 && a.w_kind == W_RAW_BF16 && a.mask == nullptr && a.T >= 1 && !a.s0_f32 &&
           tc::get_encode_fn() != nullptr;
}

// gw = 0 where the OPT-IN decay clamp is active (w > log(clamp)), for the streams the tensor-core kernel computed
// (flags index rows of the launch: stream = row / nseg when the call was segmented)
__global__ void __launch_bounds__(256) clamp_gw_kernel(size_t n8, const bf16 *__restrict__ w, bf16 *__restrict__ gw, float wmax,
                                                       const int *__restrict__ flags, int T, int H, int nseg) {
    const size_t C = (size_t)H * 64;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
        const size_t e0 = 8 * i, bt = e0 / C, b = bt / T, h = (e0 % C) / 64;
        if (flags && flags[(b * nseg) * H + h] != 0) continue;    // the exact route writes its own gw
        const uint4 wv = *reinterpret_cast<const uint4 *>(w + e0);
        uint4 gv = *reinterpret_cast<const uint4 *>(gw + e0);
        const __nv_bfloat16 *wp = reinterpret_cast<const __nv_bfloat16 *>(&wv);
        __nv_bfloat16 *gp = reinterpret_cast<__nv_bfloat16 *>(&gv);
        bool any = false;
#pragma unroll
        for (int e = 0; e < 8; e++)
            if (__bfloat162float(wp[e]) > wmax) { gp[e] = __float2bfloat16_rn(0.f); any = true; }
        if (any) *reinterpret_cast<uint4 *>(gw + e0) = gv;
    }
}
static inline float __logf_host(float x) { return logf(x); }

template <bool SEG, int BI>
static int launch_bwd_kernel(dim3 grid, cudaStream_t stream, const CUtensorMap *const *m, const Params &p) {
    static bool attr_done[64] = {};          // function attributes are per device (and per instantiation)
    int dev = 0;
    WKV6_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_done[dev]) {
        WKV6_CUDA_CHECK(cudaFuncSetAttribute(wkv6_tc3_bwd_kernel<SEG, BI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
        WKV6_CUDA_CHECK(cudaFuncSetAttribute(wkv6_tc3_bwd_kernel<SEG, BI>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
    wkv6_tc3_bwd_kernel<SEG, BI><<<grid, NTHREADS, SMEM_BYTES, stream>>>(*m[0], *m[1], *m[2], *m[3], *m[4], *m[5], *m[6], *m[7], *m[8], *m[9], p);
    count_launch();
    WKV6_CUDA_CHECK(cudaGetLastError());
    return WKV6_OK;
}

// one launch of the backward kernel on `a` viewed as given (B rows of T tokens), chunk-start states in ckpt
// gu_count: nullptr, or the zeroed per-head arrival counters that let an ordinary call add gu up into a.gu_total
// g_init: nullptr, or dL/dS behind every row's last token (g_init_f32: fp32, else bf16); an unsegmented call with one
// runs the SEG instantiation with nseg = 1 (which leaves gu_total to the caller)
// bi / row_len: direction of the bidirectional op (tc3_common.cuh) and the device int [B] row lengths it needs
static int launch_bwd(const Args &a, const bf16 *ckpt, const int *flags, int *gu_count, const void *g_init, int g_init_f32,
                      int nseg, int seg_chunks, bool has_s0, int bi = BI_NONE, const int *row_len = nullptr,
                      const int *row_order = nullptr) {
    const int C = a.H * 64;
    if (nseg <= 1) { nseg = 1; seg_chunks = (a.T + L - 1) / L; }
    const size_t NC = (size_t)nseg * seg_chunks;
    CUtensorMap mr, mk, mv, mw, mg, mc, ogr, ogk, ogv, ogw;
    const auto dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const void *ptrs[10] = {a.r, a.k, a.v, a.w, a.gy, ckpt, a.gr, a.gk, a.gv, a.gw};
    CUtensorMap *maps[10] = {&mr, &mk, &mv, &mw, &mg, &mc, &ogr, &ogk, &ogv, &ogw};
    for (int i = 0; i < 10; i++) {
        const bool ok = (i == 5) ? tc::make_btc_map(maps[i], ptrs[i], 1, (int)((size_t)a.B * a.H * NC * 64), 64, 64, dt, 2, 64)
                                 : tc::make_btc_map(maps[i], ptrs[i], a.B, a.T, C, L, dt, 2, 64);
        if (!ok) {
            set_error("cuTensorMapEncodeTiled failed for tensor %d (r,k,v,w,gy,ckpt,gr,gk,gv,gw), pointer %p (16-byte alignment required)", i, ptrs[i]);
            return WKV6_ECUDA;
        }
    }
    Params p;
    p.B = a.B; p.T = a.T; p.H = a.H;
    p.u = (const bf16 *)a.u;
    p.has_s0 = has_s0;
    p.g_init = g_init; p.g_init_f32 = g_init_f32;
    p.nseg = nseg; p.seg_chunks = seg_chunks;
    p.lmin = tc_lmin_log2(a);
    p.gu = (bf16 *)a.gu; p.gs = (bf16 *)a.gs;
    p.hz_flags = flags;
    p.gs_f32 = a.gs_f32;
    // an fp32 gs, like a g_init or segments, takes the SEG instantiation
    const bool seg_inst = nseg > 1 || g_init || a.gs_f32;
    // in-kernel sum of gu over the rows: ordinary call only
    const bool sum_gu = a.gu_total && gu_count && !seg_inst && bi == BI_NONE && a.H <= 512;
    p.gu_total = sum_gu ? (bf16 *)a.gu_total : nullptr;
    p.gu_count = gu_count;
    if (sum_gu) a.gu_total_done = true;
#ifdef WKV6_FINE_STAMPS
    p.dbg = (long long *)g_tc3_bwd_stamps;
#else
    p.dbg = nullptr;
#endif
    p.row_len = row_len; p.row_order = row_order;
    const bool clamp = a.lmin > -INFINITY;
    const dim3 grid(a.B * nseg * a.H);
    int rc;
    if (bi == BI_CAUSAL) rc = launch_bwd_kernel<false, BI_CAUSAL>(grid, a.stream, maps, p);
    else if (bi == BI_REV) rc = launch_bwd_kernel<false, BI_REV>(grid, a.stream, maps, p);
    else if (seg_inst) rc = launch_bwd_kernel<true, BI_NONE>(grid, a.stream, maps, p);
    else rc = launch_bwd_kernel<false, BI_NONE>(grid, a.stream, maps, p);
    if (rc != WKV6_OK) return rc;
    if (clamp) {                       // opt-in decay clamp: a clamped decay no longer depends on w (kept out of the hot kernel)
        const size_t n8 = (size_t)a.B * a.T * C / 8;
        size_t g = (n8 + 255) / 256;
        if (g > 148 * 16) g = 148 * 16;
        clamp_gw_kernel<<<(int)g, 256, 0, a.stream>>>(n8, (const bf16 *)a.w, (bf16 *)a.gw, __logf_host(-a.lmin), flags, a.T, a.H, nseg);
        count_launch();
        WKV6_CUDA_CHECK(cudaGetLastError());
    }
    return WKV6_OK;
}

// Backward over `nseg` time segments run as independent batch rows (seg_scan.cu).  dL/dS at the end of each
// segment comes from the SAME recurrence as the forward state, run on time-reversed (r, gy, w):
//     G_{t-1} = d_t G_t + r_t (x) gy_t      <->      S_{tau+1} = d'_tau S_tau + k'_tau (x) v'_tau
// so: reverse the three tensors inside every segment, a state-only forward pass (k := r_rev, v := gy_rev) gives
// each segment's own contribution, a reverse scan over the segments chains them, and the ordinary backward
// kernel starts every segment from its scanned G.  The forward of the training pair was segmented the same
// way, so `saved` holds the chunk-start states in segment-row order.
static int tc3_backward_segmented(const Args &a, int nseg, int seg_chunks) {
    const int Bs = a.B * nseg, C = a.H * 64, seg_tokens = seg_chunks * L;
    const bf16 *ckpt = (const bf16 *)((uint8_t *)a.saved + TC3_SAVED_HEADER);
    const size_t n_el = (size_t)a.B * a.T * C, st = (size_t)Bs * a.H * 4096;
    // scratch lives in the caller's workspace, behind the part the exact route uses
    const size_t simt_ws = (simt_backward_workspace_bytes(a.B, a.T, a.H) + 1023) / 1024 * 1024;
    uint8_t *buf = (uint8_t *)a.workspace + simt_ws;
    bf16 *r_rev = (bf16 *)buf, *gy_rev = r_rev + n_el, *w_rev = gy_rev + n_el;
    float *g_loc = (float *)(w_rev + n_el), *g_end = g_loc + st, *lam = g_end + st;
    bf16 *gs_tmp = (bf16 *)(lam + (size_t)Bs * C), *gu_tmp = gs_tmp + st;
    int rc = seg_reverse3(a.B, a.T, C, nseg, seg_tokens, a.r, a.gy, a.w, r_rev, gy_rev, w_rev, a.stream);
    Args f = a;                                   // state-only pass: the "state" it ends with is each segment's own dL/dS_start
    f.r = r_rev; f.k = r_rev; f.v = gy_rev; f.w = w_rev;
    f.s0 = nullptr; f.s0_bstride = 0; f.s0_f32 = 0; f.sT = g_loc; f.sT_f32 = 1; f.y = nullptr; f.saved = nullptr; f.gy = nullptr;
    if (rc == WKV6_OK) rc = tc3_forward(f, nullptr, nullptr, nseg, seg_chunks);
    if (rc == WKV6_OK) rc = seg_decay(a.B, a.T, C, nseg, seg_tokens, a.w, lam, tc_lmin_nats(a), a.stream);
    // the chain starts from the caller's final-state gradient (or 0), which the last segment then reads like the others
    if (rc == WKV6_OK) rc = seg_scan(a.B, nseg, a.H, lam, g_loc, a.gT, a.gT_f32, (long long)a.H * 4096, g_end, nullptr, 0, 1, nullptr, a.stream);
    Args v = a;
    // an fp32 gs is staged in g_loc, which nothing reads once the scan has produced g_end
    void *gs_stage = a.gs_f32 ? (void *)g_loc : (void *)gs_tmp;
    const size_t gs_el = a.gs_f32 ? 4 : 2;
    v.gu = gu_tmp; v.gs = a.gs ? gs_stage : nullptr;
    if (rc == WKV6_OK) rc = launch_bwd(v, ckpt, nullptr, nullptr, g_end, 1, nseg, seg_chunks, a.s0 != nullptr);
    if (rc == WKV6_OK) rc = seg_sum_gu(a.B, nseg, C, gu_tmp, a.gu, a.stream);
    if (rc == WKV6_OK && a.gs)                    // dL/dS_0 is what segment 0 of every sequence produced
        rc = cudaMemcpy2DAsync(a.gs, (size_t)a.H * 4096 * gs_el, gs_stage, (size_t)nseg * a.H * 4096 * gs_el, (size_t)a.H * 4096 * gs_el,
                               a.B, cudaMemcpyDeviceToDevice, a.stream) == cudaSuccess ? WKV6_OK : WKV6_ECUDA;
    return rc;
}

// One direction of the bidirectional backward (wkv6_bi_tc.cu): recompute the chunk-start states of that direction
// (state-only forward in the same mode), then the backward kernel in that mode.  ckpt: bf16 [B*H][ceil(T/64)][64][64].
int tc3_backward_bi(const Args &a, void *ckpt, int *flags, int bi, const int *row_len, const int *row_order) {
    if (a.B * a.H == 0 || a.T == 0) return WKV6_OK;
    Args f = a;
    f.y = nullptr; f.sT = nullptr; f.s0 = nullptr;
    if (int rc = tc3_forward(f, ckpt, flags, 1, 0, bi, row_len, row_order)) return rc;
    return launch_bwd(a, (const bf16 *)ckpt, flags, nullptr, nullptr, 0, 1, 0, false, bi, row_len, row_order);
}

int tc3_backward(const Args &a, int *flags) {
    if (a.B * a.H == 0 || a.T == 0) return WKV6_OK;
    const size_t need = tc3_backward_workspace_bytes(a.B, a.T, a.H, a.saved != nullptr);
    if (!a.workspace || a.workspace_bytes < need) {
        set_error("workspace too small: need %zu bytes", need);
        return WKV6_EWORKSPACE;
    }
    if (a.saved) {
        int nseg = 1, seg_chunks = 0;
        seg_plan_train(a.B, a.T, a.H, &nseg, &seg_chunks);
        if (nseg > 1) return tc3_backward_segmented(a, nseg, seg_chunks);
    }
    // `saved`, or without a training pair the same layout in the workspace, behind the part the caller's exact route uses
    uint8_t *sv = a.saved ? (uint8_t *)a.saved : (uint8_t *)a.workspace + simt_backward_workspace_bytes(a.B, a.T, a.H);
    int *gu_count = (int *)sv;
    bf16 *ckpt = (bf16 *)(sv + TC3_SAVED_HEADER);
    if (!a.saved) {
        // recompute the chunk-start states first
        if (a.gu_total) WKV6_CUDA_CHECK(cudaMemsetAsync(gu_count, 0, TC3_SAVED_HEADER, a.stream));
        Args f = a;
        f.y = nullptr;
        f.sT = nullptr;
        if (int rc = tc3_forward(f, ckpt, flags)) return rc;
    }
    return launch_bwd(a, ckpt, flags, gu_count, a.gT, a.gT_f32, 1, 0, a.s0 != nullptr);
}

}  // namespace wkv6
