// wkv6_bi on the tensor-core kernels (cuda/wkv6_bi_cuda.cu:7-112, semantics 3 of SURVEY.md 2.3), fused: no reversed
// copies, no scratch tensors, no combine pass.
//
//   y_t = r_t^T (diag(u) kv_t + S_t) + r_t^T S'_t   for t <= p,   0 for t > p        (p = first masked token, or T-1)
//   S'_{t-1} = diag(d_t) S'_t + kv_t,  S'_p = 0                                       (reverse pass: exclusive, no u)
//
// In reversed time tau = p - t the reverse pass IS the causal recurrence with u = 0 (Z_{tau+1} = d Z_tau + kv,
// y'_tau = r^T Z_tau).  Both directions run on the chunked tcgen05 kernels in their BI modes (tc3_common.cuh): the
// causal direction with the row's own length p + 1 (zeros behind it), the reverse direction reading the SAME r, k, v,
// w (and gy) tiles through TMA at token offsets p - 64c - 63 and mirroring the rows inside the tile -- free for
// everything that goes through ldmatrix / stmatrix, an in-place row swap for the two tiles the tensor cores read as
// they arrive -- and ADDING its output tiles to the causal pass's with TMA reduce stores (bf16 accumulation across
// the two passes, like the reference).  Forward: 2 launches; backward: per direction a state-only forward for the
// chunk-start states and the backward kernel.  Both take raw bf16 logits; the flagged streams (common.cuh) are left to
// the caller's exact route.
#include <stdlib.h>

#include "common.cuh"
#include "tc3_common.cuh"

namespace wkv6 {
namespace {

typedef __nv_bfloat16 bf16;

// row_len[b] = p + 1, p = first t with mask == 0, or T-1 (cuda/wkv6_bi_cuda.cu:25-69)
__global__ void __launch_bounds__(256) bi_last_kernel(int T, const int *__restrict__ mask, int *__restrict__ p) {
    const int *row = mask + (size_t)blockIdx.x * T;
    __shared__ int best;
    if (threadIdx.x == 0) best = T;
    __syncthreads();
    int mine = T;
    for (int t = threadIdx.x; t < T; t += blockDim.x)
        if (row[t] == 0) { mine = t; break; }
    atomicMin(&best, mine);
    __syncthreads();
    if (threadIdx.x == 0) p[blockIdx.x] = (best >= T ? T - 1 : best) + 1;       // row length p + 1
}

// order[rank] = b with the rows ranked by length, longest first (ties by index): the CTAs of long rows start first, so
// the last wave of the grid is made of short rows.  One block; B is a batch size.
__global__ void __launch_bounds__(256) bi_order_kernel(int B, const int *__restrict__ len, int *__restrict__ order) {
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const int lb = len[b];
        int rank = 0;
        for (int j = 0; j < B; j++) {
            const int lj = len[j];
            rank += (lj > lb) | ((lj == lb) & (j < b));
        }
        order[rank] = b;
    }
}

}  // namespace

// WKV6_B200_SYNC_DEBUG=1: synchronise after every step of the bidirectional op and name the one that failed
static int dbg_sync(cudaStream_t st, const char *what) {
    static const bool on = getenv("WKV6_B200_SYNC_DEBUG") != nullptr;
    if (!on) return WKV6_OK;
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("wkv6_bi %s: %s", what, cudaGetErrorString(e)); return WKV6_ECUDA; }
    return WKV6_OK;
}

bool bi_forward_tc_supported(const Args &a) {
    Args t = a;
    t.mask = nullptr;
    return a.mask != nullptr && a.s0 == nullptr && a.sT == nullptr && tc3_forward_supported(t);
}

int bi_forward_tc(const Args &a, int *flags) {
    if (a.B * a.H == 0 || a.T == 0) return WKV6_OK;
    // stream-ordered scratch, kept cached in the pool: zero u, row lengths
    wkv6::ensure_pool_keeps_memory();
    const size_t usz = ((size_t)a.H * N * sizeof(bf16) + 255) / 256 * 256;
    uint8_t *sc = nullptr;
    WKV6_CUDA_CHECK(cudaMallocAsync((void **)&sc, usz + (size_t)2 * a.B * sizeof(int), a.stream));
    bf16 *u0 = (bf16 *)sc;
    int *row_len = (int *)(sc + usz), *row_order = row_len + a.B;
    int rc = WKV6_OK;
    if (cudaMemsetAsync(u0, 0, (size_t)a.H * N * sizeof(bf16), a.stream) != cudaSuccess) rc = WKV6_ECUDA;
    if (rc == WKV6_OK) {
        bi_last_kernel<<<a.B, 256, 0, a.stream>>>(a.T, a.mask, row_len);
        bi_order_kernel<<<1, 256, 0, a.stream>>>(a.B, row_len, row_order);
        count_launch(2);
        if (cudaGetLastError() != cudaSuccess) { set_error("wkv6_bi row-length launch failed"); rc = WKV6_ECUDA; }
    }
    if (rc == WKV6_OK) {
        Args f = a;                       // causal direction: stores y (zeros behind p)
        f.mask = nullptr;
        rc = tc3_forward(f, nullptr, flags, 1, 0, tc3::BI_CAUSAL, row_len, row_order);
        if (rc == WKV6_OK) rc = dbg_sync(a.stream, "forward, causal direction");
        if (rc == WKV6_OK) {              // reverse direction: u = 0, adds to y
            f.u = u0;
            rc = tc3_forward(f, nullptr, flags, 1, 0, tc3::BI_REV, row_len, row_order);
        }
        if (rc == WKV6_OK) rc = dbg_sync(a.stream, "forward, reverse direction");
    }
    cudaFreeAsync(sc, a.stream);
    return rc;
}

// wkv6_bi backward: per direction, the chunk-start states (state-only forward) and the backward kernel; the reverse
// direction adds its four gradient tiles to the causal direction's.  a.workspace must hold
// tc3_backward_workspace_bytes(B, T, H, false) (the chunk-state checkpoints live there, one direction after the other).
int bi_backward_tc(const Args &a, int *flags) {
    if (a.B * a.H == 0 || a.T == 0) return WKV6_OK;
    const int C = a.H * N;
    const size_t base = tc3_backward_workspace_bytes(a.B, a.T, a.H, false);
    if (!a.workspace || a.workspace_bytes < base) { set_error("workspace too small: need %zu bytes", base); return WKV6_EWORKSPACE; }
    wkv6::ensure_pool_keeps_memory();
    const size_t usz = ((size_t)a.H * N * sizeof(bf16) + 255) / 256 * 256, lsz = ((size_t)2 * a.B * sizeof(int) + 255) / 256 * 256;
    uint8_t *sc = nullptr;
    WKV6_CUDA_CHECK(cudaMallocAsync((void **)&sc, usz + lsz + (size_t)a.B * C * sizeof(bf16), a.stream));
    bf16 *u0 = (bf16 *)sc;
    int *row_len = (int *)(sc + usz), *row_order = row_len + a.B;
    bf16 *gu2 = (bf16 *)(sc + usz + lsz);
    // the checkpoints sit where tc3_backward keeps them: behind the part of the workspace the caller's exact route uses
    void *ckpt = (uint8_t *)a.workspace + simt_backward_workspace_bytes(a.B, a.T, a.H) + TC3_SAVED_HEADER;
    int rc = WKV6_OK;
    auto ck = [&](cudaError_t e) { if (e != cudaSuccess && rc == WKV6_OK) { set_error("wkv6_bi backward: %s", cudaGetErrorString(e)); rc = WKV6_ECUDA; } };
    ck(cudaMemsetAsync(u0, 0, (size_t)a.H * N * sizeof(bf16), a.stream));
    if (rc == WKV6_OK) {
        bi_last_kernel<<<a.B, 256, 0, a.stream>>>(a.T, a.mask, row_len);
        bi_order_kernel<<<1, 256, 0, a.stream>>>(a.B, row_len, row_order);
        count_launch(2);
        ck(cudaGetLastError());
    }
    Args d = a;
    d.mask = nullptr;
    if (rc == WKV6_OK) rc = tc3_backward_bi(d, ckpt, flags, tc3::BI_CAUSAL, row_len, row_order);
    if (rc == WKV6_OK) rc = dbg_sync(a.stream, "backward, causal direction");
    if (rc == WKV6_OK) {
        d.u = u0; d.gu = gu2;
        rc = tc3_backward_bi(d, ckpt, flags, tc3::BI_REV, row_len, row_order);
    }
    if (rc == WKV6_OK) rc = dbg_sync(a.stream, "backward, reverse direction");
    cudaFreeAsync(sc, a.stream);
    return rc;
}

}  // namespace wkv6
