// Shared declarations of libwkv6_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <initializer_list>

#include "../../include/wkv6_b200.h"

namespace wkv6 {

constexpr int N = WKV6_HEAD_SIZE;  // head size, fixed like the reference's -D_N_=64

// how the decay tensor is encoded at the boundary
enum WKind : int {
    W_RAW_BF16 = 0,   // raw logits w, bf16           (wkv6state / wkv6infctx / RUN_CUDA_RWKV6)
    W_LOG_F32 = 1,    // l = -exp(w), fp32            (wkv6 / wkv6_bi native entry, src/model.py:210)
    W_DECAY_F32 = 2,  // d = exp(-exp(w)), fp32       (rwkv6 inference entry, src/model_run.py:64)
};

// Opt-in decay clamp (wkv6b200_set_decay_clamp): the per-token log-decay is floored at this many nats
// (a negative number; -inf = off).  Every Args picks up the setting current at its construction.
float decay_clamp_nats();

// One generic description of a WKV6 call; every C-ABI entry point fills one of these.
struct Args {
    int B = 0, T = 0, H = 0;
    float lmin = decay_clamp_nats();
    int io_dtype = WKV6_BF16;         // element type of r,k,v,u,y,(gy,g*)
    const void *r = nullptr, *k = nullptr, *v = nullptr, *u = nullptr;
    const void *w = nullptr;
    int w_kind = W_RAW_BF16;
    // initial state: nullptr (zero) | bf16/fp32 [.,H,64(value),64(key)], batch stride 0 or H*64*64
    const void *s0 = nullptr;
    int s0_f32 = 0;
    long long s0_bstride = 0;
    // final state out (may alias s0): nullptr | bf16/fp32 [B,H,64,64]
    void *sT = nullptr;
    int sT_f32 = 0;
    void *y = nullptr;
    // tensor-core forward: split Kh into bf16 hi + lo for the state update (wkv6_tc3_fwd.cu, KLO).  -1: decided by
    // whether THIS pass returns a state (sT); the forward entry points fix it for the whole call (every internal pass of
    // a segmented call then rounds like the unsegmented one).
    int hi_lo = -1;
    // bidirectional (wkv6_bi): mask int32 [B,T]; nullptr = plain causal op
    const int *mask = nullptr;
    // backward only
    const void *gy = nullptr;
    void *gr = nullptr, *gk = nullptr, *gv = nullptr, *gw = nullptr, *gu = nullptr, *gs = nullptr;
    void *gu_total = nullptr;         // training pair only: bf16 [C], sum of gu over the batch rows
    // training pair only: nullptr (the final state feeds nothing) | dL/dS_T, bf16/fp32 [B,H,64(value),64(key)]
    const void *gT = nullptr;
    int gT_f32 = 0;
    mutable bool gu_total_done = false;   // set by the route whose kernel added the rows itself
    void *workspace = nullptr;
    size_t workspace_bytes = 0;
    // SIMT kernels only: nullptr, or one device int per (b,h) stream: block `s` runs only when
    // stream_flags[s] != 0 (lets the exact fallback be enqueued without a host round trip)
    const int *stream_flags = nullptr;
    // training pair: forward fills it (gu arrival counters + bf16 chunk-start states), backward reads it
    void *saved = nullptr;
    cudaStream_t stream = nullptr;
};

// The tensor-core kernels floor the per-token log2-decay at -13 (tc3_common.cuh LCLAMP2); an opt-in clamp
// that is tighter wins.  Returned in log2 units (kernels) / nats (seg_decay).
inline float tc_lmin_nats(const Args &a) { return a.lmin > -13.0f * 0.6931471805599453f ? a.lmin : -13.0f * 0.6931471805599453f; }
inline float tc_lmin_log2(const Args &a) { return tc_lmin_nats(a) * 1.4426950408889634f; }

// implementations (each returns a WKV6_* code)
int simt_forward(const Args &a);
int simt_backward(const Args &a);
size_t simt_backward_workspace_bytes(int B, int T, int H);

// The tensor-core routes below take raw bf16 logits.  hz_flags / flags: nullptr (no stream is flagged), or one device int
// per (b,h) stream; the kernels skip the flagged streams, which the caller recomputes on the exact SIMT kernels.  Only the
// conversion of fp32 decays (capi.cu) flags streams: the tensor-core kernels never raise a flag.
//
// role-uniform tcgen05 forward.  nseg > 1: every sequence is cut into nseg segments of
// seg_chunks 64-token chunks (the last may be shorter) that run as separate grid rows; s0 / sT / flags / ckpt
// are then indexed by row = b*nseg + seg (seg_scan.cu)
// bi != 0: one direction of the bidirectional op (tc3_common.cuh BI_CAUSAL / BI_REV) with per-row lengths row_len[B]
// (+ row_order[B]: the batch rows sorted by length, longest first)
int tc3_forward(const Args &a, void *ckpt, int *hz_flags, int nseg = 1, int seg_chunks = 0, int bi = 0,
                const int *row_len = nullptr, const int *row_order = nullptr);
bool tc3_forward_supported(const Args &a);
// role-uniform tcgen05 backward
int tc3_backward(const Args &a, int *flags = nullptr);
int tc3_backward_bi(const Args &a, void *ckpt, int *flags, int bi, const int *row_len, const int *row_order);
// wkv6_bi forward and backward, both directions on the chunked tensor-core kernels
int bi_forward_tc(const Args &a, int *flags);
bool bi_forward_tc_supported(const Args &a);
int bi_backward_tc(const Args &a, int *flags);
// fp32 ew = -exp(w) (or decay = exp(-exp(w)) with from_decay) -> raw bf16 logits; raises flags[b*H+h] where the round trip is not exact
int ew_to_raw_bf16(int B, int T, int H, const float *ew, void *w_raw, int *flags, cudaStream_t stream, int from_decay = 0);
bool tc3_backward_supported(const Args &a);
// `saved` of the training pair and the backward's own copy of it: the per-head arrival counters of the in-kernel gu sum
// (H <= 512), then the bf16 chunk-start states
constexpr size_t TC3_SAVED_HEADER = 512 * sizeof(int);
size_t tc3_saved_bytes(int B, int T, int H);
size_t tc3_backward_workspace_bytes(int B, int T, int H, bool has_saved);

void set_error(const char *fmt, ...);
void count_launch(int n = 1);

// The memory-bound kernels read and write caller tensors with single 16-byte accesses, so their entry points reject a
// pointer that is not 16-byte aligned (a contiguous view at an element offset is not) before anything is launched.
// nullptr passes (optional arguments).  On failure the error names the entry and the first misaligned argument.
struct NamedPtr { const char *name; const void *p; };
inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline bool check_aligned16(const char *fn, std::initializer_list<NamedPtr> args) {
    for (const NamedPtr &a : args)
        if (!aligned16(a.p)) {
            set_error("%s: %s is not 16-byte aligned", fn, a.name);
            return false;
        }
    return true;
}

#define WKV6_CUDA_CHECK(expr)                                                            \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            ::wkv6::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),    \
                              __FILE__, __LINE__);                                       \
            return WKV6_ECUDA;                                                           \
        }                                                                                \
    } while (0)

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T x);
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }
template <> __device__ __forceinline__ float to_f32<__half>(__half x) { return __half2float(x); }
template <> __device__ __forceinline__ float to_f32<float>(float x) { return x; }

template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }
template <> __device__ __forceinline__ __half from_f32<__half>(float x) { return __float2half_rn(x); }
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }

// log-decay l = log d (<= 0) from whatever the boundary carries
template <int WK> __device__ __forceinline__ float load_logdecay(const void *w, size_t idx, float lmin) {
    float l;
    if (WK == W_RAW_BF16) l = -__expf(__bfloat162float(((const __nv_bfloat16 *)w)[idx]));
    else if (WK == W_LOG_F32) l = ((const float *)w)[idx];
    else l = __logf(fmaxf(((const float *)w)[idx], 1e-38f));
    return fmaxf(l, lmin);
}

// ddlerp_tma.cu: TMA-fed token-shift ddlerp backward (nout = 5 with m, or 1 / 2 without).  The caller has checked
// C % 8 == 0, the pointer alignment and, with m, 5*B <= INT_MAX (the five m planes are one tensor map of 5*B rows).
// Returns WKV6_OK or an error.
size_t ddlerp_tma_partial_slots(int nout, int B, int T, int C);
int ddlerp_backward_tma(int nout, int B, int T, int C, const void *x, const void *shift, const void *maa, const void *m,
                        const void *const *gouts, void *gx, void *gm, void *gshift, float *partial, int *slots,
                        cudaStream_t stream);
// seg_scan.cu: time-axis segmentation for calls with few streams (see the file header)
void ensure_pool_keeps_memory();   // cudaMallocAsync scratch stays cached in the device pool
void seg_plan(int B, int T, int H, int *nseg, int *seg_chunks);
void seg_plan_train(int B, int T, int H, int *nseg, int *seg_chunks);
int seg_reverse3(int B, int T, int C, int nseg, int seg_tokens, const void *a, const void *b, const void *c, void *ra, void *rb,
                 void *rc, cudaStream_t stream);
int seg_sum_gu(int B, int nseg, int C, const void *part, void *gu, cudaStream_t stream);
int seg_decay(int B, int T, int C, int nseg, int seg_tokens, const void *w, float *lam, float lmin, cudaStream_t stream);
int seg_scan(int B, int nseg, int H, const float *lam, const float *s_loc, const void *s0, int s0_f32,
             long long s0_bstride, float *s_start, void *sT, int sT_f32, int reverse, const int *stream_flags,
             cudaStream_t stream);
int seg_flags_merge(int B, int nseg, int H, int *seg_flags, int *stream_flags, cudaStream_t stream);
// ddlerp_lora.cu: ddlerp forward with the LoRA product on the tensor cores
bool ddlerp_lora_supported(int B, int T, int C, int R);
int ddlerp_lora_forward(int B, int T, int C, const void *x, const void *shift, const void *maa, const void *h,
                        const void *w2, void *out, cudaStream_t stream);
}  // namespace wkv6
