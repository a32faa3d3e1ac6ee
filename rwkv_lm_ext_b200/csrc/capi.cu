// extern "C" entry points of libwkv6_b200.so -- see include/wkv6_b200.h for the contract.
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace wkv6 {

#ifdef WKV6_FINE_STAMPS
extern void *g_tc3_bwd_stamps;
#endif
static thread_local char g_err[512] = "";
static std::atomic<int> g_impl{-1};
static std::atomic<uint64_t> g_launches{0};
static std::atomic<float> g_lmin{-INFINITY};
float decay_clamp_nats() {
    static const bool env_read = [] {          // WKV6_B200_DECAY_CLAMP=3.7 in the environment == wkv6b200_set_decay_clamp(3.7)
        const char *e = getenv("WKV6_B200_DECAY_CLAMP");
        const float v = e ? (float)atof(e) : 0.f;
        if (v > 0.f) g_lmin.store(-v);
        return true;
    }();
    (void)env_read;
    return g_lmin.load(std::memory_order_relaxed);
}

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

static int current_impl() {
    int v = g_impl.load();
    if (v < 0) {
        const char *e = getenv("WKV6_B200_IMPL");   // "simt" | "tc" | "auto"
        v = WKV6_IMPL_AUTO;
        if (e && !strcmp(e, "simt")) v = WKV6_IMPL_SIMT;
        if (e && !strcmp(e, "tc")) v = WKV6_IMPL_TC;
        g_impl.store(v);
    }
    return v;
}

static int check_shape(int B, int T, int C, int H) {
    if (B < 0 || T < 0 || H <= 0 || C != H * N) {
        set_error("bad shape B=%d T=%d C=%d H=%d (need C == H*%d)", B, T, C, H, N);
        return WKV6_EINVAL;
    }
    return WKV6_OK;
}
#define REQUIRE_PTRS(...)                                                        \
    do {                                                                         \
        const void *_p[] = {__VA_ARGS__};                                        \
        for (size_t _i = 0; _i < sizeof(_p) / sizeof(_p[0]); _i++)               \
            if (!_p[_i]) { set_error("%s: null pointer argument #%zu", __func__, _i); return WKV6_EINVAL; } \
    } while (0)

// Forward over `nseg` time segments that run as separate grid rows (seg_scan.cu): state-only pass from zero
// states, scan over the segment states, ordinary pass with the scanned initial states.
// flags: nullptr, or the stream flags of the fp32-decay conversion ([B*H]); ckpt: nullptr, or (training pair) where
// the chunk-start states go.
static int tc3_forward_segmented(const Args &a, int *flags, int nseg, int seg_chunks, void *ckpt) {
    wkv6::ensure_pool_keeps_memory();
    const int Bs = a.B * nseg, C = a.H * 64, seg_tokens = seg_chunks * 64;
    const size_t st = (size_t)Bs * a.H * 4096, nl = (size_t)Bs * C, nf = (size_t)Bs * a.H;
    float *buf = nullptr;
    WKV6_CUDA_CHECK(cudaMallocAsync((void **)&buf, (2 * st + nl) * sizeof(float) + (flags ? nf * sizeof(int) : 0), a.stream));
    float *s_loc = buf, *s_start = buf + st, *lam = s_start + st;
    int *sflags = flags ? (int *)(lam + nl) : nullptr;      // the stream flags broadcast to the segment rows
    int rc = WKV6_OK;
    if (flags) {
        rc = cudaMemsetAsync(sflags, 0, nf * sizeof(int), a.stream) == cudaSuccess ? WKV6_OK : WKV6_ECUDA;
        if (rc == WKV6_OK) rc = seg_flags_merge(a.B, nseg, a.H, sflags, flags, a.stream);
    }
    Args a1 = a;
    a1.s0 = nullptr; a1.s0_bstride = 0; a1.sT = s_loc; a1.sT_f32 = 1; a1.y = nullptr; a1.saved = nullptr;
    if (rc == WKV6_OK) rc = tc3_forward(a1, nullptr, sflags, nseg, seg_chunks);
    if (rc == WKV6_OK) rc = seg_decay(a.B, a.T, C, nseg, seg_tokens, a.w, lam, tc_lmin_nats(a), a.stream);
    if (rc == WKV6_OK) rc = seg_scan(a.B, nseg, a.H, lam, s_loc, a.s0, a.s0_f32, a.s0_bstride, s_start, a.sT, a.sT_f32, 0, flags, a.stream);
    Args a2 = a;
    a2.s0 = s_start; a2.s0_f32 = 1; a2.s0_bstride = (long long)a.H * 4096; a2.sT = nullptr; a2.saved = nullptr;
    if (rc == WKV6_OK) rc = tc3_forward(a2, ckpt, sflags, nseg, seg_chunks);
    cudaFreeAsync(buf, a.stream);
    return rc;
}
// the tensor-core forward on raw bf16 logits; flags: nullptr, or the stream flags of the fp32-decay conversion
static int forward3(const Args &a, int *flags = nullptr) {
    void *ckpt = nullptr;
    if (a.saved) {
        // the training pair's header: per-head arrival counters of the backward's in-kernel gu reduction
        WKV6_CUDA_CHECK(cudaMemsetAsync(a.saved, 0, TC3_SAVED_HEADER, a.stream));
        ckpt = (uint8_t *)a.saved + TC3_SAVED_HEADER;
    }
    // the training pair segments forward and backward alike (the saved chunk states are in segment-row order)
    int nseg = 1, seg_chunks = 0;
    if (a.saved) seg_plan_train(a.B, a.T, a.H, &nseg, &seg_chunks);
    else seg_plan(a.B, a.T, a.H, &nseg, &seg_chunks);
    return nseg > 1 ? tc3_forward_segmented(a, flags, nseg, seg_chunks, ckpt) : tc3_forward(a, ckpt, flags);
}

// fp32 decays (-exp(w) of wkv6 / wkv6_bi, exp(-exp(w)) of rwkv6 inference): the tensor-core routes on the raw bf16
// logits they convert to, then the exact SIMT kernels on the original values for the streams where that conversion is
// not lossless (the only streams that are ever flagged)
static Args with_raw_w(const Args &a, void *w_raw) {
    Args t = a;
    t.w = w_raw;
    t.w_kind = W_RAW_BF16;
    return t;
}
static bool ew_convertible(const Args &a, bool backward) {
    if ((a.w_kind != W_LOG_F32 && a.w_kind != W_DECAY_F32) || a.saved) return false;
    const Args t = with_raw_w(a, const_cast<void *>(a.w));
    return bi_forward_tc_supported(t) || (backward ? tc3_backward_supported(t) : tc3_forward_supported(t));
}
static int forward_ew(const Args &a) {
    // the reference's entries have no workspace argument: stream-ordered scratch, kept cached in the pool
    wkv6::ensure_pool_keeps_memory();
    const size_t nw = (size_t)a.B * a.T * a.H * N * 2;
    uint8_t *buf = nullptr;
    WKV6_CUDA_CHECK(cudaMallocAsync((void **)&buf, nw + (size_t)a.B * a.H * sizeof(int), a.stream));
    int *flags = (int *)(buf + nw);
    int rc = cudaMemsetAsync(flags, 0, (size_t)a.B * a.H * sizeof(int), a.stream) == cudaSuccess ? WKV6_OK : WKV6_ECUDA;
    if (rc == WKV6_OK) rc = ew_to_raw_bf16(a.B, a.T, a.H, (const float *)a.w, buf, flags, a.stream, a.w_kind == W_DECAY_F32);
    if (rc == WKV6_OK) rc = a.mask ? bi_forward_tc(with_raw_w(a, buf), flags) : forward3(with_raw_w(a, buf), flags);
    if (rc == WKV6_OK) {
        Args s = a;
        s.stream_flags = flags;
        rc = simt_forward(s);
    }
    cudaFreeAsync(buf, a.stream);
    return rc;
}
static int backward_ew(const Args &a) {
    // workspace: [tensor-core backward workspace][raw bf16 logits][stream flags]
    const size_t base = tc3_backward_workspace_bytes(a.B, a.T, a.H, false), nw = (size_t)a.B * a.T * a.H * N * 2;
    const size_t need = base + nw + (size_t)a.B * a.H * sizeof(int);
    if (!a.workspace || a.workspace_bytes < need) { set_error("workspace too small: need %zu bytes", need); return WKV6_EWORKSPACE; }
    void *w_raw = (uint8_t *)a.workspace + base;
    int *flags = (int *)((uint8_t *)w_raw + nw);
    if (cudaMemsetAsync(flags, 0, (size_t)a.B * a.H * sizeof(int), a.stream) != cudaSuccess) { set_error("cudaMemsetAsync failed"); return WKV6_ECUDA; }
    if (int rc = ew_to_raw_bf16(a.B, a.T, a.H, (const float *)a.w, w_raw, flags, a.stream)) return rc;
    Args t = with_raw_w(a, w_raw);
    t.workspace_bytes = base;
    if (int rc = a.mask ? bi_backward_tc(t, flags) : tc3_backward(t, flags)) return rc;
    Args s = a;                   // (the exact route's scratch is the front of the workspace)
    s.stream_flags = flags;
    return simt_backward(s);
}

static int dispatch_forward(const Args &a0) {
    Args a = a0;
    if (a.hi_lo < 0) a.hi_lo = a.sT != nullptr;      // one precision class for every internal pass of this call
    const int impl = current_impl();
    if (impl != WKV6_IMPL_SIMT && tc3_forward_supported(a)) return forward3(a);
    if (impl != WKV6_IMPL_SIMT && bi_forward_tc_supported(a)) return bi_forward_tc(a, nullptr);
    if (impl != WKV6_IMPL_SIMT && ew_convertible(a, false)) return forward_ew(a);
    if (impl == WKV6_IMPL_TC) { set_error("tensor-core forward does not support this call"); return WKV6_EUNSUPPORTED; }
    return simt_forward(a);
}
static int dispatch_backward(const Args &a) {
    const int impl = current_impl();
    if (impl != WKV6_IMPL_SIMT && tc3_backward_supported(a)) return tc3_backward(a);
    if (impl != WKV6_IMPL_SIMT && bi_forward_tc_supported(a)) return bi_backward_tc(a, nullptr);
    if (impl != WKV6_IMPL_SIMT && ew_convertible(a, true)) return backward_ew(a);
    if (impl == WKV6_IMPL_TC) { set_error("tensor-core backward does not support this call"); return WKV6_EUNSUPPORTED; }
    return simt_backward(a);
}

}  // namespace wkv6

using namespace wkv6;

extern "C" {

int wkv6b200_abi_version(void) { return 4; }
float wkv6b200_set_decay_clamp(float nats_per_token) {
    const float prev = -decay_clamp_nats();
    g_lmin.store(nats_per_token > 0.f ? -nats_per_token : -INFINITY);
    return prev == INFINITY ? 0.f : prev;
}
// host logic only (no device access): the time-segmentation plan of a call, for tests and diagnostics
void wkv6b200_seg_plan(int B, int T, int H, int training, int *nseg, int *seg_chunks) {
    int n = 1, sc = 0;
    if (training) seg_plan_train(B, T, H, &n, &sc);
    else seg_plan(B, T, H, &n, &sc);
    if (nseg) *nseg = n;
    if (seg_chunks) *seg_chunks = sc;
}
const char *wkv6b200_last_error(void) { return g_err; }
int wkv6b200_set_impl(int impl) {
    int prev = current_impl();
    g_impl.store(impl);
    return prev;
}
int wkv6b200_get_impl(void) { return current_impl(); }
uint64_t wkv6b200_launch_count(void) { return g_launches.load(); }
#ifdef WKV6_FINE_STAMPS
// Profiling BUILD only (-DWKV6_FINE_STAMPS, profiles/stage_times.py; not in the product library): device buffer
// [B*H][chunks][32] of int64 that the backward kernel fills with clock64() stamps inside its stages; NULL = off.
__attribute__((visibility("default"))) void wkv6b200_debug_stamps(void *dev_buf) { wkv6::g_tc3_bwd_stamps = dev_buf; }
#endif

// ------------------------------------------------------------------------------------ wkv6
static int wkv6_fwd_common(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                           const void *w, int w_kind, const void *u, void *y, const int *mask, void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if ((size_t)B * T == 0) return WKV6_OK;
    REQUIRE_PTRS(r, k, v, w, u, y);
    Args a;
    a.B = B; a.T = T; a.H = H; a.r = r; a.k = k; a.v = v; a.w = w; a.w_kind = w_kind; a.u = u; a.y = y;
    a.mask = mask; a.stream = (cudaStream_t)stream;
    return dispatch_forward(a);
}
static int wkv6_bwd_common(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                           const void *w, int w_kind, const void *u, const void *s0, long long s0_bstride,
                           const void *gy, void *gr, void *gk, void *gv, void *gw, void *gu, void *gs,
                           const int *mask, void *ws, size_t ws_bytes, void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if ((size_t)B * T == 0) return WKV6_OK;
    REQUIRE_PTRS(r, k, v, w, u, gy, gr, gk, gv, gw, gu);
    Args a;
    a.B = B; a.T = T; a.H = H; a.r = r; a.k = k; a.v = v; a.w = w; a.w_kind = w_kind; a.u = u;
    a.s0 = s0; a.s0_bstride = s0_bstride; a.gy = gy; a.gr = gr; a.gk = gk; a.gv = gv; a.gw = gw;
    a.gu = gu; a.gs = gs; a.mask = mask; a.workspace = ws; a.workspace_bytes = ws_bytes;
    a.stream = (cudaStream_t)stream;
    return dispatch_backward(a);
}

int wkv6_forward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                 const float *ew, const void *u, void *y, void *stream) {
    return wkv6_fwd_common(B, T, C, H, r, k, v, ew, W_LOG_F32, u, y, nullptr, stream);
}
int wkv6_forward_raww(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                      const void *w, const void *u, void *y, void *stream) {
    return wkv6_fwd_common(B, T, C, H, r, k, v, w, W_RAW_BF16, u, y, nullptr, stream);
}
size_t wkv6_backward_workspace_bytes(int B, int T, int C, int H) {
    (void)C;
    // superset: SIMT scratch + chunk-start states (+ raw bf16 logits and per-stream flags for the fp32-ew entries)
    return tc3_backward_workspace_bytes(B, T, H, false) + (size_t)B * T * H * N * 2 + (size_t)B * H * sizeof(int);
}
int wkv6_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                  const float *ew, const void *u, const void *gy, void *gr, void *gk, void *gv,
                  void *gw, void *gu, void *workspace, size_t workspace_bytes, void *stream) {
    return wkv6_bwd_common(B, T, C, H, r, k, v, ew, W_LOG_F32, u, nullptr, 0, gy, gr, gk, gv, gw, gu,
                           nullptr, nullptr, workspace, workspace_bytes, stream);
}
int wkv6_backward_raww(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                       const void *w, const void *u, const void *gy, void *gr, void *gk, void *gv,
                       void *gw, void *gu, void *workspace, size_t workspace_bytes, void *stream) {
    return wkv6_bwd_common(B, T, C, H, r, k, v, w, W_RAW_BF16, u, nullptr, 0, gy, gr, gk, gv, gw, gu,
                           nullptr, nullptr, workspace, workspace_bytes, stream);
}

// ---------------------------------------------------------------------------- training pair
size_t wkv6_saved_bytes(int B, int T, int C, int H) {
    (void)C;
    return tc3_saved_bytes(B, T, H);
}
size_t wkv6_train_backward_workspace_bytes(int B, int T, int C, int H, int has_saved) {
    (void)C;
    return has_saved ? tc3_backward_workspace_bytes(B, T, H, true) + 1024 : wkv6_backward_workspace_bytes(B, T, C, H);
}
int wkv6_train_forward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                       const void *w, const void *u, const void *s0, int s0_batched, int s0_f32,
                       void *sT, int sT_f32, void *y, void *saved, int *saved_valid, void *stream) {
    if (saved_valid) *saved_valid = 0;
    if (int rc = check_shape(B, T, C, H)) return rc;
    if ((size_t)B * T == 0) return WKV6_OK;
    REQUIRE_PTRS(r, k, v, w, u, y);
    Args a;
    a.B = B; a.T = T; a.H = H; a.r = r; a.k = k; a.v = v; a.w = w; a.w_kind = W_RAW_BF16; a.u = u;
    a.s0 = s0; a.s0_f32 = s0_f32; a.s0_bstride = s0_batched ? (long long)H * N * N : 0;
    a.sT = sT; a.sT_f32 = sT_f32; a.y = y; a.stream = (cudaStream_t)stream;
    const bool save = saved && current_impl() != WKV6_IMPL_SIMT && tc3_forward_supported(a);
    if (save) a.saved = saved;
    const int rc = dispatch_forward(a);
    if (rc == WKV6_OK && save && saved_valid) *saved_valid = 1;
    return rc;
}
// the training pair's backward, with (gT) or without (gT = NULL) a gradient arriving at the final state
static int train_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v, const void *w,
                          const void *u, const void *s0, int s0_batched, const void *gy, void *gr, void *gk, void *gv,
                          void *gw, void *gu, void *gu_total, void *gs, int gs_f32, const void *gT, int gT_f32,
                          const void *saved, void *workspace, size_t workspace_bytes, void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if ((size_t)B * T == 0) return WKV6_OK;
    REQUIRE_PTRS(r, k, v, w, u, gy, gr, gk, gv, gw, gu);
    if (s0) REQUIRE_PTRS(gs);
    Args a;
    a.B = B; a.T = T; a.H = H; a.r = r; a.k = k; a.v = v; a.w = w; a.w_kind = W_RAW_BF16; a.u = u;
    a.s0 = s0; a.s0_bstride = s0_batched ? (long long)H * N * N : 0; a.gy = gy; a.gr = gr; a.gk = gk;
    a.gv = gv; a.gw = gw; a.gu = gu; a.gs = gs; a.workspace = workspace; a.workspace_bytes = workspace_bytes;
    a.gT = gT; a.gT_f32 = gT_f32; a.gs_f32 = gs_f32;
    a.saved = const_cast<void *>(saved);
    a.stream = (cudaStream_t)stream;
    a.gu_total = gu_total;
    const int rc = dispatch_backward(a);
    if (rc != WKV6_OK || !gu_total || a.gu_total_done) return rc;
    return seg_sum_gu(1, B, C, gu, gu_total, a.stream);      // routes whose kernels do not add the rows themselves
}
int wkv6_train_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                        const void *w, const void *u, const void *s0, int s0_batched, const void *gy,
                        void *gr, void *gk, void *gv, void *gw, void *gu, void *gu_total, void *gs,
                        const void *saved, void *workspace, size_t workspace_bytes, void *stream) {
    return train_backward(B, T, C, H, r, k, v, w, u, s0, s0_batched, gy, gr, gk, gv, gw, gu, gu_total, gs, 0, nullptr, 0,
                          saved, workspace, workspace_bytes, stream);
}
int wkv6_train_backward_state_grad(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                                   const void *w, const void *u, const void *s0, int s0_batched, const void *gy,
                                   void *gr, void *gk, void *gv, void *gw, void *gu, void *gu_total, void *gs,
                                   const void *gT, int gT_f32, const void *saved, void *workspace,
                                   size_t workspace_bytes, void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if (!gT) { set_error("%s: gT is NULL (wkv6_train_backward is the call without a final-state gradient)", __func__); return WKV6_EINVAL; }
    if (gT_f32 != 0 && gT_f32 != 1) { set_error("%s: gT_f32 = %d (0: bf16 gT, 1: fp32 gT)", __func__, gT_f32); return WKV6_EINVAL; }
    if (!check_aligned16(__func__, {{"gT", gT}})) return WKV6_EINVAL;
    return train_backward(B, T, C, H, r, k, v, w, u, s0, s0_batched, gy, gr, gk, gv, gw, gu, gu_total, gs, 0, gT, gT_f32,
                          saved, workspace, workspace_bytes, stream);
}
int wkv6_train_backward_state_grad_ex(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                                      const void *w, const void *u, const void *s0, int s0_batched, const void *gy,
                                      void *gr, void *gk, void *gv, void *gw, void *gu, void *gu_total,
                                      const void *gT, int gT_f32, void *gs, int gs_f32, const void *saved,
                                      void *workspace, size_t workspace_bytes, void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if (gT_f32 != 0 && gT_f32 != 1) { set_error("%s: gT_f32 = %d (0: bf16 gT, 1: fp32 gT)", __func__, gT_f32); return WKV6_EINVAL; }
    if (gs_f32 != 0 && gs_f32 != 1) { set_error("%s: gs_f32 = %d (0: bf16 gs, 1: fp32 gs)", __func__, gs_f32); return WKV6_EINVAL; }
    if (!gs) { set_error("%s: gs is NULL", __func__); return WKV6_EINVAL; }
    if (!check_aligned16(__func__, {{"gT", gT}, {"gs", gs}})) return WKV6_EINVAL;
    return train_backward(B, T, C, H, r, k, v, w, u, s0, s0_batched, gy, gr, gk, gv, gw, gu, gu_total, gs, gs_f32, gT, gT_f32,
                          saved, workspace, workspace_bytes, stream);
}

// ------------------------------------------------------------------------------- wkv6state
int wkv6state_forward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                      const void *w, const void *u, const void *s, void *y, void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if ((size_t)B * T == 0) return WKV6_OK;
    REQUIRE_PTRS(r, k, v, w, u, s, y);
    Args a;
    a.B = B; a.T = T; a.H = H; a.r = r; a.k = k; a.v = v; a.w = w; a.w_kind = W_RAW_BF16; a.u = u;
    a.s0 = s; a.s0_bstride = 0; a.y = y; a.stream = (cudaStream_t)stream;
    return dispatch_forward(a);
}
int wkv6state_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                       const void *w, const void *u, const void *s, const void *gy, void *gr,
                       void *gk, void *gv, void *gw, void *gu, void *gs, void *workspace,
                       size_t workspace_bytes, void *stream) {
    REQUIRE_PTRS(s, gs);
    return wkv6_bwd_common(B, T, C, H, r, k, v, w, W_RAW_BF16, u, s, 0, gy, gr, gk, gv, gw, gu, gs,
                           nullptr, workspace, workspace_bytes, stream);
}

// ------------------------------------------------------------------------------ wkv6infctx
static int infctx_fwd(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                      const void *w, const void *u, void *s, int f32, void *y, void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if ((size_t)B * T == 0) return WKV6_OK;
    REQUIRE_PTRS(r, k, v, w, u, s, y);
    Args a;
    a.B = B; a.T = T; a.H = H; a.r = r; a.k = k; a.v = v; a.w = w; a.w_kind = W_RAW_BF16; a.u = u;
    a.s0 = s; a.s0_f32 = f32; a.s0_bstride = (long long)H * N * N; a.sT = s; a.sT_f32 = f32;
    a.y = y; a.stream = (cudaStream_t)stream;
    return dispatch_forward(a);
}
int wkv6infctx_forward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                       const void *w, const void *u, void *s, void *y, void *stream) {
    return infctx_fwd(B, T, C, H, r, k, v, w, u, s, 0, y, stream);
}
int wkv6infctx_forward_f32state(int B, int T, int C, int H, const void *r, const void *k,
                                const void *v, const void *w, const void *u, float *s, void *y,
                                void *stream) {
    return infctx_fwd(B, T, C, H, r, k, v, w, u, s, 1, y, stream);
}
int wkv6infctx_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                        const void *w, const void *u, const void *s_initial, const void *gy,
                        void *gr, void *gk, void *gv, void *gw, void *gu, void *gs,
                        void *workspace, size_t workspace_bytes, void *stream) {
    REQUIRE_PTRS(s_initial, gs);
    return wkv6_bwd_common(B, T, C, H, r, k, v, w, W_RAW_BF16, u, s_initial, (long long)H * N * N, gy,
                           gr, gk, gv, gw, gu, gs, nullptr, workspace, workspace_bytes, stream);
}

// --------------------------------------------------------------------------------- wkv6_bi
int wkv6_bi_forward(int B, int T, int C, int H, const int *mask, const void *r, const void *k,
                    const void *v, const float *ew, const void *u, void *y, void *stream) {
    REQUIRE_PTRS(mask);
    return wkv6_fwd_common(B, T, C, H, r, k, v, ew, W_LOG_F32, u, y, mask, stream);
}
int wkv6_bi_forward_raww(int B, int T, int C, int H, const int *mask, const void *r,
                         const void *k, const void *v, const void *w, const void *u, void *y,
                         void *stream) {
    REQUIRE_PTRS(mask);
    return wkv6_fwd_common(B, T, C, H, r, k, v, w, W_RAW_BF16, u, y, mask, stream);
}
int wkv6_bi_backward(int B, int T, int C, int H, const int *mask, const void *r, const void *k,
                     const void *v, const float *ew, const void *u, const void *gy, void *gr,
                     void *gk, void *gv, void *gw, void *gu, void *workspace,
                     size_t workspace_bytes, void *stream) {
    REQUIRE_PTRS(mask);
    return wkv6_bwd_common(B, T, C, H, r, k, v, ew, W_LOG_F32, u, nullptr, 0, gy, gr, gk, gv, gw, gu,
                           nullptr, mask, workspace, workspace_bytes, stream);
}
int wkv6_bi_backward_raww(int B, int T, int C, int H, const int *mask, const void *r,
                          const void *k, const void *v, const void *w, const void *u,
                          const void *gy, void *gr, void *gk, void *gv, void *gw, void *gu,
                          void *workspace, size_t workspace_bytes, void *stream) {
    REQUIRE_PTRS(mask);
    return wkv6_bwd_common(B, T, C, H, r, k, v, w, W_RAW_BF16, u, nullptr, 0, gy, gr, gk, gv, gw, gu,
                           nullptr, mask, workspace, workspace_bytes, stream);
}

// ------------------------------------------------------------------------- rwkv6 inference
int rwkv6_forward(int dtype, int B, int T, int C, int H, float *state, const void *r,
                  const void *k, const void *v, const float *w_decay, const void *u, void *y,
                  void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if (dtype < WKV6_BF16 || dtype > WKV6_FP32) { set_error("bad dtype %d", dtype); return WKV6_EINVAL; }
    if ((size_t)B * T == 0) return WKV6_OK;
    REQUIRE_PTRS(state, r, k, v, w_decay, u, y);
    Args a;
    a.B = B; a.T = T; a.H = H; a.io_dtype = dtype; a.r = r; a.k = k; a.v = v; a.w = w_decay;
    a.w_kind = W_DECAY_F32; a.u = u; a.s0 = state; a.s0_f32 = 1; a.s0_bstride = (long long)H * N * N;
    a.sT = state; a.sT_f32 = 1; a.y = y; a.stream = (cudaStream_t)stream;
    return dispatch_forward(a);
}

int rwkv6_forward_raww(int B, int T, int C, int H, float *state, const void *r, const void *k,
                       const void *v, const void *w, const void *u, void *y, void *stream) {
    if (int rc = check_shape(B, T, C, H)) return rc;
    if ((size_t)B * T == 0) return WKV6_OK;
    REQUIRE_PTRS(state, r, k, v, w, u, y);
    Args a;
    a.B = B; a.T = T; a.H = H; a.io_dtype = WKV6_BF16; a.r = r; a.k = k; a.v = v; a.w = w;
    a.w_kind = W_RAW_BF16; a.u = u; a.s0 = state; a.s0_f32 = 1; a.s0_bstride = (long long)H * N * N;
    a.sT = state; a.sT_f32 = 1; a.y = y; a.stream = (cudaStream_t)stream;
    return dispatch_forward(a);
}

}  // extern "C"
