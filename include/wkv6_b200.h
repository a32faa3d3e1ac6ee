/* wkv6_b200.h -- C ABI of the B200-native WKV6 hot path (libwkv6_b200.so).
 *
 * Drop-in boundary for yynil/RWKV_LM_EXT.  Every entry point replaces one launcher the
 * reference's pybind modules bind (file:line cited per function).  Plain pointers and sizes only:
 * no torch types.  All pointers are DEVICE pointers unless marked "host".  Every function
 *   - returns 0 on success, a negative WKV6_E* code otherwise (wkv6b200_last_error() has text);
 *   - is asynchronous: work is enqueued on `stream` (a cudaStream_t; NULL = legacy default
 *     stream, which is what the reference's bare <<<>>> launches use, cuda/wkv6_cuda.cu:233);
 *   - the caller owns every buffer, including the workspace (size from the matching
 *     *_workspace_bytes) -- the reference wrappers likewise pre-allocate all outputs with
 *     torch.empty (src/model.py:211,225-230).  The library keeps no device memory of its own: what
 *     an entry needs beyond its arguments is stream-ordered scratch (cudaMallocAsync, e.g. wkv6_forward).
 *
 * Layout contract (identical to the reference): r,k,v,w,y,gy,g* are [B,T,C] contiguous,
 * C = H*64 (head size is fixed at 64 like -D_N_=64, src/model.py:189); u is [H,64];
 * states are [.,H,64(value j),64(key i)] (cuda/wkv6state_cuda.cu:15,24).
 */
#ifndef WKV6_B200_H
#define WKV6_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* exported symbol (the library is built with -fvisibility=hidden) */
#if defined(__GNUC__)
#define WKV6_API __attribute__((visibility("default")))
#else
#define WKV6_API
#endif

#define WKV6_HEAD_SIZE 64

/* error codes */
#define WKV6_OK            0
#define WKV6_EINVAL       -1   /* bad shape / null pointer / C != H*64 */
#define WKV6_EWORKSPACE   -2   /* workspace too small */
#define WKV6_ECUDA        -3   /* CUDA runtime / driver error (text in wkv6b200_last_error) */
#define WKV6_EUNSUPPORTED -4   /* the selected implementation cannot run this shape */

/* element types of r,k,v,u,y for the inference entry (cuda/rwkv6_op.cpp:12-34) */
#define WKV6_BF16 0
#define WKV6_FP16 1
#define WKV6_FP32 2

/* route of the WKV6 recurrence, see wkv6b200_set_impl; it selects nothing else (every other kernel has one route) */
#define WKV6_IMPL_AUTO 0       /* tensor-core chunked kernels where the shape allows, else SIMT */
#define WKV6_IMPL_SIMT 1       /* exact fp32 step recurrence on CUDA cores (all shapes)          */
#define WKV6_IMPL_TC   2       /* tcgen05/TMA chunked kernels only; WKV6_EUNSUPPORTED otherwise  */

WKV6_API int         wkv6b200_abi_version(void);
/* How a call with B*H streams of T tokens is cut along the time axis when it has too few streams to fill the
 * GPU (csrc/seg_scan.cu): nseg segments of seg_chunks 64-token chunks, the last one possibly shorter;
 * nseg = 1 = not segmented.  training != 0: the forward/backward pair.  Host logic only. */
WKV6_API void        wkv6b200_seg_plan(int B, int T, int H, int training, int *nseg, int *seg_chunks);
WKV6_API const char *wkv6b200_last_error(void);              /* host string, thread-local */
WKV6_API int         wkv6b200_set_impl(int impl);            /* returns the previous value */
WKV6_API int         wkv6b200_get_impl(void);
/* number of kernels this library launched since process start (bench.py's gpu_launches) */
WKV6_API uint64_t    wkv6b200_launch_count(void);
/* Opt-in: floor the per-token log-decay at -nats_per_token, i.e. compute with w' = min(w, log(nats_per_token))
 * (and a zero w-gradient where the floor is active).  A channel that decays faster than e^-3.7 per token keeps
 * < 2.5 % of the previous token; with a floor of 3.7 no stream can exceed what the tensor-core kernels' block
 * references allow, so none is handed to the (much slower) exact kernels.  This CHANGES the function for such
 * channels: it is off by default (0 turns it off again).  Returns the previous setting (0 = off).  Process-wide;
 * applies to every entry point, the exact kernels included.  Environment: WKV6_B200_DECAY_CLAMP=3.7. */
WKV6_API float       wkv6b200_set_decay_clamp(float nats_per_token);

/* ------------------------------------------------------------------------------------------
 * (a1/a2) wkv6 -- replaces cuda_forward / cuda_backward of cuda/wkv6_cuda.cu:229-242, bound by
 * cuda/wkv6_op.cpp:8-22 as forward(B,T,C,H,r,k,v,w,u,y) / backward(...,gy,gr,gk,gv,gw,gu).
 * r,k,v,u,y,gy,gr,gk,gv,gw,gu: bf16.  ew: fp32 [B,T,C] = -exp(w) (src/model.py:210).
 * gu: [B,C] per-batch partials (the wrapper sums over B, src/model.py:232).
 * gw[:,0] and gw[:,T-1] are exact zeros (cuda/wkv6_cuda.cu:201,226).
 * Implementation note: the tensor-core kernels read raw bf16 logits, so these two entries first
 * recover them (bf16(log(-ew)), exact when ew was built from bf16 logits as src/model.py:210 does);
 * streams where that round trip is not exact are computed by the fp32 SIMT kernels from ew itself.
 * wkv6_forward has no workspace argument in the reference, so it takes B*T*C*2 + B*H*4 bytes of
 * stream-ordered scratch (cudaMallocAsync, kept cached) for the logits and one flag per (b,h) stream;
 * wkv6_backward keeps both in its workspace.
 * ------------------------------------------------------------------------------------------ */
WKV6_API int wkv6_forward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                 const float *ew, const void *u, void *y, void *stream);
WKV6_API size_t wkv6_backward_workspace_bytes(int B, int T, int C, int H);
WKV6_API int wkv6_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                  const float *ew, const void *u, const void *gy, void *gr, void *gk, void *gv,
                  void *gw, void *gu, void *workspace, size_t workspace_bytes, void *stream);

/* Same operator taking the raw bf16 decay logits w (what RUN_CUDA_RWKV6 receives,
 * src/model.py:235) so the host wrapper can skip the three fp32 elementwise passes that build
 * `ew`.  gw is d/d(raw w) in both forms. */
WKV6_API int wkv6_forward_raww(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                      const void *w, const void *u, void *y, void *stream);
WKV6_API int wkv6_backward_raww(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                       const void *w, const void *u, const void *gy, void *gr, void *gk, void *gv,
                       void *gw, void *gu, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * Training pair behind the torch.autograd.Function wrappers (WKV_6 src/model.py:191-233, WKV_6STATE
 * :137-182 and :83-128): the reference forward keeps r,k,v,w,u(,s) for backward with
 * ctx.save_for_backward and its backward re-runs the whole state recurrence; here the forward also
 * leaves, in `saved` (caller-owned, wkv6_saved_bytes), the bf16 state at the start of every
 * 64-token chunk, and the backward consumes it instead of recomputing it.
 *   s0: NULL (zero state) | [H,64,64] (s0_batched = 0, wkv6state) | [B,H,64,64] (s0_batched = 1,
 *       wkv6infctx); bf16, or fp32 in the forward when s0_f32.  sT: NULL or [B,H,64,64] final state
 *       out (may alias s0).  *saved_valid (host int) is set to 1 when `saved` was filled; pass
 *       saved = NULL to wkv6_train_backward otherwise (it then recomputes, needing the larger
 *       workspace of wkv6_backward_workspace_bytes).  gs: NULL iff s0 is NULL, else bf16 [B,H,64,64].
 *   gu: bf16 [B,C], one row per sample like the reference's launcher (src/model.py:232 then sums over B);
 *       gu_total: NULL, or bf16 [C] that receives that sum (fp32 accumulation over the bf16 rows, what
 *       torch.sum(gu, 0) computes) from the backward kernel itself -- the last CTA of every head adds the rows.
 * `saved` is opaque: its layout depends on how the pair schedules the call (few (b,h) streams and T >= 2048:
 * both directions run as time segments, wkv6b200_seg_plan), so it must go to the backward of the same
 * B, T, H and the same library; the workspace then also holds the segmented backward's scratch.
 * ------------------------------------------------------------------------------------------ */
WKV6_API size_t wkv6_saved_bytes(int B, int T, int C, int H);
WKV6_API size_t wkv6_train_backward_workspace_bytes(int B, int T, int C, int H, int has_saved);
WKV6_API int wkv6_train_forward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                       const void *w, const void *u, const void *s0, int s0_batched, int s0_f32,
                       void *sT, int sT_f32, void *y, void *saved, int *saved_valid, void *stream);
WKV6_API int wkv6_train_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                        const void *w, const void *u, const void *s0, int s0_batched, const void *gy,
                        void *gr, void *gk, void *gv, void *gw, void *gu, void *gu_total, void *gs,
                        const void *saved, void *workspace, size_t workspace_bytes, void *stream);
/* The same backward when the loss also depends on the final state S_T (chunked long-context training that
 * carries the state from one chunk to the next and lets its gradient flow back): gT = dL/dS_T, bf16
 * (gT_f32 = 0) or fp32 (gT_f32 = 1) [B,H,64(value),64(key)] like sT, 16-byte aligned, non-NULL (wkv6_train_backward
 * is this call with gT = NULL).  The reverse sweep starts from gT instead of 0, so gw[:,T-1] is no longer forced
 * to 0 (the last decay feeds the final state); it is an exact 0 again where gT is 0.  Same `saved` and workspace as wkv6_train_backward;
 * the exact SIMT route (wkv6b200_set_impl) takes B*H*64*4 bytes of stream-ordered scratch on top. */
WKV6_API int wkv6_train_backward_state_grad(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                                   const void *w, const void *u, const void *s0, int s0_batched, const void *gy,
                                   void *gr, void *gk, void *gv, void *gw, void *gu, void *gu_total, void *gs,
                                   const void *gT, int gT_f32, const void *saved, void *workspace,
                                   size_t workspace_bytes, void *stream);
/* The same backward with the precision of dL/dS_0 chosen by the caller: gs is bf16 (gs_f32 = 0) or fp32
 * (gs_f32 = 1) [B,H,64(value),64(key)], non-NULL and 16-byte aligned.  A reverse sweep over many chunks hands each
 * chunk's dL/dS_0 to the previous chunk as its gT; with gs_f32 = 1 that carry is never rounded to bf16, like the
 * fp32 state carry of the forward (sT_f32).  gT may be NULL here (the last chunk: no final-state gradient); gT_f32
 * and gs_f32 must be 0 or 1.  Same `saved` and workspace as wkv6_train_backward. */
WKV6_API int wkv6_train_backward_state_grad_ex(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                                      const void *w, const void *u, const void *s0, int s0_batched, const void *gy,
                                      void *gr, void *gk, void *gv, void *gw, void *gu, void *gu_total,
                                      const void *gT, int gT_f32, void *gs, int gs_f32, const void *saved,
                                      void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * (a3) wkv6state -- cuda/wkv6state_cuda.cu:298-311 bound by cuda/wkv6state_op.cpp:8-21.
 * w: raw bf16 logits.  s: bf16 [H,64,64], shared by the batch, read-only.
 * gs: bf16 [B,H,64,64] per-batch partials (wrapper sums over B, src/model.py:182).
 * Gradients are those of the mathematical operator (fp64-autograd parity); the reference
 * kernel_backward_111 mis-indexes `s` (cuda/wkv6state_cuda.cu:79,91) -- not reproduced.
 * ------------------------------------------------------------------------------------------ */
WKV6_API int wkv6state_forward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                      const void *w, const void *u, const void *s, void *y, void *stream);
WKV6_API int wkv6state_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                       const void *w, const void *u, const void *s, const void *gy, void *gr,
                       void *gk, void *gv, void *gw, void *gu, void *gs, void *workspace,
                       size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * (a4) wkv6infctx -- cuda/wkv6infctx_cuda.cu:298-311 bound by cuda/wkv6infctx_op.cpp:8-22.
 * s: bf16 [B,H,64,64]; forward OVERWRITES it with the final state (cuda/wkv6infctx_cuda.cu:65-67).
 * backward takes the INITIAL state (the reference wrapper hands its kernel the mutated tensor,
 * src/model.py:104-106 -- a defect; the host wrapper here keeps a copy of the initial state).
 * wkv6infctx_forward_f32state: same with an fp32 state that is carried without the bf16 round trip.
 * ------------------------------------------------------------------------------------------ */
WKV6_API int wkv6infctx_forward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                       const void *w, const void *u, void *s, void *y, void *stream);
WKV6_API int wkv6infctx_forward_f32state(int B, int T, int C, int H, const void *r, const void *k,
                                const void *v, const void *w, const void *u, float *s, void *y,
                                void *stream);
WKV6_API int wkv6infctx_backward(int B, int T, int C, int H, const void *r, const void *k, const void *v,
                        const void *w, const void *u, const void *s_initial, const void *gy,
                        void *gr, void *gk, void *gv, void *gw, void *gu, void *gs,
                        void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * (a5) wkv6_bi -- cuda/wkv6_bi_cuda.cu:363-376 bound by cuda/wkv6_bi_op.cpp:8-21.
 * mask: int32 [B,T].  p[b] = first t with mask==0, or T-1.  y[t>p] = 0 (reference: unwritten).
 * ew: fp32 -exp(w).  Backward = gradient of this forward (SURVEY.md section 8c).
 * Implementation: two runs of the chunked tensor-core kernels (tokens as they are / each row's first
 * p+1 tokens reversed with u = 0) around a reverse-gather and a combine pass; they take B*T*C*2 x 5
 * (forward) or x 10 (backward) bytes of stream-ordered scratch (cudaMallocAsync).
 * ------------------------------------------------------------------------------------------ */
WKV6_API int wkv6_bi_forward(int B, int T, int C, int H, const int *mask, const void *r, const void *k,
                    const void *v, const float *ew, const void *u, void *y, void *stream);
WKV6_API int wkv6_bi_backward(int B, int T, int C, int H, const int *mask, const void *r, const void *k,
                     const void *v, const float *ew, const void *u, const void *gy, void *gr,
                     void *gk, void *gv, void *gw, void *gu, void *workspace,
                     size_t workspace_bytes, void *stream);
WKV6_API int wkv6_bi_forward_raww(int B, int T, int C, int H, const int *mask, const void *r,
                         const void *k, const void *v, const void *w, const void *u, void *y,
                         void *stream);
WKV6_API int wkv6_bi_backward_raww(int B, int T, int C, int H, const int *mask, const void *r,
                          const void *k, const void *v, const void *w, const void *u,
                          const void *gy, void *gr, void *gk, void *gv, void *gw, void *gu,
                          void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * (a6) rwkv6 inference -- cuda/rwkv6.cu:73-87 bound by cuda/rwkv6_op.cpp:12-34
 * (forward_bf16 / forward_fp16 / forward_fp32).  state: fp32 [B,H,64,64] in and out (the
 * reference is only correct for B = 1, cuda/rwkv6.cu:17; here every batch row has its own state).
 * w_decay: fp32 [B,T,C] = exp(-exp(w)) (src/model_run.py:64).  dtype: WKV6_BF16/FP16/FP32.
 * ------------------------------------------------------------------------------------------ */
WKV6_API int rwkv6_forward(int dtype, int B, int T, int C, int H, float *state, const void *r,
                  const void *k, const void *v, const float *w_decay, const void *u, void *y,
                  void *stream);
/* The same op for a caller that still holds the raw bf16 decay logits w (what `RWKV_6.forward`,
 * src/model_run.py:58-66, starts from before it materialises exp(-exp(w.float()))): no fp32 decay tensor is
 * built (2 eager passes and 4 B/element saved) and nothing has to be recovered from it.  bf16 r,k,v,w,u,y. */
WKV6_API int rwkv6_forward_raww(int B, int T, int C, int H, float *state, const void *r,
                       const void *k, const void *v, const void *w, const void *u, void *y,
                       void *stream);

/* ------------------------------------------------------------------------------------------
 * Memory-bound neighbours of the recurrence.
 * Their kernels read and write tensors with 16-byte vector accesses: every tensor argument of these
 * entries, and of their gradients and the channel-mix pieces below, must start at a 16-byte aligned
 * address (a contiguous view at an element offset, x[1:], does not).  A misaligned pointer is rejected
 * with WKV6_EINVAL, naming the argument, before anything is launched.  int64 index tensors, fp32
 * pooling outputs, fp32 parameter gradients and workspaces are exempt, and so are gather_rows_bf16,
 * gather_tokens_bf16 and pooling_bf16 when D % 8 != 0 (they then copy element by element).
 * ------------------------------------------------------------------------------------------ */
/* (a9) pos[b] = first t with idx[b,t]==token_id, 0 if absent
 * (== torch.eq(idx,id).int().argmax(-1), src/model_ext.py:209,1765); idx int64 [B,T]; pos int64 [B]. */
WKV6_API int eos_index_i64(int B, int T, const int64_t *idx, int64_t token_id, int64_t *pos, void *stream);
/* out[b,:] = x[b,pos[b],:]  (src/model_ext.py:210-211); x bf16 [B,T,D], out bf16 [B,D]. */
WKV6_API int gather_rows_bf16(int B, int T, int D, const void *x, const int64_t *pos, void *out,
                     void *stream);
/* (a10) pooling (src/model_ext.py:1708-1738, src/model_run.py:777-797).
 * kind: 0 weightedmean, 1 lasttoken, 2 avg.  variant: 0 train (L = actual_len), 1 infer
 * (L = actual_len + 1).  x bf16 [B,T,D]; actual_len int64 [B]; out_f32 fp32 [B,D] (the host
 * wrapper casts to bf16 where the reference does). */
WKV6_API int pooling_bf16(int kind, int variant, int B, int T, int D, const void *x,
                 const int64_t *actual_len, float *out_f32, void *stream);
/* (a12) mask = (idx != pad) & (idx != emb) as int32; rev_idx[b] = [len-1..0, len..T-1],
 * len = sum(mask[b]) (src/model_ext.py:398-417). */
WKV6_API int create_mask_rev_idx(int B, int T, const int64_t *idx, int64_t emb_id, int64_t pad_id,
                        int32_t *mask, int64_t *rev_idx, void *stream);
/* out[b,t,:] = x[b,rev_idx[b,t],:]  (reverse_x, src/model_ext.py:418-419); bf16 [B,T,D]. */
WKV6_API int gather_tokens_bf16(int B, int T, int D, const void *x, const int64_t *rev_idx, void *out,
                       void *stream);
/* out [2B,T,D]: out[b] = x[b], out[B + b] = reverse_x(x)[b] -- the plain and the reversed sequences of
 * bi_att_forward_batch (src/model_encoder_run.py:64-75) stacked as one batch, one read of x.  D % 8 == 0. */
WKV6_API int stack_reversed_bf16(int B, int T, int D, const void *x, const int64_t *rev_idx, void *out,
                        void *stream);

/* (a7) token-shift + ddlerp of RWKV_Tmix_x060.jit_func (src/model.py:437-449), mixing stage:
 * given x [B,T,C], the five data-dependent coefficients m [5,B,T,C] (output of the rank-R LoRA
 * bmm) and maa [5,C], writes xw,xk,xv,xr,xg = x + (shift(x)-x)*(maa_n + m_n) into out [5,B,T,C].
 * shift_state: NULL (zero pad) or bf16 [B,C] (infctx, src/model.py:738-745).  All bf16. */
WKV6_API int tmix_ddlerp_mix_bf16(int B, int T, int C, const void *x, const void *shift_state,
                         const void *maa, const void *m, void *out, void *stream);
/* The same with the rank-R LoRA product fused in (src/model.py:442-448): m_n = h_n @ W2_n is computed on
 * the tensor cores inside the kernel and never written to memory.  h bf16 [B*T, 5*R] = tanh(xxx @ W1)
 * (row-major, the five R-wide slices side by side), w2 bf16 [5,R,C], out bf16 [5,B,T,C].
 * R = 32 and C % 64 == 0 only (WKV6_EUNSUPPORTED otherwise: use a bmm + tmix_ddlerp_mix_bf16).
 * Misaligned tensors are WKV6_EINVAL, as for every entry of this section. */
WKV6_API int tmix_ddlerp_lora_bf16(int B, int T, int C, int R, const void *x, const void *shift_state,
                          const void *maa, const void *h, const void *w2, void *out, void *stream);
/* xxx = x + (shift(x)-x)*maa_x  (src/model.py:439-441), the LoRA input.  bf16. */
WKV6_API int tmix_shift_lerp_bf16(int B, int T, int C, const void *x, const void *shift_state,
                         const void *maa_x, void *out, void *stream);
/* (a8) GroupNorm(H groups, eps) * g  of jit_func_2 (src/model.py:461-467).
 * y,g,out bf16 [B*T,C]; ln_w, ln_b bf16 [C].  gate_act: 0 = g is the gate itself; 1 = g is the
 * gate Linear's output and silu (src/model.py:454) is applied here, saving a pass over [B,T,C]. */
WKV6_API int groupnorm_gate_bf16(int BT, int C, int H, float eps, int gate_act, const void *y, const void *g,
                        const void *ln_w, const void *ln_b, void *out, void *stream);

/* The same for the bi-directional encoders (src/model_encoder_run.py:72-74): the normalised input is
 * (y + reverse_x(y_rev, rev_idx)) / 2, gathered and averaged inside the kernel.  rev_idx int64 [B,T]. */
WKV6_API int groupnorm_gate_pair_bf16(int B, int T, int C, int H, float eps, int gate_act, const void *y,
                             const void *y_rev, const int64_t *rev_idx, const void *g, const void *ln_w,
                             const void *ln_b, void *out, void *stream);

/* ------------------------------------------------------------------------------------------
 * Gradients of the memory-bound neighbours, so the fused forwards above can replace the eager
 * chains of src/model.py:434-468 / src/model_ext.py:1708-1738 inside a training graph.  Data
 * gradients are bf16 like their tensors; parameter gradients (sums over all B*T rows) are fp32
 * (deterministic two-stage reduction).  ws: caller-owned scratch of
 * elementwise_backward_workspace_bytes(B, T, C, nparam) bytes (nparam = 5 ddlerp, 1 shift-lerp,
 * 2 GroupNorm).  gshift (bf16 [B,C]) is written only when shift_state is given; may be NULL.
 * ------------------------------------------------------------------------------------------ */
WKV6_API size_t elementwise_backward_workspace_bytes(int B, int T, int C, int nparam);
/* gx [B,T,C], gm [5,B,T,C], gmaa fp32 [5,C] from the gradients of xw,xk,xv,xr,xg (five separate
 * [B,T,C] tensors: they come out of five different Linear backward passes).  B > INT_MAX / 5 is
 * rejected with WKV6_EINVAL: the kernel reads the m planes through one tensor map of 5*B rows. */
WKV6_API int tmix_ddlerp_mix_backward_bf16(int B, int T, int C, const void *x, const void *shift_state,
                                  const void *maa, const void *m, const void *gxw, const void *gxk,
                                  const void *gxv, const void *gxr, const void *gxg, void *gx, void *gm,
                                  float *gmaa, void *gshift, void *ws, size_t ws_bytes, void *stream);
WKV6_API int tmix_shift_lerp_backward_bf16(int B, int T, int C, const void *x, const void *shift_state,
                                  const void *maa_x, const void *gout, void *gx, float *gmaa_x,
                                  void *gshift, void *ws, size_t ws_bytes, void *stream);
/* gy, gg bf16 [B*T,C]; gln_w, gln_b fp32 [C], or both NULL (frozen affine parameters: their reduction is skipped;
 * the same holds for gmaa / gmaa_x / gmaa_kr of the other backward entries). */
WKV6_API int groupnorm_gate_backward_bf16(int BT, int C, int H, float eps, int gate_act, const void *y,
                                 const void *g, const void *ln_w, const void *ln_b, const void *gout, void *gy, void *gg,
                                 float *gln_w, float *gln_b, void *ws, size_t ws_bytes, void *stream);
/* gx[b,t,:] = gout[b,:] * weight(t) / L inside the pooled range, 0 outside (kind 0 or 2). */
WKV6_API int pooling_backward_bf16(int kind, int variant, int B, int T, int D, const int64_t *actual_len,
                          const float *gout_f32, void *gx, void *stream);
/* gradient of gather_rows_bf16: gx[b,t,:] = (t == pos[b]) ? gout[b,:] : 0.  Writes all of gx. */
WKV6_API int scatter_rows_bf16(int B, int T, int D, const void *gout, const int64_t *pos, void *gx,
                      void *stream);
/* gradient of gather_tokens_bf16 for a per-row permutation (what reverse_x_idx builds):
 * gx[b,rev_idx[b,t],:] = gout[b,t,:]. */
WKV6_API int scatter_tokens_bf16(int B, int T, int D, const void *gout, const int64_t *rev_idx, void *gx,
                        void *stream);
/* gradient of groupnorm_gate_pair_bf16.  With G = the bf16 gradient of the averaged GroupNorm input (what
 * groupnorm_gate_backward_bf16 writes for it):  gy[b,t] = G[b,t] / 2,  gy_rev[b, rev_idx[b,t]] = G[b,t] / 2,  gg and
 * gln_w / gln_b (fp32 [C], or both NULL when frozen) as groupnorm_gate_backward_bf16 -- one pass, the average recomputed
 * as the forward computes it.  gy and gy_rev may be the two halves of one [2B,T,C] buffer (the gradient of one WKV6 call
 * over both directions).  rev_idx is a per-row permutation (what create_mask_rev_idx builds), else rows of gy_rev no
 * entry points at are left unwritten; an entry outside [0, T) writes nothing.  B*T <= INT_MAX.
 * ws: elementwise_backward_workspace_bytes(B, T, C, 2) bytes. */
WKV6_API int groupnorm_gate_pair_backward_bf16(int B, int T, int C, int H, float eps, int gate_act, const void *y,
                                      const void *y_rev, const int64_t *rev_idx, const void *g, const void *ln_w,
                                      const void *ln_b, const void *gout, void *gy, void *gy_rev, void *gg,
                                      float *gln_w, float *gln_b, void *ws, size_t ws_bytes, void *stream);
/* gradient of stack_reversed_bf16:  gx[b,t,:] = gxx[b,t,:] + gxx[B+b, rev_idx[b,t],:]  (one bf16 rounding), gxx [2B,T,D].
 * Precondition: rev_idx is a per-row involution (rev[b, rev[b,t]] == t), as create_mask_rev_idx builds it; the
 * scatter of the reversed half is then this gather.  An entry outside [0, T) reads gxx[B+b, t].  D % 8 == 0,
 * 2*B*T <= INT_MAX. */
WKV6_API int stack_reversed_backward_bf16(int B, int T, int D, const void *gxx, const int64_t *rev_idx, void *gx,
                                 void *stream);

/* ------------------------------------------------------------------------------------------
 * Channel mix (RWKV_CMix_x060.forward, src/model.py:635-644; infctx :804-812): the elementwise pieces
 * around its two GEMMs, bit-identical to the eager bf16 chain.
 * ------------------------------------------------------------------------------------------ */
/* out[0] = xk, out[1] = xr = x + (shift(x)-x) * time_maa_{k,r};  maa_kr bf16 [2,C];  out bf16 [2,B,T,C]. */
/* Residual add + LayerNorm (the glue of `Block.forward`, src/model.py:904-933), rows = B*T, D % 256 == 0:
 *   x_new = bf16(x + delta);  y = LayerNorm(x_new; w, b, eps)   (fp32 statistics, bf16 result)
 * delta == NULL: plain LayerNorm of x (x_new unused).  stats: NULL or fp32 [rows][2] receiving (mean, rstd) for the backward. */
WKV6_API int add_layernorm_bf16(long long rows, int D, float eps, const void *x, const void *delta, const void *w,
                       const void *b, void *x_new, void *y, float *stats, void *stream);
WKV6_API size_t add_layernorm_backward_workspace_bytes(long long rows, int D);
/* g = g_xnew + dLN(g_y): the gradient of BOTH x and delta (g_xnew may be NULL).  gw / gb: fp32 [D] or both NULL
 * (frozen affine parameters: the column pass is skipped); workspace only needed for gw / gb. */
WKV6_API int add_layernorm_backward_bf16(long long rows, int D, const void *x_new, const float *stats, const void *w,
                                const void *g_y, const void *g_xnew, void *g, float *gw, float *gb,
                                void *workspace, size_t workspace_bytes, void *stream);
WKV6_API int cmix_shift_lerp2_bf16(int B, int T, int C, const void *x, const void *shift_state,
                          const void *maa_kr, void *out, void *stream);
/* ws: elementwise_backward_workspace_bytes(B, T, C, 3) bytes; gmaa_kr fp32 [2,C]. */
WKV6_API int cmix_shift_lerp2_backward_bf16(int B, int T, int C, const void *x, const void *shift_state,
                                   const void *maa_kr, const void *gxk, const void *gxr, void *gx,
                                   float *gmaa_kr, void *gshift, void *ws, size_t ws_bytes, void *stream);
/* y = relu(x)^2 and its gradient gx = 2 relu(x) gy;  n elements (n % 8 == 0). */
WKV6_API int relu_sq_bf16(size_t n, const void *x, void *y, void *stream);
WKV6_API int relu_sq_backward_bf16(size_t n, const void *x, const void *gy, void *gx, void *stream);
/* out = sigmoid(r) * kv and its gradients. */
WKV6_API int sigmoid_mul_bf16(size_t n, const void *r, const void *kv, void *out, void *stream);
WKV6_API int sigmoid_mul_backward_bf16(size_t n, const void *r, const void *kv, const void *gout, void *gr,
                              void *gkv, void *stream);

/* ------------------------------------------------------------------------------------------
 * SFT loss (src/model.py:1244-1283 `training_step`, my_qa_mask == 0 branch, + `L2Wrap` src/model.py:960-974) on bf16
 * logits [rows, V] (rows = B*T, V % 8 == 0, V <= 65536), fp32 arithmetic:
 *   mean_out[0] = mean over the rows with target != ignore_index of  logsumexp(x_row) - x_row[target];  mean_out[1] = their number
 *   row_stats fp32 [3][rows] (row loss, logsumexp, maximum) and row_argmax int [rows] are kept for the backward
 *   glogits[r,j] = gloss[0] * (softmax(x_r)_j - [j == target_r]) / mean_out[1]   (0 for an ignored row)
 *                  + [j == row_argmax[r]] * maximum_r * l2_factor                 (L2Wrap: l2_factor = 1e-4 / rows)
 * gloss: device fp32 scalar (the gradient arriving at the loss). */
WKV6_API int cross_entropy_l2wrap_bf16(long long rows, int V, const void *logits, const int64_t *targets, long long ignore_index,
                              float *row_stats, int *row_argmax, float *mean_out, void *stream);
WKV6_API int cross_entropy_l2wrap_backward_bf16(long long rows, int V, const void *logits, const int64_t *targets,
                                       long long ignore_index, const float *row_stats, const int *row_argmax,
                                       const float *mean_out, const float *gloss, float l2_factor, void *glogits, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* WKV6_B200_H */
