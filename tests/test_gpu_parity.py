"""Parity of the CUDA path (through the C ABI / the reference-shaped Python surface) against the
oracle.  Needs a B200: run with `pytest -m gpu`.  Tolerances are in tests/util.py."""
import os

import pytest
import torch

from tests.util import (BF16_MAXABS_REL, STATE_RELRMS, assert_bf16_close, load_golden, make_inputs, relrms)

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def M():
    import rwkv_lm_ext_b200 as M
    M.load()
    return M


@pytest.fixture(scope="module")
def O():
    from oracle import wkv6_oracle
    return wkv6_oracle


def _impls(M):
    # every forward test runs on both implementations once the tensor-core one exists
    return ["simt", "auto"]


def _run_fwd_bwd(M, r, k, v, w, u, gy):
    B, T, C = r.shape
    H = u.shape[0]
    leaves = [t.detach().clone().to(DEV).requires_grad_(True) for t in (r, k, v, w, u)]
    y = M.RUN_CUDA_RWKV6(B, T, C, H, *leaves)
    y.backward(gy.to(DEV))
    return y.detach(), [t.grad for t in leaves]


# ---------------------------------------------------------------------------------------------
# golden fixtures produced by the reference itself
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", ["simt", "auto"])
@pytest.mark.parametrize("name", ["wkv6_2x10x256_randn", "wkv6_2x150x128_decay"])
def test_golden_forward_backward(M, name, impl):
    c = load_golden(name)
    M.set_impl(impl)
    try:
        bf = lambda t: t.bfloat16()
        y, grads = _run_fwd_bwd(M, bf(c["r"]), bf(c["k"]), bf(c["v"]), bf(c["w"]), bf(c["u"]), bf(c["gy"]))
    finally:
        M.set_impl("auto")
    assert_bf16_close(y, c["y_run_rwkv6_forward"], f"{name} y vs run_rwkv6_forward")
    # the author's own bar (tests/test_cpu.py:290)
    assert torch.allclose(y.float().cpu(), c["y_run_rwkv6_forward"], atol=1e-2 + 2 ** -7 * c["y_run_rwkv6_forward"].abs().max().item())
    for g, key in zip(grads, ("gr", "gk", "gv", "gw", "gu")):
        assert_bf16_close(g, c[key], f"{name} {key}")


def test_golden_initial_state(M):
    c = load_golden("wkv6state_2x70x128")
    bf = lambda t: t.bfloat16().to(DEV)
    B, T, C = c["r"].shape
    H = 2
    s_vk = c["s0_kv"].transpose(-1, -2).contiguous()
    leaves = [bf(c[n]).requires_grad_(True) for n in ("r", "k", "v", "w", "u")]
    s = bf(s_vk).requires_grad_(True)
    s_work = s.clone()
    y, s_out = M.RUN_CUDA_RWKV6_STATE(B, T, C, H, *leaves, s_work)
    y.backward(bf(c["gy"]))
    assert_bf16_close(y, c["y_fla"], "state y")
    for t, key in zip(leaves, ("gr", "gk", "gv", "gw", "gu")):
        assert_bf16_close(t.grad, c[key], f"state {key}")
    assert_bf16_close(s.grad.transpose(-1, -2), c["gs_kv"], "state gs")


# ---------------------------------------------------------------------------------------------
# wkv6 forward / backward against the fp64 oracle, shapes around every tile boundary
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", ["simt", "auto", "tc"])
@pytest.mark.parametrize("decay", ["randn", "model"])
@pytest.mark.parametrize("B,T,H", [(1, 1, 1), (2, 2, 1), (1, 15, 2), (2, 16, 1), (1, 17, 1), (1, 63, 2),
                                   (2, 64, 2), (1, 65, 1), (1, 130, 3), (1, 257, 1)])
def test_wkv6_vs_oracle(M, O, B, T, H, decay, impl):
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=B * 1000 + T, decay=decay)
    ref = O.wkv6_backward(r, k, v, w, u, gy)
    M.set_impl(impl)
    try:
        y, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
    finally:
        M.set_impl("auto")
    assert_bf16_close(y, ref["y"], "y")
    for g, key in zip(grads, ("gr", "gk", "gv", "gw", "gu")):
        assert_bf16_close(g, ref[key], key)
    # exact zeros at the edges like cuda/wkv6_cuda.cu:201,226
    assert grads[3][:, 0].abs().max().item() == 0.0
    assert grads[3][:, -1].abs().max().item() == 0.0


def test_mixed_hazard_streams(M, O):
    """One (b,h) stream decays by far more than e^-60 inside 16 tokens, the others are model-like: the
    tensor-core kernels handle it themselves (16-token reference blocks + the 2^-13 per-token floor, no
    exact-route hand-off), forward and backward, through the training pair."""
    B, T, H = 2, 200, 2
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=11, decay="model")
    w[1, 40:120, 64:128] = 3.0            # stream (b=1, h=1): exp(3) = 20 nats per token
    ref = O.wkv6_backward(r, k, v, w, u, gy)
    y, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
    assert_bf16_close(y, ref["y"], "y")
    for g, key in zip(grads, ("gr", "gk", "gv", "gw", "gu")):
        assert_bf16_close(g, ref[key], key)
    # and the in-place state variant: the flagged stream's final state must come from the exact kernel
    s0 = (torch.randn(B, H, 64, 64, generator=torch.Generator().manual_seed(3)) * 0.5).bfloat16()
    y_ref, s_ref = O.wkv6infctx_forward(r, k, v, w, u, s0)
    s = s0.clone().to(DEV)
    with torch.no_grad():
        y2, _ = M.RUN_CUDA_RWKV6_STATE(B, T, H * 64, H, *(t.to(DEV) for t in (r, k, v, w, u)), s)
    assert_bf16_close(y2, y_ref, "infctx y")
    assert_bf16_close(s, s_ref, "infctx final state")


@pytest.mark.parametrize("dist", ["randn", "hot", "all_clamped", "spiky"])
def test_strong_decays_stay_on_the_tensor_cores(M, O, dist):
    """The reference tests' own distribution (w ~ N(0,1), tests/test_cpu.py:266) and hotter ones, forced onto the
    tensor-core kernels (impl = "tc": an exact-route hand-off would raise), against the UNCLAMPED fp64 recurrence:
    the built-in floor of 2^-13 per token and the 16-token reference blocks must stay inside the stated tolerance."""
    B, T, H = 2, 333, 2
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=77, decay="randn")
    gw_tol = 1e-2
    # max-abs bound of these stress distributions: 2^-6 max|ref| instead of 2^-7.  With few surviving terms per sum
    # the bf16 rounding of ONE operand and of the output can add up to 1.2 ulp on the largest elements (the CPU
    # emulation tests/tc_emulation.py shows the same 1.02 x 2^-7 on this input, and 0.26 without operand rounding:
    # it is rounding noise, not the decay floor); rel-RMS keeps the stated 1e-2.
    if dist == "hot":
        w = (w.float() * 1.5 + 1.0).bfloat16()
    elif dist == "all_clamped":
        # every token decays by more than the floor: the true gw is ~0 everywhere, the floor's own gradient
        # l 2^l <S,G> (1e-3 of a term) is what is left -- relative to a vanishing reference, hence the wider bound
        w = (w.float() + 2.5).bfloat16()
        gw_tol = 3e-2
    elif dist == "spiky":
        g = torch.Generator().manual_seed(5)
        w = torch.where(torch.rand(w.shape, generator=g) < 0.1, torch.full_like(w, 4.5), (w.float() - 3.0).bfloat16())
    ref = O.wkv6_backward(r, k, v, w, u, gy)
    M.set_impl("tc")
    try:
        with M.exact_route_report() as rep:
            y, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
    finally:
        M.set_impl("auto")
    assert rep.streams() == (0, B * H)
    assert_bf16_close(y, ref["y"], f"{dist} y", maxabs_rel=2.0 ** -6)
    for g_, key in zip(grads, ("gr", "gk", "gv", "gw", "gu")):
        assert_bf16_close(g_, ref[key], f"{dist} {key}", relrms_tol=gw_tol if key == "gw" else 1e-2, maxabs_rel=2.0 ** -6)


def test_exact_route_report(M):
    """Diagnostics: how many streams of the training forwards went to the exact route."""
    B, T, H = 2, 200, 2
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=12, decay="model", device=DEV)
    w[1, 40:120, 64:128] = 3.0
    leaves = [t.clone().requires_grad_(True) for t in (r, k, v, w, u)]
    with M.exact_route_report() as rep:
        M.RUN_CUDA_RWKV6(B, T, H * 64, H, *leaves)
        M.RUN_CUDA_RWKV6(B, T, H * 64, H, *leaves)
    assert rep.streams() == (0, 8)             # no stream ever leaves the tensor-core kernels


def test_native_raww_backward_without_saved_state(M):
    """wkv6_backward_raww (no training pair): the library recomputes the chunk-start states itself."""
    import ctypes
    from rwkv_lm_ext_b200 import _lib
    B, T, H = 2, 130, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=8, decay="model", device=DEV)
    lib = _lib.load()
    gr, gk, gv, gw = (torch.empty_like(r) for _ in range(4))
    gu = torch.empty(B, C, device=DEV, dtype=torch.bfloat16)
    n = lib.wkv6_backward_workspace_bytes(B, T, C, H)
    ws = torch.empty(n, dtype=torch.uint8, device=DEV)
    _lib.check(lib.wkv6_backward_raww(B, T, C, H, *(t.data_ptr() for t in (r, k, v, w, u, gy, gr, gk, gv, gw, gu)),
                                      ws.data_ptr(), n, torch.cuda.current_stream().cuda_stream), "wkv6_backward_raww")
    _, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
    for a, b_ in zip((gr, gk, gv, gw, gu.sum(0).view(H, 64)), grads):
        assert relrms(a, b_) < 1e-6


def test_native_fp32_logdecay_entries(M, O):
    """cuda/wkv6_op.cpp surface: w is fp32 -exp(w).  When it was made from bf16 logits (what the reference
    does, src/model.py:210) the tensor-core kernels run on the recovered logits; a stream whose values do
    not survive the bf16 round trip is computed exactly by the SIMT kernels -- both in one call."""
    B, T, H = 2, 150, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=13, decay="model")
    ew = -torch.exp(w.float())
    ew[1, :, 64:] = -torch.exp(w.float()[1, :, 64:] + 0.001)       # stream (1,1): not representable as bf16 logits
    dv = lambda t: t.to(DEV).contiguous()
    rd, kd, vd, ud, gyd, ewd = map(dv, (r, k, v, u, gy, ew))
    y = torch.empty_like(rd)
    M.wkv6_cuda.forward(B, T, C, H, rd, kd, vd, ewd, ud, y)
    gr, gk, gv, gw = (torch.empty_like(rd) for _ in range(4))
    gu = torch.empty(B, C, device=DEV, dtype=torch.bfloat16)
    M.wkv6_cuda.backward(B, T, C, H, rd, kd, vd, ewd, ud, gyd, gr, gk, gv, gw, gu)
    # reference values: fp64 recurrence on the same fp32 log-decay
    y_ref, _ = O.wkv6_recurrence(r, k, v, ew, u, w_is_log_decay=True)
    assert_bf16_close(y, y_ref, "y (fp32 log-decay entry)")
    M.set_impl("simt")
    try:
        y_s = torch.empty_like(rd)
        M.wkv6_cuda.forward(B, T, C, H, rd, kd, vd, ewd, ud, y_s)
        g_s = [torch.empty_like(rd) for _ in range(4)]
        gu_s = torch.empty(B, C, device=DEV, dtype=torch.bfloat16)
        M.wkv6_cuda.backward(B, T, C, H, rd, kd, vd, ewd, ud, gyd, *g_s, gu_s)
    finally:
        M.set_impl("auto")
    # the inexact stream must be bit-identical to the SIMT result, the others within tensor-core rounding
    assert torch.equal(y[1, :, 64:], y_s[1, :, 64:])
    for a, b_ in zip((gr, gk, gv, gw), g_s):
        assert torch.equal(a[1, :, 64:], b_[1, :, 64:])
        assert relrms(a, b_) < 6e-3
    assert relrms(gu, gu_s) < 6e-3


def test_native_surface_matches_python_surface(M):
    """cuda/wkv6_op.cpp signatures (fp32 ew = -exp(w), caller-allocated outputs)."""
    B, T, H = 2, 70, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=5, decay="model", device=DEV)
    ew = (-torch.exp(w.float())).contiguous()
    y = torch.empty_like(r)
    M.wkv6_cuda.forward(B, T, C, H, r, k, v, ew, u, y)
    gr, gk, gv, gw = (torch.empty_like(r) for _ in range(4))
    gu = torch.empty(B, C, device=DEV, dtype=torch.bfloat16)
    M.wkv6_cuda.backward(B, T, C, H, r, k, v, ew, u, gy, gr, gk, gv, gw, gu)
    y2, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
    # same kernels, decay read in fp32 instead of recomputed from bf16 w: near-identical
    assert relrms(y, y2) < 6e-3      # tcgen05 path rounds scaled operands to bf16
    for a, b in zip((gr, gk, gv, gw, gu.sum(0).view(H, 64)), grads):
        assert relrms(a, b) < 5e-3


# ---------------------------------------------------------------------------------------------
# state variants
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [1, 33, 64, 100])
def test_wkv6state_vs_oracle(M, O, T):
    B, H = 2, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=T, decay="model")
    s = (torch.randn(H, 64, 64, generator=torch.Generator().manual_seed(T)) * 0.5).bfloat16()
    ref = O.wkv6_backward(r, k, v, w, u, gy, s=s, s_layout="state")
    leaves = [t.clone().to(DEV).requires_grad_(True) for t in (r, k, v, w, u, s)]
    os.environ["RWKV_TRAIN_TYPE"] = "states"
    try:
        y = M.RUN_CUDA_RWKV6_STATE(B, T, C, H, *leaves)
    finally:
        os.environ.pop("RWKV_TRAIN_TYPE")
    assert isinstance(y, torch.Tensor)
    y.backward(gy.to(DEV))
    assert_bf16_close(y, ref["y"], "y")
    for t, key in zip(leaves, ("gr", "gk", "gv", "gw", "gu", "gs")):
        assert_bf16_close(t.grad, ref[key], key)
    assert leaves[3].grad[:, -1].abs().max().item() == 0.0
    if T > 1:
        assert leaves[3].grad[:, 0].abs().max().item() > 0.0      # real value at t = 0 (cuda/wkv6state_cuda.cu:254)


def test_wkv6infctx_in_place_state_and_chain(M, O):
    B, T, H = 2, 96, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=77, decay="model")
    s0 = (torch.randn(B, H, 64, 64, generator=torch.Generator().manual_seed(1)) * 0.5).bfloat16()
    y_ref, s_ref = O.wkv6infctx_forward(r, k, v, w, u, s0)
    dv = lambda t: t.clone().to(DEV)
    # one call, bf16 state written back in place (cuda/wkv6infctx_cuda.cu:65-67)
    s = dv(s0)
    y, s_ret = M.RUN_CUDA_RWKV6_STATE(B, T, C, H, dv(r), dv(k), dv(v), dv(w), dv(u), s)
    assert s_ret.data_ptr() == s.data_ptr()
    assert_bf16_close(y, y_ref, "infctx y")
    assert_bf16_close(s, s_ref, "infctx final state (bf16)")
    # chain of chunks with an fp32 carried state == one long call, fp32 tolerance
    sf = dv(s0).float()
    ys = []
    for a in range(0, T, 32):
        sl = slice(a, a + 32)
        yc, sf = M.RUN_CUDA_RWKV6_STATE(B, 32, C, H, dv(r[:, sl]).contiguous(), dv(k[:, sl]).contiguous(),
                                        dv(v[:, sl]).contiguous(), dv(w[:, sl]).contiguous(), dv(u), sf)
        ys.append(yc)
    assert_bf16_close(torch.cat(ys, 1), y_ref, "infctx chained y")
    assert relrms(sf, s_ref) < STATE_RELRMS
    # gradient w.r.t. the INITIAL state (the reference kernel sees the final one: a defect)
    ref = O.wkv6_backward(r, k, v, w, u, gy, s=s0, s_layout="infctx")
    leaves = [dv(t).requires_grad_(True) for t in (r, k, v, w, u)]
    s_leaf = dv(s0).requires_grad_(True)
    y2, _ = M.RUN_CUDA_RWKV6_STATE(B, T, C, H, *leaves, s_leaf.clone())
    y2.backward(dv(gy))
    for t, key in zip(leaves + [s_leaf], ("gr", "gk", "gv", "gw", "gu", "gs")):
        assert_bf16_close(t.grad, ref[key], f"infctx {key}")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
@pytest.mark.parametrize("T", [50, 700])
def test_rwkv6_inference_op(M, O, dtype, T):
    H = 3
    C = H * 64
    r, k, v, w, u, _ = make_inputs(1, T, H, seed=9, decay="model")
    cast = lambda t: t.float().to(dtype)
    r, k, v, w, u = (cast(t[0]) if t.dim() == 3 else cast(t) for t in (r, k, v, w, u))
    st0 = torch.randn(H, 64, 64, generator=torch.Generator().manual_seed(2)) * 0.3
    decay = torch.exp(-torch.exp(w.float()))
    y_ref, s_ref = O.rwkv6_inference_forward(st0, r, k, v, decay, u)
    st = st0.clone().to(DEV)
    y, st_ret = M.RUN_RWKV_6(1, T, C, H, st, r.to(DEV), k.to(DEV), v.to(DEV), w.to(DEV), u.to(DEV))
    assert st_ret.data_ptr() == st.data_ptr() and tuple(y.shape) == (1, T, C) and y.dtype == dtype
    if dtype == torch.float32:
        assert relrms(y[0], y_ref) < 1e-5
    else:
        assert_bf16_close(y[0], y_ref, "inference y")
    assert relrms(st, s_ref) < STATE_RELRMS


# ---------------------------------------------------------------------------------------------
# bidirectional op
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("decay,T", [("randn", 64), ("model", 64), ("model", 200), ("randn", 200)])
def test_wkv6_bi_vs_oracle(M, O, decay, T):
    """Both directions run on the tensor-core kernels (BI modes: per-row lengths, in-tile time reversal)."""
    B, H = 4, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=21, decay=decay)
    mask = torch.ones(B, T, dtype=torch.int32)
    mask[0, 60:] = 0          # cuda/wkv6_bi.py:66-67 smoke masks
    mask[1, 40:] = 0
    mask[2, 0:] = 0           # empty row: p = 0
    ref = O.wkv6_bi_backward(mask, r, k, v, w, u, gy)
    leaves = [t.clone().to(DEV).requires_grad_(True) for t in (r, k, v, w, u)]
    y = M.RUN_CUDA_RWKV6_BI(B, T, C, H, mask.to(DEV), *leaves)
    y.backward(gy.to(DEV))
    assert_bf16_close(y, ref["y"], "bi y")
    assert y[0, 61:].abs().max().item() == 0.0 and y[1, 41:].abs().max().item() == 0.0
    # native entry (fp32 log-decay, cuda/wkv6_bi_op.cpp:8-14) gives the same forward
    y_n = torch.empty_like(y)
    M.wkv6_bi_cuda.forward(B, T, C, H, mask.to(DEV), *(t.detach() for t in leaves[:3]),
                           (-torch.exp(leaves[3].detach().float())).contiguous(), leaves[4].detach(), y_n)
    assert relrms(y_n, y.detach()) < 1e-6
    for t, key in zip(leaves, ("gr", "gk", "gv", "gw", "gu")):
        assert_bf16_close(t.grad, ref[key], f"bi {key}")
    assert leaves[0].grad[0, 61:].abs().max().item() == 0.0 and leaves[3].grad[1, 41:].abs().max().item() == 0.0


@pytest.mark.parametrize("T", [130, 513])
def test_wkv6_bi_row_lengths_around_chunk_boundaries(M, O, T):
    """p on, just before and just behind 64-token chunk boundaries, p = 0, p = T-1 (no masked token), several chunks per
    row: the reverse direction reads tiles at token offsets p - 64c - 63 (negative for the last one) and mirrors their
    rows; the causal direction stops at p and writes zeros behind it.  Against the fp64 oracle, per row."""
    ps = [0, 1, 62, 63, 64, 65, 127, 128, 129, T - 2, T - 1, None]        # None: no masked token at all
    ps = [p for p in ps if p is None or p < T]
    B, H = len(ps), 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=33, decay="model")
    mask = torch.ones(B, T, dtype=torch.int32)
    for b, p in enumerate(ps):
        if p is not None:
            mask[b, p:] = 0
    ref = O.wkv6_bi_backward(mask, r, k, v, w, u, gy)
    leaves = [t.clone().to(DEV).requires_grad_(True) for t in (r, k, v, w, u)]
    y = M.RUN_CUDA_RWKV6_BI(B, T, C, H, mask.to(DEV), *leaves)
    y.backward(gy.to(DEV))
    for b, p in enumerate(ps):
        n = T if p is None else p + 1
        # y = bf16(bf16(y_causal) + bf16(y_reverse)) like the reference (three roundings, and the two addends may be
        # larger than their sum): twice the single-rounding max-abs allowance, same rel-RMS bar
        assert_bf16_close(y[b, :n], ref["y"][b, :n], f"bi y row {b} (p={p})", maxabs_rel=2 * BF16_MAXABS_REL)
        for t, key in zip(leaves[:4], ("gr", "gk", "gv", "gw")):
            assert_bf16_close(t.grad[b, :n], ref[key][b, :n], f"bi {key} row {b} (p={p})")
            assert t.grad[b, n:].abs().sum().item() == 0.0, f"{key} behind p in row {b}"
        assert y[b, n:].abs().sum().item() == 0.0
    assert_bf16_close(leaves[4].grad, ref["gu"], "bi gu")


def test_wkv6_bi_native_entry_with_an_inexact_stream(M, O):
    """cuda/wkv6_bi_op.cpp surface (fp32 -exp(w)): a stream whose decays are not bf16 logits is recomputed by the exact
    SIMT bidirectional kernels (bit-identical to impl="simt"), the others run both directions on the tensor-core
    kernels -- in one call, forward and backward."""
    B, T, H = 3, 200, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=41, decay="model")
    ew = -torch.exp(w.float())
    ew[1, :, 64:] = -torch.exp(w.float()[1, :, 64:] + 0.001)        # stream (1,1): not representable as bf16 logits
    mask = torch.ones(B, T, dtype=torch.int32)
    mask[0, 150:] = 0
    mask[1, 77:] = 0
    dv = lambda t: t.to(DEV).contiguous()
    rd, kd, vd, ud, gyd, ewd, md = map(dv, (r, k, v, u, gy, ew, mask))
    out = {}
    for impl in ("auto", "simt"):
        M.set_impl(impl)
        try:
            y = torch.empty_like(rd)
            M.wkv6_bi_cuda.forward(B, T, C, H, md, rd, kd, vd, ewd, ud, y)
            g = [torch.empty_like(rd) for _ in range(4)]
            gu = torch.empty(B, C, device=DEV, dtype=torch.bfloat16)
            M.wkv6_bi_cuda.backward(B, T, C, H, md, rd, kd, vd, ewd, ud, gyd, *g, gu)
        finally:
            M.set_impl("auto")
        out[impl] = [y] + g
    y_ref = O.wkv6_bi_forward(mask, r, k, v, ew, u, w_is_log_decay=True) if "w_is_log_decay" in O.wkv6_bi_forward.__code__.co_varnames else None
    for a, b_, name in zip(out["auto"], out["simt"], ("y", "gr", "gk", "gv", "gw")):
        assert torch.equal(a[1, :, 64:], b_[1, :, 64:]), f"{name}: the inexact stream must come from the exact kernels"
        assert_bf16_close(a, b_.float().cpu(), f"bi native {name} auto vs simt", maxabs_rel=2 * BF16_MAXABS_REL)
    if y_ref is not None:
        assert_bf16_close(out["auto"][0], y_ref, "bi native y vs oracle", maxabs_rel=2 * BF16_MAXABS_REL)


def test_gu_total_is_the_row_sum(M):
    """The training pair's backward adds the per-sample gu rows over the batch in the kernel (last CTA of every head):
    the result must be what torch.sum(gu, 0) gives (src/model.py:232) -- fp32 accumulation of the bf16 rows."""
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    B, T, H = 5, 192, 3
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=9, decay="model", device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    y = torch.empty_like(r)
    saved = torch.empty(lib.wkv6_saved_bytes(B, T, C, H), dtype=torch.uint8, device=DEV)
    import ctypes
    valid = ctypes.c_int(0)
    p = lambda t: t.data_ptr()
    assert lib.wkv6_train_forward(B, T, C, H, p(r), p(k), p(v), p(w), p(u), None, 0, 0, None, 0, p(y), p(saved), ctypes.byref(valid), st) == 0
    assert valid.value == 1
    n = lib.wkv6_train_backward_workspace_bytes(B, T, C, H, 1)
    ws = torch.empty(n, dtype=torch.uint8, device=DEV)
    g = [torch.empty_like(r) for _ in range(4)]
    gu = torch.empty(B, C, device=DEV, dtype=torch.bfloat16)
    for _ in range(2):                       # twice on the same saved buffer: the arrival counters return to zero
        gu_total = torch.full((C,), float("nan"), device=DEV, dtype=torch.bfloat16)
        assert lib.wkv6_train_backward(B, T, C, H, p(r), p(k), p(v), p(w), p(u), None, 0, p(gy), *(p(t) for t in g), p(gu),
                                       p(gu_total), None, p(saved), p(ws), n, st) == 0
        assert torch.equal(gu_total, torch.sum(gu.float(), 0).bfloat16())
    # and the Python surface returns it
    leaves = [t.clone().requires_grad_(True) for t in (r, k, v, w, u)]
    M.RUN_CUDA_RWKV6(B, T, C, H, *leaves).backward(gy)
    assert torch.equal(leaves[4].grad.reshape(-1), gu_total)


def test_tensor_on_another_device_is_refused(M):
    """The library takes scratch from the CURRENT device: a tensor on a different one must raise, not misbehave."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from rwkv_lm_ext_b200._lib import Wkv6B200Error
    r, k, v, w, u, _ = make_inputs(1, 64, 1, seed=0, decay="model", device=torch.device("cuda", 1))
    with torch.cuda.device(0), pytest.raises(Wkv6B200Error):
        M.RUN_CUDA_RWKV6(1, 64, 64, 1, r, k, v, w, u)


def test_wkv6_bi_tensor_core_route_equals_exact_route(M):
    """Mid-size shape (many streams, 8 chunks): the fused tensor-core route against the exact SIMT bidirectional kernels."""
    B, T, H = 8, 512, 4
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=5, decay="model", device=DEV)
    mask = torch.ones(B, T, dtype=torch.int32, device=DEV)
    for b, n in enumerate([512, 511, 300, 257, 256, 129, 64, 7]):
        mask[b, n - 1:] = 0
    out = {}
    for impl in ("tc", "simt"):
        M.set_impl(impl)
        leaves = [t.clone().requires_grad_(True) for t in (r, k, v, w, u)]
        y = M.RUN_CUDA_RWKV6_BI(B, T, C, H, mask, *leaves)
        y.backward(gy)
        out[impl] = [y.detach()] + [t.grad for t in leaves]
    M.set_impl("auto")
    for a, b_, name in zip(out["tc"], out["simt"], ("y", "gr", "gk", "gv", "gw", "gu")):
        assert_bf16_close(a, b_.float().cpu(), f"bi {name} tc vs simt")


# ---------------------------------------------------------------------------------------------
# against the reference's own CUDA kernels (oracle/_ref, built from /root/reference/cuda/*.cu)
# ---------------------------------------------------------------------------------------------
def test_against_reference_cuda_kernels(M):
    from oracle import ref_cuda
    if not ref_cuda.available("wkv6"):
        pytest.skip("oracle/_ref not built (make -C oracle ref)")
    B, T, H = 2, 512, 4
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=3, decay="model", device=DEV)
    y_ref, ew = ref_cuda.wkv6_forward(r, k, v, w, u)
    g_ref = ref_cuda.wkv6_backward(r, k, v, ew, u, gy)
    torch.cuda.synchronize()
    y, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
    assert_bf16_close(y, y_ref.float(), "y vs reference CUDA", relrms_tol=6e-3)
    for a, b, key in zip(grads, g_ref, ("gr", "gk", "gv", "gw", "gu")):
        assert_bf16_close(a, b.float(), f"{key} vs reference CUDA", relrms_tol=8e-3)


# ---------------------------------------------------------------------------------------------
# long sequences: C oracle (fp32, multi-threaded) at T = 4096, and size-independent properties at
# BASELINE.json's full shape
# ---------------------------------------------------------------------------------------------
def test_long_sequence_vs_c_oracle(M):
    from oracle import c_oracle
    B, T, H = 1, 4096, 2
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=4096, decay="model")
    y_ref = c_oracle.forward(r, k, v, w, u)
    g_ref = c_oracle.backward(r, k, v, w, u, gy)
    y, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
    assert_bf16_close(y, y_ref, "T=4096 y")
    for a, key in zip(grads[:4], ("gr", "gk", "gv", "gw")):
        assert_bf16_close(a, g_ref[key], f"T=4096 {key}")
    assert_bf16_close(grads[4], g_ref["gu"].sum(0).view(H, 64), "T=4096 gu")


@pytest.mark.parametrize("decay", ["model", "randn"])
def test_full_shape_forward_backward_vs_c_oracle(M, decay):
    """BASELINE.json configs[1] at full size, B=8, T=4096, H=32, forward AND backward against the oracle's C port
    (fp32 step recurrence with the reference kernels' arithmetic, about a second of CPU per batch row), for the
    model-like decays and for the reference tests' w ~ N(0,1) -- with no stream on the exact route."""
    from oracle import c_oracle
    B, T, H = 8, 4096, 32
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=2, decay=decay)
    with M.exact_route_report() as rep:
        y, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
    assert rep.streams() == (0, B * H)
    gu_ref = torch.zeros(H, 64, dtype=torch.float64)
    for b in range(B):
        sl = slice(b, b + 1)
        y_ref = c_oracle.forward(r[sl], k[sl], v[sl], w[sl], u)
        g_ref = c_oracle.backward(r[sl], k[sl], v[sl], w[sl], u, gy[sl])
        assert_bf16_close(y[sl], y_ref, f"{decay} row {b} y")
        for a, key in zip(grads[:4], ("gr", "gk", "gv", "gw")):
            assert_bf16_close(a[sl], g_ref[key], f"{decay} row {b} {key}")
        gu_ref += g_ref["gu"].sum(0).view(H, 64).double()
    assert_bf16_close(grads[4], gu_ref, f"{decay} gu")


def test_full_shape_properties(M):
    """B=8, T=4096, H=32 (BASELINE.json configs[1]): too big for the oracle, so check
    (1) split-and-carry == one call, (2) batch rows are independent, (3) SIMT == AUTO."""
    B, T, H = 8, 4096, 32
    C = H * 64
    r, k, v, w, u, _ = make_inputs(B, T, H, seed=1, decay="model", device=DEV)
    y = M.RUN_CUDA_RWKV6(B, T, C, H, r, k, v, w, u)
    assert torch.isfinite(y.float()).all()
    # (1) two halves chained through an fp32 state
    s = torch.zeros(B, H, 64, 64, device=DEV)
    h = T // 2
    ya, s = M.RUN_CUDA_RWKV6_STATE(B, h, C, H, *(t[:, :h].contiguous() for t in (r, k, v, w)), u, s)
    yb, s = M.RUN_CUDA_RWKV6_STATE(B, h, C, H, *(t[:, h:].contiguous() for t in (r, k, v, w)), u, s)
    assert relrms(torch.cat([ya, yb], 1), y) < 3e-3
    # (2) row 3 alone gives the same numbers
    y3 = M.RUN_CUDA_RWKV6(1, T, C, H, *(t[3:4].contiguous() for t in (r, k, v, w)), u)
    assert relrms(y3, y[3:4]) < 1e-6
    # (3) implementations agree
    M.set_impl("simt")
    try:
        ys = M.RUN_CUDA_RWKV6(B, T, C, H, r, k, v, w, u)
    finally:
        M.set_impl("auto")
    assert relrms(y, ys) < 6e-3


def test_bidirectional_encoder_composition(M, O):
    """BASELINE config 3 in miniature: padded passages -> mask / reverse index (our kernel) -> the
    reverse-gather + WKV6 + un-reverse composition of the bidirectional models (src/model_bi.py:345-348,
    src/model_ext.py:398-437) built from this library's pieces, against the oracle."""
    B, T, H = 3, 200, 2
    C = H * 64
    g = torch.Generator().manual_seed(5)
    idx = torch.randint(2, 1000, (B, T), generator=g)
    lens = [200, 131, 64]
    for b_, n in enumerate(lens):
        idx[b_, n - 1] = 1            # embedding / eos id
        idx[b_, n:] = 0               # padding
    r, k, v, w, u, _ = make_inputs(B, T, H, seed=17, decay="model")
    mask_ref = O.create_mask(idx, 1, 0)
    rev_ref = O.reverse_x_idx(mask_ref, T)
    y_ref = O.wkv6_bi_sum_forward(r, k, v, w, u, rev_ref)
    mask, rev = M.create_mask_and_rev_idx(idx.to(DEV), 1, 0)
    assert torch.equal(mask.cpu(), mask_ref.to(torch.int32)) and torch.equal(rev.cpu(), rev_ref)
    dv = lambda t: t.to(DEV)
    with torch.no_grad():
        y1 = M.RUN_CUDA_RWKV6(B, T, C, H, dv(r), dv(k), dv(v), dv(w), dv(u))
        y2 = M.RUN_CUDA_RWKV6(B, T, C, H, dv(r), M.reverse_x(dv(k), rev), M.reverse_x(dv(v), rev), dv(w), dv(u))
        y = y1.float() + M.reverse_x(y2, rev).float()
    assert_bf16_close(y, y_ref, "bidirectional sum")
    pos = M.eos_index(idx.to(DEV), 1)
    assert pos.cpu().tolist() == [n - 1 for n in lens]


def test_infctx_long_context_chain_3b_shape(M):
    """BASELINE config 5 in miniature: 3B shape (H = 40), a 16k-token context as 4 chunks of 4096 tokens
    with the state carried in fp32 (extension) and in bf16 (the reference's container,
    src/infctx_module.py:36-38), against one uninterrupted SIMT pass."""
    B, T, H, NCH = 1, 4096, 40, 4
    C = H * 64
    r, k, v, w, u, _ = make_inputs(B, T * NCH, H, seed=21, decay="model", device=DEV)
    with torch.no_grad():
        M.set_impl("simt")
        try:
            s_ref = torch.zeros(B, H, 64, 64, device=DEV)
            y_ref, s_ref = M.RUN_CUDA_RWKV6_STATE(B, T * NCH, C, H, r, k, v, w, u, s_ref)
        finally:
            M.set_impl("auto")
        for dt, tol in ((torch.float32, STATE_RELRMS), (torch.bfloat16, 1e-2)):
            s = torch.zeros(B, H, 64, 64, device=DEV, dtype=dt)
            ys = []
            for c in range(NCH):
                sl = slice(c * T, (c + 1) * T)
                yc, s = M.RUN_CUDA_RWKV6_STATE(B, T, C, H, *(t[:, sl].contiguous() for t in (r, k, v, w)), u, s)
                ys.append(yc)
            assert relrms(torch.cat(ys, 1), y_ref) < 6e-3, dt
            assert relrms(s, s_ref) < tol, (dt, relrms(s, s_ref))


def test_very_long_single_call_and_many_streams(M):
    """T = 65536 in one call (1024 chunks per stream) and a grid of 4096 streams: tensor-core path == SIMT."""
    for (B, T, H) in ((1, 65536, 2), (64, 128, 64)):
        C = H * 64
        r, k, v, w, u, gy = make_inputs(B, T, H, seed=31, decay="model", device=DEV)
        y, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
        M.set_impl("simt")
        try:
            ys, gs = _run_fwd_bwd(M, r, k, v, w, u, gy)
        finally:
            M.set_impl("auto")
        assert relrms(y, ys) < 6e-3
        for a, b_ in zip(grads, gs):
            assert relrms(a, b_) < 8e-3


def test_segmented_forward_few_streams(M):
    """Forward-only calls with few streams and T >= 8192 are cut into time segments that run as
    independent batch rows (csrc/seg_scan.cu); y and the carried state must match the exact SIMT route."""
    from rwkv_lm_ext_b200 import _lib
    B, T, H = 1, 16384, 3
    C = H * 64
    r, k, v, w, u, _ = make_inputs(B, T, H, seed=41, decay="model", device=DEV)
    g = torch.Generator().manual_seed(42)
    s0 = (torch.randn(B, H, 64, 64, generator=g) * 0.3).to(DEV)
    lib = _lib.load()
    outs = []
    for impl in ("auto", "simt"):
        M.set_impl(impl)
        try:
            st = s0.clone()
            y = torch.empty_like(r)
            _lib.check(lib.wkv6infctx_forward_f32state(B, T, C, H, _lib.ptr(r), _lib.ptr(k), _lib.ptr(v), _lib.ptr(w),
                                                       _lib.ptr(u), _lib.ptr(st), _lib.ptr(y), _lib.stream_of(r)), "infctx fwd")
            with torch.no_grad():
                y0 = M.RUN_CUDA_RWKV6(B, T, C, H, r, k, v, w, u)
            outs.append((y, st, y0))
        finally:
            M.set_impl("auto")
    (y, st, y0), (ys, sts, y0s) = outs
    assert relrms(y, ys) < 6e-3 and relrms(y0, y0s) < 6e-3
    assert relrms(st, sts) < 2e-3


def test_empty_inputs(M):
    z = torch.empty(0, 8, 64, device=DEV, dtype=torch.bfloat16)
    u = torch.zeros(1, 64, device=DEV, dtype=torch.bfloat16)
    assert M.RUN_CUDA_RWKV6(0, 8, 64, 1, z, z, z, z, u).shape == (0, 8, 64)


def test_cuda_graph_capture_fwd_bwd(M):
    """The operator (forward + backward through autograd) is capturable in a CUDA graph: no host
    synchronisation, no legacy-stream work, scratch from torch's allocator.  Replays reproduce the eager
    results bit for bit on new input values."""
    B, T, H = 2, 192, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=51, decay="model", device=DEV)
    static = [t.clone().requires_grad_(True) for t in (r, k, v, w, u)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                       # warm-up on a side stream, as torch's recipe asks
        for _ in range(3):
            y = M.RUN_CUDA_RWKV6(B, T, C, H, *static)
            y.backward(gy)
    torch.cuda.current_stream().wait_stream(side)
    for t in static:
        t.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        y_static = M.RUN_CUDA_RWKV6(B, T, C, H, *static)
        y_static.backward(gy)
    # new values into the captured buffers, replay, compare with an eager run on the same values
    r2, k2, v2, w2, u2, _ = make_inputs(B, T, H, seed=52, decay="model", device=DEV)
    with torch.no_grad():
        for dst, src in zip(static, (r2, k2, v2, w2, u2)):
            dst.copy_(src)
    graph.replay()
    torch.cuda.synchronize()
    y_e, g_e = _run_fwd_bwd(M, r2, k2, v2, w2, u2, gy)
    assert torch.equal(y_static, y_e)
    for t, g in zip(static, g_e):
        assert torch.equal(t.grad, g)


@pytest.mark.parametrize("with_state", [False, True])
def test_segmented_training_pair(M, with_state):
    """Few streams and T >= 2048: forward AND backward of the training pair run as time segments (state scan
    forward, state-gradient scan backward on time-reversed r, gy, w).  Must agree with the exact SIMT kernels,
    keep the exact zeros at the edges of gw, deliver dL/dS_0, and leave the one hazardous stream to the
    exact route."""
    B, T, H = 2, 2048, 3
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=61, decay="model", device=DEV)
    w[1, 700:760, 128:192] = 3.0                 # stream (b=1, h=2): decays by > e^-60 inside 16 tokens
    s0 = (torch.randn(B, H, 64, 64, generator=torch.Generator().manual_seed(62)) * 0.3).bfloat16().to(DEV)
    launches = []

    def run(impl):
        M.set_impl(impl)
        try:
            leaves = [t.clone().requires_grad_(True) for t in (r, k, v, w, u)]
            n0 = M.launch_count()
            if with_state:
                s = s0.clone().requires_grad_(True)
                y, sT = M.RUN_CUDA_RWKV6_STATE(B, T, C, H, *leaves, s.clone())
            else:
                s, sT = None, None
                y = M.RUN_CUDA_RWKV6(B, T, C, H, *leaves)
            y.backward(gy)
            torch.cuda.synchronize()
            launches.append(M.launch_count() - n0)
            return y.detach(), [t.grad for t in leaves], (None if s is None else s.grad), sT
        finally:
            M.set_impl("auto")
    y, grads, gs, sT = run("auto")
    ys, gss, gs_s, sTs = run("simt")
    assert launches[0] > launches[1] + 6         # the segmented route really ran (scan / reverse / sum kernels)
    assert relrms(y, ys) < 6e-3
    for name, a, b_ in zip(("gr", "gk", "gv", "gw", "gu"), grads, gss):
        assert relrms(a, b_) < 8e-3, name
    assert grads[3][:, -1].abs().max().item() == 0.0
    if with_state:
        assert relrms(gs, gs_s) < 8e-3 and relrms(sT, sTs) < 6e-3
    else:
        assert grads[3][:, 0].abs().max().item() == 0.0


def test_concurrent_streams_do_not_share_scratch(M):
    """Calls in flight on different CUDA streams (forward-only path on raw logits; one of the inputs has a stream with
    decays far beyond the block references) give the same results as serial calls."""
    B, T, H = 2, 320, 3
    C = H * 64
    sets = []
    for i in range(4):
        r, k, v, w, u, _ = make_inputs(B, T, H, seed=70 + i, decay="model", device=DEV)
        if i % 2:
            w[0, 100:140, :64] = 3.0
        sets.append((r, k, v, w, u))
    with torch.no_grad():
        serial = [M.RUN_CUDA_RWKV6(B, T, C, H, *s) for s in sets]
        torch.cuda.synchronize()
        streams = [torch.cuda.Stream() for _ in range(4)]
        outs = [None] * 4
        for rep in range(5):
            for i, st in enumerate(streams):
                with torch.cuda.stream(st):
                    outs[i] = M.RUN_CUDA_RWKV6(B, T, C, H, *sets[i])
        torch.cuda.synchronize()
    for a, b_ in zip(outs, serial):
        assert torch.equal(a, b_)


def test_concurrent_fp32_decay_entries(M):
    """wkv6_cuda.forward / .backward (fp32 -exp(w), one stream per input set not representable as bf16 logits) in flight
    on four CUDA streams at once: every call keeps its stream flags in its own stream-ordered scratch (forward) or
    workspace (backward), so the results equal serial calls bit for bit."""
    B, T, H = 2, 320, 3
    C = H * 64
    sets = []
    for i in range(4):
        r, k, v, w, u, gy = make_inputs(B, T, H, seed=90 + i, decay="model", device=DEV)
        ew = -torch.exp(w.float())
        b, c0 = i % B, 64 * (i % H)
        ew[b, :, c0:c0 + 64] = -torch.exp(w.float()[b, :, c0:c0 + 64] + 0.001)
        sets.append((r, k, v, ew.contiguous(), u, gy))

    def run(r, k, v, ew, u, gy):
        y = torch.empty_like(r)
        M.wkv6_cuda.forward(B, T, C, H, r, k, v, ew, u, y)
        g = [torch.empty_like(r) for _ in range(4)]
        gu = torch.empty(B, C, device=DEV, dtype=torch.bfloat16)
        M.wkv6_cuda.backward(B, T, C, H, r, k, v, ew, u, gy, *g, gu)
        return [y, *g, gu]

    serial = [run(*s) for s in sets]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(4)]
    outs = [None] * 4
    for rep in range(5):
        for i, st in enumerate(streams):
            with torch.cuda.stream(st):
                outs[i] = run(*sets[i])
    torch.cuda.synchronize()
    for a, b_ in zip(outs, serial):
        for x, x_serial, name in zip(a, b_, ("y", "gr", "gk", "gv", "gw", "gu")):
            assert torch.equal(x, x_serial), name


def test_launch_counts_on_raw_logits(M):
    """Raw bf16 logits carry no stream flags: the calls launch their tensor-core kernels and nothing else (no exact-route
    launch whose blocks would all exit at once)."""
    B, T, H = 2, 192, 2
    C = H * 64
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=95, decay="model", device=DEV)
    mask = torch.ones(B, T, dtype=torch.int32, device=DEV)
    mask[0, 150:] = 0

    def launches(fn):
        n0 = M.launch_count()
        out = fn()
        return M.launch_count() - n0, out

    with torch.no_grad():
        assert launches(lambda: M.RUN_CUDA_RWKV6(B, T, C, H, r, k, v, w, u))[0] == 1
    leaves = [t.clone().requires_grad_(True) for t in (r, k, v, w, u)]
    assert launches(lambda: M.RUN_CUDA_RWKV6(B, T, C, H, *leaves).backward(gy))[0] == 2     # forward + backward kernel
    leaves = [t.clone().requires_grad_(True) for t in (r, k, v, w, u)]
    n, y = launches(lambda: M.RUN_CUDA_RWKV6_BI(B, T, C, H, mask, *leaves))
    assert n == 4                 # row lengths, row order, causal and reverse forward
    assert launches(lambda: y.backward(gy))[0] == 6      # row lengths, row order, per direction: states + backward


def test_decay_clamp_opt_in(M, O):
    """wkv6b200_set_decay_clamp(3.7): the op computes with w' = min(w, log 3.7) (zero w-gradient where the floor is
    active), on the tensor-core kernels for EVERY stream -- the one that would otherwise be handed to the exact
    route included -- and on the exact kernels alike.  Off again afterwards: the default semantics are untouched."""
    import math
    B, T, H = 2, 200, 2
    r, k, v, w, u, gy = make_inputs(B, T, H, seed=81, decay="model")
    w[1, 40:120, 64:128] = 3.0                     # exp(3) = 20 nats per token: far beyond the block references
    wc = torch.clamp(w.float(), max=math.log(3.7)).double().requires_grad_(True)
    leaves = [t.double().requires_grad_(True) for t in (r, k, v)] + [wc, u.double().requires_grad_(True)]
    y_ref, _ = O.wkv6_recurrence(*leaves)
    (y_ref * gy.double()).sum().backward()
    gw_ref = wc.grad * (w.float() <= math.log(3.7)).double()      # d/dw of min(w, c)
    assert M.set_decay_clamp(3.7) == 0.0
    try:
        for impl in ("auto", "simt"):
            M.set_impl(impl)
            with M.exact_route_report() as rep:
                y, grads = _run_fwd_bwd(M, r, k, v, w, u, gy)
            if impl == "auto":
                assert rep.streams() == (0, B * H)                 # nobody left the tensor-core kernels
            assert_bf16_close(y, y_ref, f"clamped y ({impl})")
            for g, ref, name in zip(grads, (leaves[0].grad, leaves[1].grad, leaves[2].grad, gw_ref, leaves[4].grad),
                                    ("gr", "gk", "gv", "gw", "gu")):
                assert_bf16_close(g, ref, f"clamped {name} ({impl})")
            assert grads[3][1, 41:119, 64:128].abs().max().item() == 0.0
    finally:
        M.set_impl("auto")
        assert abs(M.set_decay_clamp(0.0) - 3.7) < 1e-6
    with M.exact_route_report() as rep:
        _run_fwd_bwd(M, r, k, v, w, u, gy)
    assert rep.streams() == (0, B * H)                             # default semantics: still no exact-route hand-off


def test_long_prefill_through_the_fp32_decay_entries(M):
    """The pybind-shaped entries that receive fp32 decays (rwkv6 inference: exp(-exp(w)); wkv6: -exp(w)) with a long
    sequence and few streams: logits are recovered, the call is time-segmented, one stream whose decays do not
    survive the bf16 round trip goes to the exact route -- all in one call, equal to the exact kernels."""
    B, T, H = 1, 4096 + 64, 3
    C = H * 64
    r, k, v, w, u, _ = make_inputs(B, T, H, seed=91, decay="model", device=DEV)
    ew = -torch.exp(w.float())
    ew[0, :, 128:] = -torch.exp(w.float()[0, :, 128:] + 0.001)          # stream h=2: not representable as bf16 logits
    decay = torch.exp(ew)[0].contiguous()
    st0 = (torch.randn(H, 64, 64, generator=torch.Generator().manual_seed(5)) * 0.3).to(DEV)
    outs = {}
    for impl in ("auto", "simt"):
        M.set_impl(impl)
        try:
            st = st0.clone()
            y, _ = M.RUN_RWKV_6(1, T, C, H, st, r[0].contiguous(), k[0].contiguous(), v[0].contiguous(), decay, u)
            y2 = torch.empty_like(r)
            M.wkv6_cuda.forward(B, T, C, H, r, k, v, ew.contiguous(), u, y2)
            outs[impl] = (y, st, y2)
        finally:
            M.set_impl("auto")
    (y, st, y2), (ys, sts, y2s) = outs["auto"], outs["simt"]
    assert relrms(y, ys) < 6e-3 and relrms(st, sts) < 2e-3 and relrms(y2, y2s) < 6e-3
    assert torch.equal(y[..., 128:], ys[..., 128:])                     # the inexact stream ran on the exact kernels
