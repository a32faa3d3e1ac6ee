"""Gradients through the carried WKV state (ops.WKV_6STATE_BPTT, wkv6_train_backward_state_grad): the loss may
depend on the final state, and its gradient flows back into r, k, v, w, u and the initial state.  Checked against
fp64 autograd of the oracle, chunk by chunk against one pass, against the truncated operator where the final-state
gradient is 0, across the SIMT and tensor-core routes, at the layer level and under CUDA-graph replay.
`pytest -m gpu`."""
import ctypes

import pytest
import torch

from tests.util import assert_bf16_close, make_inputs, relrms

pytestmark = pytest.mark.gpu
DEV = "cuda"


def nseg_of(B, T, H):
    from rwkv_lm_ext_b200 import _lib
    n, sc = ctypes.c_int(0), ctypes.c_int(0)
    _lib.load().wkv6b200_seg_plan(B, T, H, 1, ctypes.byref(n), ctypes.byref(sc))
    return n.value


def inputs(B, T, H, seed, carry, s0_kind="random"):
    r, k, v, w, u, gy = make_inputs(B, T, H, seed)
    g = torch.Generator().manual_seed(seed + 1000)
    s0 = torch.zeros(B, H, 64, 64) if s0_kind == "zero" else torch.randn(B, H, 64, 64, generator=g) * 0.3
    gT = torch.randn(B, H, 64, 64, generator=g)
    return r, k, v, w, u, gy, s0.to(carry), gT.to(carry)


def oracle(r, k, v, w, u, s0, gy, gT):
    """fp64 autograd of  <y, gy> + <s_final, gT>;  s0, s_final, gT in the [B,H,value,key] layout."""
    from oracle import wkv6_oracle as O
    leaves = [t.detach().double().clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    y, S = O.wkv6_recurrence(*leaves[:5], leaves[5].transpose(-1, -2))
    sT = S.transpose(-1, -2)
    ((y * gy.double()).sum() + (sT * gT.double()).sum()).backward()
    return y.detach(), sT.detach(), [t.grad for t in leaves]


def run_op(r, k, v, w, u, s0, gy, gT):
    import rwkv_lm_ext_b200 as M
    B, T, C = r.shape
    H = C // 64
    leaves = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    s_in = leaves[5].detach().clone()
    y, sT = M.RUN_CUDA_RWKV6_STATE_BPTT(B, T, C, H, *leaves)
    assert torch.equal(leaves[5].detach(), s_in), "the initial state must not be modified"
    assert sT.dtype == s0.dtype and sT.data_ptr() != leaves[5].data_ptr()
    loss = (y.float() * gy.to(DEV).float()).sum()
    if gT is not None:
        loss = loss + (sT.float() * gT.to(DEV).float()).sum()
    loss.backward()
    return y.detach(), sT.detach(), [t.grad for t in leaves]


def check_against_oracle(B, T, H, seed, carry, s0_kind):
    r, k, v, w, u, gy, s0, gT = inputs(B, T, H, seed, carry, s0_kind)
    y_ref, sT_ref, g_ref = oracle(r, k, v, w, u, s0, gy, gT)
    y, sT, g = run_op(r, k, v, w, u, s0, gy, gT)
    assert_bf16_close(y, y_ref, "y")
    assert relrms(sT, sT_ref) <= 1e-2, "s_final"
    for name, got, ref in zip(("gr", "gk", "gv", "gw", "gu", "gs"), g, g_ref):
        assert got.dtype == (s0.dtype if name == "gs" else torch.bfloat16), name
        assert_bf16_close(got, ref, name)
    # the last decay now feeds the final state: gw[:, T-1] is no longer 0
    gw_last_ref = g_ref[3][:, -1]
    if T > 1 or s0_kind == "random":
        assert gw_last_ref.abs().max() > 1e-3
    assert_bf16_close(g[3][:, -1], gw_last_ref, "gw[:, T-1]")


@pytest.mark.parametrize("T", [1, 63, 64, 65, 130, 1000])
@pytest.mark.parametrize("carry", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("s0_kind", ["zero", "random"])
def test_against_fp64_oracle(T, carry, s0_kind):
    assert nseg_of(2, T, 2) == 1
    check_against_oracle(2, T, 2, 7 + T, carry, s0_kind)


@pytest.mark.parametrize("B, H, T", [(1, 2, 4096), (2, 3, 8192), (2, 37, 4096)])
@pytest.mark.parametrize("carry", [torch.bfloat16, torch.float32])
def test_segmented_route_against_fp64_oracle(B, H, T, carry):
    assert B * H <= 74 and nseg_of(B, T, H) > 1
    check_against_oracle(B, T, H, 11, carry, "random")


@pytest.mark.parametrize("B, H, T, chunks", [(1, 2, 4096, 4), (2, 40, 4096, 4), (1, 2, 8192, 4)])
def test_chunks_equal_one_pass(B, H, T, chunks):
    """4 chained calls with the fp32 carry and the state gradient flowing back == one call over the sequence.
    (1,2,4096): the whole call is segmented, the 1024-token chunks are not; (2,40,4096): neither is (80 streams);
    (1,2,8192): every call is."""
    import rwkv_lm_ext_b200 as M
    C = H * 64
    r, k, v, w, u, gy, s0, _ = inputs(B, T, H, 3, torch.float32)
    L = T // chunks
    whole = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    y, _ = M.RUN_CUDA_RWKV6_STATE_BPTT(B, T, C, H, *whole)
    (y.float() * gy.to(DEV).float()).sum().backward()

    part = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    s, loss = part[5], 0.0
    for c in range(chunks):
        sl = slice(c * L, (c + 1) * L)
        yc, s = M.RUN_CUDA_RWKV6_STATE_BPTT(B, L, C, H, *(t[:, sl].contiguous() for t in part[:4]), part[4], s)
        loss = loss + (yc.float() * gy[:, sl].to(DEV).float()).sum()
    loss.backward()
    for name, a, b in zip(("gr", "gk", "gv", "gw", "gu", "gs0"), part, whole):
        rr = relrms(a.grad, b.grad)
        assert rr <= 1e-2, f"{name}: rel-RMS {rr:.3g} (B={B} H={H} T={T}, segmented {nseg_of(B, T, H) > 1}/{nseg_of(B, L, H) > 1})"


@pytest.mark.parametrize("B, H, T", [(2, 2, 130), (1, 2, 4096)])
@pytest.mark.parametrize("carry", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("zero_gT", [True, False])
def test_zero_final_state_gradient_changes_nothing(B, H, T, carry, zero_gT):
    """gT = 0 (a zero tensor) or None (s_final unused): bit-equal to WKV_6STATE_INFCTX, gw[:, T-1] exactly 0."""
    import rwkv_lm_ext_b200 as M
    C = H * 64
    r, k, v, w, u, gy, s0, _ = inputs(B, T, H, 5, carry)
    gy = gy.to(DEV)

    a = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    y_a, s_a = M.RUN_CUDA_RWKV6_STATE_BPTT(B, T, C, H, *a)
    out = [y_a, s_a] if zero_gT else [y_a]
    torch.autograd.backward(out, [gy, torch.zeros_like(s_a)] if zero_gT else [gy])

    b = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    y_b, s_b = M.WKV_6STATE_INFCTX.apply(B, T, C, H, *b[:5], b[5].clone())
    y_b.backward(gy)

    assert torch.equal(y_a, y_b) and torch.equal(s_a, s_b)
    for name, ga, gb in zip(("gr", "gk", "gv", "gw", "gu", "gs"), (t.grad for t in a), (t.grad for t in b)):
        assert torch.equal(ga, gb), name
    assert (a[3].grad[:, -1] == 0).all()
    assert (nseg_of(B, T, H) > 1) == (T >= 2048)          # both routes


@pytest.mark.parametrize("B, H, T", [(2, 2, 130), (1, 2, 4096)])
def test_simt_agrees_with_tensor_cores(B, H, T):
    import rwkv_lm_ext_b200 as M
    r, k, v, w, u, gy, s0, gT = inputs(B, T, H, 9, torch.float32)
    tc = run_op(r, k, v, w, u, s0, gy, gT)
    prev = M.set_impl("simt")
    try:
        simt = run_op(r, k, v, w, u, s0, gy, gT)
    finally:
        M.set_impl(prev)
    assert_bf16_close(simt[0], tc[0], "y")
    assert relrms(simt[1], tc[1]) <= 1e-3, "s_final"
    for name, a, b in zip(("gr", "gk", "gv", "gw", "gu", "gs"), simt[2], tc[2]):
        assert_bf16_close(a, b, name)


def test_simt_against_fp64_oracle():
    import rwkv_lm_ext_b200 as M
    prev = M.set_impl("simt")
    try:
        check_against_oracle(2, 130, 2, 13, torch.bfloat16, "random")
    finally:
        M.set_impl(prev)


class _Cmix(torch.nn.Module):
    def __init__(self, C, F, g):
        super().__init__()
        self.time_maa_k = torch.nn.Parameter(torch.rand(1, 1, C, generator=g))
        self.time_maa_r = torch.nn.Parameter(torch.rand(1, 1, C, generator=g))
        self.key = torch.nn.Linear(C, F, bias=False)
        self.receptance = torch.nn.Linear(C, C, bias=False)
        self.value = torch.nn.Linear(F, C, bias=False)
        with torch.no_grad():
            self.key.weight.copy_(torch.randn(F, C, generator=g) / C ** 0.5)
            self.receptance.weight.copy_(torch.randn(C, C, generator=g) / C ** 0.5)
            self.value.weight.copy_(torch.randn(C, F, generator=g) / F ** 0.5)


def test_layer_chunks_equal_whole_sequence():
    """Tmix_x060 + the infctx channel mix over 2 chunks with exact_state_grad=True == the whole-sequence layer, output
    and every parameter / input gradient (the bounds of test_gpu_tmix.py)."""
    import rwkv_lm_ext_b200 as M
    from tests.test_gpu_tmix import assert_chain_close, make_layer
    B, T, H = 2, 256, 2
    C = H * 64
    att = make_layer(M, C, H, 31).to(DEV)
    ffn = _Cmix(C, 4 * C, torch.Generator().manual_seed(32)).bfloat16().to(DEV)
    g = torch.Generator().manual_seed(33)
    x = torch.randn(B, T, C, generator=g).bfloat16().to(DEV)
    gout = torch.randn(B, T, C, generator=g).bfloat16().to(DEV)

    def block(xc, state):
        if state is None:
            h = xc + att(xc)
            return h + M.cmix_x060_forward(ffn, h), None
        a, tms = att(xc, state[0], exact_state_grad=True)
        h = xc + a
        f, cms = M.cmix_x060_forward(ffn, h, state[1])
        return h + f, (tms, cms)

    def grads(chunks):
        att.zero_grad(set_to_none=True)
        ffn.zero_grad(set_to_none=True)
        xd = x.clone().requires_grad_(True)
        if chunks == 1:
            out, _ = block(xd, None)
        else:
            states = M.BlockStateList.create(1, B, C, H, DEV, torch.bfloat16, wkv_dtype=torch.float32)
            st = (states[0].time_mix_state, states[0].channel_mix_state)
            outs, L = [], T // chunks
            for c in range(chunks):
                o, st = block(xd[:, c * L:(c + 1) * L].contiguous(), st)
                outs.append(o)
            out = torch.cat(outs, 1)
        out.backward(gout)
        params = {f"att.{n}": p.grad.clone() for n, p in att.named_parameters()}
        params.update({f"ffn.{n}": p.grad.clone() for n, p in ffn.named_parameters()})
        return out.detach(), xd.grad, params

    out1, gx1, p1 = grads(1)
    out2, gx2, p2 = grads(2)
    assert_chain_close(out2, out1, "out", 2e-2)
    assert_chain_close(gx2, gx1, "gx", 3e-2)
    for name in p1:
        rr = relrms(p2[name], p1[name])
        assert rr < 4e-2, f"grad {name}: rel-RMS {rr:.3g}"


@pytest.mark.parametrize("B, H, T", [(2, 2, 130), (1, 2, 4096)])
def test_cuda_graph_replay_is_bit_identical(B, H, T):
    import rwkv_lm_ext_b200 as M
    C = H * 64
    r, k, v, w, u, gy, s0, gT = inputs(B, T, H, 17, torch.float32)
    leaves = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    gy, gT = gy.to(DEV), gT.to(DEV)

    def step():
        y, sT = M.RUN_CUDA_RWKV6_STATE_BPTT(B, T, C, H, *leaves)
        return (y, sT) + torch.autograd.grad((y, sT), leaves, (gy, gT))

    eager = [t.detach().clone() for t in step()]        # (holding the autograd graph would pin its AccumulateGrad streams)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        for name, a, b in zip(("y", "s_final", "gr", "gk", "gv", "gw", "gu", "gs"), static, eager):
            assert torch.equal(a, b), name
