"""Whole-model infctx training chunk by chunk (infctx.infctx_train_step) and the fp32 state gradient under it
(ops.WKV_6STATE_BPTT(fp32_state_grad=True), wkv6_train_backward_state_grad_ex).  Checked against the fp64 oracle,
against one pass over the whole sequence (exact mode), against the reference's truncated graph written out by hand
(truncated mode), for bit-exact recomputation, and for a peak memory that does not grow with the chunk count.
`pytest -m gpu`; the measured errors are printed (-s)."""
import pytest
import torch

from tests.test_gpu_state_grad import inputs, nseg_of, oracle
from tests.util import assert_bf16_close, relrms

pytestmark = pytest.mark.gpu
DEV = "cuda"


# ------------------------------------------------------------------------------------------------
# operator: fp32 dL/dS_0
# ------------------------------------------------------------------------------------------------
def _op_grads(r, k, v, w, u, s0, gy, gT, fp32_gs):
    import rwkv_lm_ext_b200 as M
    B, T, C = r.shape
    leaves = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    y, sT = M.RUN_CUDA_RWKV6_STATE_BPTT(B, T, C, C // 64, *leaves, fp32_state_grad=fp32_gs)
    outs, grads = [y], [gy.to(DEV)]
    if gT is not None:
        outs.append(sT)
        grads.append(gT.to(DEV))
    torch.autograd.backward(outs, grads)
    return [t.grad for t in leaves]


def _check_fp32_gs(B, T, H, seed):
    r, k, v, w, u, gy, s0, gT = inputs(B, T, H, seed, torch.float32)
    _, _, g_ref = oracle(r, k, v, w, u, s0, gy, gT)
    g16 = _op_grads(r, k, v, w, u, s0, gy, gT, False)
    g32 = _op_grads(r, k, v, w, u, s0, gy, gT, True)
    assert g32[5].dtype == torch.float32
    assert_bf16_close(g32[5], g_ref[5], "gs (fp32)")
    e16, e32 = relrms(g16[5], g_ref[5]), relrms(g32[5], g_ref[5])
    print(f"\n[fp32 gs] B={B} T={T} H={H}: rel-RMS vs fp64  bf16 gs {e16:.3e}  fp32 gs {e32:.3e}")
    assert e32 <= e16, (e32, e16)
    for name, a, b in zip(("gr", "gk", "gv", "gw", "gu"), g32, g16):    # only the store of gs differs
        assert torch.equal(a, b), name


@pytest.mark.parametrize("T", [1, 63, 65, 1000])
def test_fp32_state_grad_against_fp64_oracle(T):
    assert nseg_of(2, T, 2) == 1
    _check_fp32_gs(2, T, 2, 21 + T)


@pytest.mark.parametrize("B, H, T", [(1, 2, 4096), (2, 3, 8192)])
def test_fp32_state_grad_segmented_route(B, H, T):
    assert nseg_of(B, T, H) > 1
    _check_fp32_gs(B, T, H, 23)


def test_fp32_state_grad_simt_route():
    import rwkv_lm_ext_b200 as M
    prev = M.set_impl("simt")
    try:
        _check_fp32_gs(2, 130, 2, 25)
    finally:
        M.set_impl(prev)


def test_fp32_state_grad_without_final_state_gradient():
    """The last chunk of a reverse sweep has no gT: the fp32 gs then matches the bf16 one to bf16 rounding."""
    r, k, v, w, u, gy, s0, _ = inputs(2, 130, 2, 27, torch.float32)
    g16 = _op_grads(r, k, v, w, u, s0, gy, None, False)
    g32 = _op_grads(r, k, v, w, u, s0, gy, None, True)
    assert torch.equal(g32[5].to(torch.bfloat16).float(), g16[5])
    for name, a, b in zip(("gr", "gk", "gv", "gw"), g32, g16):
        assert torch.equal(a, b), name


def _slow_decays(B, T, H):
    """Per-channel decay logits constant in time, init_like_reference's time_decay of a model's last layer (-6 ... -1,
    exponent 2): the slowest channels keep exp(-exp(-6) * 1024) = 8 % of the state across a 1024-token chunk, so the
    gradient carried across chunk boundaries reaches dL/dS_0, as in a model."""
    C = H * 64
    n = torch.arange(C, dtype=torch.float32)
    return (-6 + 5 * (n / (C - 1)) ** 2.0).view(1, 1, C).expand(B, T, C).contiguous().bfloat16()


def test_long_chain_state_gradient_carry():
    """16 chained calls of 1024 tokens, fp32 state carry, the state gradient flowing back through all of them, with
    the carried gradient in bf16 and in fp32, against fp64 autograd of the oracle over the 16384 tokens (and one call
    over them): dL/dS_0 and gw.  The decays carry the state across chunks, and dL/dS_0 is checked to depend on the
    gradient that crosses the boundaries."""
    import rwkv_lm_ext_b200 as M
    from oracle import wkv6_oracle as O
    from rwkv_lm_ext_b200.synthetic import make_inputs
    B, H, L, n = 1, 2, 1024, 16
    T, C = L * n, H * 64
    r, k, v, _, u, gy = make_inputs(B, T, H, 29)
    w = _slow_decays(B, T, H)
    g = torch.Generator().manual_seed(30)
    s0 = torch.randn(B, H, 64, 64, generator=g) * 0.3
    gT = torch.randn(B, H, 64, 64, generator=g)
    gy, gT = gy.to(DEV), gT.to(DEV)

    lv = [t.detach().to(DEV).double().requires_grad_(True) for t in (r, k, v, w, u, s0)]
    y, S = O.wkv6_recurrence(*lv[:5], lv[5].transpose(-1, -2))
    ((y * gy.double()).sum() + (S.transpose(-1, -2) * gT.double()).sum()).backward()
    gs_ref, gw_ref = lv[5].grad, lv[3].grad
    del y, S, lv

    def whole():
        lv = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
        y, sT = M.RUN_CUDA_RWKV6_STATE_BPTT(B, T, C, H, *lv, fp32_state_grad=True)
        torch.autograd.backward([y, sT], [gy, gT])
        return lv[5].grad, lv[3].grad

    def chained(fp32_gs, gy_=gy, gT_=gT):
        lv = [t.detach().to(DEV).clone().requires_grad_(True) for t in (r, k, v, w, u, s0)]
        s, ys = lv[5], []
        for c in range(n):
            sl = slice(c * L, (c + 1) * L)
            yc, s = M.RUN_CUDA_RWKV6_STATE_BPTT(B, L, C, H, *(t[:, sl].contiguous() for t in lv[:4]), lv[4], s,
                                                fp32_state_grad=fp32_gs)
            ys.append(yc)
        torch.autograd.backward([torch.cat(ys, 1), s], [gy_, gT_])
        return lv[5].grad, lv[3].grad

    (gs1, gw1), (gs16, gw16), (gs32, gw32) = whole(), chained(False), chained(True)
    # the same chain with the loss of chunk 0 only: what dL/dS_0 would be without the carried gradient
    gy0 = gy.clone()
    gy0[:, L:] = 0
    gs_local, _ = chained(True, gy0, torch.zeros_like(gT))
    carried = relrms(gs_local, gs32)
    # gs_fp32_carry_bf16out: the fp32-carry result rounded to bf16 once at the end, like the bf16-carry one, so that
    # the difference to gs_bf16_carry is what the 15 roundings of the carried gradient cost
    e = {"gs_one_call": relrms(gs1, gs_ref), "gs_bf16_carry": relrms(gs16, gs_ref), "gs_fp32_carry": relrms(gs32, gs_ref),
         "gs_fp32_carry_bf16out": relrms(gs32.bfloat16().float(), gs_ref),
         "gw_one_call": relrms(gw1, gw_ref), "gw_bf16_carry": relrms(gw16, gw_ref), "gw_fp32_carry": relrms(gw32, gw_ref),
         "gw0_bf16_carry": relrms(gw16[:, :L], gw_ref[:, :L]), "gw0_fp32_carry": relrms(gw32[:, :L], gw_ref[:, :L])}
    print(f"\n[carry 16 x 1024] carried share of dL/dS_0 {carried:.3f}; rel-RMS vs fp64: "
          + "  ".join(f"{k_} {v_:.3e}" for k_, v_ in e.items())
          + f"  ratio gs bf16/fp32 {e['gs_bf16_carry'] / e['gs_fp32_carry']:.2f}")
    assert carried > 0.02                          # the boundaries' gradient reaches chunk 0
    assert_bf16_close(gs32, gs_ref, "gs (fp32 carry)")
    assert_bf16_close(gw32, gw_ref, "gw (fp32 carry)")
    assert e["gs_fp32_carry"] < e["gs_bf16_carry"]
    assert e["gs_fp32_carry_bf16out"] <= e["gs_bf16_carry"] * 1.01
    assert e["gw_fp32_carry"] <= e["gw_bf16_carry"] * 1.01


# ------------------------------------------------------------------------------------------------
# the model driver
# ------------------------------------------------------------------------------------------------
def _model(seed=0, layers=3, D=128, H=2, vocab=512):
    from rwkv_lm_ext_b200 import sft
    m = sft.RwkvSft(layers=layers, D=D, H=H, ffn=int(3.5 * D) // 32 * 32, vocab=vocab, train_type="full")
    return sft.init_like_reference(m, seed=seed).bfloat16().to(DEV)


def _data(B, T, vocab=512, seed=1):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(0, vocab, (B, T + 1), generator=g)
    return idx[:, :-1].contiguous().to(DEV), idx[:, 1:].contiguous().to(DEV)


def _grads(model):
    out = {n: p.grad.detach().float().clone() for n, p in model.named_parameters()}
    model.zero_grad(set_to_none=True)
    return out


def _states(model, B, wkv_dtype=torch.float32):
    import rwkv_lm_ext_b200 as M
    L, C, H = len(model.blocks), model.emb.weight.shape[1], model.blocks[0].att.time_faaaa.shape[0]
    return M.BlockStateList.create(L, B, C, H, DEV, torch.bfloat16, wkv_dtype=wkv_dtype)


def _whole_pass(model, idx, tgt):
    import rwkv_lm_ext_b200 as M
    from rwkv_lm_ext_b200.sft import sft_loss
    logits, _ = M.infctx_forward(model, idx, _states(model, idx.shape[0]))
    loss = sft_loss(logits, tgt)
    loss.backward()
    return float(loss), _grads(model)


@pytest.mark.parametrize("B, T, chunk", [(2, 4 * 512, 512), (2, 3 * 512 + 130, 512), (1, 2 * 2048, 2048)])
def test_exact_mode_equals_one_pass(B, T, chunk):
    """Exact mode against one pass over the whole sequence: the loss to 1e-3, all parameter gradients as one vector to
    1e-2 rel-RMS, every parameter to 4e-2 (the bound of test_gpu_state_grad's chunked layer: the parameters with the
    smallest gradients, such as time_maa_w, are sums of many bf16 terms), and closer than the truncated gradient on
    the recurrence's decay."""
    import rwkv_lm_ext_b200 as M
    model = _model()
    H = 2
    if chunk == 2048:
        assert B * H <= 74 and nseg_of(B, chunk, H) > 1                    # every WKV call is time-segmented
    idx, tgt = _data(B, T)
    loss1, g1 = _whole_pass(model, idx, tgt)
    loss, final = M.infctx_train_step(model, idx, tgt, chunk, exact=True)
    g = _grads(model)
    M.infctx_train_step(model, idx, tgt, chunk, exact=False)
    g_tr = _grads(model)
    names = [n for n in g1 if g1[n].norm() > 0]
    rr = {n: relrms(g[n], g1[n]) for n in names}
    worst = max(rr, key=rr.get)

    def flat(d):
        return torch.cat([d[n].flatten() for n in names])
    e_all = relrms(flat(g), flat(g1))
    key = "blocks.0.att.time_decay"
    print(f"\n[exact vs one pass] B={B} T={T} chunk={chunk}: loss {float(loss):.6f} vs {loss1:.6f}, all grads "
          f"rel-RMS {e_all:.3e}, worst {rr[worst]:.3e} ({worst}); {key}: exact {rr[key]:.3e} truncated "
          f"{relrms(g_tr[key], g1[key]):.3e}")
    assert abs(float(loss) - loss1) <= 1e-3 * abs(loss1)
    assert e_all <= 1e-2
    assert rr[worst] <= 4e-2, (worst, rr[worst])
    assert rr[key] < relrms(g_tr[key], g1[key])
    assert final.wkv_states.dtype == torch.float32 and not final.wkv_states.requires_grad


def _hand_truncated(model, idx, tgt, chunk):
    """The reference's truncated graph: the layer functions chained without detach(), one backward()."""
    import rwkv_lm_ext_b200 as M
    from rwkv_lm_ext_b200.sft import sft_loss
    B, T = idx.shape
    st, total = _states(model, B), 0.0
    for t0 in range(0, T, chunk):
        t1 = min(T, t0 + chunk)
        logits, st = M.infctx_forward(model, idx[:, t0:t1], st, exact_state_grad=False)
        total = total + sft_loss(logits, tgt[:, t0:t1]) * ((t1 - t0) / T)
    total.backward()
    return float(total), _grads(model), st


@pytest.mark.parametrize("B, T, chunk", [(2, 4 * 512, 512), (2, 3 * 512 + 130, 512)])
def test_truncated_mode_equals_the_reference_graph(B, T, chunk):
    import rwkv_lm_ext_b200 as M
    model = _model(seed=3)
    idx, tgt = _data(B, T, seed=4)
    loss_h, g_h, st_h = _hand_truncated(model, idx, tgt, chunk)
    loss, final = M.infctx_train_step(model, idx, tgt, chunk, exact=False)
    g = _grads(model)
    assert abs(float(loss) - loss_h) <= 1e-6 * abs(loss_h)
    for n in g_h:
        assert relrms(g[n], g_h[n]) <= 1e-3 if g_h[n].norm() > 0 else torch.equal(g[n], g_h[n]), n
    assert torch.equal(final.wkv_states, st_h.wkv_states) and torch.equal(final.shift_states, st_h.shift_states)
    # the exact gradient differs from the truncated one as soon as there is a boundary to cross
    M.infctx_train_step(model, idx, tgt, chunk, exact=True)
    g_x = _grads(model)
    assert any(not torch.equal(g_x[n], g[n]) for n in g)
    assert relrms(g_x["blocks.0.att.time_decay"], g["blocks.0.att.time_decay"]) > 1e-3


def test_dropout_draws_the_same_masks_in_both_sweeps():
    """LoRA dropout in training mode: the recompute runs from the random-number state the first sweep started each
    chunk from, so the driver's loss, gradients and final states are those of the hand-chained graph drawn from the
    same seed, and the generator ends where that one pass leaves it."""
    import rwkv_lm_ext_b200 as M
    from rwkv_lm_ext_b200 import sft
    m = sft.RwkvSft(layers=3, D=128, H=2, ffn=448, vocab=512, lora_r=8, lora_alpha=16, lora_dropout=0.2)
    sft.init_like_reference(m, seed=11)
    with torch.no_grad():
        for name, p in m.named_parameters():
            if "lora_B" in name:
                p.copy_(torch.randn(p.shape, generator=torch.Generator().manual_seed(12)) * 0.05)
    model = m.bfloat16().to(DEV).train()
    idx, tgt = _data(2, 3 * 512, seed=13)
    torch.manual_seed(123)
    loss_h, g_h, st_h = _hand_truncated(model, idx, tgt, 512)
    after_h = torch.cuda.get_rng_state()
    torch.manual_seed(123)
    loss, final = M.infctx_train_step(model, idx, tgt, 512, exact=False)
    g = _grads(model)
    assert torch.equal(torch.cuda.get_rng_state(), after_h)
    assert abs(float(loss) - loss_h) <= 1e-6 * abs(loss_h)
    assert torch.equal(final.wkv_states, st_h.wkv_states) and torch.equal(final.shift_states, st_h.shift_states)
    for n in g_h:
        assert relrms(g[n], g_h[n]) <= 1e-3 if g_h[n].norm() > 0 else torch.equal(g[n], g_h[n]), n


def test_one_chunk_exact_equals_truncated():
    import rwkv_lm_ext_b200 as M
    model = _model(seed=5)
    idx, tgt = _data(2, 700, seed=6)
    la, _ = M.infctx_train_step(model, idx, tgt, 700, exact=False)
    ga = _grads(model)
    lb, _ = M.infctx_train_step(model, idx, tgt, 1024, exact=True)
    gb = _grads(model)
    assert torch.equal(la, lb)
    for n in ga:
        assert torch.equal(ga[n], gb[n]), n


@pytest.mark.parametrize("B, chunk, n", [(2, 512, 3), (1, 2048, 2), (1, 1000, 3)])
def test_recompute_reproduces_the_stored_states(B, chunk, n):
    """The driver's final states (the last chunk recomputed from the states its first sweep stored) are bit-equal to
    the chain of chunk forwards with autograd on.  A forward-only chunk takes the forward-only segment plan: equal
    where it is the training plan, within 1e-3 rel-RMS where it is not (1 x 2048 x 2 streams)."""
    import rwkv_lm_ext_b200 as M
    H = 2
    model = _model(seed=7)
    idx, tgt = _data(B, chunk * n, seed=8)
    _, final = M.infctx_train_step(model, idx, tgt, chunk, exact=True)
    model.zero_grad(set_to_none=True)
    st_grad = _states(model, B)
    for c in range(n):
        _, st_grad = M.infctx_forward(model, idx[:, c * chunk:(c + 1) * chunk], st_grad)
        st_grad = st_grad.detach()
    assert torch.equal(final.wkv_states, st_grad.wkv_states)
    assert torch.equal(final.shift_states, st_grad.shift_states)
    with torch.no_grad():
        st_ng = _states(model, B)
        for c in range(n):
            _, st_ng = M.infctx_forward(model, idx[:, c * chunk:(c + 1) * chunk], st_ng)
    plans_agree = nseg_of(B, chunk, H) == _nseg_fwd(B, chunk, H)
    rr = relrms(st_ng.wkv_states, st_grad.wkv_states)
    print(f"\n[recompute] B={B} chunk={chunk} x{n}: plans agree {plans_agree}, forward-only vs training route "
          f"wkv-state rel-RMS {rr:.3e}")
    if plans_agree:
        assert torch.equal(st_ng.wkv_states, st_grad.wkv_states)
    else:
        assert rr <= 1e-3


def _nseg_fwd(B, T, H):
    import ctypes
    from rwkv_lm_ext_b200 import _lib
    nseg, sc = ctypes.c_int(0), ctypes.c_int(0)
    _lib.load().wkv6b200_seg_plan(B, T, H, 0, ctypes.byref(nseg), ctypes.byref(sc))
    return nseg.value


def _peak(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def test_peak_memory_is_one_chunk():
    """exact=True at 8 chunks needs at most the 6 extra stored boundaries (+ 1 MB) more than at 2 chunks; chaining
    infctx_forward(exact_state_grad=True) over the chunks with one backward() grows by about a chunk's activations
    per chunk."""
    import rwkv_lm_ext_b200 as M
    B, chunk = 2, 512
    model = _model(seed=9)
    L, C, H = len(model.blocks), model.emb.weight.shape[1], 2
    boundary = L * B * H * 64 * 64 * 4 + L * 2 * B * C * 2
    data = {n: _data(B, n * chunk, seed=10 + n) for n in (2, 8)}

    def driver(n):
        M.infctx_train_step(model, *data[n], chunk, exact=True)
        model.zero_grad(set_to_none=True)

    def naive(n):
        from rwkv_lm_ext_b200.sft import sft_loss
        idx, tgt = data[n]
        st, total = _states(model, B), 0.0
        for c in range(n):
            logits, st = M.infctx_forward(model, idx[:, c * chunk:(c + 1) * chunk], st, exact_state_grad=True)
            total = total + sft_loss(logits, tgt[:, c * chunk:(c + 1) * chunk]) / n
        total.backward()
        model.zero_grad(set_to_none=True)

    for fn in (driver, naive):                      # warm-up: gradients and allocator state of both shapes
        fn(2)
    d2, d8 = _peak(lambda: driver(2)), _peak(lambda: driver(8))
    n2, n8 = _peak(lambda: naive(2)), _peak(lambda: naive(8))
    print(f"\n[memory] driver 2 chunks {d2 / 2**20:.1f} MiB, 8 chunks {d8 / 2**20:.1f} MiB; naive chain {n2 / 2**20:.1f} / "
          f"{n8 / 2**20:.1f} MiB; boundary {boundary / 2**20:.3f} MiB")
    assert d8 - d2 <= 6 * boundary + 2**20
    assert n8 - n2 >= d2 / 2 and n8 - n2 > 10 * (max(d8 - d2, 0) + 2**20)
