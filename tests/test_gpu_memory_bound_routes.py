"""The memory-bound kernels around the recurrence on the routes and at the sizes the per-op tests do not reach:

A. the token-shift backward at shapes whose splits start in the middle of a sequence, against fp64 autograd, and the
   same kernel under every setting of the WKV6 route selector;
B. the later passes of every grid-stride loop (the grid is capped at 148*16 blocks of 256 threads), with a shift
   state so that the t == 0 rows of later passes must find their own row of it;
C. tensors that are contiguous views at an element offset, which the wrappers must copy to 16-byte aligned storage.

Forwards that reproduce the eager bf16 chain op by op are compared bit for bit; gradients against fp64.  `pytest -m gpu`."""
import pytest
import torch

from oracle import wkv6_oracle as O
from rwkv_lm_ext_b200 import heads
from tests.util import assert_bf16_close

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def M():
    import rwkv_lm_ext_b200 as M
    M.load()
    return M


def _randn(*shape, scale=1.0, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(*shape, generator=g, device=DEV) * scale).bfloat16()


def _rand(*shape, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.rand(*shape, generator=g, device=DEV).bfloat16()


def _prev64(x, st):
    """fp64 token shift of the reference (nn.ZeroPad2d((0,0,1,-1)), or the infctx shift state)"""
    B, _, C = x.shape
    prev = torch.zeros(B, 1, C, dtype=x.dtype, device=x.device) if st is None else st.unsqueeze(1)
    return torch.cat([prev, x[:, :-1]], 1) - x


def _eager_shift(x, st):
    """the reference's bf16 xx = shift(x) - x"""
    prev = torch.zeros_like(x[:, :1]) if st is None else st.unsqueeze(1)
    return torch.cat([prev, x[:, :-1]], 1) - x


# --------------------------------------------------------------------------------------------------
# A. token-shift backward
# --------------------------------------------------------------------------------------------------
SHIFT_SHAPES = [
    (3, 130, 768, True),
    (7, 333, 256, True),
    (16, 1, 2048, True),      # every row reads its row of the shift state
    (1, 4097, 64, False),     # C = 64 leaves 3/4 of the column lanes idle
    (9, 129, 512, True),
    (5, 77, 320, False),      # C = 320: the second column block is 1/4 live
]
SHAPE_IDS = [f"{B}x{T}x{C}{'_state' if s else ''}" for B, T, C, s in SHIFT_SHAPES]


def _shift_inputs(B, T, C, with_state, seed):
    x = _randn(B, T, C, seed=seed)
    maa_x = _rand(C, seed=seed + 1)
    maa = _rand(5, C, seed=seed + 2)
    m = _randn(5, B, T, C, scale=0.3, seed=seed + 3)
    st = _randn(B, C, seed=seed + 4) if with_state else None
    go1 = _randn(B, T, C, seed=seed + 5)
    go5 = _randn(5, B, T, C, seed=seed + 6)
    return x, maa_x, maa, m, st, go1, go5


def _run_shift_backward(M, impl, x, maa_x, maa, m, st, go1, go5):
    """gradients of tmix_shift_lerp (x, maa_x, st) and tmix_ddlerp_mix (x, maa, m, st) under one route setting"""
    M.set_impl(impl)
    try:
        leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (x, maa_x, maa, m, st)]
        lx, lmaa_x, lmaa, lm, lst = leaves
        out1 = M.tmix_shift_lerp(lx, lmaa_x, lst)
        g1 = torch.autograd.grad(out1, [t for t in (lx, lmaa_x, lst) if t is not None], go1)
        out5 = M.tmix_ddlerp_mix(lx, lmaa, lm, lst)
        g5 = torch.autograd.grad(list(out5), [t for t in (lx, lmaa, lm, lst) if t is not None], list(go5.unbind(0)))
        torch.cuda.synchronize()
    finally:
        M.set_impl("auto")
    return g1, g5


@pytest.mark.parametrize("B,T,C,with_state", SHIFT_SHAPES, ids=SHAPE_IDS)
def test_shift_lerp_backward_against_fp64(M, B, T, C, with_state):
    x, maa_x, maa, m, st, go1, go5 = _shift_inputs(B, T, C, with_state, seed=B * 1000 + T)
    g1, g5 = _run_shift_backward(M, "auto", x, maa_x, maa, m, st, go1, go5)

    l64 = [t.double().requires_grad_(True) if t is not None else None for t in (x, maa_x, maa, m, st)]
    x64, maa_x64, maa64, m64, st64 = l64
    xx = _prev64(x64, st64)
    want1 = torch.autograd.grad(x64 + xx * maa_x64, [t for t in (x64, maa_x64, st64) if t is not None], go1.double())
    out5 = torch.stack([x64 + xx * (maa64[n] + m64[n]) for n in range(5)])
    want5 = torch.autograd.grad(out5, [t for t in (x64, maa64, m64, st64) if t is not None], go5.double())
    for name, got, want in zip(("gx", "gmaa_x", "gshift"), g1, want1):
        assert_bf16_close(got, want, f"shift_lerp {name}")
    for name, got, want in zip(("gx", "gmaa", "gm", "gshift"), g5, want5):
        assert_bf16_close(got, want, f"ddlerp {name}")


@pytest.mark.parametrize("B,T,C,with_state", SHIFT_SHAPES, ids=SHAPE_IDS)
def test_shift_lerp_backward_is_the_same_kernel_under_simt(M, B, T, C, with_state):
    """set_impl chooses the route of the WKV6 recurrence only: under "simt" the profiler shows the TMA-fed kernel of
    "auto" and nothing else, and every gradient is bit-equal (the kernel and the partial sums have no atomics)."""
    args = _shift_inputs(B, T, C, with_state, seed=B * 1000 + T + 7)
    got = {}
    for impl in ("auto", "simt"):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            got[impl] = _run_shift_backward(M, impl, *args)
        names = {e.name for e in prof.events()}
        assert any("ddlerp_bwd_tma_kernel" in n for n in names) and not any("ddlerp_bwd_kernel" in n for n in names), \
            (impl, sorted(n for n in names if "ddlerp" in n))
    (a1, a5), (s1, s5) = got["auto"], got["simt"]
    for name, a, s in zip(("shift_lerp gx", "shift_lerp gmaa_x", "shift_lerp gshift"), a1, s1):
        assert torch.equal(a, s), name
    for name, a, s in zip(("ddlerp gx", "ddlerp gmaa", "ddlerp gm", "ddlerp gshift"), a5, s5):
        assert torch.equal(a, s), name


@pytest.mark.parametrize("B,T,C,with_state", SHIFT_SHAPES, ids=SHAPE_IDS)
def test_cmix_shift_lerp2_backward_against_fp64(M, B, T, C, with_state):
    x, maa_k, maa_r = _randn(B, T, C, seed=T), _rand(C, seed=T + 1), _rand(C, seed=T + 2)
    st = _randn(B, C, seed=T + 3) if with_state else None
    gk, gr = _randn(B, T, C, seed=T + 4), _randn(B, T, C, seed=T + 5)
    leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (x, maa_k, maa_r, st)]
    xk, xr = M.cmix_shift_lerp2(*leaves)
    xx = _eager_shift(x, st)
    assert torch.equal(xk, x + xx * maa_k) and torch.equal(xr, x + xx * maa_r)
    got = torch.autograd.grad([xk, xr], [t for t in leaves if t is not None], [gk, gr])
    l64 = [t.double().requires_grad_(True) if t is not None else None for t in (x, maa_k, maa_r, st)]
    xx64 = _prev64(l64[0], l64[3])
    want = torch.autograd.grad([l64[0] + xx64 * l64[1], l64[0] + xx64 * l64[2]], [t for t in l64 if t is not None],
                               [gk.double(), gr.double()])
    for name, a, b in zip(("gx", "gmaa_k", "gmaa_r", "gshift"), got, want):
        assert_bf16_close(a, b, f"cmix {name}")


# --------------------------------------------------------------------------------------------------
# B. later passes of the grid-stride loops
# --------------------------------------------------------------------------------------------------
GRID_THREADS = 148 * 16 * 256       # grid_for (cmix.cu, elementwise.cu, elementwise_bwd.cu): 606,208 threads
GRID_WARPS = GRID_THREADS // 32     # the warp-per-token kernels: 18,944 tokens per pass


def _assert_passes(items, per_pass, what):
    """at least three full passes of the capped grid and a ragged last one"""
    assert items > 3 * per_pass and items % per_pass, f"{what}: {items} items = {items / per_pass:.2f} passes"


def test_cmix_pieces_at_the_model_shape(M):
    """B=8, T=4096, D=2048, FFN 7168: shift_lerp_n 13.8 passes (the t = 0 rows of b = 1..7 fall in passes 1..12),
    sigmoid_mul 13.8, relu_sq 48.4."""
    B, T, D, F = 8, 4096, 2048, 7168
    _assert_passes(B * T * D // 8, GRID_THREADS, "shift_lerp_n / sigmoid_mul")
    _assert_passes(B * T * F // 8, GRID_THREADS, "relu_sq")
    x, st = _randn(B, T, D, seed=1), _randn(B, D, seed=2)
    maa_k, maa_r = _rand(D, seed=3), _rand(D, seed=4)
    xk, xr = M.cmix_shift_lerp2(x, maa_k, maa_r, st)
    xx = _eager_shift(x, st)
    assert torch.equal(xk, x + xx * maa_k) and torch.equal(xr, x + xx * maa_r)
    del x, xx, xk, xr

    k = _randn(B, T, F, scale=2.0, seed=5).requires_grad_(True)
    y = M.relu_sq(k)
    assert torch.equal(y, torch.relu(k.detach()) ** 2)
    gy = _randn(B, T, F, seed=6)
    (gk,) = torch.autograd.grad(y, k, gy)
    # 2 * relu(k) * gy of two bf16 numbers is exact in fp32 and in fp64: the kernel's one rounding is the fp64 value's
    assert torch.equal(gk, (2.0 * torch.relu(k.detach().double()) * gy.double()).bfloat16())
    del k, y, gy, gk

    r = _randn(B, T, D, scale=2.0, seed=7).requires_grad_(True)
    kv = _randn(B, T, D, seed=8).requires_grad_(True)
    z = M.sigmoid_mul(r, kv)
    assert torch.equal(z, torch.sigmoid(r.detach()) * kv.detach())
    go = _randn(B, T, D, seed=9)
    gr, gkv = torch.autograd.grad(z, [r, kv], go)
    r64, kv64 = r.detach().double().requires_grad_(True), kv.detach().double().requires_grad_(True)
    gr64, gkv64 = torch.autograd.grad(torch.sigmoid(r64) * kv64, [r64, kv64], go.double())
    assert_bf16_close(gr, gr64, "sigmoid_mul gr")
    assert_bf16_close(gkv, gkv64, "sigmoid_mul gkv")


def test_tmix_and_groupnorm_kernels_over_three_passes(M):
    """ddlerp_mix and GroupNorm*gate stride over B*T*C/8 = 1,844,736 vectors: 3.04 passes, the t = 0 rows of b = 1
    and b = 2 in passes 1 and 2.  shift_lerp has no grid-stride loop (one block per 16 rows of one sequence)."""
    B, T, C, H = 3, 1201, 4096, 64
    _assert_passes(B * T * C // 8, GRID_THREADS, "ddlerp_mix / gn_gate")
    assert all((b * T * C // 8) // GRID_THREADS == b for b in range(B))
    x, st = _randn(B, T, C, seed=11), _randn(B, C, seed=12)
    maa_x, maa = _rand(C, seed=13), _rand(5, C, seed=14)
    m = _randn(5, B, T, C, scale=0.3, seed=15)
    xx = _eager_shift(x, st)
    assert torch.equal(M.tmix_shift_lerp(x, maa_x, st), x + xx * maa_x)
    out = M.tmix_ddlerp_mix(x, maa, m, st)
    for n in range(5):
        assert torch.equal(out[n], x + xx * (maa[n] + m[n])), n
    del m, out, xx

    y, yr, g = _randn(B, T, C, scale=3.0, seed=16), _randn(B, T, C, seed=17), _randn(B, T, C, seed=18)
    lw, lb = (_rand(C, seed=19).float() + 0.5).bfloat16(), _randn(C, scale=0.1, seed=20)
    eps = 64e-5
    idx = torch.full((B, T), 5, dtype=torch.int64, device=DEV)
    idx[1, 700:] = 0                                        # padded rows: lengths T, 700 and 1
    idx[2, 1:] = 0
    _, rev = M.create_mask_and_rev_idx(idx, 1, 0)
    y64, g64 = y.double(), g.double()
    for act in (None, "silu"):
        gate64 = torch.nn.functional.silu(g64) if act else g64
        got = M.groupnorm_gate(y, g, lw, lb, H, eps, gate_act=act)
        assert_bf16_close(got, O.groupnorm_gate(y64, gate64, lw, lb, H, eps), f"gn_gate {act}")
        pair = M.groupnorm_gate_pair(y, yr, rev, g, lw, lb, H, eps, gate_act=act)
        assert torch.equal(pair, M.groupnorm_gate((y + M.reverse_x(yr, rev)) / 2, g, lw, lb, H, eps, gate_act=act))
        ref = O.groupnorm_gate((y64 + O.reverse_x(yr.double(), rev)) / 2, gate64, lw, lb, H, eps)
        assert_bf16_close(pair, ref, f"gn_gate_pair {act}")


def test_gathers_and_scatters_over_three_passes(M):
    """58,000 tokens of D = 264 (a ragged 256-channel inner loop): gather_tokens, stack_reversed and scatter_tokens
    take 3.06 passes of 18,944 warps, scatter_rows 3.16 passes over its 1,914,000 vectors."""
    B, T, D = 29, 2000, 264
    _assert_passes(B * T, GRID_WARPS, "gather_tokens / stack_reversed / scatter_tokens")
    _assert_passes(B * T * D // 8, GRID_THREADS, "scatter_rows")
    g = torch.Generator(device=DEV).manual_seed(21)
    x = _randn(B, T, D, seed=22)
    lens = torch.randint(1, T + 1, (B,), generator=g, device=DEV)
    lens[0], lens[1] = T, 1
    idx = torch.where(torch.arange(T, device=DEV) < lens[:, None], 5, 0)
    _, rev = M.create_mask_and_rev_idx(idx, 1, 0)
    want = torch.gather(x, 1, rev.unsqueeze(-1).expand(-1, -1, D))
    assert torch.equal(M.reverse_x(x, rev), want)
    assert torch.equal(heads.stack_reversed(x, rev), torch.cat([x, want], 0))

    go = _randn(B, T, D, seed=23)
    xg = x.clone().requires_grad_(True)
    (got,) = torch.autograd.grad(M.reverse_x(xg, rev), xg, go)
    (ref,) = torch.autograd.grad(torch.gather(xg, 1, rev.unsqueeze(-1).expand(-1, -1, D)), xg, go)
    assert torch.equal(got, ref)

    pos = torch.randint(-T, T, (B,), generator=g, device=DEV)
    go_rows = _randn(B, D, seed=24)
    (got,) = torch.autograd.grad(M.gather_rows(xg, pos), xg, go_rows)
    ref = torch.zeros_like(x)
    ref[torch.arange(B, device=DEV), pos] = go_rows
    assert torch.equal(got, ref)


# --------------------------------------------------------------------------------------------------
# C. contiguous views at an element offset
# --------------------------------------------------------------------------------------------------
def _offset_copy(t, requires_grad):
    """(storage, view): a contiguous view, one element past a 16-byte boundary, of a copy of t"""
    n = t.numel()
    buf = torch.zeros(n + 16 // t.element_size(), dtype=t.dtype, device=t.device)
    buf[1:1 + n].copy_(t.reshape(-1))
    buf.requires_grad_(requires_grad)
    view = buf[1:1 + n].view(t.shape)
    assert view.is_contiguous() and view.data_ptr() % 16 != 0
    return buf, view


def _same_on_offset_views(fn, inputs, gouts=None):
    """fn on aligned leaves and on offset views of copies of them: outputs, and the gradients of all inputs for the
    (likewise offset) output gradients, bit-equal"""
    grad = gouts is not None
    leaves = [t.clone().requires_grad_(grad) for t in inputs]
    outs = fn(*leaves)
    outs = list(outs) if isinstance(outs, (tuple, list)) else [outs]
    bufs, views = zip(*[_offset_copy(t, grad) for t in inputs])
    outs_v = fn(*views)
    outs_v = list(outs_v) if isinstance(outs_v, (tuple, list)) else [outs_v]
    for a, b in zip(outs, outs_v):
        assert torch.equal(a, b)
    if grad:
        torch.autograd.backward(outs, gouts)
        torch.autograd.backward(outs_v, [_offset_copy(g, False)[1] for g in gouts])
        for leaf, buf in zip(leaves, bufs):
            assert torch.equal(leaf.grad, buf.grad[1:1 + leaf.numel()].view(leaf.shape))


def test_offset_views_give_the_results_of_aligned_copies(M):
    B, T, C, H, R = 2, 37, 128, 2, 32
    x, st = _randn(B, T, C, seed=31), _randn(B, C, seed=32)
    maa_x, maa = _rand(C, seed=33), _rand(5, C, seed=34)
    m = _randn(5, B, T, C, scale=0.3, seed=35)
    h, w2 = torch.tanh(_randn(B * T, 5 * R, seed=36).float()).bfloat16(), _randn(5, R, C, scale=0.1, seed=37)
    go = [_randn(B, T, C, seed=40 + n) for n in range(5)]
    _same_on_offset_views(lambda *a: M.tmix_shift_lerp(*a), [x, maa_x, st], go[:1])
    _same_on_offset_views(lambda *a: M.tmix_ddlerp_mix(*a), [x, maa, m, st], go)
    _same_on_offset_views(lambda *a: M.tmix_ddlerp_lora(*a), [x, maa, h, w2, st], go)
    _same_on_offset_views(lambda *a: M.cmix_shift_lerp2(*a), [x, maa_x, maa[0], st], go[:2])
    _same_on_offset_views(lambda a: M.relu_sq(a), [x], go[:1])
    _same_on_offset_views(lambda a, b: M.sigmoid_mul(a, b), [x, go[1]], go[2:3])

    lw, lb = (_rand(C, seed=50).float() + 0.5).bfloat16(), _randn(C, scale=0.1, seed=51)
    for act in (None, "silu"):
        _same_on_offset_views(lambda y, g, w, b: M.groupnorm_gate(y, g, w, b, H, 64e-5, gate_act=act), [x, go[0], lw, lb], go[1:2])
    idx = torch.full((B, T), 5, dtype=torch.int64, device=DEV)
    idx[1, 20:] = 0
    _, rev = M.create_mask_and_rev_idx(idx, 1, 0)
    with torch.no_grad():
        _same_on_offset_views(lambda y, yr, g: M.groupnorm_gate_pair(y, yr, rev, g, lw, lb, H, 64e-5), [x, go[0], go[1]])
        _same_on_offset_views(lambda a: heads.stack_reversed(a, rev), [x])
    _same_on_offset_views(lambda a: M.reverse_x(a, rev), [x], go[:1])
    pos = torch.tensor([3, -1], device=DEV)
    _same_on_offset_views(lambda a: M.gather_rows(a, pos), [x], [go[0][:, 0]])
    alen = torch.tensor([36, 20], device=DEV)
    gpool = torch.randn(B, C, device=DEV)
    _same_on_offset_views(lambda a: M.pooling(a, alen, "weightedmean", "infer"), [x], [gpool])
    _same_on_offset_views(lambda a: M.pooling(a, alen, "avg", "train"), [x], [gpool.bfloat16()])
