"""Forward + backward time of the infctx operator with the truncated gradient (WKV_6STATE_INFCTX, the reference's
semantics: the final state is a constant) against the exact one (WKV_6STATE_BPTT: the gradient of the carried state
flows back through every chunk).  Two shapes:
  * BASELINE config 5: 3B shape (H = 40), B = 1, 16 chained calls of 4096 tokens -- the time-segmented route;
  * B = 8, T = 4096, H = 32 (256 streams): the unsegmented route, one call.
fp32 carry, CUDA events, bf16 inputs from rwkv_lm_ext_b200.synthetic; the card's name and power limit are read in
the same run.  Prints one JSON line."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import rwkv_lm_ext_b200 as M
from rwkv_lm_ext_b200.synthetic import make_inputs

M.load()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def chain(chunks, B, T, H, exact):
    """One pass over the chunks carrying the fp32 state; loss = sum <y, gy>; backward through all of them."""
    C = H * 64
    s = torch.zeros(B, H, 64, 64, device="cuda", dtype=torch.float32)
    outs = []
    for (r, k, v, w, u, gy) in chunks:
        leaves = [t.detach().requires_grad_(True) for t in (r, k, v, w, u)]
        if exact:
            y, s = M.RUN_CUDA_RWKV6_STATE_BPTT(B, T, C, H, *leaves, s)
            outs.append((y, gy))
        else:
            y, s = M.WKV_6STATE_INFCTX.apply(B, T, C, H, *leaves, s.detach().clone())
            y.backward(gy)                      # truncated: every chunk's backward stands alone
    if exact:
        torch.autograd.backward([y for y, _ in outs], [gy for _, gy in outs])


def timeit(fn, n=5):
    for _ in range(2):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    res = {"card": card()}
    for name, (B, T, H, n) in {"config5_3b_64k": (1, 4096, 40, 16), "b8_t4096_h32": (8, 4096, 32, 1)}.items():
        chunks = [make_inputs(B, T, H, seed=100 + i, decay="model", device="cuda") for i in range(n)]
        ms = {}
        for rep in range(2):                   # alternate the two settings
            for exact in (False, True):
                key = "exact" if exact else "truncated"
                ms.setdefault(key, []).append(timeit(lambda: chain(chunks, B, T, H, exact)))
        res[name] = {"B": B, "T": T, "H": H, "chunks": n,
                     **{f"fwd_bwd_ms_{k}": round(min(v), 3) for k, v in ms.items()},
                     "exact_over_truncated": round(min(ms["exact"]) / min(ms["truncated"]), 3)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
