"""ctypes binding of the reference's OWN CUDA kernels, compiled by `make -C oracle ref REF=<RWKV_LM_EXT checkout>`
from its cuda/*.cu into oracle/_ref/ (git-ignored).
TEST / BENCH INFRASTRUCTURE ONLY: used as a second checker on the GPU and as the
"reference wkv6_cuda" timing beside ours (BASELINE.json configs[1]).  Entry points are the
`cuda_forward` / `cuda_backward` launchers at cuda/wkv6_cuda.cu:229-242 etc. (C++-mangled names).
They launch on the legacy default stream, like the reference does."""
import ctypes
import os

import torch

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
_BF = "PN3c108BFloat16E"
_SYMS = {
    "wkv6": ("_Z12cuda_forwardiiiiPN3c108BFloat16ES1_S1_PfS1_S1_",
             "_Z13cuda_backwardiiiiPN3c108BFloat16ES1_S1_PfS1_S1_S1_S1_S1_S1_S1_"),
    "wkv6state": ("_Z12cuda_forwardiiiiPN3c108BFloat16ES1_S1_S1_S1_S1_S1_",
                  "_Z13cuda_backwardiiiiPN3c108BFloat16ES1_S1_S1_S1_S1_S1_S1_S1_S1_S1_S1_S1_"),
    "wkv6infctx": ("_Z12cuda_forwardiiiiPN3c108BFloat16ES1_S1_S1_S1_S1_S1_",
                   "_Z13cuda_backwardiiiiPN3c108BFloat16ES1_S1_S1_S1_S1_S1_S1_S1_S1_S1_S1_S1_"),
    "wkv6_bi": ("_Z12cuda_forwardiiiiPKiPN3c108BFloat16ES3_S3_PfS3_S3_",
                "_Z13cuda_backwardiiiiPKiPN3c108BFloat16ES3_S3_PfS3_S3_S3_S3_S3_S3_S3_"),
    "rwkv6": ("_Z17cuda_forward_bf16iiiiPfPN3c108BFloat16ES2_S2_S_S2_S2_", None),
}
_libs = {}


def available(name: str = "wkv6") -> bool:
    return os.path.exists(os.path.join(_DIR, f"libref_{name}.so"))


def _lib(name):
    if name not in _libs:
        _libs[name] = ctypes.CDLL(os.path.join(_DIR, f"libref_{name}.so"), mode=ctypes.RTLD_LOCAL)
    return _libs[name]


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def wkv6_forward(r, k, v, w, u):
    """`WKV_6.forward` as the reference runs it (src/model.py:193-214), incl. the fp32 ew pre-pass."""
    B, T, C = r.shape
    H = u.shape[0]
    ew = (-torch.exp(w.float())).contiguous()
    y = torch.empty_like(r)
    getattr(_lib("wkv6"), _SYMS["wkv6"][0])(B, T, C, H, _p(r), _p(k), _p(v), _p(ew), _p(u), _p(y))
    return y, ew


def wkv6_backward(r, k, v, ew, u, gy):
    """`WKV_6.backward` (src/model.py:216-233)."""
    B, T, C = r.shape
    H = u.shape[0]
    gr, gk, gv, gw = (torch.empty_like(r) for _ in range(4))
    gu = torch.empty(B, C, device=r.device, dtype=torch.bfloat16)
    getattr(_lib("wkv6"), _SYMS["wkv6"][1])(B, T, C, H, _p(r), _p(k), _p(v), _p(ew), _p(u), _p(gy),
                                           _p(gr), _p(gk), _p(gv), _p(gw), _p(gu))
    return gr, gk, gv, gw, torch.sum(gu, 0).view(H, C // H)


def state_forward(name, r, k, v, w, u, s):
    """wkv6state / wkv6infctx forward (src/model.py:83-185).  infctx overwrites ``s`` in place."""
    B, T, C = r.shape
    H = u.shape[0]
    y = torch.empty_like(r)
    getattr(_lib(name), _SYMS[name][0])(B, T, C, H, _p(r), _p(k), _p(v), _p(w), _p(u), _p(s), _p(y))
    return y


def bi_forward(mask, r, k, v, w, u):
    """`WKV_6_BI.forward` (cuda/wkv6_bi.py:15-39); y is torch.empty there -- zero it here so the
    positions the reference never writes are comparable."""
    B, T, C = r.shape
    H = u.shape[0]
    ew = (-torch.exp(w.float())).contiguous()
    y = torch.zeros_like(r)
    getattr(_lib("wkv6_bi"), _SYMS["wkv6_bi"][0])(B, T, C, H, _p(mask), _p(r), _p(k), _p(v), _p(ew), _p(u), _p(y))
    return y


def rwkv6_forward_bf16(state, r, k, v, w_decay, u):
    """`RWKV_6.forward` bf16 branch (src/model_run.py:58-66); state fp32 [H,64,64] updated in place."""
    T, C = r.shape
    H = u.shape[0]
    y = torch.empty_like(r)
    getattr(_lib("rwkv6"), _SYMS["rwkv6"][0])(1, T, C, H, _p(state), _p(r), _p(k), _p(v), _p(w_decay), _p(u), _p(y))
    return y
