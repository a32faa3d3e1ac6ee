"""ctypes loader of libwkv6_b200.so (the C ABI declared in include/wkv6_b200.h).

There is NO fallback: if the library is missing and cannot be built, importing any operator fails
loudly.  Nothing here imports ``oracle/``.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# WKV6_B200_LIB: load another build of the same library instead (A/B timing of kernel variants, profiles/variants.py)
LIB_PATH = os.environ.get("WKV6_B200_LIB") or os.path.join(_PKG, "libwkv6_b200.so")

c_p, c_i, c_sz, c_i64, c_f = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t, ctypes.c_int64, ctypes.c_float

# name -> (restype, argtypes); mirrors include/wkv6_b200.h one to one
_BTCH = [c_i, c_i, c_i, c_i]
SIGNATURES = {
    "wkv6b200_abi_version": (c_i, []),
    "wkv6b200_seg_plan": (None, [c_i, c_i, c_i, c_i, ctypes.POINTER(c_i), ctypes.POINTER(c_i)]),
    "wkv6b200_last_error": (ctypes.c_char_p, []),
    "wkv6b200_set_impl": (c_i, [c_i]),
    "wkv6b200_get_impl": (c_i, []),
    "wkv6b200_launch_count": (ctypes.c_uint64, []),
    "wkv6b200_set_decay_clamp": (c_f, [c_f]),
    "wkv6_forward": (c_i, _BTCH + [c_p] * 7),
    "wkv6_forward_raww": (c_i, _BTCH + [c_p] * 7),
    "wkv6_backward_workspace_bytes": (c_sz, _BTCH),
    "wkv6_backward": (c_i, _BTCH + [c_p] * 12 + [c_sz, c_p]),
    "wkv6_backward_raww": (c_i, _BTCH + [c_p] * 12 + [c_sz, c_p]),
    "wkv6_saved_bytes": (c_sz, _BTCH),
    "wkv6_train_backward_workspace_bytes": (c_sz, _BTCH + [c_i]),
    "wkv6_train_forward": (c_i, _BTCH + [c_p] * 6 + [c_i, c_i, c_p, c_i, c_p, c_p, ctypes.POINTER(c_i), c_p]),
    "wkv6_train_backward": (c_i, _BTCH + [c_p] * 6 + [c_i] + [c_p] * 10 + [c_sz, c_p]),
    "wkv6_train_backward_state_grad": (c_i, _BTCH + [c_p] * 6 + [c_i] + [c_p] * 9 + [c_i] + [c_p] * 2 + [c_sz, c_p]),
    "wkv6state_forward": (c_i, _BTCH + [c_p] * 8),
    "wkv6state_backward": (c_i, _BTCH + [c_p] * 14 + [c_sz, c_p]),
    "wkv6infctx_forward": (c_i, _BTCH + [c_p] * 8),
    "wkv6infctx_forward_f32state": (c_i, _BTCH + [c_p] * 8),
    "wkv6infctx_backward": (c_i, _BTCH + [c_p] * 14 + [c_sz, c_p]),
    "wkv6_bi_forward": (c_i, _BTCH + [c_p] * 8),
    "wkv6_bi_forward_raww": (c_i, _BTCH + [c_p] * 8),
    "wkv6_bi_backward": (c_i, _BTCH + [c_p] * 13 + [c_sz, c_p]),
    "wkv6_bi_backward_raww": (c_i, _BTCH + [c_p] * 13 + [c_sz, c_p]),
    "rwkv6_forward": (c_i, [c_i] + _BTCH + [c_p] * 8),
    "rwkv6_forward_raww": (c_i, _BTCH + [c_p] * 8),
    "eos_index_i64": (c_i, [c_i, c_i, c_p, c_i64, c_p, c_p]),
    "gather_rows_bf16": (c_i, [c_i, c_i, c_i, c_p, c_p, c_p, c_p]),
    "pooling_bf16": (c_i, [c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p]),
    "create_mask_rev_idx": (c_i, [c_i, c_i, c_p, c_i64, c_i64, c_p, c_p, c_p]),
    "gather_tokens_bf16": (c_i, [c_i, c_i, c_i, c_p, c_p, c_p, c_p]),
    "stack_reversed_bf16": (c_i, [c_i, c_i, c_i, c_p, c_p, c_p, c_p]),
    "tmix_ddlerp_mix_bf16": (c_i, [c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p]),
    "tmix_ddlerp_lora_bf16": (c_i, [c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "tmix_shift_lerp_bf16": (c_i, [c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p]),
    "groupnorm_gate_bf16": (c_i, [c_i, c_i, c_i, c_f, c_i, c_p, c_p, c_p, c_p, c_p, c_p]),
    "groupnorm_gate_pair_bf16": (c_i, [c_i, c_i, c_i, c_i, c_f, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "elementwise_backward_workspace_bytes": (c_sz, [c_i, c_i, c_i, c_i]),
    "tmix_ddlerp_mix_backward_bf16": (c_i, [c_i, c_i, c_i] + [c_p] * 14 + [c_sz, c_p]),
    "tmix_shift_lerp_backward_bf16": (c_i, [c_i, c_i, c_i] + [c_p] * 8 + [c_sz, c_p]),
    "groupnorm_gate_backward_bf16": (c_i, [c_i, c_i, c_i, c_f, c_i] + [c_p] * 10 + [c_sz, c_p]),
    "pooling_backward_bf16": (c_i, [c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p]),
    "scatter_rows_bf16": (c_i, [c_i, c_i, c_i, c_p, c_p, c_p, c_p]),
    "add_layernorm_bf16": (c_i, [ctypes.c_longlong, c_i, c_f] + [c_p] * 8),
    "add_layernorm_backward_workspace_bytes": (c_sz, [ctypes.c_longlong, c_i]),
    "add_layernorm_backward_bf16": (c_i, [ctypes.c_longlong, c_i] + [c_p] * 9 + [c_sz, c_p]),
    "cmix_shift_lerp2_bf16": (c_i, [c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p]),
    "cmix_shift_lerp2_backward_bf16": (c_i, [c_i, c_i, c_i] + [c_p] * 9 + [c_sz, c_p]),
    "relu_sq_bf16": (c_i, [c_sz, c_p, c_p, c_p]),
    "relu_sq_backward_bf16": (c_i, [c_sz, c_p, c_p, c_p, c_p]),
    "sigmoid_mul_bf16": (c_i, [c_sz, c_p, c_p, c_p, c_p]),
    "sigmoid_mul_backward_bf16": (c_i, [c_sz, c_p, c_p, c_p, c_p, c_p, c_p]),
    "scatter_tokens_bf16": (c_i, [c_i, c_i, c_i, c_p, c_p, c_p, c_p]),
    "cross_entropy_l2wrap_bf16": (c_i, [ctypes.c_longlong, c_i, c_p, c_p, ctypes.c_longlong, c_p, c_p, c_p, c_p]),
    "cross_entropy_l2wrap_backward_bf16": (c_i, [ctypes.c_longlong, c_i, c_p, c_p, ctypes.c_longlong, c_p, c_p, c_p, c_p, c_f, c_p, c_p]),
}

_lib = None
ABI_VERSION = 4   # == wkv6b200_abi_version() of the library this signature table was written for


class Wkv6B200Error(RuntimeError):
    pass


def load(build_if_missing: bool = True):
    """Return the loaded library; raise if it is not there (never falls back to anything else)."""
    global _lib
    if _lib is not None:
        return _lib
    have_nvcc = os.path.exists(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"))
    if build_if_missing and have_nvcc and not os.environ.get("WKV6_B200_LIB"):
        from .build import build_library
        build_library()                  # returns at once unless a source or the header is newer than the library
    elif not os.path.exists(LIB_PATH):
        raise Wkv6B200Error(f"{LIB_PATH} is missing: run `python -m rwkv_lm_ext_b200.build` "
                            "(there is no CPU or eager fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header and library disagree
        fn.restype, fn.argtypes = res, args
    if lib.wkv6b200_abi_version() != ABI_VERSION:
        raise Wkv6B200Error(f"{LIB_PATH} has ABI version {lib.wkv6b200_abi_version()}, this package needs {ABI_VERSION}: rebuild it")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().wkv6b200_last_error().decode(errors="replace")
        raise Wkv6B200Error(f"{what} failed with code {rc}: {msg}")


def require_current_device(t):
    """The library takes its stream from the tensor's device but its scratch (memory pool, function attributes)
    from the CURRENT device: a tensor on another device must be used under `torch.cuda.device(t.device)`."""
    import torch
    if not t.is_cuda:
        raise Wkv6B200Error("rwkv_lm_ext_b200 runs on CUDA tensors only (no CPU fallback)")
    if t.device.index != torch.cuda.current_device():
        raise Wkv6B200Error(f"tensor on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}: "
                            "wrap the call in `with torch.cuda.device(t.device):`")


def ptr(t):
    return None if t is None else t.data_ptr()


def stream_of(t):
    import torch
    return torch.cuda.current_stream(t.device).cuda_stream


def launch_count() -> int:
    return int(load().wkv6b200_launch_count())


IMPL = {"auto": 0, "simt": 1, "tc": 2}


def set_decay_clamp(nats_per_token: float) -> float:
    """Opt-in floor of the per-token log-decay (include/wkv6_b200.h); 0 = off.  Returns the previous value."""
    return float(load().wkv6b200_set_decay_clamp(float(nats_per_token)))


def set_impl(name: str) -> str:
    prev = load().wkv6b200_set_impl(IMPL[name])
    return {v: k for k, v in IMPL.items()}[prev]
