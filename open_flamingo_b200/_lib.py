"""ctypes binding of libofk.so (the C ABI declared in include/ofk.h).

There is deliberately NO fallback: if the library is missing or a call fails, a RuntimeError is raised.
torch is used only to own device memory and streams; raw pointers cross the boundary.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# OFK_LIB_VARIANT=<name> loads open_flamingo_b200/libofk_<name>.so instead (A/B builds of a kernel made with
# tools/build_variant.sh; measurement tooling only -- the default and every test use libofk.so)
_VARIANT = os.environ.get("OFK_LIB_VARIANT", "")
LIB_PATH = os.path.join(_HERE, f"libofk_{_VARIANT}.so" if _VARIANT else "libofk.so")

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_ll = ctypes.c_longlong
c_float = ctypes.c_float

# epilogue ids (include/ofk.h)
EPI_STORE_BF16 = 0
EPI_STORE_F32 = 1
EPI_ATOMIC_F32 = 2
EPI_BIAS_BF16 = 3
EPI_BIAS_QGELU_BF16 = 4
EPI_GELU_DUAL = 5
EPI_GATE_RESID_F32 = 6
EPI_DGELU_BF16 = 7
EPI_BIAS_RESID_F32 = 8
EPI_BIAS_GELU_BF16 = 9
EPI_SWIGLU_DUAL = 10
SWIGLU_GROUP = 16   # OFK_SWIGLU_GROUP: gate / up rows interleaved in groups of 16 in the packed SwiGLU weight

MASK_NONE = 0
MASK_MEDIA_EQ = 1
MASK_MEDIA_GE = 2

_SIGNATURES = {
    "ofk_last_error": (ctypes.c_char_p, []),
    "ofk_abi_version": (c_int, []),
    "ofk_launch_count": (c_ll, []),
    "ofk_gemm_bf16": (c_int, [c_int, c_int, c_int, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_int,
                              c_int, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_void_p,
                              c_void_p]),
    "ofk_make_labels": (c_int, [c_void_p, c_ll, c_int, c_int, c_ll, c_ll, c_ll, c_int, c_void_p, c_ll, c_void_p]),
    "ofk_gemm_workspace_bytes": (c_ll, []),
    "ofk_gemm_reserve_sms": (c_int, [c_int]),
    "ofk_gemm_bf16_ws": (c_int, [c_int, c_int, c_int, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_int,
                                 c_int, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_void_p,
                                 c_void_p, c_ll, c_void_p]),
    "ofk_gemm_bf16_grouped": (c_int, [c_int, c_int, c_int, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_int,
                                      c_int, c_void_p, c_ll, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                      c_void_p]),
    "ofk_layernorm_fwd": (c_int, [c_void_p, c_ll, c_void_p, c_void_p, c_float, c_int, c_int, c_void_p,
                                  c_int, c_ll, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "ofk_layernorm_bwd_workspace": (c_ll, [c_int, c_int]),
    "ofk_layernorm_bwd": (c_int, [c_void_p, c_int, c_ll, c_int, c_int, c_int, c_void_p, c_ll, c_void_p, c_void_p,
                                  c_void_p, c_int, c_int, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_void_p,
                                  c_void_p, c_void_p]),
    "ofk_rmsnorm_fwd": (c_int, [c_void_p, c_ll, c_void_p, c_float, c_int, c_int, c_void_p, c_ll, c_void_p, c_void_p]),
    "ofk_rmsnorm_bwd": (c_int, [c_void_p, c_int, c_ll, c_void_p, c_ll, c_void_p, c_void_p, c_int, c_int, c_void_p, c_ll,
                                c_void_p, c_ll, c_void_p]),
    "ofk_rope": (c_int, [c_void_p, c_ll, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_ll, c_int, c_void_p]),
    "ofk_swiglu_bwd": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_void_p, c_ll, c_void_p]),
    "ofk_attn_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                             c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_float, c_int, c_void_p, c_int,
                             c_void_p]),
    "ofk_attn_bwd_workspace_bytes": (c_ll, [c_int, c_int, c_int, c_int, c_int]),
    "ofk_attn_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                             c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll,
                             c_float, c_int, c_void_p, c_int, c_void_p, c_ll, c_void_p]),
    "ofk_attn_dense_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                   c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_ll, c_float, c_int, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "ofk_attn_dense_bwd": (c_int, [c_void_p] * 10 + [c_int] * 5 + [c_ll] * 14 + [c_float, c_int, c_void_p, c_void_p,
                                                                              c_void_p, c_void_p, c_ll, c_void_p]),
    "ofk_attn_force_legacy": (c_int, [c_int]),
    "ofk_attn_tc_launch_count": (c_ll, []),
    "ofk_text_time": (c_int, [c_void_p, c_ll, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "ofk_cast_f32_bf16": (c_int, [c_void_p, c_void_p, c_ll, c_void_p]),
    "ofk_gate_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_void_p]),
    "ofk_add_f32": (c_int, [c_void_p, c_void_p, c_ll, c_void_p]),
    "ofk_patchify": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_ll, c_void_p]),
    "ofk_vit_assemble": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ofk_ce_fwd": (c_int, [c_void_p, c_int, c_ll, c_ll, c_int, c_void_p, c_int, c_int, c_ll, c_void_p, c_void_p, c_void_p,
                           c_void_p]),
    "ofk_ce_bwd": (c_int, [c_void_p, c_int, c_ll, c_ll, c_int, c_void_p, c_int, c_int, c_ll, c_void_p, c_void_p, c_void_p,
                           c_void_p, c_ll, c_void_p]),
    "ofk_adamw": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_float, c_float, c_float,
                          c_float, c_float, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "ofk_sumsq": (c_int, [c_void_p, c_ll, c_void_p, c_void_p]),
}

_lib = None


def exported_symbols():
    """Names every entry point include/ofk.h declares (used by the CPU-side ABI test)."""
    return sorted(_SIGNATURES)


def lib():
    """Load libofk.so (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU/PyTorch fallback for the hot path.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if L.ofk_abi_version() != 2:
            raise RuntimeError("libofk.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().ofk_last_error()
        raise RuntimeError(f"libofk error {rc}: {msg.decode() if msg else ''}")


def launch_count():
    return int(lib().ofk_launch_count())


def ptr(t):
    return 0 if t is None else t.data_ptr()


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    """Every tensor must live on the CURRENT CUDA device: kernels are enqueued on that device's current stream
    (a model moved to cuda:1 without torch.cuda.set_device(1) would otherwise be launched on the wrong GPU)."""
    cur = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("open_flamingo_b200 kernels need CUDA tensors (sm_100a); there is no CPU path")
        if cur is None:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            raise RuntimeError(f"tensor on cuda:{t.device.index} but the current device is cuda:{cur}: call "
                               "torch.cuda.set_device() (one process per GPU) before running the model")
