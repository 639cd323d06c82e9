"""ctypes binding of libagcn_b200.so (the C ABI declared in include/agcn_b200.h).

There is no CPU fallback: if the shared library is missing or does not load, every
kernel entry point raises ``RuntimeError``.  Build it with ``python -m fusion_gcn_b200.build``
(or ``__graft_entry__.build()``).
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# AGCN_B200_LIB: another build of the same library (e.g. the -DAGCN_PROBES build of tools/, never the product path)
LIB_PATH = os.environ.get("AGCN_B200_LIB") or os.path.join(_HERE, "libagcn_b200.so")

PREC_FP32 = 0          # fp32 parity: 3xTF32 tensor cores where possible, FFMA otherwise
PREC_TF32 = 1          # single-pass TF32 tensor cores
PREC_FP32_FFMA = 2     # force FFMA
PREC_BF16X3 = 3        # fp32 parity on bf16 triple products (h.h + h.m + m.h, tcgen05 kind::f16)
MIX_AGG_FWD, MIX_AGG_BWD, MIX_SCORE_BWD = 0, 1, 2
RES_NONE, RES_TENSOR, RES_AFFINE = 0, 1, 2

_c_int, _c_ll, _c_float, _c_void_p, _c_size_t = ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t
_c_double = ctypes.c_double

# name -> (restype, argtypes); mirrors include/agcn_b200.h one to one
SIGNATURES = {
    "agcn_version": (_c_int, []),
    "agcn_last_error_string": (ctypes.c_char_p, []),
    "agcn_launch_count": (_c_ll, []),
    "agcn_conv_fwd_workspace_bytes": (_c_size_t, [_c_int] * 4),
    "agcn_conv_fwd": (_c_int, [_c_void_p] * 4 + [_c_int] * 12 + [_c_void_p, _c_size_t, _c_void_p]),
    "agcn_conv_fwd_post": (_c_int, [_c_void_p] * 6 + [_c_int, _c_void_p] + [_c_int] * 10 + [_c_void_p, _c_size_t, _c_void_p]),
    "agcn_conv_fwd_stats_bytes": (_c_size_t, [_c_int]),
    "agcn_conv_fwd_stats": (_c_int, [_c_void_p] * 4 + [_c_int] * 10 + [_c_void_p, _c_size_t, _c_void_p, _c_size_t, ctypes.POINTER(_c_int), _c_void_p]),
    "agcn_conv_wgrad_workspace_bytes": (_c_size_t, [_c_int] * 7),
    "agcn_conv_wgrad": (_c_int, [_c_void_p] * 4 + [_c_int] * 9 + [_c_void_p, _c_size_t, _c_int, _c_void_p]),
    "agcn_conv_wgrad_presplit": (_c_int, [_c_void_p] * 3 + [_c_int] * 9 + [_c_void_p, _c_size_t, _c_void_p]),
    "agcn_joint_gram": (_c_int, [_c_void_p] * 3 + [_c_int] * 13 + [_c_void_p]),
    "agcn_attention_fwd": (_c_int, [_c_void_p] * 5 + [_c_int] * 4 + [_c_float, _c_void_p]),
    "agcn_attention_bwd": (_c_int, [_c_void_p] * 5 + [_c_int] * 4 + [_c_float, _c_void_p]),
    "agcn_joint_mix_workspace_bytes": (_c_size_t, [_c_int]),
    "agcn_joint_mix": (_c_int, [_c_void_p] * 3 + [_c_int] * 9 + [_c_void_p, _c_size_t, _c_void_p]),
    "agcn_joint_mix_score_bwd_colsum_workspace_bytes": (_c_size_t, [_c_int, _c_int]),
    "agcn_joint_mix_score_bwd_colsum": (_c_int, [_c_void_p] * 4 + [_c_int] * 5 + [_c_void_p, _c_size_t, _c_void_p]),
    "agcn_bn_workspace_bytes": (_c_size_t, [_c_int]),
    "agcn_bn_stats": (_c_int, [_c_void_p, _c_int, _c_int, _c_ll, _c_int] + [_c_void_p] * 5 + [_c_float, _c_float, _c_int]
                      + [_c_void_p] * 4 + [_c_void_p, _c_size_t, _c_void_p]),
    "agcn_bn_finalize": (_c_int, [_c_void_p, _c_int, _c_ll, _c_int] + [_c_void_p] * 5 + [_c_float, _c_float] + [_c_void_p] * 5),
    "agcn_bn_apply": (_c_int, [_c_void_p] * 3 + [_c_int] + [_c_void_p] * 3 + [_c_int] + [_c_void_p] * 3 + [_c_int, _c_int, _c_ll, _c_int, _c_void_p]),
    "agcn_bn_mask_words": (_c_size_t, [_c_int] * 3),
    "agcn_bn_bwd": (_c_int, [_c_void_p] * 12 + [_c_int, _c_int, _c_int, _c_int, _c_ll, _c_int, _c_int, _c_int, _c_void_p, _c_double,
                             _c_void_p, _c_size_t, _c_void_p]),
    "agcn_pool_fwd": (_c_int, [_c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_void_p]),
    "agcn_pool_bwd": (_c_int, [_c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_void_p]),
    "agcn_bn_apply_pool_workspace_bytes": (_c_size_t, [_c_int, _c_int]),
    "agcn_bn_apply_pool": (_c_int, [_c_void_p] * 3 + [_c_int] + [_c_void_p] * 3 + [_c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_void_p, _c_size_t, _c_void_p]),
    "agcn_bn_bwd_bits_dual": (_c_int, [_c_void_p] * 17 + [_c_int, _c_int, _c_int, _c_void_p, _c_size_t, _c_void_p]),
    "agcn_bn_stats_partials_bytes": (_c_size_t, [_c_int]),
    "agcn_bn_stats_partials": (_c_int, [_c_void_p, _c_int, _c_int, _c_ll, _c_int, _c_void_p, _c_size_t, _c_void_p, _c_void_p, _c_size_t, _c_void_p]),
    "agcn_linear_ce_fwd": (_c_int, [_c_void_p] * 8 + [_c_int] * 3 + [_c_void_p]),
    "agcn_linear_ce_bwd": (_c_int, [_c_void_p] * 7 + [_c_int] * 3 + [_c_void_p]),
    "agcn_node_mix": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_int, _c_int, _c_void_p]),
    "agcn_bucket_copy": (_c_int, [_c_void_p, _c_void_p, _c_int, _c_int, _c_float, _c_void_p]),
    "agcn_optim_chunk": (_c_int, []),
    "agcn_optim_sgd": (_c_int, [_c_void_p, _c_void_p, _c_int, _c_double, _c_void_p, _c_double, _c_double, _c_double, _c_int, _c_int,
                                _c_int, _c_void_p, _c_void_p, _c_void_p]),
    "agcn_optim_adam": (_c_int, [_c_void_p, _c_void_p, _c_int, _c_double, _c_void_p, _c_double, _c_double, _c_double, _c_double, _c_int,
                                 _c_int, _c_int, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "agcn_optim_asgd": (_c_int, [_c_void_p, _c_void_p, _c_int, _c_double, _c_void_p, _c_double, _c_double, _c_double, _c_double, _c_int]
                        + [_c_void_p] * 7),
}

_lock = threading.Lock()
_lib = None
launch_count = 0          # C-ABI calls issued through this binding; kernel launches: lib().agcn_launch_count()


def lib():
    """The loaded library; raises loudly when it is absent (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.isfile(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} not found: the CUDA extension is not built. Run `python -m fusion_gcn_b200.build` "
                    "(needs nvcc with sm_100a support). fusion_gcn_b200 has no CPU or PyTorch fallback.")
            handle = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(handle, name)       # AttributeError here = header/library mismatch
                fn.restype = res
                fn.argtypes = args
            _lib = handle
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().agcn_last_error_string().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed with status {rc}: {msg}")
