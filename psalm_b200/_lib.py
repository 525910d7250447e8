"""ctypes binding of libpsalm_b200.so (the C ABI declared in include/psalm_b200.h).

There is NO fallback: if the shared library is missing or a call fails, we raise.  (The reference
silently falls back to a slow PyTorch path on *any* exception — ops/modules/ms_deform_attn.py:117 —
which is exactly what this package must never do.)
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpsalm_b200.so")

F32, F16, BF16, U8 = 0, 1, 2, 3
_DT = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16, torch.uint8: U8}


class PsalmKernelError(RuntimeError):
    pass


_lib = None

_c_vp, _c_i, _c_i64p = ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int64)

# name -> argtypes; every symbol declared in include/psalm_b200.h must be listed here
# (tests/test_abi.py cross-checks this table against the header).
SIGNATURES = {
    "psalm_abi_version": ([], _c_i),
    "psalm_last_error": ([], ctypes.c_char_p),
    "psalm_compiled_arch": ([], _c_i),
    "psalm_msda_forward": ([_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp] + [_c_i] * 11 + [_c_vp], _c_i),
    "psalm_msda_encoder_fused": ([_c_vp, _c_vp, _c_vp, _c_i64p, _c_i64p] + [_c_i] * 8 + [_c_vp], _c_i),
    "psalm_set_attention_impl": ([_c_i], _c_i),
    "psalm_window_attention": ([_c_vp] * 4 + [_c_i] * 8 + [_c_vp], _c_i),
    "psalm_causal_attention": ([_c_vp] * 3 + [_c_i] * 5 + [_c_vp], _c_i),
    "psalm_rotary_inplace": ([_c_vp] * 3 + [_c_i] * 6 + [_c_vp], _c_i),
    "psalm_cross_attention_workspace_bytes": ([_c_i] * 5, ctypes.c_size_t),
    "psalm_cross_attention": ([_c_vp] * 7 + [_c_i] * 7 + [_c_vp], _c_i),
    "psalm_mask_bits_fused": ([_c_vp] * 4 + [_c_i] * 5 + [_c_vp], _c_i),
    "psalm_set_mask_proj_impl": ([_c_i], _c_i),
    "psalm_mask_logits": ([_c_vp] * 3 + [_c_i] * 6 + [_c_vp], _c_i),
    "psalm_bilinear_tokens": ([_c_vp] * 2 + [_c_i] * 9 + [_c_vp], _c_i),
    "psalm_attn_mask_bits": ([_c_vp] * 3 + [_c_i] * 3 + [_c_vp], _c_i),
    "psalm_set_postproc_impl": ([_c_i], _c_i),
    "psalm_set_msda_impl": ([_c_i], _c_i),
    "psalm_set_msda_halo": ([_c_i], _c_i),
    "psalm_set_causal_impl": ([_c_i], _c_i),
    "psalm_postproc_partials": ([_c_i] * 8 + [ctypes.POINTER(_c_i)], _c_i),
    "psalm_postproc_fused": ([_c_vp] * 10 + [_c_i] * 8 + [_c_vp], _c_i),
    "psalm_postproc_crop_supported": ([_c_i] * 10, _c_i),
    "psalm_postproc_crop_partials": ([_c_i] * 2 + [ctypes.POINTER(_c_i)], _c_i),
    "psalm_postproc_fused_crop": ([_c_vp] * 10 + [_c_i] * 12 + [_c_vp], _c_i),
    "psalm_add_layernorm": ([_c_vp] * 7 + [ctypes.c_longlong, _c_i, ctypes.c_float, _c_i, _c_vp], _c_i),
    "psalm_set_cross_impl": ([_c_i], _c_i),
    "psalm_masked_cross_attention_workspace_bytes": ([_c_i] * 3, ctypes.c_size_t),
    "psalm_masked_cross_attention": ([_c_vp] * 3 + [ctypes.c_longlong] + [_c_vp] * 4 + [ctypes.c_size_t] + [_c_i] * 6 + [_c_vp], _c_i),
    "psalm_kv_cache_write": ([_c_vp] * 5 + [_c_i] * 7 + [_c_vp], _c_i),
    "psalm_paged_decode_attention": ([_c_vp, ctypes.c_longlong] + [_c_vp] * 5 + [_c_i] * 6 + [_c_vp], _c_i),
    "psalm_patchify": ([_c_vp] * 4 + [_c_i] * 7 + [_c_vp], _c_i),
    "psalm_region_pool": ([_c_vp] * 4 + [_c_i] * 7 + [_c_vp], _c_i),
    "psalm_patch_merge_layernorm": ([_c_vp] * 4 + [_c_i] * 4 + [ctypes.c_float, _c_i, _c_vp], _c_i),
    "psalm_linear_fused_supported": ([ctypes.c_longlong, _c_i, _c_i, _c_i, ctypes.c_longlong, _c_i], _c_i),
    "psalm_linear_fused": ([_c_vp, ctypes.c_longlong, _c_vp, _c_vp, _c_vp, ctypes.c_longlong, _c_i, _c_i, _c_i,
                            ctypes.c_longlong, _c_i, _c_vp], _c_i),
    "psalm_groupnorm_tokens": ([_c_vp] * 6 + [_c_i] * 4 + [ctypes.c_float, _c_i, _c_i, _c_vp], _c_i),
    "psalm_mask_rle_workspace_bytes": ([_c_i] * 3, ctypes.c_size_t),
    "psalm_mask_rle_sizes": ([_c_vp, _c_vp, ctypes.c_size_t, _c_vp] + [_c_i] * 4 + [_c_vp], _c_i),
    "psalm_mask_rle_runs": ([_c_vp, ctypes.c_size_t, _c_vp, _c_vp, _c_vp] + [_c_i] * 3 + [_c_vp], _c_i),
    "psalm_mask_rle_write": ([_c_vp] * 4 + [_c_i, _c_vp], _c_i),
}


def lib():
    """Load (once) and return the ctypes handle.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PsalmKernelError(
            "psalm_b200: %s not found — run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `python psalm_b200/build.py`). There is no CPU / PyTorch fallback." % LIB_PATH)
    h = ctypes.CDLL(LIB_PATH)
    for name, (argtypes, restype) in SIGNATURES.items():
        fn = getattr(h, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = h
    return h


def dtype_code(t):
    try:
        return _DT[t]
    except KeyError:
        raise PsalmKernelError("psalm_b200: unsupported dtype %s" % t)


def check(rc, what):
    if rc != 0:
        msg = lib().psalm_last_error()
        raise PsalmKernelError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise PsalmKernelError("psalm_b200 kernels need CUDA tensors; got a %s tensor. "
                                   "There is no CPU implementation." % t.device)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def i64_array(vals):
    arr = (ctypes.c_int64 * len(vals))(*[int(v) for v in vals])
    return arr
