"""ctypes binding of include/vqvae_b200.h (the C-ABI boundary).

The library is built in-tree by vqvae_b200/build.py (nvcc, sm_100a).  Loading never
falls back to anything: if the shared object is missing the import of the product
fails loudly.
"""
import ctypes as C
import os

from .build import LIB, build

_lib = None

# enums of include/vqvae_b200.h
NCHW, NHWC = 0, 1
FP32, TF32, BF16 = 0, 1, 2
PRECISIONS = {"fp32": FP32, "tf32": TF32, "bf16": BF16}
# enum vqb_conv_kind
CONV_K1, CONV_K3, CONVT_K3, CONV_K4S2, CONVT_K4S2, CONVT_K4S2_OUT, RES_W2 = range(7)

_vp, _i, _i64, _sz, _f = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float

# name -> (restype, argtypes); mirrors the header one to one (tests check this)
SIGNATURES = {
    "vqb_abi_version": (_i, []),
    "vqb_diag_build": (_i, []),
    "vqb_error_string": (C.c_char_p, [_i]),
    "vqb_device_info": (_i, [C.POINTER(_i)] * 3),
    "vqb_pack_conv_weight_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "vqb_conv2d_f32": (_i, [_vp] * 5 + [_i] * 14 + [_vp]),
    "vqb_vq_workspace_bytes": (_sz, [_i64, _i, _i]),
    "vqb_vq_forward_f32": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "vqb_vq_forward_deferred_f32": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "vqb_memcpy_async": (_i, [_vp, _vp, _sz, _i, _vp]),
    "vqb_vq_reduce_sse_f32": (_i, [_vp, _i64, _i, _i, _vp, _vp]),
    "vqb_vq_finish_f32": (_i, [_vp, _vp, _i64, _i, _i, _f, _vp, _vp, _vp]),
    "vqb_vq_backward_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _f, _vp, _vp, _vp]),
    "vqb_onehot_f32": (_i, [_vp, _i64, _i, _vp, _vp]),
    "vqb_gather_rows_f32": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp]),
    "vqb_nchw_to_nhwc_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "vqb_nhwc_to_nchw_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "vqb_relu_f32": (_i, [_vp, _i64, _vp]),
    "vqb_launch_count": (C.c_ulonglong, []),
    "vqb_set_vq_kernel": (_i, [_i]),
    "vqb_debug_read_trace": (_i, [_vp, _i]),
    "vqb_debug_read_trace_vq": (_i, [_vp, _i]),
    "vqb_debug_read_cta_times": (_i, [_vp, _i]),
    "vqb_residual_layer_f32": (_i, [_vp] * 5 + [_i] * 7 + [_vp]),
    "vqb_residual_stack_f32": (_i, [_vp] * 6 + [_i] * 7 + [_vp]),
    "vqb_latent_encoder_f32": (_i, [_vp] * 8 + [_i] * 7 + [_vp]),
    "vqb_latent_decoder_f32": (_i, [_vp] * 8 + [_i] * 8 + [_vp]),
    "vqb_conv_bf16_packed_bytes": (_sz, [_i, _i, _i]),
    "vqb_pack_conv_weight_bf16": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "vqb_conv2d_bf16": (_i, [_vp, _vp, _vp, _vp] + [_i] * 8 + [_vp]),
    "vqb_conv_in_bf16": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "vqb_vq_forward_bf16zq_f32": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "vqb_residual_layer_bf16": (_i, [_vp] * 4 + [_i] * 6 + [_vp]),
    "vqb_debug_vq_scores_f32": (_i, [_vp, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
}


def lib():
    """The loaded C-ABI library (built on first use if the .so is absent/stale)."""
    global _lib
    if _lib is None:
        path = LIB if os.path.exists(LIB) and os.environ.get("VQB_NO_REBUILD") else build()
        handle = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)   # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        if handle.vqb_abi_version() != 2:
            raise RuntimeError("libvqvae_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(code, what):
    if code != 0:
        msg = lib().vqb_error_string(int(code)).decode()
        raise RuntimeError(f"{what}: {msg} (code {code})")
