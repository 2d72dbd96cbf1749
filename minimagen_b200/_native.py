"""ctypes binding of the C ABI declared in include/minimagen_b200.h (built by minimagen_b200/build_ext.py).

This is the ONLY compute backend of the package: if the shared library is missing, or a tensor is not on a CUDA
device, the ops raise -- there is no CPU / PyTorch fallback on the product path.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_longlong, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libminimagen_b200.so")

_P, _I, _L, _F = c_void_p, c_int, c_longlong, c_float

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/minimagen_b200.h one to one
SIGNATURES = {
    "mi_abi_version": [],
    "mi_last_error": [],
    "mi_device_ok": [],
    "mi_set_launch_mode": [_I],
    "mi_pack_conv_weight_f16": [_P, _I, _I, _I, _I, _F, _P, _P],
    "mi_pack_conv_weight_dgrad_f16": [_P, _I, _I, _I, _I, _P, _P],
    "mi_conv2d_igemm_supported": [_I, _I, _I, _I],
    "mi_conv2d_igemm_f16": [_P, _I, _I, _I, _I, _I, _I, _P, _I, _I, _I, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _L, _L, _L, _L,
                            _I, _I, _P, _P, _L, _P],
    "mi_conv3x3_res1x1_supported": [_I, _I, _I, _I, _I],
    "mi_conv3x3_res1x1_f16": [_P, _I, _I, _I, _I, _I, _P, _I, _I, _P, _I, _I, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P],
    "mi_conv2d_igemm_workspace_bytes": [],
    "mi_conv3x3_gn_supported": [_I, _I, _I, _I, _I, _I],
    "mi_conv3x3_gn_silu_f16": [_P, _I, _P, _I, _F, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _F, _P, _I, _P, _P, _P, _P, _P, _P,
                               _P],
    "mi_conv2d_direct_f32": [_P, _I, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _P, _P, _P, _I, _I, _L, _L, _L, _L, _P],
    "mi_gn_stats": [_P, _I, _P, _I, _F, _I, _I, _I, _I, _P, _P],
    "mi_gn_apply_silu": [_P, _I, _P, _I, _F, _I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _P, _I, _F, _P, _I, _P],
    "mi_cast_act": [_P, _I, _P, _I, _F, _I, _I, _I, _I, _I, _P, _I, _P],
    "mi_ln_rows": [_P, _L, _I, _P, _P, _F, _I, _P, _P, _P, _P],
    "mi_linear_f32": [_P, _I, _I, _P, _P, _I, _I, _I, _P, _P, _P, _F, _P],
    "mi_sinusoidal_posemb": [_P, _I, _I, _P, _P],
    "mi_text_tokens": [_P, _I, _I, _I, _P, _P, _P, _I, _P, _I, _I, _P, _P],
    "mi_place_rows": [_P, _I, _I, _I, _P, _I, _I, _P],
    "mi_select_rows": [_P, _P, _P, _P, _I, _I, _P, _P],
    "mi_nchw_to_nhwc": [_P, _I, _P, _I, _I, _I, _I, _P, _P],
    "mi_stem_unroll_f16": [_P, _I, _P, _I, _I, _I, _I, _P, _P],
    "mi_resize_separable": [_P, _L, _I, _I, _P, _I, _I, _P, _P, _I, _P, _P, _I, _I, _F, _F, _P],
    "mi_silu_f32": [_P, _L, _P, _P],
    "mi_attention_workspace_bytes": [_I, _I, _I, _I],
    "mi_attention_fwd": [_P, _L, _I, _P, _P, _L, _I, _I, _P, _P, _I, _I, _I, _I, _P, _L, _I, _P, _L, _P],
    "mi_step_x0": [_P, _P, _P, _F, _P, _P, _P, _I, _I, _P, _P],
    "mi_step_quantile": [_P, _I, _I, _I, _I, _F, _F, _P, _P],
    "mi_step_posterior": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P],
    "mi_step_epilogue_workspace_floats": [_I, _I],
    "mi_step_epilogue": [_P, _P, _P, _F, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _F, _P, _P, _P, _P],
    "mi_step_advance_t": [_P, _I, _P],
    "mi_step_finalize": [_P, _L, _I, _P, _P],
    "mi_q_sample": [_P, _P, _P, _P, _P, _I, _I, _F, _F, _P, _P],
    "mi_inpaint_blend": [_P, _P, _P, _I, _I, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "mi_inpaint_advance": [_P, _P, _I, _I, _P],
    # training side (backward)
    "mi_gemm_f32": [_P, _P, _P, _I, _I, _I, _L, _L, _L, _L, _L, _L, _I, _I, _L, _L, _L, _L, _L, _L, _F, _I, _P],
    "mi_colsum_f32": [_P, _L, _I, _P, _I, _P],
    "mi_conv2d_dgrad_f32": [_P, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _P, _I, _I, _P],
    "mi_conv2d_wgrad_f32": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "mi_conv2d_wgrad_f16_supported": [_I, _I, _I, _I, _I, _I, _I],
    "mi_conv2d_wgrad_f16_workspace_bytes": [_I, _I, _I, _I, _I, _I, _I, _I],
    "mi_conv2d_wgrad_f16": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _L, _P],
    "mi_gn_silu_bwd": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _I, _F, _P, _P, _P, _P, _I, _P, _P],
    "mi_ln_rows_bwd": [_P, _P, _L, _I, _P, _F, _I, _P, _P, _P, _P],
    "mi_softmax_rows": [_P, _L, _I, _P],
    "mi_softmax_rows_bwd": [_P, _P, _L, _I, _P],
    "mi_upsample2x_bwd": [_P, _I, _I, _I, _I, _P, _P],
}
_RESTYPES = {"mi_last_error": c_char_p, "mi_conv2d_igemm_workspace_bytes": c_longlong,
             "mi_attention_workspace_bytes": c_longlong, "mi_conv2d_wgrad_f16_workspace_bytes": c_longlong, "mi_step_epilogue_workspace_floats": c_longlong}

_lib = None
launch_count = 0   # number of kernel launches issued through this binding (bench.py reports it)


def load():
    """Load the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"minimagen_b200: native library not found at {LIB_PATH}. Build it with "
            f"`python -m minimagen_b200.build_ext` (or __graft_entry__.build()). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, c_int)
    if lib.mi_abi_version() != 2:
        raise RuntimeError("minimagen_b200: ABI version mismatch between _native.py and the shared library")
    _lib = lib
    return lib


def last_error():
    return load().mi_last_error().decode()


_FN = {}       # resolved entry points (ctypes attribute lookup + argtypes binding once per name)


def call(name, *args):
    """Invoke an entry point; raise RuntimeError (the reference's convention is a Python exception) on failure."""
    global launch_count
    fn = _FN.get(name)
    if fn is None:
        fn = _FN[name] = getattr(load(), name)
    rc = fn(*args)
    if rc != 0:
        raise RuntimeError(f"minimagen_b200.{name} failed: {last_error()}")
    launch_count += 1
    return rc


# Fast paths of torch.cuda.current_device() / current_stream(): the training step makes ~2000 native calls with ~5 pointers each,
# and the Python-object versions (torch.device, torch.cuda.Stream) were a third of its host time.
_cur_dev = getattr(torch._C, "_cuda_getDevice", None) or torch.cuda.current_device
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  Refuses non-CUDA tensors: no CPU path exists."""
    if t is None:
        return None
    d = t.get_device()                     # -1 for CPU tensors
    if d < 0:
        raise RuntimeError("minimagen_b200: tensor is not on a CUDA device; the kernels have no CPU fallback")
    if d != _cur_dev():
        # kernels are enqueued on the CURRENT device's current stream (and size grids / build tensor maps for it)
        raise RuntimeError(
            f"minimagen_b200: tensor lives on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
            f"enter `torch.cuda.device(tensor.device)` (Unet.forward / Imagen.sample do this for their inputs)")
    return t.data_ptr()


def stream():
    """Raw handle of the current stream of the current device (the capture stream while a CUDA graph is being captured)."""
    if _raw_stream is not None:
        return _raw_stream(_cur_dev())
    return torch.cuda.current_stream().cuda_stream


def device_of(*tensors):
    """`torch.cuda.device` context of the first CUDA tensor among `tensors` (a no-op context if there is none):
    the public entry points wrap their work in it so that a model on cuda:1 runs there whatever the current device is."""
    for t in tensors:
        if t is not None and getattr(t, "is_cuda", False):
            return torch.cuda.device(t.device)
    import contextlib
    return contextlib.nullcontext()
