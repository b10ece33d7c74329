"""ctypes binding of libedvr_b200.so (the C ABI in include/edvr_b200.h).

The library is the product; there is NO fallback.  If it is missing or a call returns a
non-zero status, a RuntimeError is raised with the library's own error text.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EDVR_B200_LIB", os.path.join(_HERE, "libedvr_b200.so"))   # override: A/B-test a build
if os.environ.get("EDVR_B200_LIB"):      # development builds (e.g. the -DDP_PROF timing build of tools/dp_prof.py)
    LIB_PATH = os.environ["EDVR_B200_LIB"]

ACT_NONE, ACT_RELU, ACT_LRELU, ACT_SIGMOID = 0, 1, 2, 4
OUT_SAME, OUT_PIXSHUF2, OUT_STRIDE2 = 0, 1, 2

c_int, c_void_p, c_float, c_size_t, c_ll = (ctypes.c_int, ctypes.c_void_p, ctypes.c_float,
                                            ctypes.c_size_t, ctypes.c_longlong)


class Src(ctypes.Structure):
    _fields_ = [("ptr", c_void_p), ("C", c_int), ("pix_stride", c_int), ("ch_off", c_int),
                ("div", c_int), ("mul", c_int), ("keep", c_int), ("add", c_int)]


class Epilogue(ctypes.Structure):
    _fields_ = [("bias", c_void_p), ("act", c_int),
                ("res16", c_void_p), ("res32", c_void_p), ("res_pix_stride", c_int), ("res_ch_off", c_int),
                ("out16", c_void_p), ("out16_pix_stride", c_int), ("out16_ch_off", c_int),
                ("out32", c_void_p), ("out32_pix_stride", c_int), ("out32_ch_off", c_int),
                ("out_nchw", c_void_p), ("nchw_C", c_int), ("out_mode", c_int),
                ("f32_blocked", c_int), ("bf16", c_int)]


_SIGS = {
    "eb_version": (c_int, []),
    "eb_last_error": (ctypes.c_char_p, []),
    "eb_selftest_umma": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "eb_packed_weight_bytes": (c_size_t, [c_int] * 4),
    "eb_pack_weight": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "eb_conv2d": (c_int, [ctypes.POINTER(Src), c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int,
                          ctypes.POINTER(Epilogue), c_void_p]),
    "eb_conv2d_stats": (c_int, [ctypes.POINTER(Src), c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                ctypes.POINTER(Epilogue), c_void_p, c_void_p]),
    "eb_conv2d_pair_supported": (c_int, [c_int] * 4),
    "eb_pack_weight_pair": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "eb_pack_weight_pair_ex": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "eb_pack_weight_pair_dgrad": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "eb_conv_wgrad_workspace": (c_size_t, [c_int] * 6),
    "eb_conv_wgrad": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int] + [c_int] * 7 + [c_float, c_void_p, c_void_p, c_void_p,
                                                                                           c_size_t, c_void_p]),
    "eb_conv2d_pair": (c_int, [ctypes.POINTER(Src), c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int,
                               ctypes.POINTER(Epilogue), c_void_p]),
    "eb_dcn_site_offset_weight_bytes": (c_size_t, [c_int]),
    "eb_dcn_site_pack_offset_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "eb_dcn_site": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                            c_void_p, c_void_p, c_ll, c_ll, c_int,
                            c_void_p, c_int, c_int, c_void_p, c_void_p,
                            c_void_p, c_int, c_int, ctypes.POINTER(Epilogue), c_void_p, c_void_p]),
    "eb_dcn_pair_prof_read": (c_int, [c_void_p]),
    "eb_dcn_pair_supported": (c_int, [c_int] * 4),
    "eb_dcn_pair_offset_weight_bytes": (c_size_t, [c_int]),
    "eb_dcn_pair_pack_offset_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "eb_dcn_site_pair": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                 c_void_p, c_int, c_int, c_void_p, c_void_p,
                                 c_void_p, c_int, ctypes.POINTER(Epilogue), c_void_p, c_void_p]),
    "eb_mdcn_forward_workspace": (c_size_t, [c_int] * 7),
    "eb_mdcn_forward": (c_int, [c_void_p] * 6 + [c_int] * 12 + [c_void_p, c_size_t, c_void_p]),
    "eb_mdcn_forward_f16_workspace": (c_size_t, [c_int] * 8),
    "eb_mdcn_forward_f16": (c_int, [c_void_p] * 6 + [c_int] * 12 + [c_void_p, c_size_t, c_void_p]),
    "eb_mdcn_backward_workspace": (c_size_t, [c_int] * 10),
    "eb_mdcn_backward": (c_int, [c_void_p] * 10 + [c_int] * 12 + [c_void_p, c_size_t, c_void_p]),
    "eb_selftest_mma_rate": (c_int, [c_int] * 10 + [c_void_p, c_void_p, c_void_p]),
    "eb_dcn1_forward": (c_int, [c_void_p] * 4 + [c_int] * 15 + [c_void_p, c_size_t, c_void_p]),
    "eb_dcn1_backward_workspace": (c_size_t, [c_int] * 13),
    "eb_dcn1_backward_input": (c_int, [c_void_p] * 6 + [c_int] * 15 + [c_void_p, c_size_t, c_void_p]),
    "eb_dcn1_backward_parameters": (c_int, [c_void_p] * 4 + [c_float] + [c_int] * 15 + [c_void_p, c_size_t, c_void_p]),
    "eb_mdcn_forward_f64": (c_int, [c_void_p] * 6 + [c_int] * 12 + [c_void_p]),
    "eb_mdcn_backward_f64_workspace": (c_size_t, [c_int] * 10),
    "eb_mdcn_backward_f64": (c_int, [c_void_p] * 10 + [c_int] * 12 + [c_void_p, c_size_t, c_void_p]),
    "eb_dcn1_forward_f64": (c_int, [c_void_p] * 4 + [c_int] * 15 + [c_void_p]),
    "eb_dcn1_backward_input_f64_workspace": (c_size_t, [c_int] * 13),
    "eb_dcn1_backward_parameters_f64_workspace": (c_size_t, [c_int] * 13),
    "eb_dcn1_backward_input_f64": (c_int, [c_void_p] * 6 + [c_int] * 15 + [c_void_p, c_size_t, c_void_p]),
    "eb_dcn1_backward_parameters_f64": (c_int, [c_void_p] * 4 + [ctypes.c_double] + [c_int] * 15 +
                                        [c_void_p, c_size_t, c_void_p]),
    "eb_nchw_f32_to_nhwc_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "eb_nhwc_f16_to_nchw_f32": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "eb_conv_first": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "eb_conv_last": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_ll, c_int, c_void_p, c_int, c_int,
                             c_int, c_int, c_void_p]),
    "eb_add_base": (c_int, [c_void_p, ctypes.c_longlong, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "eb_upsample2x": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                              c_void_p, c_int, c_int, c_void_p]),
    "eb_frames_u8_to_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "eb_tensor2img_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_void_p]),
    "eb_pool_max_avg": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "eb_tsa_temporal": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "eb_tsa_modulate": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                c_int, c_void_p]),
    "eb_f32_blocked_elems": (c_size_t, [c_int] * 4),
    "eb_add": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
}

EXPORTS = tuple(_SIGS)
_lib = None


def lib():
    """Load (once) and return the CDLL; raises if the shared library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(the CUDA extension is the product; there is no fallback path)")
        h = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(h, name)
            fn.restype, fn.argtypes = res, args
        _lib = h
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().eb_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libedvr_b200 {what} failed with status {rc}: {msg}")


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return ctypes.c_void_p(None if t is None else t.data_ptr())
