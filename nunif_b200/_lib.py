"""ctypes binding of libnunif_b200.so (the C ABI in include/nunif_b200.h).

PyTorch is only used for device memory and streams: tensors are passed to the
library as raw device pointers.  There is NO fallback: if the shared library is
missing, or no sm_100 device is present, calls raise RuntimeError.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnunif_b200.so")
_lib = None
_lock = threading.Lock()

c_void_p, c_int, c_float, c_size_t, c_char_p = (ctypes.c_void_p, ctypes.c_int, ctypes.c_float,
                                                 ctypes.c_size_t, ctypes.c_char_p)
c_double = ctypes.c_double


class TileConfig(ctypes.Structure):
    """nb200_tile_config == SeamBlending.create_config (seam_blending.py:109-143)."""
    _fields_ = [(n, ctypes.c_int32) for n in (
        "y_h", "y_w", "h_blocks", "w_blocks", "pad_l", "pad_r", "pad_t", "pad_b",
        "y_buffer_h", "y_buffer_w", "input_tile_step", "output_tile_step")]

    def as_dict(self):
        return {
            "y_h": self.y_h, "y_w": self.y_w, "h_blocks": self.h_blocks, "w_blocks": self.w_blocks,
            "pad": (self.pad_l, self.pad_r, self.pad_t, self.pad_b),
            "y_buffer_h": self.y_buffer_h, "y_buffer_w": self.y_buffer_w,
            "input_tile_step": self.input_tile_step, "output_tile_step": self.output_tile_step,
        }


# name -> (restype, argtypes).  Must list every symbol declared in include/nunif_b200.h
# (tests/test_abi.py parses the header and checks this table and the .so against it).
SIGNATURES = {
    "nb200_last_error": (c_char_p, []),
    "nb200_abi_version": (c_int, []),
    "nb200_check_device": (c_int, [c_int]),
    "nb200_launch_count": (ctypes.c_uint64, []),
    "nb200_tile_config_create": (c_int, [c_int] * 6 + [ctypes.POINTER(TileConfig)]),
    "nb200_tile_unfold": (c_int, [c_void_p, c_int, c_int, c_int, ctypes.POINTER(TileConfig), c_int, c_int, c_int,
                                  c_void_p, c_int, c_void_p]),
    "nb200_tile_gather_blend": (c_int, [c_void_p, c_int, ctypes.POINTER(TileConfig), c_int, c_int, c_int, c_int,
                                        c_void_p, c_void_p]),
    "nb200_model_create": (c_int, [c_int, c_int, ctypes.POINTER(c_char_p), ctypes.POINTER(c_void_p),
                                   ctypes.POINTER(ctypes.c_int64), c_int, ctypes.POINTER(c_void_p)]),
    "nb200_model_destroy": (None, [c_void_p]),
    "nb200_model_info": (c_int, [c_void_p, ctypes.POINTER(c_int), ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "nb200_model_weight_blob": (c_int, [c_void_p, ctypes.POINTER(c_void_p), ctypes.POINTER(c_size_t)]),
    "nb200_model_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_tiled_render": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_tiled_render_host": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_depth_anything_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_zoedepth_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_zoe_rel_pos_table": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "nb200_depth_aa": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_mlbw_delta": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "nb200_mlbw_num_layers": (c_int, [c_void_p]),
    "nb200_row_flow_delta": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_backward_warp_delta": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_double, c_void_p, c_void_p]),
    "nb200_alpha_border_padding_workspace": (c_size_t, [c_int, c_int]),
    "nb200_alpha_border_padding": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "nb200_tta_transform": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_tta_merge": (c_int, [ctypes.POINTER(c_void_p), c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_hwc_to_chw_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_chw_f32_to_hwc": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_da_preprocess_size": (c_int, [c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "nb200_da_preprocess": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_zoe_preprocess_size": (c_int, [c_int] * 5 + [ctypes.POINTER(c_int)] * 6),
    "nb200_zoe_preprocess": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_anaglyph": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_resize_bicubic_aa": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_equirectangular_size": (c_int, [c_int, c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "nb200_equirectangular": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_backward_warp": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_double, c_double, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p]),
    "nb200_forward_warp_workspace": (c_size_t, [c_int] * 5),
    "nb200_forward_warp": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_double, c_double, c_int, c_int,
                                   c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nb200_depth_resize_aa": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_dilate_edge_workspace": (c_size_t, [c_int] * 3),
    "nb200_dilate_edge": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "nb200_minmax_map": (c_int, [c_void_p, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "nb200_ema_scaler_create": (c_int, [c_int, c_double, c_int, ctypes.POINTER(c_void_p)]),
    "nb200_ema_scaler_destroy": (None, [c_void_p]),
    "nb200_ema_scaler_reset": (c_int, [c_void_p, c_double, c_int]),
    "nb200_ema_scaler_update": (c_int, [c_void_p, c_void_p, c_int, ctypes.POINTER(c_int), c_void_p]),
    "nb200_ema_scaler_normalize": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "nb200_depth_mapper": (c_int, [c_void_p, ctypes.c_longlong, c_float, c_void_p, c_void_p]),
    "nb200_anaglyph_dubois": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_conv_gemm_f16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int,
                                    c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                    c_void_p]),
    "nb200_tune_set": (c_int, [c_int, c_int]),
    "nb200_debug_timeline": (c_int, [c_void_p]),
    "nb200_debug_tap": (c_int, [c_int, c_void_p, ctypes.c_size_t]),
    "nb200_profile_enable": (c_int, [c_int]),
    "nb200_profile_report": (c_int, [ctypes.c_char_p, c_size_t]),
    "nb200_profile_dump": (c_int, [c_char_p, c_size_t]),
    "nb200_swin_mlp_fused_f16": (c_int, [c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p]),
    "nb200_swin_attn_fused_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                          c_void_p]),
    "nb200_swin_attn_tc_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                       c_void_p]),
    "nb200_window_attention_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "nb200_vit_attention_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "nb200_vit_add_layernorm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_longlong, c_int, c_void_p]),
    "nb200_zoe_expand_rel_bias": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "nb200_zoe_attractor": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "nb200_zoe_clb_final": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                    c_void_p]),
    "nb200_dpt_upsample_bilinear_f16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
}


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m nunif_b200.build` "
                "(nvcc, sm_100a).  nunif_b200 has no CPU / PyTorch fallback.")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status):
    if status != 0:
        raise RuntimeError("nunif_b200: " + lib().nb200_last_error().decode("utf-8", "replace"))


def require_cuda(t, name="tensor"):
    import torch
    if not torch.is_tensor(t) or not t.is_cuda:
        raise RuntimeError(f"nunif_b200: {name} must be a CUDA tensor (the B200 engine has no CPU fallback)")


def stream_ptr(device=None):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)
