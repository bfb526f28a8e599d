"""ctypes binding of libvittrack_b200.so — the C ABI declared in include/vt_tracker.h.

The library is hand-written CUDA for sm_100a and has no CPU fallback: loading works anywhere
(so symbol checks can run on a CPU box) but every device entry point fails with VT_ERR_CUDA
when no GPU is present.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VT_B200_LIB") or os.path.join(_HERE, "libvittrack_b200.so")  # (override: A/B runs of two builds)

VT_OK, VT_ERR_INVALID, VT_ERR_CUDA, VT_ERR_WEIGHTS, VT_ERR_CROP_OUTSIDE, VT_ERR_NOT_INIT, VT_ERR_GLYPH = 0, -1, -2, -3, -4, -5, -6
VT_FMT_NV12, VT_FMT_RGB24, VT_FMT_GRAY8, VT_FMT_YUY2, VT_FMT_RGBA, VT_FMT_BGRA, VT_FMT_I420 = 0, 1, 2, 3, 5, 6, 8
VT_GEMM_FP32_SIMT, VT_GEMM_TCGEN05_BF16X3, VT_GEMM_TCGEN05_BF16, VT_GEMM_TCGEN05_FP16 = 0, 1, 2, 3
VT_RUN_HOST_SYNC, VT_RUN_HOST_PIPELINED, VT_RUN_DEVICE_SYNC, VT_RUN_DEVICE_PIPELINED = range(4)
VT_DECODE_CEIL4, VT_DECODE_4FLOOR = 0, 1
VT_WINDOW_HANN, VT_WINDOW_ONE_MINUS_HANN = 0, 1
VT_OV_RECT, VT_OV_CROSSHAIR, VT_OV_TEXT, VT_OV_BACKGROUND, VT_OV_CURSOR, VT_OV_SELECTION = range(6)


class vt_bbox(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("width", C.c_int32), ("height", C.c_int32)]

    def tuple(self):
        return (self.x, self.y, self.width, self.height)


class vt_result(C.Structure):
    _fields_ = [("success", C.c_int32), ("score", C.c_float), ("bbox", vt_bbox), ("status", C.c_int32), ("reserved", C.c_int32)]


class vt_config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("weights_path", C.c_char_p), ("device", C.c_int32), ("format", C.c_int32),
        ("width", C.c_int32), ("height", C.c_int32), ("max_targets", C.c_int32), ("score_threshold", C.c_float),
        ("gemm_mode", C.c_int32), ("use_cuda_graph", C.c_int32), ("box_overlay", C.c_int32), ("overlay_gate", C.c_float),
        ("debug_capture", C.c_int32), ("upload_window", C.c_int32),
        # SURVEY.md App. A.7 variant switches (VT_ABI_VERSION 2)
        ("pad_plus1", C.c_int32), ("decode_window", C.c_int32), ("window", C.c_int32), ("norm_custom", C.c_int32),
        ("norm_scale", C.c_float * 3), ("norm_bias", C.c_float * 3), ("reserved", C.c_int32 * 4),
    ]


class vt_overlay_cmd(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("x", C.c_int32), ("y", C.c_int32), ("w", C.c_int32), ("h", C.c_int32), ("a", C.c_int32),
        ("r", C.c_uint8), ("g", C.c_uint8), ("b", C.c_uint8), ("strict_glyphs", C.c_uint8), ("text", C.c_char * 48),
    ]


class vt_surface(C.Structure):
    """A pitched device frame: planes[0] = Y / RGB / gray, planes[1] = NV12 interleaved UV; pitch[i] = row pitch in bytes."""
    _fields_ = [("planes", C.c_void_p * 2), ("pitch", C.c_size_t * 2)]


class vt_stream_geometry(C.Structure):
    """The format and size of one target slot's frames in a stream group of mixed cameras (vt_tracker_set_stream_geometry)."""
    _fields_ = [("format", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("reserved", C.c_int32)]


class vt_timing(C.Structure):
    _fields_ = [
        ("fps", C.c_double), ("avg_conv_ms", C.c_double), ("avg_track_ms", C.c_double),
        ("h2d_ms", C.c_float), ("preprocess_ms", C.c_float), ("vit_ms", C.c_float), ("decode_ms", C.c_float),
        ("overlay_ms", C.c_float), ("d2h_ms", C.c_float), ("total_ms", C.c_float),
        ("avg_h2d_ms", C.c_float), ("avg_preprocess_ms", C.c_float), ("avg_vit_ms", C.c_float), ("avg_decode_ms", C.c_float),
        ("avg_overlay_ms", C.c_float), ("avg_d2h_ms", C.c_float), ("avg_total_ms", C.c_float),
        ("frames", C.c_uint64), ("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
    ]


class vt_selection(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("cursor_x", "cursor_y", "start_x", "start_y", "phase", "step", "fast_step")]


_u8p = C.POINTER(C.c_uint8)
_f32p = C.POINTER(C.c_float)
_vp = C.c_void_p

# name -> (restype, argtypes): every symbol include/vt_tracker.h declares
SYMBOLS = {
    "vt_abi_version": (C.c_int32, []),
    "vt_last_error": (C.c_char_p, []),
    "vt_config_default": (None, [C.POINTER(vt_config)]),
    "vt_alloc_pinned": (C.c_int32, [C.c_size_t, C.POINTER(_vp)]),
    "vt_free_pinned": (None, [_vp]),
    "vt_weights_probe": (C.c_int32, [C.c_char_p, C.POINTER(C.c_int32)]),
    "vt_tracker_create": (C.c_int32, [C.POINTER(vt_config), C.POINTER(_vp)]),
    "vt_tracker_destroy": (None, [_vp]),
    "vt_tracker_init": (C.c_int32, [_vp, C.c_int32, _vp, C.c_size_t, vt_bbox]),
    "vt_tracker_update": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(vt_result)]),
    "vt_tracker_submit": (C.c_int32, [_vp, _vp, C.c_size_t]),
    "vt_tracker_submit_device": (C.c_int32, [_vp, _vp, C.c_size_t]),
    "vt_tracker_wait": (C.c_int32, [_vp, C.POINTER(vt_result)]),
    "vt_tracker_update_device": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(vt_result)]),
    "vt_tracker_init_surface": (C.c_int32, [_vp, C.c_int32, C.POINTER(vt_surface), vt_bbox]),
    "vt_tracker_update_surface": (C.c_int32, [_vp, C.POINTER(vt_surface), C.POINTER(vt_result)]),
    "vt_tracker_submit_surface": (C.c_int32, [_vp, C.POINTER(vt_surface)]),
    "vt_tracker_update_streams_surface": (C.c_int32, [_vp, C.POINTER(vt_surface), C.c_int32, C.POINTER(vt_result)]),
    "vt_tracker_run_streams_ring": (C.c_int32, [_vp, C.POINTER(C.c_void_p), C.c_int32, C.c_size_t, C.c_size_t, C.c_int32, C.c_int32, C.c_int32,
                                    C.POINTER(C.c_void_p), C.POINTER(vt_result), C.POINTER(C.c_double)]),
    "vt_tracker_update_streams": (C.c_int32, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_int32, C.POINTER(vt_result)]),
    "vt_tracker_set_stream_geometry": (C.c_int32, [_vp, C.c_int32, C.POINTER(vt_stream_geometry)]),
    "vt_tracker_get_stream_geometry": (C.c_int32, [_vp, C.c_int32, C.POINTER(vt_stream_geometry)]),
    "vt_tracker_run_ring": (C.c_int32, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp, C.POINTER(vt_result),
                                        C.POINTER(C.c_double)]),
    "vt_context_run_ring": (C.c_int32, [_vp, _vp, C.c_size_t, C.c_size_t, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_char_p), _vp,
                                        C.POINTER(C.c_double)]),
    "vt_tracker_get_rect": (C.c_int32, [_vp, C.c_int32, C.POINTER(vt_bbox)]),
    "vt_tracker_set_rect": (C.c_int32, [_vp, C.c_int32, vt_bbox]),
    "vt_tracker_drop": (C.c_int32, [_vp, C.c_int32]),
    "vt_tracker_debug_read": (C.c_int32, [_vp, C.c_int32, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p]),
    "vt_tracker_model_dim": (C.c_int32, [_vp, C.c_int32]),
    "vt_tracker_debug_tokens": (C.c_int32, [_vp, C.c_int32, C.c_int32, _f32p]),
    "vt_tracker_debug_trace": (C.c_int32, [_vp, C.POINTER(C.c_uint64), C.c_int32, C.POINTER(C.c_int32)]),
    "vt_tracker_stream": (_vp, [_vp]),
    "vt_tracker_sync": (C.c_int32, [_vp]),
    "vt_debug_gemm": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _f32p, _f32p, _f32p, C.c_int32, C.c_int32, _f32p,
                                  C.POINTER(C.c_int32)]),
    "vt_convert_nv12_rgb": (C.c_int32, [_vp, _vp, C.c_size_t, _vp]),
    "vt_convert_nv12_rgb_device": (C.c_int32, [_vp, _vp, C.c_size_t, _vp, C.c_size_t, C.c_int32]),
    "vt_convert_yuy2_rgb": (C.c_int32, [_vp, _vp, C.c_size_t, C.c_int32, C.c_int32, _vp]),
    "vt_convert_yuy2_rgb_device": (C.c_int32, [_vp, _vp, C.c_size_t, _vp, C.c_size_t, C.c_int32, C.c_int32, C.c_int32]),
    "vt_resize_rgb": (C.c_int32, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32]),
    "vt_resize_rgb_device": (C.c_int32, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32]),
    "vt_resize_rgb_device_batch": (C.c_int32, [_vp, _vp, C.c_size_t, C.c_int32, C.c_int32, _vp, C.c_size_t, C.c_int32, C.c_int32, C.c_int32]),
    "vt_overlay": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(vt_overlay_cmd), C.c_int32]),
    "vt_overlay_current": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(vt_overlay_cmd), C.c_int32]),
    "vt_timing_get": (C.c_int32, [_vp, C.POINTER(vt_timing)]),
    "vt_timing_add_interval": (C.c_int32, [_vp, C.c_uint64]),
    "vt_timing_add_times": (C.c_int32, [_vp, C.c_uint64, C.c_uint64]),
    "vt_timing_stats_create": (_vp, []),
    "vt_timing_stats_destroy": (None, [_vp]),
    "vt_timing_stats_add_interval": (None, [_vp, C.c_uint64]),
    "vt_timing_stats_add_times": (None, [_vp, C.c_uint64, C.c_uint64]),
    "vt_timing_stats_fps": (C.c_double, [_vp]),
    "vt_timing_stats_avg_conv_ms": (C.c_double, [_vp]),
    "vt_timing_stats_avg_track_ms": (C.c_double, [_vp]),
    "vt_command_from_key": (C.c_int32, [C.c_uint8, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "vt_context_create": (C.c_int32, [C.POINTER(vt_config), C.POINTER(_vp)]),
    "vt_context_create_scripted": (C.c_int32, [C.c_int32, C.c_int32, C.POINTER(_vp)]),
    "vt_context_process_scripted": (C.c_int32, [_vp, C.POINTER(vt_result), C.c_int32, C.POINTER(C.c_int32), C.POINTER(vt_bbox)]),
    "vt_context_destroy": (None, [_vp]),
    "vt_context_handle_command": (C.c_int32, [_vp, C.c_int32, C.c_int32]),
    "vt_context_process_frame": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(vt_bbox)]),
    "vt_context_state": (C.c_int32, [_vp]),
    "vt_context_state_name": (C.c_char_p, [_vp]),
    "vt_context_current_score": (C.c_float, [_vp]),
    "vt_context_current_bbox": (C.c_int32, [_vp, C.POINTER(vt_bbox)]),
    "vt_context_selection": (None, [_vp, C.POINTER(vt_selection)]),
    "vt_context_lost_frames": (C.c_uint64, [_vp]),
    "vt_context_tracker": (_vp, [_vp]),
    "vt_probe_frame": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(C.c_char_p)]),
    "vt_probe_frame_surface": (C.c_int32, [_vp, C.POINTER(vt_surface), C.POINTER(C.c_char_p)]),
    "vt_probe_group_create": (C.c_int32, [C.POINTER(vt_config), C.c_int32, C.POINTER(vt_stream_geometry), C.POINTER(_vp)]),
    "vt_probe_group_destroy": (None, [_vp]),
    "vt_probe_group_size": (C.c_int32, [_vp]),
    "vt_probe_group_context": (_vp, [_vp, C.c_int32]),
    "vt_probe_group_frame": (C.c_int32, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(C.c_char_p)]),
    "vt_probe_group_frame_surface": (C.c_int32, [_vp, C.POINTER(vt_surface), C.c_int32, C.POINTER(C.c_char_p)]),
    "vt_probe_group_run_ring": (C.c_int32, [_vp, C.POINTER(C.c_void_p), C.c_size_t, C.c_size_t, C.c_int32, C.c_int32, C.c_int32,
                                            C.POINTER(C.c_char_p), C.POINTER(C.c_void_p), C.POINTER(C.c_double)]),
}

_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load the CUDA library.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU or PyTorch fallback for the tracker hot path.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


class VtError(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        msg = lib().vt_last_error().decode(errors="replace")
        super().__init__(f"{where} failed with vt_status {status}: {msg}")


def check(status: int, where: str) -> None:
    if status != VT_OK:
        raise VtError(status, where)
