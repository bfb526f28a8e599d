"""Host-side mirror of the reference's interface for the per-frame path, over the C ABI.

Names, argument meaning and error behaviour follow the reference so that parity tests read like
tests of the reference itself:

    nv12_full_to_rgb_parallel(nv12, w, h)            ≙ src/nv12_convert.rs:46
    draw_rect_nv12 / draw_crosshair_nv12 / draw_text_nv12 / draw_background_nv12   ≙ src/nv12_convert.rs:172-343
    draw_cursor / draw_selection                     ≙ src/drawing.rs:5-50
    draw_*_rgb                                       ≙ src/drawing_rgb.rs:30-128
    VitTrack.new / init / update                     ≙ vit_tracker::VitTrack (call sites src/tracker_context.rs:21,88,90,120)
    TrackerContext.new / handle_command / process_frame / state_name   ≙ src/tracker_context.rs:19-166
    UserCommand                                      ≙ src/user_commands.rs
    TimingStats                                      ≙ src/timing_stats.rs

Everything here runs on the GPU through libvittrack_b200.so; nothing falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
from collections import deque
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from ._lib import VtError, check, lib, vt_bbox, vt_config, vt_overlay_cmd, vt_result, vt_selection, vt_stream_geometry, vt_surface, vt_timing


@dataclass(frozen=True)
class BBox:
    """≙ vit_tracker::BBox {x, y, width, height: i32}"""
    x: int
    y: int
    width: int
    height: int

    @staticmethod
    def new(x, y, w, h) -> "BBox":
        return BBox(int(x), int(y), int(w), int(h))

    @staticmethod
    def from_array(a: Sequence[int]) -> "BBox":
        return BBox(int(a[0]), int(a[1]), int(a[2]), int(a[3]))

    def tuple(self) -> Tuple[int, int, int, int]:
        return (self.x, self.y, self.width, self.height)

    def _c(self) -> vt_bbox:
        return vt_bbox(self.x, self.y, self.width, self.height)


@dataclass(frozen=True)
class TrackResult:
    """≙ the Ok(result) of VitTrack::update (src/tracker_context.rs:92-94)"""
    success: bool
    score: float
    bbox: Tuple[int, int, int, int]
    status: int = 0


class UserCommand:
    """≙ enum UserCommand (src/user_commands.rs); Move* carry the `fast` bool."""
    MoveUp, MoveDown, MoveLeft, MoveRight, Confirm, Cancel, Quit = range(7)


# ---- pinned frames ----------------------------------------------------------------------------
class PinnedBuffer:
    """Page-locked host memory (vt_alloc_pinned) exposed as a uint8 numpy array."""

    def __init__(self, nbytes: int):
        p = C.c_void_p()
        check(lib().vt_alloc_pinned(nbytes, C.byref(p)), "vt_alloc_pinned")
        self._p = p
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(nbytes,))

    def close(self):
        if self._p:
            self.array = None
            lib().vt_free_pinned(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _ptr(a: np.ndarray) -> C.c_void_p:
    if not isinstance(a, np.ndarray) or a.dtype != np.uint8 or not a.flags["C_CONTIGUOUS"]:
        raise ValueError("frames are C-contiguous uint8 numpy arrays")
    return C.c_void_p(a.ctypes.data)


FORMATS = {"nv12": L.VT_FMT_NV12, "rgb24": L.VT_FMT_RGB24, "gray8": L.VT_FMT_GRAY8, "yuy2": L.VT_FMT_YUY2, "rgba": L.VT_FMT_RGBA,
           "bgra": L.VT_FMT_BGRA, "i420": L.VT_FMT_I420}


def row_bytes(fmt: str, width: int) -> int:
    """Bytes of one packed row of plane 0 (the Y plane, the RGB / gray image, the packed YUY2 words: 4 * ceil(width / 2), the 32-bit
    RGBA / BGRA pixels: 4 * width; I420: the Y stride of GStreamer's layout, width rounded up to a multiple of 4)."""
    if fmt == "yuy2":
        return 4 * ((width + 1) // 2)
    if fmt == "i420":
        return (width + 3) & ~3
    return width * {"rgb24": 3, "rgba": 4, "bgra": 4}.get(fmt, 1)


Surface = Tuple[Sequence[int], Sequence[int]]  # ((plane 0 address, plane 1 address), (pitch 0, pitch 1)): device addresses, bytes


def _surface(s: Surface) -> vt_surface:
    planes, pitches = s
    c = vt_surface()
    for i in range(2):
        c.planes[i] = int(planes[i]) if i < len(planes) and planes[i] else None
        c.pitch[i] = int(pitches[i]) if i < len(pitches) else 0
    return c


class PitchedFrame:
    """A packed frame laid out as a pitched device surface in torch buffers, like a decoder's output surface: rows `pitch` bytes apart
    and, for NV12, the chroma plane `chroma_row` rows after the start of the Y plane (NVDEC: the surface height), or in an allocation
    of its own (`separate_uv`).  Every byte outside the visible pixels (pitch padding, the gap between the planes) holds `fill`.
    `surface` is the (planes, pitches) tuple the *_surface methods of VitTrack take."""

    def __init__(self, width: int, height: int, fmt: str = "nv12", pitch: Optional[int] = None, chroma_row: Optional[int] = None,
                 separate_uv: bool = False, fill: int = 0, device: int = 0):
        import torch

        self.width, self.height, self.fmt = width, height, fmt
        self.row = row_bytes(fmt, width)
        self.pitch = pitch if pitch is not None else self.row
        if self.pitch < self.row:
            raise ValueError("pitch is smaller than a row")
        self.nv12 = fmt == "nv12"
        self.uv_rows = (height + 1) // 2 if self.nv12 else 0
        dev = torch.device("cuda", device)
        if not self.nv12 or separate_uv:
            self.buf = torch.full((height * self.pitch,), fill, dtype=torch.uint8, device=dev)
            self.uv_buf = torch.full((self.uv_rows * self.pitch,), fill, dtype=torch.uint8, device=dev) if self.nv12 else None
            self.uv_offset = 0
        else:
            crow = chroma_row if chroma_row is not None else height
            if crow < height:
                raise ValueError("the chroma plane overlaps the Y plane")
            self.buf = torch.full(((crow + self.uv_rows) * self.pitch,), fill, dtype=torch.uint8, device=dev)
            self.uv_buf, self.uv_offset = None, crow * self.pitch

    def _planes(self):
        y = self.buf[: self.height * self.pitch].view(self.height, self.pitch)[:, : self.row]
        if not self.nv12:
            return y, None
        base = self.uv_buf if self.uv_buf is not None else self.buf[self.uv_offset:]
        return y, base[: self.uv_rows * self.pitch].view(self.uv_rows, self.pitch)[:, : self.width]

    def write(self, frame) -> None:
        """Copies a packed frame (numpy array or torch tensor, host or device) into the visible pixels."""
        import torch

        f = torch.as_tensor(np.ascontiguousarray(frame) if isinstance(frame, np.ndarray) else frame).reshape(-1)
        y, uv = self._planes()
        n = self.height * self.row
        y.copy_(f[:n].view(self.height, self.row))
        if uv is not None:
            uv.copy_(f[n: n + self.uv_rows * self.width].view(self.uv_rows, self.width))
        torch.cuda.synchronize(self.buf.device)  # the tracker's stream does not order behind torch's

    def read(self) -> np.ndarray:
        """The visible pixels as a packed frame (host)."""
        import torch

        y, uv = self._planes()
        return torch.cat([y.reshape(-1)] + ([uv.reshape(-1)] if uv is not None else [])).cpu().numpy()

    @property
    def surface(self) -> Surface:
        if not self.nv12:
            return (self.buf.data_ptr(), 0), (self.pitch, 0)
        uv = self.uv_buf.data_ptr() if self.uv_buf is not None else self.buf.data_ptr() + self.uv_offset
        return (self.buf.data_ptr(), uv), (self.pitch, self.pitch)


def make_config(weights: str, width: int, height: int, fmt: str = "nv12", max_targets: int = 1, device: int = 0,
                use_cuda_graph: bool = True, box_overlay: bool = False, score_threshold: float = 0.20,
                gemm_mode: int = L.VT_GEMM_TCGEN05_BF16X3, debug_capture: bool = False, upload_window: bool = False,
                pad_plus1: bool = False, decode_window: int = L.VT_DECODE_CEIL4, window: int = L.VT_WINDOW_HANN,
                norm: Optional[Tuple[Sequence[float], Sequence[float]]] = None) -> vt_config:
    """`pad_plus1`, `decode_window`, `window`, `norm=(scale[3], bias[3])` are the SURVEY.md App. A.7 variant switches (defaults: OpenCV 4.13
    TrackerVit with the intended (u8/255 - mean)/std normalisation; `norm` replaces it by blob = u8*scale[c] + bias[c])."""
    cfg = vt_config()
    lib().vt_config_default(C.byref(cfg))
    if weights.lower().endswith(".onnx"):  # ≙ VitTrack::new(model_path) with the network in its public ONNX form
        weights = _import_onnx_cached(weights)
    cfg.weights_path = weights.encode()
    cfg.device = device
    cfg.format = FORMATS[fmt]
    cfg.width, cfg.height, cfg.max_targets = width, height, max_targets
    cfg.score_threshold = score_threshold
    cfg.gemm_mode = gemm_mode
    cfg.use_cuda_graph = int(use_cuda_graph)
    cfg.box_overlay = int(box_overlay)
    cfg.debug_capture = int(debug_capture)
    cfg.upload_window = int(upload_window)
    cfg.pad_plus1, cfg.decode_window, cfg.window = int(pad_plus1), int(decode_window), int(window)
    if norm is not None:
        cfg.norm_custom = 1
        for k in range(3):
            cfg.norm_scale[k], cfg.norm_bias[k] = float(norm[0][k]), float(norm[1][k])
    return cfg


def weights_probe(path: str) -> Tuple[int, int, int, int, int]:
    """(D, depth, heads, hidden, head_channels) of a VTW1 model file; raises VtError(VT_ERR_WEIGHTS) when `VitTrack.new` would reject
    it.  Needs no GPU."""
    shape = (C.c_int32 * 5)()
    check(lib().vt_weights_probe(path.encode(), shape), "vt_weights_probe")
    return tuple(int(v) for v in shape)


def _import_onnx_cached(onnx_path: str) -> str:
    """ONNX model file -> flat VTW1 file next to the system temp dir (keyed by path, size, mtime); see onnx_import.py."""
    import hashlib
    import os
    import tempfile

    from . import onnx_import

    st = os.stat(onnx_path)
    key = hashlib.sha1(f"{os.path.abspath(onnx_path)}|{st.st_size}|{st.st_mtime_ns}".encode()).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), "vt_b200_weights", f"onnx_{key}.vtw")
    if not os.path.exists(out):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        try:
            onnx_import.import_onnx(onnx_path, out + ".tmp")
        except onnx_import.OnnxImportError as e:
            raise VtError(L.VT_ERR_WEIGHTS, f"{onnx_path}: {e}") from None
        os.replace(out + ".tmp", out)
    return out


# ---- VitTrack ------------------------------------------------------------------------------------
class VitTrack:
    """≙ vit_tracker::VitTrack.  One handle tracks up to `max_targets` targets on one video stream."""

    def __init__(self, cfg: vt_config, _handle=None, _owned=True):
        self._cfg = cfg
        self.width, self.height = cfg.width, cfg.height
        self.max_targets = cfg.max_targets
        self.fmt = cfg.format
        self._owned = _owned
        if _handle is not None:
            self._h = _handle
        else:
            h = C.c_void_p()
            check(lib().vt_tracker_create(C.byref(cfg), C.byref(h)), "vt_tracker_create")
            self._h = h
        self._res = (vt_result * self.max_targets)()
        # frames handed to submit() and not yet returned by wait(): the C side keeps the raw pointer until wait() (the overlay writes
        # into it), so the arrays must stay alive — a temporary like submit(fr.copy()) would otherwise be freed under the library
        self._inflight = deque()

    @classmethod
    def new(cls, model_path: str, width: int = 1920, height: int = 1080, **kw) -> "VitTrack":
        """≙ VitTrack::new(model_path) — raises VtError(VT_ERR_WEIGHTS) like the reference's Err."""
        return cls(make_config(model_path, width, height, **kw))

    def close(self):
        if getattr(self, "_h", None) and self._owned:
            lib().vt_tracker_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference API
    def init(self, frame: np.ndarray, bbox: BBox, target: int = 0) -> None:
        check(lib().vt_tracker_init(self._h, target, _ptr(frame), frame.size, bbox._c()), "vt_tracker_init")

    def update(self, frame: np.ndarray) -> TrackResult:
        """Single-target form: returns the result of target 0, raising on the Err branch."""
        r = self.update_all(frame)[0]
        if r.status != L.VT_OK:
            raise VtError(r.status, "VitTrack.update")
        return r

    # -- extensions
    def _results(self) -> List[TrackResult]:
        return [TrackResult(bool(r.success), float(r.score), r.bbox.tuple(), int(r.status)) for r in self._res]

    def update_all(self, frame: np.ndarray) -> List[TrackResult]:
        check(lib().vt_tracker_update(self._h, _ptr(frame), frame.size, self._res), "vt_tracker_update")
        return self._results()

    def set_stream_geometry(self, target: int, width: Optional[int] = None, height: Optional[int] = None, fmt: Optional[str] = None) -> None:
        """Stream groups of mixed cameras (vt_tracker_set_stream_geometry): target slot `target` takes frames of `fmt` ("nv12", "rgb24",
        "gray8", "yuy2", "rgba", "bgra", "i420") at width x height instead of the handle's geometry — init() on that slot and its stream in update_streams /
        update_streams_surface / run_streams_ring.  Only a slot that is not initialised may change; no arguments: back to the handle's
        geometry.  A handle with a slot of its own geometry takes frames through the stream-group calls only."""
        if width is None and height is None and fmt is None:
            check(lib().vt_tracker_set_stream_geometry(self._h, target, None), "vt_tracker_set_stream_geometry")
            return
        if width is None or height is None or fmt is None:
            raise ValueError("set_stream_geometry takes width, height and fmt together (or none of them)")
        g = vt_stream_geometry(FORMATS[fmt], int(width), int(height), 0)
        check(lib().vt_tracker_set_stream_geometry(self._h, target, C.byref(g)), "vt_tracker_set_stream_geometry")

    def get_stream_geometry(self, target: int) -> Tuple[int, int, str]:
        """(width, height, fmt) of target slot `target`'s frames."""
        g = vt_stream_geometry()
        check(lib().vt_tracker_get_stream_geometry(self._h, target, C.byref(g)), "vt_tracker_get_stream_geometry")
        return g.width, g.height, {v: k for k, v in FORMATS.items()}[g.format]

    def update_streams(self, frames: Sequence[np.ndarray]) -> List[TrackResult]:
        """Stream group (vt_tracker_update_streams): frames[i] — a full frame in pinned host memory (PinnedBuffer) — is the current
        frame of the i-th active target's own video stream, of that target's geometry (set_stream_geometry); all targets go through one
        batched forward, each stream's box overlay is drawn into its own frame.  ≙ n TrackerContexts (src/pipeline.rs:55) stepped
        together."""
        n = len(frames)
        ptrs = (C.c_void_p * n)(*[_ptr(f).value for f in frames])
        lens = (C.c_size_t * n)(*[f.size for f in frames])
        check(lib().vt_tracker_update_streams(self._h, ptrs, lens, n, self._res), "vt_tracker_update_streams")
        return self._results()

    def submit_device(self, d_ptr: int, nbytes: int) -> None:
        """Frame already in device memory, tracked in place.  The caller keeps the device buffer alive until the matching wait()."""
        check(lib().vt_tracker_submit_device(self._h, C.c_void_p(d_ptr), nbytes), "vt_tracker_submit_device")
        self._inflight.append(None)

    def submit(self, frame: np.ndarray) -> None:
        """Enqueue one frame (up to two may be in flight).  Lifetime rule of the C ABI: `frame` must stay valid until the matching
        wait() returns — with box_overlay the library WRITES the box pixels into it.  This binding holds a reference to the array
        until then, so temporaries are safe; the caller must still not resize / free the underlying buffer."""
        p = _ptr(frame)
        check(lib().vt_tracker_submit(self._h, p, frame.size), "vt_tracker_submit")
        self._inflight.append(frame)

    def wait(self) -> List[TrackResult]:
        try:
            check(lib().vt_tracker_wait(self._h, self._res), "vt_tracker_wait")
        finally:
            if self._inflight:
                self._inflight.popleft()
        return self._results()

    def update_device(self, d_ptr: int, nbytes: int) -> List[TrackResult]:
        check(lib().vt_tracker_update_device(self._h, C.c_void_p(d_ptr), nbytes, self._res), "vt_tracker_update_device")
        return self._results()

    # -- pitched device surfaces (decoder output: NVDEC, NvBufSurface), tracked in place; PitchedFrame makes one in torch memory
    def init_surface(self, surface: Surface, bbox: BBox, target: int = 0) -> None:
        s = _surface(surface)
        check(lib().vt_tracker_init_surface(self._h, target, C.byref(s), bbox._c()), "vt_tracker_init_surface")

    def update_surface(self, surface: Surface) -> List[TrackResult]:
        s = _surface(surface)
        check(lib().vt_tracker_update_surface(self._h, C.byref(s), self._res), "vt_tracker_update_surface")
        return self._results()

    def submit_surface(self, surface: Surface) -> None:
        """The caller keeps the surface's memory alive until the matching wait()."""
        s = _surface(surface)
        check(lib().vt_tracker_submit_surface(self._h, C.byref(s)), "vt_tracker_submit_surface")
        self._inflight.append(None)

    def update_streams_surface(self, surfaces: Sequence[Surface]) -> List[TrackResult]:
        """Stream group on device surfaces: surfaces[i] is the current frame of the i-th active target's stream (see update_streams)."""
        n = len(surfaces)
        arr = (vt_surface * n)(*[_surface(s) for s in surfaces])
        check(lib().vt_tracker_update_streams_surface(self._h, arr, n, self._res), "vt_tracker_update_streams_surface")
        return self._results()

    def run_ring(self, base_ptr: int, stride: int, frame_len: int, ring: int, first: int, n: int, mode: int, pristine_ptr: int = 0,
                 want_latency: bool = False):
        """n frames of a ring through this handle in one native call (vt_tracker_run_ring; the GIL is released for its duration, so
        one Python thread per stream drives many streams).  Returns (results of the last frame, latencies in us or None)."""
        lat = np.empty(n, np.float64) if want_latency else None
        check(lib().vt_tracker_run_ring(self._h, C.c_void_p(base_ptr), stride, frame_len, ring, first, n, mode,
                                        C.c_void_p(pristine_ptr) if pristine_ptr else None, self._res,
                                        lat.ctypes.data_as(C.POINTER(C.c_double)) if want_latency else None), "vt_tracker_run_ring")
        return self._results(), lat

    def run_streams_ring(self, ring_ptrs: Sequence[int], stride: int, frame_len: int, ring: int, first: int, n: int,
                         pristine_ptrs: Optional[Sequence[int]] = None, want_latency: bool = False):
        """n steps of a stream group in one native call (vt_tracker_run_streams_ring): ring_ptrs[i] = pinned host ring of stream i.  With
        streams of mixed geometries `frame_len` and `stride` cover the largest stream's frame."""
        k = len(ring_ptrs)
        rings = (C.c_void_p * k)(*ring_ptrs)
        clean = (C.c_void_p * k)(*pristine_ptrs) if pristine_ptrs is not None else None
        lat = np.empty(n, np.float64) if want_latency else None
        check(lib().vt_tracker_run_streams_ring(self._h, rings, k, stride, frame_len, ring, first, n, clean, self._res,
                                                lat.ctypes.data_as(C.POINTER(C.c_double)) if want_latency else None), "vt_tracker_run_streams_ring")
        return self._results(), lat

    def get_rect(self, target: int = 0) -> Tuple[int, int, int, int]:
        b = vt_bbox()
        check(lib().vt_tracker_get_rect(self._h, target, C.byref(b)), "vt_tracker_get_rect")
        return b.tuple()

    def set_rect(self, box, target: int = 0) -> None:
        check(lib().vt_tracker_set_rect(self._h, target, vt_bbox(*box)), "vt_tracker_set_rect")

    def drop(self, target: int) -> None:
        check(lib().vt_tracker_drop(self._h, target), "vt_tracker_drop")

    def model_dim(self, which: int) -> int:
        return lib().vt_tracker_model_dim(self._h, which)

    def debug_read(self, target: int = 0):
        D = self.model_dim(0)
        sb, tb = np.empty((3, 256, 256), np.float32), np.empty((3, 128, 128), np.float32)
        cw, sm, om, tok = np.empty(256, np.float32), np.empty(512, np.float32), np.empty(512, np.float32), np.empty((320, D), np.float32)
        f = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
        check(lib().vt_tracker_debug_read(self._h, target, f(sb), f(tb), f(cw), f(sm), f(om), f(tok)), "vt_tracker_debug_read")
        return dict(search_blob=sb, template_blob=tb, conf_win=cw, size_map=sm, off_map=om, tokens=tok)

    def debug_tokens(self, which: int, target: int = 0) -> np.ndarray:
        out = np.empty((320, self.model_dim(0)), np.float32)
        check(lib().vt_tracker_debug_tokens(self._h, target, which, out.ctypes.data_as(C.POINTER(C.c_float))), "vt_tracker_debug_tokens")
        return out

    def debug_trace(self, max_records: int = 2048) -> np.ndarray:
        """Device timeline since the last call: rows of (kernel id, t_entry, t_after_wait, t_end, m4..m7) in ns (VT_B200_TRACE=1)."""
        out = np.zeros((max_records, 8), np.uint64)
        n = C.c_int32(0)
        check(lib().vt_tracker_debug_trace(self._h, out.ctypes.data_as(C.POINTER(C.c_uint64)), max_records, C.byref(n)), "vt_tracker_debug_trace")
        return out[: n.value]

    def timing(self) -> vt_timing:
        t = vt_timing()
        check(lib().vt_timing_get(self._h, C.byref(t)), "vt_timing_get")
        return t

    @property
    def stream(self) -> int:
        return lib().vt_tracker_stream(self._h) or 0

    def sync(self) -> None:
        check(lib().vt_tracker_sync(self._h), "vt_tracker_sync")

    # -- conversion / overlay on this handle's geometry
    def nv12_to_rgb(self, nv12: np.ndarray) -> np.ndarray:
        out = np.empty((self.height, self.width, 3), np.uint8)
        check(lib().vt_convert_nv12_rgb(self._h, _ptr(nv12), nv12.size, _ptr(out)), "vt_convert_nv12_rgb")
        return out

    def nv12_to_rgb_device(self, d_in: int, stride_in: int, d_out: int, stride_out: int, n_frames: int) -> None:
        check(lib().vt_convert_nv12_rgb_device(self._h, C.c_void_p(d_in), stride_in, C.c_void_p(d_out), stride_out, n_frames),
              "vt_convert_nv12_rgb_device")

    # ---- format steps either side of the RGB probe (SURVEY.md §8(f) row 1) ----
    def yuy2_to_rgb(self, yuy2: np.ndarray, width: int, height: int) -> np.ndarray:
        """≙ the videoconvert YUY2 -> RGB step of src/pipeline_ir.rs:27-56."""
        yuy2 = np.ascontiguousarray(yuy2, dtype=np.uint8).reshape(-1)
        out = np.empty((height, width, 3), np.uint8)
        check(lib().vt_convert_yuy2_rgb(self._h, _ptr(yuy2), yuy2.size, width, height, _ptr(out)), "vt_convert_yuy2_rgb")
        return out

    def yuy2_to_rgb_device(self, d_in: int, stride_in: int, d_out: int, stride_out: int, width: int, height: int, n_frames: int) -> None:
        check(lib().vt_convert_yuy2_rgb_device(self._h, C.c_void_p(d_in), stride_in, C.c_void_p(d_out), stride_out, width, height, n_frames),
              "vt_convert_yuy2_rgb_device")

    def resize_rgb(self, rgb: np.ndarray, dst_w: int, dst_h: int) -> np.ndarray:
        """≙ the rgaconvert display upscale of src/pipeline_ir.rs:62-73 (bilinear, bit-exact with cv2.resize INTER_LINEAR)."""
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        sh, sw = rgb.shape[0], rgb.shape[1]
        out = np.empty((dst_h, dst_w, 3), np.uint8)
        check(lib().vt_resize_rgb(self._h, _ptr(rgb), sw, sh, _ptr(out), dst_w, dst_h), "vt_resize_rgb")
        return out

    def resize_rgb_device(self, d_in: int, sw: int, sh: int, d_out: int, dw: int, dh: int) -> None:
        check(lib().vt_resize_rgb_device(self._h, C.c_void_p(d_in), sw, sh, C.c_void_p(d_out), dw, dh), "vt_resize_rgb_device")

    def resize_rgb_device_batch(self, d_in: int, stride_in: int, sw: int, sh: int, d_out: int, stride_out: int, dw: int, dh: int, n: int) -> None:
        check(lib().vt_resize_rgb_device_batch(self._h, C.c_void_p(d_in), stride_in, sw, sh, C.c_void_p(d_out), stride_out, dw, dh, n),
              "vt_resize_rgb_device_batch")

    def overlay(self, frame: np.ndarray, cmds: Sequence[vt_overlay_cmd], current: bool = False) -> None:
        arr = (vt_overlay_cmd * len(cmds))(*cmds)
        fn = lib().vt_overlay_current if current else lib().vt_overlay
        check(fn(self._h, _ptr(frame), frame.size, arr, len(cmds)), "vt_overlay")


def debug_gemm(A: np.ndarray, W: np.ndarray, bias: Optional[np.ndarray] = None, nsplit: int = 3, gelu: bool = False, device: int = 0):
    """C = A @ W.T (+bias) through the tcgen05 GEMM kernel; returns (C, err_flag)."""
    A = np.ascontiguousarray(A, np.float32)
    W = np.ascontiguousarray(W, np.float32)
    M, K = A.shape
    N = W.shape[0]
    out = np.empty((M, N), np.float32)
    err = C.c_int32(0)
    f = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    b = np.ascontiguousarray(bias, np.float32) if bias is not None else None
    check(lib().vt_debug_gemm(device, M, N, K, f(A), f(W), f(b) if b is not None else None, nsplit, int(gelu), f(out), C.byref(err)),
          "vt_debug_gemm")
    return out, err.value


def overlay_cmd(kind: int, x=0, y=0, w=0, h=0, a=0, r=255, g=0, b=0, text: str = "", strict: bool = False) -> vt_overlay_cmd:
    c = vt_overlay_cmd()
    c.kind, c.x, c.y, c.w, c.h, c.a, c.r, c.g, c.b, c.strict_glyphs = kind, x, y, w, h, a, r, g, b, int(strict)
    c.text = text.encode("latin-1")[:47]
    return c


# ---- reference-named free functions (each is one overlay command on the GPU) ----------------------
_scratch = {}


def _handle_for(width: int, height: int, fmt: str) -> VitTrack:
    """A weight-less use of the pixel kernels still needs a handle (stream + device buffers)."""
    key = (width, height, fmt)
    if key not in _scratch:
        import os
        import tempfile

        from .weights import ensure_weight_file
        path = ensure_weight_file("nano", os.path.join(tempfile.gettempdir(), "vt_b200_weights"))
        _scratch[key] = VitTrack.new(path, width, height, fmt=fmt)
    return _scratch[key]


def nv12_full_to_rgb_parallel(nv12_data: np.ndarray, width: int, height: int) -> np.ndarray:
    """≙ nv12_full_to_rgb_parallel (src/nv12_convert.rs:46): (h, w, 3) uint8 in R,G,B order; short input -> zeros."""
    return _handle_for(width, height, "nv12").nv12_to_rgb(nv12_data)


def draw_rect_nv12(data, width, height, x, y, w, h, thickness, brightness):
    _handle_for(width, height, "nv12").overlay(data, [overlay_cmd(L.VT_OV_RECT, x, y, w, h, thickness, brightness)])


def draw_crosshair_nv12(data, width, height, cx, cy, size, brightness):
    _handle_for(width, height, "nv12").overlay(data, [overlay_cmd(L.VT_OV_CROSSHAIR, cx, cy, 0, 0, size, brightness)])


def draw_text_nv12(data, width, height, text, x, y, scale, brightness):
    _handle_for(width, height, "nv12").overlay(data, [overlay_cmd(L.VT_OV_TEXT, x, y, 0, 0, scale, brightness, text=text)])


def draw_background_nv12(data, width, height, x, y, w, h, darkness):
    _handle_for(width, height, "nv12").overlay(data, [overlay_cmd(L.VT_OV_BACKGROUND, x, y, w, h, darkness)])


def draw_cursor(data, w, h, x, y):
    _handle_for(w, h, "nv12").overlay(data, [overlay_cmd(L.VT_OV_CURSOR, x, y)])


def draw_selection(data, w, h, start_x, start_y, cursor_x, cursor_y, selecting_area=True):
    if selecting_area:
        _handle_for(w, h, "nv12").overlay(data, [overlay_cmd(L.VT_OV_SELECTION, start_x, start_y, cursor_x, cursor_y)])


def draw_background_rgb(data, w, h, x, y, bw, bh, dim=150):
    _handle_for(w, h, "rgb24").overlay(data, [overlay_cmd(L.VT_OV_BACKGROUND, x, y, bw, bh, dim)])


def draw_rect_rgb(data, w, h, x, y, rw, rh, thickness, r, g, b):
    _handle_for(w, h, "rgb24").overlay(data, [overlay_cmd(L.VT_OV_RECT, x, y, rw, rh, thickness, r, g, b)])


def draw_crosshair_rgb(data, w, h, cx, cy, size, r, g, b):
    _handle_for(w, h, "rgb24").overlay(data, [overlay_cmd(L.VT_OV_CROSSHAIR, cx, cy, 0, 0, size, r, g, b)])


def draw_cursor_rgb(data, w, h, cx, cy):
    _handle_for(w, h, "rgb24").overlay(data, [overlay_cmd(L.VT_OV_CURSOR, cx, cy, r=0, g=255, b=0)])


def draw_text_rgb(data, w, h, text, x, y, scale, luma):
    """Unknown characters raise VtError(VT_ERR_GLYPH) ≙ the get_glyph panic (src/drawing.rs:99)."""
    _handle_for(w, h, "rgb24").overlay(data, [overlay_cmd(L.VT_OV_TEXT, x, y, 0, 0, scale, luma, text=text, strict=True)])


def draw_selection_rgb(data, w, h, start_x, start_y, cursor_x, cursor_y, selecting_area=True):
    if selecting_area:
        _handle_for(w, h, "rgb24").overlay(data, [overlay_cmd(L.VT_OV_SELECTION, start_x, start_y, cursor_x, cursor_y, r=255, g=255, b=0)])


# ---- TrackerContext -------------------------------------------------------------------------------
class TrackerContext:
    """≙ TrackerContext (src/tracker_context.rs:7-167)."""

    def __init__(self, cfg: Optional[vt_config], _scripted_size: Optional[Tuple[int, int]] = None):
        h = C.c_void_p()
        if cfg is None:
            w, hh = _scripted_size
            check(lib().vt_context_create_scripted(w, hh, C.byref(h)), "vt_context_create_scripted")
            self._h, self._cfg, self.tracker = h, None, None
            self.frame_width, self.frame_height = w, hh
            return
        check(lib().vt_context_create(C.byref(cfg), C.byref(h)), "vt_context_create")
        self._h = h
        self._cfg = cfg
        self.frame_width, self.frame_height = cfg.width, cfg.height
        self.tracker = VitTrack(cfg, _handle=C.c_void_p(lib().vt_context_tracker(h)), _owned=False)

    @classmethod
    def scripted(cls, width: int, height: int) -> "TrackerContext":
        """The state machine alone: update() outcomes are supplied to process_scripted (no GPU)."""
        return cls(None, (width, height))

    def process_scripted(self, result: Optional[TrackResult], err: bool = False) -> Optional[BBox]:
        r = vt_result()
        if result is not None:
            r.success, r.score, r.bbox, r.status = int(result.success), result.score, vt_bbox(*result.bbox), 0
        has, b = C.c_int32(0), vt_bbox()
        check(lib().vt_context_process_scripted(self._h, C.byref(r), int(err), C.byref(has), C.byref(b)), "vt_context_process_scripted")
        return BBox(*b.tuple()) if has.value else None

    @classmethod
    def new(cls, model_path: str, width: int, height: int, **kw) -> "TrackerContext":
        return cls(make_config(model_path, width, height, **kw))

    @classmethod
    def _member(cls, handle: C.c_void_p, cfg: vt_config, width: int, height: int) -> "TrackerContext":
        """A non-owning view of a probe group's member context (close() leaves it to the group)."""
        self = cls.__new__(cls)
        self._h, self._cfg, self._owned = handle, cfg, False
        self.frame_width, self.frame_height = width, height
        self.tracker = VitTrack(cfg, _handle=C.c_void_p(lib().vt_context_tracker(handle)), _owned=False)
        return self

    def close(self):
        if getattr(self, "_h", None) and getattr(self, "_owned", True):
            lib().vt_context_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def handle_command(self, cmd: int, fast: bool = False) -> None:
        check(lib().vt_context_handle_command(self._h, cmd, int(fast)), "vt_context_handle_command")

    def process_frame(self, full_image: np.ndarray) -> Optional[BBox]:
        has, b = C.c_int32(0), vt_bbox()
        check(lib().vt_context_process_frame(self._h, _ptr(full_image), full_image.size, C.byref(has), C.byref(b)),
              "vt_context_process_frame")
        return BBox(*b.tuple()) if has.value else None

    def state_name(self) -> str:
        return lib().vt_context_state_name(self._h).decode()

    @property
    def current_score(self) -> float:
        return lib().vt_context_current_score(self._h)

    @property
    def current_bbox(self) -> Optional[BBox]:
        b = vt_bbox()
        return BBox(*b.tuple()) if lib().vt_context_current_bbox(self._h, C.byref(b)) else None

    @property
    def selection(self) -> vt_selection:
        s = vt_selection()
        lib().vt_context_selection(self._h, C.byref(s))
        return s

    @property
    def lost_frames(self) -> int:
        return lib().vt_context_lost_frames(self._h)

    def run_ring(self, base_ptr: int, stride: int, frame_len: int, ring: int, first: int, n: int, hud: Optional[Tuple[str, str]] = None,
                 pristine_ptr: int = 0, want_latency: bool = False):
        """n frames of a host ring through vt_probe_frame in one native call (vt_context_run_ring)."""
        arr = (C.c_char_p * 2)(hud[0].encode(), hud[1].encode()) if hud is not None else None
        lat = np.empty(n, np.float64) if want_latency else None
        check(lib().vt_context_run_ring(self._h, C.c_void_p(base_ptr), stride, frame_len, ring, first, n, arr,
                                        C.c_void_p(pristine_ptr) if pristine_ptr else None,
                                        lat.ctypes.data_as(C.POINTER(C.c_double)) if want_latency else None), "vt_context_run_ring")
        return lat

    def probe(self, frame: np.ndarray, hud: Optional[Tuple[str, str]] = None) -> None:
        """≙ one invocation of the pad-probe closure (src/pipeline.rs:67-184 / src/pipeline_ir.rs:100-228)."""
        arr = None
        if hud is not None:
            arr = (C.c_char_p * 2)(hud[0].encode(), hud[1].encode())
        check(lib().vt_probe_frame(self._h, _ptr(frame), frame.size, arr), "vt_probe_frame")

    def probe_surface(self, surface: Surface, hud: Optional[Tuple[str, str]] = None) -> None:
        """probe() on a pitched device surface of the context's geometry (PitchedFrame.surface, a decoder's output): HUD, cursor /
        selection and box drawn in place into its plane 0 (vt_probe_frame_surface)."""
        arr = (C.c_char_p * 2)(hud[0].encode(), hud[1].encode()) if hud is not None else None
        s = _surface(surface)
        check(lib().vt_probe_frame_surface(self._h, C.byref(s), arr), "vt_probe_frame_surface")


class TimingStats:
    """≙ TimingStats (src/timing_stats.rs): free-standing (TimingStats.new()) or bound to a tracker handle's windows."""

    def __init__(self, tracker: Optional[VitTrack] = None):
        self._t = tracker
        self._s = None if tracker is not None else C.c_void_p(lib().vt_timing_stats_create())

    @classmethod
    def new(cls) -> "TimingStats":
        return cls()

    def __del__(self):
        try:
            if self._s:
                lib().vt_timing_stats_destroy(self._s)
                self._s = None
        except Exception:
            pass

    def add_interval(self, us: int) -> None:
        if self._s:
            lib().vt_timing_stats_add_interval(self._s, int(us))
        else:
            check(lib().vt_timing_add_interval(self._t._h, int(us)), "vt_timing_add_interval")

    def add_times(self, conv: int, track: int) -> None:
        if self._s:
            lib().vt_timing_stats_add_times(self._s, int(conv), int(track))
        else:
            check(lib().vt_timing_add_times(self._t._h, int(conv), int(track)), "vt_timing_add_times")

    def fps(self) -> float:
        return lib().vt_timing_stats_fps(self._s) if self._s else self._t.timing().fps

    def avg_conv_ms(self) -> float:
        return lib().vt_timing_stats_avg_conv_ms(self._s) if self._s else self._t.timing().avg_conv_ms

    def avg_track_ms(self) -> float:
        return lib().vt_timing_stats_avg_track_ms(self._s) if self._s else self._t.timing().avg_track_ms


class ProbeGroup:
    """Probe groups (vt_probe_group_*): the drop-in probe for up to 16 cameras in one batched forward.  Stream i behaves exactly like a
    TrackerContext of its own geometry probing the same frames with the same commands; one step runs ONE batched forward over the streams
    whose state machine calls VitTrack on that frame and draws every stream's HUD in place, with one synchronisation.

    `contexts[i]` is a non-owning TrackerContext view of stream i (commands, state, score, box, selection; its `tracker` is the group's
    shared tracker, on which stream i is target i); `tracker` is that shared tracker."""

    def __init__(self, cfg: vt_config, cams: Sequence[Tuple[int, int, str]]):
        n = len(cams)
        geoms = (vt_stream_geometry * max(n, 1))(*[vt_stream_geometry(FORMATS[f], int(w), int(h), 0) for (w, h, f) in cams])
        cfg.max_targets = max(n, 1)  # (the group's tracker has one target slot per stream)
        h = C.c_void_p()
        check(lib().vt_probe_group_create(C.byref(cfg), n, geoms, C.byref(h)), "vt_probe_group_create")
        self._h, self._cfg = h, cfg
        self.cams = [(int(w), int(h_), f) for (w, h_, f) in cams]
        self.contexts = [TrackerContext._member(C.c_void_p(lib().vt_probe_group_context(h, i)), cfg, w, h_) for i, (w, h_, _) in enumerate(self.cams)]
        self.tracker = self.contexts[0].tracker if n else None

    @classmethod
    def new(cls, model_path: str, cams: Sequence[Tuple[int, int, str]], **kw) -> "ProbeGroup":
        """cams = [(width, height, fmt), ...] (1..16 streams); kw: make_config's (the format / size there default to cams[0]'s)."""
        w, h, f = cams[0] if cams else (1920, 1080, "nv12")
        kw.setdefault("fmt", f)
        return cls(make_config(model_path, w, h, **kw), cams)

    def __len__(self) -> int:
        return lib().vt_probe_group_size(self._h) if self._h else 0

    def close(self):
        if getattr(self, "_h", None):
            for c in self.contexts:
                c._h = None
            self.tracker = None
            lib().vt_probe_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def probe(self, frames: Sequence[np.ndarray], hud: Optional[Tuple[str, str]] = None) -> None:
        """One step: frames[i] — a full frame of stream i in pinned host memory (PinnedBuffer) — probed and drawn on in place."""
        n = len(frames)
        ptrs = (C.c_void_p * n)(*[_ptr(f).value for f in frames])
        lens = (C.c_size_t * n)(*[f.size for f in frames])
        arr = (C.c_char_p * 2)(hud[0].encode(), hud[1].encode()) if hud is not None else None
        check(lib().vt_probe_group_frame(self._h, ptrs, lens, arr), "vt_probe_group_frame")

    def probe_surfaces(self, surfaces: Sequence[Surface], hud: Optional[Tuple[str, str]] = None) -> None:
        """One step on device surfaces: surfaces[i] — stream i's current frame, of its geometry — probed and drawn on in place
        (vt_probe_group_frame_surface)."""
        n = len(surfaces)
        arr_s = (vt_surface * max(n, 1))(*[_surface(s) for s in surfaces])
        arr = (C.c_char_p * 2)(hud[0].encode(), hud[1].encode()) if hud is not None else None
        check(lib().vt_probe_group_frame_surface(self._h, arr_s, n, arr), "vt_probe_group_frame_surface")

    def run_ring(self, ring_ptrs: Sequence[int], stride: int, frame_len: int, ring: int, first: int, n: int,
                 hud: Optional[Tuple[str, str]] = None, pristine_ptrs: Optional[Sequence[int]] = None, want_latency: bool = False):
        """n steps over per-stream host rings (pinned) in one native call (vt_probe_group_run_ring); returns the step latencies (us)."""
        k = len(ring_ptrs)
        rings = (C.c_void_p * k)(*ring_ptrs)
        pr = (C.c_void_p * k)(*pristine_ptrs) if pristine_ptrs is not None else None
        arr = (C.c_char_p * 2)(hud[0].encode(), hud[1].encode()) if hud is not None else None
        lat = np.empty(n, np.float64) if want_latency else None
        check(lib().vt_probe_group_run_ring(self._h, rings, stride, frame_len, ring, first, n, arr, pr,
                                            lat.ctypes.data_as(C.POINTER(C.c_double)) if want_latency else None), "vt_probe_group_run_ring")
        return lat
