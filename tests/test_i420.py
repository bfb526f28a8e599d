"""Planar I420 frames, the parts that need no GPU: the ABI constant, create-time validation of the format (single handles and probe-group
stream geometries), and synth.rgb_to_i420 in GStreamer's default layout."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from gstreamer_vit_tracker_b200 import synth


def test_fmt_i420_matches_header(built, tmp_path):
    """_lib.VT_FMT_I420 is the header's value (C99 program built with gcc): 8."""
    from gstreamer_vit_tracker_b200 import _lib

    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    src = tmp_path / "f.c"
    src.write_text('#include "vt_tracker.h"\n#include <stdio.h>\nint main(void) { printf("%d\\n", VT_FMT_I420); return 0; }\n')
    exe = tmp_path / "f"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True, capture_output=True)
    got = int(subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout)
    assert got == _lib.VT_FMT_I420 == 8


def test_create_accepts_i420_and_rejects_4_7_9(built):
    """Format 8 passes the configuration check at 1920x1080 and 641x481 (on a box without a GPU create then fails with VT_ERR_CUDA; with
    one, on the missing weights file); 4, 7 and 9 are VT_ERR_INVALID."""
    import torch

    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    past = _lib.VT_ERR_WEIGHTS if torch.cuda.is_available() else _lib.VT_ERR_CUDA
    cases = [(_lib.VT_FMT_I420, 1920, 1080, past), (_lib.VT_FMT_I420, 641, 481, past)]
    cases += [(f, 641, 481, _lib.VT_ERR_INVALID) for f in (4, 7, 9)]
    for fmt, w, h, want in cases:
        cfg = _lib.vt_config()
        L.vt_config_default(C.byref(cfg))
        cfg.weights_path = b"/nonexistent/weights.vtw"
        cfg.format, cfg.width, cfg.height = fmt, w, h
        out = C.c_void_p()
        assert L.vt_tracker_create(C.byref(cfg), C.byref(out)) == want, (fmt, w, h)
        assert not out.value


def test_probe_group_takes_i420_stream_geometry(built):
    """vt_probe_group_create with an I420 stream geometry gets as far as the same call with an all-NV12 geometry on this box (the weights,
    or the device): the geometry passes its check and is never VT_ERR_INVALID."""
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()

    def create(f):
        cfg = _lib.vt_config()
        L.vt_config_default(C.byref(cfg))
        cfg.weights_path = b"/nonexistent/model.vtw"
        cfg.width, cfg.height, cfg.format = 1920, 1080, _lib.VT_FMT_NV12
        geoms = (_lib.vt_stream_geometry * 2)(_lib.vt_stream_geometry(_lib.VT_FMT_NV12, 1920, 1080, 0), _lib.vt_stream_geometry(f, 641, 481, 0))
        out = C.c_void_p()
        st = L.vt_probe_group_create(C.byref(cfg), 2, geoms, C.byref(out))
        assert not out.value
        return st

    got, ref = create(_lib.VT_FMT_I420), create(_lib.VT_FMT_NV12)
    assert got == ref and got != _lib.VT_ERR_INVALID


@pytest.mark.parametrize("w,h,size,s0,s1", [(1920, 1080, 3110400, 1920, 960), (640, 512, 491520, 640, 320), (641, 481, 466576, 644, 324)])
def test_rgb_to_i420_layout(w, h, size, s0, s1):
    """Frame sizes, strides and plane offsets of GStreamer's default I420 layout (1920x1080 is W*H*3/2; 641x481 has a Y padding row)."""
    f = synth.rgb_to_i420(synth.hash_u8(w * h, (h, w, 3)))
    assert f.dtype == np.uint8 and f.size == size
    y_rows = h + (h & 1)
    assert synth.i420_layout(w, h) == (s0, s1, s0 * y_rows, s0 * y_rows + s1 * ((h + 1) // 2), size)
    from gstreamer_vit_tracker_b200 import api

    assert api.row_bytes("i420", w) == s0


def test_rgb_to_i420_interleaves_to_rgb_to_nv12():
    """At even sizes, interleaving the U and V planes gives exactly synth.rgb_to_nv12 of the same image (same Y, same 2x2 chroma)."""
    for w, h in ((640, 512), (46, 30), (18, 10)):  # 46: chroma rows of 23 bytes, padded to 24
        rgb = synth.hash_u8(w + h, (h, w, 3))
        f, nv = synth.rgb_to_i420(rgb), synth.rgb_to_nv12(rgb)
        s0, s1, uo, vo, _ = synth.i420_layout(w, h)
        y = f[: s0 * h].reshape(h, s0)[:, :w]
        u = f[uo:vo].reshape(h // 2, s1)[:, : w // 2]
        v = f[vo:].reshape(h // 2, s1)[:, : w // 2]
        uv = np.stack([u, v], axis=-1).reshape(h // 2, w)
        assert np.array_equal(np.concatenate([y.reshape(-1), uv.reshape(-1)]), nv), (w, h)


def test_rgb_to_i420_odd_sizes_and_padding():
    """641x481: every padding byte (Y row padding, the Y padding row, chroma row padding) is zero; the visible samples are those of
    rgb_to_nv12 on the image with its last column and row replicated."""
    w, h = 641, 481
    rgb = synth.hash_u8(5, (h, w, 3))
    f = synth.rgb_to_i420(rgb)
    s0, s1, uo, vo, n = synth.i420_layout(w, h)
    Y = f[:uo].reshape(h + 1, s0)
    assert not Y[:, w:].any() and not Y[h].any()
    cw, ch = (w + 1) // 2, (h + 1) // 2
    U, V = f[uo:vo].reshape(ch, s1), f[vo:].reshape(ch, s1)
    assert not U[:, cw:].any() and not V[:, cw:].any()
    ext = np.pad(rgb, ((0, 1), (0, 1), (0, 0)), mode="edge")
    nv = synth.rgb_to_nv12(ext)
    W2, H2 = w + 1, h + 1
    assert np.array_equal(Y[:h, :w], nv[: W2 * H2].reshape(H2, W2)[:h, :w])
    uv = nv[W2 * H2:].reshape(ch, cw, 2)
    assert np.array_equal(U[:, :cw], uv[..., 0]) and np.array_equal(V[:, :cw], uv[..., 1])
