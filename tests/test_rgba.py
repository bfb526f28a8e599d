"""32-bit RGBA / BGRA frames, the parts that need no GPU: the ABI constants, create-time validation of the formats (single handles and
probe-group stream geometries), and synth.rgb_to_rgba / rgb_to_bgra."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from gstreamer_vit_tracker_b200 import synth


def test_fmt_rgba_bgra_match_header(built, tmp_path):
    """_lib.VT_FMT_RGBA / VT_FMT_BGRA are the header's values (C99 program built with gcc): 5 and 6, so 4 stays unassigned."""
    from gstreamer_vit_tracker_b200 import _lib

    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    src = tmp_path / "f.c"
    src.write_text('#include "vt_tracker.h"\n#include <stdio.h>\n'
                   'int main(void) { printf("%d %d\\n", VT_FMT_RGBA, VT_FMT_BGRA); return 0; }\n')
    exe = tmp_path / "f"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True, capture_output=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [_lib.VT_FMT_RGBA, _lib.VT_FMT_BGRA] == [5, 6]


def test_create_accepts_rgba_bgra_and_rejects_4_and_7(built):
    """Formats 5 and 6 pass the configuration check (on a box without a GPU create then fails with VT_ERR_CUDA; with one, on the missing
    weights file), at odd sizes too; 4 and 7 are VT_ERR_INVALID."""
    import torch

    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    past = _lib.VT_ERR_WEIGHTS if torch.cuda.is_available() else _lib.VT_ERR_CUDA
    for fmt, want in ((_lib.VT_FMT_RGBA, past), (_lib.VT_FMT_BGRA, past), (4, _lib.VT_ERR_INVALID), (7, _lib.VT_ERR_INVALID)):
        cfg = _lib.vt_config()
        L.vt_config_default(C.byref(cfg))
        cfg.weights_path = b"/nonexistent/weights.vtw"
        cfg.format, cfg.width, cfg.height = fmt, 641, 481
        h = C.c_void_p()
        assert L.vt_tracker_create(C.byref(cfg), C.byref(h)) == want, fmt
        assert not h.value


@pytest.mark.parametrize("fmt", [5, 6])
def test_probe_group_takes_rgba_bgra_stream_geometries(built, fmt):
    """vt_probe_group_create with a 5 / 6 stream geometry gets as far as the same call with an all-NV12 geometry on this box (the
    weights, or the device): the geometry passes its check and is never VT_ERR_INVALID."""
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

    got, ref = create(fmt), create(_lib.VT_FMT_NV12)
    assert got == ref and got != _lib.VT_ERR_INVALID


def test_rgb_to_rgba_bgra_known_answers():
    """Byte order R G B pad / B G R pad, rows of 4 * W bytes; pad is a constant or one byte per pixel."""
    rgb = np.array([[(1, 2, 3), (4, 5, 6), (7, 8, 9)]], np.uint8)  # odd width
    assert synth.rgb_to_rgba(rgb).tolist() == [1, 2, 3, 255, 4, 5, 6, 255, 7, 8, 9, 255]
    assert synth.rgb_to_bgra(rgb).tolist() == [3, 2, 1, 255, 6, 5, 4, 255, 9, 8, 7, 255]
    assert synth.rgb_to_rgba(rgb, pad=0).tolist() == [1, 2, 3, 0, 4, 5, 6, 0, 7, 8, 9, 0]
    pad = np.array([[10, 20, 30]], np.uint8)
    assert synth.rgb_to_bgra(rgb, pad=pad).tolist() == [3, 2, 1, 10, 6, 5, 4, 20, 9, 8, 7, 30]
    two = synth.rgb_to_rgba(np.concatenate([rgb, rgb], axis=0), pad=np.arange(6, dtype=np.uint8).reshape(2, 3))
    assert two.dtype == np.uint8 and two.size == 4 * 3 * 2
    assert two.reshape(2, 3, 4)[..., 3].tolist() == [[0, 1, 2], [3, 4, 5]]


def test_rgba_colour_bytes_are_the_rgb_image():
    """Any size: bytes 0..2 of RGBA and bytes 2..0 of BGRA are the RGB image; byte 3 is the pad."""
    rgb = synth.hash_u8(9, (5, 7, 3))
    pad = synth.hash_u8(10, (5, 7))
    a = synth.rgb_to_rgba(rgb, pad).reshape(5, 7, 4)
    b = synth.rgb_to_bgra(rgb, pad).reshape(5, 7, 4)
    assert np.array_equal(a[..., :3], rgb) and np.array_equal(b[..., 2::-1], rgb)
    assert np.array_equal(a[..., 3], pad) and np.array_equal(b[..., 3], pad)
