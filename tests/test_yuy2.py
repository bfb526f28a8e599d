"""Packed YUY2 frames, the parts that need no GPU: the ABI constant, create-time validation of the format, and synth.rgb_to_yuy2."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from gstreamer_vit_tracker_b200 import synth


def test_fmt_yuy2_matches_header(built, tmp_path):
    """_lib.VT_FMT_YUY2 is the header's value (C99 program built with gcc), next to the formats that were there before."""
    from gstreamer_vit_tracker_b200 import _lib

    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    src = tmp_path / "f.c"
    src.write_text('#include "vt_tracker.h"\n#include <stdio.h>\n'
                   'int main(void) { printf("%d %d %d %d\\n", VT_FMT_NV12, VT_FMT_RGB24, VT_FMT_GRAY8, VT_FMT_YUY2); return 0; }\n')
    exe = tmp_path / "f"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True, capture_output=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [_lib.VT_FMT_NV12, _lib.VT_FMT_RGB24, _lib.VT_FMT_GRAY8, _lib.VT_FMT_YUY2] == [0, 1, 2, 3]


def test_create_accepts_yuy2_and_rejects_the_next_format(built):
    """Format 3 passes the configuration check (on a box without a GPU create then fails with VT_ERR_CUDA; with one, on the missing
    weights file); format 4 is still VT_ERR_INVALID."""
    import torch

    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    for fmt, want in ((_lib.VT_FMT_YUY2, _lib.VT_ERR_WEIGHTS if torch.cuda.is_available() else _lib.VT_ERR_CUDA), (4, _lib.VT_ERR_INVALID)):
        cfg = _lib.vt_config()
        L.vt_config_default(C.byref(cfg))
        cfg.weights_path = b"/nonexistent/weights.vtw"
        cfg.format, cfg.width, cfg.height = fmt, 641, 481
        h = C.c_void_p()
        assert L.vt_tracker_create(C.byref(cfg), C.byref(h)) == want, fmt
        assert not h.value


@pytest.mark.parametrize("rgb,want", [
    ([(0, 0, 0), (0, 0, 0)], [16, 128, 16, 128]),            # black
    ([(255, 255, 255)] * 2, [235, 128, 235, 128]),           # white
    ([(255, 0, 0)] * 2, [82, 90, 82, 240]),                  # red
    ([(0, 255, 0)] * 2, [144, 54, 144, 34]),                 # green
    ([(0, 0, 255)] * 2, [41, 240, 41, 110]),                 # blue
    ([(0, 0, 0), (255, 0, 0)], [16, 109, 82, 184]),          # a pair that differs: chroma of the rounded mean (128, 0, 0)
    ([(255, 255, 255), (0, 0, 0), (0, 0, 255)], [235, 128, 16, 128, 41, 240, 41, 110]),  # odd width: the last word pads with its pixel
])
def test_rgb_to_yuy2_known_answers(rgb, want):
    """Hand-computed BT.601 limited-range words (Y = ((66 R + 129 G + 25 B + 128) >> 8) + 16, U / V likewise from the pair's mean)."""
    img = np.array(rgb, np.uint8).reshape(1, -1, 3)
    got = synth.rgb_to_yuy2(img)
    assert got.dtype == np.uint8 and got.tolist() == want
    # rows are 4 * ceil(W / 2) bytes
    two = synth.rgb_to_yuy2(np.concatenate([img, img], axis=0))
    assert two.tolist() == want + want


def test_rgb_to_yuy2_shape_and_luma_agree_with_nv12():
    """Any size; the Y samples are the luma rgb_to_nv12 computes for the same image."""
    rgb = synth.hash_u8(5, (6, 10, 3))
    y2 = synth.rgb_to_yuy2(rgb).reshape(6, 20)
    assert np.array_equal(y2[:, 0::2], synth.rgb_to_nv12(rgb)[:60].reshape(6, 10))
    assert synth.rgb_to_yuy2(synth.hash_u8(6, (3, 7, 3))).size == 4 * 4 * 3
