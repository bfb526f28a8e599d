"""The stream-geometry part of the C ABI (stream groups of mixed cameras) on a CPU-only box: the ctypes struct matches the header's
layout as a C99 compiler sees it, and examples/mixed_group.c builds warning-free against the library."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

from conftest import ROOT

GCC = ["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror"]


def _need_gcc():
    if not shutil.which("gcc"):
        pytest.skip("no gcc")


def test_stream_geometry_layout_matches_header(built, tmp_path):
    from gstreamer_vit_tracker_b200 import _lib

    _need_gcc()
    src = tmp_path / "g.c"
    src.write_text('#include "vt_tracker.h"\n#include <stddef.h>\n#include <stdio.h>\n'
                   "int main(void) {\n"
                   '  printf("%d %d %d %d %d\\n", (int)sizeof(vt_stream_geometry), (int)offsetof(vt_stream_geometry, format),\n'
                   "         (int)offsetof(vt_stream_geometry, width), (int)offsetof(vt_stream_geometry, height),\n"
                   "         (int)offsetof(vt_stream_geometry, reserved));\n  return 0; }\n")
    exe = tmp_path / "g"
    subprocess.run(GCC + ["-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True, capture_output=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    G = _lib.vt_stream_geometry
    assert got == [C.sizeof(G), G.format.offset, G.width.offset, G.height.offset, G.reserved.offset]


def test_stream_geometry_calls_reject_bad_arguments(built):
    """No handle, no output, no device: the geometry calls fail with VT_ERR_INVALID and a message (never touch memory)."""
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    g = _lib.vt_stream_geometry(_lib.VT_FMT_YUY2, 640, 512, 0)
    assert L.vt_tracker_set_stream_geometry(None, 0, C.byref(g)) == _lib.VT_ERR_INVALID
    assert L.vt_last_error()
    assert L.vt_tracker_get_stream_geometry(None, 0, C.byref(g)) == _lib.VT_ERR_INVALID


def test_mixed_group_example_builds(built, tmp_path):
    from gstreamer_vit_tracker_b200 import _lib

    _need_gcc()
    inc, libdir = os.path.join(ROOT, "include"), os.path.dirname(_lib.LIB_PATH)
    subprocess.run(GCC + ["-I", inc, os.path.join(ROOT, "examples", "mixed_group.c"), "-L", libdir, "-lvittrack_b200", f"-Wl,-rpath,{libdir}",
                          "-o", str(tmp_path / "mixed_group")], check=True, capture_output=True)
