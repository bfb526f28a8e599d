"""The probe's surface entry points on a CPU-only box: both are exported, a C99 program calling them builds warning-free against the
header, and NULL contexts, groups or surfaces fail with VT_ERR_INVALID and a message before anything touches a device."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

from conftest import ROOT

GCC = ["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror"]

PROGRAM = r"""
#include <stdio.h>
#include "vt_tracker.h"

int main(void) {
    vt_context* c = NULL;
    vt_probe_group* g = NULL;
    vt_surface s[2] = {{{NULL, NULL}, {0, 0}}, {{NULL, NULL}, {0, 0}}};
    const char* const hud[2] = {"FPS: 60", "conv:0.1ms trk:0.5ms"};
    vt_status a = vt_probe_frame_surface(c, &s[0], hud);
    vt_status b = vt_probe_group_frame_surface(g, s, 2, NULL);
    printf("%d %d\n", (int)a, (int)b);
    return a == VT_ERR_INVALID && b == VT_ERR_INVALID ? 0 : 1;
}
"""


def _invalid(L, _lib, status):
    assert status == _lib.VT_ERR_INVALID
    msg = L.vt_last_error()
    assert msg, "no message for VT_ERR_INVALID"
    return msg.decode()


def test_surface_probe_symbols_exported(built):
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    for name in ("vt_probe_frame_surface", "vt_probe_group_frame_surface"):
        assert hasattr(L, name) and name in _lib.SYMBOLS


def test_c99_program_builds_and_gets_invalid(built, tmp_path):
    from gstreamer_vit_tracker_b200 import _lib

    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    src = tmp_path / "p.c"
    src.write_text(PROGRAM)
    exe = tmp_path / "p"
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.run(GCC + ["-I", os.path.join(ROOT, "include"), str(src), "-L", libdir, "-lvittrack_b200", f"-Wl,-rpath,{libdir}", "-o", str(exe)],
                   check=True, capture_output=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr


def test_null_arguments_are_invalid_without_a_device(built):
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    s = _lib.vt_surface()
    arr = (_lib.vt_surface * 2)()
    assert "surface" in _invalid(L, _lib, L.vt_probe_frame_surface(None, C.byref(s), None))
    assert "group" in _invalid(L, _lib, L.vt_probe_group_frame_surface(None, arr, 2, None))
    # a context without a tracker (the scripted state machine) and a NULL surface
    ctx = C.c_void_p()
    assert L.vt_context_create_scripted(640, 480, C.byref(ctx)) == _lib.VT_OK
    _invalid(L, _lib, L.vt_probe_frame_surface(ctx, C.byref(s), None))
    _invalid(L, _lib, L.vt_probe_frame_surface(ctx, None, None))
    L.vt_context_destroy(ctx)
