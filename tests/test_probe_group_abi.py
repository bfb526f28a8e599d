"""The probe-group part of the C ABI on a CPU-only box: every group call with NULL or bad arguments fails with VT_ERR_INVALID and a message
before anything touches a device, and examples/probe_group.c builds warning-free against the library."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

from conftest import ROOT

GCC = ["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror"]


def _cfg(_lib, L):
    cfg = _lib.vt_config()
    L.vt_config_default(C.byref(cfg))
    cfg.weights_path = b"/nonexistent/model.vtw"
    cfg.width, cfg.height, cfg.format = 1920, 1080, _lib.VT_FMT_NV12
    return cfg


def _invalid(L, _lib, status):
    assert status == _lib.VT_ERR_INVALID
    msg = L.vt_last_error()
    assert msg, "no message for VT_ERR_INVALID"
    return msg.decode()


def test_group_calls_reject_null_arguments(built):
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    out = C.c_void_p(1)
    _invalid(L, _lib, L.vt_probe_group_create(None, 2, None, C.byref(out)))
    assert not out.value  # cleared, never a dangling handle
    _invalid(L, _lib, L.vt_probe_group_create(C.byref(_cfg(_lib, L)), 2, None, None))
    _invalid(L, _lib, L.vt_probe_group_frame(None, None, None, None))
    _invalid(L, _lib, L.vt_probe_group_run_ring(None, None, 0, 0, 1, 0, 1, None, None, None))
    assert L.vt_probe_group_size(None) == _lib.VT_ERR_INVALID
    assert not L.vt_probe_group_context(None, 0)
    L.vt_probe_group_destroy(None)  # a no-op


@pytest.mark.parametrize("n", [0, -1, 17, 64])
def test_group_size_outside_1_to_16_is_invalid(built, n):
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    out = C.c_void_p()
    msg = _invalid(L, _lib, L.vt_probe_group_create(C.byref(_cfg(_lib, L)), n, None, C.byref(out)))
    assert "streams" in msg and not out.value


@pytest.mark.parametrize("geom", [(_f, w, h, r) for (_f, w, h, r) in [(7, 640, 512, 0), (3, 0, 512, 0), (3, 640, -1, 0), (0, 640, 480, 1)]])
def test_bad_stream_geometry_is_invalid_before_any_device_work(built, geom):
    """validated as vt_tracker_set_stream_geometry, ahead of creating the tracker: no device is needed to be told"""
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    geoms = (_lib.vt_stream_geometry * 2)(_lib.vt_stream_geometry(_lib.VT_FMT_NV12, 1920, 1080, 0), _lib.vt_stream_geometry(*geom))
    out = C.c_void_p()
    msg = _invalid(L, _lib, L.vt_probe_group_create(C.byref(_cfg(_lib, L)), 2, geoms, C.byref(out)))
    assert "stream 1" in msg and not out.value


def test_probe_group_example_builds(built, tmp_path):
    from gstreamer_vit_tracker_b200 import _lib

    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    inc, libdir = os.path.join(ROOT, "include"), os.path.dirname(_lib.LIB_PATH)
    subprocess.run(GCC + ["-I", inc, os.path.join(ROOT, "examples", "probe_group.c"), "-L", libdir, "-lvittrack_b200", f"-Wl,-rpath,{libdir}",
                          "-o", str(tmp_path / "probe_group")], check=True, capture_output=True)
