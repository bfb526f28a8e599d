"""Pitched device surfaces (vt_surface): frames in device memory with any row pitch and a chroma plane anywhere, as decoders hand them
over (NVDEC, NvBufSurface), tracked in place.  Every comparison is between handles alive at the same time, so both sides run the same
kernel forms; results must be equal, blobs and overlay pixels bit-identical, and nothing outside the visible pixels may be written."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from gstreamer_vit_tracker_b200 import synth, weights

FILL = 0x5A  # sentinel of every byte outside the visible pixels


@pytest.fixture(scope="module")
def api(built):
    from gstreamer_vit_tracker_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import oracle as _o
    return _o


def test_surface_struct_matches_header(tmp_path):
    """The ctypes vt_surface has the size and field offsets of the header's struct (C99 program built with gcc)."""
    from gstreamer_vit_tracker_b200 import _lib

    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    src = tmp_path / "s.c"
    src.write_text('#include "vt_tracker.h"\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(vt_surface), offsetof(vt_surface, planes), offsetof(vt_surface, pitch),'
                   ' sizeof(((vt_surface*)0)->pitch[0])); return 0; }\n')
    exe = tmp_path / "s"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True, capture_output=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S = _lib.vt_surface
    assert got == [C.sizeof(S), S.planes.offset, S.pitch.offset, C.sizeof(C.c_size_t)]


# ---- helpers -----------------------------------------------------------------------------------------------------------------------
def _gray(st, n):
    W, H = st.spec.width, st.spec.height
    rgb = np.asarray(st.frame(n)).reshape(H, W, 3).astype(np.uint32)
    return ((rgb[..., 0] * 77 + rgb[..., 1] * 150 + rgb[..., 2] * 29 + 128) >> 8).astype(np.uint8).reshape(-1)


def _frames(fmt):
    """(W, H, frame(n) -> packed uint8 frame) of the stream a format is tested on: cfg1 (NV12 1280x720), cfg3 (RGB24 / GRAY8 640x512)."""
    st = synth.SyntheticStream(synth.CONFIGS["cfg1" if fmt == "nv12" else "cfg3"])
    if fmt == "gray8":
        return st, (lambda n: _gray(st, n))
    return st, (lambda n: np.ascontiguousarray(st.frame(n)).reshape(-1))


def _layout(kind, W, H, fmt):
    """packed; "nvdec": rows padded to a multiple of 512 bytes, chroma after the surface height rounded to 32 rows (1280x720 NV12:
    pitch 1536, chroma at row 736); "odd": pitch = row + 3, chroma plane in an allocation of its own."""
    row = W * (3 if fmt == "rgb24" else 1)
    if kind == "packed":
        return dict(pitch=row)
    if kind == "nvdec":
        return dict(pitch=(row + 511) // 512 * 512, chroma_row=(H + 31) // 32 * 32)
    return dict(pitch=row + 3, separate_uv=True)


def _pitched(api, fmt, W, H, kind, frame):
    pf = api.PitchedFrame(W, H, fmt=fmt, fill=FILL, **_layout(kind, W, H, fmt))
    pf.write(frame)
    return pf


def _outside_visible_intact(pf):
    """Every byte of pitch padding, of the gap between the planes (and past the last plane) still holds the sentinel."""
    ok = True
    bufs = [(pf.buf, [(0, pf.height, pf.row)] + ([(pf.uv_offset // pf.pitch, pf.uv_rows, pf.width)] if pf.nv12 and pf.uv_buf is None else []))]
    if pf.uv_buf is not None:
        bufs.append((pf.uv_buf, [(0, pf.uv_rows, pf.width)]))
    for buf, planes in bufs:
        b = buf.cpu().numpy().reshape(-1, pf.pitch)
        mask = np.ones(b.shape, bool)
        for r0, rows, cols in planes:
            mask[r0:r0 + rows, :cols] = False
        ok = ok and bool((b[mask] == FILL).all())
    return ok


def _draw_box(oracle, frame, fmt, W, H, r):
    """The oracle's box overlay (rect thickness 3 + crosshair 15, src/pipeline.rs:165-168) on a packed frame, for a gated result."""
    if not (r.status == 0 and r.success and r.score > 0.25):
        return frame
    x, y, w, h = r.bbox
    if fmt == "rgb24":
        oracle.draw_rect_rgb(frame, W, H, x, y, w, h, 3, (0, 255, 0))
        oracle.draw_crosshair_rgb(frame, W, H, x + w // 2, y + h // 2, 15, (0, 255, 0))
        return frame
    full = frame if fmt == "nv12" else np.concatenate([frame, np.zeros(W * H // 2, np.uint8)])  # GRAY8: NV12 luma semantics
    oracle.draw_rect_nv12(full, W, H, x, y, w, h, 3, 255)
    oracle.draw_crosshair_nv12(full, W, H, x + w // 2, y + h // 2, 15, 255)
    frame[:] = full[:frame.size]
    return frame


# ---- single handle -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["packed", "nvdec", "odd"])
@pytest.mark.parametrize("fmt", ["nv12", "rgb24", "gray8"])
def test_surface_equals_packed_frames(api, oracle, weight_dir, fmt, kind):
    """init_surface + 8 x update_surface == init + update on the packed host frames: results equal, search / template blobs bit-identical,
    the box drawn into the surface's visible pixels exactly as the oracle draws it, and nothing written outside them."""
    st, frame = _frames(fmt)
    W, H = st.spec.width, st.spec.height
    wpath = weights.ensure_weight_file("nano", weight_dir)
    a = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True)
    b = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True)
    box = api.BBox(*st.target_boxes(0)[0])
    f0 = frame(0)
    a.init(f0.copy(), box)
    pf = _pitched(api, fmt, W, H, kind, f0)
    b.init_surface(pf.surface, box)
    assert np.array_equal(a.debug_read(0)["template_blob"], b.debug_read(0)["template_blob"])
    drawn = 0
    for n in range(1, 9):
        fr = frame(n)
        host = fr.copy()
        pf.write(fr)
        ra = a.update_all(host)[0]
        rb = b.update_surface(pf.surface)[0]
        assert ra == rb, (n, ra, rb)
        da, db = a.debug_read(0), b.debug_read(0)
        assert np.array_equal(da["search_blob"], db["search_blob"]), n
        assert np.array_equal(da["template_blob"], db["template_blob"]), n
        want = _draw_box(oracle, fr.copy(), fmt, W, H, rb)
        drawn += int(not np.array_equal(want, fr))
        assert np.array_equal(pf.read(), want), (n, int((pf.read() != want).sum()))
        assert np.array_equal(host, want), n
        assert _outside_visible_intact(pf), n
    assert drawn > 0, "no box was drawn: the overlay check saw nothing"


@pytest.mark.gpu
def test_graph_replays_surfaces_of_different_layouts(api, weight_dir):
    """Plane addresses and pitches travel in the per-frame control block, never in the captured graph: one graph handle alternates
    between two surfaces of different pitch and plane placement every frame, and equals an eager handle and the packed host path."""
    st, frame = _frames("nv12")
    W, H = st.spec.width, st.spec.height
    wpath = weights.ensure_weight_file("nano", weight_dir)
    g = api.VitTrack.new(wpath, W, H, box_overlay=True, use_cuda_graph=True)
    e = api.VitTrack.new(wpath, W, H, box_overlay=True, use_cuda_graph=False)
    p = api.VitTrack.new(wpath, W, H, box_overlay=True)
    box = api.BBox(*st.target_boxes(0)[0])
    f0 = frame(0)
    g_s = [_pitched(api, "nv12", W, H, k, f0) for k in ("nvdec", "odd")]
    e_s = [_pitched(api, "nv12", W, H, k, f0) for k in ("nvdec", "odd")]
    g.init_surface(g_s[1].surface, box)
    e.init_surface(e_s[0].surface, box)
    p.init(f0.copy(), box)
    for n in range(1, 11):
        fr = frame(n)
        k = n % 2
        g_s[k].write(fr)
        e_s[k].write(fr)
        host = fr.copy()
        rg, re_, rp = g.update_surface(g_s[k].surface)[0], e.update_surface(e_s[k].surface)[0], p.update_all(host)[0]
        assert rg == re_ == rp, (n, rg, re_, rp)
        assert np.array_equal(g_s[k].read(), host) and np.array_equal(e_s[k].read(), host), n
        assert _outside_visible_intact(g_s[k]), n
    assert len(g_s[0].surface[0]) == 2 and g_s[0].pitch != g_s[1].pitch


@pytest.mark.gpu
def test_pipelined_submit_surface(api, weight_dir):
    """submit_surface with two frames in flight, then wait == synchronous update_surface."""
    st, frame = _frames("nv12")
    W, H = st.spec.width, st.spec.height
    wpath = weights.ensure_weight_file("nano", weight_dir)
    a = api.VitTrack.new(wpath, W, H, box_overlay=True)
    b = api.VitTrack.new(wpath, W, H, box_overlay=True)
    box = api.BBox(*st.target_boxes(0)[0])
    f0 = frame(0)
    for t in (a, b):
        t.init_surface(_pitched(api, "nv12", W, H, "nvdec", f0).surface, box)
    N = 8
    sa = [_pitched(api, "nv12", W, H, "nvdec" if n % 2 else "odd", frame(n)) for n in range(1, N + 1)]
    sb = [_pitched(api, "nv12", W, H, "nvdec" if n % 2 else "odd", frame(n)) for n in range(1, N + 1)]
    got = []
    a.submit_surface(sa[0].surface)
    for n in range(1, N):
        a.submit_surface(sa[n].surface)
        got.append(a.wait()[0])
    got.append(a.wait()[0])
    for n in range(N):
        want = b.update_surface(sb[n].surface)[0]
        assert got[n] == want, (n, got[n], want)
        assert np.array_equal(sa[n].read(), sb[n].read()), n


@pytest.mark.gpu
def test_mixing_frame_kinds(api, weight_dir):
    """One handle alternates surface frames, pinned host frames (search-window uploads) and update_device frames, and equals a handle fed
    only host frames."""
    import torch

    st, frame = _frames("nv12")
    W, H = st.spec.width, st.spec.height
    wpath = weights.ensure_weight_file("nano", weight_dir)
    m = api.VitTrack.new(wpath, W, H, box_overlay=True, upload_window=True)
    h = api.VitTrack.new(wpath, W, H, box_overlay=True, upload_window=True)
    box = api.BBox(*st.target_boxes(0)[0])
    f0 = frame(0)
    pin_m, pin_h = api.PinnedBuffer(f0.size), api.PinnedBuffer(f0.size)
    pin_h.array[:] = f0
    h.init(pin_h.array, box)
    m.init_surface(_pitched(api, "nv12", W, H, "odd", f0).surface, box)
    for n in range(1, 13):
        fr = frame(n)
        pin_h.array[:] = fr
        rh = h.update(pin_h.array)
        kind = n % 3
        if kind == 0:
            pf = _pitched(api, "nv12", W, H, "nvdec", fr)
            rm = m.update_surface(pf.surface)[0]
            out = pf.read()
        elif kind == 1:
            pin_m.array[:] = fr
            rm = m.update(pin_m.array)
            out = pin_m.array
        else:
            d = torch.from_numpy(fr.copy()).cuda()
            torch.cuda.synchronize()
            rm = m.update_device(d.data_ptr(), fr.size)[0]
            out = d.cpu().numpy()
        assert rm == rh, (n, kind, rm, rh)
        assert np.array_equal(out, pin_h.array), (n, kind)


# ---- stream groups -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 4, 16])
def test_stream_group_of_surfaces(api, weight_dir, G):
    """update_streams_surface on G cfg5 streams whose surfaces differ in pitch and plane placement == update_streams on pinned copies of
    the same frames (search-window uploads): results equal, each surface carries exactly its own stream's overlay, sentinels intact."""
    import gc
    gc.collect()
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    streams = [synth.SyntheticStream(synth.cfg5_stream(i)) for i in range(G)]
    spec = streams[0].spec
    W, H = spec.width, spec.height
    fb = streams[0].frame_bytes()
    gs = api.VitTrack.new(w, W, H, gemm_mode=1, max_targets=G, box_overlay=True)
    gh = api.VitTrack.new(w, W, H, gemm_mode=1, max_targets=G, box_overlay=True, upload_window=True)
    kinds = ("nvdec", "odd", "packed")
    surf = []
    pins = [api.PinnedBuffer(fb) for _ in range(G)]
    for i, st in enumerate(streams):
        f0 = np.ascontiguousarray(st.frame(0)).reshape(-1)
        box = api.BBox(*st.target_boxes(0)[0])
        surf.append(_pitched(api, "nv12", W, H, kinds[i % 3], f0))
        gs.init_surface(surf[i].surface, box, target=i)
        pins[i].array[:] = f0
        gh.init(pins[i].array, box, target=i)
    drawn = 0
    for k in range(1, 4):
        frames = [np.ascontiguousarray(st.frame(k)).reshape(-1) for st in streams]
        for i in range(G):
            surf[i].write(frames[i])
            pins[i].array[:] = frames[i]
        got = gs.update_streams_surface([s.surface for s in surf])
        want = gh.update_streams([p.array for p in pins])
        assert got == want, (k, got, want)
        for i in range(G):
            assert np.array_equal(surf[i].read(), pins[i].array), (k, i, "overlay pixels differ")
            assert _outside_visible_intact(surf[i]), (k, i)
            drawn += int(not np.array_equal(pins[i].array, frames[i]))
    assert drawn > 0, "no overlay was drawn"
    gs.close()
    gh.close()
    for p in pins:
        p.close()


# ---- validation --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_surface_argument_errors(api, weight_dir):
    """Every rejected surface call returns VT_ERR_INVALID (template window outside the frame: VT_ERR_CROP_OUTSIDE, as vt_tracker_init),
    and the handle tracks exactly as an untouched one afterwards."""
    from gstreamer_vit_tracker_b200 import _lib

    st, frame = _frames("nv12")
    W, H = st.spec.width, st.spec.height
    wpath = weights.ensure_weight_file("nano", weight_dir)
    t = api.VitTrack.new(wpath, W, H, max_targets=2)
    ref = api.VitTrack.new(wpath, W, H, max_targets=2)
    box = api.BBox(*st.target_boxes(0)[0])
    f0 = frame(0)
    good = _pitched(api, "nv12", W, H, "nvdec", f0)
    (y, uv), (p0, p1) = good.surface
    host = np.zeros(p0 * H * 2, np.uint8)
    pin = api.PinnedBuffer(p0 * H * 2)

    def status(fn, *a):
        with pytest.raises(api.VtError) as e:
            fn(*a)
        return e.value.status

    bad = [((0, uv), (p0, p1)), ((y, 0), (p0, p1)),                         # null plane
           ((y, uv), (W - 1, p1)), ((y, uv), (p0, W - 1)),                  # pitch below the row
           ((host.ctypes.data, uv), (p0, p1)), ((y, host.ctypes.data), (p0, p1)),          # pageable host memory
           ((pin.array.ctypes.data, uv), (p0, p1))]                          # pinned host memory
    L = _lib.lib()
    res = (_lib.vt_result * 2)()
    assert L.vt_tracker_init_surface(t._h, 0, None, box._c()) == _lib.VT_ERR_INVALID
    for s in bad:
        assert status(t.init_surface, s, box) == _lib.VT_ERR_INVALID, s
        assert L.vt_last_error()
    assert status(t.init_surface, good.surface, api.BBox(5000, 5000, 40, 40)) == _lib.VT_ERR_CROP_OUTSIDE
    t.init_surface(good.surface, box)
    ref.init(f0.copy(), box)
    assert L.vt_tracker_update_surface(t._h, None, res) == _lib.VT_ERR_INVALID
    assert L.vt_tracker_submit_surface(t._h, None) == _lib.VT_ERR_INVALID
    for s in bad:
        assert status(t.update_surface, s) == _lib.VT_ERR_INVALID, s
        assert status(t.submit_surface, s) == _lib.VT_ERR_INVALID, s
        assert status(t.update_streams_surface, [s]) == _lib.VT_ERR_INVALID, s
    # stream groups: n must equal the number of active targets (1 here), at most 16
    assert status(t.update_streams_surface, [good.surface] * 2) == _lib.VT_ERR_INVALID
    assert status(t.update_streams_surface, [good.surface] * 17) == _lib.VT_ERR_INVALID
    assert status(t.update_streams_surface, []) == _lib.VT_ERR_INVALID
    # synchronous calls with a frame in flight
    fr1 = _pitched(api, "nv12", W, H, "odd", frame(1))
    t.submit_surface(fr1.surface)
    assert status(t.update_surface, good.surface) == _lib.VT_ERR_INVALID
    assert status(t.init_surface, good.surface, box, 1) == _lib.VT_ERR_INVALID
    assert status(t.update_streams_surface, [good.surface]) == _lib.VT_ERR_INVALID
    r1 = t.wait()[0]
    assert r1 == ref.update(frame(1).copy())
    # the handle still tracks as the untouched one
    for n in range(2, 6):
        pf = _pitched(api, "nv12", W, H, "nvdec", frame(n))
        assert t.update_surface(pf.surface)[0] == ref.update(frame(n).copy()), n
    # probe (HUD) handles take packed frames only
    ctx = api.TrackerContext.new(wpath, W, H)
    assert status(ctx.tracker.init_surface, good.surface, box) == _lib.VT_ERR_INVALID
    assert status(ctx.tracker.update_surface, good.surface) == _lib.VT_ERR_INVALID
    assert status(ctx.tracker.submit_surface, good.surface) == _lib.VT_ERR_INVALID
    assert status(ctx.tracker.update_streams_surface, [good.surface]) == _lib.VT_ERR_INVALID
    ctx.close()
    pin.close()
