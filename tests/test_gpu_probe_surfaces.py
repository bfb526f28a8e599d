"""The drop-in probe on pitched device surfaces (vt_probe_frame_surface, vt_probe_group_frame_surface): the state machine, HUD, cursor /
selection and box drawn in place into a decoder-like surface.  Every comparison is between handles alive at the same time, so both sides run
the same kernel forms: a context (or group) probing surfaces must match one probing the same frames in pinned host memory — state, box, lost
frames, score and the visible pixels after every step — and nothing outside plane 0's visible pixels may be written."""
import hashlib

import numpy as np
import pytest

from gstreamer_vit_tracker_b200 import weights
from test_gpu_probe_groups import HUD, Cam, select_script

pytestmark = pytest.mark.gpu

FILL = 0x5A  # sentinel of every byte outside the visible pixels


@pytest.fixture(scope="module")
def api(built):
    from gstreamer_vit_tracker_b200 import api as _api
    return _api


def _layout(kind, fmt, W, H):
    """packed; "nvdec": pitch a multiple of 512 bytes, NV12 chroma after the surface height rounded to 32 rows; "odd": pitch = row + 3
    (unaligned rows: the background dim's bytewise path), NV12 chroma in an allocation of its own"""
    row = 4 * ((W + 1) // 2) if fmt == "yuy2" else W * (3 if fmt == "rgb24" else 1)
    if kind == "packed":
        return dict(pitch=row)
    if kind == "nvdec":
        return dict(pitch=(row + 511) // 512 * 512, chroma_row=(H + 31) // 32 * 32)
    return dict(pitch=row + 3, separate_uv=True)


def _surface(api, cam, kind):
    return api.PitchedFrame(cam.W, cam.H, fmt=cam.fmt, fill=FILL, **_layout(kind, cam.fmt, cam.W, cam.H))


def _load(pf, frame):
    """the sentinel into every byte of the surface's allocations, then the frame into the visible pixels"""
    pf.buf.fill_(FILL)
    if pf.uv_buf is not None:
        pf.uv_buf.fill_(FILL)
    pf.write(frame)


def _outside_visible_intact(pf):
    """pitch padding, the gap between the NV12 planes and whatever follows the last plane still hold the sentinel"""
    bufs = [(pf.buf, [(0, pf.height, pf.row)] + ([(pf.uv_offset // pf.pitch, pf.uv_rows, pf.width)] if pf.nv12 and pf.uv_buf is None else []))]
    if pf.uv_buf is not None:
        bufs.append((pf.uv_buf, [(0, pf.uv_rows, pf.width)]))
    for buf, planes in bufs:
        b = buf.cpu().numpy().reshape(-1, pf.pitch)
        mask = np.ones(b.shape, bool)
        for r0, rows, cols in planes:
            mask[r0:r0 + rows, :cols] = False
        if not (b[mask] == FILL).all():
            return False
    return True


def _untouched_outside_plane0(cam, got, frame):
    """the NV12 UV plane and the YUY2 U / V bytes are the frame's own"""
    if cam.fmt == "nv12":
        return np.array_equal(got[cam.W * cam.H:], frame[cam.W * cam.H:])
    if cam.fmt == "yuy2":
        return np.array_equal(got[1::2], frame[1::2])
    return True


def _record(ctx, frame):
    b = ctx.current_bbox
    return (ctx.state_name(), b.tuple() if b else None, int(ctx.lost_frames), float(ctx.current_score), hashlib.sha1(frame.tobytes()).hexdigest())


def _session(api, cam, at=1):
    """cursor moves + confirm, drag (dashed selection), confirm (init + update), >= 10 TRACKING frames, a forced loss at `at + 13`
    (LOST), Cancel at `at + 15`, a fresh selection from `at + 16` on"""
    U = api.UserCommand
    s = select_script(api, cam, at)
    s[at + 15] = [(U.Cancel, False)]
    s.update(select_script(api, cam, at + 16))
    return s, {at + 13: (-5000, -5000, 20, 20)}, at + 20


def _step_ctx(ctx, script, losses, n):
    for cmd, fast in script.get(n, []):
        ctx.handle_command(cmd, fast)
    if n in losses and ctx.state_name() == "TRACKING":
        ctx.tracker.set_rect(losses[n])


SINGLE = [("nv12", 1280, 720, k) for k in ("packed", "nvdec", "odd")] + \
         [(f, 640, 512, k) for f in ("rgb24", "gray8", "yuy2") for k in ("packed", "odd")] + \
         [("gray8", 320, 240, "odd"), ("yuy2", 320, 240, "odd")]  # narrower than the 400 x 80 HUD block: the clipped background


def _cam(fmt, W, H):
    if W == 1280:
        return Cam(fmt, W, H, 1001, (580, 315, 120, 90, 5, 3))
    if W == 640:
        return Cam(fmt, W, H, 1003, (288, 232, 64, 48, 3, 2))
    return Cam(fmt, W, H, 301, (140, 100, 48, 40, 1, 1))


@pytest.mark.parametrize("fmt,W,H,kind", SINGLE, ids=[f"{f}_{w}x{h}_{k}" for f, w, h, k in SINGLE])
def test_single_context_surface_equals_pinned(api, weight_dir, fmt, W, H, kind):
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cam = _cam(fmt, W, H)
    script, losses, steps = _session(api, cam)
    kw = dict(fmt=fmt, gemm_mode=1, upload_window=True)
    a, b = api.TrackerContext.new(wpath, W, H, **kw), api.TrackerContext.new(wpath, W, H, **kw)
    pin, pf = api.PinnedBuffer(cam.nbytes), _surface(api, cam, kind)
    seen = set()
    for n in range(steps):
        for c in (a, b):
            _step_ctx(c, script, losses, n)
        f = cam.frame(n)
        pin.array[:] = f
        _load(pf, f)
        a.probe(pin.array, HUD)
        b.probe_surface(pf.surface, HUD)
        got = pf.read()
        ra, rb = _record(a, pin.array), _record(b, got)
        assert ra[:3] == rb[:3] and abs(ra[3] - rb[3]) <= 1e-6, (n, ra[:4], rb[:4])
        assert ra[4] == rb[4], (n, ra[0], "pixels differ", int((got != pin.array).sum()))
        assert _outside_visible_intact(pf), (n, "a byte outside the visible pixels was written")
        assert _untouched_outside_plane0(cam, got, f), (n, "UV plane / YUY2 chroma written")
        seen.add(ra[0])
    assert {"SELECT START", "SELECT END", "TRACKING", "LOST"} <= seen, seen
    a.close(), b.close(), pin.close()


GROUP = [("nv12", 1280, 720, "nvdec"), ("nv12", 1280, 720, "nvdec"), ("yuy2", 640, 512, "odd"), ("rgb24", 640, 512, "packed")]


def _group_scripts(api, cams):
    """stream 0: selects, tracks, is forced lost at step 8; stream 1: a confirm on the background corner at step 4, then its target;
    stream 2: selects and tracks; stream 3: never selects (HUD and cursor only).  Step 0: no stream in the forward."""
    U = api.UserCommand
    s1 = select_script(api, cams[1], 2, box=(0, 0, 30, 30))
    s1.update(select_script(api, cams[1], 6))
    return [select_script(api, cams[0], 1), s1, select_script(api, cams[2], 1), {3: [(U.MoveLeft, True)], 5: [(U.MoveUp, False)]}], {(8, 0): (-5000, -5000, 20, 20)}


def _step_group(g, scripts, losses, n):
    for i, ctx in enumerate(g.contexts):
        for cmd, fast in scripts[i].get(n, []):
            ctx.handle_command(cmd, fast)
        if (n, i) in losses and ctx.state_name() == "TRACKING":
            g.tracker.set_rect(losses[(n, i)], target=i)


def test_group_surfaces_equal_pinned(api, weight_dir):
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cams = [_cam(f, w, h) for f, w, h, _ in GROUP]
    scripts, losses = _group_scripts(api, cams)
    geo = [(c.W, c.H, c.fmt) for c in cams]
    a = api.ProbeGroup.new(wpath, geo, gemm_mode=1, upload_window=True)
    b = api.ProbeGroup.new(wpath, geo, gemm_mode=1, upload_window=True)
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    pfs = [_surface(api, c, k) for c, (_, _, _, k) in zip(cams, GROUP)]
    seen = [set() for _ in cams]
    for n in range(16):
        _step_group(a, scripts, losses, n)
        _step_group(b, scripts, losses, n)
        for i, c in enumerate(cams):
            pins[i].array[:] = c.frame(n)
            _load(pfs[i], c.frame(n))
        a.probe([p.array for p in pins], HUD)
        b.probe_surfaces([pf.surface for pf in pfs], HUD)
        for i, c in enumerate(cams):
            got = pfs[i].read()
            ra, rb = _record(a.contexts[i], pins[i].array), _record(b.contexts[i], got)
            assert ra[:3] == rb[:3] and abs(ra[3] - rb[3]) <= 1e-6, (n, i, ra[:4], rb[:4])
            assert ra[4] == rb[4], (n, i, ra[0], "pixels differ", int((got != pins[i].array).sum()))
            assert _outside_visible_intact(pfs[i]) and _untouched_outside_plane0(c, got, c.frame(n)), (n, i)
            seen[i].add(ra[0])
    assert "TRACKING" in seen[0] and "LOST" in seen[0], seen[0]
    assert "TRACKING" in seen[2] and seen[3] <= {"SELECT START"}, (seen[2], seen[3])
    a.close(), b.close()
    for p in pins:
        p.close()


def test_mixing_pinned_frames_and_surfaces(api, weight_dir):
    """one context (and one group) alternating pinned frames and surfaces == an all-pinned one"""
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cam = _cam("nv12", 1280, 720)
    script, losses, steps = _session(api, cam)
    a, b = api.TrackerContext.new(wpath, cam.W, cam.H, gemm_mode=1, upload_window=True), api.TrackerContext.new(wpath, cam.W, cam.H, gemm_mode=1, upload_window=True)
    pa, pb, pf = api.PinnedBuffer(cam.nbytes), api.PinnedBuffer(cam.nbytes), _surface(api, cam, "nvdec")
    for n in range(steps):
        for c in (a, b):
            _step_ctx(c, script, losses, n)
        pa.array[:] = cam.frame(n)
        a.probe(pa.array, HUD)
        if n % 2:
            _load(pf, cam.frame(n))
            b.probe_surface(pf.surface, HUD)
            got = pf.read()
        else:
            pb.array[:] = cam.frame(n)
            b.probe(pb.array, HUD)
            got = pb.array
        assert _record(a, pa.array) == _record(b, got), n
    a.close(), b.close(), pa.close(), pb.close()

    cams = [_cam(f, w, h) for f, w, h, _ in GROUP]
    scripts, losses = _group_scripts(api, cams)
    geo = [(c.W, c.H, c.fmt) for c in cams]
    ga, gb = api.ProbeGroup.new(wpath, geo, gemm_mode=1, upload_window=True), api.ProbeGroup.new(wpath, geo, gemm_mode=1, upload_window=True)
    pa = [api.PinnedBuffer(c.nbytes) for c in cams]
    pb = [api.PinnedBuffer(c.nbytes) for c in cams]
    pfs = [_surface(api, c, k) for c, (_, _, _, k) in zip(cams, GROUP)]
    for n in range(12):
        _step_group(ga, scripts, losses, n)
        _step_group(gb, scripts, losses, n)
        for i, c in enumerate(cams):
            pa[i].array[:] = c.frame(n)
            pb[i].array[:] = c.frame(n)
            _load(pfs[i], c.frame(n))
        ga.probe([p.array for p in pa], HUD)
        if n % 2:
            gb.probe_surfaces([pf.surface for pf in pfs], HUD)
            got = [pf.read() for pf in pfs]
        else:
            gb.probe([p.array for p in pb], HUD)
            got = [p.array for p in pb]
        for i in range(len(cams)):
            assert _record(ga.contexts[i], pa[i].array) == _record(gb.contexts[i], got[i]), (n, i)
    ga.close(), gb.close()
    for p in pa + pb:
        p.close()


def test_no_pcie_frame_traffic(api, weight_dir):
    """surface probes upload nothing; each step brings back the result block only (32 bytes per target slot + 8 stage stamps + 2 flags)"""
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cam = _cam("nv12", 1280, 720)
    script, losses, _ = _session(api, cam)
    ctx = api.TrackerContext.new(wpath, cam.W, cam.H, gemm_mode=1, upload_window=True)
    pf = _surface(api, cam, "nvdec")
    block = 32 * 1 + 8 * 8 + 2 * 4
    for n in range(14):
        _step_ctx(ctx, script, {}, n)
        _load(pf, cam.frame(n))
        ctx.probe_surface(pf.surface, HUD)
        t = ctx.tracker.timing()
        assert t.h2d_bytes == 0 and t.d2h_bytes == (n + 1) * block, (n, t.h2d_bytes, t.d2h_bytes)
    assert ctx.state_name() == "TRACKING"
    ctx.close()

    cams = [_cam(f, w, h) for f, w, h, _ in GROUP]
    scripts, _ = _group_scripts(api, cams)
    g = api.ProbeGroup.new(wpath, [(c.W, c.H, c.fmt) for c in cams], gemm_mode=1, upload_window=True)
    pfs = [_surface(api, c, k) for c, (_, _, _, k) in zip(cams, GROUP)]
    block = 32 * len(cams) + 8 * 8 + 2 * 4
    for n in range(8):
        _step_group(g, scripts, {}, n)
        for i, c in enumerate(cams):
            _load(pfs[i], c.frame(n))
        g.probe_surfaces([pf.surface for pf in pfs], HUD)
        t = g.tracker.timing()
        assert t.h2d_bytes == 0 and t.d2h_bytes == (n + 1) * block, (n, t.h2d_bytes, t.d2h_bytes)
    assert g.contexts[0].state_name() == "TRACKING"
    g.close()


def test_surface_errors_leave_the_probe_untouched(api, weight_dir):
    """every refused call is VT_ERR_INVALID with a message, and the context / group then probes exactly as an untouched one"""
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    wpath = weights.ensure_weight_file("nano", weight_dir)

    def refused(fn, *a):
        with pytest.raises(api.VtError) as e:
            fn(*a)
        assert e.value.status == _lib.VT_ERR_INVALID and L.vt_last_error()

    cam = _cam("nv12", 1280, 720)
    script, losses, _ = _session(api, cam)
    e, r = api.TrackerContext.new(wpath, cam.W, cam.H, gemm_mode=1, upload_window=True), api.TrackerContext.new(wpath, cam.W, cam.H, gemm_mode=1, upload_window=True)
    pe, pr = _surface(api, cam, "nvdec"), _surface(api, cam, "nvdec")
    pin = api.PinnedBuffer(pe.buf.numel())
    (y, uv), (p0, p1) = pe.surface
    bad = [((0, uv), (p0, p1)), ((y, 0), (p0, p1)), ((y, uv), (cam.W - 1, p1)), ((y, uv), (p0, cam.W - 1)),
           ((pin.array.ctypes.data, uv), (p0, p1)), ((y, pin.array.ctypes.data), (p0, p1))]
    for n in range(8):
        for c in (e, r):
            _step_ctx(c, script, losses, n)
        if n in (3, 6):  # a pending confirm (SELECT END) and TRACKING: neither may step on a refused call
            for s in bad:
                refused(e.probe_surface, s, HUD)
            assert L.vt_probe_frame_surface(e._h, None, None) == _lib.VT_ERR_INVALID and L.vt_last_error()
        _load(pe, cam.frame(n))
        _load(pr, cam.frame(n))
        e.probe_surface(pe.surface, HUD)
        r.probe_surface(pr.surface, HUD)
        assert _record(e, pe.read()) == _record(r, pr.read()), n
    assert e.state_name() == "TRACKING"
    e.close(), r.close()

    cams = [_cam(f, w, h) for f, w, h, _ in GROUP]
    scripts, losses = _group_scripts(api, cams)
    geo = [(c.W, c.H, c.fmt) for c in cams]
    ge, gr = api.ProbeGroup.new(wpath, geo, gemm_mode=1, upload_window=True), api.ProbeGroup.new(wpath, geo, gemm_mode=1, upload_window=True)
    fe = [_surface(api, c, k) for c, (_, _, _, k) in zip(cams, GROUP)]
    fr = [_surface(api, c, k) for c, (_, _, _, k) in zip(cams, GROUP)]
    for n in range(8):
        _step_group(ge, scripts, losses, n)
        _step_group(gr, scripts, losses, n)
        for i, c in enumerate(cams):
            _load(fe[i], c.frame(n))
            _load(fr[i], c.frame(n))
        s = [pf.surface for pf in fe]
        if n in (3, 5):
            refused(ge.probe_surfaces, s[:3], HUD)                      # n != the group's size
            refused(ge.probe_surfaces, s + [s[0]], HUD)
            refused(ge.probe_surfaces, s[:2] + [s[3], s[2]], HUD)       # a 640x512 YUY2 surface for the RGB24 stream: its pitch is short
            refused(ge.probe_surfaces, [((0, 0), (0, 0))] + s[1:], HUD)
            refused(ge.contexts[0].probe_surface, s[0], HUD)            # a member context
            assert L.vt_probe_group_frame_surface(ge._h, None, 4, None) == _lib.VT_ERR_INVALID and L.vt_last_error()
        ge.probe_surfaces(s, HUD)
        gr.probe_surfaces([pf.surface for pf in fr], HUD)
        for i in range(len(cams)):
            assert _record(ge.contexts[i], fe[i].read()) == _record(gr.contexts[i], fr[i].read()), (n, i)
    ge.close(), gr.close(), pin.close()
