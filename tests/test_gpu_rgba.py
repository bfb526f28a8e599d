"""32-bit RGBA / BGRA frames (VT_FMT_RGBA, VT_FMT_BGRA) tracked natively: the tracker must see exactly the RGB24 frame of their colour
bytes (bytes 0 1 2, resp. 2 1 0), every overlay must leave those colour bytes as the RGB24 overlay leaves the converted frame, and byte 3
must never be read or written.  Every 4-byte frame here carries a seeded random byte 3; every surface a sentinel outside its pixels."""
import dataclasses

import numpy as np
import pytest

from gstreamer_vit_tracker_b200 import synth, weights
from test_gpu_mixed_groups import Cam as MixedCam
from test_gpu_mixed_groups import assert_same, group, singles
from test_gpu_probe_groups import Cam as ProbeCam
from test_gpu_probe_groups import assert_same_runs, run_group, run_singles, select_script
from test_gpu_tracker import compare_step, finish_stats, new_stats

pytestmark = pytest.mark.gpu

FILL = 0x5A  # sentinel of every byte outside the visible pixels of a surface
ODD = synth.StreamSpec("odd", 641, 481, 91, [(575, 425, 60, 50, 2, 1)], fmt="rgb24")  # odd W and H, search window over the right / bottom edges
RGB32 = ("rgba", "bgra")
HUD = ("FPS: 60", "conv:0.1ms trk:0.5ms")


@pytest.fixture(scope="module")
def api(built):
    from gstreamer_vit_tracker_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import oracle as _o
    return _o


def pad_bytes(seed, n, H, W):
    """byte 3 of every pixel of frame n: seeded noise, so that a kernel that read it (or wrote it) shows"""
    return synth.hash_u8(seed * 7919 + n, (H, W))


def pack(fmt, rgb, pad):
    return synth.rgb_to_rgba(rgb, pad) if fmt == "rgba" else synth.rgb_to_bgra(rgb, pad)


def colour(fmt, frame, W, H):
    """the RGB24 frame (HWC) of a 4-byte frame's colour bytes"""
    p = np.asarray(frame, np.uint8).reshape(H, W, 4)
    return np.ascontiguousarray(p[..., :3] if fmt == "rgba" else p[..., 2::-1])


def byte3(frame, W, H):
    return np.asarray(frame, np.uint8).reshape(H, W, 4)[..., 3]


def remap(fmt, frame, rgb):
    """`frame` with its colour bytes replaced by the RGB24 image `rgb` (byte 3 kept): an RGB24 result mapped back"""
    out = np.array(frame, np.uint8).reshape(rgb.shape[0], rgb.shape[1], 4)
    out[..., :3] = rgb if fmt == "rgba" else rgb[..., ::-1]
    return out.reshape(-1)


class Rgb32Stream:
    """A synthetic stream (synth.SyntheticStream on the RGB composite) delivered as packed 4-byte frames with a random byte 3."""

    def __init__(self, spec, fmt):
        self.st = synth.SyntheticStream(dataclasses.replace(spec, fmt="rgb24"))
        self.fmt, self.W, self.H, self.seed = fmt, spec.width, spec.height, spec.seed
        self.row = 4 * self.W
        self.frame_bytes = self.row * self.H

    def rgb(self, n):
        return np.ascontiguousarray(self.st.frame_rgb(n))

    def frame(self, n):
        return pack(self.fmt, self.rgb(n), pad_bytes(self.seed, n, self.H, self.W))

    def box(self, n=0):
        return self.st.target_boxes(n)[0]


def _geom(name, fmt):
    return Rgb32Stream(ODD if name == "odd" else synth.CONFIGS["cfg3"], fmt)


def _blobs(trk):
    d = trk.debug_read(0)
    return np.asarray(d["search_blob"]), np.asarray(d["template_blob"])


def _same_blobs(a, b):
    (sa, ta), (sb, tb) = _blobs(a), _blobs(b)
    return np.array_equal(sa, sb) and np.array_equal(ta, tb)


# ---- tracking parity -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pad_plus1", [False, True], ids=["pad0", "pad_plus1"])
@pytest.mark.parametrize("geom", ["cfg3", "odd"])
@pytest.mark.parametrize("fmt", RGB32)
def test_parity_with_rgb24_on_converted_frames(api, oracle, weight_dir, fmt, geom, pad_plus1):
    """cfg3 and 641x481 with an edge target, teacher-forced over 8 frames: the 4-byte handle against an RGB24 handle alive at the same
    time fed the converted frames (search / template blobs bit-identical, results equal) and against the oracle on the converted frames
    (compare_step).  A buffer shorter than a packed frame is read as RGB24 reads a short buffer: border everywhere."""
    ys = _geom(geom, fmt)
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    q = api.VitTrack.new(wpath, W, H, fmt=fmt, pad_plus1=pad_plus1)
    c = api.VitTrack.new(wpath, W, H, fmt="rgb24", pad_plus1=pad_plus1)
    ref = oracle.VitTrack(wpath, threads=8)
    ref.set_variant(pad_plus1=pad_plus1)
    box = ys.box()
    f0, rgb0 = ys.frame(0), ys.rgb(0)
    assert f0.size == 4 * W * H and np.array_equal(colour(fmt, f0, W, H), rgb0)
    q.init(f0, api.BBox(*box))
    c.init(rgb0, api.BBox(*box))
    ref.init(rgb0, box)
    assert _same_blobs(q, c)
    stats = new_stats()
    frames = 8
    for n in range(1, frames + 1):
        f, rgb = ys.frame(n), ys.rgb(n)
        before = ref.rect
        q.set_rect(before)
        c.set_rect(before)
        rq, rc_ = q.update_all(f)[0], c.update_all(rgb)[0]
        rc, ok, score, bb = ref.update(rgb)
        assert rc == 0 and rq.status == 0, n
        assert rq == rc_, (n, rq, rc_)
        assert _same_blobs(q, c), n
        sb, tb = ref.last_blobs()
        assert np.array_equal(_blobs(q)[0].reshape(-1), np.asarray(sb).reshape(-1)), n
        assert np.array_equal(_blobs(q)[1].reshape(-1), np.asarray(tb).reshape(-1)), n
        compare_step(q, rq, ref, before, stats, (fmt, geom, pad_plus1, n))
    finish_stats(f"teacher_forced/nano/{geom}_{fmt}_pad{int(pad_plus1)}", stats, frames)
    short32 = np.full(ys.frame_bytes - 5, 180, np.uint8)
    short24 = np.full(3 * W * H - 5, 180, np.uint8)
    q.set_rect(box)
    c.set_rect(box)
    assert q.update_all(short32)[0] == c.update_all(short24)[0]
    assert np.array_equal(_blobs(q)[0], _blobs(c)[0])


# ---- uploads -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("geom", ["cfg3", "odd"])
@pytest.mark.parametrize("fmt", RGB32)
def test_window_uploads_equal_whole_frame_updates(api, weight_dir, monkeypatch, fmt, geom):
    """upload_window from pinned frames (whole 4-byte pixels of the search window; any W and H), windows shrunk by 60 px so that the
    crop kernel falls back to the pinned host frame (VT_B200_WINDOW_SHRINK), and pipelined submit / wait on predicted windows (also
    shrunk): results and overlay pixels equal to whole-frame synchronous updates."""
    ys = _geom(geom, fmt)
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    n = 8
    frames = [ys.frame(i) for i in range(n)]
    box = api.BBox(*ys.box())
    kw = dict(fmt=fmt, box_overlay=True, gemm_mode=1)
    ref = api.VitTrack.new(wpath, W, H, upload_window=False, **kw)
    win = api.VitTrack.new(wpath, W, H, upload_window=True, **kw)
    piped = api.VitTrack.new(wpath, W, H, upload_window=True, **kw)
    monkeypatch.setenv("VT_B200_WINDOW_SHRINK", "60")
    a = api.VitTrack.new(wpath, W, H, upload_window=True, **kw)
    b = api.VitTrack.new(wpath, W, H, upload_window=True, **kw)
    monkeypatch.delenv("VT_B200_WINDOW_SHRINK")
    pr, pw, pa = (api.PinnedBuffer(ys.frame_bytes) for _ in range(3))
    pins_p = [api.PinnedBuffer(ys.frame_bytes) for _ in range(n)]
    pins_b = [api.PinnedBuffer(ys.frame_bytes) for _ in range(n)]
    for t in (ref, win, piped, a, b):
        t.init(frames[0], box)
    want, want_px = [], []
    h2d0, h2d0_a = win.timing().h2d_bytes, a.timing().h2d_bytes
    for i in range(n):
        for p in (pr, pw, pa):
            p.array[:] = frames[i]
        want.append(ref.update(pr.array))
        assert win.update(pw.array) == want[-1], i
        assert a.update(pa.array) == want[-1], i
        assert np.array_equal(pw.array, pr.array) and np.array_equal(pa.array, pr.array), i
        assert np.array_equal(byte3(pr.array, W, H), byte3(frames[i], W, H)), i
        want_px.append(pr.array.copy())
        pins_p[i].array[:] = frames[i]
        pins_b[i].array[:] = frames[i]
    assert win.timing().h2d_bytes - h2d0 < 0.5 * n * ys.frame_bytes  # the windows really are smaller than the frame
    assert a.timing().h2d_bytes - h2d0_a < 0.3 * n * ys.frame_bytes
    assert any(not np.array_equal(want_px[i], frames[i]) for i in range(n)), "no box was drawn"
    for t, pins in ((piped, pins_p), (b, pins_b)):
        got = []
        t.submit(pins[0].array)
        for i in range(1, n):
            t.submit(pins[i].array)
            got.append(t.wait()[0])
        got.append(t.wait()[0])
        assert got == want
        for i in range(n):
            assert np.array_equal(pins[i].array, want_px[i]), i


# ---- overlays ------------------------------------------------------------------------------------------------------------------------
def _rgb_cmds(api, W, H):
    """every overlay kind, boxes over the edges, distinct R / G / B, and a background whose y + h wraps (src/drawing_rgb.rs:45)"""
    return [api.overlay_cmd(3, 10, 10, 400, 80, 150), api.overlay_cmd(2, 15, 15, a=2, r=255, text="TRACKING"),
            api.overlay_cmd(2, 15, 65, a=1, r=200, text="conv:0.1ms trk:0.4ms"),
            api.overlay_cmd(0, W - 50, H - 40, 90, 70, 3, r=255, g=40, b=7), api.overlay_cmd(1, W - 5, 30, a=15, r=220, g=10, b=90),
            api.overlay_cmd(4, 7, H - 3), api.overlay_cmd(5, 40, 200, W - 1, H - 2), api.overlay_cmd(3, 301, 151, 77, 33, 90),
            api.overlay_cmd(0, -20, -10, 60, 50, 2, r=1, g=128, b=250), api.overlay_cmd(3, 100, 5, 50, -10)]


def _rgb_draws(oracle, rgb, W, H):
    d = np.ascontiguousarray(rgb).reshape(-1).copy()
    oracle.draw_background_rgb(d, W, H, 10, 10, 400, 80)
    oracle.draw_text_rgb(d, W, H, "TRACKING", 15, 15, 2, 255)
    oracle.draw_text_rgb(d, W, H, "conv:0.1ms trk:0.4ms", 15, 65, 1, 200)
    oracle.draw_rect_rgb(d, W, H, W - 50, H - 40, 90, 70, 3, (255, 40, 7))
    oracle.draw_crosshair_rgb(d, W, H, W - 5, 30, 15, (220, 10, 90))
    oracle.draw_cursor_rgb(d, W, H, 7, H - 3)
    oracle.draw_selection_rgb(d, W, H, 40, 200, W - 1, H - 2)
    oracle.draw_background_rgb(d, W, H, 301, 151, 77, 33)
    oracle.draw_rect_rgb(d, W, H, -20, -10, 60, 50, 2, (1, 128, 250))
    oracle.draw_background_rgb(d, W, H, 100, 5, 50, -10)
    return d.reshape(H, W, 3)


def _boxed(oracle, fmt, frame, W, H, r):
    """the oracle's RGB box overlay (rect thickness 3 + crosshair 15, green) for a gated result, on the converted frame, mapped back"""
    if not (r.status == 0 and r.success and r.score > 0.25):
        return np.array(frame)
    x, y, w, h = r.bbox
    d = colour(fmt, frame, W, H).reshape(-1).copy()
    oracle.draw_rect_rgb(d, W, H, x, y, w, h, 3, (0, 255, 0))
    oracle.draw_crosshair_rgb(d, W, H, x + w // 2, y + h // 2, 15, (0, 255, 0))
    return remap(fmt, frame, d.reshape(H, W, 3))


@pytest.mark.parametrize("geom", ["cfg3", "odd"])
@pytest.mark.parametrize("fmt", RGB32)
def test_overlays_write_colour_bytes_only(api, oracle, weight_dir, fmt, geom):
    """The box overlay into pinned frames (zero-copy mirror) and pageable frames (row copy-back), and vt_overlay / vt_overlay_current with
    every overlay kind: the colour bytes equal the oracle's draw_*_rgb on the converted frame, byte 3 is unchanged everywhere.  A frame
    shorter than 4 * W * H is VT_ERR_INVALID for vt_overlay[_current]."""
    ys = _geom(geom, fmt)
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir)
    box = api.BBox(*ys.box())
    pinned = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True, upload_window=True)
    pageable = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True)
    pin = api.PinnedBuffer(ys.frame_bytes)
    f0 = ys.frame(0)
    pinned.init(f0, box)
    pageable.init(f0, box)
    drawn = 0
    for n in range(1, 7):
        f = ys.frame(n)
        pin.array[:] = f
        pg = f.copy()
        r1, r2 = pinned.update(pin.array), pageable.update(pg)
        assert r1 == r2, n
        want = _boxed(oracle, fmt, f, W, H, r1)
        assert np.array_equal(pin.array, want) and np.array_equal(pg, want), (n, int((pin.array != want).sum()), int((pg != want).sum()))
        drawn += int(not np.array_equal(want, f))
    assert drawn > 0, "no box was drawn"
    cmds = _rgb_cmds(api, W, H)
    f = ys.frame(3)
    want = remap(fmt, f, _rgb_draws(oracle, ys.rgb(3), W, H))
    assert not np.array_equal(want, f)
    d = f.copy()
    pinned.overlay(d, cmds)                            # vt_overlay (uploads the frame), pageable
    assert np.array_equal(d, want), int((d != want).sum())
    p2 = api.PinnedBuffer(ys.frame_bytes)
    p2.array[:] = f
    pinned.overlay(p2.array, cmds)                     # pinned
    assert np.array_equal(p2.array, want), int((p2.array != want).sum())
    cur = api.VitTrack.new(wpath, W, H, fmt=fmt)       # vt_overlay_current: the device copy of the frame update() just read
    cur.init(f0, box)
    d = f.copy()
    cur.update_all(d)
    cur.overlay(d, cmds, current=True)
    assert np.array_equal(d, want), int((d != want).sum())
    for current, t in ((False, pinned), (True, cur)):
        short = f[:-1].copy()
        with pytest.raises(api.VtError) as e:
            t.overlay(short, cmds, current=current)
        assert e.value.status == -1
        assert np.array_equal(short, f[:-1])


# ---- surfaces ------------------------------------------------------------------------------------------------------------------------
def _padding_intact(pf):
    b = pf.buf.cpu().numpy().reshape(pf.height, pf.pitch)
    return bool((b[:, pf.row:] == FILL).all())


@pytest.mark.parametrize("kind", ["packed", "pitch7936", "row_plus2"])
@pytest.mark.parametrize("fmt", RGB32)
def test_surfaces_equal_pinned_frames(api, oracle, weight_dir, fmt, kind):
    """init_surface / update_surface / submit_surface on 4-byte surfaces (packed cfg3; 1920 px at a pitch of 7936 bytes, as a DeepStream
    RGBA NvBufSurface; pitch = row + 2, unaligned rows: the crop kernel's byte loads) == pinned frames of the same pixels: results equal,
    blobs bit-identical, the box drawn into the colour bytes as the oracle draws it, byte 3 and the sentinel in the row padding intact."""
    if kind == "pitch7936":
        ys = Rgb32Stream(synth.CONFIGS["cfg2"], fmt)
        pitch = 7936
    else:
        ys = _geom("cfg3", fmt)
        pitch = ys.row if kind == "packed" else ys.row + 2
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir)
    a = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True, upload_window=True)
    b = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True)
    c = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True)
    box = api.BBox(*ys.box())
    f0 = ys.frame(0)
    pin = api.PinnedBuffer(ys.frame_bytes)

    def surf(fr):
        pf = api.PitchedFrame(W, H, fmt=fmt, pitch=pitch, fill=FILL)
        pf.write(fr)
        return pf
    pin.array[:] = f0
    a.init(pin.array, box)
    b.init_surface(surf(f0).surface, box)
    c.init_surface(surf(f0).surface, box)
    assert np.array_equal(_blobs(a)[1], _blobs(b)[1])
    N = 6
    pfs = [surf(ys.frame(n)) for n in range(1, N + 1)]
    want, drawn = [], 0
    for n in range(1, N + 1):
        fr = ys.frame(n)
        pin.array[:] = fr
        pf = surf(fr)
        ra, rb = a.update_all(pin.array)[0], b.update_surface(pf.surface)[0]
        assert ra == rb, (n, ra, rb)
        assert _same_blobs(a, b), n
        px = _boxed(oracle, fmt, fr, W, H, rb)
        drawn += int(not np.array_equal(px, fr))
        assert np.array_equal(pf.read(), px) and np.array_equal(pin.array, px), n
        assert _padding_intact(pf), n
        want.append((ra, px))
    assert drawn > 0, "no box was drawn"
    got = []
    c.submit_surface(pfs[0].surface)
    for n in range(1, N):
        c.submit_surface(pfs[n].surface)
        got.append(c.wait()[0])
    got.append(c.wait()[0])
    for n in range(N):
        assert got[n] == want[n][0], (n, got[n], want[n][0])
        assert np.array_equal(pfs[n].read(), want[n][1]) and _padding_intact(pfs[n]), n
    pin.close()


# ---- groups --------------------------------------------------------------------------------------------------------------------------
class GroupCam(MixedCam):
    """test_gpu_mixed_groups.Cam, plus RGBA / BGRA cameras (the RGB composite packed with a random byte 3)"""

    def __init__(self, fmt, W, H, seed, target):
        super().__init__("rgb24" if fmt in RGB32 else fmt, W, H, seed, target)
        self.fmt, self.seed = fmt, seed
        if fmt in RGB32:
            self.nbytes = 4 * W * H

    def frame(self, n):
        if self.fmt not in RGB32:
            return super().frame(n)
        rgb = np.ascontiguousarray(self.st.frame_rgb(n)[: self.H, : self.W])
        return pack(self.fmt, rgb, pad_bytes(self.seed, n, self.H, self.W))


def _mixed_cams():
    return [GroupCam("nv12", 1920, 1080, 2000, (880, 480, 160, 120, 6, 3)), GroupCam("rgba", 1920, 1080, 2001, (880, 480, 160, 120, -5, 3)),
            GroupCam("bgra", 641, 481, 2002, (300, 200, 60, 50, 3, 2)), GroupCam("yuy2", 640, 512, 1003, (288, 232, 64, 48, 3, 2))]


@pytest.mark.parametrize("src", ["pinned", "surfaces"])
def test_mixed_stream_group_equals_single_handles(api, weight_dir, src):
    """1080p NV12 + 1080p RGBA + 641x481 BGRA + 640x512 YUY2 in one stream group, from pinned frames (window uploads) or from surfaces
    (padded and unaligned pitches), against one single-target handle per stream of its geometry: boxes equal, scores within 1e-5, the
    overlaid pixels equal, the search blobs bit-identical, and nothing outside each surface's pixels written."""
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    cams = _mixed_cams()
    kw = dict(box_overlay=True, upload_window=True)
    grp = group(api, w, cams, **kw) if src == "pinned" else group(api, w, cams, box_overlay=True)
    refs = singles(api, w, cams, **kw)
    pin_s = [api.PinnedBuffer(c.nbytes) for c in cams]
    pin_g = [api.PinnedBuffer(c.nbytes) for c in cams] if src == "pinned" else None
    pitches = [2048, 7936, 4 * 641 + 2, 1283]
    surfs = ([api.PitchedFrame(c.W, c.H, fmt=c.fmt, pitch=p, separate_uv=(c.fmt == "nv12"), fill=FILL) for c, p in zip(cams, pitches)]
             if src == "surfaces" else None)
    for i, c in enumerate(cams):
        if surfs:
            surfs[i].write(c.frame(0))
            grp.init_surface(surfs[i].surface, api.BBox(*c.box(0)), target=i)
        else:
            grp.init(c.frame(0), api.BBox(*c.box(0)), target=i)
        refs[i].init(c.frame(0), api.BBox(*c.box(0)))
    drawn = 0
    for k in range(1, 6):
        for i, c in enumerate(cams):
            pin_s[i].array[:] = c.frame(k)
            if surfs:
                surfs[i].write(c.frame(k))
            else:
                pin_g[i].array[:] = c.frame(k)
        got = grp.update_streams_surface([s.surface for s in surfs]) if surfs else grp.update_streams([p.array for p in pin_g])
        for i, c in enumerate(cams):
            ref = refs[i].update_all(pin_s[i].array)[0]
            assert got[i].status == 0, (k, i, got[i])
            assert_same(got[i], ref, (src, k, i))
            out = surfs[i].read() if surfs else pin_g[i].array
            assert np.array_equal(out, pin_s[i].array), (src, k, i, "overlay pixels differ")
            drawn += not np.array_equal(out, c.frame(k))
            assert np.array_equal(grp.debug_read(i)["search_blob"], refs[i].debug_read(0)["search_blob"]), (src, k, i, "search blob")
            if c.fmt in RGB32:
                assert np.array_equal(byte3(out, c.W, c.H), byte3(c.frame(k), c.W, c.H)), (src, k, i, "byte 3 written")
            if surfs:
                s = surfs[i]
                rows = s.buf[: c.H * s.pitch].view(c.H, s.pitch)[:, s.row:].cpu().numpy()
                assert (rows == FILL).all(), (k, i, "pitch padding written")
    assert drawn > 0, "no overlay was drawn"
    for t in [grp] + refs:
        t.close()
    for p in pin_s + (pin_g or []):
        p.close()


class ProbeGroupCam(ProbeCam):
    """test_gpu_probe_groups.Cam, plus RGBA / BGRA cameras"""

    def __init__(self, fmt, W, H, seed, target):
        super().__init__("rgb24" if fmt in RGB32 else fmt, W, H, seed, target)
        self.fmt, self.seed = fmt, seed
        if fmt in RGB32:
            self.nbytes = 4 * W * H

    def frame(self, n):
        if self.fmt not in RGB32:
            return super().frame(n)
        return pack(self.fmt, np.ascontiguousarray(self.st.frame_rgb(n)), pad_bytes(self.seed, n, self.H, self.W))


def test_mixed_probe_group_equals_single_contexts(api, weight_dir):
    """A probe group of 1080p NV12 + 1080p BGRA (the BGRA stream with the RGB HUD) against two single contexts, step by step: state,
    box, lost frames, score and the pinned frame's bytes."""
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    cams = [ProbeGroupCam("nv12", 1920, 1080, 2000, (880, 480, 160, 120, 6, 3)), ProbeGroupCam("bgra", 1920, 1080, 2001, (880, 480, 160, 120, -5, 3))]
    scripts = [select_script(api, cams[0], 1), select_script(api, cams[1], 2)]
    a = run_group(api, wpath, cams, scripts, 10)
    b = run_singles(api, wpath, cams, scripts, 10)
    assert "TRACKING" in assert_same_runs(a, b, "nv12+bgra")


# ---- probe ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mem", ["pinned", "pinned_window", "surface"])
@pytest.mark.parametrize("fmt", RGB32)
def test_probe_flow_equals_rgb24_context(api, weight_dir, fmt, mem):
    """vt_probe_frame on pinned 4-byte frames (whole-frame and window uploads) or vt_probe_frame_surface on padded surfaces, through
    select -> confirm -> track -> lost -> cancel with a pinned HUD text, against an RGB24 context alive at the same time fed the converted
    frames and the same commands: state, box and score equal after every frame, the colour bytes equal the RGB24 frame's (RGB HUD,
    cursor / selection, box), byte 3 and the surface padding untouched.  vt_context_run_ring with `pristine` then leaves every frame of a
    4-byte ring byte-identical to its clean copy."""
    ys = _geom("cfg3", fmt)
    W, H, fb = ys.W, ys.H, ys.frame_bytes
    wpath = weights.ensure_weight_file("nano", weight_dir)
    win = mem == "pinned_window"
    g = api.TrackerContext.new(wpath, W, H, fmt=fmt, upload_window=win)
    r24 = api.TrackerContext.new(wpath, W, H, fmt="rgb24", upload_window=win)
    pin = api.PinnedBuffer(fb)
    pin24 = api.PinnedBuffer(3 * W * H)
    pf = api.PitchedFrame(W, H, fmt=fmt, pitch=4 * W + 256, fill=FILL) if mem == "surface" else None
    U = api.UserCommand
    n = 0
    seen = set()

    def cmd(c, fast=False):
        g.handle_command(c, fast)
        r24.handle_command(c, fast)

    def frame():
        nonlocal n
        fr = ys.frame(n)
        pin24.array[:] = ys.rgb(n).reshape(-1)
        n += 1
        if pf is not None:
            pf.write(fr)
            g.probe_surface(pf.surface, HUD)
            got = pf.read()
            assert _padding_intact(pf), n
        else:
            pin.array[:] = fr
            g.probe(pin.array, HUD)
            got = pin.array
        r24.probe(pin24.array, HUD)
        assert g.state_name() == r24.state_name(), n
        gb, rb = g.current_bbox, r24.current_bbox
        assert (gb.tuple() if gb else None) == (rb.tuple() if rb else None), n
        assert abs(g.current_score - r24.current_score) <= 1e-5, n
        assert np.array_equal(colour(fmt, got, W, H), pin24.array.reshape(H, W, 3)), (n, g.state_name())
        assert np.array_equal(byte3(got, W, H), byte3(fr, W, H)), n
        seen.add(g.state_name())

    cmd(U.Confirm)
    frame()                                   # start point set -> SELECT END
    cmd(U.MoveRight, True)
    cmd(U.MoveDown, True)
    frame()                                   # selection visible
    cmd(U.Confirm)
    for _ in range(6):                        # init + update on the confirm frame, then tracking
        frame()
    assert g.state_name() == "TRACKING"
    for c in (g, r24):
        c.tracker.set_rect((-5000, -5000, 20, 20))
    frame()
    assert g.state_name() == "LOST"
    frame()
    cmd(U.Cancel)
    frame()
    assert g.state_name() == "SELECT START" and {"SELECT END", "TRACKING", "LOST"} <= seen
    g.close()
    r24.close()
    if mem == "surface":
        return
    # ring replay on clean copies: a context driven to TRACKING, 4 frames of a 3-frame ring through vt_context_run_ring
    r = api.TrackerContext.new(wpath, W, H, fmt=fmt, upload_window=win)
    r.handle_command(U.Confirm)
    pin.array[:] = ys.frame(0)
    r.probe(pin.array, HUD)
    r.handle_command(U.MoveRight, True)
    r.handle_command(U.MoveDown, True)
    r.handle_command(U.Confirm)
    pin.array[:] = ys.frame(1)
    r.probe(pin.array, HUD)
    assert r.state_name() == "TRACKING"
    ring = 3
    clean = np.concatenate([ys.frame(2 + i) for i in range(ring)])
    buf = api.PinnedBuffer(clean.size)
    buf.array[:] = clean
    r.run_ring(buf.array.ctypes.data, fb, fb, ring, 0, 4, HUD, pristine_ptr=clean.ctypes.data)
    assert np.array_equal(buf.array, clean), int((buf.array != clean).sum())
    r.close()
