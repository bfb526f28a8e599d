"""Planar I420 frames (VT_FMT_I420) tracked natively, in GStreamer's default layout: the tracker must see exactly what it sees for the NV12
frame of the same Y and interleaved chroma (blobs bit-identical), every overlay must write only the Y samples of the W x H image (never
U, V, the Y row padding or the padding row of an odd height), and pitched I420 surfaces are refused."""
import math

import numpy as np
import pytest

from gstreamer_vit_tracker_b200 import synth, weights
from test_gpu_mixed_groups import Cam as MixedCam
from test_gpu_mixed_groups import assert_same, group, singles
from test_gpu_probe_groups import Cam as ProbeCam
from test_gpu_probe_groups import assert_same_runs, run_group, run_singles, select_script
from test_gpu_tracker import compare_step, finish_stats, new_stats

pytestmark = pytest.mark.gpu

HUD = ("FPS: 60", "conv:0.1ms trk:0.5ms")
ODD = synth.StreamSpec("odd", 642, 482, 91, [(575, 425, 60, 50, 2, 1)], fmt="rgb24")  # cut to 641x481: a target over the right / bottom edges


@pytest.fixture(scope="module")
def api(built):
    from gstreamer_vit_tracker_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import oracle as _o
    return _o


def planes(f, W, H):
    """views of the visible Y, U and V samples of a packed I420 frame"""
    s0, s1, uo, vo, _ = synth.i420_layout(W, H)
    cw, ch = (W + 1) // 2, (H + 1) // 2
    f = np.asarray(f, np.uint8).reshape(-1)
    return f[: s0 * H].reshape(H, s0)[:, :W], f[uo:vo].reshape(ch, s1)[:, :cw], f[vo: vo + s1 * ch].reshape(ch, s1)[:, :cw]


def hidden(f, W, H):
    """every byte of an I420 frame that no overlay may write: U, V, the Y row padding and the Y padding row"""
    s0, _, uo, _, _ = synth.i420_layout(W, H)
    f = np.asarray(f, np.uint8).reshape(-1)
    return np.concatenate([f[: s0 * H].reshape(H, s0)[:, W:].reshape(-1), f[s0 * H:]])


def to_nv12(f, W, H):
    """the NV12 frame of the same Y and interleaved chroma, padded to even W / H (edge replicated)"""
    y, u, v = planes(f, W, H)
    W2, H2 = W + (W & 1), H + (H & 1)
    y = np.pad(y, ((0, H2 - H), (0, W2 - W)), mode="edge")
    return np.concatenate([y.reshape(-1), np.stack([u, v], axis=-1).reshape(-1)])


def to_rgb(oracle, f, W, H):
    """what the tracker must see: the padded NV12 frame through oracle.nv12_to_rgb, cropped back to W x H"""
    W2, H2 = W + (W & 1), H + (H & 1)
    return np.ascontiguousarray(oracle.nv12_to_rgb(to_nv12(f, W, H), W2, H2, 8)[:H, :W])


class I420Stream:
    """synth.SyntheticStream's RGB composite cut to W x H and delivered as packed I420 (synth.rgb_to_i420)."""

    def __init__(self, spec, W=None, H=None):
        self.st = synth.SyntheticStream(spec)
        self.W, self.H = W or spec.width, H or spec.height
        self.frame_bytes = synth.i420_layout(self.W, self.H)[4]

    def frame(self, n):
        return synth.rgb_to_i420(np.ascontiguousarray(self.st.frame_rgb(n)[: self.H, : self.W]))

    def box(self, n=0):
        return self.st.target_boxes(n)[0]


def _stream(geom):
    return I420Stream(ODD, 641, 481) if geom == "odd" else I420Stream(synth.CONFIGS["cfg2"])


def _blobs(trk, target=0):
    d = trk.debug_read(target)
    return np.asarray(d["search_blob"]), np.asarray(d["template_blob"])


def _same_blobs(a, b):
    (sa, ta), (sb, tb) = _blobs(a), _blobs(b)
    return np.array_equal(sa, sb) and np.array_equal(ta, tb)


# ---- tracking parity -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model,geom,pad_plus1", [("nano", "1080p", False), ("tiny", "1080p", False), ("nano", "odd", False),
                                                  ("nano", "odd", True)])
def test_parity_with_nv12_and_oracle(api, oracle, weight_dir, model, geom, pad_plus1):
    """Teacher-forced over 10 frames: the I420 handle against an NV12 handle fed the interleaved frames (even sizes: results equal, blobs
    bit-identical) and against the oracle on the converted RGB (blobs bit-identical, compare_step).  641x481 (strides 644 / 324, a Y
    padding row) with an edge target, pad_plus1 on and off.  A buffer shorter than the frame gives the result of an all-zero RGB24 frame."""
    ys = _stream(geom)
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file(model, weight_dir, variant="wild")
    q = api.VitTrack.new(wpath, W, H, fmt="i420", pad_plus1=pad_plus1)
    nv = api.VitTrack.new(wpath, W, H, fmt="nv12", pad_plus1=pad_plus1) if geom != "odd" else None
    ref = oracle.VitTrack(wpath, threads=8)
    ref.set_variant(pad_plus1=pad_plus1)
    box = ys.box()
    f0 = ys.frame(0)
    assert f0.size == ys.frame_bytes
    q.init(f0, api.BBox(*box))
    ref.init(to_rgb(oracle, f0, W, H), box)
    if nv:
        nv.init(to_nv12(f0, W, H), api.BBox(*box))
        assert _same_blobs(q, nv)
    stats = new_stats()
    frames = 10
    for n in range(1, frames + 1):
        f = ys.frame(n)
        rgb = to_rgb(oracle, f, W, H)
        before = ref.rect
        q.set_rect(before)
        rq = q.update_all(f)[0]
        rc, ok, score, bb = ref.update(rgb)
        assert rc == 0 and rq.status == 0, n
        if nv:
            nv.set_rect(before)
            assert rq == nv.update_all(to_nv12(f, W, H))[0], n
            assert _same_blobs(q, nv), n
        sb, tb = ref.last_blobs()
        assert np.array_equal(_blobs(q)[0].reshape(-1), np.asarray(sb).reshape(-1)), n
        assert np.array_equal(_blobs(q)[1].reshape(-1), np.asarray(tb).reshape(-1)), n
        compare_step(q, rq, ref, before, stats, (model, geom, pad_plus1, n))
    finish_stats(f"teacher_forced/{model}/i420_{geom}_pad{int(pad_plus1)}", stats, frames)
    c = api.VitTrack.new(wpath, W, H, fmt="rgb24", pad_plus1=pad_plus1)
    c.init(to_rgb(oracle, f0, W, H), api.BBox(*box))
    q.set_rect(box)
    c.set_rect(box)
    assert q.update_all(np.full(ys.frame_bytes - 1, 180, np.uint8))[0] == c.update_all(np.zeros(3 * W * H, np.uint8))[0]
    assert np.array_equal(_blobs(q)[0], _blobs(c)[0])


# ---- uploads -------------------------------------------------------------------------------------------------------------------------
def search_window(W, H, box):
    """the library's synchronous search window (App. A.1, factor 4), clipped and grown to even coordinates"""
    x, y, w, h = box
    c = int(math.ceil(math.sqrt(w * h) * 4.0))
    wx, wy = x + int((w - c) / 2), y + int((h - c) / 2)
    x0, y0 = max(wx, 0) & ~1, max(wy, 0) & ~1
    x1, y1 = min((min(wx + c, W) + 1) & ~1, W), min((min(wy + c, H) + 1) & ~1, H)
    return x0, y0, x1, y1


def window_bytes(win):
    x0, y0, x1, y1 = win
    return (x1 - x0) * (y1 - y0) + 2 * ((x1 + 1) // 2 - x0 // 2) * ((y1 + 1) // 2 - y0 // 2)


@pytest.mark.parametrize("geom", ["1080p", "odd"])
def test_window_uploads_equal_whole_frame_updates(api, weight_dir, monkeypatch, geom):
    """upload_window from pinned frames (Y window + the U / V blocks under it), windows shrunk by 60 px so that the crop kernel reads the
    rest of all three planes from the pinned host frame (VT_B200_WINDOW_SHRINK), and pipelined submit / wait on predicted windows: results
    and overlay pixels equal to whole-frame synchronous updates; h2d_bytes of the synchronous window handle grows by exactly the Y + U + V
    window bytes of every frame."""
    ys = _stream(geom)
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    n = 8
    frames = [ys.frame(i) for i in range(n)]
    box = api.BBox(*ys.box())
    kw = dict(fmt="i420", box_overlay=True, gemm_mode=1)
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
    rect = box.tuple()
    for i in range(n):
        for p in (pr, pw, pa):
            p.array[:] = frames[i]
        h2d = win.timing().h2d_bytes
        want.append(ref.update(pr.array))
        assert win.update(pw.array) == want[-1], i
        assert win.timing().h2d_bytes - h2d == window_bytes(search_window(W, H, rect)), i
        if want[-1].status == 0 and want[-1].success:
            rect = tuple(want[-1].bbox)
        assert a.update(pa.array) == want[-1], i
        assert np.array_equal(pw.array, pr.array) and np.array_equal(pa.array, pr.array), i
        assert np.array_equal(hidden(pr.array, W, H), hidden(frames[i], W, H)), i
        want_px.append(pr.array.copy())
        pins_p[i].array[:] = frames[i]
        pins_b[i].array[:] = frames[i]
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
def _luma_cmds(api, W, H):
    """every overlay kind, boxes over the edges"""
    return [api.overlay_cmd(3, 10, 10, 400, 80, 150), api.overlay_cmd(2, 15, 15, a=2, r=255, text="TRACKING"),
            api.overlay_cmd(2, 15, 65, a=1, r=200, text="conv:0.1ms trk:0.4ms"), api.overlay_cmd(0, W - 50, H - 40, 90, 70, 3, r=255),
            api.overlay_cmd(1, W - 5, 30, a=15, r=220), api.overlay_cmd(4, 7, H - 3), api.overlay_cmd(5, 40, 200, W - 1, H - 2),
            api.overlay_cmd(3, 301, 151, 77, 33, 90)]


def _luma_draws(oracle, y, W, H):
    d = np.ascontiguousarray(y).reshape(-1).copy()
    oracle.draw_background_nv12(d, W, H, 10, 10, 400, 80, 150)
    oracle.draw_text_nv12(d, W, H, "TRACKING", 15, 15, 2, 255)
    oracle.draw_text_nv12(d, W, H, "conv:0.1ms trk:0.4ms", 15, 65, 1, 200)
    oracle.draw_rect_nv12(d, W, H, W - 50, H - 40, 90, 70, 3, 255)
    oracle.draw_crosshair_nv12(d, W, H, W - 5, 30, 15, 220)
    oracle.draw_cursor_nv12(d, W, H, 7, H - 3)
    oracle.draw_selection_nv12(d, W, H, 40, 200, W - 1, H - 2)
    oracle.draw_background_nv12(d, W, H, 301, 151, 77, 33, 90)
    return d.reshape(H, W)


def _with_y(f, W, H, y):
    out = np.array(f, np.uint8)
    planes(out, W, H)[0][:] = y
    return out


def _boxed(oracle, f, W, H, r):
    """the oracle's luma box overlay (rect thickness 3 + crosshair 15) for a gated result, on the Y plane"""
    if not (r.status == 0 and r.success and r.score > 0.25):
        return np.array(f)
    x, y, w, h = r.bbox
    d = np.ascontiguousarray(planes(f, W, H)[0]).reshape(-1).copy()
    oracle.draw_rect_nv12(d, W, H, x, y, w, h, 3, 255)
    oracle.draw_crosshair_nv12(d, W, H, x + w // 2, y + h // 2, 15, 255)
    return _with_y(f, W, H, d.reshape(H, W))


@pytest.mark.parametrize("geom", ["1080p", "odd"])
def test_overlays_write_y_samples_only(api, oracle, weight_dir, geom):
    """The box overlay into pinned frames (zero-copy mirror) and pageable frames (row copy-back), and vt_overlay / vt_overlay_current with
    every overlay kind: the Y plane equals the oracle's draw_*_nv12 on it; U, V, the Y row padding and the padding row are unchanged."""
    ys = _stream(geom)
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir)
    box = api.BBox(*ys.box())
    pinned = api.VitTrack.new(wpath, W, H, fmt="i420", box_overlay=True, upload_window=True)
    pageable = api.VitTrack.new(wpath, W, H, fmt="i420", box_overlay=True)
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
        want = _boxed(oracle, f, W, H, r1)
        assert np.array_equal(pin.array, want) and np.array_equal(pg, want), (n, int((pin.array != want).sum()), int((pg != want).sum()))
        assert np.array_equal(hidden(pin.array, W, H), hidden(f, W, H)), n
        drawn += int(not np.array_equal(want, f))
    assert drawn > 0, "no box was drawn"
    cmds = _luma_cmds(api, W, H)
    f = ys.frame(3)
    want = _with_y(f, W, H, _luma_draws(oracle, planes(f, W, H)[0], W, H))
    assert not np.array_equal(want, f)
    d = f.copy()
    pinned.overlay(d, cmds)                            # vt_overlay (uploads the frame), pageable
    assert np.array_equal(d, want), int((d != want).sum())
    p2 = api.PinnedBuffer(ys.frame_bytes)
    p2.array[:] = f
    pinned.overlay(p2.array, cmds)                     # pinned
    assert np.array_equal(p2.array, want), int((p2.array != want).sum())
    cur = api.VitTrack.new(wpath, W, H, fmt="i420")    # vt_overlay_current: the device copy of the frame update() just read
    cur.init(f0, box)
    d = f.copy()
    cur.update_all(d)
    cur.overlay(d, cmds, current=True)
    assert np.array_equal(d, want), int((d != want).sum())


# ---- frames in device memory ---------------------------------------------------------------------------------------------------------
def test_device_frames_and_refused_surfaces(api, oracle, weight_dir):
    """update_device, submit_device and vt_tracker_run_ring in both device modes on packed 641x481 I420 device frames equal host frames:
    results equal, the box drawn into the device frame's Y plane only.  Every surface entry point on an I420 handle or slot is
    VT_ERR_INVALID with a message naming I420."""
    import torch

    ys = _stream("odd")
    W, H, fb = ys.W, ys.H, ys.frame_bytes
    wpath = weights.ensure_weight_file("nano", weight_dir)
    box = api.BBox(*ys.box())
    host = api.VitTrack.new(wpath, W, H, fmt="i420", box_overlay=True)
    dev = api.VitTrack.new(wpath, W, H, fmt="i420", box_overlay=True)
    sub = api.VitTrack.new(wpath, W, H, fmt="i420", box_overlay=True)
    f0 = ys.frame(0)
    for t in (host, dev, sub):
        t.init(f0, box)
    N = 6
    frames = [ys.frame(n) for n in range(1, N + 1)]
    bufs = [torch.from_numpy(f).cuda() for f in frames]
    torch.cuda.synchronize()
    want, drawn = [], 0
    for n in range(N):
        h = frames[n].copy()
        rh = host.update_all(h)[0]
        rd = dev.update_device(bufs[n].data_ptr(), fb)[0]
        assert rh == rd, (n, rh, rd)
        got = bufs[n].cpu().numpy()
        assert np.array_equal(got, h) and np.array_equal(got, _boxed(oracle, frames[n], W, H, rh)), n
        assert np.array_equal(hidden(got, W, H), hidden(frames[n], W, H)), n
        drawn += int(not np.array_equal(got, frames[n]))
        want.append(rh)
    assert drawn > 0, "no box was drawn"
    bufs = [torch.from_numpy(f).cuda() for f in frames]
    torch.cuda.synchronize()
    got = []
    sub.submit_device(bufs[0].data_ptr(), fb)
    for n in range(1, N):
        sub.submit_device(bufs[n].data_ptr(), fb)
        got.append(sub.wait()[0])
    got.append(sub.wait()[0])
    assert got == want
    L = api.L
    for mode in (L.VT_RUN_DEVICE_SYNC, L.VT_RUN_DEVICE_PIPELINED):
        ring = torch.from_numpy(np.concatenate(frames)).cuda()
        torch.cuda.synchronize()
        r = api.VitTrack.new(wpath, W, H, fmt="i420", box_overlay=True)
        r.init(f0, box)
        last, _ = r.run_ring(ring.data_ptr(), fb, fb, N, 0, N, mode)
        assert last[0] == want[-1], (mode, last[0], want[-1])
        r.close()
    # surfaces: refused for an I420 handle and for an I420 slot of a stream group
    yb = torch.zeros(fb, dtype=torch.uint8, device="cuda")
    s = ((yb.data_ptr(), yb.data_ptr() + synth.i420_layout(W, H)[2]), (api.row_bytes("i420", W), synth.i420_layout(W, H)[1]))
    calls = [lambda: host.init_surface(s, box), lambda: host.update_surface(s), lambda: host.submit_surface(s)]
    g = api.VitTrack.new(wpath, 640, 512, fmt="nv12", max_targets=2)
    g.set_stream_geometry(1, W, H, "i420")
    nvf = synth.rgb_to_nv12(synth.SyntheticStream(synth.CONFIGS["cfg3"]).frame_rgb(0))
    g.init(nvf, api.BBox(288, 232, 64, 48), target=0)
    g.init(f0, box, target=1)
    nvb = torch.from_numpy(nvf).cuda()
    nvs = ((nvb.data_ptr(), nvb.data_ptr() + 640 * 512), (640, 640))
    calls.append(lambda: g.update_streams_surface([nvs, s]))
    ctx = api.TrackerContext.new(wpath, W, H, fmt="i420")
    calls.append(lambda: ctx.probe_surface(s, HUD))
    pg = api.ProbeGroup.new(wpath, [(640, 512, "nv12"), (W, H, "i420")])
    calls.append(lambda: pg.probe_surfaces([nvs, s], HUD))
    for i, call in enumerate(calls):
        with pytest.raises(api.VtError) as e:
            call()
        assert e.value.status == -1 and "I420" in str(e.value), (i, str(e.value))
    for x in (host, dev, sub, g, ctx, pg):
        x.close()


# ---- groups --------------------------------------------------------------------------------------------------------------------------
class GroupCam(MixedCam):
    """test_gpu_mixed_groups.Cam, plus I420 cameras"""

    def __init__(self, fmt, W, H, seed, target):
        super().__init__("rgb24" if fmt == "i420" else fmt, W, H, seed, target)
        self.fmt = fmt
        if fmt == "i420":
            self.nbytes = synth.i420_layout(W, H)[4]

    def frame(self, n):
        if self.fmt != "i420":
            return super().frame(n)
        return synth.rgb_to_i420(np.ascontiguousarray(self.st.frame_rgb(n)[: self.H, : self.W]))


def test_mixed_stream_group_equals_single_handles(api, weight_dir):
    """1080p NV12 + 1080p I420 + 641x481 I420 + 640x512 YUY2 in one stream group on pinned frames (window uploads) against one
    single-target handle per stream of its geometry: boxes equal, scores within 1e-5, the overlaid pixels and the search blobs equal."""
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    cams = [GroupCam("nv12", 1920, 1080, 2000, (880, 480, 160, 120, 6, 3)), GroupCam("i420", 1920, 1080, 2001, (880, 480, 160, 120, -5, 3)),
            GroupCam("i420", 641, 481, 2002, (300, 200, 60, 50, 3, 2)), GroupCam("yuy2", 640, 512, 1003, (288, 232, 64, 48, 3, 2))]
    kw = dict(box_overlay=True, upload_window=True)
    grp = group(api, w, cams, **kw)
    refs = singles(api, w, cams, **kw)
    pin_s = [api.PinnedBuffer(c.nbytes) for c in cams]
    pin_g = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        grp.init(c.frame(0), api.BBox(*c.box(0)), target=i)
        refs[i].init(c.frame(0), api.BBox(*c.box(0)))
    drawn = 0
    for k in range(1, 6):
        for i, c in enumerate(cams):
            pin_s[i].array[:] = c.frame(k)
            pin_g[i].array[:] = c.frame(k)
        got = grp.update_streams([p.array for p in pin_g])
        for i, c in enumerate(cams):
            ref = refs[i].update_all(pin_s[i].array)[0]
            assert got[i].status == 0, (k, i, got[i])
            assert_same(got[i], ref, (k, i))
            assert np.array_equal(pin_g[i].array, pin_s[i].array), (k, i, "overlay pixels differ")
            drawn += not np.array_equal(pin_g[i].array, c.frame(k))
            assert np.array_equal(grp.debug_read(i)["search_blob"], refs[i].debug_read(0)["search_blob"]), (k, i, "search blob")
            if c.fmt == "i420":
                assert np.array_equal(hidden(pin_g[i].array, c.W, c.H), hidden(c.frame(k), c.W, c.H)), (k, i)
    assert drawn > 0, "no overlay was drawn"
    for t in [grp] + refs:
        t.close()
    for p in pin_s + pin_g:
        p.close()


class ProbeGroupCam(ProbeCam):
    """test_gpu_probe_groups.Cam, plus I420 cameras"""

    def __init__(self, fmt, W, H, seed, target):
        super().__init__("rgb24" if fmt == "i420" else fmt, W, H, seed, target)
        self.fmt = fmt
        if fmt == "i420":
            self.nbytes = synth.i420_layout(W, H)[4]

    def frame(self, n):
        if self.fmt != "i420":
            return super().frame(n)
        return synth.rgb_to_i420(np.ascontiguousarray(self.st.frame_rgb(n)))


def test_mixed_probe_group_equals_single_contexts(api, weight_dir):
    """A probe group of 1080p NV12 + 1080p I420 against two single contexts, step by step: state, box, lost frames, score and the pinned
    frame's bytes."""
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    cams = [ProbeGroupCam("nv12", 1920, 1080, 2000, (880, 480, 160, 120, 6, 3)), ProbeGroupCam("i420", 1920, 1080, 2001, (880, 480, 160, 120, -5, 3))]
    scripts = [select_script(api, cams[0], 1), select_script(api, cams[1], 2)]
    a = run_group(api, wpath, cams, scripts, 10)
    b = run_singles(api, wpath, cams, scripts, 10)
    assert "TRACKING" in assert_same_runs(a, b, "nv12+i420")


# ---- probe ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mem", ["pageable", "pinned", "pinned_window"])
def test_probe_flow_equals_nv12_context(api, weight_dir, mem):
    """vt_probe_frame on 1080p I420 frames (pageable, pinned, pinned with window uploads) through select -> confirm -> track -> lost ->
    cancel with a pinned HUD text, against an NV12 context alive at the same time fed the interleaved frames and the same commands: state,
    box and score equal after every frame, the Y plane equal to the NV12 frame's, U and V untouched.  vt_context_run_ring with
    `pristine` then leaves every frame of an I420 ring byte-identical to its clean copy."""
    ys = _stream("1080p")
    W, H, fb = ys.W, ys.H, ys.frame_bytes
    wpath = weights.ensure_weight_file("nano", weight_dir)
    win = mem == "pinned_window"
    g = api.TrackerContext.new(wpath, W, H, fmt="i420", upload_window=win)
    r12 = api.TrackerContext.new(wpath, W, H, fmt="nv12", upload_window=win)
    pin = api.PinnedBuffer(fb) if mem != "pageable" else None
    pin12 = api.PinnedBuffer(W * H * 3 // 2) if mem != "pageable" else None
    U = api.UserCommand
    n = 0
    seen = set()

    def cmd(c, fast=False):
        g.handle_command(c, fast)
        r12.handle_command(c, fast)

    def frame():
        nonlocal n
        fr = ys.frame(n)
        n += 1
        if pin is not None:
            pin.array[:] = fr
            pin12.array[:] = to_nv12(fr, W, H)
            got, got12 = pin.array, pin12.array
        else:
            got, got12 = fr.copy(), to_nv12(fr, W, H)
        g.probe(got, HUD)
        r12.probe(got12, HUD)
        assert g.state_name() == r12.state_name(), n
        gb, rb = g.current_bbox, r12.current_bbox
        assert (gb.tuple() if gb else None) == (rb.tuple() if rb else None), n
        assert abs(g.current_score - r12.current_score) <= 1e-5, n
        assert np.array_equal(got[: W * H], got12[: W * H]), (n, g.state_name())
        assert np.array_equal(got[W * H:], fr[W * H:]), n
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
    for c in (g, r12):
        c.tracker.set_rect((-5000, -5000, 20, 20))
    frame()
    assert g.state_name() == "LOST"
    frame()
    cmd(U.Cancel)
    frame()
    assert g.state_name() == "SELECT START" and {"SELECT END", "TRACKING", "LOST"} <= seen
    g.close()
    r12.close()
    if pin is None:
        return
    # ring replay on clean copies: a context driven to TRACKING, 4 frames of a 3-frame ring through vt_context_run_ring
    r = api.TrackerContext.new(wpath, W, H, fmt="i420", upload_window=win)
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
