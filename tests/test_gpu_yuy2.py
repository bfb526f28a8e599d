"""Packed YUY2 frames (VT_FMT_YUY2) tracked natively: the tracker must see exactly the RGB of vto_yuy2_to_rgb(frame), and every overlay
writes only the Y samples (byte 2x of row y) with the NV12 luma semantics.  Every comparison runs once, against handles alive at the
same time (so both sides run the same kernel forms) and against the oracle on the converted frames."""
import dataclasses

import numpy as np
import pytest

from gstreamer_vit_tracker_b200 import synth, weights
from test_gpu_tracker import compare_step, finish_stats, new_stats

pytestmark = pytest.mark.gpu

FILL = 0x5A  # sentinel of every byte outside the visible pixels of a surface
ODD = synth.StreamSpec("odd", 641, 481, 91, [(575, 425, 60, 50, 2, 1)], fmt="rgb24")  # odd W and H, search window over the right / bottom edges


@pytest.fixture(scope="module")
def api(built):
    from gstreamer_vit_tracker_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import oracle as _o
    return _o


class Yuy2Stream:
    """A synthetic stream (synth.SyntheticStream on the RGB composite) delivered as packed YUY2 frames."""

    def __init__(self, spec):
        self.st = synth.SyntheticStream(dataclasses.replace(spec, fmt="rgb24"))
        self.W, self.H = spec.width, spec.height
        self.row = 4 * ((self.W + 1) // 2)
        self.frame_bytes = self.row * self.H

    def frame(self, n):
        return synth.rgb_to_yuy2(self.st.frame_rgb(n))

    def box(self, n=0):
        return self.st.target_boxes(n)[0]


def _geom(name):
    return Yuy2Stream(ODD if name == "odd" else synth.CONFIGS["cfg3"])


def _luma(frame, W, H, draws):
    """The frame as the luma overlays must leave it: `draws(nv12, W, H)` (oracle draw_*_nv12 calls) applied to its Y samples laid out as
    an NV12 Y plane, written back into bytes 0, 2, .. of every row; the U / V bytes and the pad byte of an odd row stay as they were."""
    row = 4 * ((W + 1) // 2)
    out = np.array(frame, np.uint8).reshape(H, row)
    nv = np.zeros(W * H * 3 // 2 + 2, np.uint8)
    nv[:W * H] = out[:, 0:2 * W:2].reshape(-1)
    draws(nv, W, H)
    out[:, 0:2 * W:2] = nv[:W * H].reshape(H, W)
    return out.reshape(-1)


def _boxed(oracle, frame, W, H, r):
    """The oracle's box overlay (rect thickness 3 + crosshair 15, src/pipeline.rs:165-168) for a gated result."""
    if not (r.status == 0 and r.success and r.score > 0.25):
        return np.array(frame)
    x, y, w, h = r.bbox

    def draw(nv, W, H):
        oracle.draw_rect_nv12(nv, W, H, x, y, w, h, 3, 255)
        oracle.draw_crosshair_nv12(nv, W, H, x + w // 2, y + h // 2, 15, 255)
    return _luma(frame, W, H, draw)


def _blobs_equal(trk, ref):
    sb, tb = ref.last_blobs()
    d = trk.debug_read(0)
    return (np.array_equal(np.asarray(d["search_blob"]).reshape(-1), np.asarray(sb).reshape(-1)) and
            np.array_equal(np.asarray(d["template_blob"]).reshape(-1), np.asarray(tb).reshape(-1)))


# ---- parity --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["nano", "tiny"])
def test_teacher_forced_parity_on_converted_frames(api, oracle, weight_dir, model):
    """cfg3 (640x512, a 64x48 target) teacher-forced over 10 frames: the YUY2 handle against the oracle fed vto_yuy2_to_rgb(frame) —
    search / template blobs bit-identical, success equal, boxes equal on decidable frames, |dscore| within the suite's tolerance — and
    an RGB24 handle fed the converted frames returns exactly the YUY2 handle's results."""
    ys = _geom("cfg3")
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file(model, weight_dir)
    y = api.VitTrack.new(wpath, W, H, fmt="yuy2")
    c = api.VitTrack.new(wpath, W, H, fmt="rgb24")
    ref = oracle.VitTrack(wpath, threads=8)
    box = ys.box()
    f0 = ys.frame(0)
    rgb0 = oracle.yuy2_to_rgb(f0, W, H, 8)
    y.init(f0, api.BBox(*box))
    c.init(rgb0, api.BBox(*box))
    ref.init(rgb0, box)
    stats = new_stats()
    frames = 10
    for n in range(1, frames + 1):
        f = ys.frame(n)
        rgb = oracle.yuy2_to_rgb(f, W, H, 8)
        before = ref.rect
        y.set_rect(before)
        c.set_rect(before)
        ry, rc_ = y.update_all(f)[0], c.update_all(rgb)[0]
        rc, ok, score, bb = ref.update(rgb)
        assert rc == 0 and ry.status == 0, n
        assert ry == rc_, (n, ry, rc_)
        assert _blobs_equal(y, ref), n
        assert ry.success == ok, (n, ry, ok, score)
        compare_step(y, ry, ref, before, stats, ("yuy2", model, n))
    finish_stats(f"teacher_forced/{model}/cfg3_yuy2", stats, frames)


@pytest.mark.parametrize("pad_plus1", [False, True], ids=["pad0", "pad_plus1"])
def test_odd_size_edge_target_and_short_buffer(api, oracle, weight_dir, pad_plus1):
    """641x481 (odd W: the last word of a row is half padding; odd H), a target whose search window overhangs the right and bottom
    edges, with and without pad_plus1: blobs bit-identical to the oracle's on the converted frames, results equal to an RGB24 handle's.
    A buffer shorter than a packed frame is an all-black image: the same results as an all-zero RGB24 frame."""
    ys = _geom("odd")
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    y = api.VitTrack.new(wpath, W, H, fmt="yuy2", pad_plus1=pad_plus1)
    c = api.VitTrack.new(wpath, W, H, fmt="rgb24", pad_plus1=pad_plus1)
    ref = oracle.VitTrack(wpath, threads=8)
    ref.set_variant(pad_plus1=pad_plus1)
    box = ys.box()
    f0 = ys.frame(0)
    assert f0.size == 1284 * 481
    rgb0 = oracle.yuy2_to_rgb(f0, W, H, 8)
    y.init(f0, api.BBox(*box))
    c.init(rgb0, api.BBox(*box))
    ref.init(rgb0, box)
    stats = new_stats()
    for n in range(1, 9):
        f = ys.frame(n)
        rgb = oracle.yuy2_to_rgb(f, W, H, 8)
        before = ref.rect
        y.set_rect(before)
        c.set_rect(before)
        ry, rc_ = y.update_all(f)[0], c.update_all(rgb)[0]
        rc, ok, score, bb = ref.update(rgb)
        assert rc == 0 and ry == rc_, (n, ry, rc_)
        assert _blobs_equal(y, ref), n
        compare_step(y, ry, ref, before, stats, ("odd", pad_plus1, n))
    finish_stats(f"teacher_forced/nano/odd641x481_yuy2_pad{int(pad_plus1)}", stats, 8)
    short = np.full(ys.frame_bytes - 5, 180, np.uint8)
    black = np.zeros((H, W, 3), np.uint8)
    y.set_rect(box)
    c.set_rect(box)
    assert y.update_all(short)[0] == c.update_all(black)[0]
    assert np.array_equal(y.debug_read(0)["search_blob"], c.debug_read(0)["search_blob"])


# ---- uploads -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("geom", ["cfg3", "odd"])
def test_window_uploads_equal_whole_frame_updates(api, weight_dir, monkeypatch, geom):
    """upload_window from pinned frames (whole YUY2 words of the search window; any W and H), windows shrunk by 60 px so that the crop
    kernel falls back to the pinned host frame (VT_B200_WINDOW_SHRINK), and pipelined submit / wait on predicted windows: results and
    overlay pixels equal to whole-frame synchronous updates."""
    ys = _geom(geom)
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    n = 8
    frames = [ys.frame(i) for i in range(n)]
    box = api.BBox(*ys.box())
    kw = dict(fmt="yuy2", box_overlay=True, gemm_mode=1)
    ref = api.VitTrack.new(wpath, W, H, upload_window=False, **kw)
    win = api.VitTrack.new(wpath, W, H, upload_window=True, **kw)
    monkeypatch.setenv("VT_B200_WINDOW_SHRINK", "60")
    a = api.VitTrack.new(wpath, W, H, upload_window=True, **kw)
    b = api.VitTrack.new(wpath, W, H, upload_window=True, **kw)
    monkeypatch.delenv("VT_B200_WINDOW_SHRINK")
    pr, pw, pa = (api.PinnedBuffer(ys.frame_bytes) for _ in range(3))
    pins = [api.PinnedBuffer(ys.frame_bytes) for _ in range(n)]
    for t in (ref, win, a, b):
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
        want_px.append(pr.array.copy())
        pins[i].array[:] = frames[i]
    assert win.timing().h2d_bytes - h2d0 < 0.5 * n * ys.frame_bytes  # the windows really are smaller than the frame
    assert a.timing().h2d_bytes - h2d0_a < 0.3 * n * ys.frame_bytes
    assert any(not np.array_equal(want_px[i], frames[i]) for i in range(n)), "no box was drawn"
    got = []
    b.submit(pins[0].array)
    for i in range(1, n):
        b.submit(pins[i].array)
        got.append(b.wait()[0])
    got.append(b.wait()[0])
    assert got == want
    for i in range(n):
        assert np.array_equal(pins[i].array, want_px[i]), i


# ---- overlays ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("geom", ["cfg3", "odd"])
def test_overlays_write_only_y_samples(api, oracle, weight_dir, geom):
    """The box overlay into pinned frames (zero-copy mirror) and pageable frames (row copy-back), and vt_overlay / vt_overlay_current with
    every overlay kind: the Y samples equal the oracle's draw_*_nv12 on the extracted Y plane, every U / V byte and pad byte is unchanged."""
    ys = _geom(geom)
    W, H = ys.W, ys.H
    wpath = weights.ensure_weight_file("nano", weight_dir)
    box = api.BBox(*ys.box())
    pinned = api.VitTrack.new(wpath, W, H, fmt="yuy2", box_overlay=True, upload_window=True)
    pageable = api.VitTrack.new(wpath, W, H, fmt="yuy2", box_overlay=True)
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
        drawn += int(not np.array_equal(want, f))
    assert drawn > 0, "no box was drawn"
    # explicit commands: every kind, boxes over the edges, a dim that is not first in the list
    cmds = [api.overlay_cmd(3, 10, 10, 400, 80, 150), api.overlay_cmd(2, 15, 15, a=2, r=255, text="TRACKING"),
            api.overlay_cmd(2, 15, 65, a=1, r=200, text="conv:0.1ms trk:0.4ms"), api.overlay_cmd(0, W - 50, H - 40, 90, 70, 3, 255),
            api.overlay_cmd(1, W - 5, 30, a=15, r=220), api.overlay_cmd(4, 7, H - 3), api.overlay_cmd(5, 40, 200, W - 1, H - 2),
            api.overlay_cmd(3, 301, 151, 77, 33, 90), api.overlay_cmd(0, -20, -10, 60, 50, 2, 128)]

    def draws(nv, W, H):
        oracle.draw_background_nv12(nv, W, H, 10, 10, 400, 80, 150)
        oracle.draw_text_nv12(nv, W, H, "TRACKING", 15, 15, 2, 255)
        oracle.draw_text_nv12(nv, W, H, "conv:0.1ms trk:0.4ms", 15, 65, 1, 200)
        oracle.draw_rect_nv12(nv, W, H, W - 50, H - 40, 90, 70, 3, 255)
        oracle.draw_crosshair_nv12(nv, W, H, W - 5, 30, 15, 220)
        oracle.draw_cursor_nv12(nv, W, H, 7, H - 3)
        oracle.draw_selection_nv12(nv, W, H, 40, 200, W - 1, H - 2)
        oracle.draw_background_nv12(nv, W, H, 301, 151, 77, 33, 90)
        oracle.draw_rect_nv12(nv, W, H, -20, -10, 60, 50, 2, 128)
    f = ys.frame(3)
    want = _luma(f, W, H, draws)
    d = f.copy()
    pinned.overlay(d, cmds)                            # vt_overlay (uploads the frame)
    assert np.array_equal(d, want), int((d != want).sum())
    cur = api.VitTrack.new(wpath, W, H, fmt="yuy2")   # vt_overlay_current: the device copy of the frame update() just read
    cur.init(f0, box)
    d = f.copy()
    cur.update_all(d)
    cur.overlay(d, cmds, current=True)
    assert np.array_equal(d, want), int((d != want).sum())
    p2 = api.PinnedBuffer(ys.frame_bytes)
    p2.array[:] = f
    pinned.overlay(p2.array, cmds)
    assert np.array_equal(p2.array, want)


# ---- surfaces ------------------------------------------------------------------------------------------------------------------------
def _padding_intact(pf):
    b = pf.buf.cpu().numpy().reshape(pf.height, pf.pitch)
    return bool((b[:, pf.row:] == FILL).all())


@pytest.mark.parametrize("kind", ["packed", "pitch512", "row_plus3"])
def test_surfaces_equal_packed_frames(api, oracle, weight_dir, kind):
    """init_surface / update_surface / submit_surface on YUY2 surfaces (packed; pitch rounded up to 512; pitch = row + 3, unaligned rows:
    the crop kernel's byte loads) == the packed host path: results equal, blobs bit-identical, the box drawn into the Y samples as the
    oracle draws it, U / V bytes unchanged and the sentinel in the row padding intact."""
    ys = _geom("cfg3")
    W, H, row = ys.W, ys.H, ys.row
    pitch = {"packed": row, "pitch512": (row + 511) // 512 * 512, "row_plus3": row + 3}[kind]
    wpath = weights.ensure_weight_file("nano", weight_dir)
    a = api.VitTrack.new(wpath, W, H, fmt="yuy2", box_overlay=True)
    b = api.VitTrack.new(wpath, W, H, fmt="yuy2", box_overlay=True)
    c = api.VitTrack.new(wpath, W, H, fmt="yuy2", box_overlay=True)
    box = api.BBox(*ys.box())
    f0 = ys.frame(0)

    def surf(fr):
        pf = api.PitchedFrame(W, H, fmt="yuy2", pitch=pitch, fill=FILL)
        pf.write(fr)
        return pf
    a.init(f0.copy(), box)
    b.init_surface(surf(f0).surface, box)
    c.init_surface(surf(f0).surface, box)
    assert np.array_equal(a.debug_read(0)["template_blob"], b.debug_read(0)["template_blob"])
    N = 8
    pfs = [surf(ys.frame(n)) for n in range(1, N + 1)]
    want, drawn = [], 0
    for n in range(1, N + 1):
        fr = ys.frame(n)
        host = fr.copy()
        pf = surf(fr)
        ra, rb = a.update_all(host)[0], b.update_surface(pf.surface)[0]
        assert ra == rb, (n, ra, rb)
        da, db = a.debug_read(0), b.debug_read(0)
        assert np.array_equal(da["search_blob"], db["search_blob"]) and np.array_equal(da["template_blob"], db["template_blob"]), n
        px = _boxed(oracle, fr, W, H, rb)
        drawn += int(not np.array_equal(px, fr))
        assert np.array_equal(pf.read(), px) and np.array_equal(host, px), n
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


# ---- stream groups -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src", ["pinned", "surfaces"])
def test_stream_group_of_four(api, weight_dir, src):
    """Four YUY2 streams (1280 rows: where the many-row kernel forms start) stepped together from pinned frames (search-window uploads)
    or from surfaces of different pitches, each against its own single-target handle: boxes equal, scores within 1e-5, each stream's
    frame carries exactly its own overlay."""
    import gc
    gc.collect()
    G = 4
    streams = [Yuy2Stream(synth.StreamSpec(f"y{i}", 640, 512, 3000 + i, [(288, 232, 64, 48, 3, 2)], fmt="rgb24")) for i in range(G)]
    W, H, fb, row = streams[0].W, streams[0].H, streams[0].frame_bytes, streams[0].row
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    kw = dict(fmt="yuy2", gemm_mode=1, box_overlay=True, upload_window=True)
    grp = api.VitTrack.new(w, W, H, max_targets=G, **kw)
    singles = [api.VitTrack.new(w, W, H, **kw) for _ in range(G)]
    pin_s = [api.PinnedBuffer(fb) for _ in range(G)]
    pin_g = [api.PinnedBuffer(fb) for _ in range(G)] if src == "pinned" else None
    pitches = [row, row + 3, 1536, row + 64]
    surfs = [api.PitchedFrame(W, H, fmt="yuy2", pitch=pitches[i], fill=FILL) for i in range(G)] if src == "surfaces" else None
    for i, st in enumerate(streams):
        f0 = st.frame(0)
        box = api.BBox(*st.box())
        if surfs:
            surfs[i].write(f0)
            grp.init_surface(surfs[i].surface, box, target=i)
        else:
            grp.init(f0, box, target=i)
        singles[i].init(f0, box)
    drawn = 0
    for k in range(1, 5):
        frames = [st.frame(k) for st in streams]
        for i in range(G):
            pin_s[i].array[:] = frames[i]
            if surfs:
                surfs[i].write(frames[i])
            else:
                pin_g[i].array[:] = frames[i]
        got = grp.update_streams_surface([s.surface for s in surfs]) if surfs else grp.update_streams([p.array for p in pin_g])
        for i in range(G):
            ref = singles[i].update(pin_s[i].array)
            a = got[i]
            assert a.status == 0 and a.success == ref.success and a.bbox == ref.bbox and abs(a.score - ref.score) < 1e-5, (k, i, a, ref)
            out = surfs[i].read() if surfs else pin_g[i].array
            assert np.array_equal(out, pin_s[i].array), (k, i, "overlay pixels differ")
            if surfs:
                assert _padding_intact(surfs[i]), (k, i)
            drawn += int(not np.array_equal(pin_s[i].array, frames[i]))
    assert drawn > 0, "no overlay was drawn"
    grp.close()
    for t in singles:
        t.close()
    for p in pin_s + (pin_g or []):
        p.close()


# ---- probe ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mem", ["pageable", "pinned", "pinned_window"])
def test_probe_flow_yuy2(api, oracle, weight_dir, mem):
    """vt_context on YUY2 frames through select -> confirm -> track -> lost -> cancel with a pinned HUD text: pinned frames take the
    one-synchronisation path (HUD queued with the frame, mirrored zero-copy), pageable frames the two-step path.  The Y samples equal
    the oracle's luma HUD and box drawn on the Y plane, driven by the oracle TrackerContext on the converted frames; the chroma bytes
    are untouched.  vt_context_run_ring with `pristine` then leaves every frame of a ring byte-identical to its clean copy."""
    ys = _geom("cfg3")
    W, H, fb = ys.W, ys.H, ys.frame_bytes
    wpath = weights.ensure_weight_file("nano", weight_dir)
    g = api.TrackerContext.new(wpath, W, H, fmt="yuy2", upload_window=(mem == "pinned_window"))
    pin = api.PinnedBuffer(fb) if mem != "pageable" else None
    otrk = oracle.VitTrack(wpath, threads=8)
    o = oracle.TrackerContext(otrk, W, H)
    U = api.UserCommand
    names = {U.MoveUp: "up", U.MoveDown: "down", U.MoveLeft: "left", U.MoveRight: "right", U.Confirm: "confirm", U.Cancel: "cancel"}
    hud = ("FPS: 60", "conv:0.1ms trk:0.5ms")
    n = 0

    def load(fr):
        if pin is None:
            return fr.copy()
        pin.array[:] = fr
        return pin.array

    def cmd(c, fast=False):
        g.handle_command(c, fast)
        o.handle_command(names[c], fast)

    def frame():
        nonlocal n
        fr = ys.frame(n)
        n += 1
        got = load(fr)
        g.probe(got, hud)
        bb = o.process_frame(oracle.yuy2_to_rgb(fr, W, H, 8))
        name = o.state_name()
        sel = o.selection
        box = bb if bb is not None else (o.current_bbox if name == "TRACKING" else None)

        def draws(nv, W, H):
            oracle.draw_background_nv12(nv, W, H, 10, 10, 400, 80, 150)
            oracle.draw_text_nv12(nv, W, H, name, 15, 15, 2, 255)
            oracle.draw_text_nv12(nv, W, H, hud[0], 15, 40, 2, 255)
            oracle.draw_text_nv12(nv, W, H, hud[1], 15, 65, 1, 200)
            if name == "TRACKING":
                oracle.draw_text_nv12(nv, W, H, "score: %.0f%%" % (o.current_score * 100.0), 250, 15, 2, 255)
            if name.startswith("SELECT"):
                oracle.draw_cursor_nv12(nv, W, H, sel[0], sel[1])
                oracle.draw_selection_nv12(nv, W, H, sel[2], sel[3], sel[0], sel[1], sel[4] == 1)
            if box is not None:
                oracle.draw_rect_nv12(nv, W, H, box[0], box[1], box[2], box[3], 3, 255)
                oracle.draw_crosshair_nv12(nv, W, H, box[0] + box[2] // 2, box[1] + box[3] // 2, 15, 255)
        want = _luma(fr, W, H, draws)
        assert g.state_name() == name, n
        gb = g.current_bbox
        assert (gb.tuple() if gb else None) == o.current_bbox, n
        assert abs(g.current_score - o.current_score) <= 1e-3, n
        assert np.array_equal(got, want), (n, name, int((got != want).sum()))

    cmd(U.Confirm)
    frame()                                   # start point set -> SELECT END
    cmd(U.MoveRight, True)
    cmd(U.MoveDown, True)
    frame()                                   # selection visible
    cmd(U.Confirm)
    for _ in range(6):                        # init + update on the confirm frame, then tracking
        frame()
    assert g.state_name() == "TRACKING"
    g.tracker.set_rect((-5000, -5000, 20, 20))
    otrk.rect = (-5000, -5000, 20, 20)
    frame()
    assert g.state_name() == "LOST"
    frame()
    cmd(U.Cancel)
    frame()
    assert g.state_name() == "SELECT START"
    g.close()
    # ring replay on clean copies: a context driven to TRACKING, 4 frames of a 3-frame ring through vt_context_run_ring
    r = api.TrackerContext.new(wpath, W, H, fmt="yuy2", upload_window=(mem == "pinned_window"))
    r.handle_command(U.Confirm)
    r.probe(load(ys.frame(0)), hud)
    r.handle_command(U.MoveRight, True)
    r.handle_command(U.MoveDown, True)
    r.handle_command(U.Confirm)
    r.probe(load(ys.frame(1)), hud)
    assert r.state_name() == "TRACKING"
    ring = 3
    clean = np.concatenate([ys.frame(2 + i) for i in range(ring)])
    buf = api.PinnedBuffer(clean.size) if pin is not None else None
    arr = buf.array if buf is not None else clean.copy()
    arr[:] = clean
    r.run_ring(arr.ctypes.data, fb, fb, ring, 0, 4, hud, pristine_ptr=clean.ctypes.data)
    assert np.array_equal(arr, clean), int((arr != clean).sum())
    r.close()
