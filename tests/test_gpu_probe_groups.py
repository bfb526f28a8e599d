"""Probe groups (vt_probe_group_*): n cameras probed in one step — one batched forward over the streams that call VitTrack on that frame,
every stream's HUD drawn in place, one synchronisation.  Each stream must behave exactly like a single TrackerContext of its geometry
that probes the same frames with the same commands: state, box, lost frames, score and the pixels of the pinned frame after every step."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from gstreamer_vit_tracker_b200 import synth, weights

pytestmark = pytest.mark.gpu

HUD = ("FPS: 60", "conv:0.1ms trk:0.5ms")


@pytest.fixture(scope="module")
def api(built):
    from gstreamer_vit_tracker_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import oracle as _o
    return _o


def frame_bytes(fmt, W, H):
    if fmt == "nv12":
        return W * H + (H + 1) // 2 * W + (W & 1)
    return (4 * ((W + 1) // 2) if fmt == "yuy2" else W * (3 if fmt == "rgb24" else 1)) * H


class Cam:
    """A synthetic camera (synth.SyntheticStream, one moving target) delivering packed frames of `fmt` (even sizes)."""

    def __init__(self, fmt, W, H, seed, target):
        self.fmt, self.W, self.H = fmt, W, H
        self.st = synth.SyntheticStream(synth.StreamSpec(f"{fmt}{W}x{H}", W, H, seed, [target], fmt="rgb24"))
        self.nbytes = frame_bytes(fmt, W, H)
        self._cache = {}

    def box(self, n):
        return self.st.target_boxes(n)[0]

    def frame(self, n):
        if n in self._cache:
            return self._cache[n]
        rgb = self.st.frame_rgb(n)
        if self.fmt == "nv12":
            out = synth.rgb_to_nv12(rgb)
        elif self.fmt == "yuy2":
            out = synth.rgb_to_yuy2(np.ascontiguousarray(rgb))
        elif self.fmt == "rgb24":
            out = rgb.reshape(-1)
        else:
            p = rgb.astype(np.int32)
            out = np.clip(((66 * p[..., 0] + 129 * p[..., 1] + 25 * p[..., 2] + 128) >> 8) + 16, 0, 255).astype(np.uint8).reshape(-1)
        out = np.ascontiguousarray(out, dtype=np.uint8).reshape(-1)
        assert out.size == self.nbytes
        if len(self._cache) > 8:
            self._cache.clear()
        self._cache[n] = out
        return out


def _moves(d, neg, pos):
    """cursor moves covering d pixels (fast = 50, slow = 10)"""
    c = neg if d < 0 else pos
    d = abs(d)
    return [(c, True)] * (d // 50) + [(c, False)] * ((d % 50) // 10)


def select_script(api, cam, at, confirm=True, box=None):
    """{step: commands} of a stream that selects `box` (default: its target in frame `at`): cursor to the top-left corner and confirm
    at step `at`, drag to the bottom-right corner at `at + 1` (dashed selection), confirm at `at + 2` (init + update)"""
    U = api.UserCommand
    x, y, w, h = box if box is not None else cam.box(at)
    cx, cy = cam.W // 2, cam.H // 2
    s = {at: _moves(x - cx, U.MoveLeft, U.MoveRight) + _moves(y - cy, U.MoveUp, U.MoveDown) + [(U.Confirm, False)],
         at + 1: _moves(w, U.MoveLeft, U.MoveRight) + _moves(h, U.MoveUp, U.MoveDown)}
    if confirm:
        s[at + 2] = [(U.Confirm, False)]
    return s


def record(ctx, frame):
    b = ctx.current_bbox
    return (ctx.state_name(), b.tuple() if b else None, int(ctx.lost_frames), float(ctx.current_score), hashlib.sha1(frame.tobytes()).hexdigest())


def run_group(api, wpath, cams, scripts, steps, losses=None, kw=None):
    """the group alone (one live handle): per step and stream, (state, box, lost frames, score, frame digest)"""
    kw = dict(gemm_mode=1, upload_window=True, **(kw or {}))
    g = api.ProbeGroup.new(wpath, [(c.W, c.H, c.fmt) for c in cams], **kw)
    assert len(g) == len(cams)
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    out = []
    for n in range(steps):
        for i, c in enumerate(cams):
            for cmd, fast in scripts[i].get(n, []):
                g.contexts[i].handle_command(cmd, fast)
            if losses and (n, i) in losses and g.contexts[i].state_name() == "TRACKING":
                g.tracker.set_rect(losses[(n, i)], target=i)
            pins[i].array[:] = c.frame(n)
        g.probe([p.array for p in pins], HUD)
        out.append([record(g.contexts[i], pins[i].array) for i in range(len(cams))])
    g.close()
    for p in pins:
        p.close()
    return out


def run_singles(api, wpath, cams, scripts, steps, losses=None, kw=None):
    """one TrackerContext per stream, of its geometry, the same frames and commands"""
    kw = dict(gemm_mode=1, upload_window=True, **(kw or {}))
    ctxs = [api.TrackerContext.new(wpath, c.W, c.H, fmt=c.fmt, **kw) for c in cams]
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    out = []
    for n in range(steps):
        rec = []
        for i, c in enumerate(cams):
            for cmd, fast in scripts[i].get(n, []):
                ctxs[i].handle_command(cmd, fast)
            if losses and (n, i) in losses and ctxs[i].state_name() == "TRACKING":
                ctxs[i].tracker.set_rect(losses[(n, i)])
            pins[i].array[:] = c.frame(n)
            ctxs[i].probe(pins[i].array, HUD)
            rec.append(record(ctxs[i], pins[i].array))
        out.append(rec)
    for c in ctxs:
        c.close()
    for p in pins:
        p.close()
    return out


def assert_same_runs(a, b, where):
    seen = set()
    for n, (ra, rb) in enumerate(zip(a, b)):
        for i, (x, y) in enumerate(zip(ra, rb)):
            assert x[:3] == y[:3], (where, n, i, x[:3], y[:3])
            assert abs(x[3] - y[3]) <= 1e-5, (where, n, i, x[3], y[3])
            assert x[4] == y[4], (where, n, i, x[0], "pixels differ")
            seen.add(x[0])
    return seen


def test_group_of_2_equals_single_contexts(api, weight_dir):
    """a uniform group of 2 x 1080p NV12 (one handle: the latency forms) against two single contexts"""
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    cams = [Cam("nv12", 1920, 1080, synth.cfg5_stream(i).seed, (880, 480, 160, 120, 6, 3)) for i in range(2)]
    scripts = [select_script(api, cams[0], 1), select_script(api, cams[1], 3)]
    a = run_group(api, wpath, cams, scripts, 12)
    b = run_singles(api, wpath, cams, scripts, 12)
    assert "TRACKING" in assert_same_runs(a, b, "uniform2")


def test_mixed_group_of_4_equals_single_contexts(api, weight_dir):
    """1080p NV12 + 640x512 YUY2 + 720p RGB24 + 640x480 GRAY8: each stream's HUD in its format's style, throughput forms"""
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    cams = [Cam("nv12", 1920, 1080, 2000, (880, 480, 160, 120, 6, 3)), Cam("yuy2", 640, 512, 1003, (288, 232, 64, 48, 3, 2)),
            Cam("rgb24", 1280, 720, 1001, (580, 315, 120, 90, 5, 3)), Cam("gray8", 640, 480, 91, (300, 200, 60, 50, 3, 2))]
    scripts = [select_script(api, c, 1 + i % 2) for i, c in enumerate(cams)]
    a = run_group(api, wpath, cams, scripts, 10)
    b = run_singles(api, wpath, cams, scripts, 10)
    assert "TRACKING" in assert_same_runs(a, b, "mixed4")


def test_group_of_16_equals_single_contexts(api, weight_dir):
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    cams = [Cam("nv12", 1920, 1080, synth.cfg5_stream(i).seed, (880, 480, 160, 120, 6, 3)) for i in range(16)]
    scripts = [select_script(api, c, 1 + i % 3) for i, c in enumerate(cams)]
    a = run_group(api, wpath, cams, scripts, 8)
    b = run_singles(api, wpath, cams, scripts, 8)
    assert "TRACKING" in assert_same_runs(a, b, "uniform16")


def test_staggered_states_in_one_step(api, weight_dir):
    """Streams in different states in the same steps: SELECT START, SELECT END with a dashed selection, a confirm that passes the gate,
    a confirm on the background, TRACKING, a forced loss -> LOST and the auto-reset 61 lost frames later, Cancel and a fresh init."""
    U = api.UserCommand
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cams = [Cam("nv12" if i % 3 else "gray8", 320, 240, 300 + i, (140, 100, 48, 40, 1, 1)) for i in range(6)]
    steps = 72
    scripts = [
        {20: [(U.Cancel, False)]},                                   # idle: SELECT START (and a Cancel there)
        select_script(api, cams[1], 1, confirm=False),               # SELECT END, dashed selection, forever
        select_script(api, cams[2], 2),                              # confirm -> TRACKING, stays
        select_script(api, cams[3], 1, box=(0, 0, 30, 30)),          # confirm on the background (corner)
        select_script(api, cams[4], 1),                              # TRACKING, forced loss, LOST, auto reset
        select_script(api, cams[5], 1),                              # TRACKING, Cancel, a fresh init later
    ]
    scripts[5][7] = [(U.Cancel, False)]
    scripts[5].update({k + 9: v for k, v in select_script(api, cams[5], 0).items()})
    losses = {(6, 4): (-5000, -5000, 20, 20)}
    a = run_group(api, wpath, cams, scripts, steps, losses)
    b = run_singles(api, wpath, cams, scripts, steps, losses)
    seen = assert_same_runs(a, b, "staggered")
    assert seen >= {"SELECT START", "SELECT END", "TRACKING", "LOST"}, seen
    assert a[6][4][0] == "LOST" and a[-1][4][0] == "SELECT START", (a[6][4], a[-1][4])
    assert a[8][5][0] == "SELECT START" and a[-1][1][0] == "SELECT END"
    assert len({r[i][0] for r in a[5:7] for i in range(6)}) >= 3  # different states inside the same steps


def test_group_vs_oracle(api, oracle, weight_dir):
    """4 NV12 streams against one oracle TrackerContext per stream, drawn with the oracle's draw_* functions"""
    U = api.UserCommand
    names = {U.MoveUp: "up", U.MoveDown: "down", U.MoveLeft: "left", U.MoveRight: "right", U.Confirm: "confirm", U.Cancel: "cancel"}
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cams = [Cam("nv12", 1280, 720, 1001 + 7 * i, (580, 315, 120, 90, 5, 3)) for i in range(4)]
    scripts = [select_script(api, c, 1 + i) for i, c in enumerate(cams)]
    g = api.ProbeGroup.new(wpath, [(c.W, c.H, c.fmt) for c in cams], gemm_mode=1, upload_window=True)
    refs = [oracle.TrackerContext(oracle.VitTrack(wpath, threads=8), c.W, c.H) for c in cams]
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for n in range(9):
        for i, c in enumerate(cams):
            for cmd, fast in scripts[i].get(n, []):
                g.contexts[i].handle_command(cmd, fast)
                refs[i].handle_command(names[cmd], fast)
            pins[i].array[:] = c.frame(n)
        g.probe([p.array for p in pins], HUD)
        for i, c in enumerate(cams):
            W, H, fr, o = c.W, c.H, c.frame(n), refs[i]
            bb = o.process_frame(oracle.nv12_to_rgb(fr, W, H, 8))
            ref = fr.copy()
            name = o.state_name()
            oracle.draw_background_nv12(ref, W, H, 10, 10, 400, 80, 150)
            oracle.draw_text_nv12(ref, W, H, name, 15, 15, 2, 255)
            oracle.draw_text_nv12(ref, W, H, HUD[0], 15, 40, 2, 255)
            oracle.draw_text_nv12(ref, W, H, HUD[1], 15, 65, 1, 200)
            if name == "TRACKING":
                oracle.draw_text_nv12(ref, W, H, "score: %.0f%%" % (o.current_score * 100.0), 250, 15, 2, 255)
            sel = o.selection
            if name.startswith("SELECT"):
                oracle.draw_cursor_nv12(ref, W, H, sel[0], sel[1])
                oracle.draw_selection_nv12(ref, W, H, sel[2], sel[3], sel[0], sel[1], sel[4] == 1)
            box = bb if bb is not None else (o.current_bbox if name == "TRACKING" else None)
            if box is not None:
                oracle.draw_rect_nv12(ref, W, H, box[0], box[1], box[2], box[3], 3, 255)
                oracle.draw_crosshair_nv12(ref, W, H, box[0] + box[2] // 2, box[1] + box[3] // 2, 15, 255)
            ctx = g.contexts[i]
            assert ctx.state_name() == name, (n, i)
            gb = ctx.current_bbox
            assert (gb.tuple() if gb else None) == o.current_bbox, (n, i)
            assert abs(ctx.current_score - o.current_score) <= 1e-3, (n, i)
            assert np.array_equal(pins[i].array, ref), (n, i, name, int((pins[i].array != ref).sum()))
    assert any(c.state_name() == "TRACKING" for c in g.contexts)
    g.close()
    for p in pins:
        p.close()


def test_no_stream_in_the_forward(api, weight_dir):
    """every stream selecting: no forward; the step is the stamp kernel + one overlay kernel, and only the HUD regions are uploaded"""
    U = api.UserCommand
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cams = [Cam("nv12", 640, 360, 50 + i, (280, 150, 80, 60, 2, 1)) for i in range(3)] + [Cam("rgb24", 640, 360, 60, (280, 150, 80, 60, 2, 1))]
    scripts = [{0: [(U.MoveLeft, True)]}, select_script(api, cams[1], 0, confirm=False), {}, {1: [(U.MoveUp, False)]}]
    a = run_group(api, wpath, cams, scripts, 3)
    b = run_singles(api, wpath, cams, scripts, 3)
    assert assert_same_runs(a, b, "selecting") <= {"SELECT START", "SELECT END"}
    g = api.ProbeGroup.new(wpath, [(c.W, c.H, c.fmt) for c in cams], gemm_mode=1, upload_window=True)
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        pins[i].array[:] = c.frame(0)
    t0 = g.tracker.timing()
    g.probe([p.array for p in pins], HUD)
    t1 = g.tracker.timing()
    assert t1.kernel_launches - t0.kernel_launches == 2
    assert t1.h2d_bytes - t0.h2d_bytes == 3 * 400 * 80  # the three NV12 HUD regions (RGB24 draws without reading)
    g.close()


def test_one_forward_and_one_sync_per_step(api, weight_dir):
    """k tracking streams: the step launches what vt_tracker_update_streams with k streams launches on a plain group handle, and uploads
    what that one uploads at the same search windows plus every luma stream's HUD region"""
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    cams = [Cam("nv12", 1280, 720, 1001 + i, (580, 315, 120, 90, 5, 3)) for i in range(4)]
    scripts = [select_script(api, cams[0], 0), select_script(api, cams[1], 0), {}, {}]
    g = api.ProbeGroup.new(wpath, [(c.W, c.H, c.fmt) for c in cams], gemm_mode=1, upload_window=True)
    plain = api.VitTrack.new(wpath, 1280, 720, max_targets=4, gemm_mode=1, upload_window=True)
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for n in range(4):
        for i, c in enumerate(cams):
            for cmd, fast in scripts[i].get(n, []):
                g.contexts[i].handle_command(cmd, fast)
            pins[i].array[:] = c.frame(n)
        g.probe([p.array for p in pins], HUD)
    assert [c.state_name() for c in g.contexts] == ["TRACKING", "TRACKING", "SELECT START", "SELECT START"]
    for i in range(2):
        plain.init(cams[i].frame(3), api.BBox(*cams[i].box(3)), target=i)
    ppins = [api.PinnedBuffer(c.nbytes) for c in cams[:2]]
    for n in range(4, 7):
        for i in range(2):
            plain.set_rect(g.tracker.get_rect(i), target=i)  # the same search windows
            ppins[i].array[:] = cams[i].frame(n)
        for i, c in enumerate(cams):
            pins[i].array[:] = c.frame(n)
        p0 = plain.timing()
        plain.update_streams([p.array for p in ppins])
        p1 = plain.timing()
        t0 = g.tracker.timing()
        g.probe([p.array for p in pins], HUD)
        t1 = g.tracker.timing()
        assert t1.kernel_launches - t0.kernel_launches == p1.kernel_launches - p0.kernel_launches, n
        assert t1.h2d_bytes - t0.h2d_bytes == (p1.h2d_bytes - p0.h2d_bytes) + 4 * 400 * 80, n
    g.close()
    plain.close()


def test_ring_runner(api, weight_dir):
    """vt_probe_group_run_ring with pristine rings: the states and results of step-by-step calls, and clean rings afterwards"""
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    cams = [Cam("nv12", 1280, 720, 1001 + i, (580, 315, 120, 90, 5, 3)) for i in range(2)] + [Cam("yuy2", 640, 512, 1003, (288, 232, 64, 48, 3, 2))]
    scripts = [select_script(api, c, 0) for c in cams]
    R, N = 6, 10
    groups = [api.ProbeGroup.new(wpath, [(c.W, c.H, c.fmt) for c in cams], gemm_mode=1, upload_window=True) for _ in range(2)]
    stride = max(c.nbytes for c in cams)
    rings = [api.PinnedBuffer(stride * R) for _ in cams]
    clean = [api.PinnedBuffer(stride * R) for _ in cams]
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        for k in range(R):
            rings[i].array[k * stride: k * stride + c.nbytes] = c.frame(3 + k)
        clean[i].array[:] = rings[i].array
    for n in range(3):  # select and confirm step by step on both groups
        for g in groups:
            for i, c in enumerate(cams):
                for cmd, fast in scripts[i].get(n, []):
                    g.contexts[i].handle_command(cmd, fast)
                pins[i].array[:] = c.frame(n)
            g.probe([p.array for p in pins], HUD)
    lat = groups[0].run_ring([r.array.ctypes.data for r in rings], stride, max(c.nbytes for c in cams), R, 0, N, HUD,
                             [c_.array.ctypes.data for c_ in clean], want_latency=True)
    assert lat.shape == (N,) and (lat > 0).all()
    for i in range(len(cams)):
        assert np.array_equal(rings[i].array, clean[i].array), (i, "ring not restored")
    for n in range(N):
        for i, c in enumerate(cams):
            pins[i].array[:] = c.frame(3 + n % R)
        groups[1].probe([p.array for p in pins], HUD)
    for a, b in zip(groups[0].contexts, groups[1].contexts):
        assert a.state_name() == b.state_name() == "TRACKING"
        assert a.current_bbox == b.current_bbox and abs(a.current_score - b.current_score) <= 1e-6
    for g in groups:
        g.close()


def test_validation(api, weight_dir):
    from gstreamer_vit_tracker_b200 import _lib

    L = _lib.lib()
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cams = [Cam("nv12", 640, 360, 70, (280, 150, 80, 60, 2, 1)), Cam("yuy2", 320, 240, 71, (140, 100, 48, 40, 1, 1))]
    g = api.ProbeGroup.new(wpath, [(c.W, c.H, c.fmt) for c in cams], gemm_mode=1)
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        pins[i].array[:] = c.frame(0)

    def invalid(fn, what):
        with pytest.raises(_lib.VtError) as e:
            fn()
        assert e.value.status == _lib.VT_ERR_INVALID and what in str(e.value), str(e.value)

    invalid(lambda: g.probe([c.frame(0).copy() for c in cams]), "pinned")                      # pageable
    invalid(lambda: g.probe([pins[0].array, pins[1].array[:-2]]), "full frame")                 # short
    ptrs = (C.c_void_p * 2)(pins[0].array.ctypes.data, None)
    lens = (C.c_size_t * 2)(cams[0].nbytes, cams[1].nbytes)
    assert L.vt_probe_group_frame(g._h, ptrs, lens, None) == _lib.VT_ERR_INVALID and b"frame 1" in L.vt_last_error()  # NULL frame
    for n in (0, 17):
        invalid(lambda: api.ProbeGroup.new(wpath, [(640, 360, "nv12")] * n if n else [], gemm_mode=1), "streams")
    with pytest.raises(_lib.VtError):
        api.ProbeGroup(api.make_config(wpath, 640, 360), [(640, 0, "nv12")])
    m = g.contexts[0]
    invalid(lambda: m.probe(pins[0].array), "probe group")
    invalid(lambda: m.process_frame(pins[0].array), "probe group")
    invalid(lambda: m.run_ring(pins[0].array.ctypes.data, cams[0].nbytes, cams[0].nbytes, 1, 0, 1), "probe group")
    invalid(lambda: g.tracker.update_all(pins[0].array), "probe group")
    invalid(lambda: g.tracker.init(pins[0].array, api.BBox(280, 150, 80, 60), target=0), "probe group")
    invalid(lambda: g.tracker.update_streams([pins[0].array]), "probe group")
    invalid(lambda: g.tracker.submit(pins[0].array), "probe group")
    invalid(lambda: g.tracker.run_ring(pins[0].array.ctypes.data, cams[0].nbytes, cams[0].nbytes, 1, 0, 1, 0), "probe group")
    L.vt_context_destroy(m._h)  # does nothing on a member
    g.probe([p.array for p in pins], HUD)
    assert [c.state_name() for c in g.contexts] == ["SELECT START"] * 2
    assert g.tracker.timing().frames == 1
    g.close()
