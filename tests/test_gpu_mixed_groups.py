"""Stream groups of mixed cameras (vt_tracker_set_stream_geometry): streams of different sizes and formats stepped through one batched
forward must track exactly as single handles of their own geometries do — boxes, scores, overlays, search blobs — on host frames and
on pitched surfaces, against the oracle, at the frame edges, and through the ring runner; and the geometry rules must be enforced."""
import numpy as np
import pytest

from gstreamer_vit_tracker_b200 import synth, weights

pytestmark = pytest.mark.gpu

FILL = 0x5A


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
    """A synthetic camera: the RGB composite of synth.SyntheticStream (seed, one moving target) delivered as packed frames of `fmt`.
    Odd NV12 sizes are cut out of the NV12 encoding of the next even size (the chroma rows keep W bytes, plus the odd-width pad byte)."""

    def __init__(self, fmt, W, H, seed, target):
        self.fmt, self.W, self.H = fmt, W, H
        self.st = synth.SyntheticStream(synth.StreamSpec(f"{fmt}{W}x{H}", W + (W & 1), H + (H & 1), seed, [target], fmt="rgb24"))
        self.nbytes = frame_bytes(fmt, W, H)

    def box(self, n):
        return self.st.target_boxes(n)[0]

    def rgb(self, oracle, n):
        """the RGB image the tracker sees in frame n (the oracle's input): the oracle's own conversions of the packed frame"""
        f, W, H = self.frame(n), self.W, self.H
        if self.fmt == "nv12":
            return oracle.nv12_to_rgb(f, W, H, 16)
        if self.fmt == "yuy2":
            return oracle.yuy2_to_rgb(f, W, H, 16)
        if self.fmt == "gray8":
            return np.ascontiguousarray(np.repeat(f.reshape(H, W)[..., None], 3, axis=2))
        return np.ascontiguousarray(f.reshape(H, W, 3))

    def frame(self, n):
        rgb = self.st.frame_rgb(n)
        W, H = self.W, self.H
        if self.fmt == "nv12":
            Wp, Hp = W + (W & 1), H + (H & 1)
            full = synth.rgb_to_nv12(rgb)
            y = full[: Wp * Hp].reshape(Hp, Wp)[:H, :W]
            uv = full[Wp * Hp:].reshape(Hp // 2, Wp)[: (H + 1) // 2, :W]
            out = np.concatenate([y.reshape(-1), uv.reshape(-1), np.zeros(W & 1, np.uint8)])
        elif self.fmt == "yuy2":
            out = synth.rgb_to_yuy2(np.ascontiguousarray(rgb[:H, :W]))
        elif self.fmt == "rgb24":
            out = rgb[:H, :W].reshape(-1)
        else:
            p = rgb[:H, :W].astype(np.int32)
            out = np.clip(((66 * p[..., 0] + 129 * p[..., 1] + 25 * p[..., 2] + 128) >> 8) + 16, 0, 255).astype(np.uint8).reshape(-1)
        out = np.ascontiguousarray(out, dtype=np.uint8)
        assert out.size == self.nbytes
        return out


def four_cams():
    return [Cam("nv12", 1920, 1080, synth.cfg5_stream(0).seed, (880, 480, 160, 120, 6, 3)),
            Cam("yuy2", 640, 512, synth.CONFIGS["cfg3"].seed, (288, 232, 64, 48, 3, 2)),
            Cam("rgb24", 1280, 720, 1001, (580, 315, 120, 90, 5, 3)),
            Cam("gray8", 641, 481, 91, (300, 200, 60, 50, 3, 2))]


def odd_cams():
    return [Cam("nv12", 637, 359, 71, (300, 160, 56, 44, 3, -2)), Cam("yuy2", 641, 481, 72, (320, 220, 60, 48, -3, 2))]


def group(api, w, cams, **kw):
    """one handle (cfg geometry = the first camera's) with slot i of camera i's geometry"""
    g = api.VitTrack.new(w, cams[0].W, cams[0].H, fmt=cams[0].fmt, max_targets=len(cams), gemm_mode=1, **kw)
    for i, c in enumerate(cams):
        g.set_stream_geometry(i, c.W, c.H, c.fmt)
        assert g.get_stream_geometry(i) == (c.W, c.H, c.fmt)
    return g


def singles(api, w, cams, **kw):
    return [api.VitTrack.new(w, c.W, c.H, fmt=c.fmt, gemm_mode=1, **kw) for c in cams]


def assert_same(a, b, where):
    assert a.status == b.status and a.success == b.success and a.bbox == b.bbox, (where, a, b)
    assert abs(a.score - b.score) <= 1e-5, (where, a, b)


@pytest.mark.parametrize("upload_window", [True, False], ids=["windows", "whole"])
@pytest.mark.parametrize("case", ["four", "odd"])
def test_mixed_group_equals_single_handles(api, weight_dir, case, upload_window):
    """1080p NV12 + 640x512 YUY2 + 720p RGB24 + 641x481 GRAY8 (and two odd-sized NV12 / YUY2 streams) in one group against one
    single-target handle per stream of that stream's geometry: boxes equal, scores within 1e-5, the pinned frames byte-equal after the
    box overlay, the search blobs bit-identical."""
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    cams = four_cams() if case == "four" else odd_cams()
    kw = dict(box_overlay=True, upload_window=upload_window)
    grp, refs = group(api, w, cams, **kw), singles(api, w, cams, **kw)
    pin_g = [api.PinnedBuffer(c.nbytes) for c in cams]
    pin_s = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        grp.init(c.frame(0), api.BBox(*c.box(0)), target=i)
        refs[i].init(c.frame(0), api.BBox(*c.box(0)))
    drawn = 0
    for k in range(1, 7):
        for i, c in enumerate(cams):
            pin_g[i].array[:] = c.frame(k)
            pin_s[i].array[:] = c.frame(k)
        got = grp.update_streams([p.array for p in pin_g])
        for i, c in enumerate(cams):
            ref = refs[i].update_all(pin_s[i].array)[0]
            assert got[i].status == 0, (k, i, got[i])
            assert_same(got[i], ref, (case, k, i))
            assert np.array_equal(pin_g[i].array, pin_s[i].array), (case, k, i, "overlay pixels differ")
            drawn += not np.array_equal(pin_g[i].array, c.frame(k))
            assert np.array_equal(grp.debug_read(i)["search_blob"], refs[i].debug_read(0)["search_blob"]), (case, k, i, "search blob")
    assert drawn > 0, "no overlay was drawn"
    for t in [grp] + refs:
        t.close()
    for p in pin_g + pin_s:
        p.close()


def test_mixed_group_of_surfaces(api, weight_dir):
    """The same four streams as pitched device surfaces — padded pitches, the NV12 chroma behind its own pointer, an unaligned YUY2
    pitch — give the results and overlays of the host-frame mixed group, and nothing outside each stream's plane 0 is written."""
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    cams = four_cams()
    host = group(api, w, cams, box_overlay=True, upload_window=True)
    dev = group(api, w, cams, box_overlay=True)
    pitches = [2048, 1283, 3904, 700]
    surfs = [api.PitchedFrame(c.W, c.H, fmt=c.fmt, pitch=p, separate_uv=(c.fmt == "nv12"), fill=FILL) for c, p in zip(cams, pitches)]
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        host.init(c.frame(0), api.BBox(*c.box(0)), target=i)
        surfs[i].write(c.frame(0))
        dev.init_surface(surfs[i].surface, api.BBox(*c.box(0)), target=i)
    for k in range(1, 6):
        for i, c in enumerate(cams):
            pins[i].array[:] = c.frame(k)
            surfs[i].write(c.frame(k))
        a = host.update_streams([p.array for p in pins])
        b = dev.update_streams_surface([s.surface for s in surfs])
        for i, c in enumerate(cams):
            assert a[i].status == 0 and a[i] == b[i], (k, i, a[i], b[i])
            got = surfs[i].read()
            assert np.array_equal(got, pins[i].array), (k, i, "surface overlay differs from the host frame's")
            clean = c.frame(k)
            ny = c.H * c.W
            if c.fmt == "nv12":
                assert np.array_equal(got[ny:], clean[ny:]), (k, i, "UV plane written")
            if c.fmt == "yuy2":
                assert np.array_equal(got[1::2], clean[1::2]), (k, i, "YUY2 chroma written")
            s = surfs[i]
            rows = s.buf[: c.H * s.pitch].view(c.H, s.pitch)[:, s.row:].cpu().numpy()
            assert (rows == FILL).all(), (k, i, "pitch padding written")
            if s.uv_buf is not None:
                assert (s.uv_buf.view(s.uv_rows, s.pitch)[:, c.W:].cpu().numpy() == FILL).all(), (k, i, "chroma pitch padding written")
    for t in (host, dev):
        t.close()
    for p in pins:
        p.close()


def test_mixed_group_16_streams_vs_oracle(api, oracle, weight_dir):
    """16 streams, four geometries x 4 (1080p NV12, 640x512 YUY2, 720p RGB24, 640x480 GRAY8), one batched forward of 5120 rows (the
    many-row kernel forms), teacher-forced against one oracle tracker per stream on what that stream's camera delivers: search blobs
    bit-exact, scores within 1e-3, boxes equal off floor ties."""
    from test_gpu_tracker import compare_step, new_stats

    geo = [("nv12", 1920, 1080, (880, 480, 160, 120, 6, 3)), ("yuy2", 640, 512, (288, 232, 64, 48, 3, 2)),
           ("rgb24", 1280, 720, (580, 315, 120, 90, 5, 3)), ("gray8", 640, 480, (280, 200, 64, 48, -3, 2))]
    cams = [Cam(f, W, H, 4000 + 4 * j + r, t) for j, (f, W, H, t) in enumerate(geo) for r in range(4)]
    G = len(cams)
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    trk = group(api, wpath, cams, upload_window=True)
    refs = [oracle.VitTrack(wpath, threads=16) for _ in range(G)]
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        trk.init(c.frame(0), api.BBox(*c.box(0)), target=i)
        assert refs[i].init(c.rgb(oracle, 0), c.box(0)) == 0
    stats = new_stats()
    for n in range(1, 5):
        before = [refs[i].rect for i in range(G)]
        for i, c in enumerate(cams):
            pins[i].array[:] = c.frame(n)
            trk.set_rect(before[i], target=i)
        rs = trk.update_streams([p.array for p in pins])
        for i, c in enumerate(cams):
            assert rs[i].status == 0, (n, i, rs[i])
            assert refs[i].update(c.rgb(oracle, n))[0] == 0
            assert np.array_equal(trk.debug_read(i)["search_blob"], refs[i].last_blobs()[0]), (n, i, c.fmt, "search blob")
            compare_step(trk, rs[i], refs[i], before[i], stats, ("mixed16", n, i), target=i)
    assert stats["ties"] + stats["boundary"] <= 2, stats
    trk.close()
    for p in pins:
        p.close()


@pytest.mark.parametrize("pad_plus1", [False, True], ids=["pad0", "pad1"])
def test_mixed_group_edges(api, weight_dir, pad_plus1):
    """A small stream whose search window overhangs its right and bottom edges matches its single handle (pad_plus1 on and off); a
    target whose window lies entirely outside its own, smaller frame gets VT_ERR_CROP_OUTSIDE for that stream only."""
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    big = Cam("nv12", 1920, 1080, 2000, (880, 480, 160, 120, 6, 3))
    edge = Cam("yuy2", 641, 481, 91, (575, 425, 60, 50, 2, 1))
    cams = [big, edge]
    kw = dict(box_overlay=True, upload_window=True, pad_plus1=pad_plus1)
    grp, refs = group(api, w, cams, **kw), singles(api, w, cams, **kw)
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    pin_s = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        grp.init(c.frame(0), api.BBox(*c.box(0)), target=i)
        refs[i].init(c.frame(0), api.BBox(*c.box(0)))
    for k in range(1, 5):
        for i, c in enumerate(cams):
            pins[i].array[:] = c.frame(k)
            pin_s[i].array[:] = c.frame(k)
        got = grp.update_streams([p.array for p in pins])
        for i in range(2):
            assert_same(got[i], refs[i].update_all(pin_s[i].array)[0], (pad_plus1, k, i))
            assert np.array_equal(pins[i].array, pin_s[i].array), (k, i)
    # a rect far outside the small frame (but inside the big one): only that stream fails
    grp.set_rect((1500, 900, 60, 50), target=1)
    for i, c in enumerate(cams):
        pins[i].array[:] = c.frame(5)
    got = grp.update_streams([p.array for p in pins])
    assert got[1].status == -4, got[1]
    assert got[0].status == 0 and got[0].success, got[0]
    for t in [grp] + refs:
        t.close()
    for p in pins + pin_s:
        p.close()


def test_uniform_group_unchanged(api, weight_dir):
    """Slots explicitly set to the cfg geometry give bit-identical results, overlays and kernel launches per frame to a group never
    touched by the new call; a mixed group launches as many kernels per frame as a uniform group of as many streams."""
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    cams = [Cam("nv12", 1920, 1080, 2000 + i, (880, 480, 160, 120, 6, 3)) for i in range(4)]
    kw = dict(gemm_mode=1, max_targets=4, box_overlay=True, upload_window=True)
    plain = api.VitTrack.new(w, 1920, 1080, **kw)
    touched = api.VitTrack.new(w, 1920, 1080, **kw)
    for i in range(4):
        touched.set_stream_geometry(i, 1920, 1080, "nv12")
    mixed = group(api, w, four_cams(), box_overlay=True, upload_window=True)
    pa, pb = [api.PinnedBuffer(c.nbytes) for c in cams], [api.PinnedBuffer(c.nbytes) for c in cams]
    pm = [api.PinnedBuffer(c.nbytes) for c in four_cams()]
    for i, c in enumerate(cams):
        plain.init(c.frame(0), api.BBox(*c.box(0)), target=i)
        touched.init(c.frame(0), api.BBox(*c.box(0)), target=i)
    for i, c in enumerate(four_cams()):
        mixed.init(c.frame(0), api.BBox(*c.box(0)), target=i)
    for k in range(1, 5):
        for i, c in enumerate(cams):
            pa[i].array[:] = c.frame(k)
            pb[i].array[:] = c.frame(k)
        for i, c in enumerate(four_cams()):
            pm[i].array[:] = c.frame(k)
        l0, l1, l2 = plain.timing().kernel_launches, touched.timing().kernel_launches, mixed.timing().kernel_launches
        a = plain.update_streams([p.array for p in pa])
        b = touched.update_streams([p.array for p in pb])
        mixed.update_streams([p.array for p in pm])
        da, db, dm = plain.timing().kernel_launches - l0, touched.timing().kernel_launches - l1, mixed.timing().kernel_launches - l2
        assert a == b, (k, a, b)
        assert all(np.array_equal(x.array, y.array) for x, y in zip(pa, pb)), k
        assert da == db == dm, (k, da, db, dm)
        for i in range(4):
            assert np.array_equal(plain.debug_read(i)["search_blob"], touched.debug_read(i)["search_blob"]), (k, i)
    for t in (plain, touched, mixed):
        t.close()
    for p in pa + pb + pm:
        p.close()


def test_mixed_ring_runner(api, weight_dir):
    """run_streams_ring over a mixed group with pristine copies: every ring ends equal to its pristine copy, and the last results
    equal those of stepping update_streams by hand."""
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    cams = four_cams()
    ring, n = 3, 5
    stride = max(c.nbytes for c in cams)
    a = group(api, w, cams, box_overlay=True, upload_window=True)
    b = group(api, w, cams, box_overlay=True, upload_window=True)
    rings = [api.PinnedBuffer(stride * ring) for _ in cams]
    clean = [api.PinnedBuffer(stride * ring) for _ in cams]
    for i, c in enumerate(cams):
        for r in range(ring):
            rings[i].array[r * stride: r * stride + c.nbytes] = c.frame(1 + r)
        clean[i].array[:] = rings[i].array
        a.init(c.frame(0), api.BBox(*c.box(0)), target=i)
        b.init(c.frame(0), api.BBox(*c.box(0)), target=i)
    last, _ = a.run_streams_ring([r._p.value for r in rings], stride, stride, ring, 0, n, [p._p.value for p in clean])
    for i in range(len(cams)):
        assert np.array_equal(rings[i].array, clean[i].array), (i, "ring not restored")
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for s in range(n):
        for i, c in enumerate(cams):
            pins[i].array[:] = c.frame(1 + s % ring)
        ref = b.update_streams([p.array for p in pins])
    assert last == ref, (last, ref)
    # frame_len below the largest stream's frame
    with pytest.raises(Exception):
        a.run_streams_ring([r._p.value for r in rings], stride, cams[1].nbytes, ring, 0, 1)
    for t in (a, b):
        t.close()
    for p in rings + clean + pins:
        p.close()


def test_mixed_geometry_validation(api, weight_dir):
    """Each rule of vt_tracker_set_stream_geometry is VT_ERR_INVALID with a message; NULL restores the cfg behaviour."""
    from gstreamer_vit_tracker_b200 import _lib as L

    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    cams = four_cams()[:2]
    t = group(api, w, cams, upload_window=True)

    def invalid(fn, *a):
        with pytest.raises(L.VtError) as e:
            fn(*a)
        assert e.value.status == L.VT_ERR_INVALID, e.value
        assert L.lib().vt_last_error(), "no message"
        return str(e.value)

    for i, c in enumerate(cams):
        t.init(c.frame(0), api.BBox(*c.box(0)), target=i)
    assert "drop" in invalid(t.set_stream_geometry, 1, 320, 240, "rgb24")
    t.drop(1)
    for bad in [(0, 240, "nv12"), (320, 0, "nv12"), (-4, 240, "gray8")]:
        invalid(t.set_stream_geometry, 1, *bad)
    g = L.vt_stream_geometry(7, 320, 240, 0)
    assert L.lib().vt_tracker_set_stream_geometry(t._h, 1, g) == L.VT_ERR_INVALID
    t.set_stream_geometry(1, cams[1].W, cams[1].H, cams[1].fmt)
    t.init(cams[1].frame(0), api.BBox(*cams[1].box(0)), target=1)
    # single-frame entry points on a mixed handle
    pin = api.PinnedBuffer(cams[0].nbytes)
    pin.array[:] = cams[0].frame(1)
    invalid(t.update_all, pin.array)
    invalid(t.submit, pin.array)
    invalid(t.run_ring, pin._p.value, cams[0].nbytes, cams[0].nbytes, 1, 0, 1, L.VT_RUN_HOST_SYNC)
    invalid(t.overlay, pin.array, [api.overlay_cmd(L.VT_OV_RECT, 10, 10, 20, 20, 2)], True)
    # lens[i] shorter than stream i's frame
    pins = [api.PinnedBuffer(c.nbytes) for c in cams]
    for i, c in enumerate(cams):
        pins[i].array[:] = c.frame(1)
    invalid(t.update_streams, [pins[0].array, pins[1].array[:-1]])
    # a surface pitch below stream i's row bytes
    surfs = [api.PitchedFrame(c.W, c.H, fmt=c.fmt) for c in cams]
    bad = (surfs[1].surface[0], (api.row_bytes("yuy2", cams[1].W) - 2, 0))
    invalid(t.update_streams_surface, [surfs[0].surface, bad])
    assert t.update_streams([p.array for p in pins])[1].status == 0
    # a probe (HUD) handle
    ctx = api.TrackerContext.new(w, 640, 360)
    invalid(ctx.tracker.set_stream_geometry, 0, 320, 240, "nv12")
    ctx.close()
    # NULL: back to the cfg geometry — the single-frame calls work again
    t.drop(1)
    t.set_stream_geometry(1)
    assert t.get_stream_geometry(1) == (cams[0].W, cams[0].H, cams[0].fmt)
    assert t.update_all(pin.array)[0].status == 0
    t.close()
    for p in pins + [pin]:
        p.close()
