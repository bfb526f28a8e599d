"""GPU parity of the tracker path (crop/convert/resize/normalise -> ViT -> decode) through the C ABI
against the CPU oracle and the cv2.TrackerVit fixtures.

Tolerances (BASELINE.json north_star): NV12 conversion and the u8 preprocessing bit-exact; score within
1e-3 absolute; boxes IoU >= 0.99.  Boxes are floor()s of fp32 expressions scaled by the crop size, so a
relative error e in the size/offset maps moves a pre-floor coordinate by ~e*crop px.  Two kinds of frame are
numerically undecidable and are counted, bounded (<= 3 % of the frames of a sequence, together) and recorded:
  * boundary: an oracle pre-floor coordinate lies within BOUNDARY_PX of an integer -> that coordinate may differ by one pixel;
  * tie: the oracle's hann-weighted top-1/top-2 margin is below TIE_MARGIN -> the GPU may pick another of the tied cells; the
    cell it picked must be one of the oracle's tied maxima and its score / box must equal the oracle's values FOR THAT CELL.
Everything else must match exactly.  The per-test counts go to gpurun_out/parity_stats.json (and are asserted on at the end of
this file), so they survive `pytest -q`."""
import hashlib
import json
import math
import os

import numpy as np
import pytest

from conftest import ROOT, golden
from gstreamer_vit_tracker_b200 import synth, weights

pytestmark = pytest.mark.gpu

SCORE_TOL = 1e-3
IOU_MIN = 0.99
TIE_MARGIN = 1e-4        # fp32 / bf16x3 paths (measured |dscore| ~1e-5): top-1/top-2 margin under which the argmax is undecidable
TIE_MARGIN_FP16 = 2e-3   # single-pass fp16 operands (opt-in mode, |dscore| ~3e-4)
BOUNDARY_PX = 0.02       # distance of a pre-floor coordinate from an integer under which +-1 px is accepted
EXEMPT_FRAC = 0.03       # ties + boundary frames per sequence
THRESHOLD = 0.2

PARITY_STATS = {}        # test id -> stats dict, written to gpurun_out/parity_stats.json by the last test of this file


@pytest.fixture(scope="module")
def api(built):
    from gstreamer_vit_tracker_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def oracle(built):
    from oracle import oracle as _o
    return _o


def iou(a, b):
    ax, ay, aw, ah = a
    bx, by, bw, bh = b
    ix = max(0, min(ax + aw, bx + bw) - max(ax, bx))
    iy = max(0, min(ay + ah, by + bh) - max(ay, by))
    inter = ix * iy
    union = aw * ah + bw * bh - inter
    return inter / union if union > 0 else 1.0


def oracle_prefloor(ref, rect_before, cell=None, decode_window=0):
    """Pre-floor bbox coordinates the oracle's last update gives for map cell `cell` (default: its own argmax), in the fp32
    arithmetic of App. A.6, and the hann-weighted top-1/top-2 margin."""
    cw, sm, om, _ = ref.last_maps()
    best = int(np.argmax(cw)) if cell is None else int(cell)
    my, mx = divmod(best, 16)
    f = np.float32
    cx = (f(mx) + om[best]) / f(16)
    cy = (f(my) + om[256 + best]) / f(16)
    bw, bh = sm[best], sm[256 + best]
    x, y, w, h = rect_before
    c = 4 * int(np.floor(np.sqrt(float(w * h)))) if decode_window else int(np.ceil(np.sqrt(float(w * h)) * 4))  # App. A.7 / A.6
    x0, y0 = x + int((w - c) / 2), y + int((h - c) / 2)
    vals = [(cx - bw / f(2)) * f(c) + f(x0), (cy - bh / f(2)) * f(c) + f(y0), bw * f(c), bh * f(c)]
    srt = np.sort(cw)[::-1]
    return [float(v) for v in vals], float(srt[0] - srt[1])


def compare_step(trk, r, ref, rect_before, stats, where, target=0, tie_margin=TIE_MARGIN, decode_window=0):
    """One step from the same rect_last: GPU result r (target `target` of handle trk) vs the oracle tracker `ref`, which has just
    run update() on the same frame.  Returns True when the step matched exactly."""
    cw = ref.last_maps()[0]
    best = int(np.argmax(cw))
    srt = np.sort(cw)[::-1]
    margin = float(srt[0] - srt[1])
    cell = best
    if margin < tie_margin:  # undecidable argmax: the GPU's cell must be one of the oracle's tied maxima
        stats["ties"] += 1
        cell = int(np.argmax(trk.debug_read(target)["conf_win"]))
        assert cw[cell] >= cw[best] - tie_margin, (where, "argmax outside the oracle's tied set", cell, best, float(cw[cell]), float(cw[best]))
    score = float(cw[cell])
    d = abs(r.score - score)
    stats["max_dscore"] = max(stats["max_dscore"], d)
    assert d <= SCORE_TOL, (where, r.score, score)
    if abs(score - THRESHOLD) > SCORE_TOL:
        assert r.success == (score >= THRESHOLD), where
    if not r.success:
        stats["exact"] += cell == best
        return cell == best
    pre, _ = oracle_prefloor(ref, rect_before, cell, decode_window)
    want = tuple(int(math.floor(v)) for v in pre)
    if tuple(r.bbox) == want:
        stats["exact"] += cell == best
        return cell == best
    near = [abs(v - round(v)) < BOUNDARY_PX for v in pre]
    diff = [abs(a - b) for a, b in zip(r.bbox, want)]
    assert all(dd <= 1 for dd in diff) and all(n for dd, n in zip(diff, near) if dd), (where, r.bbox, want, pre)
    stats["boundary"] += 1
    stats["min_iou_boundary"] = min(stats["min_iou_boundary"], iou(r.bbox, want))
    return False


def new_stats():
    return {"frames": 0, "exact": 0, "boundary": 0, "ties": 0, "max_dscore": 0.0, "min_iou_boundary": 1.0}


def finish_stats(name, stats, frames):
    """Bounds of a teacher-forced sequence + the record that survives `pytest -q`."""
    stats["frames"] = frames
    PARITY_STATS[name] = dict(stats)
    print(f"\n[parity {name}] {frames} steps: exact {stats['exact']}, boundary(+-1px) {stats['boundary']}, ties {stats['ties']}, "
          f"max|dscore| {stats['max_dscore']:.2e}, min IoU on boundary steps {stats['min_iou_boundary']:.4f}")
    assert stats["max_dscore"] <= SCORE_TOL
    assert stats["ties"] + stats["boundary"] <= max(1, math.ceil(EXEMPT_FRAC * frames)), (name, stats)
    assert stats["exact"] >= frames - stats["ties"] - stats["boundary"], (name, stats)


# ---- preprocessing: bit-exact ----------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["nv12", "rgb24"])
def test_search_and_template_blobs_bit_exact(api, oracle, weight_dir, fmt):
    """K2 (fused crop + NV12->RGB + OpenCV bilinear + normalise) == oracle crop/resize/norm on the converted frame,
    for boxes inside, hanging over each edge, tiny (up-scale) and huge."""
    W, H = 1280, 720
    wpath = weights.ensure_weight_file("nano", weight_dir)
    spec = synth.StreamSpec("pp", W, H, 41, [(500, 300, 120, 90, 3, 2)], fmt=fmt)
    st = synth.SyntheticStream(spec)
    frame = st.frame(3)
    rgb = frame if fmt == "rgb24" else oracle.nv12_to_rgb(frame, W, H, 8)
    trk = api.VitTrack.new(wpath, W, H, fmt=fmt)
    ref = oracle.VitTrack(wpath, threads=4)
    boxes = [(500, 300, 120, 90), (0, 0, 60, 40), (-30, -20, 100, 80), (1200, 650, 120, 90), (640, -40, 90, 100), (-50, 400, 150, 60),
             (600, 700, 40, 40), (100, 100, 21, 23), (300, 200, 10, 12), (200, 100, 400, 300), (0, 0, 1280, 720), (639, 359, 2, 2),
             (700, 300, 64, 64), (700, 300, 63, 65), (50, 60, 33, 31)]
    for box in boxes:
        flat = np.ascontiguousarray(frame).reshape(-1)
        trk.init(flat, api.BBox(*box))
        ref.init(rgb, box)
        trk.update_all(flat)
        ref.rect = box
        rc = ref.update(rgb)[0]
        assert rc == 0
        sb, tb = ref.last_blobs()
        d = trk.debug_read(0)
        assert np.array_equal(d["template_blob"], tb), ("template", box, int((d["template_blob"] != tb).sum()))
        assert np.array_equal(d["search_blob"], sb), ("search", box, int((d["search_blob"] != sb).sum()))


def test_short_nv12_frame_is_black(api, oracle, weight_dir):
    """A too-short NV12 buffer is an all-zero image to the tracker (src/nv12_convert.rs:48-50)."""
    W, H = 640, 360
    wpath = weights.ensure_weight_file("nano", weight_dir)
    trk = api.VitTrack.new(wpath, W, H)
    ref = oracle.VitTrack(wpath, threads=2)
    short = np.full(W * H * 3 // 2 - 7, 180, np.uint8)
    black = np.zeros((H, W, 3), np.uint8)
    trk.init(short, api.BBox(300, 150, 60, 50))
    ref.init(black, (300, 150, 60, 50))
    r = trk.update(short)
    rc, ok, score, bb = ref.update(black)
    assert abs(r.score - score) <= SCORE_TOL and r.success == ok and (not ok or tuple(r.bbox) == tuple(bb))


# ---- network: layer-wise ------------------------------------------------------------------------------
@pytest.mark.parametrize("gemm_mode", [0, 1], ids=["fp32simt", "tcgen05x3"])
@pytest.mark.parametrize("model", ["nano", "tiny"])
def test_layerwise_tokens(api, oracle, weight_dir, model, gemm_mode):
    """Token features after the embeddings and after every block vs the fp32 oracle (relative 2e-4 of the layer's scale)."""
    W, H = 1280, 720
    wpath = weights.ensure_weight_file(model, weight_dir, variant="wild")
    st = synth.SyntheticStream(synth.CONFIGS["cfg1"])
    frame = st.frame(0)
    rgb = oracle.nv12_to_rgb(frame, W, H, 8)
    box = st.target_boxes(0)[0]
    trk = api.VitTrack.new(wpath, W, H, debug_capture=True, gemm_mode=gemm_mode)
    ref = oracle.VitTrack(wpath, threads=8)
    trk.init(frame, api.BBox(*box))
    ref.init(rgb, box)
    trk.update_all(frame)
    assert ref.update(rgb)[0] == 0
    depth = trk.model_dim(1)
    for which in range(depth + 1):
        a, b = trk.debug_tokens(which), ref.debug_tokens(which)
        scale = float(np.abs(b).max())
        err = float(np.abs(a - b).max())
        assert err <= 2e-4 * scale, (model, which, err, scale)
    fin = trk.debug_read(0)["tokens"][64:]
    b = ref.debug_tokens(depth + 1)[64:]
    assert float(np.abs(fin - b).max()) <= 2e-4 * float(np.abs(b).max())
    cw, sm, om, _ = ref.last_maps()
    d = trk.debug_read(0)
    assert float(np.abs(d["conf_win"] - cw).max()) <= SCORE_TOL
    assert float(np.abs(d["size_map"] - sm).max()) <= 1e-4
    assert float(np.abs(d["off_map"] - om).max()) <= 1e-3


# ---- against the third-party cv2.TrackerVit fixtures -----------------------------------------------------
@pytest.mark.parametrize("gemm_mode", [0, 1], ids=["fp32simt", "tcgen05x3"])
@pytest.mark.parametrize("variant", ["stable", "wild"])
@pytest.mark.parametrize("model", ["nano", "tiny"])
def test_sequences_vs_cv2_golden(api, weight_dir, model, variant, gemm_mode):
    """Free-running sequences recorded from the third-party cv2.TrackerVit (nano and the bench model tiny; cfg2 leads the tiny set)."""
    g = golden(f"trackervit_{model}.json")["models"][variant]
    wpath = weights.ensure_weight_file(model, weight_dir, variant=variant)
    assert hashlib.sha256(open(wpath, "rb").read()).hexdigest() == g["weights_sha256"]
    for seq in g["sequences"]:
        sp = seq["spec"]
        spec = synth.StreamSpec(seq["name"], sp["w"], sp["h"], sp["seed"], [tuple(t) for t in sp["targets"]])
        st = synth.SyntheticStream(spec)
        trk = api.VitTrack.new(wpath, spec.width, spec.height, gemm_mode=gemm_mode)
        trk.init(st.frame(0), api.BBox(*seq["init_box"]))
        n_exact, dmax = 0, 0.0
        for i, fr in enumerate(seq["frames"]):
            r = trk.update(st.frame(i))
            dmax = max(dmax, abs(r.score - fr["score"]))
            assert abs(r.score - fr["score"]) <= SCORE_TOL, (seq["name"], i, r.score, fr["score"])
            assert r.success == fr["ok"]
            if fr["ok"]:
                if list(r.bbox) == fr["bbox"]:
                    n_exact += 1
                else:  # resynchronise on cv2's box so that one boundary flip cannot cascade
                    assert iou(r.bbox, fr["bbox"]) >= 0.95 and max(abs(a - b) for a, b in zip(r.bbox, fr["bbox"])) <= 1, (seq["name"], i, r.bbox, fr["bbox"])
                    trk.set_rect(fr["bbox"])
        PARITY_STATS[f"cv2_sequence/{model}/{variant}/{seq['name']}/gemm{gemm_mode}"] = {
            "frames": len(seq["frames"]), "exact": n_exact, "max_dscore": dmax}
        assert n_exact >= len(seq["frames"]) - 2, (seq["name"], n_exact)


@pytest.mark.parametrize("gemm_mode", [0, 1], ids=["fp32simt", "tcgen05x3"])
@pytest.mark.parametrize("variant", ["stable", "wild"])
@pytest.mark.parametrize("model", ["nano", "tiny"])
def test_single_steps_vs_cv2_golden(api, weight_dir, model, variant, gemm_mode):
    g = golden(f"trackervit_{model}.json")["models"][variant]
    wpath = weights.ensure_weight_file(model, weight_dir, variant=variant)
    sp = g["steps_spec"]
    spec = synth.StreamSpec("steps", sp["w"], sp["h"], sp["seed"], [tuple(t) for t in sp["targets"]])
    st = synth.SyntheticStream(spec)
    f0, f1 = st.frame(sp["frames"][0]), st.frame(sp["frames"][1])
    trk = api.VitTrack.new(wpath, spec.width, spec.height, gemm_mode=gemm_mode)
    n_exact = n = 0
    for s in g["single_steps"]:
        if s.get("error"):
            with pytest.raises(api.VtError) as e:
                trk.init(f0, api.BBox(*s["box"]))
                trk.update(f1)
            assert e.value.status == -4  # VT_ERR_CROP_OUTSIDE ≙ Err
            continue
        trk.init(f0, api.BBox(*s["box"]))
        r = trk.update(f1)
        assert abs(r.score - s["score"]) <= SCORE_TOL, (s, r.score)
        assert r.success == s["ok"]
        n += 1
        if s["ok"]:
            d = max(abs(a - b) for a, b in zip(r.bbox, s["bbox"]))
            assert d <= 1, (s, r.bbox)
            n_exact += d == 0
    assert n_exact >= n - 2, (n_exact, n)


# ---- teacher-forced long sequences vs the oracle ------------------------------------------------------------
@pytest.mark.parametrize("gemm_mode", [0, 1, 3], ids=["fp32simt", "tcgen05x3", "tcgen05fp16"])
@pytest.mark.parametrize("model,cfg,frames", [("nano", "cfg1", 120), ("tiny", "cfg2", 60)])
def test_teacher_forced_sequence(api, oracle, weight_dir, model, cfg, frames, gemm_mode):
    spec = synth.CONFIGS[cfg]
    W, H = spec.width, spec.height
    wpath = weights.ensure_weight_file(model, weight_dir)
    st = synth.SyntheticStream(spec)
    trk = api.VitTrack.new(wpath, W, H, gemm_mode=gemm_mode)
    ref = oracle.VitTrack(wpath, threads=8)
    f0 = st.frame(0)
    box = st.target_boxes(0)[0]
    trk.init(f0, api.BBox(*box))
    ref.init(oracle.nv12_to_rgb(f0, W, H, 8), box)
    stats = new_stats()
    fp16 = gemm_mode == 3
    for n in range(frames):
        fr = st.frame(n)
        before = ref.rect
        trk.set_rect(before)
        r = trk.update(fr)
        rc = ref.update(oracle.nv12_to_rgb(fr, W, H, 8))[0]
        assert rc == 0
        compare_step(trk, r, ref, before, stats, (model, cfg, n), tie_margin=TIE_MARGIN_FP16 if fp16 else TIE_MARGIN)
    if fp16:  # opt-in mode: its wider tie window is not held to the 3 % bound of the default paths; the score bar is the same
        PARITY_STATS[f"teacher_forced/{model}/{cfg}/gemm{gemm_mode}"] = dict(stats, frames=frames)
        assert stats["max_dscore"] <= SCORE_TOL and stats["exact"] >= 0.85 * frames, stats
    else:
        finish_stats(f"teacher_forced/{model}/{cfg}/gemm{gemm_mode}", stats, frames)


@pytest.mark.parametrize("model,cfg,frames,first_min", [("nano", "cfg1", 120, 30), ("tiny", "cfg2", 300, 100)])
def test_free_running_sequence_iou(api, oracle, weight_dir, model, cfg, frames, first_min):
    """No teacher forcing: the GPU tracker and the oracle run free from the same init box (cfg2 / tiny = the bench workload, 300 frames).
    IoU >= 0.99 and |dscore| <= 1e-3 on every frame up to the first numerically undecidable one (tie / floor boundary), which must not
    come before frame `first_min`; there the GPU state is resynchronised on the oracle's rect (a one-pixel difference would otherwise
    feed back through the crop) and the run continues under the same rules; undecidable frames stay <= 3 %."""
    spec = synth.CONFIGS[cfg]
    W, H = spec.width, spec.height
    wpath = weights.ensure_weight_file(model, weight_dir)
    st = synth.SyntheticStream(spec)
    trk = api.VitTrack.new(wpath, W, H, gemm_mode=1)
    ref = oracle.VitTrack(wpath, threads=16)
    box = st.target_boxes(0)[0]
    trk.init(st.frame(0), api.BBox(*box))
    ref.init(oracle.nv12_to_rgb(st.frame(0), W, H, 16), box)
    stats = new_stats()
    first = None
    min_iou = 1.0
    for n in range(frames):
        fr = st.frame(n)
        before = ref.rect
        assert trk.get_rect() == tuple(before), n   # both trackers enter the frame with the same rect_last
        r = trk.update(fr)
        rc, ok, score, bb = ref.update(oracle.nv12_to_rgb(fr, W, H, 16))
        assert rc == 0
        same = compare_step(trk, r, ref, before, stats, (model, cfg, n))
        if same:
            assert r.success == ok and (not ok or (tuple(r.bbox) == tuple(bb) and iou(r.bbox, bb) >= IOU_MIN)), (n, r, bb)
        else:
            first = n if first is None else first
            if ok:
                min_iou = min(min_iou, iou(r.bbox, bb))
            trk.set_rect(ref.rect)
    stats["first_undecidable_frame"] = first
    stats["min_iou_undecidable"] = min_iou
    finish_stats(f"free_running/{model}/{cfg}", stats, frames)
    assert first is None or first > first_min, (first, stats)


@pytest.mark.gpu
def test_cfg4_full_size_16_targets_vs_oracle(api, oracle, weight_dir):
    """BASELINE config 4 at full size: 3840x2160 NV12, tiny, 16 targets through ONE batched forward (M = 5120 rows: the many-row
    forms — A-stationary QKV, chained MLP with the hidden tile in tensor memory, three partial planes), 5 teacher-forced frames, EVERY target against its own oracle.VitTrack (one fp32 forward per target
    and frame): score within 1e-3, box equal off floor ties (reference semantics: /root/reference/src/tracker_context.rs:120-125,
    one VitTrack per target)."""
    spec = synth.CONFIGS["cfg4"]
    W, H = spec.width, spec.height
    st = synth.SyntheticStream(spec)
    nt = len(spec.targets)
    assert nt == 16
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    trk = api.VitTrack.new(wpath, W, H, max_targets=nt, gemm_mode=1)
    refs = [oracle.VitTrack(wpath, threads=16) for _ in range(nt)]
    f0 = st.frame(0)
    rgb0 = oracle.nv12_to_rgb(f0, W, H, 16)
    for k, b in enumerate(st.target_boxes(0)):
        trk.init(f0, api.BBox(*b), target=k)
        assert refs[k].init(rgb0, b) == 0
    stats = new_stats()
    frames = 5
    for n in range(frames):
        fr = st.frame(n)
        rgb = oracle.nv12_to_rgb(fr, W, H, 16)
        before = [refs[k].rect for k in range(nt)]
        for k in range(nt):
            trk.set_rect(before[k], target=k)
        rs = trk.update_all(fr)
        for k in range(nt):
            assert rs[k].status == 0, (n, k, rs[k])
            assert refs[k].update(rgb)[0] == 0
            compare_step(trk, rs[k], refs[k], before[k], stats, ("cfg4", n, k), target=k)
    finish_stats("teacher_forced/tiny/cfg4x16/gemm1", stats, frames * nt)


def test_stream_group_16_streams_vs_oracle(api, oracle, weight_dir):
    """BASELINE config 5's unit of work as this repo runs it: 16 independent 1080p NV12 streams (cfg5 seeds) stepped together through
    vt_tracker_update_streams (one batched forward of 5120 rows, every stream its own pinned frame, search-window upload and device-side
    rect_last), 4 teacher-forced steps, EVERY stream against its own oracle.VitTrack on its own frames (one TrackerContext per
    pipeline, /root/reference/src/pipeline.rs:55): score within 1e-3, box equal off floor ties."""
    G, steps = 16, 4
    streams = [synth.SyntheticStream(synth.cfg5_stream(i)) for i in range(G)]
    spec = streams[0].spec
    W, H = spec.width, spec.height
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    trk = api.VitTrack.new(wpath, W, H, max_targets=G, gemm_mode=1, upload_window=True)
    refs = [oracle.VitTrack(wpath, threads=16) for _ in range(G)]
    pins = [api.PinnedBuffer(s_.frame_bytes()) for s_ in streams]
    for i, s_ in enumerate(streams):
        f0 = np.ascontiguousarray(s_.frame(0)).reshape(-1)
        b = s_.target_boxes(0)[0]
        trk.init(f0, api.BBox(*b), target=i)
        assert refs[i].init(oracle.nv12_to_rgb(f0, W, H, 16), b) == 0
    stats = new_stats()
    for n in range(1, steps + 1):
        before = [refs[i].rect for i in range(G)]
        for i, s_ in enumerate(streams):
            pins[i].array[:] = np.ascontiguousarray(s_.frame(n)).reshape(-1)
            trk.set_rect(before[i], target=i)
        rs = trk.update_streams([p.array for p in pins])
        for i, s_ in enumerate(streams):
            assert rs[i].status == 0, (n, i, rs[i])
            assert refs[i].update(oracle.nv12_to_rgb(np.ascontiguousarray(s_.frame(n)).reshape(-1), W, H, 16))[0] == 0
            compare_step(trk, rs[i], refs[i], before[i], stats, ("group16", n, i), target=i)
    finish_stats("teacher_forced/tiny/stream_group16/gemm1", stats, steps * G)
    trk.close()
    for p in pins:
        p.close()


# ---- multi-target, formats, errors -----------------------------------------------------------------------------
@pytest.mark.parametrize("gemm_mode", [0, 1], ids=["fp32simt", "tcgen05x3"])
def test_multi_target_equals_independent_singles(api, weight_dir, gemm_mode):
    """16 targets batched through one forward (cfg4 geometry at 1/2 scale for speed) == 16 single-target trackers: bit for bit while
    the same kernel forms run (fp32 path; tensor-core path below 8 targets, checked with a 4-target handle); from 8 targets on the
    tensor-core MLP runs unchained (FC2 as its own GEMM instead of 12 partial products) — a re-association of the same sums, boxes
    equal and scores within 1e-5."""
    spec = synth.StreamSpec("mt", 1920, 1080, 1004, [(190 + (i % 4) * 450, 110 + (i // 4) * 250, 100, 75, 3 + i % 4, 2 + i // 4) for i in range(16)])
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    multi = api.VitTrack.new(wpath, spec.width, spec.height, max_targets=16, gemm_mode=gemm_mode)
    multi4 = api.VitTrack.new(wpath, spec.width, spec.height, max_targets=4, gemm_mode=gemm_mode)
    singles = [api.VitTrack.new(wpath, spec.width, spec.height, gemm_mode=gemm_mode) for _ in range(16)]
    f0 = st.frame(0)
    for i, b in enumerate(st.target_boxes(0)):
        multi.init(f0, api.BBox(*b), target=i)
        singles[i].init(f0, api.BBox(*b))
        if i < 4:
            multi4.init(f0, api.BBox(*b), target=i)
    tol = 0.0 if gemm_mode == 0 else 1e-5
    for n in range(5):
        fr = st.frame(n)
        rs, rs4 = multi.update_all(fr), multi4.update_all(fr)
        for i in range(16):
            r1 = singles[i].update(fr)
            assert rs[i].status == 0 and rs[i].success == r1.success and rs[i].bbox == r1.bbox and abs(rs[i].score - r1.score) <= tol, (n, i, rs[i], r1)
            if i < 4:
                assert rs4[i] == r1, (n, i, rs4[i], r1)
    # dropping a target leaves the others untouched; un-initialised slots report VT_ERR_NOT_INIT
    multi.drop(3)
    rs = multi.update_all(st.frame(5))
    assert rs[3].status == -5
    assert rs[4].bbox == singles[4].update(st.frame(5)).bbox


def test_graph_and_eager_paths_agree(api, weight_dir):
    spec = synth.CONFIGS["cfg1"]
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir)
    a = api.VitTrack.new(wpath, spec.width, spec.height, use_cuda_graph=True)
    b = api.VitTrack.new(wpath, spec.width, spec.height, use_cuda_graph=False)
    box = api.BBox(*st.target_boxes(0)[0])
    a.init(st.frame(0), box)
    b.init(st.frame(0), box)
    for n in range(8):
        ra, rb = a.update(st.frame(n)), b.update(st.frame(n))
        assert ra == rb, (n, ra, rb)
    assert a.timing().kernel_launches == b.timing().kernel_launches > 0


def test_submit_wait_and_device_resident_frame(api, weight_dir):
    import torch

    spec = synth.CONFIGS["cfg1"]
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir)
    a = api.VitTrack.new(wpath, spec.width, spec.height)
    b = api.VitTrack.new(wpath, spec.width, spec.height)
    c = api.VitTrack.new(wpath, spec.width, spec.height)
    box = api.BBox(*st.target_boxes(0)[0])
    for t in (a, b, c):
        t.init(st.frame(0), box)
    pin = api.PinnedBuffer(st.frame_bytes())
    for n in range(6):
        fr = st.frame(n)
        ra = a.update(fr)
        pin.array[:] = fr
        b.submit(pin.array)
        rb = b.wait()[0]
        d = torch.from_numpy(fr).cuda()
        torch.cuda.synchronize()
        rc = c.update_device(d.data_ptr(), fr.size)[0]
        assert ra == rb == rc, (n, ra, rb, rc)


def test_error_paths(api, weight_dir):
    spec = synth.CONFIGS["cfg1"]
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir)
    with pytest.raises(api.VtError) as e:
        api.VitTrack.new("/nonexistent/model.vtw", 640, 480)
    assert e.value.status == -3  # ≙ VitTrack::new Err -> TrackerContext::new fails (src/tracker_context.rs:21)
    trk = api.VitTrack.new(wpath, spec.width, spec.height)
    r = trk.update_all(st.frame(0))[0]
    assert r.status == -5 and not r.success  # update before init
    with pytest.raises(api.VtError) as e:
        trk.init(st.frame(0), api.BBox(5000, 5000, 40, 40))
    assert e.value.status == -4
    trk.init(st.frame(0), api.BBox(600, 300, 100, 80))
    trk.set_rect((-900, -900, 30, 30))  # search window now entirely outside
    r = trk.update_all(st.frame(1))[0]
    assert r.status == -4 and not r.success


def test_box_overlay_fused_path(api, oracle, weight_dir):
    """cfg.box_overlay: update() draws rect + crosshair of the gated result on the device and returns the touched rows."""
    spec = synth.CONFIGS["cfg1"]
    W, H = spec.width, spec.height
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir)
    trk = api.VitTrack.new(wpath, W, H, box_overlay=True)
    trk.init(st.frame(0), api.BBox(*st.target_boxes(0)[0]))
    for n in range(4):
        fr = st.frame(n)
        ref = fr.copy()
        r = trk.update(fr)
        if r.success and r.score > 0.25:
            x, y, w, h = r.bbox
            oracle.draw_rect_nv12(ref, W, H, x, y, w, h, 3, 255)
            oracle.draw_crosshair_nv12(ref, W, H, x + w // 2, y + h // 2, 15, 255)
        assert np.array_equal(fr, ref), (n, int((fr != ref).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["nv12", "rgb24"])
def test_box_overlay_zero_copy_mirror_into_pinned_frame(api, oracle, weight_dir, fmt):
    """With a pinned caller frame the overlay kernel writes the box pixels straight into host memory (no row copy): the frame must
    equal the oracle's draw_rect + draw_crosshair on the same result, and the pageable (row-copy) path must give the same bytes."""
    spec = synth.CONFIGS["cfg1"] if fmt == "nv12" else synth.CONFIGS["cfg3"]
    W, H = spec.width, spec.height
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir)
    a = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True)
    b = api.VitTrack.new(wpath, W, H, fmt=fmt, box_overlay=True)
    f0 = np.asarray(st.frame(0)).reshape(-1)
    box = api.BBox(*st.target_boxes(0)[0])
    a.init(f0, box)
    b.init(f0, box)
    pin = api.PinnedBuffer(f0.size)
    for n in range(4):
        fr = np.asarray(st.frame(n)).reshape(-1).copy()
        ref = fr.copy()
        pin.array[:] = fr
        ra = a.update(pin.array)   # pinned: zero-copy mirror
        rb = b.update(fr)          # pageable: touched rows copied back
        assert ra == rb
        if ra.success and ra.score > 0.25:
            x, y, w, h = ra.bbox
            if fmt == "nv12":
                oracle.draw_rect_nv12(ref, W, H, x, y, w, h, 3, 255)
                oracle.draw_crosshair_nv12(ref, W, H, x + w // 2, y + h // 2, 15, 255)
            else:
                oracle.draw_rect_rgb(ref, W, H, x, y, w, h, 3, (0, 255, 0))
                oracle.draw_crosshair_rgb(ref, W, H, x + w // 2, y + h // 2, 15, (0, 255, 0))
        assert np.array_equal(pin.array, ref), (n, int((pin.array != ref).sum()))
        assert np.array_equal(fr, ref), (n, int((fr != ref).sum()))


@pytest.mark.gpu
def test_concurrent_streams_equal_sequential(api, weight_dir):
    """Independent handles driven from different host threads (one CUDA stream + graph each, sharing the GPU) reproduce the
    single-stream results bit for bit — the multi-stream / multi-GPU sharding has no cross-stream state."""
    import threading

    wpath = weights.ensure_weight_file("tiny", weight_dir)
    specs = [synth.cfg5_stream(i) for i in range(4)]
    frames = [[synth.SyntheticStream(s).frame(n) for n in range(6)] for s in specs]
    boxes = [synth.SyntheticStream(s).target_boxes(0)[0] for s in specs]

    def run_stream(i, out):
        trk = api.VitTrack.new(wpath, specs[i].width, specs[i].height, gemm_mode=1, box_overlay=True)
        trk.init(frames[i][0], api.BBox(*boxes[i]))
        out[i] = [trk.update(frames[i][n].copy()) for n in range(6)]

    seq, par = {}, {}
    for i in range(4):
        run_stream(i, seq)
    th = [threading.Thread(target=run_stream, args=(i, par)) for i in range(4)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert seq == par


@pytest.mark.gpu
def test_device_stage_stamps(api, weight_dir):
    """vt_timing_get: stage times come from device stamps; they are positive, ordered and add up to less than the wall time."""
    spec = synth.CONFIGS["cfg2"]
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    trk = api.VitTrack.new(wpath, spec.width, spec.height, gemm_mode=1, box_overlay=True)
    trk.init(st.frame(0), api.BBox(*st.target_boxes(0)[0]))
    for n in range(5):
        trk.update(st.frame(n))
    t = trk.timing()
    for f in ("h2d_ms", "preprocess_ms", "vit_ms", "decode_ms", "overlay_ms", "total_ms"):
        assert getattr(t, f) > 0, f
    dev = t.h2d_ms + t.preprocess_ms + t.vit_ms + t.decode_ms + t.overlay_ms
    assert dev <= t.total_ms * 1.001 and t.vit_ms > 0.5 * dev
    assert t.frames == 5 and t.kernel_launches > 5 * 30 and t.h2d_bytes == 6 * st.frame_bytes()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["cfg2", "cfg4"])
def test_full_size_properties(api, oracle, weight_dir, cfg):
    """BASELINE.json sizes (1080p one target, 2160p 16 targets), properties that do not need the fp32 oracle forward at that size:
    (1) the search blob of every target is bit-exact against the oracle's crop/resize/normalise of the same frame and rect,
    (2) the result is invariant to pixels outside every search window (the fused kernel reads only the crop),
    (3) replaying the same frame from the same state is idempotent in (score, box)."""
    spec = synth.CONFIGS[cfg]
    W, H = spec.width, spec.height
    st = synth.SyntheticStream(spec)
    nt = len(spec.targets)
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    trk = api.VitTrack.new(wpath, W, H, max_targets=nt, gemm_mode=1)
    f0, f1 = st.frame(0), st.frame(1)
    boxes = st.target_boxes(0)
    for k, b in enumerate(boxes):
        trk.init(f0, api.BBox(*b), target=k)
    r1 = trk.update_all(f1)
    rgb1 = oracle.nv12_to_rgb(f1, W, H, 4)
    for k in (0, nt - 1):
        blob = np.asarray(trk.debug_read(target=k)["search_blob"]).reshape(-1)
        rc, crop = oracle.crop_square(rgb1, boxes[k], 4)
        assert rc == 0
        ref = oracle.normalize_chw(oracle.resize_linear(crop, 256, 256)).reshape(-1)
        assert np.array_equal(blob, ref), (cfg, k, int((blob != ref).sum()))
    # (3) same state, same frame -> same answer
    for k, b in enumerate(boxes):
        trk.set_rect(tuple(b), target=k)
    assert trk.update_all(f1) == r1
    # (2) scribble outside all search windows (Y plane rows far from every target)
    f2 = f1.copy()
    wins = []
    for b in boxes:
        c = int(np.ceil(np.sqrt(float(b[2] * b[3])) * 4))
        wins.append((b[1] + (b[3] - c) // 2 - 2, b[1] + (b[3] - c) // 2 + c + 2))
    rows = [y for y in range(0, H, 2) if all(not (lo <= y <= hi) for lo, hi in wins)]
    assert rows, "no row outside the search windows"
    for y in rows[:64]:
        f2[y * W:(y + 1) * W] = 255 - f2[y * W:(y + 1) * W]
    for k, b in enumerate(boxes):
        trk.set_rect(tuple(b), target=k)
    assert trk.update_all(f2) == r1


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,cfg", [("nv12", "cfg1"), ("rgb24", "cfg3"), ("nv12", "mt")])
def test_window_upload_equals_full_upload(api, weight_dir, fmt, cfg):
    """cfg.upload_window: only the search windows travel over PCIe; results and the overlaid host frame are identical to the
    whole-frame upload, frame after frame (free running, so the host mirror of rect_last is exercised), incl. borders / 16 targets."""
    if cfg == "mt":
        spec = synth.StreamSpec("mt", 1920, 1080, 1004, [(190 + (i % 4) * 450, 110 + (i // 4) * 250, 100, 75, 3 + i % 4, 2 + i // 4) for i in range(16)])
    else:
        spec = synth.CONFIGS[cfg]
    st = synth.SyntheticStream(spec)
    nt = len(spec.targets)
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    a = api.VitTrack.new(wpath, spec.width, spec.height, fmt=fmt, max_targets=nt, box_overlay=True, gemm_mode=1, upload_window=True)
    b = api.VitTrack.new(wpath, spec.width, spec.height, fmt=fmt, max_targets=nt, box_overlay=True, gemm_mode=1, upload_window=False)
    f0 = np.asarray(st.frame(0)).reshape(-1)
    pa, pb = api.PinnedBuffer(f0.size), api.PinnedBuffer(f0.size)
    pa.array[:] = f0
    for k, box in enumerate(st.target_boxes(0)):
        a.init(pa.array, api.BBox(*box), target=k)
        b.init(pa.array, api.BBox(*box), target=k)
    h2d0 = a.timing().h2d_bytes
    for n in range(1, 9):
        fr = np.asarray(st.frame(n)).reshape(-1)
        pa.array[:] = fr
        pb.array[:] = fr
        ra, rb = a.update_all(pa.array), b.update_all(pb.array)
        assert ra == rb, (n, ra, rb)
        assert np.array_equal(pa.array, pb.array), n
    if nt == 1:
        assert a.timing().h2d_bytes - h2d0 < 0.5 * 8 * f0.size  # the window really is smaller than the frame
    # a box pushed against / over the border still matches
    a.set_rect((-20, -10, 90, 70))
    b.set_rect((-20, -10, 90, 70))
    pa.array[:] = f0
    pb.array[:] = f0
    assert a.update_all(pa.array) == b.update_all(pb.array)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,cfg", [("nv12", "cfg1"), ("rgb24", "cfg3")])
def test_window_miss_falls_back_to_the_pinned_host_frame(api, weight_dir, monkeypatch, fmt, cfg):
    """Window uploads are predictions when a frame is in flight (rect_last on the host lags by one frame): whatever the uploaded
    window misses, the crop kernel reads from the caller's pinned frame (zero-copy), so results never depend on the prediction.
    Forced here by uploading windows that are 60 px too small on every side (VT_B200_WINDOW_SHRINK): synchronous and pipelined
    results and overlay pixels must equal the whole-frame upload."""
    spec = synth.CONFIGS[cfg]
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    n = 8
    frames = [np.asarray(st.frame(i)).reshape(-1) for i in range(n)]
    box = api.BBox(*st.target_boxes(0)[0])
    ref = api.VitTrack.new(wpath, spec.width, spec.height, fmt=fmt, box_overlay=True, gemm_mode=1, upload_window=False)
    monkeypatch.setenv("VT_B200_WINDOW_SHRINK", "60")
    a = api.VitTrack.new(wpath, spec.width, spec.height, fmt=fmt, box_overlay=True, gemm_mode=1, upload_window=True)
    b = api.VitTrack.new(wpath, spec.width, spec.height, fmt=fmt, box_overlay=True, gemm_mode=1, upload_window=True)
    monkeypatch.delenv("VT_B200_WINDOW_SHRINK")
    pr, pa = api.PinnedBuffer(frames[0].size), api.PinnedBuffer(frames[0].size)
    pins = [api.PinnedBuffer(frames[0].size) for _ in range(n)]
    for t in (ref, a, b):
        t.init(frames[0], box)
    want, want_px = [], []
    h2d0 = a.timing().h2d_bytes
    for i in range(n):
        pr.array[:] = frames[i]
        pa.array[:] = frames[i]
        want.append(ref.update(pr.array))
        assert a.update(pa.array) == want[-1], i                 # synchronous, exact mirror, shrunk window
        assert np.array_equal(pa.array, pr.array), i
        want_px.append(pr.array.copy())
        pins[i].array[:] = frames[i]
    assert a.timing().h2d_bytes - h2d0 < 0.3 * n * frames[0].size  # the windows really were small
    got = []
    b.submit(pins[0].array)
    for i in range(1, n):                                         # pipelined: lagging mirror, predicted + shrunk windows
        b.submit(pins[i].array)
        got.append(b.wait()[0])
    got.append(b.wait()[0])
    assert got == want
    for i in range(n):
        assert np.array_equal(pins[i].array, want_px[i]), i


@pytest.mark.gpu
def test_bench_workload_teacher_forced_300_frames(api, oracle, weight_dir):
    """The exact bench workload (cfg2, tiny, bf16x3, box overlay, window upload from a pinned frame) against the fp32 oracle over 300
    teacher-forced frames: boxes equal except numerically undecidable floor ties, |dscore| <= 1e-3, overlay pixels as the oracle draws."""
    spec = synth.CONFIGS["cfg2"]
    W, H = spec.width, spec.height
    wpath = weights.ensure_weight_file("tiny", weight_dir)
    st = synth.SyntheticStream(spec)
    trk = api.VitTrack.new(wpath, W, H, gemm_mode=1, box_overlay=True, upload_window=True)
    ref = oracle.VitTrack(wpath, threads=16)
    f0 = st.frame(0)
    pin = api.PinnedBuffer(f0.size)
    pin.array[:] = f0
    box = st.target_boxes(0)[0]
    trk.init(pin.array, api.BBox(*box))
    ref.init(oracle.nv12_to_rgb(f0, W, H, 16), box)
    stats = new_stats()
    frames = 300
    for n in range(frames):
        fr = st.frame(n)
        before = ref.rect
        trk.set_rect(before)
        pin.array[:] = fr
        r = trk.update(pin.array)
        rc = ref.update(oracle.nv12_to_rgb(fr, W, H, 16))[0]
        assert rc == 0
        compare_step(trk, r, ref, before, stats, ("tiny", "cfg2", n))
        if n % 50 == 0 and r.success and r.score > 0.25:
            want = fr.copy()
            x, y, w, h = r.bbox
            oracle.draw_rect_nv12(want, W, H, x, y, w, h, 3, 255)
            oracle.draw_crosshair_nv12(want, W, H, x + w // 2, y + h // 2, 15, 255)
            assert np.array_equal(pin.array, want), n
    finish_stats("teacher_forced/tiny/cfg2/bench_workload_300", stats, frames)


@pytest.mark.gpu
def test_pipelined_submit_wait_depth_two(api, weight_dir):
    """Two frames in flight per handle (rect_last lives on the device): results, overlay pixels and final state equal the synchronous
    call sequence; a third submit, a pipelined pageable frame and update() with frames in flight are refused."""
    import torch

    spec = synth.CONFIGS["cfg1"]
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    a = api.VitTrack.new(wpath, spec.width, spec.height, box_overlay=True, upload_window=True)
    b = api.VitTrack.new(wpath, spec.width, spec.height, box_overlay=True, upload_window=True)
    c = api.VitTrack.new(wpath, spec.width, spec.height, box_overlay=True)
    box = api.BBox(*st.target_boxes(0)[0])
    n = 10
    frames = [st.frame(i) for i in range(n)]
    pins = [api.PinnedBuffer(frames[0].size) for _ in range(n)]
    sync_frames = []
    for t in (a, b, c):
        t.init(frames[0], box)
    want = []
    for i in range(n):
        p = api.PinnedBuffer(frames[0].size)
        p.array[:] = frames[i]
        want.append(a.update(p.array))
        sync_frames.append(p.array.copy())
    # host frames, pipelined
    for i in range(n):
        pins[i].array[:] = frames[i]
    got = []
    b.submit(pins[0].array)
    for i in range(1, n):
        b.submit(pins[i].array)
        got.append(b.wait()[0])
    with pytest.raises(api.VtError):
        b.update(pins[0].array)          # a frame is still in flight
    got.append(b.wait()[0])
    assert got == want
    for i in range(n):
        assert np.array_equal(pins[i].array, sync_frames[i]), i
    # device frames, pipelined, tracked in place
    dev = [torch.from_numpy(frames[i]).cuda() for i in range(n)]
    torch.cuda.synchronize()
    got = []
    c.submit_device(dev[0].data_ptr(), frames[0].size)
    c.submit_device(dev[1].data_ptr(), frames[0].size)
    with pytest.raises(api.VtError):
        c.submit_device(dev[2].data_ptr(), frames[0].size)   # queue depth is two
    got.append(c.wait()[0])
    for i in range(2, n):
        c.submit_device(dev[i].data_ptr(), frames[0].size)
        got.append(c.wait()[0])
    got.append(c.wait()[0])
    assert got == want
    for i in range(n):
        assert np.array_equal(dev[i].cpu().numpy(), sync_frames[i]), i   # the box was drawn into the caller's device frame
    # pageable frames cannot be pipelined
    c.submit_device(dev[0].data_ptr(), frames[0].size)
    with pytest.raises(api.VtError):
        c.submit(frames[1].copy())
    c.wait()


@pytest.mark.gpu
def test_gray8_input_format(api, oracle, weight_dir):
    """BASELINE config "IR/GRAY8 at 640x512": a GRAY8 frame is tracked as r = g = b = gray (search blob bit-exact against the oracle on the
    replicated RGB frame, boxes / scores as the oracle's), and the box overlay follows the NV12 luma-plane semantics."""
    spec = synth.CONFIGS["cfg3"]
    W, H = spec.width, spec.height
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir)

    def gray(n):
        rgb = np.asarray(st.frame(n)).reshape(H, W, 3).astype(np.uint32)
        return ((rgb[..., 0] * 77 + rgb[..., 1] * 150 + rgb[..., 2] * 29 + 128) >> 8).astype(np.uint8).reshape(-1)

    trk = api.VitTrack.new(wpath, W, H, fmt="gray8", box_overlay=True, upload_window=True)
    ref = oracle.VitTrack(wpath, threads=4)
    box = st.target_boxes(0)[0]
    g0 = gray(0)
    pin = api.PinnedBuffer(g0.size)
    pin.array[:] = g0
    trk.init(pin.array, api.BBox(*box))
    ref.init(np.repeat(g0.reshape(H, W, 1), 3, axis=2), box)
    for n in range(6):
        g = gray(n)
        rgb = np.ascontiguousarray(np.repeat(g.reshape(H, W, 1), 3, axis=2))
        before = ref.rect
        trk.set_rect(before)
        pin.array[:] = g
        r = trk.update(pin.array)
        rc, ok, score, bb = ref.update(rgb)
        assert rc == 0 and r.success == ok and abs(r.score - score) <= SCORE_TOL, (n, r, ok, score)
        sb, _ = ref.last_blobs()
        assert np.array_equal(np.asarray(trk.debug_read(0)["search_blob"]).reshape(-1), np.asarray(sb).reshape(-1)), n
        if tuple(r.bbox) == tuple(bb) and ok and score > 0.25:
            want = np.concatenate([g, np.zeros(W * H // 2, np.uint8)])  # the oracle's NV12 drawing code on a bare luma plane
            x, y, w, h = bb
            oracle.draw_rect_nv12(want, W, H, x, y, w, h, 3, 255)
            oracle.draw_crosshair_nv12(want, W, H, x + w // 2, y + h // 2, 15, 255)
            assert np.array_equal(pin.array, want[:W * H]), n
    # pageable frames and the explicit overlay entry point work on the luma plane too
    fr = gray(2).copy()
    want = np.concatenate([fr, np.zeros(W * H // 2, np.uint8)])
    trk.overlay(fr, [api.overlay_cmd(api.L.VT_OV_RECT, 100, 80, 60, 40, 3, 200)])
    oracle.draw_rect_nv12(want, W, H, 100, 80, 60, 40, 3, 200)
    assert np.array_equal(fr, want[:W * H])


def test_live_handles_are_counted_across_processes(api, weight_dir):
    """The latency / throughput form switch counts tracker handles per GPU, not per process (one process per stream under torchrun, one
    pipeline per camera process): handles of other processes are seen, and the slot of a process that died without destroying its
    handle is reclaimed."""
    import gc
    import subprocess
    import sys
    gc.collect()
    w = weights.ensure_weight_file("nano", weight_dir)
    trk = api.VitTrack.new(w, 640, 360)
    base = trk.model_dim(5)
    assert base >= 1
    child = ("import sys; sys.path.insert(0, %r)\nfrom gstreamer_vit_tracker_b200 import api\n"
             "t = api.VitTrack.new(%r, 640, 360)\nprint('up', flush=True)\nsys.stdin.readline()\n") % (ROOT, w)
    procs = [subprocess.Popen([sys.executable, "-c", child], stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True) for _ in range(2)]
    try:
        for p in procs:
            assert p.stdout.readline().strip() == "up"
        assert trk.model_dim(5) == base + 2
        procs[0].stdin.write("\n")
        procs[0].stdin.flush()
        procs[0].wait(timeout=60)              # clean exit: the handle is destroyed
        procs[1].kill()                        # no destructor runs
        procs[1].wait(timeout=60)
        t2 = api.VitTrack.new(w, 640, 360)     # creating a handle sweeps the slots of dead processes
        assert trk.model_dim(5) == base + 1
        t2.close()
        assert trk.model_dim(5) == base
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()


def test_kernel_forms_agree(api, weight_dir, monkeypatch):
    """The latency-mode "spread" forms (used while <= 2 handles are alive on the GPU: FC1 tile computed by three CTAs with one
    64-column slice of the chained FC2 product each, proj folded into the attention kernel, hi / lo replicas of the QKV scatter), the
    plain chained forms and the unchained FC1 / FC2 GEMMs (>= 8 targets) are re-associations of the same sums: boxes equal, scores
    within 1e-5 of each other over a sequence (parity bar: 1e-3).  One and two targets per handle (different forms qualify)."""
    import gc
    gc.collect()  # handles of earlier tests would count as live streams
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    spec1 = synth.CONFIGS["cfg1"]
    spec2 = synth.StreamSpec("two", 1920, 1080, 1005, [(400, 300, 140, 100, 4, 2), (1300, 600, 120, 160, -3, 3)])
    for spec in (spec1, spec2):
        st = synth.SyntheticStream(spec)
        nt = len(spec.targets)
        frames = [np.ascontiguousarray(st.frame(i)).reshape(-1) for i in range(6)]

        def run(env):
            for k in ("VT_B200_NO_SPREAD", "VT_B200_UNCHAIN_N", "VT_B200_NO_ATT_CHAIN"):
                monkeypatch.delenv(k, raising=False)
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            trk = api.VitTrack.new(w, spec.width, spec.height, gemm_mode=1, max_targets=nt)
            for k, b in enumerate(st.target_boxes(0)):
                trk.init(frames[0], api.BBox(*b), target=k)
            out = [trk.update_all(f) for f in frames[1:]]
            trk.close()
            return out

        ref = run({"VT_B200_NO_SPREAD": "1"})
        for env in ({}, {"VT_B200_NO_ATT_CHAIN": "1"}, {"VT_B200_UNCHAIN_N": "1"}):
            got = run(env)
            for fa, fb in zip(got, ref):
                for a, b in zip(fa, fb):
                    assert a.success and a.status == 0 and a.bbox == b.bbox, (spec.name, env, a, b)
                    assert abs(a.score - b.score) < 1e-5, (spec.name, env, a, b)


@pytest.mark.parametrize("gemm_mode", [1, 2, 3], ids=["tcgen05x3", "tcgen05", "tcgen05fp16"])
def test_throughput_gemm_forms_bit_identical(api, weight_dir, monkeypatch, gemm_mode):
    """The throughput forms that run from 1024 rows on (cfg4 / stream groups: QKV and FC1 in the A-stationary kernel of gemm_as.cu)
    add the same products in the same order as the one-tile kernels: forced onto a 2-target handle (640 rows, 5 row tiles with a
    ragged last one), scores and boxes must be IDENTICAL."""
    import gc
    gc.collect()
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    spec = synth.StreamSpec("two", 1920, 1080, 1005, [(400, 300, 140, 100, 4, 2), (1300, 600, 120, 160, -3, 3)])
    st = synth.SyntheticStream(spec)
    frames = [np.ascontiguousarray(st.frame(i)).reshape(-1) for i in range(5)]

    def run(env):
        for k in ("VT_B200_NO_SPREAD", "VT_B200_UNCHAIN_N", "VT_B200_AS_ROWS", "VT_B200_NO_AS_MLP", "VT_B200_AS_SPLIT"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        trk = api.VitTrack.new(w, spec.width, spec.height, gemm_mode=gemm_mode, max_targets=2)
        for k, b in enumerate(st.target_boxes(0)):
            trk.init(frames[0], api.BBox(*b), target=k)
        out = [trk.update_all(f) for f in frames[1:]]
        trk.close()
        return out

    base = {"VT_B200_NO_SPREAD": "1", "VT_B200_UNCHAIN_N": "1"}
    ref = run(dict(base, VT_B200_AS_ROWS="0"))
    got = run(dict(base, VT_B200_AS_ROWS="1", VT_B200_NO_AS_MLP="1"))
    for fa, fb in zip(got, ref):
        for a, b in zip(fa, fb):
            assert a.success and a.status == 0, a
            assert a.bbox == b.bbox and a.score == b.score, (a, b)
    # the chained A-stationary MLP (hidden tile in tensor memory, chained product accumulated over a CTA's hidden chunks) re-associates
    # the FC2 sum: same boxes, scores within 1e-5 (bf16x3 only; the other operand modes keep FC1 / FC2 as separate GEMMs)
    got = run(dict(base, VT_B200_AS_ROWS="1"))
    for fa, fb in zip(got, ref):
        for a, b in zip(fa, fb):
            assert a.success and a.status == 0 and a.bbox == b.bbox, (a, b)
            assert abs(a.score - b.score) < 1e-5, (a, b)
    # three CTAs per row tile (what 5120 rows get on 148 SMs): three partial planes per row tile for reduce_ln_kernel
    if gemm_mode == 1:
        planes = run(dict(base, VT_B200_AS_ROWS="1", VT_B200_AS_SPLIT="3"))
        for fa, fb in zip(planes, ref):
            for a, b in zip(fa, fb):
                assert a.success and a.status == 0 and a.bbox == b.bbox, (a, b)
                assert abs(a.score - b.score) < 1e-5, (a, b)


@pytest.mark.parametrize("upload_window", [True, False], ids=["windows", "whole"])
def test_stream_group_equals_independent_handles(api, weight_dir, upload_window):
    """vt_tracker_update_streams: 5 independent 1080p streams (cfg5 seeds) stepped together through one batched forward (1600 rows: the
    many-row GEMM forms) against 5 single-stream handles on the same frames: boxes equal, scores within 1e-5 (re-association of the FC2
    sum in the chained A-stationary MLP), and every stream's pinned frame carries exactly the overlay pixels its own handle draws."""
    import gc
    gc.collect()
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    G, steps = 5, 6
    streams = [synth.SyntheticStream(synth.cfg5_stream(i)) for i in range(G)]
    spec = streams[0].spec
    fb = streams[0].frame_bytes()
    grp = api.VitTrack.new(w, spec.width, spec.height, gemm_mode=1, max_targets=G, box_overlay=True, upload_window=upload_window)
    singles = [api.VitTrack.new(w, spec.width, spec.height, gemm_mode=1, box_overlay=True, upload_window=upload_window) for _ in range(G)]
    pin_g = [api.PinnedBuffer(fb) for _ in range(G)]
    pin_s = [api.PinnedBuffer(fb) for _ in range(G)]
    for i, st in enumerate(streams):
        f0 = np.ascontiguousarray(st.frame(0)).reshape(-1)
        box = api.BBox(*st.target_boxes(0)[0])
        grp.init(f0, box, target=i)
        singles[i].init(f0, box)
    for k in range(1, steps + 1):
        for i, st in enumerate(streams):
            f = np.ascontiguousarray(st.frame(k)).reshape(-1)
            pin_g[i].array[:] = f
            pin_s[i].array[:] = f
        got = grp.update_streams([p.array for p in pin_g])
        for i in range(G):
            ref = singles[i].update(pin_s[i].array)
            a = got[i]
            # (the group runs the many-row kernel forms, the single handles the one-tile forms: a pre-floor coordinate within ~1e-3 px of an
            # integer may land on the other side — the IoU >= 0.99 bar, never seen on these streams)
            assert a.status == 0 and a.success == ref.success and iou(a.bbox, ref.bbox) >= IOU_MIN, (k, i, a, ref)
            assert all(abs(p - q) <= 1 for p, q in zip(a.bbox, ref.bbox)), (k, i, a, ref)
            assert abs(a.score - ref.score) < 1e-5, (k, i, a, ref)
            if a.bbox == ref.bbox:
                assert np.array_equal(pin_g[i].array, pin_s[i].array), (k, i, "overlay pixels differ")
            else:
                singles[i].set_rect(a.bbox)  # keep the two trajectories on the same state
            assert not np.array_equal(pin_g[i].array, np.ascontiguousarray(streams[i].frame(k)).reshape(-1)), "no overlay was drawn"
    # argument checks: frame count, pageable frames
    with pytest.raises(Exception):
        grp.update_streams([p.array for p in pin_g[:3]])
    with pytest.raises(Exception):
        grp.update_streams([np.zeros(fb, np.uint8) for _ in range(G)])
    grp.close()
    for t in singles:
        t.close()
    for p in pin_g + pin_s:
        p.close()


# ---- SURVEY.md App. A.7 variant switches ----------------------------------------------------------------------------------------
def _quirk_norm():
    g = golden("trackervit_variants.json")
    return (g["norm_scale"], g["norm_bias"])


@pytest.mark.parametrize("gemm_mode", [0, 1], ids=["fp32simt", "tcgen05x3"])
@pytest.mark.parametrize("switch", ["pad_plus1", "decode_window", "window", "norm", "all"])
def test_variant_switch_vs_oracle(api, oracle, weight_dir, switch, gemm_mode):
    """One GPU-vs-oracle test per App. A.7 switch in vt_config (and all of them together): 12 teacher-forced frames of a target whose
    search window overhangs the right and bottom frame edges (so pad_plus1 matters), blobs bit-exact, score within 1e-3, boxes equal."""
    kw = {"pad_plus1": dict(pad_plus1=True), "decode_window": dict(decode_window=1), "window": dict(window=1), "norm": dict(norm=_quirk_norm()),
          "all": dict(pad_plus1=True, decode_window=1, window=1, norm=_quirk_norm())}[switch]
    W, H = 640, 360
    spec = synth.StreamSpec("v", W, H, 77, [(560, 300, 80, 60, 2, 1)])
    st = synth.SyntheticStream(spec)
    wpath = weights.ensure_weight_file("nano", weight_dir, variant="wild")
    trk = api.VitTrack.new(wpath, W, H, gemm_mode=gemm_mode, **kw)
    ref = oracle.VitTrack(wpath, threads=4)
    ref.set_variant(**kw)
    base = oracle.VitTrack(wpath, threads=4)   # default variant: the switch must actually change something
    f0 = st.frame(0)
    rgb0 = oracle.nv12_to_rgb(f0, W, H, 4)
    box = st.target_boxes(0)[0]
    trk.init(f0, api.BBox(*box))
    ref.init(rgb0, box)
    base.init(rgb0, box)
    stats = new_stats()
    changed = False
    for n in range(12):
        fr = st.frame(n)
        rgb = oracle.nv12_to_rgb(fr, W, H, 4)
        before = ref.rect
        trk.set_rect(before)
        base.rect = before
        r = trk.update(fr)
        assert ref.update(rgb)[0] == 0 and base.update(rgb)[0] == 0
        sb, tb = ref.last_blobs()
        d = trk.debug_read(0)
        assert np.array_equal(d["search_blob"], sb) and np.array_equal(d["template_blob"], tb), (switch, n)
        compare_step(trk, r, ref, before, stats, (switch, n), decode_window=kw.get("decode_window", 0))
        changed |= (not np.array_equal(base.last_blobs()[0], sb)) or (not np.array_equal(base.last_maps()[0], ref.last_maps()[0])) or base.rect != ref.rect
    assert changed, "the switch changed nothing on this sequence"
    finish_stats(f"variant/{switch}/gemm{gemm_mode}", stats, 12)


def test_custom_norm_vs_cv2_default_std_golden(api, weight_dir):
    """vt_config.norm_custom against the third party: cv2.TrackerVit with its default stdvalue (Scalar-division quirk, SURVEY.md §8c)."""
    g = golden("trackervit_variants.json")
    wpath = weights.ensure_weight_file(g["model"], weight_dir, variant=g["variant"])
    assert hashlib.sha256(open(wpath, "rb").read()).hexdigest() == g["weights_sha256"]
    for seq in g["sequences"]:
        sp = seq["spec"]
        spec = synth.StreamSpec(seq["name"], sp["w"], sp["h"], sp["seed"], [tuple(t) for t in sp["targets"]])
        st = synth.SyntheticStream(spec)
        trk = api.VitTrack.new(wpath, spec.width, spec.height, gemm_mode=1, norm=(g["norm_scale"], g["norm_bias"]))
        trk.init(st.frame(0), api.BBox(*seq["init_box"]))
        for i, fr in enumerate(seq["frames"]):
            r = trk.update(st.frame(i))
            assert abs(r.score - fr["score"]) <= SCORE_TOL and r.success == fr["ok"], (seq["name"], i, r, fr)
            if fr["ok"] and list(r.bbox) != fr["bbox"]:
                assert max(abs(a - b) for a, b in zip(r.bbox, fr["bbox"])) <= 1, (seq["name"], i, r.bbox, fr["bbox"])
                trk.set_rect(fr["bbox"])


def test_config_struct_size_evolution(api, weight_dir):
    """vt_config.struct_size: a caller built against the v1 header (no App. A.7 fields) gets the defaults for what its struct lacks;
    0 and oversized values are rejected (ADVICE r1)."""
    import ctypes as C
    L = api.L
    wpath = weights.ensure_weight_file("nano", weight_dir)
    cfg = api.make_config(wpath, 640, 360, pad_plus1=True, window=1)   # v2 fields set ...
    cfg.struct_size = L.vt_config.pad_plus1.offset                     # ... but the caller claims the v1 size: they must be ignored
    h = C.c_void_p()
    api.check(L.lib().vt_tracker_create(C.byref(cfg), C.byref(h)), "create v1-sized")
    a = api.VitTrack(cfg, _handle=h)
    b = api.VitTrack.new(wpath, 640, 360)
    st = synth.SyntheticStream(synth.StreamSpec("v", 640, 360, 77, [(560, 300, 80, 60, 2, 1)]))
    for t in (a, b):
        t.init(st.frame(0), api.BBox(*st.target_boxes(0)[0]))
    assert a.update(st.frame(1)) == b.update(st.frame(1))
    for bad in (0, C.sizeof(L.vt_config) + 8, 12):
        cfg.struct_size = bad
        h2 = C.c_void_p()
        assert L.lib().vt_tracker_create(C.byref(cfg), C.byref(h2)) == L.VT_ERR_INVALID and not h2.value


def test_one_process_two_devices(api, weight_dir):
    """One process driving two GPUs (cfg.device): a handle per device, the same stream on both, driven alternately and from two threads —
    results identical to each other (same kernels, same forms: one handle per GPU).  Skipped on a single-GPU box."""
    import threading

    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    w = weights.ensure_weight_file("tiny", weight_dir)
    spec = synth.CONFIGS["cfg1"]
    st = synth.SyntheticStream(spec)
    frames = [np.ascontiguousarray(st.frame(i)).reshape(-1) for i in range(8)]
    trks = [api.VitTrack.new(w, spec.width, spec.height, device=d, box_overlay=True) for d in (0, 1)]
    for t in trks:
        t.init(frames[0].copy(), api.BBox(*st.target_boxes(0)[0]))
    outs = [[], []]
    for f in frames[1:4]:                       # alternately from one thread
        for d, t in enumerate(trks):
            outs[d].append(t.update(f.copy()))

    def worker(d):                              # concurrently from two threads
        for f in frames[4:]:
            outs[d].append(trks[d].update(f.copy()))
    th = [threading.Thread(target=worker, args=(d,)) for d in (0, 1)]
    [x.start() for x in th]
    [x.join() for x in th]
    for a, b in zip(*outs):
        assert a.success and a.bbox == b.bbox and a.score == b.score, (a, b)
    for t in trks:
        t.close()


def test_zz_parity_stats_recorded():
    """Last test of the file: the tie / boundary / |dscore| counts of every sequence above go to gpurun_out/parity_stats.json (the
    numbers behind the 1e-3 / IoU claims survive `pytest -q`), and the global bounds hold over everything that ran."""
    if not PARITY_STATS:
        pytest.skip("no parity sequence ran in this session")
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    tot = {"frames": 0, "exact": 0, "boundary": 0, "ties": 0, "max_dscore": 0.0}
    for name, stt in PARITY_STATS.items():
        if "gemm3" in name:
            continue  # opt-in fp16 mode: recorded, not part of the default-path totals
        tot["frames"] += stt["frames"]
        tot["exact"] += stt["exact"]
        tot["boundary"] += stt.get("boundary", 0)
        tot["ties"] += stt.get("ties", 0)
        tot["max_dscore"] = max(tot["max_dscore"], stt["max_dscore"])
    with open(os.path.join(out, "parity_stats.json"), "w") as f:
        json.dump({"bars": {"score_tol": SCORE_TOL, "tie_margin": TIE_MARGIN, "boundary_px": BOUNDARY_PX, "exempt_frac": EXEMPT_FRAC},
                   "total_default_paths": tot, "sequences": PARITY_STATS}, f, indent=1, sort_keys=True)
    assert tot["max_dscore"] <= SCORE_TOL
    assert tot["ties"] + tot["boundary"] <= EXEMPT_FRAC * tot["frames"], tot
