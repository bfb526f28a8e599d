#!/usr/bin/env python
"""32-bit RGBA / BGRA frames against the formats a pipeline would otherwise convert them to (GPU only), on the cfg2 scene (1920x1080, one
target, tiny model, bf16x3), arms alternated over --rounds rounds in one process:

  update_surface:  vt_tracker_update_surface (box overlay on) on RGBA surfaces laid out as a DeepStream RGBA NvBufSurface (pitch 7936)
                   against NV12 surfaces of the same frames laid out as NVDEC's (pitch 2048, chroma at row 1088).
  probe_surface:   vt_probe_frame_surface, the probe in TRACKING, on the same two surface layouts.
  probe_pinned:    vt_probe_frame with upload_window = 1 on pinned BGRA frames (GStreamer BGRx) against pinned RGB24 frames.

Every arm runs the same Python loop over a ring of RING frames; after each timed call the drawn frame is restored from its clean copy
outside the timed region.  Reported per arm: calls/s over the summed timed calls, p50 / p99 call latency, H2D / D2H bytes per call from
vt_timing, and (update arms) the share of successful results.  The probes must stay in TRACKING.  The card's name, power limit and SM
clocks are read (nvidia-smi --query-gpu, read-only) in the same run.  Writes <out>/bench_rgba.json and prints one JSON line.

    python tools/bench_rgba.py --out DIR [--steps 300] [--warmup 30] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gstreamer_vit_tracker_b200 import api, synth, weights  # noqa: E402

RING = 8
HUD = ("FPS: 60", "conv:0.1ms trk:0.5ms")
PITCH = {"nv12": 2048, "rgba": 7936}  # NVDEC's 1080p NV12 surface (chroma after 1088 rows); a DeepStream 1080p RGBA surface
CHROMA_ROW = 1088


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def packed(fmt, rgb, n):
    """frame n of the scene in `fmt` (4-byte formats: a random byte 3, as RGBx / BGRx padding may hold)"""
    if fmt == "nv12":
        return synth.rgb_to_nv12(rgb)
    if fmt == "rgb24":
        return np.ascontiguousarray(rgb).reshape(-1)
    pad = synth.hash_u8(77 + n, rgb.shape[:2])
    return synth.rgb_to_rgba(rgb, pad) if fmt == "rgba" else synth.rgb_to_bgra(rgb, pad)


class Ring:
    """RING frames of the cfg2 scene in one format, as pinned host frames or as device surfaces, each with a clean copy"""

    def __init__(self, fmt, surface):
        import torch

        spec = synth.CONFIGS["cfg2"]
        st = synth.SyntheticStream(synth.StreamSpec(spec.name, spec.width, spec.height, spec.seed, spec.targets, fmt="rgb24"))
        self.fmt, self.surface, self.W, self.H, self.box = fmt, surface, spec.width, spec.height, st.target_boxes(0)[0]
        self.clean = [packed(fmt, st.frame_rgb(n), n) for n in range(RING)]
        if surface:
            self.surfs = [api.PitchedFrame(self.W, self.H, fmt, pitch=PITCH[fmt], chroma_row=CHROMA_ROW if fmt == "nv12" else None) for _ in range(RING)]
            for s, f in zip(self.surfs, self.clean):
                s.write(f)
            self.dclean = [s.buf.clone() for s in self.surfs]
            torch.cuda.synchronize()
        else:
            self.pins = [api.PinnedBuffer(self.clean[0].size) for _ in range(RING)]
            for p, f in zip(self.pins, self.clean):
                p.array[:] = f

    def frame(self, k):
        return self.surfs[k].surface if self.surface else self.pins[k].array

    def restore(self, k):
        import torch

        if self.surface:
            self.surfs[k].buf.copy_(self.dclean[k])
            torch.cuda.synchronize()
        else:
            self.pins[k].array[:] = self.clean[k]


def select_commands(r):
    """steps 0..2 of a scripted selection of the target: cursor to its top-left corner + confirm, drag, confirm (init + update)"""
    U = api.UserCommand
    x, y, w, h = r.box

    def moves(d, neg, pos):
        c = neg if d < 0 else pos
        return [(c, True)] * (abs(d) // 50) + [(c, False)] * ((abs(d) % 50) // 10)

    return [moves(x - r.W // 2, U.MoveLeft, U.MoveRight) + moves(y - r.H // 2, U.MoveUp, U.MoveDown) + [(U.Confirm, False)],
            moves(w, U.MoveLeft, U.MoveRight) + moves(h, U.MoveUp, U.MoveDown), [(U.Confirm, False)]]


class Arm:
    """kind "update": a tracker handle, vt_tracker_update_surface; kind "probe": a context, vt_probe_frame[_surface]"""

    def __init__(self, wpath, kind, fmt, surface):
        self.kind, self.ring = kind, Ring(fmt, surface)
        r = self.ring
        kw = dict(gemm_mode=1, upload_window=not surface)
        self.ok = 0
        if kind == "update":
            self.h = api.VitTrack.new(wpath, r.W, r.H, fmt=fmt, box_overlay=True, **kw)
            self.tracker = self.h
            self.h.init(r.clean[0], api.BBox(*r.box))
        else:
            self.h = api.TrackerContext.new(wpath, r.W, r.H, fmt=fmt, **kw)
            self.tracker = self.h.tracker
            for s in range(3):
                for cmd, fast in select_commands(r)[s]:
                    self.h.handle_command(cmd, fast)
                self.call(s)
                r.restore(s)

    def call(self, k):
        f = self.ring.frame(k)
        if self.kind == "update":
            self.ok += int(self.h.update_surface(f)[0].success)
        elif self.ring.surface:
            self.h.probe_surface(f, HUD)
        else:
            self.h.probe(f, HUD)

    def tracking(self):
        return self.kind == "update" or self.h.state_name() == "TRACKING"

    def run(self, first, n):
        """n timed calls; returns the latencies (us), and the H2D / D2H bytes they moved"""
        t0 = self.tracker.timing()
        lat = np.empty(n)
        for i in range(n):
            k = (first + i) % RING
            a = time.perf_counter()
            self.call(k)
            lat[i] = (time.perf_counter() - a) * 1e6
            self.ring.restore(k)
            assert self.tracking(), "a probe left TRACKING"
        t1 = self.tracker.timing()
        return lat, t1.h2d_bytes - t0.h2d_bytes, t1.d2h_bytes - t0.d2h_bytes


def compare(name, arms, steps, warmup, rounds):
    assert all(a.tracking() for a in arms.values()), "a probe is not TRACKING after its selection"
    acc = {k: {"lat": [], "h2d": 0, "d2h": 0, "calls": 0} for k in arms}
    first = 3
    for a in arms.values():
        a.run(first, warmup)
        a.ok = 0
    first += warmup
    keys = list(arms)
    for r in range(rounds):
        for k in (keys if r % 2 == 0 else keys[::-1]):
            lat, h2d, d2h = arms[k].run(first, steps)
            acc[k]["lat"].append(lat)
            acc[k]["h2d"] += h2d
            acc[k]["d2h"] += d2h
            acc[k]["calls"] += steps
        first += steps
    out = {"case": name}
    for k, v in acc.items():
        lat = np.concatenate(v["lat"])
        out[k] = {"calls_per_s": round(len(lat) / (lat.sum() * 1e-6), 1), "p50_us": round(float(np.percentile(lat, 50)), 1),
                  "p99_us": round(float(np.percentile(lat, 99)), 1), "round_calls_per_s": [round(len(x) / (x.sum() * 1e-6), 1) for x in v["lat"]],
                  "h2d_bytes_per_call": v["h2d"] / v["calls"], "d2h_bytes_per_call": v["d2h"] / v["calls"]}
        if arms[k].kind == "update":
            out[k]["success_share"] = round(arms[k].ok / v["calls"], 3)
    for a in arms.values():
        a.h.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    wpath = weights.ensure_weight_file("tiny", os.path.join(tempfile.gettempdir(), "vt_b200_weights"))
    res = {"gpu": gpu_info(), "scene": "cfg2", "model": "tiny", "gemm": "bf16x3", "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
           "ring": RING, "surface_pitch": PITCH, "nv12_chroma_row": CHROMA_ROW, "cases": []}
    res["cases"].append(compare("update_surface", {"nv12": Arm(wpath, "update", "nv12", True), "rgba": Arm(wpath, "update", "rgba", True)},
                                a.steps, a.warmup, a.rounds))
    res["cases"].append(compare("probe_surface", {"nv12": Arm(wpath, "probe", "nv12", True), "rgba": Arm(wpath, "probe", "rgba", True)},
                                a.steps, a.warmup, a.rounds))
    res["cases"].append(compare("probe_pinned", {"rgb24": Arm(wpath, "probe", "rgb24", False), "bgra": Arm(wpath, "probe", "bgra", False)},
                                a.steps, a.warmup, a.rounds))
    res["gpu_after"] = gpu_info()
    with open(os.path.join(a.out, "bench_rgba.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
