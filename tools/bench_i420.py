#!/usr/bin/env python
"""Planar I420 frames against NV12 frames of the same scene (GPU only), on the cfg2 scene (1920x1080, one target per stream, tiny model,
bf16x3, pinned frames, upload_window = 1), arms alternated over --rounds rounds in one process:

  update:   vt_tracker_update (box overlay on) on I420 frames against NV12 frames.
  probe:    vt_probe_frame, the probe in TRACKING, on I420 frames against NV12 frames, and the path a software-decoder pipeline had before
            I420 was a format: a CPU repack of the I420 frame into a pinned NV12 frame inside the timed call, then vt_probe_frame on it.
  group16:  vt_tracker_update_streams of a 16-stream group (cfg5 streams 0..15, box overlay on) on I420 frames against NV12 frames.

Every arm runs the same Python loop over a ring of frames; after each timed call the drawn frame is restored from its clean copy outside
the timed region.  Reported per arm: calls/s over the summed timed calls, p50 / p99 call latency, the mean h2d_ms stage of vt_timing
(device-stamped: submit to crop start, the window uploads), and H2D bytes per call.  The probes must stay in TRACKING.  The card's name,
power limit and SM clocks are read (nvidia-smi --query-gpu, read-only) in the same run.  Writes <out>/bench_i420.json and prints one JSON
line.

    python tools/bench_i420.py --out DIR [--steps 300] [--warmup 30] [--rounds 3]
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
GROUP_RING = 4
HUD = ("FPS: 60", "conv:0.1ms trk:0.5ms")


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def packed(fmt, rgb):
    return synth.rgb_to_nv12(rgb) if fmt == "nv12" else synth.rgb_to_i420(rgb)


def repack_i420_to_nv12(src, dst, W, H):
    """the CPU conversion a pipeline without native I420 runs in front of the probe (videoconvert I420 -> NV12, even W and H)"""
    n, c = W * H, W * H // 4
    dst[:n] = src[:n]
    uv = dst[n:].reshape(c, 2)
    uv[:, 0] = src[n: n + c]
    uv[:, 1] = src[n + c: n + 2 * c]


class Ring:
    """`size` pinned frames of one stream in one format, each with a clean copy"""

    def __init__(self, spec, fmt, size):
        st = synth.SyntheticStream(synth.StreamSpec(spec.name, spec.width, spec.height, spec.seed, spec.targets, fmt="rgb24"))
        self.W, self.H, self.box, self.size = spec.width, spec.height, st.target_boxes(0)[0], size
        self.clean = [packed(fmt, st.frame_rgb(n)) for n in range(size)]
        self.pins = [api.PinnedBuffer(self.clean[0].size) for _ in range(size)]
        for p, f in zip(self.pins, self.clean):
            p.array[:] = f

    def restore(self, k):
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
    """kind "update": vt_tracker_update; "probe": vt_probe_frame; "repack": CPU I420 -> NV12 repack + vt_probe_frame on NV12;
    "group": vt_tracker_update_streams of 16 streams"""

    def __init__(self, wpath, kind, fmt):
        self.kind = kind
        kw = dict(gemm_mode=1, upload_window=True)
        self.ok = 0
        spec = synth.CONFIGS["cfg2"]
        if kind == "group":
            self.rings = [Ring(synth.cfg5_stream(i), fmt, GROUP_RING) for i in range(16)]
            r = self.rings[0]
            self.h = api.VitTrack.new(wpath, r.W, r.H, fmt=fmt, max_targets=16, box_overlay=True, **kw)
            self.tracker = self.h
            for i, s in enumerate(self.rings):
                self.h.init(s.clean[0], api.BBox(*s.box), target=i)
            return
        self.ring = Ring(spec, fmt, RING)
        r = self.ring
        if kind == "update":
            self.h = api.VitTrack.new(wpath, r.W, r.H, fmt=fmt, box_overlay=True, **kw)
            self.tracker = self.h
            self.h.init(r.clean[0], api.BBox(*r.box))
            return
        if kind == "repack":
            self.nv = api.PinnedBuffer(r.W * r.H * 3 // 2)
        self.h = api.TrackerContext.new(wpath, r.W, r.H, fmt="nv12" if kind == "repack" else fmt, **kw)
        self.tracker = self.h.tracker
        for s in range(3):
            for cmd, fast in select_commands(r)[s]:
                self.h.handle_command(cmd, fast)
            self.call(s)
            r.restore(s)

    @property
    def n(self):
        return GROUP_RING if self.kind == "group" else RING

    def call(self, k):
        if self.kind == "group":
            self.ok += sum(int(x.success) for x in self.h.update_streams([s.pins[k].array for s in self.rings]))
            return
        f = self.ring.pins[k].array
        if self.kind == "update":
            self.ok += int(self.h.update(f).success)
        elif self.kind == "repack":
            repack_i420_to_nv12(f, self.nv.array, self.ring.W, self.ring.H)
            self.h.probe(self.nv.array, HUD)
        else:
            self.h.probe(f, HUD)

    def restore(self, k):
        for r in (self.rings if self.kind == "group" else [self.ring]):
            r.restore(k)

    def tracking(self):
        return self.kind in ("update", "group") or self.h.state_name() == "TRACKING"

    def run(self, first, n):
        """n timed calls; returns the latencies (us), the h2d_ms stage of every call and the H2D bytes they moved"""
        t0 = self.tracker.timing()
        lat, h2d_ms = np.empty(n), np.empty(n)
        for i in range(n):
            k = (first + i) % self.n
            a = time.perf_counter()
            self.call(k)
            lat[i] = (time.perf_counter() - a) * 1e6
            h2d_ms[i] = self.tracker.timing().h2d_ms
            self.restore(k)
            assert self.tracking(), "a probe left TRACKING"
        return lat, h2d_ms, self.tracker.timing().h2d_bytes - t0.h2d_bytes


def compare(name, arms, steps, warmup, rounds):
    assert all(a.tracking() for a in arms.values()), "a probe is not TRACKING after its selection"
    acc = {k: {"lat": [], "h2d_ms": [], "h2d": 0, "calls": 0} for k in arms}
    first = 3
    for a in arms.values():
        a.run(first, warmup)
        a.ok = 0
    first += warmup
    keys = list(arms)
    for r in range(rounds):
        for k in (keys if r % 2 == 0 else keys[::-1]):
            lat, h2d_ms, h2d = arms[k].run(first, steps)
            acc[k]["lat"].append(lat)
            acc[k]["h2d_ms"].append(h2d_ms)
            acc[k]["h2d"] += h2d
            acc[k]["calls"] += steps
        first += steps
    out = {"case": name}
    for k, v in acc.items():
        lat = np.concatenate(v["lat"])
        out[k] = {"calls_per_s": round(len(lat) / (lat.sum() * 1e-6), 1), "p50_us": round(float(np.percentile(lat, 50)), 1),
                  "p99_us": round(float(np.percentile(lat, 99)), 1), "round_calls_per_s": [round(len(x) / (x.sum() * 1e-6), 1) for x in v["lat"]],
                  "mean_h2d_ms": round(float(np.concatenate(v["h2d_ms"]).mean()), 4), "h2d_bytes_per_call": v["h2d"] / v["calls"]}
        if arms[k].kind in ("update", "group"):
            out[k]["success_share"] = round(arms[k].ok / v["calls"] / (16 if arms[k].kind == "group" else 1), 3)
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
    res = {"gpu": gpu_info(), "scene": "cfg2", "model": "tiny", "gemm": "bf16x3", "upload_window": True, "frames": "pinned",
           "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds, "ring": RING, "group_ring": GROUP_RING, "cases": []}
    res["cases"].append(compare("update", {"nv12": Arm(wpath, "update", "nv12"), "i420": Arm(wpath, "update", "i420")},
                                a.steps, a.warmup, a.rounds))
    res["cases"].append(compare("probe", {"nv12": Arm(wpath, "probe", "nv12"), "i420": Arm(wpath, "probe", "i420"),
                                          "i420_cpu_repack_nv12": Arm(wpath, "repack", "i420")}, a.steps, a.warmup, a.rounds))
    res["cases"].append(compare("group16", {"nv12": Arm(wpath, "group", "nv12"), "i420": Arm(wpath, "group", "i420")},
                                max(a.steps // 3, 1), max(a.warmup // 3, 1), a.rounds))
    res["gpu_after"] = gpu_info()
    with open(os.path.join(a.out, "bench_i420.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
