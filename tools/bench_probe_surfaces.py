#!/usr/bin/env python
"""The drop-in probe on decoder surfaces against pinned host frames (GPU only), arms alternated over --rounds rounds in one process:

  single:  cfg2 (1920x1080 NV12, one target), tiny model, bf16x3, the probe in TRACKING.  Pinned arm: vt_probe_frame on a pinned ring
           with upload_window = 1 (as bench.py's e2e leg).  Surface arm: vt_probe_frame_surface on NVDEC-like surfaces (pitch 2048, chroma
           at row 1088) in device memory.
  group:   a probe group of 16 cfg2-like cameras (cfg5 streams), vt_probe_group_frame on pinned frames against
           vt_probe_group_frame_surface on surfaces of the same layout.

Both arms run the same Python loop over a ring of RING frames and treat their frames alike: after each timed call the drawn frame is
restored from its clean copy outside the timed region (numpy copy of the pinned frame; device-to-device copy of the surface).  Reported per
arm: calls/s over the summed timed calls, p50 / p99 call latency, and H2D / D2H bytes per call from vt_timing.  Every probe must stay in
TRACKING.  The card's name, power limit and SM clocks are read (nvidia-smi --query-gpu, read-only) in the same run.  Writes
<out>/bench_probe_surfaces.json and prints one JSON line.

    python tools/bench_probe_surfaces.py --out DIR [--steps 300] [--warmup 30] [--rounds 3]
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
PITCH, CHROMA_ROW = 2048, 1088  # NVDEC's 1080p NV12 surface: rows padded to 2048 bytes, chroma after 1088 rows


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


class Camera:
    """RING frames of one 1080p NV12 stream as a pinned ring and as NVDEC-like device surfaces, each with a clean copy"""

    def __init__(self, spec):
        import torch

        st = synth.SyntheticStream(spec)
        self.W, self.H, self.box = spec.width, spec.height, st.target_boxes(0)[0]
        frames = [np.ascontiguousarray(st.frame(n)).reshape(-1) for n in range(RING)]
        self.nbytes = frames[0].size
        self.pins = [api.PinnedBuffer(self.nbytes) for _ in range(RING)]
        for p, f in zip(self.pins, frames):
            p.array[:] = f
        self.clean = frames
        self.surfs = [api.PitchedFrame(self.W, self.H, "nv12", pitch=PITCH, chroma_row=CHROMA_ROW) for _ in range(RING)]
        for s, f in zip(self.surfs, frames):
            s.write(f)
        self.dclean = [s.buf.clone() for s in self.surfs]
        torch.cuda.synchronize()

    def restore(self, k, surface):
        if surface:
            self.surfs[k].buf.copy_(self.dclean[k])
        else:
            self.pins[k].array[:] = self.clean[k]


def select_commands(cam):
    """steps 0..2 of a scripted selection of the target: cursor to its top-left corner + confirm, drag, confirm (init + update)"""
    U = api.UserCommand
    x, y, w, h = cam.box

    def moves(d, neg, pos):
        c = neg if d < 0 else pos
        return [(c, True)] * (abs(d) // 50) + [(c, False)] * ((abs(d) % 50) // 10)

    return [moves(x - cam.W // 2, U.MoveLeft, U.MoveRight) + moves(y - cam.H // 2, U.MoveUp, U.MoveDown) + [(U.Confirm, False)],
            moves(w, U.MoveLeft, U.MoveRight) + moves(h, U.MoveUp, U.MoveDown), [(U.Confirm, False)]]


class Arm:
    """one probe (a context, or a group when len(cams) > 1) fed pinned frames or surfaces; step(k) probes ring frame k of every camera"""

    def __init__(self, wpath, cams, surface):
        self.cams, self.surface, self.group = cams, surface, len(cams) > 1
        kw = dict(gemm_mode=1, upload_window=True)
        self.h = api.ProbeGroup.new(wpath, [(c.W, c.H, "nv12") for c in cams], **kw) if self.group else api.TrackerContext.new(wpath, cams[0].W, cams[0].H, **kw)
        self.ctxs = self.h.contexts if self.group else [self.h]
        self.tracker = self.h.tracker
        for s in range(3):
            for ctx, c in zip(self.ctxs, cams):
                for cmd, fast in select_commands(c)[s]:
                    ctx.handle_command(cmd, fast)
            self.call(s)
        self.restore(0), self.restore(1), self.restore(2)

    def call(self, k):
        if self.group and self.surface:
            self.h.probe_surfaces([c.surfs[k].surface for c in self.cams], HUD)
        elif self.group:
            self.h.probe([c.pins[k].array for c in self.cams], HUD)
        elif self.surface:
            self.h.probe_surface(self.cams[0].surfs[k].surface, HUD)
        else:
            self.h.probe(self.cams[0].pins[k].array, HUD)

    def restore(self, k):
        import torch

        for c in self.cams:
            c.restore(k, self.surface)
        if self.surface:
            torch.cuda.synchronize()

    def tracking(self):
        return all(c.state_name() == "TRACKING" for c in self.ctxs)

    def run(self, first, n):
        """n timed calls; returns the latencies (us), and the H2D / D2H bytes they moved"""
        t0 = self.tracker.timing()
        lat = np.empty(n)
        for i in range(n):
            k = (first + i) % RING
            a = time.perf_counter()
            self.call(k)
            lat[i] = (time.perf_counter() - a) * 1e6
            self.restore(k)
            assert self.tracking(), "a probe left TRACKING"
        t1 = self.tracker.timing()
        return lat, t1.h2d_bytes - t0.h2d_bytes, t1.d2h_bytes - t0.d2h_bytes


def compare(name, wpath, cams, steps, warmup, rounds):
    arms = {"pinned": Arm(wpath, cams, False), "surface": Arm(wpath, cams, True)}
    assert all(a.tracking() for a in arms.values()), "a probe is not TRACKING after its selection"
    acc = {k: {"lat": [], "h2d": 0, "d2h": 0, "calls": 0} for k in arms}
    first = 3
    for k, a in arms.items():
        a.run(first, warmup)
    first += warmup
    for r in range(rounds):
        for k in (("pinned", "surface") if r % 2 == 0 else ("surface", "pinned")):
            lat, h2d, d2h = arms[k].run(first, steps)
            acc[k]["lat"].append(lat)
            acc[k]["h2d"] += h2d
            acc[k]["d2h"] += d2h
            acc[k]["calls"] += steps
        first += steps
    out = {"case": name, "streams": len(cams)}
    for k, v in acc.items():
        lat = np.concatenate(v["lat"])
        out[k] = {"calls_per_s": round(len(lat) / (lat.sum() * 1e-6), 1), "frames_per_s": round(len(lat) * len(cams) / (lat.sum() * 1e-6), 1),
                  "p50_us": round(float(np.percentile(lat, 50)), 1), "p99_us": round(float(np.percentile(lat, 99)), 1),
                  "round_calls_per_s": [round(len(x) / (x.sum() * 1e-6), 1) for x in v["lat"]],
                  "h2d_bytes_per_call": v["h2d"] / v["calls"], "d2h_bytes_per_call": v["d2h"] / v["calls"],
                  "tracking_after": arms[k].tracking()}
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
    res = {"gpu": gpu_info(), "model": "tiny", "gemm": "bf16x3", "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds, "ring": RING,
           "surface_layout": {"pitch": PITCH, "chroma_row": CHROMA_ROW}, "cases": []}
    res["cases"].append(compare("single_cfg2", wpath, [Camera(synth.CONFIGS["cfg2"])], a.steps, a.warmup, a.rounds))
    res["cases"].append(compare("group16_cfg5", wpath, [Camera(synth.cfg5_stream(i)) for i in range(16)], max(a.steps // 3, 20), a.warmup, a.rounds))
    res["gpu_after"] = gpu_info()
    with open(os.path.join(a.out, "bench_probe_surfaces.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
