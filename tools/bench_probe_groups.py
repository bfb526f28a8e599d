#!/usr/bin/env python
"""Probe groups (GPU only): 16 cameras probed with the full probe (state machine, HUD, box) on one GPU, served four ways:

  independent:  16 x 1920x1080 NV12 as 16 vt_context probes (vt_context_run_ring), one host thread each;
  group16:      the same 16 cameras as one probe group (vt_probe_group_run_ring), one host thread;
  group4x4:     the same 16 cameras as 4 probe groups of 4, one host thread per group;
  mixed16:      8 x 1920x1080 NV12 + 8 x 640x512 YUY2 as one probe group of 16.

Every probe is in TRACKING before the timed steps (the selection is scripted through the context commands); pinned rings of 8 frames
per camera with pristine restore (each probe draws on clean frames); tiny model, bf16x3, upload_window on.  Reported per layout:
streams x frames/s over the timed window, and p50 / p99 of the step latency (one vt_probe_group_frame, resp. one vt_probe_frame).  The
card's name, power limit and SM clocks are read (nvidia-smi --query-gpu, read-only) in the same run.  Writes <out>/bench_probe_groups.json
and prints one JSON line.

    python tools/bench_probe_groups.py --out DIR [--steps 200] [--warmup 20]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gstreamer_vit_tracker_b200 import api, synth, weights  # noqa: E402

RING = 8
HUD = ("FPS: 60", "conv:0.1ms trk:0.5ms")


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


STRIDE = 1920 * 1080 * 3 // 2  # one ring stride for every camera: a group steps all its rings with one stride


class Camera:
    """a pinned ring of RING packed frames, STRIDE apart (+ its pristine copy), and the target's box in frame 0"""

    def __init__(self, fmt, W, H, st):
        frames = [np.ascontiguousarray(st.frame(n)).reshape(-1) if fmt == "nv12" else synth.rgb_to_yuy2(st.frame_rgb(n)) for n in range(RING)]
        self.fmt, self.W, self.H, self.nbytes = fmt, W, H, frames[0].size
        self.ring, self.clean = api.PinnedBuffer(STRIDE * RING), api.PinnedBuffer(STRIDE * RING)
        for k, f in enumerate(frames):
            self.ring.array[k * STRIDE:k * STRIDE + self.nbytes] = f
        self.clean.array[:] = self.ring.array
        self.box = st.target_boxes(0)[0]

    def frame(self, k):
        return self.ring.array[k * STRIDE:k * STRIDE + self.nbytes]


def cameras(n_vis, n_ir):
    cams = [Camera("nv12", 1920, 1080, synth.SyntheticStream(synth.cfg5_stream(i))) for i in range(n_vis)]
    c3 = synth.CONFIGS["cfg3"]
    for i in range(n_ir):
        st = synth.SyntheticStream(synth.StreamSpec(f"ir{i}", c3.width, c3.height, c3.seed + 100 * i, c3.targets, fmt="rgb24"))
        cams.append(Camera("yuy2", c3.width, c3.height, st))
    return cams


def select_commands(ctx, cam):
    """steps 0..2 of a scripted selection of the target: cursor to its top-left corner + confirm, drag, confirm (init + update)"""
    U = api.UserCommand
    x, y, w, h = cam.box

    def moves(d, neg, pos):
        c = neg if d < 0 else pos
        return [(c, True)] * (abs(d) // 50) + [(c, False)] * ((abs(d) % 50) // 10)

    return [moves(x - cam.W // 2, U.MoveLeft, U.MoveRight) + moves(y - cam.H // 2, U.MoveUp, U.MoveDown) + [(U.Confirm, False)],
            moves(w, U.MoveLeft, U.MoveRight) + moves(h, U.MoveUp, U.MoveDown), [(U.Confirm, False)]]


def start_group(wpath, cams):
    g = api.ProbeGroup.new(wpath, [(c.W, c.H, c.fmt) for c in cams], gemm_mode=1, upload_window=True)
    scripts = [select_commands(ctx, c) for ctx, c in zip(g.contexts, cams)]
    for s in range(3):
        for ctx, sc in zip(g.contexts, scripts):
            for cmd, fast in sc[s]:
                ctx.handle_command(cmd, fast)
        g.probe([c.frame(s) for c in cams], HUD)
    for c in cams:
        c.ring.array[:] = c.clean.array
    return g


def start_context(wpath, cam):
    ctx = api.TrackerContext.new(wpath, cam.W, cam.H, fmt=cam.fmt, gemm_mode=1, upload_window=True)
    for s, cmds in enumerate(select_commands(ctx, cam)):
        for cmd, fast in cmds:
            ctx.handle_command(cmd, fast)
        ctx.probe(cam.frame(s), HUD)
    cam.ring.array[:] = cam.clean.array
    return ctx


def run_threads(jobs, steps, warmup):
    """jobs: callables job(first, n) -> per-step latencies (us); one thread each; returns (wall s of the timed steps, latencies)"""
    lat = [None] * len(jobs)
    for j in jobs:
        j(3, warmup)
    barrier = threading.Barrier(len(jobs) + 1)

    def work(k):
        barrier.wait()
        lat[k] = jobs[k](3 + warmup, steps)

    th = [threading.Thread(target=work, args=(k,)) for k in range(len(jobs))]
    for t in th:
        t.start()
    barrier.wait()
    t0 = time.perf_counter()
    for t in th:
        t.join()
    return time.perf_counter() - t0, np.concatenate(lat)


def layout(name, wpath, cams, groups, steps, warmup):
    """groups: None = one vt_context per camera; else a list of camera index lists, one probe group each"""
    if groups is None:
        handles = [start_context(wpath, c) for c in cams]
        jobs = [(lambda first, n, h=h, c=c: h.run_ring(c.ring.array.ctypes.data, STRIDE, c.nbytes, RING, first, n, HUD, c.clean.array.ctypes.data,
                                                       want_latency=True)) for h, c in zip(handles, cams)]
        tracking = sum(h.state_name() == "TRACKING" for h in handles)
    else:
        handles = [start_group(wpath, [cams[i] for i in idx]) for idx in groups]
        jobs = []
        for h, idx in zip(handles, groups):
            cs = [cams[i] for i in idx]
            jobs.append(lambda first, n, h=h, cs=cs: h.run_ring([c.ring.array.ctypes.data for c in cs], STRIDE,
                                                                 max(c.nbytes for c in cs), RING, first, n, HUD,
                                                                 [c.clean.array.ctypes.data for c in cs], want_latency=True))
        tracking = sum(c.state_name() == "TRACKING" for h in handles for c in h.contexts)
    wall, lat = run_threads(jobs, steps, warmup)
    after = (sum(h.state_name() == "TRACKING" for h in handles) if groups is None else
             sum(c.state_name() == "TRACKING" for h in handles for c in h.contexts))
    for h in handles:
        h.close()
    return {"layout": name, "streams": len(cams), "handles": len(handles), "tracking_before": int(tracking), "tracking_after": int(after),
            "stream_fps": round(len(cams) * steps / wall, 1), "step_p50_us": round(float(np.percentile(lat, 50)), 1),
            "step_p99_us": round(float(np.percentile(lat, 99)), 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    wpath = weights.ensure_weight_file("tiny", os.path.join(tempfile.gettempdir(), "vt_b200_weights"))
    vis = cameras(16, 0)
    res = {"gpu": gpu_info(), "model": "tiny", "gemm": "bf16x3", "steps": a.steps, "warmup": a.warmup, "ring": RING, "layouts": []}
    res["layouts"].append(layout("independent", wpath, vis, None, a.steps, a.warmup))
    res["layouts"].append(layout("group16", wpath, vis, [list(range(16))], a.steps, a.warmup))
    res["layouts"].append(layout("group4x4", wpath, vis, [list(range(4 * k, 4 * k + 4)) for k in range(4)], a.steps, a.warmup))
    mixed = cameras(8, 8)
    res["layouts"].append(layout("mixed16", wpath, mixed, [list(range(16))], a.steps, a.warmup))
    res["gpu_after"] = gpu_info()
    with open(os.path.join(a.out, "bench_probe_groups.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
