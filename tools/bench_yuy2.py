#!/usr/bin/env python
"""YUY2 camera frames three ways on cfg3 (640x512, one 64x48 target, tiny, bf16x3, box overlay; GPU only), the arms alternated within
one process and every handle alive for the whole measurement (so all arms run the same kernel forms):

  yuy2_native:       the YUY2 frame tracked as it comes from the camera — vt_tracker_update on pinned frames with search-window uploads
                     (whole YUY2 words of the window), and vt_probe_frame (the probe of src/pipeline_ir.rs with the luma HUD, TRACKING)
  convert_then_rgb24: the path before native YUY2 tracking — vt_convert_yuy2_rgb (frame up, RGB down) into a pinned RGB frame, then
                     vt_tracker_update on it with search-window uploads
  rgb24:             RGB24 frames as bench.py's cfg3 leg (vt_tracker_update, pinned, search-window uploads)

Each arm prints one JSON line: frames/s and p50 latency of one synchronous call per frame (medians over the rounds), the host<->device
bytes per step (the handle's vt_timing counters), the mean device stage times of the handle, and the card's name and power limit read
(nvidia-smi --query-gpu, read-only) in the same run.

    python tools/bench_yuy2.py [--rounds 3] [--steps 600] [--warmup 60] [--out DIR]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gstreamer_vit_tracker_b200 import api, synth, weights  # noqa: E402
from gstreamer_vit_tracker_b200._lib import lib  # noqa: E402

RING = 8
HUD = ("FPS: 60", "conv:0.1ms trk:0.5ms")


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def stages(t):
    return {k: round(getattr(t, "avg_" + k), 4) for k in ("h2d_ms", "preprocess_ms", "vit_ms", "decode_ms", "overlay_ms", "d2h_ms", "total_ms")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--warmup", type=int, default=60)
    ap.add_argument("--out", default=None, help="also write the lines to DIR/bench_yuy2.jsonl")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_yuy2.py needs a CUDA device")
    spec = synth.CONFIGS["cfg3"]
    W, H = spec.width, spec.height
    st = synth.SyntheticStream(spec)
    box = api.BBox(*st.target_boxes(0)[0])
    rgb = [np.ascontiguousarray(st.frame_rgb(i)).reshape(-1) for i in range(RING)]
    yuy2 = [synth.rgb_to_yuy2(st.frame_rgb(i)) for i in range(RING)]
    yb, rb = yuy2[0].size, rgb[0].size
    wpath = weights.ensure_weight_file("tiny", os.path.join(tempfile.gettempdir(), "vt_b200_weights"))
    kw = dict(gemm_mode=1, box_overlay=True, upload_window=True)

    # pinned rings (the box overlay draws into them; every arm replays its ring alike)
    pin_y, pin_yp, pin_r = api.PinnedBuffer(yb * RING), api.PinnedBuffer(yb * RING), api.PinnedBuffer(rb * RING)
    pin_y.array[:], pin_yp.array[:], pin_r.array[:] = np.concatenate(yuy2), np.concatenate(yuy2), np.concatenate(rgb)
    pin_c = api.PinnedBuffer(rb)  # the converted frame of the convert arm
    ny = api.VitTrack.new(wpath, W, H, fmt="yuy2", **kw)
    cv = api.VitTrack.new(wpath, W, H, fmt="rgb24", **kw)
    r24 = api.VitTrack.new(wpath, W, H, fmt="rgb24", **kw)
    ny.init(yuy2[0], box)
    cv.init(rgb[0], box)
    r24.init(rgb[0], box)
    ctx = api.TrackerContext.new(wpath, W, H, fmt="yuy2", upload_window=True, gemm_mode=1)
    U = api.UserCommand
    ctx.handle_command(U.Confirm)
    ctx.probe(pin_yp.array[:yb], HUD)
    ctx.handle_command(U.MoveRight, True)
    ctx.handle_command(U.MoveDown, True)
    ctx.handle_command(U.Confirm)
    ctx.probe(pin_yp.array[yb:2 * yb], HUD)

    def ys(i):
        return pin_y.array[(i % RING) * yb:(i % RING + 1) * yb]

    def convert_update(i):
        src = ys(i)
        rc = lib().vt_convert_yuy2_rgb(cv._h, C.c_void_p(src.ctypes.data), yb, W, H, C.c_void_p(pin_c.array.ctypes.data))
        assert rc == 0, rc
        cv.update(pin_c.array)

    arms = {
        "yuy2_native/update": (ny, lambda i: ny.update(ys(i))),
        "yuy2_native/probe": (ctx.tracker, lambda i: ctx.probe(pin_yp.array[(i % RING) * yb:(i % RING + 1) * yb], HUD)),
        "convert_then_rgb24": (cv, convert_update),
        "rgb24": (r24, lambda i: r24.update(pin_r.array[(i % RING) * rb:(i % RING + 1) * rb])),
    }
    gpu = gpu_info()
    for name, (trk, fn) in arms.items():  # warm-up: graph capture, first launches
        for i in range(a.warmup):
            fn(i)
    res = {k: [] for k in arms}
    for _ in range(a.rounds):
        for name, (trk, fn) in arms.items():
            t0 = trk.timing()
            lat = np.empty(a.steps)
            s0 = time.perf_counter()
            for i in range(a.steps):
                x = time.perf_counter()
                fn(i)
                lat[i] = time.perf_counter() - x
            dt = time.perf_counter() - s0
            t1 = trk.timing()
            res[name].append({"fps": a.steps / dt, "p50_ms": float(np.percentile(lat, 50) * 1e3),
                              "h2d_bytes_per_step": (t1.h2d_bytes - t0.h2d_bytes) / a.steps,
                              "d2h_bytes_per_step": (t1.d2h_bytes - t0.d2h_bytes) / a.steps, "stages_ms": stages(t1)})
    probe_state = ctx.state_name()
    gpu_after = gpu_info()

    def summary(name):
        rs = res[name]
        return {"frames_per_s": round(float(np.median([r["fps"] for r in rs])), 1),
                "frames_per_s_min_max": [round(min(r["fps"] for r in rs), 1), round(max(r["fps"] for r in rs), 1)],
                "p50_latency_ms": round(float(np.median([r["p50_ms"] for r in rs])), 4),
                "h2d_bytes_per_step": int(round(rs[-1]["h2d_bytes_per_step"])), "d2h_bytes_per_step": int(round(rs[-1]["d2h_bytes_per_step"])),
                "stages_ms": rs[-1]["stages_ms"]}
    common = {"workload": "cfg3 640x512, one 64x48 target, tiny, bf16x3, box overlay, pinned frames, search-window upload",
              "steps_per_round": a.steps, "rounds": a.rounds, "warmup": a.warmup, "gpu": gpu, "gpu_after": gpu_after}
    lines = [
        dict(run="yuy2_native", update=summary("yuy2_native/update"), probe=dict(summary("yuy2_native/probe"), state=probe_state), **common),
        dict(run="convert_then_rgb24", **summary("convert_then_rgb24"), **common),
        dict(run="rgb24", **summary("rgb24"), **common),
    ]
    for ln in lines:
        print(json.dumps(ln))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bench_yuy2.jsonl"), "w") as f:
            f.write("".join(json.dumps(ln) + "\n" for ln in lines))
    for t in (ny, cv, r24):
        t.close()
    ctx.close()


if __name__ == "__main__":
    main()
