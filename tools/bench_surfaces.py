#!/usr/bin/env python
"""Pitched device surfaces against the packed paths (GPU only).  Two measurements on one GPU, the arms alternated within one process:

  single: one cfg2 stream (1920x1080 NV12, tiny, bf16x3, box overlay): vt_tracker_update_surface on an NVDEC-like surface (pitch 2048,
          chroma after 1088 rows) against vt_tracker_update_device on packed frames — frames/s and p50 latency.
  groups: 64 cfg2-like streams (cfg5 seeds) as 4 groups of 16 on 4 host threads: vt_tracker_update_streams_surface on such surfaces
          against vt_tracker_update_streams on pinned frames with search-window uploads (as bench.py's cfg5 `grouped` leg) — streams x
          frames/s and host->device bytes per stream-step.

Both arms of a measurement go through the same Python calls (one ctypes call per frame / group step; the GIL is released during it).
Every frame of a ring is drawn into by the box overlay and replayed, in both arms alike.  The card's name, power limit and SM clocks are
read (nvidia-smi --query-gpu, read-only) in the same run.  Writes <out>/bench_surfaces.json.

    python tools/bench_surfaces.py --out DIR [--rounds 3] [--steps 600] [--group-steps 150]
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
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gstreamer_vit_tracker_b200 import api, synth, weights  # noqa: E402

RING = 8          # frames per stream ring
PITCH, CHROMA_ROW = 2048, 1088  # NVDEC output surface of a 1920x1080 stream


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def ring_frames(spec, n):
    st = synth.SyntheticStream(spec)
    return [np.ascontiguousarray(st.frame(i)).reshape(-1) for i in range(n)], api.BBox(*st.target_boxes(0)[0])


def single(wpath, rounds, steps, warm):
    spec = synth.CONFIGS["cfg2"]
    W, H = spec.width, spec.height
    frames, box = ring_frames(spec, RING)
    packed = torch.stack([torch.from_numpy(f) for f in frames]).cuda()
    surf = []
    for f in frames:
        pf = api.PitchedFrame(W, H, pitch=PITCH, chroma_row=CHROMA_ROW)
        pf.write(f)
        surf.append(pf)
    torch.cuda.synchronize()
    fb = frames[0].size
    # both handles alive for the whole measurement: the same latency / throughput kernel forms on both arms
    dev = api.VitTrack.new(wpath, W, H, gemm_mode=1, box_overlay=True)
    srf = api.VitTrack.new(wpath, W, H, gemm_mode=1, box_overlay=True)
    dev.init(frames[0].copy(), box)
    srf.init_surface(surf[0].surface, box)
    arms = {
        "update_device_packed": (dev, lambda i: dev.update_device(packed[i % RING].data_ptr(), fb)),
        "update_surface_pitch2048": (srf, lambda i: srf.update_surface(surf[i % RING].surface)),
    }
    res = {k: [] for k in arms}
    for name, (trk, fn) in arms.items():  # warm-up (graph capture, first launches)
        for i in range(warm):
            fn(i)
    for r in range(rounds):
        for name, (trk, fn) in arms.items():
            lat = np.empty(steps)
            t0 = time.perf_counter()
            for i in range(steps):
                a = time.perf_counter()
                fn(i)
                lat[i] = time.perf_counter() - a
            dt = time.perf_counter() - t0
            res[name].append({"fps": steps / dt, "p50_ms": float(np.percentile(lat, 50) * 1e3), "p99_ms": float(np.percentile(lat, 99) * 1e3)})
    dev.close()
    srf.close()
    return {"workload": "cfg2 1920x1080 NV12, tiny, bf16x3, box overlay, one synchronous call per frame", "steps_per_round": steps,
            "warmup": warm, "rounds": res}


def groups(wpath, rounds, steps, warm):
    G, NG = 16, 4
    specs = [synth.cfg5_stream(i) for i in range(G * NG)]
    W, H = specs[0].width, specs[0].height
    rings, boxes = [], []
    for sp in specs:
        f, b = ring_frames(sp, RING)
        rings.append(f)
        boxes.append(b)
    fb = rings[0][0].size
    pins = [api.PinnedBuffer(fb * RING) for _ in specs]
    for p, r in zip(pins, rings):
        p.array[:] = np.concatenate(r)
    surfs = []
    for r in rings:
        row = []
        for f in r:
            pf = api.PitchedFrame(W, H, pitch=PITCH, chroma_row=CHROMA_ROW)
            pf.write(f)
            row.append(pf)
        surfs.append(row)
    torch.cuda.synchronize()
    host_h = [api.VitTrack.new(wpath, W, H, gemm_mode=1, box_overlay=True, upload_window=True, max_targets=G) for _ in range(NG)]
    surf_h = [api.VitTrack.new(wpath, W, H, gemm_mode=1, box_overlay=True, max_targets=G) for _ in range(NG)]
    for g in range(NG):
        for k in range(G):
            s = g * G + k
            host_h[g].init(pins[s].array[:fb], boxes[s], target=k)
            surf_h[g].init_surface(surfs[s][0].surface, boxes[s], target=k)

    def host_step(g, i):
        host_h[g].update_streams([pins[g * G + k].array[(i % RING) * fb:(i % RING + 1) * fb] for k in range(G)])

    def surf_step(g, i):
        surf_h[g].update_streams_surface([surfs[g * G + k][i % RING].surface for k in range(G)])

    def run(step, n):
        lat = [None] * NG

        def worker(g):
            x = np.empty(n)
            for i in range(n):
                a = time.perf_counter()
                step(g, i)
                x[i] = time.perf_counter() - a
            lat[g] = x
        th = [threading.Thread(target=worker, args=(g,)) for g in range(NG)]
        t0 = time.perf_counter()
        [t.start() for t in th]
        [t.join() for t in th]
        return time.perf_counter() - t0, np.concatenate(lat)

    arms = {"update_streams_pinned_windows": (host_h, host_step), "update_streams_surface_pitch2048": (surf_h, surf_step)}
    for name, (hs, step) in arms.items():
        run(step, warm)
    res = {k: [] for k in arms}
    for r in range(rounds):
        for name, (hs, step) in arms.items():
            t0 = [h.timing() for h in hs]
            dt, lat = run(step, steps)
            t1 = [h.timing() for h in hs]
            h2d = sum(b.h2d_bytes - a.h2d_bytes for a, b in zip(t0, t1))
            res[name].append({"streams_x_fps": G * NG * steps / dt, "p50_step_ms": float(np.percentile(lat, 50) * 1e3),
                              "h2d_bytes_per_stream_step": h2d / (G * NG * steps)})
    for h in host_h + surf_h:
        h.close()
    for p in pins:
        p.close()
    return {"workload": f"{G * NG} cfg5 streams (1920x1080 NV12), tiny, bf16x3, box overlay; {NG} groups of {G}, one host thread per group",
            "steps_per_round": steps, "warmup": warm, "rounds": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--group-steps", type=int, default=150)
    ap.add_argument("--warmup", type=int, default=60)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_surfaces.py needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    wpath = weights.ensure_weight_file("tiny", os.path.join(tempfile.gettempdir(), "vt_b200_weights"))
    out = {"gpu_before": gpu_info()}
    out["single"] = single(wpath, a.rounds, a.steps, a.warmup)
    out["groups"] = groups(wpath, a.rounds, a.group_steps, max(4, a.warmup // 4))
    out["gpu_after"] = gpu_info()
    for part in ("single", "groups"):
        for arm, rs in out[part]["rounds"].items():
            key = "fps" if part == "single" else "streams_x_fps"
            v = [x[key] for x in rs]
            out[part].setdefault("summary", {})[arm] = {"median_" + key: float(np.median(v)), "min": min(v), "max": max(v)}
    with open(os.path.join(a.out, "bench_surfaces.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({p: out[p]["summary"] for p in ("single", "groups")}))


if __name__ == "__main__":
    main()
