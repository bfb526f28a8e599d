#!/usr/bin/env python
"""Stream groups of mixed cameras (GPU only): 8 visible cameras (1920x1080 NV12, cfg5 seeds) and 8 IR cameras (640x512 YUY2, the cfg3
scene) on one GPU, served three ways, the arms alternated within one process:

  mixed:        one group of all 16 streams (vt_tracker_set_stream_geometry on the 8 IR slots), one host thread;
  two_uniform:  one group of the 8 NV12 streams and one of the 8 YUY2 streams, one host thread per group;
  independent:  16 single-stream handles, one host thread per handle.

Each layout is measured end to end (pinned host frames, upload_window on: vt_tracker_update_streams / vt_tracker_update) and
device-resident (pitched device surfaces: vt_tracker_update_streams_surface / vt_tracker_update_surface), tiny model, bf16x3, box
overlay, rings of 8 frames per stream replayed (the box overlay draws into them in every arm alike).  Reported: streams x frames/s.
The card's name, power limit and SM clocks are read (nvidia-smi --query-gpu, read-only) in the same run.  Writes
<out>/bench_mixed_groups.json and prints one JSON line.

    python tools/bench_mixed_groups.py --out DIR [--rounds 3] [--steps 150] [--warmup 15]
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

RING = 8
N_VIS = N_IR = 8
VIS = ("nv12", 1920, 1080)
IR = ("yuy2", 640, 512)


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def cameras():
    """[(geometry, ring of packed frames, box in frame 0)] — the 8 visible cameras, then the 8 IR cameras"""
    cams = []
    for i in range(N_VIS):
        st = synth.SyntheticStream(synth.cfg5_stream(i))
        cams.append((VIS, [np.ascontiguousarray(st.frame(n)).reshape(-1) for n in range(RING)], api.BBox(*st.target_boxes(0)[0])))
    c3 = synth.CONFIGS["cfg3"]
    for i in range(N_IR):
        st = synth.SyntheticStream(synth.StreamSpec(f"ir{i}", c3.width, c3.height, c3.seed + 100 * i, c3.targets, fmt="rgb24"))
        cams.append((IR, [synth.rgb_to_yuy2(st.frame_rgb(n)) for n in range(RING)], api.BBox(*st.target_boxes(0)[0])))
    return cams


def new_group(wpath, geoms, **kw):
    fmt, W, H = geoms[0]
    t = api.VitTrack.new(wpath, W, H, fmt=fmt, gemm_mode=1, box_overlay=True, max_targets=len(geoms), **kw)
    for k, (f, w, h) in enumerate(geoms):
        t.set_stream_geometry(k, w, h, f)
    return t


def run_threads(steps_fns, n):
    """one host thread per entry of steps_fns; returns the wall time of n steps of every thread"""
    def worker(fn):
        for i in range(n):
            fn(i)
    th = [threading.Thread(target=worker, args=(fn,)) for fn in steps_fns]
    t0 = time.perf_counter()
    [t.start() for t in th]
    [t.join() for t in th]
    return time.perf_counter() - t0


def build_arms(wpath, cams):
    """{arm: (handles, [step function per host thread])}; every layout gets its own handles, all alive for the whole measurement"""
    S = len(cams)
    pins = [api.PinnedBuffer(fr[0].size * RING) for _, fr, _ in cams]
    for p, (_, fr, _) in zip(pins, cams):
        p.array[:] = np.concatenate(fr)
    surfs = []
    for (fmt, W, H), fr, _ in cams:
        row = []
        for f in fr:
            pf = api.PitchedFrame(W, H, fmt=fmt, pitch=(api.row_bytes(fmt, W) + 255) // 256 * 256, separate_uv=(fmt == "nv12"))
            pf.write(f)
            row.append(pf)
        surfs.append(row)
    torch.cuda.synchronize()

    def frame(s, i):
        fb = cams[s][1][0].size
        return pins[s].array[(i % RING) * fb:(i % RING + 1) * fb]

    layouts = {"mixed": [list(range(S))], "two_uniform": [list(range(N_VIS)), list(range(N_VIS, S))], "independent": [[s] for s in range(S)]}
    arms, keep = {}, (pins, surfs)
    for name, parts in layouts.items():
        for mem in ("pinned_windows", "surfaces"):
            hs, fns = [], []
            for part in parts:
                geoms = [cams[s][0] for s in part]
                t = new_group(wpath, geoms, upload_window=(mem == "pinned_windows"))
                for k, s in enumerate(part):
                    if mem == "pinned_windows":
                        t.init(frame(s, 0), cams[s][2], target=k)
                    else:
                        t.init_surface(surfs[s][0].surface, cams[s][2], target=k)
                hs.append(t)
                single = len(part) == 1
                if mem == "pinned_windows":
                    fns.append((lambda t, part, single: (lambda i: t.update_all(frame(part[0], i)) if single
                                                         else t.update_streams([frame(s, i) for s in part])))(t, part, single))
                else:
                    fns.append((lambda t, part, single: (lambda i: t.update_surface(surfs[part[0]][i % RING].surface) if single
                                                         else t.update_streams_surface([surfs[s][i % RING].surface for s in part])))(t, part, single))
            arms[f"{name}/{mem}"] = (hs, fns)
    return arms, keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--warmup", type=int, default=15)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_mixed_groups.py needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    wpath = weights.ensure_weight_file("tiny", os.path.join(tempfile.gettempdir(), "vt_b200_weights"))
    out = {"gpu_before": gpu_info()}
    cams = cameras()
    S = len(cams)
    arms, keep = build_arms(wpath, cams)
    for hs, fns in arms.values():  # warm-up: graph capture and first launches of every layout
        run_threads(fns, a.warmup)
    res = {k: [] for k in arms}
    for r in range(a.rounds):
        for name, (hs, fns) in arms.items():
            dt = run_threads(fns, a.steps)
            res[name].append(S * a.steps / dt)
    out["gpu_after"] = gpu_info()
    out["workload"] = (f"{N_VIS} x {VIS[1]}x{VIS[2]} NV12 (cfg5 seeds) + {N_IR} x {IR[1]}x{IR[2]} YUY2 (cfg3 scene), tiny, bf16x3, box overlay; "
                       "one host thread per group / handle; pinned_windows: pinned host frames with search-window uploads; surfaces: pitched "
                       "device surfaces (pitch rounded up to 256 bytes, NV12 chroma in its own allocation)")
    out["steps_per_round"], out["warmup"], out["rounds_streams_x_fps"] = a.steps, a.warmup, res
    out["summary"] = {k: {"median_streams_x_fps": float(np.median(v)), "min": float(min(v)), "max": float(max(v))} for k, v in res.items()}
    for hs, _ in arms.values():
        for t in hs:
            t.close()
    for p in keep[0]:
        p.close()
    with open(os.path.join(a.out, "bench_mixed_groups.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": out["gpu_before"], "summary": out["summary"]}))


if __name__ == "__main__":
    main()
