#!/usr/bin/env python
"""HBM roofline of the byte kernels (GPU only): NV12->RGB (K1), YUY2->RGB, RGB bilinear up-scale.  Device-resident batches larger than
L2, CUDA events on the handle's stream, algorithmic bytes / time against MEASURED_PEAKS.json.  One JSON line per kernel."""
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gstreamer_vit_tracker_b200 import api, weights  # noqa: E402


def timed(trk, fn, reps=20, warm=3):
    ext = torch.cuda.ExternalStream(trk.stream)
    for _ in range(warm):
        fn()
    trk.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for _ in range(reps):
        fn()
    e1.record(ext)
    trk.sync()
    return e0.elapsed_time(e1) / reps


def main():
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    hbm = peaks.get("hbm_gbs", 6650.0)
    wpath = weights.ensure_weight_file("nano", os.path.join(tempfile.gettempdir(), "vt_b200_weights"))
    out = []
    # K1 NV12 -> RGB, 64 x 1080p
    W, H, n = 1920, 1080, 64
    trk = api.VitTrack.new(wpath, W, H, fmt="nv12")
    src = torch.randint(0, 256, (n, W * H * 3 // 2), dtype=torch.uint8, device="cuda")
    dst = torch.empty((n, W * H * 3), dtype=torch.uint8, device="cuda")
    ms = timed(trk, lambda: trk.nv12_to_rgb_device(src.data_ptr(), W * H * 3 // 2, dst.data_ptr(), W * H * 3, n))
    by = n * (W * H * 3 // 2 + W * H * 3)
    out.append({"kernel": "nv12_to_rgb_vec4_kernel", "frames": n, "resolution": "1920x1080", "bytes_per_launch": by, "ms_per_launch": ms,
                "achieved_gbs": by / ms / 1e6, "peak_gbs": hbm, "frac": by / ms / 1e6 / hbm})
    # YUY2 -> RGB, 256 x 640x512
    w, h, n2 = 640, 512, 256
    src2 = torch.randint(0, 256, (n2, w * h * 2), dtype=torch.uint8, device="cuda")
    dst2 = torch.empty((n2, w * h * 3), dtype=torch.uint8, device="cuda")
    ms = timed(trk, lambda: trk.yuy2_to_rgb_device(src2.data_ptr(), w * h * 2, dst2.data_ptr(), w * h * 3, w, h, n2))
    by = n2 * (w * h * 2 + w * h * 3)
    out.append({"kernel": "yuy2_to_rgb_vec2_kernel", "frames": n2, "resolution": "640x512", "bytes_per_launch": by, "ms_per_launch": ms,
                "achieved_gbs": by / ms / 1e6, "peak_gbs": hbm, "frac": by / ms / 1e6 / hbm})
    # RGB up-scale 640x512 -> 1280x1024, batch of 128 frames in one launch (126 MB in, 503 MB out)
    nb = 128
    srcb = dst2[: nb * w * h * 3]
    upb = torch.empty(nb * 1280 * 1024 * 3, dtype=torch.uint8, device="cuda")
    ms = timed(trk, lambda: trk.resize_rgb_device_batch(srcb.data_ptr(), w * h * 3, w, h, upb.data_ptr(), 1280 * 1024 * 3, 1280, 1024, nb), reps=10)
    by = nb * (w * h * 3 + 1280 * 1024 * 3)
    out.append({"kernel": "resize_rgb_tile_kernel", "frames": nb, "resolution": "640x512 -> 1280x1024", "bytes_per_launch": by, "ms_per_launch": ms,
                "achieved_gbs": by / ms / 1e6, "peak_gbs": hbm, "frac": by / ms / 1e6 / hbm})
    del upb
    # RGB up-scale 640x512 -> 1280x1024 (one frame per launch: 0.98 MB in, 3.9 MB out, L2 resident when repeated)
    up = torch.empty(1280 * 1024 * 3, dtype=torch.uint8, device="cuda")
    ms = timed(trk, lambda: trk.resize_rgb_device(dst2.data_ptr(), w, h, up.data_ptr(), 1280, 1024), reps=50)
    by = w * h * 3 + 1280 * 1024 * 3
    out.append({"kernel": "resize_rgb_linear_kernel", "frames": 1, "resolution": "640x512 -> 1280x1024", "bytes_per_launch": by, "ms_per_launch": ms,
                "achieved_gbs": by / ms / 1e6, "peak_gbs": hbm, "frac": by / ms / 1e6 / hbm, "note": "single frame per launch: launch/latency bound"})
    for o in out:
        print(json.dumps(o))


if __name__ == "__main__":
    main()
