#!/usr/bin/env python
"""bench.py — headline benchmark: 1080p tracked frames/s (BASELINE.json `metric`).

A "step" is one pass of the per-frame hot path (NV12 ingest -> fused crop/convert/resize/normalise -> ViT forward -> score-map
decode -> overlay) over one frame of every stream this rank owns.  Workload at N=1: BASELINE.json configs[1] — a single 1920x1080
NV12 stream, one target (SURVEY.md §8(d) cfg2).  For N>1 every rank runs its own independent stream(s) (cfg5 seeds): no data-path
collective exists, `scaling` is "weak", value = frames of all ranks / max-over-ranks device time.

  value   frames/s with the frames already resident in HBM (vt_tracker_submit_device / vt_tracker_wait, two frames in flight; box overlay
          drawn into the device frame)
  e2e     the DROP-IN call: vt_probe_frame (≙ the pad-probe closure, /root/reference/src/pipeline.rs:67-184) on pinned HOST frames — H2D of
          every frame's search window + HUD region, ViT, decode, HUD (background, 3-4 text lines, box, crosshair) mirrored into the host
          frame and the result block, all inside the timed region.  `e2e.value` / p50 / p99 are this call's; `e2e.submit_wait` (pipelined
          vt_tracker_submit / wait, box overlay only) and `e2e.sync_update` (synchronous vt_tracker_update) are reported beside it.
  roofline       dominant kernel of the step (gemm_tc_kernel: every dense contraction but attention), in-chain duration measured live
                 with device %globaltimer stamps; `roofline_convert` is the HBM-bound NV12->RGB kernel
  cpu_baseline   the CPU oracle port of the same probe body (convert + VitTrack::update + HUD overlay) on the host cores, and
                 cv2.TrackerVit (OpenCV DNN, the algorithm's upstream implementation) on the same weights as a second opinion
  cfg4 / cfg5    BASELINE.json configs 4 (2160p x 16 targets, one batched forward) and 5 (64 concurrent 1080p streams sharded over the
                 ranks of this run) — reported beside the headline, not part of `value`
  --impl reference   times the CPU path alone (same probe body, same HUD), same metric/config keys

Only the cpu_baseline / --impl reference legs (and the trajectory cross-check that uses their results) touch oracle/.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "1080p tracked frames/s"
UNIT = "frames/s"
GEMM_MODES = {"fp32simt": 0, "tcgen05x3": 1, "tcgen05": 2, "tcgen05fp16": 3}
DTYPES = {"fp32simt": "f32", "tcgen05x3": "bf16x3 (split bf16 operands, fp32 accumulate)", "tcgen05": "bf16",
          "tcgen05fp16": "f16 (single-pass fp16 operands, fp32 accumulate)"}
HUD_BG = (10, 10, 400, 80, 150)   # draw_background_nv12 call of src/pipeline.rs:125


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=600)
    ap.add_argument("--warmup", type=int, default=60)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="tiny", choices=["tiny", "nano"])
    ap.add_argument("--gemm", default="tcgen05x3", choices=list(GEMM_MODES),
                    help="precision/engine of the dense contractions (tcgen05x3 = bf16 split operands, the parity-safe default)")
    ap.add_argument("--streams-per-gpu", type=int, default=1)
    ap.add_argument("--ring", type=int, default=0,
                    help="distinct frames per stream (0 = steps + warmup, at most 1024: no frame is used twice within a timed leg).  The bytes the "
                         "step actually touches (search windows, ~0.45 MB per frame) over the ring must exceed the 126 MB L2: 660 x 0.45 MB = 297 MB")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg4 / cfg5 / multi-stream side legs")
    ap.add_argument("--cfg5-streams", type=int, default=64, help="total concurrent streams of the cfg5 leg (sharded over the ranks)")
    ap.add_argument("--full-upload", action="store_true",
                    help="e2e legs upload the whole frame every step instead of the search windows of the active targets (cfg.upload_window)")
    ap.add_argument("--cpu-sample-frames", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned for its last step as DIR/<name>.npy (float32): per "
                         "stream (rank 0's streams) and target success, status, score and bbox, and (b200 arm) the NV12 frame with the "
                         "box drawn into it. "
                         "The reference arm's frame is left out: its HUD prints the measured FPS")
    return ap.parse_args()


DUMP_BYTES = 64 << 20


def dump_outputs(directory, outputs):
    """Each array as `directory`/<name>.npy in float32, 64 MB in all.  An array larger than what is left of that is stored as a fixed
    sample: the elements at the sorted flat positions np.random.default_rng(0).choice(size, n, replace=False), the same in every run."""
    os.makedirs(directory, exist_ok=True)
    left = DUMP_BYTES
    for name, a in sorted(outputs.items(), key=lambda kv: np.asarray(kv[1]).size):
        a = np.asarray(a, dtype=np.float32)
        left -= 4096  # .npy header
        if a.nbytes > left:
            idx = np.sort(np.random.default_rng(0).choice(a.size, left // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(directory, name + ".npy"), a)
        left -= a.nbytes


def result_outputs(results):
    """results[stream][target] = (success, status, score, bbox) -> the arrays of --dump-outputs."""
    return {"success": [[r[0] for r in rs] for rs in results], "status": [[r[1] for r in rs] for rs in results],
            "score": [[r[2] for r in rs] for rs in results], "bbox": [[r[3] for r in rs] for rs in results]}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def workload_name(args):
    return (f"cfg2: single 1920x1080 NV12 synthetic stream, one target, model={args.model}, "
            f"{args.streams_per_gpu} stream(s) per GPU" + (" (cfg5 seeds, one stream set per rank)" if args.gpus > 1 else ""))


def config_dict(args):
    """`config` of the JSON line: the same keys and, for the same flags, the same values in both arms."""
    ring_n = ring_size(args)
    return {"workload": workload_name(args), "resolution": "1920x1080", "format": "NV12", "targets": 1, "model": args.model,
            "streams_per_gpu": args.streams_per_gpu, "weights": "constructed random-init (SURVEY.md §8c)",
            "call": "probe body per frame: convert + VitTrack::update + HUD overlay (src/pipeline.rs:104-174)",
            "l2": f"L2 flushed (256 MB device write) before every timed leg; within a leg every step reads a frame no earlier step of the leg "
                  f"touched ({args.steps + args.warmup} frames per stream out of a ring of {ring_n} distinct 1080p frames = "
                  f"{ring_n * 3110400 / 1e6:.0f} MB; 126 MB L2; a step reads only the ~0.4 MB search window of its frame), every frame on clean "
                  "pixels (overlays are undone / never reused)"}


def ring_size(args):
    return max(8, min(args.ring or 1024, args.steps + args.warmup))


def stream_spec(rank, k, args, world):
    """Stream k of this rank: cfg2 for the single-stream headline run, else global stream id -> rank round-robin (sharding.py)."""
    from gstreamer_vit_tracker_b200 import sharding, synth
    if world == 1 and args.streams_per_gpu == 1:
        return synth.CONFIGS["cfg2"]
    mine = sharding.streams_of_rank(world * args.streams_per_gpu, rank, world)
    return synth.cfg5_stream(mine[k] % 64)


def weight_path(model):
    from gstreamer_vit_tracker_b200 import weights
    return weights.ensure_weight_file(model, os.path.join(tempfile.gettempdir(), "vt_b200_weights"))


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.p, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])), mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's probe body restated on the CPU oracle (the Rust reference + its absent vit_tracker crate cannot be built
# in this image).  Per frame, as src/pipeline.rs:104-174: convert, process_frame (VitTrack::update), TimingStats, HUD overlay
# (background, state, FPS, timing line, score, box, crosshair).
class CpuProbe:
    def __init__(self, model, threads, tracker="oracle", cv2_threads=None):
        from gstreamer_vit_tracker_b200 import synth
        from oracle import oracle
        self.o, self.threads = oracle, threads
        self.spec = synth.CONFIGS["cfg2"]
        self.st = synth.SyntheticStream(self.spec)
        self.W, self.H = self.spec.width, self.spec.height
        self.stats = oracle.TimingStats()
        self.kind = tracker
        self.t_conv = self.t_track = self.t_ovl = 0.0
        self.last = None
        wpath = weight_path(model)
        box = self.st.target_boxes(0)[0]
        rgb0 = oracle.nv12_to_rgb(self.st.frame(0), self.W, self.H, threads)
        if tracker == "oracle":
            self.trk = oracle.VitTrack(wpath, threads=threads)
            self.trk.init(rgb0, box)
        else:  # cv2.TrackerVit on an ONNX export of the same weight file (tools/torch_model.py), intended normalisation (SURVEY.md §8c)
            import cv2
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            from torch_model import export_onnx
            onnx = os.path.join(tempfile.gettempdir(), "vt_b200_weights", f"bench_{model}.onnx")
            if not os.path.exists(onnx):
                export_onnx(wpath, onnx + ".tmp")
                os.replace(onnx + ".tmp", onnx)
            cv2.setNumThreads(cv2_threads or threads)
            s = np.array([0.229, 0.224, 0.225])
            n = 1.0 / np.sum(1.0 / s ** 2)
            prm = cv2.TrackerVit_Params()
            prm.net, prm.stdvalue, prm.tracking_score_threshold = onnx, (n / s[0], -n / s[1], -n / s[2], 0.0), 0.2
            self.trk = cv2.TrackerVit_create(prm)
            self.trk.init(rgb0, box)

    def step(self, fr):
        o, W, H = self.o, self.W, self.H
        a = time.perf_counter()
        rgb = o.nv12_to_rgb(fr, W, H, self.threads)                # conv   (src/pipeline.rs:105)
        b = time.perf_counter()
        if self.kind == "oracle":
            rc, ok, score, bb = self.trk.update(rgb)               # track  (src/pipeline.rs:112)
        else:
            ok, bb = self.trk.update(rgb)
            rc, score = 0, float(self.trk.getTrackingScore())
        c = time.perf_counter()
        self.stats.add_times(int((b - a) * 1e6), int((c - b) * 1e6))
        tracking = rc == 0 and ok and score > 0.25
        o.draw_background_nv12(fr, W, H, *HUD_BG)                  # HUD    (src/pipeline.rs:125-156)
        o.draw_text_nv12(fr, W, H, "TRACKING" if tracking else "LOST", 15, 15, 2, 255)
        o.draw_text_nv12(fr, W, H, "FPS: %.0f" % self.stats.fps(), 15, 40, 2, 255)
        o.draw_text_nv12(fr, W, H, "conv:%.1fms trk:%.1fms" % (self.stats.avg_conv_ms(), self.stats.avg_track_ms()), 15, 65, 1, 200)
        if tracking:
            o.draw_text_nv12(fr, W, H, "score: %.0f%%" % (score * 100.0), 250, 15, 2, 255)
            o.draw_rect_nv12(fr, W, H, bb[0], bb[1], bb[2], bb[3], 3, 255)          # box (src/pipeline.rs:165-168)
            o.draw_crosshair_nv12(fr, W, H, bb[0] + bb[2] // 2, bb[1] + bb[3] // 2, 15, 255)
        d = time.perf_counter()
        self.stats.add_interval(int((d - a) * 1e6))
        self.t_conv += b - a
        self.t_track += c - b
        self.t_ovl += d - c
        self.last = (rc, ok, score, tuple(int(v) for v in bb))
        return self.last


def run_reference(args):
    """--impl reference: the reference's CPU probe body (oracle port) on all host threads, same metric / config / HUD work."""
    rank, _, _ = dist_env()
    if rank != 0:
        return
    threads = len(os.sched_getaffinity(0)) or 1
    p = CpuProbe(args.model, threads)
    ring = [p.st.frame(i) for i in range(ring_size(args))]
    for i in range(args.warmup):
        p.step(ring[i % len(ring)].copy())
    t0 = time.perf_counter()
    for i in range(args.steps):
        p.step(ring[(args.warmup + i) % len(ring)].copy())
    dt = time.perf_counter() - t0
    fps = args.steps / dt
    if args.dump_outputs:
        rc, ok, score, bb = p.last
        dump_outputs(args.dump_outputs, result_outputs([[(ok, rc, score, bb)]]))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_dict(args),
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} frames of cfg2 after {args.warmup} warm-up: convert + VitTrack::update + HUD overlay (background, "
                                   f"4 text lines, box, crosshair), OpenMP {threads} threads"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference = CPU oracle port of the probe body (the Rust reference + absent vit_tracker crate cannot be built in this image)"}))


def cpu_baseline(args, n_frames):
    """Oracle port of the probe body on all host threads (+ its result trajectory for the cross-check), the conversion alone at the
    reference's pool size (8 threads, /root/reference/src/main.rs:43-46) and on 1 thread, and cv2.TrackerVit as a second opinion."""
    threads = len(os.sched_getaffinity(0)) or 1
    p = CpuProbe(args.model, threads)
    frames = [p.st.frame(i) for i in range(n_frames + 2)]
    for i in range(2):
        p.step(frames[i].copy())
    p.t_conv = p.t_track = p.t_ovl = 0.0
    traj = []
    t0 = time.perf_counter()
    for i in range(n_frames):
        traj.append(p.step(frames[2 + i].copy()))
    dt = time.perf_counter() - t0
    conv_t = {}
    for nt in (8, 1):
        a = time.perf_counter()
        for i in range(20):
            p.o.nv12_to_rgb(frames[2 + i % n_frames], p.W, p.H, nt)
        conv_t[nt] = (time.perf_counter() - a) / 20 * 1e3
    out = {"value": n_frames / dt, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": f"{n_frames} frames of cfg2 (convert + VitTrack::update + HUD overlay), OpenMP {threads} threads",
           "conv_ms": p.t_conv / n_frames * 1e3, "track_ms": p.t_track / n_frames * 1e3, "overlay_ms": p.t_ovl / n_frames * 1e3,
           "conv_ms_8_threads": conv_t[8], "conv_ms_1_thread": conv_t[1]}
    # second opinion (BASELINE.md §2): OpenCV's own TrackerVit (DNN, CPU) inside the same probe body, at the reference's 8 threads and on all cores
    try:
        cv = {}
        for nt in sorted({min(8, threads), threads}):
            q = CpuProbe(args.model, threads, tracker="cv2", cv2_threads=nt)
            m = max(20, n_frames // 4)
            for i in range(2):
                q.step(frames[i].copy())
            q.t_track = 0.0
            a = time.perf_counter()
            for i in range(m):
                q.step(frames[2 + i % n_frames].copy())
            b = time.perf_counter()
            cv[f"threads_{nt}"] = {"value": m / (b - a), "unit": UNIT, "track_ms": q.t_track / m * 1e3, "frames": m}
        import cv2
        cv["impl"] = f"cv2.TrackerVit (OpenCV {cv2.__version__}, DNN CPU backend), ONNX export of the same weight file, same probe body"
        out["cv2_trackervit"] = cv
    except Exception as e:  # the headline line must not depend on the optional leg
        out["cv2_trackervit"] = {"error": str(e)[:200]}
    return out, traj


# ---------------------------------------------------------------------------------------------------
class Stream:
    """One video stream of the bench: tracker handle (+ probe context), pinned host ring, pristine copy, device ring."""

    def __init__(self, api, torch, spec, wpath, local_rank, args, ring_n, dev_frames, with_context=True, box=None, max_targets=1):
        from gstreamer_vit_tracker_b200 import synth
        self.api, self.torch, self.spec = api, torch, spec
        self.st = synth.SyntheticStream(spec)
        self.fb = self.st.frame_bytes()
        self.ring_n, self.dev_frames = ring_n, dev_frames
        kw = dict(fmt=spec.fmt, device=local_rank, upload_window=not args.full_upload, gemm_mode=GEMM_MODES[args.gemm], max_targets=max_targets)
        self.trk = api.VitTrack.new(wpath, spec.width, spec.height, box_overlay=True, **kw)
        self.ctx = api.TrackerContext.new(wpath, spec.width, spec.height, **{k: v for k, v in kw.items() if k != "max_targets"}) if with_context else None
        self.pin = api.PinnedBuffer(ring_n * self.fb)
        self.host = self.pin.array.reshape(ring_n, self.fb)
        for i in range(ring_n):
            self.host[i] = np.asarray(self.st.frame(i)).reshape(-1)
        self.pristine = self.host.copy()                         # the same ring, never drawn on
        self.dev0 = torch.from_numpy(self.pristine).cuda(local_rank)
        self.dev = torch.empty((dev_frames, self.fb), dtype=torch.uint8, device=f"cuda:{local_rank}")
        self.boxes = self.st.target_boxes(0)

    def reset(self):
        """Clean frames and the initial tracker state (outside every timed region)."""
        self.host[:] = self.pristine
        for i in range(0, self.dev_frames, self.ring_n):   # device frames i = ring frames i % ring_n: no frame is reused within a leg
            k = min(self.ring_n, self.dev_frames - i)
            self.dev[i:i + k] = self.dev0[:k]
        for k, b in enumerate(self.boxes):
            self.trk.init(self.pristine[0], self.api.BBox(*b), target=k)

    def reset_context(self):
        """Fresh probe context steered into TRACKING on the stream's target (keyboard commands ≙ src/raw_mode_guard.rs:65-101)."""
        api = self.api
        if self.ctx is not None:
            self.ctx.close()
        kw = dict(fmt=self.spec.fmt, device=self.trk._cfg.device, upload_window=bool(self.trk._cfg.upload_window), gemm_mode=self.trk._cfg.gemm_mode)
        self.ctx = api.TrackerContext.new(self.trk._cfg.weights_path.decode(), self.spec.width, self.spec.height, **kw)
        U, c = api.UserCommand, self.ctx
        x, y, w, h = self.boxes[0]
        cx, cy = self.spec.width // 2, self.spec.height // 2

        def move(dx, dy):
            for _ in range(abs(dx) // 10):
                c.handle_command(U.MoveRight if dx > 0 else U.MoveLeft, False)
            for _ in range(abs(dy) // 10):
                c.handle_command(U.MoveDown if dy > 0 else U.MoveUp, False)
        move(x - cx, y - cy)
        c.handle_command(U.Confirm)
        c.probe(self.host[0])
        move(w, h)
        c.handle_command(U.Confirm)
        c.probe(self.host[0])
        self.host[0] = self.pristine[0]
        assert c.state_name() == "TRACKING", c.state_name()


def run_b200(args):
    import torch
    import torch.distributed as dist

    rank, local_rank, world = dist_env()
    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL may print its version banner on stdout while the communicator is created: keep stdout for the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.all_reduce(torch.zeros(1, device=f"cuda:{local_rank}"))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    from gstreamer_vit_tracker_b200 import _lib as L
    from gstreamer_vit_tracker_b200 import api, sharding, synth, weights

    wpath = weight_path(args.model)
    cfg_model = weights.MODELS[args.model]
    S = args.streams_per_gpu
    K, Wm = args.steps, args.warmup
    ring_n = ring_size(args)
    HUD = None  # live (timing dependent) HUD strings, as the reference draws them

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    l2_buf = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")

    def flush_l2():
        """Write a buffer twice the size of L2: nothing an earlier leg touched (device rings, weights, activations) stays resident."""
        l2_buf.fill_(1)
        torch.cuda.synchronize()

    def run_leg(streams, kind, n_steps, offset, want_lat=False):
        """n_steps frames on every stream of this rank, one host thread per stream, each ONE native call (the GIL is released inside);
        returns per-stream latency arrays (us) for the synchronous kinds."""
        lat = [None] * len(streams)

        def worker(si):
            s = streams[si]
            # a host ring shorter than the leg is replayed: the native loop then undoes every frame's overlay from the clean copy
            clean = s.pristine.ctypes.data if s.ring_n < offset + n_steps else 0
            if kind == "probe":
                lat[si] = s.ctx.run_ring(s.host.ctypes.data, s.fb, s.fb, s.ring_n, offset % s.ring_n, n_steps, HUD, clean, want_lat)
            elif kind in ("device", "device_sync"):
                mode = L.VT_RUN_DEVICE_PIPELINED if kind == "device" else L.VT_RUN_DEVICE_SYNC
                _, lat[si] = s.trk.run_ring(s.dev.data_ptr(), s.fb, s.fb, s.dev_frames, offset % s.dev_frames, n_steps, mode, 0, want_lat)
            else:
                mode = L.VT_RUN_HOST_PIPELINED if kind == "host_pipelined" else L.VT_RUN_HOST_SYNC
                _, lat[si] = s.trk.run_ring(s.host.ctypes.data, s.fb, s.fb, s.ring_n, offset % s.ring_n, n_steps, mode, clean, want_lat)
        if len(streams) == 1:
            worker(0)
        else:
            th = [threading.Thread(target=worker, args=(i,)) for i in range(len(streams))]
            [t.start() for t in th]
            [t.join() for t in th]
        return lat

    def timed(streams, kind, n_steps, n_warm):
        for s in streams:  # same starting state for every leg
            s.reset()
            if kind == "probe":
                s.reset_context()
        handles = [(s.ctx.tracker if kind == "probe" else s.trk) for s in streams]
        run_leg(streams, kind, n_warm, 0)
        tm0 = [h.timing() for h in handles]
        flush_l2()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ext = torch.cuda.ExternalStream(handles[0].stream, device=local_rank)  # events on the stream the kernels are launched on
        ev0.record(ext)
        lat = run_leg(streams, kind, n_steps, n_warm, want_lat=True)
        ev1.record(ext)
        for h in handles:
            h.sync()
        barrier()
        ms = ev0.elapsed_time(ev1)
        tm1 = [h.timing() for h in handles]
        if kind == "probe":
            for s in streams:
                assert s.ctx.state_name() == "TRACKING" and s.ctx.lost_frames == 0, "the probe leg must track every frame"
        return {"ms": ms, "lat": lat, "launches": sum(b.kernel_launches - a.kernel_launches for a, b in zip(tm0, tm1)),
                "h2d": sum(b.h2d_bytes - a.h2d_bytes for a, b in zip(tm0, tm1)) / n_steps,
                "d2h": sum(b.d2h_bytes - a.d2h_bytes for a, b in zip(tm0, tm1)) / n_steps,
                "stages": {k: getattr(tm1[0], "avg_" + k) for k in ("h2d_ms", "preprocess_ms", "vit_ms", "decode_ms", "overlay_ms", "d2h_ms", "total_ms")}}

    # ---- headline streams ------------------------------------------------------------------------------------------------------
    streams = [Stream(api, torch, stream_spec(rank, k, args, world), wpath, local_rank, args, ring_n, K + Wm) for k in range(S)]
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    leg_dev = timed(streams, "device", K, Wm)
    if args.dump_outputs and rank == 0:   # the headline leg's last step: the handles' results and the frame its overlay was drawn into
        dumped = result_outputs([[(r.success, r.status, r.score, r.bbox) for r in s.trk._results()] for s in streams])
        dumped["frame_nv12"] = torch.stack([s.dev[(Wm + K - 1) % s.dev_frames] for s in streams]).cpu().numpy()
    for s in streams:
        s.reset()
    lat_dev = run_leg(streams, "device_sync", min(K, 200), 0, want_lat=True)  # per-frame latency of the synchronous device-resident call
    leg_probe = timed(streams, "probe", K, Wm)
    leg_sync = timed(streams, "host", K, Wm)
    leg_pipe = timed(streams, "host_pipelined", K, Wm)
    clocks = sampler.stop()

    # ---- trajectory of the first frames (cross-checked against the CPU oracle's below): synchronous calls on clean frames -----------
    s0 = streams[0]
    n_traj = args.cpu_sample_frames or (200 if args.model == "tiny" else 1000)
    traj = []
    if world == 1 and S == 1 and not args.no_cpu_baseline:
        s0.reset()
        for i in range(n_traj + 2):
            buf = s0.host[i % ring_n]
            buf[:] = s0.st.frame(i) if i >= ring_n else s0.pristine[i]
            r = s0.trk.update(buf)
            traj.append((0, r.success, r.score, tuple(r.bbox)))
        s0.host[:] = s0.pristine

    # ---- per-kernel in-chain durations of the tensor-core kernels (device %globaltimer stamps written by the kernels themselves:
    #      an event between two kernels of the replayed graph would break the programmatic-dependent-launch edge it measures) ----
    kern = None
    for s in streams:   # (the probe contexts own a tracker handle each: the latency / throughput forms switch on the live-handle count)
        if s.ctx is not None:
            s.ctx.close()
            s.ctx = None
    if args.gemm != "fp32simt":
        os.environ["VT_B200_TRACE"] = "1"
        try:
            ttrk = api.VitTrack.new(wpath, s0.spec.width, s0.spec.height, fmt="nv12", device=local_rank, box_overlay=True, gemm_mode=GEMM_MODES[args.gemm])
        finally:
            del os.environ["VT_B200_TRACE"]
        s0.reset()
        ttrk.init(s0.pristine[0], api.BBox(*s0.boxes[0]))
        for i in range(10):
            ttrk.update_device(s0.dev[i % s0.dev_frames].data_ptr(), s0.fb)
        ttrk.debug_trace()
        nfr = 20
        for i in range(nfr):
            ttrk.update_device(s0.dev[(10 + i) % s0.dev_frames].data_ptr(), s0.fb)
        rec = ttrk.debug_trace().astype(np.int64)
        names = {1: "patch", 2: "qkv", 3: "proj", 4: "fc1+fc2partial", 5: "fc2", 6: "head", 10: "attention"}
        kern = {}
        for kid, te, tw, tend, *_ in rec:
            d = kern.setdefault(names.get(int(kid), str(int(kid))), [0, 0.0])
            d[0] += 1
            d[1] += (tend - tw) * 1e-3
        kern = {k: {"launches_per_frame": v[0] / nfr, "avg_us": v[1] / v[0]} for k, v in kern.items()}
        ttrk.close()

    # ---- NV12->RGB full-frame kernel (HBM roofline), device resident, batch larger than L2 -------------------
    nb = min(ring_n, 64)
    fb, w, h = s0.fb, s0.spec.width, s0.spec.height
    rgb_out = torch.empty((nb, h * w * 3), dtype=torch.uint8, device=f"cuda:{local_rank}")
    ext = torch.cuda.ExternalStream(s0.trk.stream, device=local_rank)
    for _ in range(3):
        s0.trk.nv12_to_rgb_device(s0.dev0.data_ptr(), fb, rgb_out.data_ptr(), h * w * 3, nb)
    s0.trk.sync()
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for _ in range(reps):
        s0.trk.nv12_to_rgb_device(s0.dev0.data_ptr(), fb, rgb_out.data_ptr(), h * w * 3, nb)
    e1.record(ext)
    s0.trk.sync()
    cvt_ms = e0.elapsed_time(e1) / reps
    cvt_bytes = nb * (w * h * 3 // 2 + w * h * 3)
    del rgb_out

    # ---- aggregate over ranks: max time, sum of frames (no data-path collective; see sharding.py) -----------------------
    frames_rank = K * S
    tm_all = sharding.combine_timings([leg_dev["ms"], leg_probe["ms"], leg_sync["ms"], leg_pipe["ms"]], float(frames_rank), float(leg_dev["launches"]),
                                      device=f"cuda:{local_rank}")
    ms_dev_g, ms_probe_g, ms_sync_g, ms_pipe_g = tm_all.ms_max
    frames_g, launches_g = tm_all.frames, tm_all.launches

    # ---- side legs: BASELINE configs 4 and 5 -------------------------------------------------------------------------------
    extras = {}
    if not args.no_extras:
        for s in streams:
            s.trk.close()
            if s.ctx is not None:
                s.ctx.close()
        hud_keep = streams  # (pinned buffers stay alive until the end)
        flops = weights.flops_per_frame(cfg_model)
        peaks_tf = None
        # cfg5: 64 concurrent 1080p streams sharded over the ranks (stream i -> rank i mod world), one handle + CUDA stream + graph each
        try:
            n5 = args.cfg5_streams
            mine = sharding.streams_of_rank(n5, rank, world)
            K5, W5 = max(20, K // 10), max(3, Wm // 6)
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(16) as ex:
                st5 = list(ex.map(lambda i: Stream(api, torch, synth.cfg5_stream(i % 64), wpath, local_rank, args, 8, K5 + W5, with_context=False), mine))
            l5d = timed(st5, "device", K5, W5)
            l5h = timed(st5, "host", K5, W5)
            l5p = timed(st5, "host_pipelined", K5, W5)
            t5 = sharding.combine_timings([l5d["ms"], l5h["ms"], l5p["ms"]], float(K5 * len(mine)), 0.0, device=f"cuda:{local_rank}")
            lat5 = np.concatenate([x for x in l5h["lat"] if x is not None]) * 1e-3
            extras["cfg5"] = {
                "workload": f"{n5} concurrent 1080p NV12 streams (cfg5 seeds) sharded over {world} GPU(s): {len(mine)} per GPU, one handle / CUDA stream / "
                            "graph / host thread per stream, no collective",
                "streams": n5, "streams_per_gpu": len(mine), "steps_per_stream": K5,
                "value": t5.frames / (t5.ms_max[0] * 1e-3), "e2e": t5.frames / (t5.ms_max[2] * 1e-3), "unit": "streams x frames/s (aggregate)",
                "e2e_mode": "vt_tracker_submit / vt_tracker_wait per stream thread (native loop; two frames in flight per stream, as the `value` leg), "
                            "pinned frames, predicted search-window uploads, box overlay",
                "e2e_sync": t5.frames / (t5.ms_max[1] * 1e-3),
                "e2e_sync_mode": "synchronous vt_tracker_update per stream thread: one frame in flight per stream (latency percentiles below)",
                "fps_per_stream_e2e": t5.frames / (t5.ms_max[2] * 1e-3) / n5, "p50_latency_ms": float(np.percentile(lat5, 50)),
                "p99_latency_ms": float(np.percentile(lat5, 99)), "h2d_bytes_per_frame": int(l5p["h2d"] / max(1, len(mine))),
                "h2d_gbs_per_gpu": l5p["h2d"] * K5 / (l5p["ms"] * 1e-3) / 1e9,
                "achieved_tflops_per_gpu": (K5 * len(mine)) / (l5d["ms"] * 1e-3) * flops / 1e12}
            for s in st5:
                s.trk.close()
            # the same streams as stream GROUPS: up to 16 streams per handle stepped together through one batched forward
            # (vt_tracker_update_streams; 320 x 16 = 5120 rows: the many-row GEMM forms), one host thread per group
            try:
                G = 16
                groups = [st5[i:i + G] for i in range(0, len(st5), G)]
                gtrk = []
                for g in groups:
                    t = api.VitTrack.new(wpath, g[0].spec.width, g[0].spec.height, fmt="nv12", device=local_rank, box_overlay=True,
                                         upload_window=not args.full_upload, gemm_mode=GEMM_MODES[args.gemm], max_targets=len(g))
                    gtrk.append(t)

                def greset():
                    for t, g in zip(gtrk, groups):
                        for k, s in enumerate(g):
                            s.host[:] = s.pristine
                            t.init(s.pristine[0], api.BBox(*s.boxes[0]), target=k)

                def grun(n_steps, offset, want_lat=False):
                    lat = [None] * len(groups)

                    def worker(gi):
                        g = groups[gi]
                        _, lat[gi] = gtrk[gi].run_streams_ring([s.host.ctypes.data for s in g], g[0].fb, g[0].fb, g[0].ring_n, offset % g[0].ring_n,
                                                               n_steps, [s.pristine.ctypes.data for s in g], want_lat)
                    th = [threading.Thread(target=worker, args=(i,)) for i in range(len(groups))]
                    [x.start() for x in th]
                    [x.join() for x in th]
                    return lat
                greset()
                grun(W5, 0)
                tm0 = [t.timing() for t in gtrk]
                barrier()
                w0 = time.perf_counter()
                glat = grun(K5, W5, True)
                for t in gtrk:
                    t.sync()
                barrier()
                gms = (time.perf_counter() - w0) * 1e3
                tm1 = [t.timing() for t in gtrk]
                tg = sharding.combine_timings([gms], float(K5 * len(mine)), 0.0, device=f"cuda:{local_rank}")
                gl = np.concatenate([x for x in glat if x is not None]) * 1e-3
                h2d = sum(b.h2d_bytes - a.h2d_bytes for a, b in zip(tm0, tm1))
                extras["cfg5"]["grouped"] = {
                    "mode": f"stream groups of up to {G}: vt_tracker_update_streams per step (one batched forward per group, search-window uploads, "
                            "each stream's box drawn into its own pinned frame), one host thread per group, timed on the host clock around all groups",
                    "groups_per_gpu": len(groups), "e2e": tg.frames / (tg.ms_max[0] * 1e-3), "unit": "streams x frames/s (aggregate)",
                    "p50_step_latency_ms": float(np.percentile(gl, 50)), "p99_step_latency_ms": float(np.percentile(gl, 99)),
                    "vit_ms_per_step": tm1[0].avg_vit_ms, "h2d_gbs_per_gpu": h2d / (gms * 1e-3) / 1e9,
                    "achieved_tflops_per_gpu": (K5 * len(mine)) / (gms * 1e-3) * flops / 1e12}
                for t in gtrk:
                    t.close()
            except Exception as e:
                extras["cfg5"]["grouped"] = {"error": repr(e)[:300]}
            del st5
        except Exception as e:
            extras["cfg5"] = {"error": repr(e)[:300]}
        # cfg4: 3840x2160 NV12, 16 targets through one batched forward (rank 0's GPU; the same on every rank)
        if world == 1:
            try:
                spec4 = synth.CONFIGS["cfg4"]
                K4, W4 = max(20, K // 6), max(3, Wm // 6)
                s4 = Stream(api, torch, spec4, wpath, local_rank, args, 8, K4 + W4, with_context=False, max_targets=len(spec4.targets))
                l4d = timed([s4], "device", K4, W4)
                l4h = timed([s4], "host", K4, W4)
                l4p = timed([s4], "host_pipelined", K4, W4)
                nt = len(spec4.targets)
                vit_ms = l4d["stages"]["vit_ms"]
                extras["cfg4"] = {
                    "workload": "3840x2160 NV12, 16 targets batched through one ViT forward (M = 5120 rows)", "targets": nt, "steps": K4,
                    "value": K4 / (l4d["ms"] * 1e-3), "e2e": K4 / (l4h["ms"] * 1e-3), "unit": "frames/s",
                    "e2e_pipelined": K4 / (l4p["ms"] * 1e-3),
                    "e2e_modes": "e2e: synchronous vt_tracker_update, the 12.4 MB frame uploaded whole (16 search windows cover it); e2e_pipelined: "
                                 "vt_tracker_submit / vt_tracker_wait, the next frame's upload under the frame in flight",
                    "target_frames_per_s": nt * K4 / (l4d["ms"] * 1e-3), "p50_latency_ms": float(np.percentile(l4h["lat"][0], 50) * 1e-3),
                    "h2d_bytes_per_step": int(l4h["h2d"]), "stages_ms": l4d["stages"],
                    "vit_tflops": nt * flops / (vit_ms * 1e-3) / 1e12 if vit_ms > 0 else None}
                s4.trk.close()
                del s4
            except Exception as e:
                extras["cfg4"] = {"error": repr(e)[:300]}

        # cfg1 / cfg3: the reference's CPU-runnable 720p NV12 case and the 640x512 RGB24 path its main() runs (src/main.rs:49), one target each
        if world == 1:
            for name in ("cfg1", "cfg3"):
                try:
                    specx = synth.CONFIGS[name]
                    Kx, Wx = max(40, K // 4), max(5, Wm // 4)
                    sx_ = Stream(api, torch, specx, wpath, local_rank, args, 8, Kx + Wx, with_context=False)
                    lxd = timed([sx_], "device", Kx, Wx)
                    lxh = timed([sx_], "host", Kx, Wx)
                    extras[name] = {
                        "workload": f"{specx.width}x{specx.height} {specx.fmt.upper()}, one target", "steps": Kx,
                        "value": Kx / (lxd["ms"] * 1e-3), "e2e": Kx / (lxh["ms"] * 1e-3), "unit": "frames/s",
                        "e2e_mode": "synchronous vt_tracker_update, pinned frames, search-window upload, box overlay",
                        "p50_latency_ms": float(np.percentile(lxh["lat"][0], 50) * 1e-3), "h2d_bytes_per_step": int(lxh["h2d"]),
                        "stages_ms": lxh["stages"]}
                    sx_.trk.close()
                    del sx_
                except Exception as e:
                    extras[name] = {"error": repr(e)[:300]}

    if rank == 0:
        peaks = {}
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peaks = json.load(open(pk))
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        tf_peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        flops = weights.flops_per_frame(cfg_model)
        stage = leg_dev["stages"]
        vit_s = stage["vit_ms"] * 1e-3
        ach_tf = (flops / vit_s / 1e12) if vit_s > 0 else None
        # dominant kernel = gemm_tc_kernel (every dense contraction except attention): algorithmic FLOPs per frame of its launches
        # (2*M*N*K each, SURVEY.md §8(d)) / summed in-chain kernel time per frame
        cm, Dm, Hm, Cm = cfg_model, cfg_model.D, cfg_model.hidden, cfg_model.head_ch
        kind_flops = {"patch": 2 * 256 * 768 * Dm, "qkv": cm.depth * 2 * 320 * Dm * 3 * Dm, "proj": cm.depth * 2 * 320 * Dm * Dm,
                      "fc1+fc2partial": cm.depth * 2 * 2 * 320 * Dm * Hm, "head": 2 * 256 * 9 * Dm * Cm}
        gemm_kinds = ("patch", "qkv", "proj", "fc1+fc2partial", "fc2", "head")
        # (in latency mode proj is folded into the attention kernel: its FLOPs then do not belong to gemm_tc_kernel)
        gemm_flops = sum(f for k, f in kind_flops.items() if kern is None or k in kern)
        gemm_us = sum(v["launches_per_frame"] * v["avg_us"] for k, v in (kern or {}).items() if k in gemm_kinds)
        gemm_n = sum(v["launches_per_frame"] for k, v in (kern or {}).items() if k in gemm_kinds)
        chain_us = sum(v["launches_per_frame"] * v["avg_us"] for v in (kern or {}).values())
        traffic = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("gemm_tc_kernel", {}).get("dram_bytes_per_launch")
        lat_probe = np.concatenate([x for x in leg_probe["lat"] if x is not None]) * 1e-3
        lat_sync = np.concatenate([x for x in leg_sync["lat"] if x is not None]) * 1e-3
        lat_d = np.concatenate([x for x in lat_dev if x is not None]) * 1e-3
        fb0 = streams[0].fb
        cfgd = config_dict(args)
        run_info = {"gemm": args.gemm,
                    "h2d": "whole frame" if args.full_upload else "search windows of the active targets (+ the HUD background region) only: 2-D copies "
                                                                  "out of the pinned frame",
                    "bytes_read_per_leg": (f"`value`: {K + Wm} device frames ({(K + Wm) * fb0 / 1e6:.0f} MB, {ring_n} distinct) of which the step reads the "
                                           f"search windows (~{(K + Wm) * leg_sync['h2d'] / 1e6:.0f} MB per leg); e2e legs: pinned host ring, every frame "
                                           "restored to clean pixels after its result")}
        out = {
            "metric": METRIC, "value": frames_g / (ms_dev_g * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_dev_g / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPES[args.gemm], "data": "synthetic", "config": cfgd, "run": run_info,
            "e2e": {"value": frames_g / (ms_probe_g * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(leg_probe["h2d"]),
                    "d2h_bytes_per_step": int(leg_probe["d2h"]),
                    "mode": "vt_probe_frame (the drop-in for the reference's pad-probe closure) on pinned host frames, synchronous, one stream thread: "
                            "window + HUD-region upload, ViT, decode, HUD (background, state / FPS / timing / score text, box, crosshair) mirrored into "
                            "the host frame, one synchronisation per frame",
                    "p50_latency_ms": float(np.percentile(lat_probe, 50)), "p99_latency_ms": float(np.percentile(lat_probe, 99)),
                    "stages_ms": leg_probe["stages"],
                    "submit_wait": {"value": frames_g / (ms_pipe_g * 1e-3), "h2d_bytes_per_step": int(leg_pipe["h2d"]), "d2h_bytes_per_step": int(leg_pipe["d2h"]),
                                    "mode": "vt_tracker_submit / vt_tracker_wait, two frames in flight, predicted search windows uploaded on a copy stream "
                                            "while the frame in flight computes, box overlay"},
                    "sync_update": {"value": frames_g / (ms_sync_g * 1e-3), "h2d_bytes_per_step": int(leg_sync["h2d"]),
                                    "p50_latency_ms": float(np.percentile(lat_sync, 50)), "p99_latency_ms": float(np.percentile(lat_sync, 99)),
                                    "mode": "synchronous vt_tracker_update (VitTrack::update + box overlay), search-window upload"}},
            "latency_ms": {"device_resident_p50": float(np.percentile(lat_d, 50)), "probe_p50": float(np.percentile(lat_probe, 50)),
                           "sync_update_p50": float(np.percentile(lat_sync, 50))},
            "gpu_launches": int(launches_g), "stages_ms": stage,
            "roofline": ({"kernel": "gemm_tc_kernel<%s> (tcgen05/TMEM/TMA GEMM: %s)" % ("3" if args.gemm == "tcgen05x3" else "1",
                              "patch-embed, QKV, proj, FC1+chained FC2, 3x3 head conv" if "proj" in kern else
                              "patch-embed, QKV, FC1+chained FC2, 3x3 head conv; proj is folded into the attention kernel in latency mode"),
                          "bound": "tensor", "achieved": gemm_flops / (gemm_us * 1e-6) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                          "frac": gemm_flops / (gemm_us * 1e-6) / 1e12 / tf_peak, "traffic": traffic, "peak_source": peak_src,
                          "flops_per_launch_avg": gemm_flops / gemm_n, "launches_per_frame": gemm_n, "avg_launch_us": gemm_us / gemm_n,
                          "share_of_chain": gemm_us / chain_us if chain_us else None,
                          "share_of_step": gemm_us * 1e-3 / (ms_dev_g / K) if ms_dev_g else None,
                          "share_note": "share_of_chain: of the in-chain time of the traced tensor-core kernels (GEMM + attention); share_of_step: of "
                                        "ms_per_step (which also holds the reduce / decode / overlay kernels and every dependency edge); the ncu launch "
                                        "list of this command (profiles/r2v_bench_launches.csv, cold cache, serialised): 43.8 % of all kernel time, "
                                        "66.7 % of GEMM + attention",
                          "timing": "device %globaltimer stamps inside the replayed graph (dependency wait -> kernel end), 20 frames",
                          "note": "one target = 320 rows: every launch is a 9..108-CTA latency-bound GEMM; algorithmic FLOPs (2MNK), the bf16x3 "
                                  "split issues 3 UMMAs per product; tensor utilisation at scale is the cfg4 / cfg5 objects' vit_tflops"} if kern and gemm_us > 0 else
                         {"kernel": "ViT forward, gemm=" + args.gemm, "bound": "tensor", "achieved": ach_tf, "peak": tf_peak, "unit": "TFLOP/s",
                          "frac": (ach_tf / tf_peak) if ach_tf else None, "traffic": None, "peak_source": peak_src}),
            "roofline_vit_stage": {"achieved": ach_tf, "unit": "TFLOP/s", "frac": (ach_tf / tf_peak) if ach_tf else None, "flops_per_frame": flops,
                                   "stage_ms": stage["vit_ms"], "timing": "device stamps, mean of the last 120 frames"},
            "kernels_in_chain": kern,
            "roofline_convert": {"kernel": "nv12_to_rgb_vec4_kernel", "bound": "hbm", "achieved": cvt_bytes / (cvt_ms * 1e-3) / 1e9, "peak": hbm_peak,
                                 "unit": "GB/s", "frac": cvt_bytes / (cvt_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                                 "frames_per_launch": nb, "bytes_per_launch": cvt_bytes, "ms_per_launch": cvt_ms, "peak_source": peak_src},
            "clocks": clocks,
        }
        tpx = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpx):
            tj = json.load(open(tpx)).get("nv12_to_rgb_vec4_kernel", {})
            if tj.get("dram_bytes_per_frame"):  # ncu capture of a 32-frame launch, scaled to this leg's frames per launch
                out["roofline_convert"]["traffic"] = int(tj["dram_bytes_per_frame"]) * nb
                out["roofline_convert"]["traffic_note"] = (f"dram__bytes_read + write per 1080p frame under ncu ({tj['dram_bytes_per_frame']} B; algorithmic "
                                                           f"{tj.get('algorithmic_bytes_per_frame')} B, the rest of the writes is still in L2 when the kernel ends) x {nb} frames")
        for k, v in extras.items():
            if isinstance(v, dict) and v.get("vit_tflops"):
                v["vit_frac_of_bf16_peak"] = v["vit_tflops"] / tf_peak
            if isinstance(v, dict) and v.get("achieved_tflops_per_gpu"):
                v["frac_of_bf16_peak"] = v["achieved_tflops_per_gpu"] / tf_peak
            out[k] = v
        if world == 1 and not args.no_cpu_baseline:
            base, cpu_traj = cpu_baseline(args, n_traj)
            out["cpu_baseline"] = base
            # the GPU arm and the CPU arm ran the same frames: their result trajectories must agree (boxes equal, |dscore| <= 1e-3)
            if traj:
                same = sum(1 for a, b in zip(traj[2:], cpu_traj) if a[1] == b[1] and a[3] == b[3])
                dmax = max(abs(a[2] - b[2]) for a, b in zip(traj[2:], cpu_traj))
                out["trajectory_check"] = {"frames": len(cpu_traj), "boxes_equal": same, "max_dscore": dmax,
                                           "what": "GPU (synchronous update, clean frames) vs CPU oracle on the first frames of the workload"}
                assert dmax <= 1e-3 and same >= 0.97 * len(cpu_traj), out["trajectory_check"]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
