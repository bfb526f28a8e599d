"""The bench.py contract: one JSON line on stdout with the keys the driver reads, for both arms.  Short runs (the numbers are not
judged here, only that the line is complete and self-consistent).  GPU only."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _run(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines  # exactly one JSON line on stdout
    return json.loads(lines[0])


def test_b200_arm_line(built):
    d = _run("--steps", "40", "--warmup", "5", "--cpu-sample-frames", "8", "--cfg5-streams", "4")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 40 and d["warmup"] == 5 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["value"] > 1000 and abs(d["ms_per_step"] * d["value"] - 1000.0) < 1.0  # frames/s and ms/frame agree (one stream)
    e = d["e2e"]   # the drop-in call: vt_probe_frame on pinned host frames, HUD included
    assert "vt_probe_frame" in e["mode"]
    assert e["value"] > 1000 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 32000 and e["unit"] == d["unit"]  # HUD block mirrored back
    assert 0 < e["p50_latency_ms"] <= e["p99_latency_ms"] < 50
    assert e["submit_wait"]["value"] > 1000 and e["sync_update"]["value"] > 1000
    assert e["submit_wait"]["h2d_bytes_per_step"] < 0.5 * 1920 * 1080 * 1.5   # pipelined frames upload predicted windows, not whole frames
    assert d["gpu_launches"] >= 40 * 60  # > 60 kernels of this library per frame
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["peak"] > 0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and "sample" in c
    assert c["cv2_trackervit"][f"threads_{min(8, c['cores'])}"]["value"] > 0, c["cv2_trackervit"]
    t = d["trajectory_check"]   # the two arms ran the same pixels
    assert t["boxes_equal"] == t["frames"] == 8 and t["max_dscore"] <= 1e-3
    assert d["cfg4"]["targets"] == 16 and d["cfg4"]["value"] > 100 and d["cfg4"]["vit_tflops"] > 10, d["cfg4"]
    assert d["cfg5"]["streams"] == 4 and d["cfg5"]["e2e"] > 1000 and d["cfg5"]["h2d_gbs_per_gpu"] > 0, d["cfg5"]
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_reference_arm_line(built):
    d = _run("--impl", "reference", "--steps", "3", "--warmup", "1")
    assert d["impl"] == "reference" and d["value"] > 0 and d["unit"] and d["higher_is_better"] is True
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]


def test_both_arms_print_the_same_config_keys(built, tmp_path):
    """The driver compares the two arms' `config`: same keys, and the same values for the workload-defining ones.  Both arms' last
    timed step tracked the same frame: their --dump-outputs results agree (|dscore| <= 1e-3, boxes within a floor tie)."""
    sys.path.insert(0, ROOT)
    import bench
    import argparse

    import numpy as np
    a = argparse.Namespace(model="tiny", streams_per_gpu=1, gpus=1, ring=0, steps=40, warmup=5)
    assert set(bench.config_dict(a)) >= {"workload", "resolution", "format", "targets", "model", "streams_per_gpu", "weights", "call", "l2"}
    g = _run("--steps", "12", "--warmup", "3", "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path / "g"))
    r = _run("--impl", "reference", "--steps", "12", "--warmup", "3", "--dump-outputs", str(tmp_path / "r"))
    assert g["config"] == r["config"]
    res = {"success", "status", "score", "bbox"}
    assert {p.stem for p in (tmp_path / "g").iterdir()} == res | {"frame_nv12"} and {p.stem for p in (tmp_path / "r").iterdir()} == res
    dg, dr = ({k: np.load(tmp_path / arm / f"{k}.npy") for k in res} for arm in ("g", "r"))
    assert all(dg[k].dtype == np.float32 and dg[k].shape == dr[k].shape for k in res)
    assert dg["success"][0, 0] == dr["success"][0, 0] == 1 and dg["status"][0, 0] == dr["status"][0, 0] == 0
    assert abs(dg["score"] - dr["score"]).max() <= 1e-3 and abs(dg["bbox"] - dr["bbox"]).max() <= 1, (dg, dr)
    fr = np.load(tmp_path / "g" / "frame_nv12.npy")
    assert fr.dtype == np.float32 and fr.shape == (1, 1920 * 1080 * 3 // 2) and fr.min() >= 0 and fr.max() <= 255
    assert np.array_equal(fr, np.round(fr))
