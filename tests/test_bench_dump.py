"""bench.py --dump-outputs: float32 .npy files, 64 MB in all, a larger output reduced to the same seeded sample in every run."""
import os

import numpy as np

import bench


def test_dump_outputs_is_float32_capped_and_repeatable(tmp_path):
    n = 20 << 20   # 80 MB as float32: has to be sampled
    outputs = {"frame": np.arange(n, dtype=np.int64).reshape(4, -1), "score": [[0.25, 0.5]], "bbox": np.array([[[1, 2, 3, 4]]], np.int32)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outputs)
    a, b = ({p.stem: np.load(p) for p in (tmp_path / run).iterdir()} for run in ("a", "b"))
    assert set(a) == {"frame", "score", "bbox"} and all(v.dtype == np.float32 for v in a.values())
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= 64 << 20
    assert a["score"].tolist() == [[0.25, 0.5]] and a["bbox"].tolist() == [[[1, 2, 3, 4]]]
    f = a["frame"]
    assert f.ndim == 1 and (16 << 20) - 4096 < f.size < n and np.all(np.diff(f) >= 0) and f[0] >= 0 and f[-1] <= n
    assert all(np.array_equal(a[k], b[k]) for k in a)
