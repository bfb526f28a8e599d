"""The chained latency-mode attention on 64-row query tiles (M = 64 UMMAs, the default for one target) against the 128-row form
(VT_B200_ATT_Q128).  The two forms add the same products; only the softmax row sums are re-associated (8 partial sums per row
instead of 4), so boxes must be equal, scores within 1e-5, and the token state after every block (where reduce_ln has added the
per-head proj partial planes) within fp32 re-association tolerance."""
import gc

import numpy as np
import pytest

from gstreamer_vit_tracker_b200 import synth, weights

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api(built):
    from gstreamer_vit_tracker_b200 import api as _api
    return _api


def _make(api, monkeypatch, w, spec, q128, **kw):
    monkeypatch.delenv("VT_B200_ATT_Q128", raising=False)
    if q128:
        monkeypatch.setenv("VT_B200_ATT_Q128", "1")
    return api.VitTrack.new(w, spec.width, spec.height, gemm_mode=1, **kw)


@pytest.mark.parametrize("model", ["nano", "tiny"])
def test_q64_matches_q128_teacher_forced(api, weight_dir, monkeypatch, model):
    """One target, every frame started from the true box of the synthetic stream (teacher forcing): both forms see the same crops."""
    gc.collect()  # handles of earlier tests would count as live streams (the chained form runs only while <= 2 handles are alive)
    w = weights.ensure_weight_file(model, weight_dir, variant="wild")
    spec = synth.CONFIGS["cfg2"]
    st = synth.SyntheticStream(spec)
    frames = [np.ascontiguousarray(st.frame(i)).reshape(-1) for i in range(12)]

    def run(q128):
        trk = _make(api, monkeypatch, w, spec, q128)
        trk.init(frames[0], api.BBox(*st.target_boxes(0)[0]))
        out = []
        for i, f in enumerate(frames[1:], 1):
            trk.set_rect(st.target_boxes(i - 1)[0])
            out.append(trk.update(f))
        trk.close()
        return out

    a, b = run(False), run(True)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.success == y.success and x.status == y.status and tuple(x.bbox) == tuple(y.bbox), (model, i, x, y)
        assert abs(x.score - y.score) <= 1e-5, (model, i, x.score, y.score)


def test_q64_block_outputs_match_q128(api, weight_dir, monkeypatch):
    """Token state after the embeddings and after every block (residual + the sum of the per-head proj partial planes + MLP)."""
    gc.collect()
    w = weights.ensure_weight_file("tiny", weight_dir, variant="wild")
    spec = synth.CONFIGS["cfg2"]
    st = synth.SyntheticStream(spec)
    f0, f1 = (np.ascontiguousarray(st.frame(i)).reshape(-1) for i in range(2))

    def run(q128):
        trk = _make(api, monkeypatch, w, spec, q128, debug_capture=True)
        trk.init(f0, api.BBox(*st.target_boxes(0)[0]))
        trk.update_all(f1)
        toks = [trk.debug_tokens(k) for k in range(trk.model_dim(1) + 1)]
        trk.close()
        return toks

    a, b = run(False), run(True)
    for k, (x, y) in enumerate(zip(a, b)):
        scale = float(np.abs(y).max())
        err = float(np.abs(x - y).max())
        assert err <= 1e-5 * scale, (k, err, scale)
