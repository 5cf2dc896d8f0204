"""KLT-7 / the facade seam (SURVEY.md 8b): the REFERENCE's own tracking/GPUKLT.cpp, SL_Track2D.cpp,
slam/SL_FeaturePoints.cpp and SL_FeaturePoint.cpp -- compiled unmodified against
coslam_b200/shim/v3d_gpuklt.h and run on top of libcoslam_b200.so: first() + next() x 4
(+ feedExternFeatPoints) on a synthetic sequence.  Their output is stored in
tests/golden/facade_ref.npz (tests/golden/make_facade_ref_golden.py).  What the reference's facade
stores in its Track2D lists must equal what the C-ABI returns for the same frames
(pos * (W, H), `GPUKLT::addToFeaturePoints`, tracking/GPUKLT.cpp:36-61)."""
import os
import sys

import numpy as np
import pytest

from helpers import live_cfg

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_facade_ref_golden as golden  # noqa: E402


def _run(name):
    """The input frames of case `name` and what the reference facade printed for them."""
    frames = golden.frames_of(name)
    z = np.load(os.path.join(ROOT, "tests", "golden", "facade_ref.npz"))
    assert np.array_equal(golden.crcs(frames), z[f"{name}_crc"]), \
        "the synthetic frames differ from those the golden output was made from"
    per_frame, counts, fed = {}, {}, {}
    for line in z[f"{name}_stdout"].tobytes().decode().splitlines():
        p = line.split()
        if p[0] == "F":
            per_frame.setdefault(int(p[1]), {})[int(p[2])] = (int(p[3]), float(p[4]), float(p[5]))
        elif p[0] == "N":
            counts[int(p[1])] = int(p[2])
        elif p[0] == "X":
            fed[int(p[1])] = int(p[2])
    return frames, per_frame, counts, fed


@pytest.mark.parametrize("gain", [True, False])
def test_reference_facade_runs_on_the_shim(api, gain):
    W, H = golden.W, golden.H
    frames, per_frame, counts, _ = _run("gain1" if gain else "gain0")
    # the same frames through the C-ABI (32 x 32 slots = SLAM_FEATURE_WIDTH/HEIGHT, slam/SL_Define.h:17-18)
    g = api.KltTracker(live_cfg(gain=gain), W, H, 6, 32, 32)
    lengths = np.zeros(1024, np.int64)
    for k in range(5):
        f, n = g.first(frames[0]) if k == 0 else g.next(frames[k])
        assert counts[k] == n
        live = np.nonzero(f["status"] >= 0)[0]
        ref = per_frame.get(k, {})
        # the facade keeps a track node for exactly the live slots
        assert sorted(ref) == sorted(int(i) for i in live)
        lengths = np.where(f["status"] == 0, lengths + 1, np.where(f["status"] == 1, 1, 0))
        for i in live:
            ln, x, y = ref[int(i)]
            assert ln == lengths[i], (k, i)
            # identical floats, converted exactly like GPUKLT.cpp:43-44 (float pos * int W -> double)
            assert x == float(np.float32(f["pos"][i, 0]) * np.float32(W)) or abs(x - f["pos"][i, 0] * W) < 1e-4
            assert abs(y - f["pos"][i, 1] * H) < 1e-4
    assert (lengths >= 4).sum() > 100  # most first-frame corners were tracked through all 5 frames


def test_reference_facade_feed_extern_points(api):
    W, H = golden.W, golden.H
    frames, per_frame, counts, fed = _run("feed")
    assert list(fed) == [2] and 1 <= fed[2] <= 5  # external points found slots (SingleSLAM::feedExtraFeatPtsToTracker)
    assert len(per_frame[3]) > 100
    # the facade's calls through the C-ABI: first, next, next, feed of 5 points + advanceFrame, next
    g = api.KltTracker(live_cfg(gain=True), W, H, 6, 32, 32)
    for k in range(4):
        f, n = g.first(frames[0]) if k == 0 else g.next(frames[k])
        assert counts[k] == n
        if k == 2:
            pts = np.array([[W * (0.2 + 0.15 * j) / W, H * (0.3 + 0.1 * j) / H, 0.0] for j in range(5)])
            _, nf = g.feed(pts)
            g.advance()
            assert nf == fed[2]
    live = np.nonzero(f["status"] >= 0)[0]
    assert sorted(per_frame[3]) == sorted(int(i) for i in live)
    for i in live:
        _, x, y = per_frame[3][int(i)]
        assert abs(x - f["pos"][i, 0] * W) < 1e-4 and abs(y - f["pos"][i, 1] * H) < 1e-4
