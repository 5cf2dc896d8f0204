"""Generates tests/golden/facade_ref.npz: what the REFERENCE's own KLT facade -- tracking/GPUKLT.cpp,
SL_Track2D.cpp, slam/SL_FeaturePoints.cpp and SL_FeaturePoint.cpp of the original CoSLAM, compiled
unmodified into oracle/_ref/gpuklt_ref_caller against coslam_b200/shim/v3d_gpuklt.h (`make -C oracle
ref REF=<CoSLAM checkout>`) -- prints when it runs on top of libcoslam_b200.so.  Needs a GPU.

    python tests/golden/make_facade_ref_golden.py [out.npz]

Per case: the stdout of tests/ref_gpuklt_caller.cpp (lines "N frame count", "X frame nFed",
"F frame slot trackLength x y") and the CRC-32 of each input frame, so that tests can tell a change
of the synthetic frames from a change of the tracker."""
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import seq  # noqa: E402

EXE = os.path.join(ROOT, "oracle", "_ref", "gpuklt_ref_caller")
W, H = 640, 480
# name: (sequence seed, frames, trackWithGain, feed external points every n-th frame)
CASES = {"gain1": (31, 5, True, 0), "gain0": (31, 5, False, 0), "feed": (32, 4, True, 2)}


def frames_of(name):
    seed, n, _, _ = CASES[name]
    return seq(H, W, seed, n=n).frames


def crcs(frames):
    return np.array([zlib.crc32(np.ascontiguousarray(f).tobytes()) for f in frames], np.int64)


def main(out_path):
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, (_, n, gain, feed_every) in CASES.items():
            frames = frames_of(name)
            raw = os.path.join(tmp, "frames.raw")
            with open(raw, "wb") as f:
                f.write(np.stack(frames).astype(np.uint8).tobytes())
            r = subprocess.run([EXE, raw, str(W), str(H), str(n), str(int(gain)), str(feed_every)],
                               capture_output=True, text=True, timeout=300)
            if r.returncode != 0:
                raise SystemExit(f"{name}: rc={r.returncode}\n{r.stdout[-2000:]}{r.stderr[-2000:]}")
            out[f"{name}_stdout"] = np.frombuffer(r.stdout.encode(), np.uint8)
            out[f"{name}_crc"] = crcs(frames)
            print(name, len(r.stdout.splitlines()), "lines")
    np.savez_compressed(out_path, **out)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "facade_ref.npz"))
