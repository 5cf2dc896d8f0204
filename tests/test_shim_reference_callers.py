"""Drop-in checks of the reference-named shim headers (syntax-only compiles, CPU).

The probe translation units in tests/stubs/ are written the way the reference's callers use
slam/SL_IntraCamPose.h (intraCamEstimate / IntraCamPoseOption) and slam/SL_GlobalPoseEstimation.h
(RobustBundleRTS::constructCameraGraphs / updateNonKeyCameraPoses).  They must compile with the shim
standing in for the header under its reference path.  LibVisualSLAM declarations come from
tests/stubs/.
"""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STUBS = os.path.join(ROOT, "tests", "stubs")
SHIM = os.path.join(ROOT, "coslam_b200", "shim")

pytestmark = pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")


def _syntax_only(tmp_path, src, *flags):
    # `#include "slam/<header>"` of the probes resolves to the shim of the same name
    os.symlink(SHIM, tmp_path / "slam")
    cmd = ["g++", "-std=c++11", "-fsyntax-only", *flags, "-I", STUBS, "-I",
           os.path.join(ROOT, "include"), "-I", str(tmp_path), src]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-4000:]


def test_pose_probe_compiles_against_the_shim_header(tmp_path):
    _syntax_only(tmp_path, os.path.join(STUBS, "probe_pose.cpp"), "-include",
                 os.path.join(SHIM, "SL_IntraCamPose.h"))


def test_posegraph_probe_compiles_against_the_shim_header(tmp_path):
    _syntax_only(tmp_path, os.path.join(STUBS, "probe_posegraph.cpp"), "-include",
                 os.path.join(SHIM, "SL_GlobalPoseEstimation.h"))
