"""Post-BA pose-graph spreading (SURVEY.md 8f-2): pins oracle/posegraph_oracle.cpp to the UNMODIFIED
reference slam/SL_GlobalPoseEstimation.cpp through the committed outputs of
oracle/_ref/libposegraph_ref.so: tests/golden/posegraph_ref.npz (with its inputs) and
posegraph_ref_seeded.npz (seeded chains), made by tests/golden/make_posegraph_ref_golden.py.
Tolerance: the two least-squares solvers differ (Householder QR vs normal equations), values are O(1):
1e-9 absolute."""
import os

import numpy as np
import pytest

from coslam_b200.synth import make_pose_chains
from oracle import orc

HERE = os.path.dirname(os.path.abspath(__file__))
TOL = 1e-9


def _golden():
    return np.load(os.path.join(HERE, "golden", "posegraph_ref.npz"))


def _case(z, i):
    return {k: z[f"c{i}_{k}"] for k in ("fixed", "R", "t", "id1", "id2", "eR_list", "et_list", "newR", "newt")}


def test_oracle_matches_reference_golden_vectors():
    z = _golden()
    for i in range(int(z["n_cases"])):
        c = _case(z, i)
        nR, nt = orc.posegraph_spread(c["fixed"], c["R"], c["t"], c["id1"], c["id2"], c["eR_list"], c["et_list"])
        assert np.abs(nR - c["newR"]).max() < TOL, i
        assert np.abs(nt - c["newt"]).max() < TOL, i


def test_oracle_matches_compiled_reference_live():
    # the reference's results for these graphs are stored; at 1e-9 the last-bit differences of
    # synthetic inputs between numpy builds do not matter
    z = np.load(os.path.join(HERE, "golden", "posegraph_ref_seeded.npz"))
    for seed in range(12):
        n = 10 + 7 * seed
        g = make_pose_chains([n], key_every=3 + seed % 6, seed=100 + seed, lead_free=seed % 3,
                             shift=0.02 * (1 + seed % 4))
        args = (g["fixed"], g["R"], g["t"], g["id1"], g["id2"], g["eR_list"], g["et_list"])
        rR, rt = z[f"c{seed}_newR"], z[f"c{seed}_newt"]
        oR, ot = orc.posegraph_spread(*args)
        assert np.abs(oR - rR).max() < TOL and np.abs(ot - rt).max() < TOL, seed


def test_unmoved_key_frames_reproduce_the_trajectory():
    """Known answer: when BA did not move the key frames every edge is satisfied exactly by the input
    poses, so the least-squares solution IS the input."""
    g = make_pose_chains([31], key_every=5, seed=3, shift=0.0)
    nR, nt = orc.posegraph_spread(g["fixed"], g["R"], g["t"], g["id1"], g["id2"], g["eR_list"], g["et_list"])
    assert np.abs(nR - g["R"]).max() < 1e-12 and np.abs(nt - g["t"]).max() < 1e-11


def test_fixed_nodes_are_copied_and_rotations_are_proper():
    g = make_pose_chains([26], key_every=6, seed=9, shift=0.3)
    nR, nt = orc.posegraph_spread(g["fixed"], g["R"], g["t"], g["id1"], g["id2"], g["eR_list"], g["et_list"])
    fx = g["fixed"].astype(bool)
    assert np.array_equal(nR[fx], g["R"][fx]) and np.array_equal(nt[fx], g["t"][fx])
    assert np.abs(np.einsum("nij,nkj->nik", nR, nR) - np.eye(3)).max() < 1e-12
    assert np.all(np.linalg.det(nR) > 0.999999)


def test_rank_deficient_graph_is_reported():
    g = make_pose_chains([6], seed=1, fixed_masks=[[0] * 6])
    with pytest.raises(RuntimeError):
        orc.posegraph_spread(g["fixed"], g["R"], g["t"], g["id1"], g["id2"], g["eR_list"], g["et_list"])
