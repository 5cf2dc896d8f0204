"""Generates tests/golden/posegraph_ref.npz and posegraph_ref_seeded.npz from the UNMODIFIED reference
file slam/SL_GlobalPoseEstimation.cpp (compiled by `make -C oracle ref REF=<CoSLAM checkout>` into
oracle/_ref/libposegraph_ref.so; needs the original CoSLAM tree, which the tests do not).
Cases: chain graphs as RobustBundleRTS::constructCameraGraphs builds them (leading / trailing free
runs, adjacent key frames, single free node), and two non-chain graphs (a skip edge, a loop closure)
that only the oracle restatement supports."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from coslam_b200.synth import make_pose_chains  # noqa: E402
from oracle import ref  # noqa: E402

cases = {}
specs = [
    dict(lengths=[23], key_every=7, seed=1),
    dict(lengths=[40], key_every=8, seed=2, lead_free=3),
    dict(lengths=[12], seed=3, fixed_masks=[[1, 1, 0, 1, 0, 0, 0, 1, 1, 1, 0, 0]]),
    dict(lengths=[9], seed=4, fixed_masks=[[0, 0, 0, 0, 1, 0, 0, 0, 0]]),
    dict(lengths=[64], key_every=16, seed=5, shift=0.2),
    dict(lengths=[5], seed=6, fixed_masks=[[1, 0, 1, 0, 1]]),
]
for i, sp in enumerate(specs):
    g = make_pose_chains(**sp)
    nR, nt = ref.posegraph_spread(g["fixed"], g["R"], g["t"], g["id1"], g["id2"], g["eR_list"], g["et_list"])
    for k in ("fixed", "R", "t", "id1", "id2", "eR_list", "et_list"):
        cases[f"c{i}_{k}"] = g[k]
    cases[f"c{i}_newR"], cases[f"c{i}_newt"] = nR, nt
# non-chain graphs: extra edges measured with noise
rng = np.random.default_rng(11)
for i, extra in ((len(specs), [(2, 9)]), (len(specs) + 1, [(0, 19), (5, 12)])):
    g = make_pose_chains([20], key_every=6, seed=20 + i)
    id1, id2 = list(g["id1"]), list(g["id2"])
    eR, et = list(g["eR_list"]), list(g["et_list"])
    from coslam_b200.synth import _rodrigues
    for a, b in extra:
        Rab = _rodrigues(rng.normal(size=3) * 0.01) @ g["R"][b] @ g["R"][a].T
        tab = g["t"][b] - Rab @ g["t"][a] + rng.normal(size=3) * 0.01
        id1.append(a), id2.append(b), eR.append(Rab), et.append(tab)
    g["id1"], g["id2"] = np.asarray(id1, np.int32), np.asarray(id2, np.int32)
    g["eR_list"], g["et_list"] = np.asarray(eR), np.asarray(et)
    nR, nt = ref.posegraph_spread(g["fixed"], g["R"], g["t"], g["id1"], g["id2"], g["eR_list"], g["et_list"])
    for k in ("fixed", "R", "t", "id1", "id2", "eR_list", "et_list"):
        cases[f"c{i}_{k}"] = g[k]
    cases[f"c{i}_newR"], cases[f"c{i}_newt"] = nR, nt
cases["n_cases"] = np.int32(len(specs) + 2)
cases["n_chain_cases"] = np.int32(len(specs))
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "posegraph_ref.npz"), **cases)
print("wrote", len(specs) + 2, "cases")

# posegraph_ref_seeded.npz: the reference's results only (tests/test_posegraph.py regenerates the
# inputs) for 12 chains of growing length, key-frame spacing, leading free runs and BA shift
seeded = {}
for seed in range(12):
    g = make_pose_chains([10 + 7 * seed], key_every=3 + seed % 6, seed=100 + seed, lead_free=seed % 3,
                         shift=0.02 * (1 + seed % 4))
    nR, nt = ref.posegraph_spread(g["fixed"], g["R"], g["t"], g["id1"], g["id2"], g["eR_list"], g["et_list"])
    seeded[f"c{seed}_newR"], seeded[f"c{seed}_newt"] = nR, nt
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "posegraph_ref_seeded.npz"), **seeded)
print("wrote 12 seeded cases")
