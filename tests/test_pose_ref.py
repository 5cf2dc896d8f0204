"""POSE-1 parity PINNED to the reference's own code.

oracle/_ref/libintracam_ref.so is the unmodified src/slam/SL_IntraCamPose.cpp of the original
CoSLAM (compiled by `make -C oracle ref` against stand-in headers for the 7 LibVisualSLAM primitives
it calls); tests/golden/pose_ref.npz and pose_ref_seeded.npz hold intraCamEstimate inputs and the
outputs produced BY that library (tests/golden/make_pose_ref_golden.py).  CPU: the oracle
restatement reproduces them bit for bit.  GPU: the CUDA kernel matches the reference vectors to 1e-8
(fused-vs-unfused fp64 rounding of the sums; the forward differences themselves are evaluated
unfused like the reference)."""
import os

import numpy as np
import pytest

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pose_ref.npz")
GS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pose_ref_seeded.npz")
OPT_KEYS = ("lambda", "lambda0", "err0", "err", "errRW", "retTypeLM", "nIterLM", "nIterRW")


def _cases():
    d = np.load(G)
    for c in range(int(d["ncases"])):
        pe = d[f"c{c}_prev"]
        yield c, dict(K=d[f"c{c}_K"], R0=d[f"c{c}_R0"], t0=d[f"c{c}_t0"], Ms=d[f"c{c}_Ms"],
                      ms=d[f"c{c}_ms"], tau=float(d[f"c{c}_tau"]), prev=None if len(pe) == 0 else pe,
                      ok=bool(d[f"c{c}_ok"]), R=d[f"c{c}_R"], t=d[f"c{c}_t"],
                      opt=dict(zip(OPT_KEYS, d[f"c{c}_opt"])))


def test_oracle_reproduces_reference_vectors_bit_for_bit(orc):
    n = 0
    for c, g in _cases():
        ok, R, t, opt = orc.pose_intracam(g["K"], g["R0"], g["t0"], g["Ms"], g["ms"], g["tau"], g["prev"])
        assert ok == g["ok"], c
        assert np.array_equal(R, g["R"]) and np.array_equal(t, g["t"]), c
        assert opt.nIterRW == int(g["opt"]["nIterRW"]) and opt.nIterLM == int(g["opt"]["nIterLM"]), c
        assert opt.err == g["opt"]["err"] and opt.lambda_ == g["opt"]["lambda"], c
        n += 1
    assert n >= 7


def test_oracle_equals_compiled_reference_live(orc):
    """40 randomised cases (6-192 points, up to 25 % outliers, tau 6/10/20, previous errors on every
    third): the oracle equals the reference's outputs stored in pose_ref_seeded.npz bit for bit."""
    d = np.load(GS)
    off = np.concatenate([[0], np.cumsum(d["npts"])])
    poff = np.concatenate([[0], np.cumsum(d["npts"] * d["has_prev"])])
    assert len(d["npts"]) == 40
    for k in range(len(d["npts"])):
        pe = d["prev"][poff[k]:poff[k + 1]] if d["has_prev"][k] else None
        ok_o, R_o, t_o, opt = orc.pose_intracam(d["K"][k], d["R0"][k], d["t0"][k], d["Ms"][off[k]:off[k + 1]],
                                                d["ms"][off[k]:off[k + 1]], float(d["tau"][k]), pe)
        assert bool(d["ok"][k]) == ok_o, k
        assert np.array_equal(d["R"][k], R_o) and np.array_equal(d["t"][k], t_o), k
        assert int(d["nIterRW"][k]) == opt.nIterRW and float(d["err"][k]) == opt.err, k


def test_so3_exp_matches_reference(orc):
    import ctypes as C
    d = np.load(GS)
    for w, R_ref in zip(d["so3_w"], d["so3_R"]):
        R = np.empty(9)
        w = np.ascontiguousarray(w)
        orc.lib().orc_so3_exp(w.ctypes.data_as(C.c_void_p), R.ctypes.data_as(C.c_void_p))
        assert np.array_equal(R.reshape(3, 3), R_ref)


@pytest.mark.gpu
def test_cuda_matches_reference_vectors(api):
    worst = 0.0
    for c, g in _cases():
        ok, R, t, opt = api.pose_intracam(g["K"], g["R0"], g["t0"], g["Ms"], g["ms"], g["tau"], g["prev"])
        assert ok == g["ok"], c
        dR, dt = np.abs(R - g["R"]).max(), np.abs(t - g["t"]).max()
        worst = max(worst, dR, dt)
        assert dR < 1e-8 and dt < 1e-8, (c, dR, dt)
        assert opt.nIterRW == int(g["opt"]["nIterRW"]), c
        assert abs(opt.err - g["opt"]["err"]) <= 1e-6 * max(1.0, g["opt"]["err"]), c
    print("max |CUDA - reference| over the golden cases:", worst)


@pytest.mark.gpu
def test_cuda_batch_matches_reference_vectors(api):
    cs = [g for _, g in _cases()][:4]
    ok, R, t, _ = api.pose_intracam_batch([g["K"] for g in cs], [g["R0"] for g in cs], [g["t0"] for g in cs],
                                          [g["Ms"] for g in cs], [g["ms"] for g in cs], 10.0,
                                          [g["prev"] for g in cs])
    for i, g in enumerate(cs):
        if g["tau"] != 10.0:
            continue
        assert ok[i] == g["ok"]
        assert np.abs(R[i] - g["R"]).max() < 1e-8 and np.abs(t[i] - g["t"]).max() < 1e-8
