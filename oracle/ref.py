"""ctypes access to oracle/_ref/libintracam_ref.so = the UNMODIFIED reference file
src/slam/SL_IntraCamPose.cpp of the original CoSLAM compiled against the stand-in headers of
oracle/ref_stubs/ (recipe: `make -C oracle ref REF=<CoSLAM checkout>`), and to libposegraph_ref.so.
TEST INFRASTRUCTURE: used only by tests/golden/make_pose_ref_golden.py and
make_posegraph_ref_golden.py, whose stored outputs pin the restatements in oracle/ and the CUDA
kernels to the reference's own code."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "_ref", "libintracam_ref.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(PATH)
        vp = C.c_void_p
        L.ref_intraCamEstimate.argtypes = [vp, vp, vp, C.c_int, vp, vp, vp, C.c_double, vp, vp, vp, vp]
        L.ref_intraCamEstimate.restype = C.c_int
        L.ref_getSO3ExpMap.argtypes = [vp, vp]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def intracam_estimate(K, R0, t0, Ms, ms, tau, prev_errs=None, opt_in=None):
    """intraCamEstimate of the reference (slam/SL_IntraCamPose.cpp:626-709).  opt_in =
    (maxIterLM, maxIterRW, epsErrorChangeLM, epsParamChangeLM, epsErrorChangeRW, lambda0) or None
    for the IntraCamPoseOption defaults.  Returns ok, R, t, dict of the option block after the call."""
    K = np.ascontiguousarray(K, np.float64).ravel()
    R0 = np.ascontiguousarray(R0, np.float64).ravel()
    t0 = np.ascontiguousarray(t0, np.float64).ravel()
    Ms = np.ascontiguousarray(Ms, np.float64).reshape(-1, 3)
    ms = np.ascontiguousarray(ms, np.float64).reshape(-1, 2)
    pe = None if prev_errs is None else np.ascontiguousarray(prev_errs, np.float64)
    oi = None if opt_in is None else np.ascontiguousarray(opt_in, np.float64)
    R, t, oo = np.empty(9), np.empty(3), np.zeros(8)
    ok = lib().ref_intraCamEstimate(_p(K), _p(R0), _p(t0), len(Ms), _p(pe), _p(Ms), _p(ms), float(tau),
                                    _p(R), _p(t), _p(oi), _p(oo))
    keys = ("lambda", "lambda0", "err0", "err", "errRW", "retTypeLM", "nIterLM", "nIterRW")
    return bool(ok), R.reshape(3, 3), t, dict(zip(keys, oo))


def so3_exp(w):
    w = np.ascontiguousarray(w, np.float64)
    R = np.empty(9)
    lib().ref_getSO3ExpMap(_p(w), _p(R))
    return R.reshape(3, 3)


# ---- post-BA pose-graph spreading: the UNMODIFIED slam/SL_GlobalPoseEstimation.cpp ----
PATH_PG = os.path.join(HERE, "_ref", "libposegraph_ref.so")
_lib_pg = None


def posegraph_spread(fixed, R, t, id1, id2, eR, et):
    """GlobalPoseGraph::computeNewCameraRotations + ::computeNewCameraTranslations of the reference
    (slam/SL_GlobalPoseEstimation.cpp:52-359) on the graph (nodes fixed/R/t, edges id1->id2 with
    eR/et), built the way RobustBundleRTS::constructCameraGraphs does.  Returns newR, newt."""
    global _lib_pg
    if _lib_pg is None:
        _lib_pg = C.CDLL(PATH_PG)
        _lib_pg.ref_posegraph_spread.argtypes = [C.c_int] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 6
        _lib_pg.ref_posegraph_spread.restype = None
    fx = np.ascontiguousarray(fixed, np.int32)
    n = fx.size
    R = np.ascontiguousarray(R, np.float64).reshape(n, 3, 3)
    t = np.ascontiguousarray(t, np.float64).reshape(n, 3)
    id1 = np.ascontiguousarray(id1, np.int32)
    id2 = np.ascontiguousarray(id2, np.int32)
    ne = id1.size
    eR = np.ascontiguousarray(eR, np.float64).reshape(ne, 3, 3)
    et = np.ascontiguousarray(et, np.float64).reshape(ne, 3)
    nR, nt = np.empty((n, 3, 3)), np.empty((n, 3))
    _lib_pg.ref_posegraph_spread(n, _p(fx), _p(R), _p(t), ne, _p(id1), _p(id2), _p(eR), _p(et), _p(nR), _p(nt))
    return nR, nt
