// Test infrastructure: uses slam/SL_IntraCamPose.h the way the reference's callers do and is compiled
// against coslam_b200/shim/SL_IntraCamPose.h (tests/test_shim_reference_callers.py).  The shim must
// accept the reference's function-pointer type and option members: it is a drop-in for the header.
#include "slam/SL_IntraCamPose.h"

typedef bool (*intraCamEstimate_t)(const double*, const double*, const double*, int, const double*,
                                   const double*, const double*, const double, double*, double*,
                                   IntraCamPoseOption*);
intraCamEstimate_t probe = &intraCamEstimate;

double use_every_member() {
  IntraCamPoseOption o;  // default constructible, as SingleSLAM::poseUpdate3D uses it
  o.maxIterLM = 100;
  o.maxIterRW = 5;
  o.epsErrorChangeLM = 1e-7;
  o.epsParamChangeLM = 1e-6;
  o.epsErrorChangeRW = 1e-6;
  o.verboseLM = 0;
  o.verboseRW = 0;
  o.lambda0 = 1e-3;
  return o.lambda + o.err0 + o.err + o.errRW + o.retTypeLM + o.npts + o.nIterLM + o.nIterRW;
}
