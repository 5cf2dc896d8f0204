// Test infrastructure: compiled against coslam_b200/shim/SL_GlobalPoseEstimation.h standing in for the
// reference's slam/SL_GlobalPoseEstimation.h (tests/test_shim_reference_callers.py).  The body
// follows the calls RobustBundleRTS::constructCameraGraphs / updateNonKeyCameraPoses make
// (reference app/SL_CoSLAMRobustBA.cpp:182-250): the shim is a drop-in for the header on that path.
#include <cassert>  // the reference header gets it through LibVisualSLAM's math/SL_Matrix.h
#include <cstring>

#include "slam/SL_GlobalPoseEstimation.h"

double probe_posegraph(int n, const double* Rs, const double* ts, const double* eR, const double* et) {
  GlobalPoseGraph graphs[2];
  GlobalPoseGraph& g = graphs[0];
  g.clear();
  g.reserve(n, n);
  for (int k = 0; k < n; ++k) {
    CamPoseNode* node = g.newNode();
    node->set(k, 0, Rs + 9 * k, ts + 3 * k);
    int id = node->id;
    (void)id;
  }
  CamPoseNode* fixedNode = &g.poseNodes[0];
  fixedNode->fixed = true;
  for (int k = 1; k < n; ++k) {
    CamPoseEdge* edge = g.addEdge();
    edge->set(k - 1, k, eR + 9 * (k - 1), et + 3 * (k - 1));
  }
  std::memcpy(g.poseNodes[0].R, Rs, sizeof(double) * 9);
  g.computeNewCameraRotations();
  g.computeNewCameraTranslations();
  double s = 0;
  for (int i = 0; i < g.nNodes; i++)
    if (!g.poseNodes[i].fixed) s += g.poseNodes[i].newR[0] + g.poseNodes[i].newt[0];
  return s + g.nEdges + g.nFixedNode + g.nConstraintEdge;
}
