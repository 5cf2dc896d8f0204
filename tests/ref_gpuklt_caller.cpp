// ref_gpuklt_caller.cpp -- runs the REFERENCE's own GPUKLT facade (tracking/GPUKLT.cpp) and its
// in-tree track / feature-point containers (tracking/SL_Track2D.cpp, slam/SL_FeaturePoints.cpp,
// slam/SL_FeaturePoint.cpp), compiled UNMODIFIED from the original CoSLAM tree, on top of
// coslam_b200/shim/v3d_gpuklt.h -> libcoslam_b200.so.  Test infrastructure: built into
// oracle/_ref/gpuklt_ref_caller by `make -C oracle ref REF=<CoSLAM checkout>`, run on a GPU by
// tests/golden/make_facade_ref_golden.py, whose stored output tests/test_gpu_ref_facade.py checks.
//
//   gpuklt_ref_caller <frames.raw> <W> <H> <nframes> <withGain> <feedEvery>
// frames.raw: nframes tightly packed W x H u8 images.  Prints, per frame, one line per live track:
//   F <frame> <slot> <track length> <x> <y>        (x, y in pixels as stored in the FeaturePoint)
// LibVisualSLAM's undistorPoint is not in the tree: identity here (k_ud = 0 means no distortion).
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "GPUKLT.h"
#include "SL_error.h"

void undistorPoint(const double*, const double*, const double* in, double* out) {
  out[0] = in[0];
  out[1] = in[1];
}

int main(int argc, char** argv) {
  if (argc < 7) return 2;
  const int W = std::atoi(argv[2]), H = std::atoi(argv[3]), nfr = std::atoi(argv[4]);
  const int gain = std::atoi(argv[5]), feedEvery = std::atoi(argv[6]);
  std::vector<unsigned char> frames((size_t)W * H * nfr);
  FILE* f = std::fopen(argv[1], "rb");
  if (!f || std::fread(frames.data(), 1, frames.size(), f) != frames.size()) return 3;
  std::fclose(f);
  // the live configuration of the reference (app/SL_GlobParam.cpp:28-34, gui/MyApp.cpp:210-211)
  V3D_GPU::KLT_SequenceTrackerConfig cfg;
  cfg.nIterations = 12;
  cfg.nLevels = 6;
  cfg.levelSkip = 2;
  cfg.windowWidth = 6;
  cfg.trackBorderMargin = 4.0f;
  cfg.convergenceThreshold = 1.0f;
  cfg.SSD_Threshold = 20000.0f;
  cfg.trackWithGain = gain != 0;
  cfg.minDistance = 8;
  cfg.minCornerness = 3000.0f;
  const double K[9] = {0.9 * W, 0, W / 2.0, 0, 0.9 * W, H / 2.0, 0, 0, 1};
  const double iK[9] = {1 / K[0], 0, -K[2] / K[0], 0, 1 / K[4], -K[5] / K[4], 0, 0, 1};
  const double kud[7] = {0, 0, 0, 0, 0, 0, 0};
  try {
    GPUKLT klt;
    FeaturePoints ips;
    klt.setIntrinsicParam(K, iK, kud);
    klt.init(0, W, H, &cfg);
    for (int fr = 0; fr < nfr; ++fr) {
      const unsigned char* img = frames.data() + (size_t)W * H * fr;
      const int n = (fr == 0) ? klt.first(0, img, ips) : klt.next(img, ips);
      if (feedEvery > 0 && fr > 0 && fr % feedEvery == 0) {
        // SingleSLAM::feedExtraFeatPtsToTracker: push a few externally matched points back in
        std::vector<FeaturePoint*> ext;
        for (int k = 0; k < 5; ++k)
          ext.push_back(ips.add(klt.currentFrame(), 0, W * (0.2 + 0.15 * k), H * (0.3 + 0.1 * k)));
        const int nf = klt.feedExternFeatPoints(ext);
        std::printf("X %d %d\n", fr, nf);
      }
      std::printf("N %d %d\n", fr, n);
      for (int i = 0; i < klt.m_nMaxCorners; ++i) {
        const Track2D& tk = klt.m_tks[i];
        if (tk.tail) std::printf("F %d %d %d %.9g %.9g\n", fr, i, tk.length(), tk.tail->x, tk.tail->y);
      }
    }
  } catch (const std::exception& e) {
    std::printf("E %s\n", e.what());
    return 1;
  }
  return 0;
}
