// Stereo visual odometry with the reference's interface (viso/viso_stereo.h:27-84): quad matching with the
// motion-predicted search window (GPU), then a 3-point RANSAC over Gauss-Newton minimisations of the reprojection error
// and a final refinement on all inliers.  process() runs that estimate on the host (double precision); it is also the
// reference the device estimate is tested against.  The sequence runner estimates the motion of many sequences with ONE
// visocu_stereo_motion call (GPU) through batchPrepare / batchFinish, which leave the same state as process().
#ifndef VISOB_VISO_STEREO_H
#define VISOB_VISO_STEREO_H
#include "viso.h"

class VisualOdometryStereo : public VisualOdometry {
public:
  struct parameters : public VisualOdometry::parameters {
    double base;              // baseline (meters)
    int32_t ransac_iters;     // number of RANSAC iterations
    double inlier_threshold;  // reprojection inlier threshold (pixels)
    bool reweighting;         // lower border weights (more robust to calibration errors)
    parameters() { base = 1.0; ransac_iters = 200; inlier_threshold = 2.0; reweighting = true; }
  };

  VisualOdometryStereo(parameters param);
  ~VisualOdometryStereo();

  // returns false if an error occurred; valid after two calls
  bool process(uint8_t* I1, uint8_t* I2, uint32_t* dims, bool replace = false);
  using VisualOdometry::process;

  // extensions for the batch runner and the tests
  // runs on a matcher owned by somebody else (a MatcherBatch sequence), with this object's calibration
  void adoptMatcher(Matcher* external);
  // The motion estimate in two halves around a batched visocu_stereo_motion call.  batchPrepare takes the matches as
  // process() does (bucketing the matcher's list) or as process(matches) does (the list given), and draws the sample table
  // (ransac_iters x 3, one getRandomSample(N, 3) per iteration, the order of estimateMotion).  It returns false, changing
  // nothing else, if there are fewer than 6 matches: the frame has failed as it does in process().  Otherwise the caller
  // runs visocu_stereo_motion on (matches, N, samples) and hands its results to batchFinish, which returns what process()
  // returns and leaves the same inliers, motion and validity.
  bool batchPrepare(const visocu_pmatch** matches, int32_t* N, const int32_t** samples);
  bool batchPrepare(const std::vector<Matcher::p_match>& p_matched_, const visocu_pmatch** matches, int32_t* N, const int32_t** samples);
  bool batchFinish(const double* tr6, int32_t ok, const uint8_t* inlier_mask);
  // the sample table of the last estimate (either path)
  const std::vector<int>& lastSamples() const { return samples_last; }

private:
  enum result { UPDATED, FAILED, CONVERGED };
  std::vector<double> estimateMotion(std::vector<Matcher::p_match> p_matched);
  bool prepareEstimate(const visocu_pmatch** matches, int32_t* N, const int32_t** samples);
  void drawSamples(int32_t N);
  result updateParameters(const std::vector<Matcher::p_match>& p_matched, const std::vector<int32_t>& active, std::vector<double>& tr,
                          double step_size, double eps);
  void residualsAndJacobian(const std::vector<Matcher::p_match>& p_matched, const std::vector<int32_t>& active,
                            const std::vector<double>& tr, bool want_jacobian);
  std::vector<int32_t> getInlier(const std::vector<Matcher::p_match>& p_matched, const std::vector<double>& tr);

  std::vector<double> X, Y, Z;                     // 3-D points of the previous stereo pair
  std::vector<double> Jac, predict, observe, residual;
  std::vector<int> samples_last;                   // ransac_iters x 3
  bool batch_ready = false;
  parameters param;
};
#endif
