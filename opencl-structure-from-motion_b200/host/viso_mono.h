// Monocular visual odometry with the reference's interface (viso/viso_mono.h:27-88).  The RANSAC step
// (ransacEstimateF, the reference's accelerator hook viso_mono.h:74 / viso_mono_cl.cpp:153-194) runs on the GPU
// through visocu_ransac_F; the remaining pose recovery stays on the host for now (SURVEY.md 8f rank 2).
#ifndef VISOB_VISO_MONO_H
#define VISOB_VISO_MONO_H
#include "viso.h"

class VisualOdometryMono : public VisualOdometry {
public:
  struct parameters : public VisualOdometry::parameters {
    double height;            // camera height above ground (meters)
    double pitch;             // camera pitch (rad, negative=pointing down)
    int32_t ransac_iters;     // number of RANSAC iterations
    double inlier_threshold;  // fundamental matrix inlier threshold
    double motion_threshold;  // directly return false on small motions
    parameters() {
      height = 1.0; pitch = 0.0; ransac_iters = 2000; inlier_threshold = 0.00001; motion_threshold = 100.0;
    }
  };

  VisualOdometryMono(parameters param);
  ~VisualOdometryMono();

  // returns false if the motion is too small or an error occurred; valid after two calls
  bool process(uint8_t* I, uint32_t* dims, bool replace = false);

  // extension: raw camera images (Matcher::setRectification); the calibration becomes the rectified projection of
  // r.cams[0].  Before the first frame only: afterwards it returns false and changes nothing.
  bool setRectification(const Rectification& r);

  // extensions for tests / the batch runner
  bool processDevice(const uint8_t* d_I, uint32_t* dims, bool replace = false);
  // the second half of process() for callers that pushed and matched through a MatcherBatch: bucketing + motion
  bool processMatched();
  // batched RANSAC (sequence runner): batchPrepare buckets, normalises and draws the samples of this sequence;
  // the caller runs visocu_ransac_F for several sequences at once and hands F and the inlier mask to batchFinish
  bool batchPrepare(const float** uv, int32_t* N, const int32_t** samples);
  bool batchFinish(const double* F9, const uint8_t* mask);
  // The same finish in three steps, so that a caller with several sequences can run the two GPU stages of the pose
  // recovery (four triangulations, ground-plane vote) as ONE batched call each: poseStageA (after RANSAC) fills the
  // triangulation request, poseStageB (after visocu_triangulate_batch) the plane-vote request, poseStageC (after
  // visocu_best_plane_batch) sets the motion.  A stage that returns false ends the frame (process() == false).
  struct PoseRequest {
    std::vector<float> uv; int32_t N; double P1[12], P2[48];          // triangulation: matches in pixels, 4 candidate cameras
    std::vector<double> X; int32_t n_front[4];                       // its results: 4 x (4 x N) points, points in front
    std::vector<double> d; double threshold, weight;                 // plane vote: distances along the road normal
  };
  bool poseStageA(const double* F9, const uint8_t* mask);
  bool poseStageB();
  bool poseStageC(int32_t best_idx);
  PoseRequest& poseRequest() { return pose; }
  const Matrix& lastF() const { return F_last; }
  const std::vector<int>& lastSamples() const { return samples_last; }

private:
  virtual Matrix ransacEstimateF(const std::vector<Matcher::p_match>& p_matched);
  virtual double findBestPlane(const Matrix& x_plane, double threshold, double weight);
  std::vector<double> estimateMotion(std::vector<Matcher::p_match> p_matched);
  std::vector<double> poseFromF(Matrix F, std::vector<Matcher::p_match>& p_matched, Matrix& Tp, Matrix& Tc);
  void drawSamples(int32_t N);
  void packNormalized(const std::vector<Matcher::p_match>& pm);
  Matrix smallerThanMedian(Matrix& X, double& median);
  bool normalizeFeaturePoints(std::vector<Matcher::p_match>& p_matched, Matrix& Tp, Matrix& Tc);
  int32_t triangulateChieral(std::vector<Matcher::p_match>& p_matched, Matrix& K, Matrix& R, Matrix& t, Matrix& X);

protected:
  parameters param;
  Matrix F_last;
  std::vector<int> samples_last;
  std::vector<float> uv_last;
  std::vector<Matcher::p_match> normalized_last;
  Matrix Tp_last, Tc_last;
  bool batch_ready = false;
  PoseRequest pose;
  Matrix pose_K, pose_Rs[4], pose_ts[4], pose_R, pose_t;
  bool poseBegin(Matrix F, std::vector<Matcher::p_match>& p_matched, Matrix& Tp, Matrix& Tc);
  bool poseMiddle();
  std::vector<double> poseEnd(int32_t best_idx);
};
#endif
