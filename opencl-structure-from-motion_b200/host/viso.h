// VisualOdometry base class with the reference's interface (viso/viso.h:28-142).
#ifndef VISOB_VISO_H
#define VISOB_VISO_H
#include <random>
#include <vector>

#include "matcher.h"
#include "matrix.h"

class VisualOdometry {
public:
  struct calibration {
    double f, cu, cv;
    calibration() { f = 1; cu = 0; cv = 0; }
  };
  struct bucketing {
    int32_t max_features;
    double bucket_width, bucket_height;
    bucketing() { max_features = 2; bucket_width = 50; bucket_height = 50; }
  };
  struct parameters {
    Matcher::parameters match;
    VisualOdometry::bucketing bucket;
    VisualOdometry::calibration calib;
  };

  VisualOdometry(parameters param);
  virtual ~VisualOdometry();

  bool process(std::vector<Matcher::p_match> p_matched_) {
    p_matched = p_matched_;
    return updateMotion();
  }
  Matrix getMotion() { return Tr_delta; }
  std::vector<Matcher::p_match> getMatches() { return matcher->getMatches(); }
  int32_t getNumberOfMatches() { return (int32_t)p_matched.size(); }
  int32_t getNumberOfInliers() { return (int32_t)inliers.size(); }
  std::vector<int32_t> getInlierIndices() { return inliers; }
  float getGain(std::vector<int32_t> inliers_) { return matcher->getGain(inliers_); }

  friend std::ostream& operator<<(std::ostream& os, VisualOdometry& viso) {
    Matrix p = viso.getMotion();
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 4; j++) os << p.val[i][j] << (i == 2 && j == 3 ? "" : " ");
    return os;
  }

  // extension: the matches fed to the last motion estimate (after bucketing)
  const std::vector<Matcher::p_match>& usedMatches() const { return p_matched; }
  Matcher* getMatcher() { return matcher; }
  // extension: run on a matcher owned by somebody else (a MatcherBatch sequence); the own one is released
  void adoptMatcher(Matcher* external);

protected:
  bool updateMotion();
  // the end of updateMotion: a 6-vector (rx, ry, rz, tx, ty, tz) becomes Tr_delta and Tr_valid; any other size is a failed
  // estimate and leaves both as they are
  bool setMotion(const std::vector<double>& tr);
  Matrix transformationVectorToMatrix(std::vector<double> tr);
  virtual std::vector<double> estimateMotion(std::vector<Matcher::p_match> p_matched) = 0;
  // num distinct indices out of 0..N-1 by a partial Fisher-Yates shuffle (viso.cpp:86-102).  The reference keeps
  // its std::default_random_engine(71) in a function-static shared by every instance of the process; here each
  // object owns one, which gives the same sequence for a single object and makes sharded runs reproducible.
  std::vector<int> getRandomSample(unsigned N, unsigned num);

  Matrix Tr_delta;
  bool Tr_valid;
  Matcher* matcher;
  bool owns_matcher;
  std::vector<int32_t> inliers;
  double* J;
  double* p_observe;
  double* p_predict;
  std::vector<Matcher::p_match> p_matched;
  std::default_random_engine sample_generator;
  std::vector<int> sample_pool;                     // identity permutation reused by getRandomSample

private:
  parameters param;
};
#endif
