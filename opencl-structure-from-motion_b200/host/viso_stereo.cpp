// Host side of stereo odometry.  Reference behaviour restated (paths relative to /root/reference/viso):
//   process ................ viso_stereo.cpp:33-40     estimateMotion ............. viso_stereo.cpp:42-145
//   getInlier .............. viso_stereo.cpp:147-165   updateParameters ........... viso_stereo.cpp:167-215
//   observations ........... viso_stereo.cpp:217-226   residuals and Jacobian ..... viso_stereo.cpp:228-316
#include "viso_stereo.h"

#include <algorithm>
#include <cmath>

using std::vector;

VisualOdometryStereo::VisualOdometryStereo(parameters param) : VisualOdometry(param), param(param) {
  matcher->setIntrinsics(param.calib.f, param.calib.cu, param.calib.cv, param.base);
}
VisualOdometryStereo::~VisualOdometryStereo() {}

bool VisualOdometryStereo::process(uint8_t* I1, uint8_t* I2, uint32_t* dims, bool replace) {
  matcher->pushBack(I1, I2, dims, replace);
  if (Tr_valid) matcher->matchFeatures(2, &Tr_delta);
  else matcher->matchFeatures(2);
  matcher->bucketFeatures(param.bucket.max_features, param.bucket.bucket_width, param.bucket.bucket_height);
  p_matched = matcher->getMatches();
  return updateMotion();
}

bool VisualOdometryStereo::setRectification(const Rectification& r) {
  if (r.n_cams != 2 || !matcher->setRectification(r)) return false;
  param.calib.f = r.cams[0].f; param.calib.cu = r.cams[0].cu; param.calib.cv = r.cams[0].cv; param.base = r.base;
  matcher->setIntrinsics(param.calib.f, param.calib.cu, param.calib.cv, param.base);
  return true;
}

void VisualOdometryStereo::adoptMatcher(Matcher* external) {
  VisualOdometry::adoptMatcher(external);
  matcher->setIntrinsics(param.calib.f, param.calib.cu, param.calib.cv, param.base);
}

// one getRandomSample(N, 3) per RANSAC iteration, whether or not that iteration's fit fails (viso_stereo.cpp:39-40)
void VisualOdometryStereo::drawSamples(int32_t N) {
  samples_last.resize((size_t)param.ransac_iters * 3);
  for (int32_t k = 0; k < param.ransac_iters; k++) {
    vector<int> s = getRandomSample(N, 3);
    std::copy(s.begin(), s.end(), samples_last.begin() + (size_t)k * 3);
  }
}

bool VisualOdometryStereo::batchPrepare(const visocu_pmatch** matches, int32_t* N, const int32_t** samples) {
  matcher->bucketFeatures(param.bucket.max_features, param.bucket.bucket_width, param.bucket.bucket_height);
  p_matched = matcher->getMatches();
  return prepareEstimate(matches, N, samples);
}

bool VisualOdometryStereo::batchPrepare(const vector<Matcher::p_match>& p_matched_, const visocu_pmatch** matches, int32_t* N,
                                        const int32_t** samples) {
  p_matched = p_matched_;
  return prepareEstimate(matches, N, samples);
}

bool VisualOdometryStereo::prepareEstimate(const visocu_pmatch** matches, int32_t* N, const int32_t** samples) {
  batch_ready = false;
  if ((int32_t)p_matched.size() < 6) return false;
  drawSamples((int32_t)p_matched.size());
  *matches = reinterpret_cast<const visocu_pmatch*>(p_matched.data());
  *N = (int32_t)p_matched.size();
  *samples = samples_last.data();
  batch_ready = true;
  return true;
}

// the state estimateMotion + updateMotion leave: the winner's inliers even if the refinement fails, the motion if it converged
bool VisualOdometryStereo::batchFinish(const double* tr6, int32_t ok, const uint8_t* inlier_mask) {
  if (!batch_ready) return false;
  batch_ready = false;
  inliers.clear();
  for (size_t i = 0; i < p_matched.size(); i++)
    if (inlier_mask[i]) inliers.push_back((int32_t)i);
  return setMotion(ok ? vector<double>(tr6, tr6 + 6) : vector<double>());
}

vector<double> VisualOdometryStereo::estimateMotion(vector<Matcher::p_match> p_matched) {
  const int32_t N = (int32_t)p_matched.size();
  if (N < 6) return vector<double>();
  drawSamples(N);
  // previous stereo matches -> 3-D points in the previous left camera frame
  X.resize(N); Y.resize(N); Z.resize(N);
  for (int32_t i = 0; i < N; i++) {
    const double d = std::max(p_matched[i].u1p - p_matched[i].u2p, 0.0001f);
    X[i] = (p_matched[i].u1p - param.calib.cu) * param.base / d;
    Y[i] = (p_matched[i].v1p - param.calib.cv) * param.base / d;
    Z[i] = param.calib.f * param.base / d;
  }
  vector<double> tr_delta, tr_curr(6);
  inliers.clear();
  // RANSAC over 3-point Gauss-Newton fits
  for (int32_t k = 0; k < param.ransac_iters; k++) {
    vector<int32_t> active(samples_last.begin() + (size_t)k * 3, samples_last.begin() + (size_t)k * 3 + 3);
    for (int32_t i = 0; i < 6; i++) tr_curr[i] = 0;
    result res = UPDATED;
    int32_t iter = 0;
    while (res == UPDATED) {
      res = updateParameters(p_matched, active, tr_curr, 1, 1e-6);
      if (iter++ > 20 || res == CONVERGED) break;
    }
    if (res != FAILED) {
      vector<int32_t> cur = getInlier(p_matched, tr_curr);
      if (cur.size() > inliers.size()) { inliers = cur; tr_delta = tr_curr; }
    }
  }
  // final refinement on all inliers
  bool success = true;
  if (inliers.size() >= 6) {
    int32_t iter = 0;
    result res = UPDATED;
    while (res == UPDATED) {
      res = updateParameters(p_matched, inliers, tr_delta, 1, 1e-8);
      if (iter++ > 100 || res == CONVERGED) break;
    }
    if (res != CONVERGED) success = false;
  } else {
    success = false;
  }
  return success ? tr_delta : vector<double>();
}

vector<int32_t> VisualOdometryStereo::getInlier(const vector<Matcher::p_match>& p_matched, const vector<double>& tr) {
  vector<int32_t> all(p_matched.size());
  for (size_t i = 0; i < all.size(); i++) all[i] = (int32_t)i;
  residualsAndJacobian(p_matched, all, tr, false);
  const double thr2 = param.inlier_threshold * param.inlier_threshold;
  vector<int32_t> in;
  for (size_t i = 0; i < all.size(); i++) {
    double e = 0;
    for (int k = 0; k < 4; k++) e += pow(observe[4 * i + k] - predict[4 * i + k], 2);
    if (e < thr2) in.push_back((int32_t)i);
  }
  return in;
}

VisualOdometryStereo::result VisualOdometryStereo::updateParameters(const vector<Matcher::p_match>& p_matched, const vector<int32_t>& active,
                                                                    vector<double>& tr, double step_size, double eps) {
  if (active.size() < 3) return FAILED;
  residualsAndJacobian(p_matched, active, tr, true);
  // normal equations J^T J x = J^T r
  Matrix A(6, 6), B(6, 1);
  const int32_t rows = 4 * (int32_t)active.size();
  for (int32_t m = 0; m < 6; m++) {
    for (int32_t n = 0; n < 6; n++) {
      double a = 0;
      for (int32_t i = 0; i < rows; i++) a += Jac[i * 6 + m] * Jac[i * 6 + n];
      A.val[m][n] = a;
    }
    double b = 0;
    for (int32_t i = 0; i < rows; i++) b += Jac[i * 6 + m] * residual[i];
    B.val[m][0] = b;
  }
  if (!B.solve(A)) return FAILED;
  bool converged = true;
  for (int32_t m = 0; m < 6; m++) {
    tr[m] += step_size * B.val[m][0];
    if (fabs(B.val[m][0]) > eps) converged = false;
  }
  return converged ? CONVERGED : UPDATED;
}

void VisualOdometryStereo::residualsAndJacobian(const vector<Matcher::p_match>& p_matched, const vector<int32_t>& active,
                                                const vector<double>& tr, bool want_jacobian) {
  const size_t n = active.size();
  observe.resize(4 * n); predict.resize(4 * n); residual.resize(4 * n);
  if (want_jacobian) Jac.resize(24 * n);
  const double sx = sin(tr[0]), cx = cos(tr[0]), sy = sin(tr[1]), cy = cos(tr[1]), sz = sin(tr[2]), cz = cos(tr[2]);
  const double tx = tr[3], ty = tr[4], tz = tr[5];
  // R = Rx(rx) Ry(ry) Rz(rz) and its derivatives with respect to the three angles
  const double R[3][3] = {{+cy * cz, -cy * sz, +sy},
                          {+sx * sy * cz + cx * sz, -sx * sy * sz + cx * cz, -sx * cy},
                          {-cx * sy * cz + sx * sz, +cx * sy * sz + sx * cz, +cx * cy}};
  const double dRx[3][3] = {{0, 0, 0},
                            {+cx * sy * cz - sx * sz, -cx * sy * sz - sx * cz, -cx * cy},
                            {+sx * sy * cz + cx * sz, -sx * sy * sz + cx * cz, -sx * cy}};
  const double dRy[3][3] = {{-sy * cz, +sy * sz, +cy},
                            {+sx * cy * cz, -sx * cy * sz, +sx * sy},
                            {-cx * cy * cz, +cx * cy * sz, -cx * sy}};
  const double dRz[3][3] = {{-cy * sz, -cy * cz, 0},
                            {-sx * sy * sz + cx * cz, -sx * sy * cz - cx * sz, 0},
                            {+cx * sy * sz + sx * cz, +cx * sy * cz - sx * sz, 0}};
  const double f = param.calib.f, cu = param.calib.cu, cv = param.calib.cv;
  for (size_t i = 0; i < n; i++) {
    const Matcher::p_match& m = p_matched[active[i]];
    observe[4 * i + 0] = m.u1c; observe[4 * i + 1] = m.v1c; observe[4 * i + 2] = m.u2c; observe[4 * i + 3] = m.v2c;
    const double Xp = X[active[i]], Yp = Y[active[i]], Zp = Z[active[i]];
    const double X1c = R[0][0] * Xp + R[0][1] * Yp + R[0][2] * Zp + tx;
    const double Y1c = R[1][0] * Xp + R[1][1] * Yp + R[1][2] * Zp + ty;
    const double Z1c = R[2][0] * Xp + R[2][1] * Yp + R[2][2] * Zp + tz;
    double weight = 1.0;
    if (param.reweighting) weight = 1.0 / (fabs(observe[4 * i + 0] - cu) / fabs(cu) + 0.05);
    const double X2c = X1c - param.base;
    if (want_jacobian) {
      for (int32_t j = 0; j < 6; j++) {
        double Xd = 0, Yd = 0, Zd = 0;        // derivative of the point in current left coordinates w.r.t. parameter j
        if (j < 3) {
          const double (*D)[3] = j == 0 ? dRx : (j == 1 ? dRy : dRz);
          Xd = D[0][0] * Xp + D[0][1] * Yp + D[0][2] * Zp;
          Yd = D[1][0] * Xp + D[1][1] * Yp + D[1][2] * Zp;
          Zd = D[2][0] * Xp + D[2][1] * Yp + D[2][2] * Zp;
        } else {
          Xd = j == 3; Yd = j == 4; Zd = j == 5;
        }
        const double zz = Z1c * Z1c;
        Jac[(4 * i + 0) * 6 + j] = weight * f * (Xd * Z1c - X1c * Zd) / zz;
        Jac[(4 * i + 1) * 6 + j] = weight * f * (Yd * Z1c - Y1c * Zd) / zz;
        Jac[(4 * i + 2) * 6 + j] = weight * f * (Xd * Z1c - X2c * Zd) / zz;
        Jac[(4 * i + 3) * 6 + j] = weight * f * (Yd * Z1c - Y1c * Zd) / zz;
      }
    }
    predict[4 * i + 0] = f * X1c / Z1c + cu; predict[4 * i + 1] = f * Y1c / Z1c + cv;
    predict[4 * i + 2] = f * X2c / Z1c + cu; predict[4 * i + 3] = f * Y1c / Z1c + cv;
    for (int k = 0; k < 4; k++) residual[4 * i + k] = weight * (observe[4 * i + k] - predict[4 * i + k]);
  }
}
