// Host side of monocular odometry.  Reference behaviour restated (paths relative to /root/reference/viso):
//   process ............... viso_mono.cpp:33-39     estimateMotion ........ viso_mono.cpp:100-190
//   ransacEstimateF ....... viso_mono.cpp:41-72     normalizeFeaturePoints  viso_mono.cpp:217-263
//   findBestPlane ......... viso_mono.cpp:74-98     smallerThanMedian ..... viso_mono.cpp:192-215
//   EtoRt ................. viso_mono.cpp:347-392   triangulateChieral .... viso_mono.cpp:394-431
#include "viso_mono.h"

#include <algorithm>
#include <cmath>
#include <iostream>
#include <numeric>

#include "visocu.h"

#include <atomic>
#include <chrono>
namespace visob {
extern std::atomic<long long> g_stage_ns[8];
extern std::atomic<long long> g_stage_calls[8];
}
namespace {
struct MonoTimer {
  int id; std::chrono::steady_clock::time_point t0;
  explicit MonoTimer(int id) : id(id), t0(std::chrono::steady_clock::now()) {}
  ~MonoTimer() {
    visob::g_stage_ns[id] += std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
    visob::g_stage_calls[id]++;
  }
};
}

using std::vector;

VisualOdometryMono::VisualOdometryMono(parameters param) : VisualOdometry(param), param(param) {}

bool VisualOdometryMono::setRectification(const Rectification& r) {
  if (!matcher->setRectification(r)) return false;
  if (r.n_cams > 0) { param.calib.f = r.cams[0].f; param.calib.cu = r.cams[0].cu; param.calib.cv = r.cams[0].cv; }
  return true;
}
VisualOdometryMono::~VisualOdometryMono() {}

bool VisualOdometryMono::process(uint8_t* I, uint32_t* dims, bool replace) {
  matcher->pushBack(I, dims, replace);
  matcher->matchFeatures(0);
  matcher->bucketFeatures(param.bucket.max_features, param.bucket.bucket_width, param.bucket.bucket_height);
  p_matched = matcher->getMatches();
  return updateMotion();
}

bool VisualOdometryMono::processDevice(const uint8_t* d_I, uint32_t* dims, bool replace) {
  matcher->pushBackDevice(d_I, 0, dims, replace);
  matcher->matchFeatures(0);
  matcher->bucketFeatures(param.bucket.max_features, param.bucket.bucket_width, param.bucket.bucket_height);
  p_matched = matcher->getMatches();
  return updateMotion();
}

bool VisualOdometryMono::processMatched() {
  matcher->bucketFeatures(param.bucket.max_features, param.bucket.bucket_width, param.bucket.bucket_height);
  p_matched = matcher->getMatches();
  return updateMotion();
}

// GPU RANSAC.  The host only draws the sample table with the reference's generator, in the reference's order
// (one getRandomSample per iteration), so a run is comparable with the reference hypothesis by hypothesis.
void VisualOdometryMono::drawSamples(int32_t N) {
  const int32_t iters = param.ransac_iters;
  samples_last.resize((size_t)iters * 8);
  for (int32_t k = 0; k < iters; k++) {
    vector<int> s = getRandomSample(N, 8);
    std::copy(s.begin(), s.end(), samples_last.begin() + (size_t)k * 8);
  }
}

void VisualOdometryMono::packNormalized(const vector<Matcher::p_match>& pm) {
  uv_last.resize(pm.size() * 4);
  for (size_t i = 0; i < pm.size(); i++) {
    uv_last[4 * i + 0] = pm[i].u1p; uv_last[4 * i + 1] = pm[i].v1p;
    uv_last[4 * i + 2] = pm[i].u1c; uv_last[4 * i + 3] = pm[i].v1c;
  }
}

Matrix VisualOdometryMono::ransacEstimateF(const vector<Matcher::p_match>& p_matched) {
  MonoTimer timer(6);
  inliers.clear();
  const int32_t N = (int32_t)p_matched.size(), iters = param.ransac_iters;
  drawSamples(N);
  packNormalized(p_matched);
  vector<uint8_t> mask(N);
  double F9[9];
  int32_t n_inl = 0, best = -1;
  const float* uvp = uv_last.data();
  const int32_t* sp = samples_last.data();
  uint8_t* mp = mask.data();
  visocu_ctx* ctx = matcher->context();
  if (!ctx || visocu_ransac_F(ctx, 1, &uvp, &N, &sp, iters, param.inlier_threshold, F9, &mp, &n_inl, &best, 0, 0) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    return Matrix();
  }
  for (int32_t i = 0; i < N; i++)
    if (mask[i]) inliers.push_back(i);
  if (inliers.size() < 10) return Matrix();
  return Matrix(3, 3, F9);
}

// ---- batched variant used by the sequence runner: the RANSAC of several sequences is ONE visocu_ransac_F call
bool VisualOdometryMono::batchPrepare(const float** uv, int32_t* N, const int32_t** samples) {
  MonoTimer timer(6);
  matcher->bucketFeatures(param.bucket.max_features, param.bucket.bucket_width, param.bucket.bucket_height);
  p_matched = matcher->getMatches();
  batch_ready = false;
  if ((int32_t)p_matched.size() < 10) return false;
  normalized_last = p_matched;
  if (!normalizeFeaturePoints(normalized_last, Tp_last, Tc_last)) return false;
  drawSamples((int32_t)normalized_last.size());
  packNormalized(normalized_last);
  *uv = uv_last.data(); *N = (int32_t)normalized_last.size(); *samples = samples_last.data();
  batch_ready = true;
  return true;
}

bool VisualOdometryMono::batchFinish(const double* F9, const uint8_t* mask) {
  MonoTimer timer(7);
  if (!batch_ready) return false;
  inliers.clear();
  for (size_t i = 0; i < normalized_last.size(); i++)
    if (mask[i]) inliers.push_back((int32_t)i);
  if (inliers.size() < 10) return false;
  Matrix F(3, 3, F9);
  F_last = F;
  vector<double> tr = poseFromF(F, p_matched, Tp_last, Tc_last);
  if (tr.size() != 6) return false;
  Tr_delta = transformationVectorToMatrix(tr);
  Tr_valid = true;
  return true;
}

// GPU Gaussian vote (the reference's second accelerator hook, viso_mono.h:75 / viso_mono_cl.cpp:255-280)
double VisualOdometryMono::findBestPlane(const Matrix& x_plane, double threshold, double weight) {
  // signed distance of every point along the plane normal, then the mode of a Gaussian kernel density
  const double ny = cos(-param.pitch), nz = sin(-param.pitch);
  const int32_t n = x_plane.n;
  vector<double> d(n);
  for (int32_t i = 0; i < n; i++) d[i] = ny * x_plane.val[0][i] + nz * x_plane.val[1][i];
  int32_t best_idx = 0;
  visocu_ctx* ctx = matcher->context();
  if (!ctx || visocu_best_plane(ctx, d.data(), n, threshold, weight, &best_idx) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    return d[0];
  }
  return d[best_idx];
}

vector<double> VisualOdometryMono::estimateMotion(vector<Matcher::p_match> p_matched) {
  MonoTimer timer(7);
  const int32_t N = (int32_t)p_matched.size();
  if (N < 10) return vector<double>();
  Matrix Tp, Tc;
  vector<Matcher::p_match> normalized = p_matched;
  if (!normalizeFeaturePoints(normalized, Tp, Tc)) return vector<double>();

  Matrix F = ransacEstimateF(normalized);
  if (F.val == 0) return vector<double>();
  F_last = F;
  return poseFromF(F, p_matched, Tp, Tc);
}

// everything of estimateMotion after the RANSAC step (viso_mono.cpp:125-189)
// Pose from F (viso_mono.cpp:100-190 after the RANSAC) in three host phases around the two GPU stages.
// Phase 1: denormalise, essential matrix, the four (R, t) candidates of EtoRt (viso_mono.cpp:347-392).
bool VisualOdometryMono::poseBegin(Matrix F, vector<Matcher::p_match>& p_matched, Matrix& Tp, Matrix& Tc) {
  double K_data[9] = {param.calib.f, 0, param.calib.cu, 0, param.calib.f, param.calib.cv, 0, 0, 1};
  pose_K = Matrix(3, 3, K_data);
  Matrix& K = pose_K;
  F = ~Tc * F * Tp;
  Matrix E = ~K * F * K;
  Matrix U, W, V;
  E.svd(U, W, V);
  W.val[2][0] = 0;
  E = U * Matrix::diag(W) * ~V;

  double W_data[9] = {0, -1, 0, +1, 0, 0, 0, 0, 1};
  double Z_data[9] = {0, +1, 0, -1, 0, 0, 0, 0, 0};
  Matrix Wm(3, 3, W_data), Z(3, 3, Z_data);
  Matrix S;
  E.svd(U, S, V);
  Matrix T = U * Z * ~U;
  Matrix Ra = U * Wm * (~V);
  Matrix Rb = U * (~Wm) * (~V);
  Matrix t(3, 1);
  t.val[0][0] = T.val[2][1]; t.val[1][0] = T.val[0][2]; t.val[2][0] = T.val[1][0];
  if (Ra.det() < 0) Ra = -Ra;
  if (Rb.det() < 0) Rb = -Rb;
  // four (R, t) candidates; all four triangulations (4 N independent 4x4 null-vector problems) run in one GPU launch
  pose_Rs[0] = Ra; pose_Rs[1] = Ra; pose_Rs[2] = Rb; pose_Rs[3] = Rb;
  pose_ts[0] = t; pose_ts[1] = -t; pose_ts[2] = t; pose_ts[3] = -t;
  const int32_t N = (int32_t)p_matched.size();
  Matrix P1(3, 4);
  P1.setMat(K, 0, 0);
  P1.getData(pose.P1);
  for (int32_t i = 0; i < 4; i++) {
    Matrix P2(3, 4);
    P2.setMat(pose_Rs[i], 0, 0);
    P2.setMat(pose_ts[i], 0, 3);
    P2 = K * P2;
    P2.getData(pose.P2 + 12 * i);
  }
  pose.N = N;
  pose.uv.resize((size_t)N * 4);
  for (int32_t i = 0; i < N; i++) {
    pose.uv[4 * i + 0] = p_matched[i].u1p; pose.uv[4 * i + 1] = p_matched[i].v1p;
    pose.uv[4 * i + 2] = p_matched[i].u1c; pose.uv[4 * i + 3] = p_matched[i].v1c;
  }
  pose.X.resize((size_t)16 * N);
  for (int i = 0; i < 4; i++) pose.n_front[i] = 0;
  return N > 0;
}

// Phase 2: keep the candidate with most points in front of both cameras (first wins on ties), normalise, median test,
// distances along the road normal for the plane vote (viso_mono.cpp:134-160, 74-98).
bool VisualOdometryMono::poseMiddle() {
  const int32_t N = pose.N;
  Matrix X;
  int32_t max_inliers = 0;
  for (int32_t i = 0; i < 4; i++) {
    if (pose.n_front[i] > max_inliers) {
      max_inliers = pose.n_front[i];
      X = Matrix(4, N, pose.X.data() + (size_t)4 * N * i);
      pose_R = pose_Rs[i];
      pose_t = pose_ts[i];
    }
  }
  if (X.val == 0) return false;
  X = X / X.getMat(3, 0, 3, -1);
  vector<int32_t> pos_idx;
  for (int32_t i = 0; i < X.n; i++)
    if (X.val[2][i] > 0) pos_idx.push_back(i);
  Matrix X_plane = X.extractCols(pos_idx);
  if (X_plane.n < 10) return false;
  double median;
  smallerThanMedian(X_plane, median);
  if (median > param.motion_threshold) return false;
  const double sigma = median / 50.0;
  pose.weight = 1.0 / (2.0 * sigma * sigma);
  pose.threshold = median / param.motion_threshold;
  // signed distance of every point along the plane normal; the vote finds the mode of a Gaussian kernel density
  const double ny = cos(-param.pitch), nz = sin(-param.pitch);
  pose.d.resize(X_plane.n);
  for (int32_t i = 0; i < X_plane.n; i++) pose.d[i] = ny * X_plane.val[1][i] + nz * X_plane.val[2][i];
  return true;
}

// Phase 3: scale the translation with the camera height over the plane distance, Euler angles.
vector<double> VisualOdometryMono::poseEnd(int32_t best_idx) {
  const double best_d = pose.d[best_idx];
  Matrix t = pose_t * param.height / best_d;
  const Matrix& R = pose_R;
  const double ry = asin(R.val[0][2]);
  const double rx = asin(-R.val[1][2] / cos(ry));
  const double rz = asin(-R.val[0][1] / cos(ry));
  vector<double> tr(6);
  tr[0] = rx; tr[1] = ry; tr[2] = rz;
  tr[3] = t.val[0][0]; tr[4] = t.val[1][0]; tr[5] = t.val[2][0];
  return tr;
}

vector<double> VisualOdometryMono::poseFromF(Matrix F, vector<Matcher::p_match>& p_matched, Matrix& Tp, Matrix& Tc) {
  if (!poseBegin(F, p_matched, Tp, Tc)) return vector<double>();
  visocu_ctx* ctx = matcher->context();
  if (!ctx || visocu_triangulate(ctx, pose.uv.data(), pose.N, pose.P1, pose.P2, 4, pose.X.data(), pose.n_front) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    return vector<double>();
  }
  if (!poseMiddle()) return vector<double>();
  int32_t best_idx = 0;
  if (visocu_best_plane(ctx, pose.d.data(), (int32_t)pose.d.size(), pose.threshold, pose.weight, &best_idx) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    best_idx = 0;
  }
  return poseEnd(best_idx);
}

bool VisualOdometryMono::poseStageA(const double* F9, const uint8_t* mask) {
  MonoTimer timer(7);
  if (!batch_ready) return false;
  inliers.clear();
  for (size_t i = 0; i < normalized_last.size(); i++)
    if (mask[i]) inliers.push_back((int32_t)i);
  if (inliers.size() < 10) return false;
  Matrix F(3, 3, F9);
  F_last = F;
  return poseBegin(F, p_matched, Tp_last, Tc_last);
}

bool VisualOdometryMono::poseStageB() {
  MonoTimer timer(7);
  return poseMiddle();
}

bool VisualOdometryMono::poseStageC(int32_t best_idx) {
  MonoTimer timer(7);
  vector<double> tr = poseEnd(best_idx);
  if (tr.size() != 6) return false;
  Tr_delta = transformationVectorToMatrix(tr);
  Tr_valid = true;
  return true;
}

Matrix VisualOdometryMono::smallerThanMedian(Matrix& X, double& median) {
  vector<double> dist(X.n);
  vector<int32_t> idx(X.n);
  for (int32_t i = 0; i < X.n; i++) dist[i] = fabs(X.val[0][i]) + fabs(X.val[1][i]) + fabs(X.val[2][i]);
  std::iota(idx.begin(), idx.end(), 0);
  std::sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return dist[a] < dist[b]; });
  const int32_t half = (int32_t)idx.size() / 2;
  median = dist[idx[half]];
  Matrix X_small(4, half + 1);
  for (int32_t j = 0; j <= half; j++)
    for (int32_t i = 0; i < 4; i++) X_small.val[i][j] = X.val[i][idx[j]];
  return X_small;
}

// Hartley normalisation.  The sums are accumulated in double but every intermediate coordinate is written back
// into the float fields of p_match, exactly like the reference (viso_mono.cpp:217-263): the rounding matters for
// the RANSAC inputs.
bool VisualOdometryMono::normalizeFeaturePoints(vector<Matcher::p_match>& p_matched, Matrix& Tp, Matrix& Tc) {
  const double n = (double)p_matched.size();
  double cpu = 0, cpv = 0, ccu = 0, ccv = 0;
  for (const Matcher::p_match& m : p_matched) { cpu += m.u1p; cpv += m.v1p; ccu += m.u1c; ccv += m.v1c; }
  cpu /= n; cpv /= n; ccu /= n; ccv /= n;
  for (Matcher::p_match& m : p_matched) { m.u1p -= cpu; m.v1p -= cpv; m.u1c -= ccu; m.v1c -= ccv; }
  double sp = 0, sc = 0;
  for (const Matcher::p_match& m : p_matched) {
    sp += std::sqrt(m.u1p * m.u1p + m.v1p * m.v1p);      // float sqrt of a float sum, as in the reference
    sc += std::sqrt(m.u1c * m.u1c + m.v1c * m.v1c);
  }
  if (fabs(sp) < 1e-10 || fabs(sc) < 1e-10) return false;
  sp = sqrt(2.0) * n / sp;
  sc = sqrt(2.0) * n / sc;
  for (Matcher::p_match& m : p_matched) { m.u1p *= sp; m.v1p *= sp; m.u1c *= sc; m.v1c *= sc; }
  double Tp_data[9] = {sp, 0, -sp * cpu, 0, sp, -sp * cpv, 0, 0, 1};
  double Tc_data[9] = {sc, 0, -sc * ccu, 0, sc, -sc * ccv, 0, 0, 1};
  Tp = Matrix(3, 3, Tp_data);
  Tc = Matrix(3, 3, Tc_data);
  return true;
}

int32_t VisualOdometryMono::triangulateChieral(vector<Matcher::p_match>& p_matched, Matrix& K, Matrix& R, Matrix& t, Matrix& X) {
  X = Matrix(4, (int32_t)p_matched.size());
  Matrix P1(3, 4), P2(3, 4);
  P1.setMat(K, 0, 0);
  P2.setMat(R, 0, 0);
  P2.setMat(t, 0, 3);
  P2 = K * P2;
  Matrix J(4, 4), U, S, V;
  for (int32_t i = 0; i < (int32_t)p_matched.size(); i++) {
    const Matcher::p_match& m = p_matched[i];
    for (int32_t j = 0; j < 4; j++) {
      J.val[0][j] = P1.val[2][j] * m.u1p - P1.val[0][j];
      J.val[1][j] = P1.val[2][j] * m.v1p - P1.val[1][j];
      J.val[2][j] = P2.val[2][j] * m.u1c - P2.val[0][j];
      J.val[3][j] = P2.val[2][j] * m.v1c - P2.val[1][j];
    }
    J.svd(U, S, V);
    for (int32_t r = 0; r < 4; r++) X.val[r][i] = V.val[r][3];
  }
  Matrix AX1 = P1 * X, BX1 = P2 * X;
  int32_t num = 0;
  for (int32_t i = 0; i < X.n; i++)
    if (AX1.val[2][i] * X.val[3][i] > 0 && BX1.val[2][i] * X.val[3][i] > 0) num++;
  return num;
}
