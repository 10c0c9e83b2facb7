// Reconstruction (reference behaviour: viso/reconstruction.cpp:27-343), see reconstruction.h.
#include "reconstruction.h"
#include <assert.h>
#include <math.h>

using std::vector;

Point3d affineTransform(const Matrix& M, const Point3d& p) {
  // double accumulation on float coordinates, rounded to float on the way out (matrix.cpp:37-44)
  return Point3d((float)(p.x * M.val[0][0] + p.y * M.val[0][1] + p.z * M.val[0][2] + M.val[0][3]),
                 (float)(p.x * M.val[1][0] + p.y * M.val[1][1] + p.z * M.val[1][2] + M.val[1][3]),
                 (float)(p.x * M.val[2][0] + p.y * M.val[2][1] + p.z * M.val[2][2] + M.val[2][3]));
}

Reconstruction::Reconstruction() : next_id(0), job() { K = Matrix::eye(3); }
Reconstruction::~Reconstruction() {}

void Reconstruction::setCalibration(FLOAT f, FLOAT cu, FLOAT cv) {
  const FLOAT kd[9] = {f, 0, cu, 0, f, cv, 0, 0, 1};
  K = Matrix(3, 3, kd);
  const FLOAT pitch = -0.08, height = 1.6;
  Tr_cam_road = Matrix(4, 4);          // note: row 3 stays zero, only rows 0..2 are ever applied
  Tr_cam_road.val[0][0] = 1;
  Tr_cam_road.val[1][1] = +cos(pitch); Tr_cam_road.val[1][2] = -sin(pitch);
  Tr_cam_road.val[2][1] = +sin(pitch); Tr_cam_road.val[2][2] = +cos(pitch);
  Tr_cam_road.val[1][3] = -height;
}

void Reconstruction::update(vector<Matcher::p_match> p_matched, Matrix Tr, int32_t point_type, int32_t min_track_length,
                            double max_dist, double min_angle) {
  const visocu_recon_job& j = batchPrepare(p_matched, Tr, point_type, min_track_length, max_dist, min_angle);
  vector<int32_t> status((size_t)j.n_tracks);
  vector<float> xyz(3 * (size_t)j.n_tracks);
  hostEval(status.data(), xyz.data());
  batchFinish(status.data(), xyz.data());
}

const visocu_recon_job& Reconstruction::batchPrepare(const vector<Matcher::p_match>& p_matched, Matrix Tr, int32_t point_type,
                                                     int32_t min_track_length, double max_dist, double min_angle) {
  // everything already reconstructed moves into the new camera frame
  for (Point3d& p : points) p = affineTransform(Tr, p);
  return batchPrepareTracks(p_matched, Tr, point_type, min_track_length, max_dist, min_angle);
}

const visocu_recon_job& Reconstruction::batchPrepareTracks(const vector<Matcher::p_match>& p_matched, Matrix Tr, int32_t point_type,
                                                           int32_t min_track_length, double max_dist, double min_angle) {
  // frames no live track starts in are dropped from the old end; the rest are re-expressed relative to the new frame
  while (!frames.empty() && frames.front().track_count == 0) frames.pop_front();
  for (Frame& f : frames) {
    f.fwd = Tr * f.fwd;
    f.inv = Matrix::inv(f.fwd);
    f.proj = K * f.inv.getMat(0, 0, 2, 3);
  }
  {
    Frame f;
    f.fwd = Matrix::eye(4); f.inv = Matrix::eye(4); f.proj = K * f.fwd.getMat(0, 0, 2, 3);
    f.id = next_id++; f.track_count = 0;
    frames.push_back(f);
  }
  assert(frames.size() <= max_track_length);
  const int64_t now = frames.back().id;

  // feature index of the previous frame -> track that ended on it (a later track wins, as in the reference's map)
  int32_t idx_max = 0;
  for (const Matcher::p_match& m : p_matched) if (m.i1p > idx_max) idx_max = m.i1p;
  for (const Track& t : tracks) if (t.last_idx > idx_max) idx_max = t.last_idx;
  vector<int32_t> by_index((size_t)idx_max + 1, -1);
  for (size_t k = 0; k < tracks.size(); k++) by_index[tracks[k].last_idx] = (int32_t)k;

  for (const Matcher::p_match& m : p_matched) {
    int32_t k = by_index[m.i1p];
    if (k < 0 || tracks[k].refreshed) {
      // new track: it starts with the observation in the previous image, but is anchored at the newest frame
      // (reconstruction.cpp:88-94) -- the projections used later are shifted by one frame accordingly
      Track t;
      t.first_id = now; t.last_idx = 0; t.refreshed = false;
      t.pixels.push_back(Obs{m.u1p, m.v1p});
      frames.back().track_count += 1;
      tracks.push_back(t);
      k = (int32_t)tracks.size() - 1;
    }
    Track& t = tracks[k];
    if (t.pixels.size() < max_track_length) {
      t.pixels.push_back(Obs{m.u1c, m.v1c});
      t.last_idx = m.i1c;
      t.refreshed = true;
    }
  }

  // tracks that were not continued end here: the long enough ones go into the job, all of them are dropped (order
  // preserved)
  job_tracks.clear();
  size_t keep = 0;
  for (size_t k = 0; k < tracks.size(); k++) {
    Track& t = tracks[k];
    if (t.refreshed) {
      t.refreshed = false;
      if (keep != k) tracks[keep] = std::move(t);
      keep++;
      continue;
    }
    if ((int32_t)t.pixels.size() >= min_track_length) {
      visocu_recon_track r;
      r.first = (int32_t)(t.first_id - frames.front().id);
      r.n_obs = (int32_t)t.pixels.size();
      for (int32_t i = 0; i < 6; i++) {
        r.u[i] = i < r.n_obs ? t.pixels[i].u : 0.0f;
        r.v[i] = i < r.n_obs ? t.pixels[i].v : 0.0f;
      }
      job_tracks.push_back(r);
    }
    frame(t.first_id).track_count -= 1;
  }
  tracks.resize(keep);

  job_frames.resize(frames.size());
  for (size_t f = 0; f < frames.size(); f++) {
    const Frame& src = frames[f];
    visocu_recon_frame& d = job_frames[f];
    for (int r = 0; r < 3; r++) {
      for (int c = 0; c < 4; c++) { d.proj[4 * r + c] = src.proj.val[r][c]; d.inv[4 * r + c] = src.inv.val[r][c]; }
      d.center[r] = src.fwd.val[r][3];
    }
  }
  job.frames = job_frames.data(); job.n_frames = (int32_t)job_frames.size();
  job.tracks = job_tracks.data(); job.n_tracks = (int32_t)job_tracks.size();
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 4; c++) job.cam_road[4 * r + c] = Tr_cam_road.val[r][c];
  job.max_dist = max_dist; job.min_angle = min_angle; job.point_type = point_type;
  return job;
}

void Reconstruction::batchFinish(const int32_t* status, const float* xyz) {
  for (int32_t k = 0; k < job.n_tracks; k++)
    if (status[k] == 0) points.push_back(Point3d(xyz[3 * k], xyz[3 * k + 1], xyz[3 * k + 2]));
}

// status and point of every prepared track, with the meaning of visocu_recon_points (include/visocu.h)
void Reconstruction::hostEval(int32_t* status, float* xyz) const {
  for (int32_t k = 0; k < job.n_tracks; k++) {
    const visocu_recon_track& t = job_tracks[k];
    Point3d p(0, 0, 0);
    int32_t s = 0;
    if (!initPoint(t, p)) { s = 1; p = Point3d(0, 0, 0); }
    else if (pointType(t, p) < job.point_type) s = 2;
    else if (!refinePoint(t, p)) { s = 3; p = Point3d(0, 0, 0); }
    else if (!(pointDistance(t, p) < job.max_dist)) s = 4;
    else if (!(rayAngle(t, p) > job.min_angle)) s = 5;
    status[k] = s;
    xyz[3 * k] = p.x; xyz[3 * k + 1] = p.y; xyz[3 * k + 2] = p.z;
  }
}

// rows 0..2 of a row-major 3x4 table applied to (p, 1): affineTransform on a job's table
static Point3d affine12(const double* M, const Point3d& p) {
  return Point3d((float)(p.x * M[0] + p.y * M[1] + p.z * M[2] + M[3]),
                 (float)(p.x * M[4] + p.y * M[5] + p.z * M[6] + M[7]),
                 (float)(p.x * M[8] + p.y * M[9] + p.z * M[10] + M[11]));
}

// linear triangulation from the first and the last observation: null vector of the 4x4 system
bool Reconstruction::initPoint(const visocu_recon_track& t, Point3d& p) const {
  const double* P1 = job_frames[t.first].proj;
  const double* P2 = job_frames.back().proj;
  const int32_t last = t.n_obs - 1;
  Matrix J(4, 4), U, S, V;
  for (int32_t j = 0; j < 4; j++) {
    J.val[0][j] = P1[8 + j] * t.u[0] - P1[j];
    J.val[1][j] = P1[8 + j] * t.v[0] - P1[4 + j];
    J.val[2][j] = P2[8 + j] * t.u[last] - P2[j];
    J.val[3][j] = P2[8 + j] * t.v[last] - P2[4 + j];
  }
  J.svd(U, S, V);
  const float w = (float)V.val[3][3];
  if (fabs(w) < 1e-10) return false;            // point at infinity
  p = Point3d((float)(V.val[0][3] / w), (float)(V.val[1][3] / w), (float)(V.val[2][3] / w));
  return true;
}

// Gauss-Newton on the reprojection error over all observations of the track; observation k is predicted with the
// projection of frame first + k.  At most 22 steps; only a converged point (all updates below 1e-5) is accepted.
bool Reconstruction::refinePoint(const visocu_recon_track& t, Point3d& p) const {
  const int32_t nf = t.n_obs;
  FLOAT J[36], res[12];
  for (int32_t iter = 0;; iter++) {
    for (int32_t k = 0; k < nf; k++) {
      const double* P = job_frames[t.first + k].proj;
      const FLOAT a = P[0] * p.x + P[1] * p.y + P[2] * p.z + P[3];
      const FLOAT b = P[4] * p.x + P[5] * p.y + P[6] * p.z + P[7];
      const FLOAT c = P[8] * p.x + P[9] * p.y + P[10] * p.z + P[11];
      const FLOAT cc = c * c;
      if (cc < 1e-10) return false;
      for (int32_t j = 0; j < 3; j++) {
        J[6 * k + j] = (P[j] * c - P[8 + j] * a) / cc;
        J[6 * k + 3 + j] = (P[4 + j] * c - P[8 + j] * b) / cc;
      }
      res[2 * k] = t.u[k] - a / c;
      res[2 * k + 1] = t.v[k] - b / c;
    }
    Matrix A(3, 3), B(3, 1);
    for (int32_t m = 0; m < 3; m++) {
      for (int32_t n = 0; n < 3; n++) {
        FLOAT s = 0;
        for (int32_t i = 0; i < 2 * nf; i++) s += J[3 * i + m] * J[3 * i + n];
        A.val[m][n] = s;
      }
      FLOAT s = 0;
      for (int32_t i = 0; i < 2 * nf; i++) s += J[3 * i + m] * res[i];
      B.val[m][0] = s;
    }
    if (!B.solve(A)) return false;
    p.x += B.val[0][0]; p.y += B.val[1][0]; p.z += B.val[2][0];
    if (fabs(B.val[0][0]) < 1e-5 && fabs(B.val[1][0]) < 1e-5 && fabs(B.val[2][0]) < 1e-5) return true;
    if (iter > 20) return false;
  }
}

// -1 not visible (closer than 1 m to either end camera), 0 below the road, 1 road, 2 obstacle
int32_t Reconstruction::pointType(const visocu_recon_track& t, const Point3d& p) const {
  const Point3d x1c = affine12(job_frames[t.first].inv, p);
  const Point3d x2c = affine12(job_frames.back().inv, p);
  const Point3d x2r = affine12(job.cam_road, x2c);
  if (x1c.z <= 1 || x2c.z <= 1) return -1;
  if (x2r.y > 0.5) return 0;
  if (x2r.y > -1) return 1;
  return 2;
}

// distance to the camera position half way along the track
double Reconstruction::pointDistance(const visocu_recon_track& t, const Point3d& p) const {
  const unsigned first_ago = (unsigned)(job_frames.size() - 1 - (size_t)t.first);
  const unsigned mid_ago = (first_ago + 0u + 1u) / 2u;
  const double* c = job_frames[job_frames.size() - 1 - mid_ago].center;
  const double dx = c[0] - p.x, dy = c[1] - p.y, dz = c[2] - p.z;
  return sqrt(dx * dx + dy * dy + dz * dz);
}

// angle (degrees) between the viewing rays from the first and the last camera centre
double Reconstruction::rayAngle(const visocu_recon_track& t, const Point3d& p) const {
  const double* C1 = job_frames[t.first].center;
  const double* C2 = job_frames.back().center;
  FLOAT v1[3], v2[3];
  const FLOAT pt[3] = {p.x, p.y, p.z};
  for (int i = 0; i < 3; i++) { v1[i] = C1[i] - pt[i]; v2[i] = C2[i] - pt[i]; }
  const FLOAT n1 = sqrt(v1[0] * v1[0] + v1[1] * v1[1] + v1[2] * v1[2]);
  const FLOAT n2 = sqrt(v2[0] * v2[0] + v2[1] * v2[1] + v2[2] * v2[2]);
  if (n1 < 1e-10 || n2 < 1e-10) return 1000;
  FLOAT dot = 0;
  for (int i = 0; i < 3; i++) dot += (v1[i] / n1) * (v2[i] / n2);
  return acos(fabs(dot)) * 180.0 / M_PI;
}
