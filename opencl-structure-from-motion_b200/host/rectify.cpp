// Rectification maps and Bouguet's stereo rectification (see rectify.h).
#include "rectify.h"

#include <cmath>

namespace visob {
namespace {
bool finite_all(const double* v, int n) {
  for (int i = 0; i < n; i++) if (!std::isfinite(v[i])) return false;
  return true;
}
bool size_ok(int32_t v, int32_t lo) { return v >= lo && v <= 8191; }

// rotation matrix of the rotation vector w (Rodrigues), row-major
void rodrigues(const double w[3], double R[9]) {
  const double th = std::sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
  for (int i = 0; i < 9; i++) R[i] = i % 4 == 0 ? 1.0 : 0.0;
  if (th < 1e-300) return;
  const double k[3] = {w[0] / th, w[1] / th, w[2] / th}, c = std::cos(th), s = std::sin(th), v = 1.0 - c;
  R[0] = c + k[0] * k[0] * v;        R[1] = k[0] * k[1] * v - k[2] * s; R[2] = k[0] * k[2] * v + k[1] * s;
  R[3] = k[1] * k[0] * v + k[2] * s; R[4] = c + k[1] * k[1] * v;        R[5] = k[1] * k[2] * v - k[0] * s;
  R[6] = k[2] * k[0] * v - k[1] * s; R[7] = k[2] * k[1] * v + k[0] * s; R[8] = c + k[2] * k[2] * v;
}

// rotation vector of the rotation matrix R (angles below pi)
void rotation_vector(const double R[9], double w[3]) {
  const double c = std::fmax(-1.0, std::fmin(1.0, 0.5 * (R[0] + R[4] + R[8] - 1.0)));
  const double a[3] = {R[7] - R[5], R[2] - R[6], R[3] - R[1]};
  const double s = 0.5 * std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
  const double th = std::atan2(s, c);
  const double g = s > 1e-300 ? th / (2.0 * s) : 0.5;     // th / sin(th) -> 1 for small angles
  for (int i = 0; i < 3; i++) w[i] = g * a[i];
}

void mul(const double A[9], const double B[9], double C[9]) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
}  // namespace

bool rectifyCheck(const visocu_camera& c, int32_t src_w, int32_t src_h, int32_t out_w, int32_t out_h, const char** why) {
  const double head[9] = {c.fx, c.fy, c.cx, c.cy, c.k1, c.k2, c.p1, c.p2, c.k3}, tail[3] = {c.f, c.cu, c.cv};
  if (!finite_all(head, 9) || !finite_all(c.R, 9) || !finite_all(tail, 3)) { *why = "non-finite camera parameter"; return false; }
  if (!(c.fx > 0) || !(c.fy > 0) || !(c.f > 0)) { *why = "fx, fy and f must be positive"; return false; }
  if (!size_ok(src_w, 16) || !size_ok(src_h, 16)) { *why = "source size outside [16, 8191]"; return false; }
  if (!size_ok(out_w, 1) || !size_ok(out_h, 1)) { *why = "output size outside [1, 8191]"; return false; }
  return true;
}

bool rectifyMap(const visocu_camera& c, int32_t src_w, int32_t src_h, int32_t out_w, int32_t out_h, int32_t* map, const char** why) {
  if (!rectifyCheck(c, src_w, src_h, out_w, out_h, why)) return false;
  const double* R = c.R;
  const double xmax = 32.0 * (src_w - 1), ymax = 32.0 * (src_h - 1);
  for (int32_t v = 0; v < out_h; v++) {
    const double b = (v - c.cv) / c.f;
    for (int32_t u = 0; u < out_w; u++) {
      const double a = (u - c.cu) / c.f;
      // R^T (a, b, 1)
      const double X = R[0] * a + R[3] * b + R[6], Y = R[1] * a + R[4] * b + R[7], Z = R[2] * a + R[5] * b + R[8];
      if (!(Z > 0)) { *why = "an output pixel looks behind the raw camera (rotated ray with z <= 0)"; return false; }
      const double x = X / Z, y = Y / Z;
      const double r2 = x * x + y * y;
      const double radial = 1.0 + r2 * (c.k1 + r2 * (c.k2 + r2 * c.k3));
      const double xd = x * radial + 2.0 * c.p1 * x * y + c.p2 * (r2 + 2.0 * x * x);
      const double yd = y * radial + c.p1 * (r2 + 2.0 * y * y) + 2.0 * c.p2 * x * y;
      double sx = 32.0 * (c.fx * xd + c.cx), sy = 32.0 * (c.fy * yd + c.cy);
      if (!std::isfinite(sx) || !std::isfinite(sy)) { *why = "the distortion model overflows inside the output image"; return false; }
      // the bounds are whole numbers: clamping before rounding gives the clamp of the rounded value
      sx = std::fmin(std::fmax(sx, 0.0), xmax);
      sy = std::fmin(std::fmax(sy, 0.0), ymax);
      int32_t* e = map + 2 * ((size_t)v * out_w + u);
      e[0] = (int32_t)std::lrint(sx);
      e[1] = (int32_t)std::lrint(sy);
    }
  }
  return true;
}

void stereoRectify(const visocu_camera& cam0, const visocu_camera& cam1, const double R[9], const double T[3], int32_t out_w,
                   int32_t out_h, visocu_camera* rect0, visocu_camera* rect1, double* base) {
  // halves: Rh Rh = R; camera 0 turns by Rh, camera 1 by Rh^T, and then X1' = X0' + Rh^T T
  double w[3], Rh[9], RhT[9];
  rotation_vector(R, w);
  for (int i = 0; i < 3; i++) w[i] *= 0.5;
  rodrigues(w, Rh);
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) RhT[3 * i + j] = Rh[3 * j + i];
  double t[3];
  for (int i = 0; i < 3; i++) t[i] = RhT[3 * i] * T[0] + RhT[3 * i + 1] * T[1] + RhT[3 * i + 2] * T[2];
  const double nt = std::sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
  // camera 1's centre sits at -t: the rotation about a x e turns a = -t / |t| onto e = +x
  const double a[3] = {-t[0] / nt, -t[1] / nt, -t[2] / nt};
  const double ax[3] = {0.0, a[2], -a[1]};
  const double s = std::sqrt(ax[1] * ax[1] + ax[2] * ax[2]), ang = std::atan2(s, a[0]);
  double W[9], ww[3] = {0.0, 0.0, 0.0};
  if (s > 1e-300) for (int i = 0; i < 3; i++) ww[i] = ax[i] / s * ang;
  rodrigues(ww, W);
  *rect0 = cam0; *rect1 = cam1;
  mul(W, Rh, rect0->R);
  mul(W, RhT, rect1->R);
  const double f = std::fmin(cam0.fy, cam1.fy);
  double px = 0.0, py = 0.0;                         // mean of the two rotated optical axes, projected with f
  visocu_camera* const rect[2] = {rect0, rect1};
  for (int k = 0; k < 2; k++) { px += 0.5 * f * rect[k]->R[2] / rect[k]->R[8]; py += 0.5 * f * rect[k]->R[5] / rect[k]->R[8]; }
  for (int k = 0; k < 2; k++) { rect[k]->f = f; rect[k]->cu = 0.5 * (out_w - 1) - px; rect[k]->cv = 0.5 * (out_h - 1) - py; }
  *base = std::sqrt(T[0] * T[0] + T[1] * T[1] + T[2] * T[2]);
}
}  // namespace visob
