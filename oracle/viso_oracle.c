/* TEST INFRASTRUCTURE ONLY -- never linked into, imported by or executed from the product path.
 *
 * Plain-C restatement of the reference's hot path (libviso2 fork under /root/reference/viso): what the reference
 * computes, written as the simplest possible loops, each function citing the reference lines it follows.  It exists so
 * that (a) the semantics the CUDA path must reproduce are written down independently of the reference's SSE code and
 * (b) CPU-only tests can check golden fixtures where /root/reference is not available.
 *
 * Parity status: PINNED.  tests/test_oracle_vs_ref.py checks every function against the unmodified reference compiled
 * into oracle/_ref/libvisoref*.so (integer stages bit-exact, FP64 stages to the tolerance stated there), and
 * tests/test_oracle_golden.py checks it against the committed fixtures in tests/golden/ (generated from oracle/_ref by
 * tests/golden/make_golden.py).  Stereo matching, the motion-predicted quad search and sub-pixel refinement have no
 * counterpart in the reference shim: tests/test_oracle_vs_ref.py pins them against the reference results stored for
 * tests/test_gpu_host_layer.py instead (integer results bit-exact, sub-pixel coordinates to 1e-4).
 *
 * FP64 note: the SVD here is a one-sided Jacobi iteration, not the reference's Numerical-Recipes svdcmp
 * (matrix.cpp:586-814); singular values and the null vectors used by the 8-point algorithm agree to rounding, which is
 * what the RANSAC parity tolerance is built on.  Compile with -ffp-contract=off.
 */
#include "viso_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define MARGIN 6 /* matcher.cpp:56 */

/* ------------------------------------------------------------------------------------------------ images */
int vo_bpl(int w) { return w + 15 - (w - 1) % 16; } /* matcher.cpp:158-160 */

void vo_pad_image(const uint8_t* I, int w, int h, int bpl_in, uint8_t* out) { /* matcher.cpp:163-175, pad = 0 */
  int bpl = vo_bpl(w);
  memset(out, 0, (size_t)bpl * h);
  for (int v = 0; v < h; v++) memcpy(out + (size_t)v * bpl, I + (size_t)v * bpl_in, (size_t)w);
}

void vo_half_dims(const int32_t dims[3], int32_t dh[3]) { /* matcher.cpp:630-634 */
  dh[0] = dims[0] / 2;
  dh[1] = dims[1] / 2;
  dh[2] = dh[0] + 15 - (dh[0] - 1) % 16;
}

void vo_half_image(const uint8_t* I, const int32_t dims[3], uint8_t* out) { /* matcher.cpp:636-647 */
  int32_t dh[3];
  vo_half_dims(dims, dh);
  memset(out, 0, (size_t)dh[2] * dh[1]);
  for (int v = 0; v < dh[1]; v++)
    for (int u = 0; u < dh[0]; u++) {
      const uint8_t* p = I + (size_t)(2 * v) * dims[2] + 2 * u;
      out[(size_t)v * dh[2] + u] = (uint8_t)((p[0] + p[1] + p[dims[2]] + p[dims[2] + 1]) / 4);
    }
}

/* ------------------------------------------------------------------------------------------------ filters */
static int pix(const uint8_t* I, int w, int x, int y) { return I[(size_t)y * w + x]; }
static uint8_t sat_u8(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); } /* packus, simd.hh:245-248 */

/* filter.cpp:316-324 (column pass 183-233, row passes 71-127): `w` is the (16-byte multiple) row stride.
 * du = out_v: (1,4,6,4,1) down the rows, (1,2,0,-2,-1) along the row; dv = out_h: the transpose. >>7 is arithmetic.
 * Defined for 2 <= x <= w-3, 2 <= y <= h-3; everything else is set to 128 here (the reference leaves wrap-around
 * garbage in the border columns and 128 in the border rows). */
void vo_sobel5x5(const uint8_t* I, int w, int h, uint8_t* du, uint8_t* dv) {
  static const int a[5] = {1, 4, 6, 4, 1}, d[5] = {1, 2, 0, -2, -1};
  memset(du, 128, (size_t)w * h);
  memset(dv, 128, (size_t)w * h);
  for (int y = 2; y <= h - 3; y++)
    for (int x = 2; x <= w - 3; x++) {
      int su = 0, sv = 0;
      for (int j = 0; j < 5; j++)
        for (int i = 0; i < 5; i++) {
          int p = pix(I, w, x - 2 + i, y - 2 + j);
          su += a[j] * d[i] * p;
          sv += d[j] * a[i] * p;
        }
      du[(size_t)y * w + x] = sat_u8((su >> 7) + 128);
      dv[(size_t)y * w + x] = sat_u8((sv >> 7) + 128);
    }
}

void vo_sobel3x3(const uint8_t* I, int w, int h, uint8_t* du, uint8_t* dv) { /* filter.cpp:306-314, 128-182, 276-303 */
  static const int a[3] = {1, 2, 1}, d[3] = {1, 0, -1};
  memset(du, 128, (size_t)w * h);
  memset(dv, 128, (size_t)w * h);
  for (int y = 1; y <= h - 2; y++)
    for (int x = 1; x <= w - 2; x++) {
      int su = 0, sv = 0;
      for (int j = 0; j < 3; j++)
        for (int i = 0; i < 3; i++) {
          int p = pix(I, w, x - 1 + i, y - 1 + j);
          su += a[j] * d[i] * p;
          sv += d[j] * a[i] * p;
        }
      du[(size_t)y * w + x] = sat_u8((su >> 2) + 128);
      dv[(size_t)y * w + x] = sat_u8((sv >> 2) + 128);
    }
}

void vo_blob5x5(const uint8_t* I, int w, int h, int16_t* out) { /* filter.cpp:343-365: -box5 + 2*box3 + 7*centre */
  memset(out, 0, (size_t)w * h * sizeof(int16_t));
  for (int y = 3; y <= h - 3; y++)
    for (int x = 3; x <= w - 3; x++) {
      int f = 0;
      for (int j = -2; j <= 2; j++)
        for (int i = -2; i <= 2; i++) {
          int ring = abs(i) > abs(j) ? abs(i) : abs(j);
          int p = pix(I, w, x + i, y + j);
          f += ring == 2 ? -p : (ring == 1 ? p : 8 * p);
        }
      out[(size_t)y * w + x] = (int16_t)f;
    }
}

void vo_checkerboard5x5(const uint8_t* I, int w, int h, int16_t* out) { /* filter.cpp:331-336, 235-274: +1 top-left */
  static const int c[5] = {1, 1, 0, -1, -1};
  memset(out, 0, (size_t)w * h * sizeof(int16_t));
  for (int y = 2; y <= h - 3; y++)
    for (int x = 2; x <= w - 3; x++) {
      int f = 0;
      for (int j = 0; j < 5; j++)
        for (int i = 0; i < 5; i++) f += c[j] * c[i] * pix(I, w, x - 2 + i, y - 2 + j);
      out[(size_t)y * w + x] = (int16_t)f;
    }
}

/* ------------------------------------------------------------------------------------------------ NMS */
int vo_sparse_nms_n(int nms_n) { /* matcher.cpp:684-688 */
  int n = nms_n * 3;
  if (n > 10) n = nms_n > 10 ? nms_n : 10;
  return n;
}

/* matcher.cpp:330-431.  out4 = (u, v, val, class) per maximum in the reference's push_back order. */
int vo_nms(const int16_t* f1, const int16_t* f2, const int32_t dims[3], int n, int tau, int32_t* out4, int cap) {
  const int width = dims[0], height = dims[1], bpl = dims[2];
  int count = 0;
  for (int i = n + MARGIN; i < width - n - MARGIN; i += n + 1)
    for (int j = n + MARGIN; j < height - n - MARGIN; j += n + 1) {
      const int16_t* planes[2] = {f1, f2};
      for (int pl = 0; pl < 2; pl++) {
        const int16_t* f = planes[pl];
        int mini = i, minj = j, maxi = i, maxj = j;
        int minv = f[(size_t)j * bpl + i], maxv = minv;
        for (int i2 = i; i2 <= i + n; i2++)
          for (int j2 = j; j2 <= j + n; j2++) {
            int v = f[(size_t)j2 * bpl + i2];
            if (v < minv) { mini = i2; minj = j2; minv = v; }
            else if (v > maxv) { maxi = i2; maxj = j2; maxv = v; }
          }
        for (int ext = 0; ext < 2; ext++) { /* 0 = minimum (class 2*pl), 1 = maximum (class 2*pl+1) */
          const int ei = ext ? maxi : mini, ej = ext ? maxj : minj, ev = ext ? maxv : minv;
          int failed = 0;
          const int iu = ei + n < width - 1 - MARGIN ? ei + n : width - 1 - MARGIN;
          const int ju = ej + n < height - 1 - MARGIN ? ej + n : height - 1 - MARGIN;
          for (int i2 = ei - n; i2 <= iu && !failed; i2++)
            for (int j2 = ej - n; j2 <= ju; j2++) {
              int v = f[(size_t)j2 * bpl + i2];
              int better = ext ? v > ev : v < ev;
              if (better && (i2 < i || i2 > i + n || j2 < j || j2 > j + n)) { failed = 1; break; }
            }
          if (failed) continue;
          if (ext ? ev >= tau : ev <= -tau) {
            if (count < cap) {
              out4[4 * count + 0] = ei; out4[4 * count + 1] = ej; out4[4 * count + 2] = ev; out4[4 * count + 3] = 2 * pl + ext;
            }
            count++;
          }
        }
      }
    }
  return count;
}

/* ------------------------------------------------------------------------------------------------ descriptors */
void vo_descriptor(const uint8_t* du, const uint8_t* dv, int bpl, int u, int v, uint8_t* out32) { /* matcher.cpp:433-477 */
  static const int ox[16] = {-3, -3, -1, -1, 3, 3, 1, 1, -1, -1, 1, 1, -5, -5, 5, 5};
  static const int oy[16] = {-1, 1, -1, 1, -1, 1, -1, 1, -5, 5, -5, 5, -3, 3, -3, 3};
  for (int k = 0; k < 16; k++) {
    size_t a = (size_t)(v + oy[k]) * bpl + (u + ox[k]);
    out32[2 * k] = du[a];
    out32[2 * k + 1] = dv[a];
  }
}

void vo_small_descriptor(const uint8_t* du, const uint8_t* dv, int bpl, int u, int v, uint8_t* out16) { /* matcher.cpp:479-506 */
  static const int pl[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1};
  static const int dx[16] = {0, -2, 0, 2, -1, 0, 0, 1, -2, 0, 2, 0, 0, -1, 1, 0};
  static const int dy[16] = {-2, -1, -1, -1, 0, 0, 0, 0, 1, 1, 1, 2, -1, 0, 0, 1};
  for (int k = 0; k < 16; k++) out16[k] = (pl[k] ? dv : du)[(size_t)(v + dy[k]) * bpl + (u + dx[k])];
}

int vo_sad(const uint8_t* a, const uint8_t* b, int nbytes) { /* simd.hh:385-394, 414-424 */
  int s = 0;
  for (int k = 0; k < nbytes; k++) s += abs((int)a[k] - (int)b[k]);
  return s;
}

/* matcher.cpp:649-732 */
int vo_compute_features(const uint8_t* Ipad, const int32_t dims[3], const vo_params* p, uint8_t* du, uint8_t* dv,
                        uint8_t* du_full, uint8_t* dv_full, int32_t* rec1, int cap1, int32_t* n1, int32_t* rec2, int cap2,
                        int32_t* n2) {
  int32_t dm[3] = {dims[0], dims[1], dims[2]};
  const uint8_t* Im = Ipad;
  uint8_t* half = NULL;
  int s = 1;
  if (p->half_resolution) {
    vo_half_dims(dims, dm);
    half = (uint8_t*)malloc((size_t)dm[2] * dm[1] + 64);
    vo_half_image(Ipad, dims, half);
    Im = half;
    s = 2;
    vo_sobel5x5(Ipad, dims[2], dims[1], du_full, dv_full);
  }
  const size_t npx = (size_t)dm[2] * dm[1];
  int16_t* f1 = (int16_t*)malloc(npx * sizeof(int16_t));
  int16_t* f2 = (int16_t*)malloc(npx * sizeof(int16_t));
  vo_sobel5x5(Im, dm[2], dm[1], du, dv);
  vo_blob5x5(Im, dm[2], dm[1], f1);
  vo_checkerboard5x5(Im, dm[2], dm[1], f2);
  int32_t* recs[2] = {rec1, rec2};
  int caps[2] = {cap1, cap2};
  int32_t* counts[2] = {n1, n2};
  int ns[2] = {vo_sparse_nms_n(p->nms_n), p->nms_n};
  for (int pass = p->multi_stage ? 0 : 1; pass < 2; pass++) {
    int cap = caps[pass];
    int32_t* mx = (int32_t*)malloc((size_t)(cap > 0 ? cap : 1) * 4 * sizeof(int32_t));
    int n = vo_nms(f1, f2, dm, ns[pass], p->nms_tau, mx, cap);
    if (n > cap) { free(mx); free(f1); free(f2); free(half); return -1; }
    for (int k = 0; k < n; k++) { /* matcher.cpp:707-731: {u*s, v*s, 0, class, 32 descriptor bytes} */
      int32_t* r = recs[pass] + (size_t)12 * k;
      r[0] = mx[4 * k] * s; r[1] = mx[4 * k + 1] * s; r[2] = 0; r[3] = mx[4 * k + 3];
      vo_descriptor(du, dv, dm[2], mx[4 * k], mx[4 * k + 1], (uint8_t*)(r + 4));
    }
    *counts[pass] = n;
    free(mx);
  }
  if (!p->multi_stage) *n1 = 0;
  free(f1); free(f2); free(half);
  return 0;
}

/* ------------------------------------------------------------------------------------------------ matching */
typedef struct { int32_t* start; int32_t* idx; } binlist; /* createIndexVector, matcher.cpp:870-890: lists in feature order */

static int bin_of(const vo_params* p, int u, int v, int c, int ub, int vb) {
  int ubin = (int)floorf((float)u / (float)p->match_binsize), vbin = (int)floorf((float)v / (float)p->match_binsize);
  if (ubin > ub - 1) ubin = ub - 1;
  if (vbin > vb - 1) vbin = vb - 1;
  return (c * vb + vbin) * ub + ubin;
}

static binlist make_bins(const int32_t* m, int n, const vo_params* p, int ub, int vb) {
  const int nb = 4 * ub * vb;
  binlist b;
  b.start = (int32_t*)calloc((size_t)nb + 1, sizeof(int32_t));
  b.idx = (int32_t*)malloc((size_t)(n > 0 ? n : 1) * sizeof(int32_t));
  for (int i = 0; i < n; i++) b.start[bin_of(p, m[12 * i], m[12 * i + 1], m[12 * i + 3], ub, vb) + 1]++;
  for (int k = 0; k < nb; k++) b.start[k + 1] += b.start[k];
  int32_t* cur = (int32_t*)malloc((size_t)nb * sizeof(int32_t));
  memcpy(cur, b.start, (size_t)nb * sizeof(int32_t));
  for (int i = 0; i < n; i++) b.idx[cur[bin_of(p, m[12 * i], m[12 * i + 1], m[12 * i + 3], ub, vb)]++] = i;
  free(cur);
  return b;
}

static int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

/* Work counters of one vo_matching call: entries of the bins a hop scans, and candidates that pass its window test
 * (what visocu_match_stats reports for the device). */
typedef struct { int64_t scanned, candidates; } counters;

/* matcher.cpp:892-963.  (up, vp): predicted position of the match (matcher.cpp:948-953), or u_ = v_ = -1 for none:
 * then every candidate in the window costs SAD + 4 * distance to it, in double precision. */
static int find_match(const int32_t* m1, int i1, const int32_t* m2, const binlist* k2, int ub, int vb, int stat_bin, int stage,
                      int flow, int use_prior, const vo_range* ranges, const vo_params* p, double up, double vp, counters* cnt) {
  int min_ind = 0;
  double min_cost = 10000000;
  const int u1 = m1[12 * i1], v1 = m1[12 * i1 + 1], c = m1[12 * i1 + 3];
  float u_min, u_max, v_min, v_max;
  if (use_prior) {
    u_min = u1 + ranges[stat_bin].u_min[stage]; u_max = u1 + ranges[stat_bin].u_max[stage];
    v_min = v1 + ranges[stat_bin].v_min[stage]; v_max = v1 + ranges[stat_bin].v_max[stage];
  } else {
    u_min = (float)(u1 - p->match_radius); u_max = (float)(u1 + p->match_radius);
    v_min = (float)(v1 - p->match_radius); v_max = (float)(v1 + p->match_radius);
  }
  if (!flow) { v_min = (float)(v1 - p->match_disp_tolerance); v_max = (float)(v1 + p->match_disp_tolerance); }
  const float bs = (float)p->match_binsize;
  const int ub0 = clampi((int)floorf(u_min / bs), 0, ub - 1), ub1 = clampi((int)floorf(u_max / bs), 0, ub - 1);
  const int vb0 = clampi((int)floorf(v_min / bs), 0, vb - 1), vb1 = clampi((int)floorf(v_max / bs), 0, vb - 1);
  const int predicted = up >= 0 && vp >= 0;
  for (int ubin = ub0; ubin <= ub1; ubin++)
    for (int vbin = vb0; vbin <= vb1; vbin++) {
      const int k = (c * vb + vbin) * ub + ubin;
      cnt->scanned += k2->start[k + 1] - k2->start[k];
      for (int e = k2->start[k]; e < k2->start[k + 1]; e++) {
        const int i2 = k2->idx[e];
        const int u2 = m2[12 * i2], v2 = m2[12 * i2 + 1];
        if (u2 >= u_min && u2 <= u_max && v2 >= v_min && v2 <= v_max) {
          cnt->candidates++;
          double cost = (double)vo_sad((const uint8_t*)(m1 + 12 * i1 + 4), (const uint8_t*)(m2 + 12 * i2 + 4), 32);
          if (predicted) {
            const double du = (double)u2 - up, dv = (double)v2 - vp;
            const double dist = sqrt(du * du + dv * dv);
            cost = cost + 4 * dist;
          }
          if (cost < min_cost) { min_ind = i2; min_cost = cost; }
        }
      }
    }
  return min_ind;
}

static int stat_bin_of(const vo_params* p, int u, int v, int ub, int vb) {
  const float bs = (float)p->match_binsize;
  int ubin = (int)floorf((float)u / bs), vbin = (int)floorf((float)v / bs);
  if (ubin > ub - 1) ubin = ub - 1;
  if (vbin > vb - 1) vbin = vb - 1;
  return vbin * ub + ubin;
}

/* matcher.cpp:965-1205: methods 0 (flow), 1 (stereo) and 2 (quad, with the motion-predicted search of
 * matcher.cpp:1112-1138 if tr_delta, rows 0..2 of Tr_delta, is given).  Nothing is matched if a set the method needs is
 * empty (matchFeatures returns early, matcher.cpp:190-212).  counts2 (optional): scanned entries, window candidates. */
int vo_matching(int method, const int32_t* m1p, int n1p, const int32_t* m2p, int n2p, const int32_t* m1c, int n1c,
                const int32_t* m2c, int n2c, const int32_t dims_c[3], const vo_params* p, int use_prior,
                const vo_range* ranges, const double* tr_delta, vo_match* out, int cap, int64_t* counts2) {
  const int ub = (int)ceilf((float)dims_c[0] / (float)p->match_binsize), vb = (int)ceilf((float)dims_c[1] / (float)p->match_binsize);
  int count = 0;
  counters cnt = {0, 0};
  if (counts2) { counts2[0] = 0; counts2[1] = 0; }
  if (method < 0 || method > 2) return -1;
  if (((method != 1) && n1p == 0) || (method == 2 && n2p == 0) || n1c == 0 || (method != 0 && n2c == 0)) return 0;
  if (method == 0 || method == 1) {
    /* flow: current left -> previous left -> back; stereo: current left -> current right -> back (matcher.cpp:1045-1084) */
    const int32_t* mo = method == 0 ? m1p : m2c;
    const int no = method == 0 ? n1p : n2c;
    binlist ko = make_bins(mo, no, p, ub, vb), k1c = make_bins(m1c, n1c, p, ub, vb);
    uint8_t* M = (uint8_t*)calloc((size_t)dims_c[0] * dims_c[1], 1);
    for (int i1c = 0; i1c < n1c; i1c++) {
      const int u1c = m1c[12 * i1c], v1c = m1c[12 * i1c + 1];
      const int stat = stat_bin_of(p, u1c, v1c, ub, vb);
      const int flow = method == 0;
      const int io = find_match(m1c, i1c, mo, &ko, ub, vb, stat, 0, flow, use_prior, ranges, p, -1, -1, &cnt);
      const int back = find_match(mo, io, m1c, &k1c, ub, vb, stat, 1, flow, use_prior, ranges, p, -1, -1, &cnt);
      if (back != i1c) continue;
      if (method == 1 && !(u1c >= mo[12 * io])) continue;       /* positive disparity, tested before the pixel rule */
      uint8_t* taken = M + (size_t)v1c * dims_c[0] + u1c;
      if (*taken) continue;
      *taken = 1;
      if (count < cap) {
        const vo_match f = {(float)mo[12 * io], (float)mo[12 * io + 1], io, -1, -1, -1, (float)u1c, (float)v1c, i1c, -1, -1, -1};
        const vo_match s = {-1, -1, -1, -1, -1, -1, (float)u1c, (float)v1c, i1c, (float)mo[12 * io], (float)mo[12 * io + 1], io};
        out[count] = method == 0 ? f : s;
      }
      count++;
    }
    free(M); free(ko.start); free(ko.idx); free(k1c.start); free(k1c.idx);
  } else {
    binlist k1p = make_bins(m1p, n1p, p, ub, vb), k2p = make_bins(m2p, n2p, p, ub, vb);
    binlist k1c = make_bins(m1c, n1c, p, ub, vb), k2c = make_bins(m2c, n2c, p, ub, vb);
    for (int i1p = 0; i1p < n1p; i1p++) {
      const int u1p = m1p[12 * i1p], v1p = m1p[12 * i1p + 1];
      const int stat = stat_bin_of(p, u1p, v1p, ub, vb);
      const int i2p = find_match(m1p, i1p, m2p, &k2p, ub, vb, stat, 0, 0, use_prior, ranges, p, -1, -1, &cnt);
      double up = -1, vp = -1, u1pd = -1, v1pd = -1;
      if (tr_delta) {
        /* the previous stereo match triangulated, moved by Tr_delta, projected into the current right image */
        const double* t = tr_delta;
        u1pd = u1p; v1pd = v1p;
        double d = u1pd - (double)m2p[12 * i2p];
        if (d < 1) d = 1;
        const double x1p = (u1pd - p->cu) * p->base / d, y1p = (v1pd - p->cv) * p->base / d, z1p = p->f * p->base / d;
        const double x2c = t[0] * x1p + t[1] * y1p + t[2] * z1p + t[3] - p->base;
        const double y2c = t[4] * x1p + t[5] * y1p + t[6] * z1p + t[7];
        const double z2c = t[8] * x1p + t[9] * y1p + t[10] * z1p + t[11];
        up = p->f * x2c / z2c + p->cu;
        vp = p->f * y2c / z2c + p->cv;
      }
      const int i2c = find_match(m2p, i2p, m2c, &k2c, ub, vb, stat, 1, 1, use_prior, ranges, p, up, vp, &cnt);
      const int i1c = find_match(m2c, i2c, m1c, &k1c, ub, vb, stat, 2, 0, use_prior, ranges, p, -1, -1, &cnt);
      const int back = find_match(m1c, i1c, m1p, &k1p, ub, vb, stat, 3, 1, use_prior, ranges, p, u1pd, v1pd, &cnt);
      if (back != i1p) continue;
      const int u2p = m2p[12 * i2p], v2p = m2p[12 * i2p + 1], u2c = m2c[12 * i2c], v2c = m2c[12 * i2c + 1];
      const int u1c = m1c[12 * i1c], v1c = m1c[12 * i1c + 1];
      if (!(u1p >= u2p && u1c >= u2c)) continue;
      if (count < cap) {
        vo_match m = {(float)u1p, (float)v1p, i1p, (float)u2p, (float)v2p, i2p, (float)u1c, (float)v1c, i1c, (float)u2c, (float)v2c, i2c};
        out[count] = m;
      }
      count++;
    }
    free(k1p.start); free(k1p.idx); free(k2p.start); free(k2p.idx);
    free(k1c.start); free(k1c.idx); free(k2c.start); free(k2c.idx);
  }
  if (counts2) { counts2[0] = cnt.scanned; counts2[1] = cnt.candidates; }
  return count;
}

/* matcher.cpp:734-868.  Only the first 2 (flow, stereo) or 4 (quad) stage entries of every range are defined. */
int vo_prior_statistics(const vo_match* pm, int n, int method, const int32_t dims_c[3], const vo_params* p, vo_range* ranges) {
  const float bs = (float)p->match_binsize;
  const int ub = (int)ceilf((float)dims_c[0] / bs), vb = (int)ceilf((float)dims_c[1] / bs);
  const int nbin = ub * vb, stages = method == 2 ? 4 : 2;
  float* lo = (float*)malloc((size_t)nbin * 8 * sizeof(float));
  float* hi = (float*)malloc((size_t)nbin * 8 * sizeof(float));
  uint8_t* seen = (uint8_t*)calloc((size_t)nbin, 1);
  for (int k = 0; k < nbin * 8; k++) { lo[k] = 1000000.f; hi[k] = -1000000.f; }
  for (int k = 0; k < n; k++) {
    const vo_match* m = pm + k;
    float d[8] = {0, 0, 0, 0, 0, 0, 0, 0}, ru, rv;
    if (method == 0) {
      d[0] = m->u1p - m->u1c; d[1] = m->v1p - m->v1c; d[2] = m->u1c - m->u1p; d[3] = m->v1c - m->v1p;
      ru = m->u1c; rv = m->v1c;
    } else if (method == 1) {
      d[0] = m->u2c - m->u1c; d[2] = m->u1c - m->u2c;
      ru = m->u1c; rv = m->v1c;
    } else {
      d[0] = m->u2p - m->u1p; d[2] = m->u2c - m->u2p; d[3] = m->v2c - m->v2p; d[4] = m->u1c - m->u2c;
      d[6] = m->u1p - m->u1c; d[7] = m->v1p - m->v1c;
      ru = m->u1p; rv = m->v1p;
    }
    const int cu = (int)floorf(ru / bs), cv = (int)floorf(rv / bs);
    for (int v = clampi(cv - 1, 0, vb - 1); v <= clampi(cv + 1, 0, vb - 1); v++)
      for (int u = clampi(cu - 1, 0, ub - 1); u <= clampi(cu + 1, 0, ub - 1); u++) {
        const int b = v * ub + u;
        seen[b] = 1;
        for (int i = 0; i < stages * 2; i++) {
          if (d[i] < lo[b * 8 + i]) lo[b * 8 + i] = d[i];
          if (d[i] > hi[b * 8 + i]) hi[b * 8 + i] = d[i];
        }
      }
  }
  for (int b = 0; b < nbin; b++) {
    memset(&ranges[b], 0, sizeof(vo_range));
    for (int i = 0; i < stages; i++)
      for (int a = 0; a < 2; a++) {
        float mn = seen[b] ? lo[b * 8 + i * 2 + a] : (float)-p->match_radius;
        float mx = seen[b] ? hi[b * 8 + i * 2 + a] : (float)p->match_radius;
        const float span = mx - mn;
        if (span < 20) { mn -= ceilf((20 - span) / 2); mx += ceilf((20 - span) / 2); }
        if (a == 0) { ranges[b].u_min[i] = mn; ranges[b].u_max[i] = mx; }
        else        { ranges[b].v_min[i] = mn; ranges[b].v_max[i] = mx; }
      }
  }
  free(lo); free(hi); free(seen);
  return nbin;
}

/* relocateMinimum, matcher.cpp:1456-1496 */
static void relocate(const uint8_t* du1, const uint8_t* dv1, const uint8_t* du2, const uint8_t* dv2, const int32_t d1[3],
                     const int32_t d2[3], float u1, float v1, float* u2, float* v2) {
  if (*u2 - 2 < MARGIN || *u2 + 2 > d2[0] - 1 - MARGIN || *v2 - 2 < MARGIN || *v2 + 2 > d2[1] - 1 - MARGIN) return;
  uint8_t ref[16], cand[16];
  vo_small_descriptor(du1, dv1, d1[2], (int)u1, (int)v1, ref);
  int best = 0, best_cost = 0;
  for (int k = 0; k < 25; k++) {
    vo_small_descriptor(du2, dv2, d2[2], (int)*u2 + k % 5 - 2, (int)*v2 + k / 5 - 2, cand);
    const int cost = vo_sad(ref, cand, 16);
    if (k == 0 || cost < best_cost) { best = k; best_cost = cost; }
  }
  *u2 += (float)(best % 5) - 2.0f;
  *v2 += (float)(best / 5) - 2.0f;
}

/* Matcher::refinement with refinement == 1, matcher.cpp:1498-1585.  The reference descriptor is always the one at
 * (u1c, v1c); the relocated points are (u1p, v1p) in the previous left image (flow, quad), (u2c, v2c) in the current
 * right image (stereo, quad) and (u2p, v2p) in the previous right image (quad). */
void vo_refine_pixel(vo_match* pm, int n, int method, const int32_t dims_p[3], const int32_t dims_c[3], const uint8_t* du1p,
                     const uint8_t* dv1p, const uint8_t* du2p, const uint8_t* dv2p, const uint8_t* du1c, const uint8_t* dv1c,
                     const uint8_t* du2c, const uint8_t* dv2c) {
  for (int k = 0; k < n; k++) {
    vo_match* m = pm + k;
    if (method == 0 || method == 2) relocate(du1c, dv1c, du1p, dv1p, dims_c, dims_p, m->u1c, m->v1c, &m->u1p, &m->v1p);
    if (method == 1 || method == 2) relocate(du1c, dv1c, du2c, dv2c, dims_c, dims_c, m->u1c, m->v1c, &m->u2c, &m->v2c);
    if (method == 2) relocate(du1c, dv1c, du2p, dv2p, dims_c, dims_p, m->u1c, m->v1c, &m->u2p, &m->v2p);
  }
}

/* Solves the 6x6 system M x = r in place (Gauss-Jordan elimination with partial pivoting, double precision).
 * Returns 0 if a pivot vanishes. */
static int solve6(double M[6][6], double r[6]) {
  for (int c = 0; c < 6; c++) {
    int piv = c;
    for (int i = c + 1; i < 6; i++) if (fabs(M[i][c]) > fabs(M[piv][c])) piv = i;
    if (fabs(M[piv][c]) < 1e-20) return 0;
    for (int k = 0; k < 6; k++) { const double t = M[c][k]; M[c][k] = M[piv][k]; M[piv][k] = t; }
    { const double t = r[c]; r[c] = r[piv]; r[piv] = t; }
    const double d = M[c][c];
    for (int k = 0; k < 6; k++) M[c][k] /= d;
    r[c] /= d;
    for (int i = 0; i < 6; i++) {
      if (i == c) continue;
      const double f = M[i][c];
      for (int k = 0; k < 6; k++) M[i][k] -= f * M[c][k];
      r[i] -= f * r[c];
    }
  }
  return 1;
}

static double min2(double a, double b) { return a < b ? a : b; }

/* parabolicFitting, matcher.cpp:1379-1454: 16-byte descriptor costs on the 7x7 positions around (u2, v2), first
 * minimum, a minimum on the border drops the match, least-squares paraboloid c = b0 j^2 + b1 i^2 + b2 i j + b3 j + b4 i
 * + b5 through the 3x3 costs around it (normal equations solved per match, as the reference's Matrix::solve does),
 * then the float offsets and their rejections.  *margin receives the smallest distance of a float decision of this fit
 * to its threshold (1 - |ddu|, 1 - |ddv|, |divisor|, |b2|; +inf if no float decision was taken).  Returns 0 if the
 * match is dropped. */
static int parabolic(const uint8_t* du1, const uint8_t* dv1, const uint8_t* du2, const uint8_t* dv2, const int32_t d1[3],
                     const int32_t d2[3], float u1, float v1, float* u2, float* v2, double* margin) {
  *margin = INFINITY;
  if (*u2 - 3 < MARGIN || *u2 + 3 > d2[0] - 1 - MARGIN || *v2 - 3 < MARGIN || *v2 + 3 > d2[1] - 1 - MARGIN) return 0;
  uint8_t ref[16], cand[16];
  vo_small_descriptor(du1, dv1, d1[2], (int)u1, (int)v1, ref);
  int cost[49];
  for (int dv = 0; dv < 7; dv++)
    for (int du = 0; du < 7; du++) {
      vo_small_descriptor(du2, dv2, d2[2], (int)*u2 + du - 3, (int)*v2 + dv - 3, cand);
      cost[dv * 7 + du] = vo_sad(ref, cand, 16);
    }
  int min_ind = 0;
  for (int i = 1; i < 49; i++) if (cost[i] < cost[min_ind]) min_ind = i;
  const int du = min_ind % 7, dv = min_ind / 7;
  if (du == 0 || du == 6 || dv == 0 || dv == 6) return 0;
  double AtA[6][6] = {{0}}, b[6] = {0, 0, 0, 0, 0, 0};
  for (int i = -1; i <= 1; i++)
    for (int j = -1; j <= 1; j++) {
      const double row[6] = {j * j, i * i, i * j, j, i, 1};
      const double c = cost[(dv + i) * 7 + (du + j)];
      for (int r = 0; r < 6; r++) {
        for (int q = 0; q < 6; q++) AtA[r][q] += row[r] * row[q];
        b[r] += row[r] * c;
      }
    }
  if (!solve6(AtA, b)) return 0;
  const float divisor = (float)(b[2] * b[2] - 4.0 * b[0] * b[1]);
  *margin = min2(fabs(divisor), fabs(b[2]));
  if (fabsf(divisor) < 1e-8 || fabs(b[2]) < 1e-8) return 0;
  const float ddv = (float)((2.0 * b[0] * b[4] - b[2] * b[3]) / divisor);
  const float ddu = (float)(-(b[4] + 2.0 * b[1] * ddv) / b[2]);
  *margin = min2(*margin, min2(fabs(1.0 - fabsf(ddu)), fabs(1.0 - fabsf(ddv))));
  if (fabsf(ddu) >= 1.0f || fabsf(ddv) >= 1.0f) return 0;
  *u2 += (float)du - 3.0 + ddu;
  *v2 += (float)dv - 3.0 + ddv;
  return 1;
}

/* Matcher::refinement with refinement == 2, matcher.cpp:1498-1585: the same hops as vo_refine_pixel with
 * parabolicFitting; the first fit that fails drops the match (keep[k] = 0, the list itself is not compacted).
 * margin[k] (optional): the smallest decision margin over the fits run for match k. */
void vo_refine_subpixel(vo_match* pm, int n, int method, const int32_t dims_p[3], const int32_t dims_c[3], const uint8_t* du1p,
                        const uint8_t* dv1p, const uint8_t* du2p, const uint8_t* dv2p, const uint8_t* du1c, const uint8_t* dv1c,
                        const uint8_t* du2c, const uint8_t* dv2c, uint8_t* keep, double* margin) {
  for (int k = 0; k < n; k++) {
    vo_match* m = pm + k;
    double mg = INFINITY, g;
    int ok = 1;
    if (method == 0 || method == 2) {
      ok = parabolic(du1c, dv1c, du1p, dv1p, dims_c, dims_p, m->u1c, m->v1c, &m->u1p, &m->v1p, &g);
      mg = min2(mg, g);
    }
    if (ok && (method == 1 || method == 2)) {
      ok = parabolic(du1c, dv1c, du2c, dv2c, dims_c, dims_c, m->u1c, m->v1c, &m->u2c, &m->v2c, &g);
      mg = min2(mg, g);
    }
    if (ok && method == 2) {
      ok = parabolic(du1c, dv1c, du2p, dv2p, dims_c, dims_p, m->u1c, m->v1c, &m->u2p, &m->v2p, &g);
      mg = min2(mg, g);
    }
    keep[k] = (uint8_t)ok;
    if (margin) margin[k] = mg;
  }
}

/* ------------------------------------------------------------------------------------------------ RANSAC (FP64) */
/* a: m x n row-major, overwritten with U*diag(w) columns; w: n singular values; v: n x n row-major.
 * Unsorted, unsigned (callers pick the smallest singular value themselves). */
void vo_svd(double* a, int m, int n, double* w, double* v) {
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) v[i * n + j] = i == j;
  double total = 0;
  for (int k = 0; k < m * n; k++) total += a[k] * a[k];
  const double tiny = 1e-28 * total; /* numerically null columns (the 8x9 system always has one) are left alone */
  for (int sweep = 0; sweep < 60; sweep++) {
    int rotated = 0;
    for (int p = 0; p < n - 1; p++)
      for (int q = p + 1; q < n; q++) {
        double alpha = 0, beta = 0, gamma = 0;
        for (int i = 0; i < m; i++) {
          alpha += a[i * n + p] * a[i * n + p]; beta += a[i * n + q] * a[i * n + q]; gamma += a[i * n + p] * a[i * n + q];
        }
        if (alpha <= tiny || beta <= tiny || fabs(gamma) <= 1e-15 * sqrt(alpha * beta)) continue;
        rotated = 1;
        const double zeta = (beta - alpha) / (2.0 * gamma);
        const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
        for (int i = 0; i < m; i++) {
          const double x = a[i * n + p], y = a[i * n + q];
          a[i * n + p] = c * x - s * y; a[i * n + q] = s * x + c * y;
        }
        for (int i = 0; i < n; i++) {
          const double x = v[i * n + p], y = v[i * n + q];
          v[i * n + p] = c * x - s * y; v[i * n + q] = s * x + c * y;
        }
      }
    if (!rotated) break;
  }
  for (int j = 0; j < n; j++) {
    double s = 0;
    for (int i = 0; i < m; i++) s += a[i * n + j] * a[i * n + j];
    w[j] = sqrt(s);
  }
}

int vo_normalize(vo_match* pm, int n, double* Tp9, double* Tc9) { /* viso_mono.cpp:217-263 (float write-backs kept) */
  double cpu = 0, cpv = 0, ccu = 0, ccv = 0;
  for (int k = 0; k < n; k++) { cpu += pm[k].u1p; cpv += pm[k].v1p; ccu += pm[k].u1c; ccv += pm[k].v1c; }
  cpu /= (double)n; cpv /= (double)n; ccu /= (double)n; ccv /= (double)n;
  for (int k = 0; k < n; k++) {
    pm[k].u1p = (float)(pm[k].u1p - cpu); pm[k].v1p = (float)(pm[k].v1p - cpv);
    pm[k].u1c = (float)(pm[k].u1c - ccu); pm[k].v1c = (float)(pm[k].v1c - ccv);
  }
  double sp = 0, sc = 0;
  for (int k = 0; k < n; k++) {
    sp += sqrtf(pm[k].u1p * pm[k].u1p + pm[k].v1p * pm[k].v1p);
    sc += sqrtf(pm[k].u1c * pm[k].u1c + pm[k].v1c * pm[k].v1c);
  }
  if (fabs(sp) < 1e-10 || fabs(sc) < 1e-10) return 0;
  sp = sqrt(2.0) * (double)n / sp;
  sc = sqrt(2.0) * (double)n / sc;
  for (int k = 0; k < n; k++) {
    pm[k].u1p = (float)(pm[k].u1p * sp); pm[k].v1p = (float)(pm[k].v1p * sp);
    pm[k].u1c = (float)(pm[k].u1c * sc); pm[k].v1c = (float)(pm[k].v1c * sc);
  }
  const double tp[9] = {sp, 0, -sp * cpu, 0, sp, -sp * cpv, 0, 0, 1}, tc[9] = {sc, 0, -sc * ccu, 0, sc, -sc * ccv, 0, 0, 1};
  memcpy(Tp9, tp, sizeof tp);
  memcpy(Tc9, tc, sizeof tc);
  return 1;
}

/* viso_mono.cpp:265-296: constraint rows from float products, null vector, rank-2 projection */
void vo_fundamental(const vo_match* pm, const int32_t* active, int nactive, double* F9) {
  double* A = (double*)malloc((size_t)nactive * 9 * sizeof(double));
  for (int i = 0; i < nactive; i++) {
    const vo_match* m = pm + active[i];
    double* r = A + 9 * i;
    r[0] = (double)(m->u1c * m->u1p); r[1] = (double)(m->u1c * m->v1p); r[2] = m->u1c;
    r[3] = (double)(m->v1c * m->u1p); r[4] = (double)(m->v1c * m->v1p); r[5] = m->v1c;
    r[6] = m->u1p; r[7] = m->v1p; r[8] = 1;
  }
  double w[9], V[81];
  vo_svd(A, nactive, 9, w, V);
  int js = 0;
  for (int j = 1; j < 9; j++) if (w[j] < w[js]) js = j;
  double F[9], w3[3], V3[9];
  for (int k = 0; k < 9; k++) F[k] = V[k * 9 + js];
  double G[9];
  memcpy(G, F, sizeof G);
  vo_svd(G, 3, 3, w3, V3);        /* G now holds sigma_j * u_j in column j */
  js = 0;
  for (int j = 1; j < 3; j++) if (w3[j] < w3[js]) js = j;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) F9[3 * r + c] = F[3 * r + c] - G[3 * r + js] * V3[3 * c + js];
  free(A);
}

int vo_get_inlier(const vo_match* pm, int n, const double* f, double thresh, int32_t* out) { /* viso_mono.cpp:298-345 */
  int count = 0;
  for (int i = 0; i < n; i++) {
    const double u1 = pm[i].u1p, v1 = pm[i].v1p, u2 = pm[i].u1c, v2 = pm[i].v1c;
    const double Fx1u = f[0] * u1 + f[1] * v1 + f[2], Fx1v = f[3] * u1 + f[4] * v1 + f[5], Fx1w = f[6] * u1 + f[7] * v1 + f[8];
    const double Ftx2u = f[0] * u2 + f[3] * v2 + f[6], Ftx2v = f[1] * u2 + f[4] * v2 + f[7];
    const double x2tFx1 = u2 * Fx1u + v2 * Fx1v + Fx1w;
    const double d = x2tFx1 * x2tFx1 / (Fx1u * Fx1u + Fx1v * Fx1v + Ftx2u * Ftx2u + Ftx2v * Ftx2v);
    if (fabs(d) < thresh) { if (out) out[count] = i; count++; }
  }
  return count;
}

/* viso_mono.cpp:41-72 with an explicit sample table (iters x 8) in place of getRandomSample */
int vo_ransac(const vo_match* pm, int n, const int32_t* samples, int iters, double thresh, double* F9, int32_t* inliers,
              int32_t* counts, double* F_all, int32_t* best_iter) {
  int32_t* cur = (int32_t*)malloc((size_t)n * sizeof(int32_t));
  int best_n = 0, best_k = -1;
  double F[9];
  for (int k = 0; k < iters; k++) {
    vo_fundamental(pm, samples + 8 * k, 8, F);
    if (F_all) memcpy(F_all + 9 * k, F, sizeof F);
    const int c = vo_get_inlier(pm, n, F, thresh, cur);
    if (counts) counts[k] = c;
    if (c > best_n) { best_n = c; best_k = k; memcpy(inliers, cur, (size_t)c * sizeof(int32_t)); }
  }
  free(cur);
  if (best_iter) *best_iter = best_k;
  if (best_n < 10) { memset(F9, 0, 9 * sizeof(double)); return -best_n - 1; }
  vo_fundamental(pm, inliers, best_n, F9);
  return best_n;
}
