/* TEST INFRASTRUCTURE ONLY (built by sgm_oracle.mk, loaded by sgm_oracle.py): the semi-global matching of
 * visocu_disparity, one pixel and one disparity at a time.
 * Written from the algorithm's statement (include/visocu.h), not from the CUDA source. */
#include "sgm_oracle.h"
#include <stdlib.h>
#include <string.h>

static int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

static uint64_t census(const uint8_t* I, int w, int h, int stride, int x, int y) {
  const int c = I[(size_t)y * stride + x];
  uint64_t bits = 0;
  int b = 0;
  for (int dy = -3; dy <= 3; dy++)
    for (int dx = -4; dx <= 4; dx++) {
      if (dx == 0 && dy == 0) continue;
      const int v = I[(size_t)clampi(y + dy, 0, h - 1) * stride + clampi(x + dx, 0, w - 1)];
      if (v < c) bits |= (uint64_t)1 << b;
      b++;
    }
  return bits;
}

static int popcount64(uint64_t v) {
  int n = 0;
  while (v) { v &= v - 1; n++; }
  return n;
}

static int floor_div(int a, int b) {   /* b > 0 */
  int q = a / b;
  if (a % b != 0 && a < 0) q--;
  return q;
}

int vo_sgm(const uint8_t* left, const uint8_t* right, int w, int h, int stride, const int32_t* params7, int16_t* out,
           uint16_t* S_out) {
  const int D = params7[0], paths = params7[1], P1 = params7[2], P2 = params7[3], U = params7[4], LR = params7[5],
            SUB = params7[6];
  if ((D != 64 && D != 128 && D != 256) || (paths != 4 && paths != 8) || P1 < 1 || P1 >= P2 || P2 > 150 || U < 0 || U > 100 ||
      LR < -1 || LR > D || (SUB != 0 && SUB != 1) || w <= 0 || h <= 0 || stride < w)
    return -1;
  const size_t n = (size_t)w * h;
  uint64_t* cl = malloc(n * sizeof(uint64_t));
  uint64_t* cr = malloc(n * sizeof(uint64_t));
  uint8_t* C = malloc(n * D);
  uint16_t* S = calloc(n * D, sizeof(uint16_t));
  int16_t* Lrow[2] = {malloc((size_t)w * D * sizeof(int16_t)), malloc((size_t)w * D * sizeof(int16_t))};
  for (int y = 0; y < h; y++)
    for (int x = 0; x < w; x++) {
      cl[(size_t)y * w + x] = census(left, w, h, stride, x, y);
      cr[(size_t)y * w + x] = census(right, w, h, stride, x, y);
    }
  for (int y = 0; y < h; y++)
    for (int x = 0; x < w; x++)
      for (int d = 0; d < D; d++)
        C[((size_t)y * w + x) * D + d] = (uint8_t)(x - d >= 0 ? popcount64(cl[(size_t)y * w + x] ^ cr[(size_t)y * w + x - d]) : 62);

  static const int dirs[8][2] = {{1, 0}, {-1, 0}, {0, 1}, {0, -1}, {1, 1}, {-1, 1}, {1, -1}, {-1, -1}};
  for (int r = 0; r < paths; r++) {
    const int rx = dirs[r][0], ry = dirs[r][1];
    /* rows in the order of ry, pixels of a row in the order of rx: p - r is always done before p.  Lrow[cur] holds the
     * row being computed, Lrow[1 - cur] the row before it in that order. */
    int cur = 0;
    for (int yi = 0; yi < h; yi++) {
      const int y = ry >= 0 ? yi : h - 1 - yi;
      for (int xi = 0; xi < w; xi++) {
        const int x = rx >= 0 ? xi : w - 1 - xi;
        const int px = x - rx, py = y - ry;
        int16_t* L = Lrow[cur] + (size_t)x * D;
        const uint8_t* c = C + ((size_t)y * w + x) * D;
        if (px < 0 || px >= w || py < 0 || py >= h) {
          for (int d = 0; d < D; d++) L[d] = c[d];
        } else {
          const int16_t* Lp = (ry == 0 ? Lrow[cur] : Lrow[1 - cur]) + (size_t)px * D;
          int M = Lp[0];
          for (int k = 1; k < D; k++) if (Lp[k] < M) M = Lp[k];
          for (int d = 0; d < D; d++) {
            int best = Lp[d];
            if (d > 0 && Lp[d - 1] + P1 < best) best = Lp[d - 1] + P1;
            if (d < D - 1 && Lp[d + 1] + P1 < best) best = Lp[d + 1] + P1;
            if (M + P2 < best) best = M + P2;
            L[d] = (int16_t)(c[d] + best - M);
          }
        }
        uint16_t* s = S + ((size_t)y * w + x) * D;
        for (int d = 0; d < D; d++) s[d] = (uint16_t)(s[d] + L[d]);
      }
      cur = 1 - cur;
    }
  }

  int* dstar = malloc(n * sizeof(int));
  int* dright = malloc(n * sizeof(int));
  for (int y = 0; y < h; y++)
    for (int x = 0; x < w; x++) {
      const uint16_t* s = S + ((size_t)y * w + x) * D;
      int best = 0;
      for (int d = 1; d < D; d++) if (s[d] < s[best]) best = d;
      dstar[(size_t)y * w + x] = best;
      /* right map: the smallest d in [0, min(D, w - x)) of min S(x + d, y, d) */
      int rb = 0, rv = S[((size_t)y * w + x) * D];
      for (int d = 1; d < D && x + d < w; d++) {
        const int v = S[((size_t)y * w + x + d) * D + d];
        if (v < rv) { rv = v; rb = d; }
      }
      dright[(size_t)y * w + x] = rb;
    }
  for (int y = 0; y < h; y++)
    for (int x = 0; x < w; x++) {
      const uint16_t* s = S + ((size_t)y * w + x) * D;
      const int ds = dstar[(size_t)y * w + x];
      int valid = 1;
      for (int d = 0; d < D; d++)
        if (abs(d - ds) > 1 && 100 * s[ds] > U * s[d]) valid = 0;
      if (LR >= 0) {
        if (x - ds < 0) valid = 0;
        else if (abs(dright[(size_t)y * w + x - ds] - ds) > LR) valid = 0;
      }
      int v = 16 * ds;
      if (SUB && ds > 0 && ds < D - 1) {
        const int a = s[ds - 1], b = s[ds], c = s[ds + 1], den = a + c - 2 * b;
        if (den > 0) v += floor_div(16 * (a - c) + den, 2 * den);
      }
      out[(size_t)y * w + x] = (int16_t)(valid ? v : -1);
    }
  if (S_out) memcpy(S_out, S, n * D * sizeof(uint16_t));
  free(cl); free(cr); free(C); free(S); free(Lrow[0]); free(Lrow[1]); free(dstar); free(dright);
  return 0;
}
