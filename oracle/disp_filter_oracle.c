/* TEST INFRASTRUCTURE ONLY (built by disp_filter_oracle.mk, loaded by disp_filter_oracle.py): the post-filters of
 * visocu_disparity and visocu_disparity_filter, one pixel at a time.
 * Written from the filters' statement (include/visocu.h), not from the CUDA source. */
#include "disp_filter_oracle.h"
#include <stdlib.h>
#include <string.h>

/* lower median of the valid values of the 3x3 window of (x, y) clipped to the image, (x, y) itself valid */
static int median3(const int16_t* m, int w, int h, int x, int y) {
  int v[9], n = 0;
  for (int yy = y - 1; yy <= y + 1; yy++)
    for (int xx = x - 1; xx <= x + 1; xx++) {
      if (xx < 0 || xx >= w || yy < 0 || yy >= h) continue;
      const int e = m[(size_t)yy * w + xx];
      if (e < 0) continue;
      int j = n++;                         /* insertion sort */
      while (j > 0 && v[j - 1] > e) { v[j] = v[j - 1]; j--; }
      v[j] = e;
    }
  return v[(n - 1) / 2];
}

int vo_disp_filter(int16_t* map, int w, int h, int median, int speckle_size, int speckle_range) {
  if ((median != 0 && median != 1) || speckle_size < 0 || speckle_range < 0 || w <= 0 || h <= 0) return -1;
  const size_t n = (size_t)w * h;
  if (median) {
    int16_t* src = malloc(n * sizeof(int16_t));
    memcpy(src, map, n * sizeof(int16_t));
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++)
        if (src[(size_t)y * w + x] >= 0) map[(size_t)y * w + x] = (int16_t)median3(src, w, h, x, y);
    free(src);
  }
  if (speckle_size > 0) {
    /* every valid pixel not yet seen starts a flood fill over the 4-neighbours that are valid and within 16 range of the
     * pixel they are reached from; the component is the queue's content when it runs dry */
    const int r16 = 16 * speckle_range;
    uint8_t* seen = calloc(n, 1);
    int32_t* queue = malloc(n * sizeof(int32_t));
    static const int nb[4][2] = {{1, 0}, {-1, 0}, {0, 1}, {0, -1}};
    for (size_t s = 0; s < n; s++) {
      if (seen[s] || map[s] < 0) continue;
      size_t head = 0, tail = 0;
      queue[tail++] = (int32_t)s;
      seen[s] = 1;
      while (head < tail) {
        const int p = queue[head++], px = p % w, py = p / w, v = map[p];
        for (int j = 0; j < 4; j++) {
          const int qx = px + nb[j][0], qy = py + nb[j][1];
          if (qx < 0 || qx >= w || qy < 0 || qy >= h) continue;
          const int q = qy * w + qx;
          if (seen[q] || map[q] < 0 || abs(map[q] - v) > r16) continue;
          seen[q] = 1;
          queue[tail++] = q;
        }
      }
      if (tail <= (size_t)speckle_size)
        for (size_t i = 0; i < tail; i++) map[queue[i]] = -1;
    }
    free(seen); free(queue);
  }
  return 0;
}
