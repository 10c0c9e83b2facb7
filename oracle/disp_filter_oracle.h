/* TEST INFRASTRUCTURE ONLY: plain-C restatement of the disparity post-filters of include/visocu.h (visocu_disparity,
 * visocu_disparity_filter). */
#ifndef DISP_FILTER_ORACLE_H
#define DISP_FILTER_ORACLE_H
#include <stdint.h>

/* The post-filters in place on a w x h int16 map (row stride w): masked 3x3 median (median = 1), then speckle removal
 * (speckle_size > 0, components by breadth-first flood fill).  Returns 0, or -1 for median outside {0, 1},
 * speckle_size < 0, speckle_range < 0, w or h <= 0. */
int vo_disp_filter(int16_t* map, int w, int h, int median, int speckle_size, int speckle_range);

#endif
