/* TEST INFRASTRUCTURE ONLY: plain-C restatement of the semi-global matching of include/visocu.h (visocu_disparity). */
#ifndef SGM_ORACLE_H
#define SGM_ORACLE_H
#include <stdint.h>

/* params7 = {max_disp, paths, p1, p2, uniqueness, lr_max_diff, subpixel}.  left / right: w x h bytes at row stride
 * `stride`.  out: w x h int16 (row stride w).  S (may be NULL): w x h x max_disp uint16, S[(y w + x) D + d].
 * Returns 0, or -1 for parameters outside the valid ranges. */
int vo_sgm(const uint8_t* left, const uint8_t* right, int w, int h, int stride, const int32_t* params7, int16_t* out,
           uint16_t* S);

#endif
