/* TEST INFRASTRUCTURE ONLY -- plain-C restatement of the reference's hot path (see viso_oracle.c).
 * Parity status: PINNED -- tests/test_oracle_vs_ref.py checks every function below against the unmodified
 * reference compiled into oracle/_ref (here) and against the committed fixtures in tests/golden (anywhere). */
#ifndef VISO_ORACLE_H
#define VISO_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {            /* Matcher::parameters, matcher.h:42-69 (same order) */
  int32_t nms_n, nms_tau, match_binsize, match_radius, match_disp_tolerance;
  int32_t outlier_disp_tolerance, outlier_flow_tolerance, multi_stage, half_resolution, refinement;
  double f, cu, cv, base;
} vo_params;

typedef struct {            /* Matcher::p_match, matcher.h:86-100 */
  float u1p, v1p; int32_t i1p;
  float u2p, v2p; int32_t i2p;
  float u1c, v1c; int32_t i1c;
  float u2c, v2c; int32_t i2c;
} vo_match;

typedef struct { float u_min[4], u_max[4], v_min[4], v_max[4]; } vo_range;   /* matcher.h:152-157 */

int  vo_bpl(int w);
void vo_pad_image(const uint8_t* I, int w, int h, int bpl_in, uint8_t* out);
void vo_half_dims(const int32_t dims[3], int32_t dims_half[3]);
void vo_half_image(const uint8_t* I, const int32_t dims[3], uint8_t* out);
void vo_sobel5x5(const uint8_t* I, int w, int h, uint8_t* du, uint8_t* dv);
void vo_sobel3x3(const uint8_t* I, int w, int h, uint8_t* du, uint8_t* dv);
void vo_blob5x5(const uint8_t* I, int w, int h, int16_t* out);
void vo_checkerboard5x5(const uint8_t* I, int w, int h, int16_t* out);
int  vo_sparse_nms_n(int nms_n);
int  vo_nms(const int16_t* f1, const int16_t* f2, const int32_t dims[3], int n, int tau, int32_t* out4, int cap);
void vo_descriptor(const uint8_t* du, const uint8_t* dv, int bpl, int u, int v, uint8_t* out32);
void vo_small_descriptor(const uint8_t* du, const uint8_t* dv, int bpl, int u, int v, uint8_t* out16);
int  vo_sad(const uint8_t* a, const uint8_t* b, int nbytes);
/* computeFeatures: Ipad is the 16-byte-stride copy; planes are caller-allocated bpl*h (full planes only
 * written when half_resolution).  rec1/rec2 receive 12-int32 records.  Returns 0, counts in n1/n2. */
int  vo_compute_features(const uint8_t* Ipad, const int32_t dims[3], const vo_params* p,
                         uint8_t* du, uint8_t* dv, uint8_t* du_full, uint8_t* dv_full,
                         int32_t* rec1, int cap1, int32_t* n1, int32_t* rec2, int cap2, int32_t* n2);
/* method 0 flow, 1 stereo, 2 quad; tr_delta (quad only, may be NULL): rows 0..2 of Tr_delta, 12 doubles, with
 * p->f, cu, cv, base.  counts2 (may be NULL): entries of the scanned bins and window candidates over all hops. */
int  vo_matching(int method, const int32_t* m1p, int n1p, const int32_t* m2p, int n2p,
                 const int32_t* m1c, int n1c, const int32_t* m2c, int n2c,
                 const int32_t dims_c[3], const vo_params* p, int use_prior, const vo_range* ranges,
                 const double* tr_delta, vo_match* out, int cap, int64_t* counts2);
int  vo_prior_statistics(const vo_match* pm, int n, int method, const int32_t dims_c[3], const vo_params* p, vo_range* ranges);
void vo_refine_pixel(vo_match* pm, int n, int method, const int32_t dims_p[3], const int32_t dims_c[3],
                     const uint8_t* du1p, const uint8_t* dv1p, const uint8_t* du2p, const uint8_t* dv2p,
                     const uint8_t* du1c, const uint8_t* dv1c, const uint8_t* du2c, const uint8_t* dv2c);
void vo_refine_subpixel(vo_match* pm, int n, int method, const int32_t dims_p[3], const int32_t dims_c[3],
                        const uint8_t* du1p, const uint8_t* dv1p, const uint8_t* du2p, const uint8_t* dv2p,
                        const uint8_t* du1c, const uint8_t* dv1c, const uint8_t* du2c, const uint8_t* dv2c,
                        uint8_t* keep, double* margin);
/* RANSAC pieces (FP64).  Compiled with -ffp-contract=off: bit-comparable to oracle/_ref/libvisoref_nofma.so */
void vo_svd(double* a, int m, int n, double* w, double* v);
int  vo_normalize(vo_match* pm, int n, double* Tp9, double* Tc9);
void vo_fundamental(const vo_match* pm, const int32_t* active, int nactive, double* F9);
int  vo_get_inlier(const vo_match* pm, int n, const double* F9, double thresh, int32_t* out);
int  vo_ransac(const vo_match* pm, int n, const int32_t* samples, int iters, double thresh,
               double* F9, int32_t* inliers, int32_t* counts, double* F_all, int32_t* best_iter);

#ifdef __cplusplus
}
#endif
#endif
