// Camera model, stereo rectification and rectification maps for raw camera images (not in the reference, which expects
// undistorted, rectified input).  A camera (visocu_camera, include/visocu.h) is a raw pinhole K = (fx, fy, cx, cy) with
// radial-tangential distortion k1, k2, p1, p2, k3 (the model of OpenCV's and KITTI's calibration files), the rectifying
// rotation R (raw camera coordinates -> rectified coordinates, row-major) and the rectified projection f, cu, cv.
//
// The map of a camera gives, for every output pixel (u, v), the raw image position it samples: the ray
// R^T ((u - cu) / f, (v - cv) / f, 1) divided by its z, distorted, projected with K, in 1/32 pixel (lrint(32 x),
// lrint(32 y)) and clamped to [0, 32 (src_w - 1)] x [0, 32 (src_h - 1)], computed in double.  The clamp replicates the
// border: a zero border would put strong artificial edges into the filter responses.  The library compiles this file
// into both of its shared libraries: libvisocu builds the maps, the host layer builds rigs.
#ifndef VISOB_RECTIFY_H
#define VISOB_RECTIFY_H
#include <stdint.h>
#include "visocu.h"

// What Matcher::setRectification and the facades take: n_cams maps (1 for a monocular matcher, 2 for a stereo rig: the
// left images use cams[0], the right ones cams[1]), raw images of src_w x src_h in, out_w x out_h rectified images to
// the matcher.  base is the rectified baseline (stereo odometry), the rectified projection of cams[0] is the calibration.
// A plain C struct: the Python binding mirrors it.
struct Rectification {
  int32_t n_cams;
  visocu_camera cams[2];
  int32_t src_w, src_h, out_w, out_h;
  double base;
};

namespace visob {
// true if the camera and the sizes are acceptable (finite parameters, fx, fy, f > 0, src in [16, 8191], out in [1, 8191]),
// else a message in *why
bool rectifyCheck(const visocu_camera& c, int32_t src_w, int32_t src_h, int32_t out_w, int32_t out_h, const char** why);
// The map of one camera (2 int32 per output pixel, row-major, x then y); false (and *why) for a camera rectifyCheck
// rejects or an output pixel whose rotated ray has z <= 0.
bool rectifyMap(const visocu_camera& c, int32_t src_w, int32_t src_h, int32_t out_w, int32_t out_h, int32_t* map, const char** why);

// Bouguet's construction for a rig whose camera 1 sees X1 = R X0 + T (R row-major).  The relative rotation is split into
// two halves (rotation vector / 2), one applied to each camera; a second rotation, common to both, turns camera 1's centre
// onto the +x axis of camera 0.  Both cameras get f = min(fy0, fy1) and one principal point (cu, cv): disparity is zero at
// infinity.  (cu, cv) puts the mean of the two rotated optical axes at the centre ((out_w - 1) / 2, (out_h - 1) / 2) of
// the output image.  The rest of each camera (K, distortion) is copied from the input.  *base = |T|.  No free scaling
// (OpenCV's alpha) is offered, and the result is not claimed equal to OpenCV's stereoRectify.
void stereoRectify(const visocu_camera& cam0, const visocu_camera& cam1, const double R[9], const double T[3], int32_t out_w,
                   int32_t out_h, visocu_camera* rect0, visocu_camera* rect1, double* base);
}  // namespace visob
#endif
