// Structure-from-motion facade with the reference's interface (viso/sfm.hh:7-83): one image in, monocular odometry on
// the GPU path, pose accumulation and track-based reconstruction on the host.  The reference picks its OpenCL or CPU
// odometry here; this library has exactly one backend (CUDA, no CPU fallback), so the third constructor argument is
// accepted for source compatibility and ignored.
#ifndef VISOB_SFM_H
#define VISOB_SFM_H
#include <array>
#include <iostream>
#include <memory>
#include "reconstruction.h"
#include "viso_mono.h"

class StructureFromMotion {
  std::unique_ptr<VisualOdometryMono> viso;
  Reconstruction reconstruction;
  bool replace = false;
  bool is_first_frame = true;
  bool verbose = true;
  std::array<uint32_t, 3> dims;
  Matrix Tr_total = Matrix::eye(4);      // first camera frame -> current camera frame, accumulated as in the reference

public:
  StructureFromMotion(VisualOdometryMono::parameters params, const std::array<uint32_t, 3> dims_, const bool /*use_accelerator*/ = true)
      : dims(dims_) {
    reconstruction.setCalibration(params.calib.f, params.calib.cu, params.calib.cv);
    viso.reset(new VisualOdometryMono(params));
  }

  void setVerbose(bool on) { verbose = on; }     // the reference always prints; tests and batch runs switch it off

  // returns whether the odometry of this frame succeeded (an extension: the reference's update returns nothing)
  bool update(uint8_t* img_data) {
    const bool ok = viso->process(img_data, &dims[0], replace);
    if (is_first_frame) {
      is_first_frame = false;
      if (verbose) std::cout << std::endl;
    } else if (ok) {
      Tr_total = Tr_total * Matrix::inv(viso->getMotion());
      if (verbose) {
        const double nm = viso->getNumberOfMatches(), ni = viso->getNumberOfInliers();
        std::cout << "Matches: " << nm << ", Inliers: " << 100.0 * ni / nm << '%' << ", Current pose: " << std::endl;
        std::cout << Tr_total << std::endl << std::endl;
      }
      reconstruction.update(viso->getMatches(), viso->getMotion(), 0, 2, 30, 3);
      replace = false;
    } else {
      if (verbose) std::cout << "No motion" << std::endl;
      replace = true;
    }
    return ok;
  }

  const std::vector<Point3d>& getPoints() { return reconstruction.getPoints(); }
  const Matrix& getPose() const { return Tr_total; }
  VisualOdometryMono& odometry() { return *viso; }
};
#endif
