// Structure-from-motion facade with the reference's interface (viso/sfm.hh:7-83): one image in, monocular odometry on
// the GPU path, pose accumulation and track-based reconstruction on the host.  The reference picks its OpenCL or CPU
// odometry here; this library has exactly one backend (CUDA, no CPU fallback), so the third constructor argument is
// accepted for source compatibility and ignored.  StructureFromMotionStereo (below) is the same facade for a stereo rig.
#ifndef VISOB_SFM_H
#define VISOB_SFM_H
#include <array>
#include <iostream>
#include <memory>
#include "reconstruction.h"
#include "viso_mono.h"
#include "viso_stereo.h"
#include "visocu.h"

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

// Extension (not in the reference): structure from motion on a stereo rig.  update() has StructureFromMotion::update's
// semantics with VisualOdometryStereo in place of the mono odometry, so the motion is metric (from the baseline) instead of
// scaled by a ground-plane guess.  Unlike StructureFromMotion, it estimates and reconstructs on the GPU: quad matching with
// the previous motion, then the batch halves of VisualOdometryStereo and Reconstruction around one single-job
// visocu_stereo_motion and one single-job visocu_recon_points on the matcher's context.  That is what the sequence
// runner's stereo structure-from-motion mode (visob_runner_create_stereo_sfm) does for each of its sequences.
class StructureFromMotionStereo {
  std::unique_ptr<VisualOdometryStereo> viso;
  VisualOdometryStereo::parameters param;
  Reconstruction reconstruction;
  bool replace = false;
  bool is_first_frame = true;
  bool verbose = true;
  std::array<uint32_t, 3> dims;
  Matrix Tr_total = Matrix::eye(4);      // first camera frame -> current camera frame

  // the motion estimate of process() (bucketing, sample table) with the device doing the RANSAC and the refinement
  bool estimateMotion(visocu_ctx* ctx) {
    const visocu_pmatch* m = 0; int32_t n = 0; const int32_t* smp = 0;
    if (!viso->batchPrepare(&m, &n, &smp)) return false;
    std::vector<uint8_t> mask((size_t)n);
    uint8_t* mp = mask.data();
    double tr[6]; int32_t ok = 0;
    const visocu_stereo_params sp = {param.calib.f, param.calib.cu, param.calib.cv, param.base, param.inlier_threshold,
                                     param.ransac_iters, param.reweighting};
    if (visocu_stereo_motion(ctx, 1, &m, &n, &smp, &sp, tr, &ok, &mp, 0, 0, 0, 0) != VISOCU_OK) {
      std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
      return false;
    }
    return viso->batchFinish(tr, ok, mp);
  }

  // Reconstruction::update with the facade's constants, the finished tracks evaluated on the device.  If the device call
  // fails, the finished tracks of this frame are lost (batchPrepare has dropped them) and the frame is reported as failed.
  bool reconstruct(visocu_ctx* ctx) {
    const visocu_recon_job& job = reconstruction.batchPrepare(viso->getMatches(), viso->getMotion(), 0, 2, 30, 3);
    std::vector<int32_t> status((size_t)job.n_tracks);
    std::vector<float> xyz(3 * (size_t)job.n_tracks);
    int32_t* sp = status.data();
    float* xp = xyz.data();
    if (visocu_recon_points(ctx, 1, &job, &sp, &xp) != VISOCU_OK) {
      std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
      return false;
    }
    reconstruction.batchFinish(sp, xp);
    return true;
  }

public:
  StructureFromMotionStereo(VisualOdometryStereo::parameters params, const std::array<uint32_t, 3> dims_)
      : viso(new VisualOdometryStereo(params)), param(params), dims(dims_) {
    reconstruction.setCalibration(params.calib.f, params.calib.cu, params.calib.cv);
  }

  void setVerbose(bool on) { verbose = on; }

  // left / right: one rectified stereo pair of dims; returns whether the odometry of this frame succeeded (and, after the
  // first frame, the reconstruction's device call)
  bool update(uint8_t* left, uint8_t* right) {
    Matcher& matcher = *viso->getMatcher();
    matcher.pushBack(left, right, &dims[0], replace);
    matcher.matchFeatures(2, viso->predictedMotion());
    bool ok = estimateMotion(matcher.context());
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
      ok = reconstruct(matcher.context());
      replace = false;
    } else {
      if (verbose) std::cout << "No motion" << std::endl;
      replace = true;
    }
    return ok;
  }

  const std::vector<Point3d>& getPoints() { return reconstruction.getPoints(); }
  const Matrix& getPose() const { return Tr_total; }
  VisualOdometryStereo& odometry() { return *viso; }
};
#endif
