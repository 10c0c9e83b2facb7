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

static_assert(sizeof(Point3d) == 12, "a device point store holds packed x, y, z floats");

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

  // extension: raw camera images of r.src_w x r.src_h for update() (VisualOdometryMono::setRectification); the
  // reconstruction uses the rectified projection.  Before the first frame only, else false and nothing changes.  update()
  // hands the constructor's dims to the push, so construct the facade with the raw size {src_w, src_h, bytes per line}.
  bool setRectification(const Rectification& r) {
    if (!viso->setRectification(r)) return false;
    if (r.n_cams > 0) reconstruction.setCalibration(r.cams[0].f, r.cams[0].cu, r.cams[0].cv);
    return true;
  }

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
// the previous motion, then the batch halves of VisualOdometryStereo around one single-job visocu_stereo_motion, and
// Reconstruction::batchPrepareTracks with one single-job visocu_recon_update on the matcher's context.  The points live in
// a device store (visocu_recon_store): they are moved and appended there, and the host never touches the cloud.  That is
// what the sequence runner's stereo structure-from-motion mode (visob_runner_create_stereo_sfm) does for each of its
// sequences.
class StructureFromMotionStereo {
  std::unique_ptr<VisualOdometryStereo> viso;
  VisualOdometryStereo::parameters param;
  Reconstruction reconstruction;
  visocu_recon_store* store = nullptr;   // the points, on the matcher's context (created by the first reconstruct)
  std::vector<Point3d> points;           // host mirror of the store, refreshed by getPoints after an update
  bool points_stale = false;
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

  // Reconstruction::update with the facade's constants, on the device: the stored points move with the motion, the
  // finished tracks are evaluated and the kept points appended.  If the device call fails, the finished tracks of this
  // frame are lost (batchPrepareTracks has dropped them) and the frame is reported as failed.
  bool reconstruct(visocu_ctx* ctx) {
    if (!store && visocu_recon_store_create(ctx, 0, &store) != VISOCU_OK) {
      std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
      return false;
    }
    const Matrix Tr = viso->getMotion();
    const visocu_recon_job& job = reconstruction.batchPrepareTracks(viso->getMatches(), Tr, 0, 2, 30, 3);
    double tr[12];
    for (int r = 0; r < 3; r++) for (int c = 0; c < 4; c++) tr[4 * r + c] = Tr.val[r][c];
    const double* trp = tr;
    points_stale = true;
    if (visocu_recon_update(ctx, 1, &store, &trp, &job, 0, 0, 0) != VISOCU_OK) {
      std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
      return false;
    }
    return true;
  }

public:
  StructureFromMotionStereo(VisualOdometryStereo::parameters params, const std::array<uint32_t, 3> dims_)
      : viso(new VisualOdometryStereo(params)), param(params), dims(dims_) {
    reconstruction.setCalibration(params.calib.f, params.calib.cu, params.calib.cv);
  }
  ~StructureFromMotionStereo() {
    if (store) visocu_recon_store_destroy(viso->getMatcher()->context(), store);
  }
  StructureFromMotionStereo(const StructureFromMotionStereo&) = delete;
  StructureFromMotionStereo& operator=(const StructureFromMotionStereo&) = delete;

  void setVerbose(bool on) { verbose = on; }

  // extension: raw stereo pairs of r.src_w x r.src_h for update() (VisualOdometryStereo::setRectification); odometry and
  // reconstruction use the rectified projection and r.base.  Before the first frame only, else false and nothing changes.
  // update() hands the constructor's dims to the push, so construct the facade with the raw size.
  bool setRectification(const Rectification& r) {
    if (!viso->setRectification(r)) return false;
    param.calib.f = r.cams[0].f; param.calib.cu = r.cams[0].cu; param.calib.cv = r.cams[0].cv; param.base = r.base;
    reconstruction.setCalibration(param.calib.f, param.calib.cu, param.calib.cv);
    return true;
  }

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

  // points of all finished tracks, in current camera coordinates: a host copy of the device store
  const std::vector<Point3d>& getPoints() {
    if (points_stale) {
      const float* d = 0; int64_t n = 0;
      visocu_recon_store_points(store, &d, &n);
      points.resize((size_t)n);
      visocu_ctx* ctx = viso->getMatcher()->context();
      if (visocu_recon_store_read(ctx, store, 0, n, (float*)points.data()) != VISOCU_OK) {
        std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
        points.clear();
      }
      points_stale = false;
    }
    return points;
  }
  // the same points in device memory (x, y, z floats per point), valid until the next update; null and 0 before the
  // first reconstruction
  void devicePoints(const float** d_xyz, int64_t* n) const {
    *d_xyz = 0; *n = 0;
    if (store) visocu_recon_store_points(store, d_xyz, n);
  }
  const Matrix& getPose() const { return Tr_total; }
  VisualOdometryStereo& odometry() { return *viso; }
  // dense disparity of the last pair (Matcher::computeDisparity)
  bool computeDisparity(const visocu_sgm_params& p, int16_t* out, bool on_device) { return viso->getMatcher()->computeDisparity(p, out, on_device); }
};
#endif
