// extern "C" access to the C++ host layer for the Python tests and bench.py (ctypes), plus the sharded
// sequence runner (SURVEY.md 8e: independent sequences, one host worker set and one CUDA stream per Matcher,
// no collective).  Plain pointers and sizes only.
#include <atomic>
#include <chrono>
#include <cstring>
#include <iostream>
#include <memory>
#include <sstream>
#include <thread>
#include <vector>

#include "delaunay.h"
#include "device.h"
#include "filter.h"
#include "matcher.h"
#include "viso_mono.h"
#include "viso_stereo.h"
#include "reconstruction.h"
#include "rectify.h"
#include "sfm.h"
#include "visocu.h"

#define VISOB_API extern "C" __attribute__((visibility("default")))

namespace {
struct MonoParamsC {          // flat mirror of VisualOdometryMono::parameters (same as oracle/pyref.py MonoParams)
  Matcher::parameters match;
  int32_t bucket_max_features; double bucket_width, bucket_height;
  double f, cu, cv;
  double height, pitch; int32_t ransac_iters; double inlier_threshold, motion_threshold;
};
VisualOdometryMono::parameters to_cpp(const MonoParamsC* p) {
  VisualOdometryMono::parameters q;
  q.match = p->match;
  q.bucket.max_features = p->bucket_max_features; q.bucket.bucket_width = p->bucket_width; q.bucket.bucket_height = p->bucket_height;
  q.calib.f = p->f; q.calib.cu = p->cu; q.calib.cv = p->cv;
  q.height = p->height; q.pitch = p->pitch; q.ransac_iters = p->ransac_iters;
  q.inlier_threshold = p->inlier_threshold; q.motion_threshold = p->motion_threshold;
  return q;
}
int copy_matches(const std::vector<Matcher::p_match>& v, void* out, int cap) {
  const int n = (int)v.size();
  if (out && n > 0) memcpy(out, v.data(), sizeof(Matcher::p_match) * (size_t)std::min(n, cap));
  return n;
}
struct MonoAccess : public VisualOdometryMono {
  explicit MonoAccess(VisualOdometryMono::parameters p) : VisualOdometryMono(p) {}
};
}  // namespace

VISOB_API void visob_set_device(int device) { visob::set_device(device); }
VISOB_API void visob_set_pipeline_depth(int depth) { visob::set_pipeline_depth(depth); }

namespace visob { extern std::atomic<long long> g_stage_ns[8]; extern std::atomic<long long> g_stage_calls[8]; }
// stage ids: 0 pushBack, 1 matching pass 1, 2 matching pass 2 (+refinement), 3 priors, 4 removeOutliers (< 2000 matches), 5 removeOutliers (larger), 6 ransacEstimateF, 7 estimateMotion (total, includes 6)
VISOB_API void visob_stage_times(double* seconds8, int64_t* calls8, int reset) {
  for (int k = 0; k < 8; k++) {
    seconds8[k] = visob::g_stage_ns[k].load() * 1e-9; calls8[k] = visob::g_stage_calls[k].load();
    if (reset) { visob::g_stage_ns[k] = 0; visob::g_stage_calls[k] = 0; }
  }
}

// ---- Matcher
VISOB_API void* visob_matcher_create(const Matcher::parameters* p) { return new Matcher(*p); }
VISOB_API void visob_matcher_destroy(void* m) { delete (Matcher*)m; }
VISOB_API void visob_matcher_push(void* m, uint8_t* I1, uint8_t* I2, const int32_t* dims, int replace) {
  uint32_t d[3] = {(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]};
  ((Matcher*)m)->pushBack(I1, I2, d, replace != 0);
}
VISOB_API void visob_matcher_push_device(void* m, const uint8_t* I1, const uint8_t* I2, const int32_t* dims, int replace) {
  uint32_t d[3] = {(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]};
  ((Matcher*)m)->pushBackDevice(I1, I2, d, replace != 0);
}
VISOB_API void visob_matcher_match_features(void* m, int method) { ((Matcher*)m)->matchFeatures(method, 0); }
VISOB_API void visob_matcher_bucket(void* m, int max_features, float bw, float bh) { ((Matcher*)m)->bucketFeatures(max_features, bw, bh); }
VISOB_API int visob_matcher_get_matches(void* m, int stage, void* out, int cap) { return copy_matches(((Matcher*)m)->matches(stage), out, cap); }
VISOB_API void visob_matcher_counts(void* m, int32_t* out8) { for (int k = 0; k < 8; k++) out8[k] = ((Matcher*)m)->featureCount(k); }
VISOB_API float visob_matcher_gain(void* m, const int32_t* inl, int n) { return ((Matcher*)m)->getGain(std::vector<int32_t>(inl, inl + n)); }
VISOB_API void* visob_matcher_context(void* m) { return ((Matcher*)m)->context(); }
VISOB_API int visob_matcher_remove_outliers(void* m, void* inout, int n, int method) {
  std::vector<Matcher::p_match> pm((Matcher::p_match*)inout, (Matcher::p_match*)inout + n);
  ((Matcher*)m)->removeOutliers(pm, method);
  return copy_matches(pm, inout, n);
}
VISOB_API int visob_matcher_prior(void* m, const void* matches, int n, int method, float* ranges_out, int cap_bins) {
  std::vector<Matcher::p_match> pm((const Matcher::p_match*)matches, (const Matcher::p_match*)matches + n);
  ((Matcher*)m)->computePriorStatistics(pm, method);
  const std::vector<Matcher::range>& r = ((Matcher*)m)->priorRanges();
  if (ranges_out) memcpy(ranges_out, r.data(), sizeof(Matcher::range) * (size_t)std::min((int)r.size(), cap_bins));
  return (int)r.size();
}

VISOB_API int visob_matcher_ranges(void* m, float* ranges_out, int cap_bins) {     // the ranges the last matchFeatures used
  const std::vector<Matcher::range>& r = ((Matcher*)m)->priorRanges();
  if (ranges_out) memcpy(ranges_out, r.data(), sizeof(Matcher::range) * (size_t)std::min((int)r.size(), cap_bins));
  return (int)r.size();
}

// ---- filter::
VISOB_API int visob_filter(int which, const uint8_t* in, uint8_t* out_a, uint8_t* out_b, int16_t* out16, int w, int h) {
  try {
    if (which == 0) filter::sobel5x5(in, out_a, out_b, w, h);
    else if (which == 1) filter::sobel3x3(in, out_a, out_b, w, h);
    else if (which == 2) filter::blob5x5(in, out16, w, h);
    else filter::checkerboard5x5(in, out16, w, h);
  } catch (const std::exception&) { return -1; }
  return 0;
}

// ---- mono odometry
VISOB_API void* visob_mono_create(const MonoParamsC* p) { return new MonoAccess(to_cpp(p)); }
VISOB_API void visob_mono_destroy(void* v) { delete (MonoAccess*)v; }
VISOB_API int visob_mono_process(void* v, uint8_t* I, const int32_t* dims, int replace) {
  uint32_t d[3] = {(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]};
  return ((MonoAccess*)v)->process(I, d, replace != 0) ? 1 : 0;
}
VISOB_API int visob_mono_process_device(void* v, const uint8_t* I, const int32_t* dims, int replace) {
  uint32_t d[3] = {(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]};
  return ((MonoAccess*)v)->processDevice(I, d, replace != 0) ? 1 : 0;
}
VISOB_API int visob_mono_process_matches(void* v, const void* matches, int n) {
  std::vector<Matcher::p_match> pm((const Matcher::p_match*)matches, (const Matcher::p_match*)matches + n);
  return ((VisualOdometry*)(MonoAccess*)v)->process(pm) ? 1 : 0;
}
VISOB_API void visob_mono_get_motion(void* v, double* out16) {
  Matrix T = ((MonoAccess*)v)->getMotion();
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) out16[4 * i + j] = T.val[i][j];
}
VISOB_API int visob_mono_get_matches(void* v, void* out, int cap) { return copy_matches(((MonoAccess*)v)->usedMatches(), out, cap); }
VISOB_API int visob_mono_get_inliers(void* v, int32_t* out, int cap) {
  std::vector<int32_t> in = ((MonoAccess*)v)->getInlierIndices();
  if (out) memcpy(out, in.data(), sizeof(int32_t) * (size_t)std::min((int)in.size(), cap));
  return (int)in.size();
}
VISOB_API int visob_mono_get_F(void* v, double* F9) {
  const Matrix& F = ((MonoAccess*)v)->lastF();
  if (!F.val) return 0;
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) F9[3 * i + j] = F.val[i][j];
  return 1;
}
VISOB_API int visob_mono_get_samples(void* v, int32_t* out, int cap) {
  const std::vector<int>& s = ((MonoAccess*)v)->lastSamples();
  if (out) for (int i = 0; i < std::min((int)s.size(), cap); i++) out[i] = s[i];
  return (int)s.size();
}
VISOB_API void* visob_mono_matcher(void* v) { return ((MonoAccess*)v)->getMatcher(); }

// ---- stereo odometry
namespace {
struct StereoParamsC {        // flat mirror of VisualOdometryStereo::parameters (same as oracle/pyref.py StereoParams)
  Matcher::parameters match;
  int32_t bucket_max_features; double bucket_width, bucket_height;
  double f, cu, cv;
  double base; int32_t ransac_iters; double inlier_threshold; int32_t reweighting;
};
VisualOdometryStereo::parameters to_cpp(const StereoParamsC* p) {
  VisualOdometryStereo::parameters q;
  q.match = p->match;
  q.bucket.max_features = p->bucket_max_features; q.bucket.bucket_width = p->bucket_width; q.bucket.bucket_height = p->bucket_height;
  q.calib.f = p->f; q.calib.cu = p->cu; q.calib.cv = p->cv;
  q.base = p->base; q.ransac_iters = p->ransac_iters; q.inlier_threshold = p->inlier_threshold; q.reweighting = p->reweighting != 0;
  return q;
}
}  // namespace
VISOB_API void* visob_stereo_create(const StereoParamsC* p) { return new VisualOdometryStereo(to_cpp(p)); }
VISOB_API void visob_stereo_destroy(void* v) { delete (VisualOdometryStereo*)v; }
VISOB_API int visob_stereo_process(void* v, uint8_t* I1, uint8_t* I2, const int32_t* dims, int replace) {
  uint32_t d[3] = {(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]};
  return ((VisualOdometryStereo*)v)->process(I1, I2, d, replace != 0) ? 1 : 0;
}
VISOB_API int visob_stereo_process_matches(void* v, const void* matches, int n) {     // host only: no image, no GPU
  std::vector<Matcher::p_match> pm((const Matcher::p_match*)matches, (const Matcher::p_match*)matches + n);
  return ((VisualOdometry*)(VisualOdometryStereo*)v)->process(pm) ? 1 : 0;
}
VISOB_API void visob_stereo_get_motion(void* v, double* out16) {
  Matrix T = ((VisualOdometryStereo*)v)->getMotion();
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) out16[4 * i + j] = T.val[i][j];
}
VISOB_API int visob_stereo_get_matches(void* v, void* out, int cap) { return copy_matches(((VisualOdometryStereo*)v)->usedMatches(), out, cap); }
VISOB_API int visob_stereo_get_inliers(void* v, int32_t* out, int cap) {
  std::vector<int32_t> in = ((VisualOdometryStereo*)v)->getInlierIndices();
  if (out) memcpy(out, in.data(), sizeof(int32_t) * (size_t)std::min((int)in.size(), cap));
  return (int)in.size();
}
VISOB_API int visob_stereo_get_samples(void* v, int32_t* out, int cap) {
  const std::vector<int>& s = ((VisualOdometryStereo*)v)->lastSamples();
  if (out) for (int i = 0; i < std::min((int)s.size(), cap); i++) out[i] = s[i];
  return (int)s.size();
}
// the two halves of the batched estimate on a stand-alone object fed with matches (process(matches) split in two)
VISOB_API int visob_stereo_batch_prepare(void* v, const void* matches, int n) {
  std::vector<Matcher::p_match> pm((const Matcher::p_match*)matches, (const Matcher::p_match*)matches + n);
  const visocu_pmatch* m = 0; int32_t N = 0; const int32_t* smp = 0;
  return ((VisualOdometryStereo*)v)->batchPrepare(pm, &m, &N, &smp) ? 1 : 0;
}
VISOB_API int visob_stereo_batch_finish(void* v, const double* tr6, int ok, const uint8_t* mask) {
  return ((VisualOdometryStereo*)v)->batchFinish(tr6, ok, mask) ? 1 : 0;
}
VISOB_API void visob_matcher_match_features_tr(void* m, int method, const double* tr16) {
  Matrix T(4, 4, tr16);
  ((Matcher*)m)->matchFeatures(method, &T);
}
VISOB_API void visob_matcher_set_intrinsics(void* m, double f, double cu, double cv, double base) { ((Matcher*)m)->setIntrinsics(f, cu, cv, base); }

// ---- reconstruction and the facade
VISOB_API void* visob_recon_create() { return new Reconstruction(); }
VISOB_API void visob_recon_destroy(void* r) { delete (Reconstruction*)r; }
VISOB_API void visob_recon_set_calibration(void* r, double f, double cu, double cv) { ((Reconstruction*)r)->setCalibration(f, cu, cv); }
VISOB_API void visob_recon_update(void* r, const void* matches, int n, const double* tr16, int point_type, int min_track_length,
                                  double max_dist, double min_angle) {
  const Matcher::p_match* m = (const Matcher::p_match*)matches;
  ((Reconstruction*)r)->update(std::vector<Matcher::p_match>(m, m + n), Matrix(4, 4, tr16), point_type, min_track_length, max_dist, min_angle);
}
VISOB_API int visob_recon_get_points(void* r, float* out3, int cap) {
  const std::vector<Point3d>& pts = ((Reconstruction*)r)->getPoints();
  for (int i = 0; i < (int)pts.size() && i < cap; i++) { out3[3 * i] = pts[i].x; out3[3 * i + 1] = pts[i].y; out3[3 * i + 2] = pts[i].z; }
  return (int)pts.size();
}
// the two halves of Reconstruction::update around the evaluation of its finished tracks (see reconstruction.h); prepare
// returns the number of tracks to evaluate; prepare_tracks is prepare without moving the stored points
VISOB_API int visob_recon_batch_prepare(void* r, const void* matches, int n, const double* tr16, int point_type, int min_track_length,
                                        double max_dist, double min_angle) {
  const Matcher::p_match* m = (const Matcher::p_match*)matches;
  return ((Reconstruction*)r)->batchPrepare(std::vector<Matcher::p_match>(m, m + n), Matrix(4, 4, tr16), point_type, min_track_length,
                                            max_dist, min_angle).n_tracks;
}
VISOB_API int visob_recon_batch_prepare_tracks(void* r, const void* matches, int n, const double* tr16, int point_type,
                                               int min_track_length, double max_dist, double min_angle) {
  const Matcher::p_match* m = (const Matcher::p_match*)matches;
  return ((Reconstruction*)r)->batchPrepareTracks(std::vector<Matcher::p_match>(m, m + n), Matrix(4, 4, tr16), point_type,
                                                  min_track_length, max_dist, min_angle).n_tracks;
}
// the prepared job: its scalar fields into *job (frames / tracks pointing into the object), and copies of the frame table
// and the tracks into `frames` and `tracks` if they are not null
VISOB_API void visob_recon_batch_job(void* r, visocu_recon_job* job, visocu_recon_frame* frames, visocu_recon_track* tracks) {
  const visocu_recon_job& j = ((Reconstruction*)r)->batchJob();
  *job = j;
  if (frames) memcpy(frames, j.frames, sizeof(visocu_recon_frame) * (size_t)j.n_frames);
  if (tracks && j.n_tracks) memcpy(tracks, j.tracks, sizeof(visocu_recon_track) * (size_t)j.n_tracks);
}
VISOB_API void visob_recon_host_eval(void* r, int32_t* status, float* xyz) { ((Reconstruction*)r)->hostEval(status, xyz); }
VISOB_API void visob_recon_batch_finish(void* r, const int32_t* status, const float* xyz) { ((Reconstruction*)r)->batchFinish(status, xyz); }
VISOB_API void* visob_sfm_create(const MonoParamsC* p, const int32_t* dims) {
  StructureFromMotion* s = new StructureFromMotion(to_cpp(p), std::array<uint32_t, 3>{{(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]}}, true);
  s->setVerbose(false);
  return s;
}
VISOB_API void visob_sfm_destroy(void* s) { delete (StructureFromMotion*)s; }
VISOB_API int visob_sfm_update(void* s, uint8_t* img) { return ((StructureFromMotion*)s)->update(img) ? 1 : 0; }
VISOB_API int visob_sfm_get_points(void* s, float* out3, int cap) {
  const std::vector<Point3d>& pts = ((StructureFromMotion*)s)->getPoints();
  for (int i = 0; i < (int)pts.size() && i < cap; i++) { out3[3 * i] = pts[i].x; out3[3 * i + 1] = pts[i].y; out3[3 * i + 2] = pts[i].z; }
  return (int)pts.size();
}
VISOB_API void visob_sfm_get_pose(void* s, double* out16) {
  const Matrix& T = ((StructureFromMotion*)s)->getPose();
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) out16[4 * i + j] = T.val[i][j];
}
// the stereo facade (host/sfm.h), created with verbose output off; _odometry gives its VisualOdometryStereo for the
// visob_stereo_get_* entries
VISOB_API void* visob_stereo_sfm_create(const StereoParamsC* p, const int32_t* dims) {
  StructureFromMotionStereo* s =
      new StructureFromMotionStereo(to_cpp(p), std::array<uint32_t, 3>{{(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]}});
  s->setVerbose(false);
  return s;
}
VISOB_API void visob_stereo_sfm_destroy(void* s) { delete (StructureFromMotionStereo*)s; }
VISOB_API int visob_stereo_sfm_update(void* s, uint8_t* left, uint8_t* right) {
  return ((StructureFromMotionStereo*)s)->update(left, right) ? 1 : 0;
}
VISOB_API int visob_stereo_sfm_get_points(void* s, float* out3, int cap) {
  const std::vector<Point3d>& pts = ((StructureFromMotionStereo*)s)->getPoints();
  for (int i = 0; i < (int)pts.size() && i < cap; i++) { out3[3 * i] = pts[i].x; out3[3 * i + 1] = pts[i].y; out3[3 * i + 2] = pts[i].z; }
  return (int)pts.size();
}
VISOB_API void visob_stereo_sfm_get_pose(void* s, double* out16) {
  const Matrix& T = ((StructureFromMotionStereo*)s)->getPose();
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) out16[4 * i + j] = T.val[i][j];
}
VISOB_API void* visob_stereo_sfm_odometry(void* s) { return &((StructureFromMotionStereo*)s)->odometry(); }
VISOB_API void visob_stereo_sfm_device_points(void* s, const float** d_xyz, int64_t* n) { ((StructureFromMotionStereo*)s)->devicePoints(d_xyz, n); }

// ---- rectification (host/rectify.h): setRectification of the classes above, 1 = done, 0 = refused
// dense disparity of the current stereo pair (Matcher::computeDisparity): 1 = done, 0 = failed (message on cerr)
VISOB_API int visob_matcher_disparity(void* m, const visocu_sgm_params* p, int16_t* out, int on_device) {
  return ((Matcher*)m)->computeDisparity(*p, out, on_device != 0) ? 1 : 0;
}
VISOB_API int visob_matcher_stereo_pair(void* m, int32_t* frames2, int32_t* wh) { return ((Matcher*)m)->stereoPair(frames2, frames2 + 1, wh, wh + 1) ? 1 : 0; }
VISOB_API void* visob_stereo_matcher(void* v) { return ((VisualOdometryStereo*)v)->getMatcher(); }
VISOB_API int visob_stereo_sfm_disparity(void* s, const visocu_sgm_params* p, int16_t* out, int on_device) {
  return ((StructureFromMotionStereo*)s)->computeDisparity(*p, out, on_device != 0) ? 1 : 0;
}
VISOB_API int visob_matcher_set_rectification(void* m, const Rectification* r) { return ((Matcher*)m)->setRectification(*r) ? 1 : 0; }
VISOB_API int visob_mono_set_rectification(void* v, const Rectification* r) { return ((MonoAccess*)v)->setRectification(*r) ? 1 : 0; }
VISOB_API int visob_stereo_set_rectification(void* v, const Rectification* r) { return ((VisualOdometryStereo*)v)->setRectification(*r) ? 1 : 0; }
VISOB_API int visob_sfm_set_rectification(void* s, const Rectification* r) { return ((StructureFromMotion*)s)->setRectification(*r) ? 1 : 0; }
VISOB_API int visob_stereo_sfm_set_rectification(void* s, const Rectification* r) {
  return ((StructureFromMotionStereo*)s)->setRectification(*r) ? 1 : 0;
}
VISOB_API void visob_stereo_rectify(const visocu_camera* cam0, const visocu_camera* cam1, const double* R9, const double* T3, int32_t out_w,
                                    int32_t out_h, visocu_camera* rect0, visocu_camera* rect1, double* base) {
  visob::stereoRectify(*cam0, *cam1, R9, T3, out_w, out_h, rect0, rect1, base);
}
// the map visocu_set_rectification builds, computed on the host (no device needed): 0, or VISOCU_EINVAL with the reason
// in why (256 bytes, optional)
VISOB_API int visob_rectify_map(const visocu_camera* cam, int32_t src_w, int32_t src_h, int32_t out_w, int32_t out_h, int32_t* out,
                                char* why256) {
  const char* why = "";
  const bool ok = visob::rectifyCheck(*cam, src_w, src_h, out_w, out_h, &why) &&
                  (!out || visob::rectifyMap(*cam, src_w, src_h, out_w, out_h, out, &why));
  if (why256) snprintf(why256, 256, "%s", ok ? "" : why);
  return ok ? VISOCU_OK : VISOCU_EINVAL;
}

// ---- host utilities exposed for tests
VISOB_API int visob_delaunay(const int32_t* x, const int32_t* y, int n, int32_t* tri_out, int cap_tri) {
  std::vector<int32_t> tri;
  visob::delaunay_triangles(x, y, n, tri);
  const int nt = (int)tri.size() / 3;
  if (tri_out) memcpy(tri_out, tri.data(), sizeof(int32_t) * 3 * (size_t)std::min(nt, cap_tri));
  return nt;
}
// edge list (a, b, triangles) of the triangulation; ctx != null: large inputs build their lower tree levels on that context
VISOB_API int visob_delaunay_edges(void* ctx, const int32_t* x, const int32_t* y, int n, int32_t* edges_out, int cap_edges, int64_t* device_nodes) {
  std::vector<int32_t> e;
  const long before = visob::delaunay_device_nodes();
  visob::delaunay_use_device((visocu_ctx*)ctx);
  visob::delaunay_edges(x, y, n, e);
  visob::delaunay_use_device(nullptr);
  if (device_nodes) *device_nodes = visob::delaunay_device_nodes() - before;
  const int ne = (int)e.size() / 3;
  if (edges_out) memcpy(edges_out, e.data(), sizeof(int32_t) * 3 * (size_t)std::min(ne, cap_edges));
  return ne;
}
// affineTransform (host/reconstruction.cpp) on n points: M16 row-major 4x4, x, y, z floats per point
VISOB_API void visob_affine_points(const double* M16, const float* in, float* out, int64_t n) {
  const Matrix M(4, 4, M16);
  for (int64_t i = 0; i < n; i++) {
    const Point3d p = affineTransform(M, Point3d(in[3 * i], in[3 * i + 1], in[3 * i + 2]));
    out[3 * i] = p.x; out[3 * i + 1] = p.y; out[3 * i + 2] = p.z;
  }
}
VISOB_API void visob_svd(const double* A, int m, int n, double* U, double* W, double* V) {
  Matrix M(m, n, A), Um, Wm, Vm;
  M.svd(Um, Wm, Vm);
  for (int i = 0; i < m; i++) for (int j = 0; j < m; j++) U[i * m + j] = Um.val[i][j];
  for (int i = 0; i < std::min(m, n); i++) W[i] = Wm.val[i][0];
  for (int i = 0; i < n; i++) for (int j = 0; j < n; j++) V[i * n + j] = Vm.val[i][j];
}

// ---------------------------------------------------------------------------------------------------------
// Sharded sequence runner.  S independent sequences live on one GPU; sequences are dealt round-robin to `threads` host
// workers.  Matcher mode: every worker drives its sequences through ONE MatcherBatch (one context, one stream, every GPU
// stage a single batched launch for all of the worker's sequences) and runs their host stages (outlier removal, priors,
// bucketing) in between; the workers' streams overlap on the GPU.  Odometry modes: one VisualOdometryMono or
// VisualOdometryStereo per sequence, running on its sequence of the worker's batch; the GPU stages of the motion estimate
// are one batched call per worker.  Structure-from-motion modes: mono (mode 3) or stereo (mode 4) odometry as above, then
// what StructureFromMotion::update or StructureFromMotionStereo::update does per sequence, with the finished tracks of all
// of the worker's sequences evaluated by one device call.
namespace {
struct SfmState {                            // what the facades keep besides their odometry object (host/sfm.h)
  Reconstruction recon;                      // track bookkeeping; the points live in `store`
  visocu_recon_store* store = nullptr;       // on the worker's context, created by the sequence's first step
  Matrix Tr_total = Matrix::eye(4);
  bool first = true, replace = false;
};
struct Runner {
  int device, S, threads, mode, method;      // mode 0 = Matcher only, 1 = VisualOdometryMono::process, 2 = VisualOdometryStereo::process,
                                             // 3 = StructureFromMotion::update, 4 = StructureFromMotionStereo::update
  int bucket_max; float bucket_w, bucket_h;
  MonoParamsC params;
  StereoParamsC sparams;
  std::vector<MatcherBatch*> batches;        // one per worker
  std::vector<MonoAccess*> monos;            // one per sequence (modes 1 and 3)
  std::vector<VisualOdometryStereo*> stereos; // one per sequence (modes 2 and 4)
  std::vector<SfmState*> sfms;               // one per sequence (modes 3 and 4)
  std::vector<int32_t> last_matches, last_ok;
  bool started = false;                      // a step has run: the rectification is fixed
  // dense disparity (modes 2 and 4): while disp_on, per sequence a device map of the last step (null: none this step)
  bool disp_on = false;
  visocu_sgm_params disp_params{};
  std::vector<int16_t*> disp_buf;            // runner-owned, w x h int16 on the sequence's worker context
  std::vector<int32_t> disp_w, disp_h;
  std::vector<uint8_t> disp_valid;          // bytes, not bits: the workers write their own sequences concurrently
  Matcher& matcher_of(int seq) { return batches[seq % threads]->sequence(seq / threads); }
};

// StructureFromMotion::update (mode 3) or StructureFromMotionStereo::update (mode 4) after the odometry of one frame, for
// every sequence of worker `tid`: pose accumulation and Reconstruction::batchPrepareTracks for the sequences whose frame is
// ok, then ONE visocu_recon_update for all of them, which moves each sequence's stored points with its motion, evaluates
// the finished tracks and appends the kept points to the sequence's device store; a failed frame is replaced by the next
// push.  If the device call fails, the finished tracks of the step are lost and the step reports ok = 0 for those
// sequences (their pose has already advanced, as the facade's does on a successful frame).
void runner_sfm(Runner* r, int tid) {
  visocu_ctx* ctx = r->batches[tid]->context();
  std::vector<int> ids;
  std::vector<visocu_recon_job> jobs;
  std::vector<visocu_recon_store*> stores;
  std::vector<double> tr;
  for (int s = tid; s < r->S; s += r->threads) {
    SfmState& q = *r->sfms[s];
    VisualOdometry& vo = r->mode == 4 ? (VisualOdometry&)*r->stereos[s] : (VisualOdometry&)*r->monos[s];
    if (q.first) {
      q.first = false;
      if (visocu_recon_store_create(ctx, 0, &q.store) != VISOCU_OK) std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
      continue;
    }
    if (!r->last_ok[s]) { q.replace = true; continue; }
    const Matrix Tr = vo.getMotion();
    q.Tr_total = q.Tr_total * Matrix::inv(Tr);
    jobs.push_back(q.recon.batchPrepareTracks(vo.getMatches(), Tr, 0, 2, 30, 3));
    for (int i = 0; i < 3; i++) for (int k = 0; k < 4; k++) tr.push_back(Tr.val[i][k]);
    stores.push_back(q.store);
    ids.push_back(s);
    q.replace = false;
  }
  if (ids.empty()) return;
  const int nj = (int)ids.size();
  std::vector<const double*> trp(nj);
  for (int j = 0; j < nj; j++) trp[j] = &tr[12 * (size_t)j];
  visocu_set_lane(ctx, 4);                         // like the odometry calls: matching stays on lane 0
  const int rc = visocu_recon_update(ctx, nj, stores.data(), trp.data(), jobs.data(), 0, 0, 0);
  visocu_set_lane(ctx, 0);
  if (rc != VISOCU_OK) {
    // the finished tracks of this step are lost (batchPrepareTracks has dropped them): the step is reported as failed
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    for (int s : ids) r->last_ok[s] = 0;
  }
}

// Dense disparity of every sequence of worker `tid` with a stereo pair this step: ONE visocu_disparity on lane 5, which
// the odometry and reconstruction calls (lane 4) and the matching (lane 0) do not use, into the runner's device buffers.
// Only reads the frames: the odometry results of the step are the same with and without it.
void runner_disparity(Runner* r, int tid) {
  visocu_ctx* ctx = r->batches[tid]->context();
  std::vector<int32_t> left, right;
  std::vector<int16_t*> out;
  std::vector<int> ids;
  for (int s = tid; s < r->S; s += r->threads) {
    r->disp_valid[s] = 0;
    int32_t l, rt, w, h;
    if (!ctx || !r->matcher_of(s).stereoPair(&l, &rt, &w, &h)) continue;
    if (r->disp_buf[s] && (r->disp_w[s] != w || r->disp_h[s] != h)) { visocu_device_free(ctx, r->disp_buf[s]); r->disp_buf[s] = nullptr; }
    if (!r->disp_buf[s]) {
      void* p = nullptr;
      if (visocu_device_alloc(ctx, (size_t)w * h * sizeof(int16_t), &p) != VISOCU_OK) { std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl; continue; }
      r->disp_buf[s] = (int16_t*)p; r->disp_w[s] = w; r->disp_h[s] = h;
    }
    left.push_back(l); right.push_back(rt); out.push_back(r->disp_buf[s]); ids.push_back(s);
  }
  if (ids.empty()) return;
  visocu_set_lane(ctx, 5);
  const int rc = visocu_disparity(ctx, (int32_t)ids.size(), left.data(), right.data(), &r->disp_params, out.data(), 1);
  visocu_set_lane(ctx, 0);
  if (rc != VISOCU_OK) { std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl; return; }
  for (int s : ids) r->disp_valid[s] = 1;
}

// host stages that follow the matching of one frame for every sequence of worker `tid`: bucketing, and for the odometry
// mode normalisation, sample tables, ONE batched RANSAC call for all of the worker's sequences, pose
void runner_post(Runner* r, int tid, int bucket, int32_t* n_matches_out, int32_t* ok_out) {
  MatcherBatch* b = r->batches[tid];
  if (r->mode == 2 || r->mode == 4) {
    // bucketing and sample tables per sequence, then ONE device motion estimate for all of the worker's sequences
    std::vector<int> ids;
    std::vector<const visocu_pmatch*> ml;
    std::vector<int32_t> N;
    std::vector<const int32_t*> smp;
    for (int s = tid; s < r->S; s += r->threads) {
      const visocu_pmatch* m = 0; int32_t n = 0; const int32_t* sp = 0;
      r->last_ok[s] = 0;
      if (r->stereos[s]->batchPrepare(&m, &n, &sp)) { ids.push_back(s); ml.push_back(m); N.push_back(n); smp.push_back(sp); }
      r->last_matches[s] = r->stereos[s]->getNumberOfMatches();
    }
    if (!ids.empty()) {
      const int nj = (int)ids.size();
      std::vector<double> tr(6 * (size_t)nj);
      std::vector<int32_t> ok(nj);
      std::vector<std::vector<uint8_t> > masks(nj);
      std::vector<uint8_t*> mptr(nj);
      for (int j = 0; j < nj; j++) { masks[j].resize(N[j]); mptr[j] = masks[j].data(); }
      const StereoParamsC& q = r->sparams;
      const visocu_stereo_params sp = {q.f, q.cu, q.cv, q.base, q.inlier_threshold, q.ransac_iters, q.reweighting};
      visocu_ctx* ctx = b->context();
      visocu_set_lane(ctx, 4);                     // odometry calls run on their own lane, matching stays on lane 0
      const int rc = visocu_stereo_motion(ctx, nj, ml.data(), N.data(), smp.data(), &sp, tr.data(), ok.data(), mptr.data(), 0, 0, 0, 0);
      if (rc != VISOCU_OK) std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
      visocu_set_lane(ctx, 0);
      if (rc == VISOCU_OK)
        for (int j = 0; j < nj; j++) r->last_ok[ids[j]] = r->stereos[ids[j]]->batchFinish(&tr[6 * (size_t)j], ok[j], mptr[j]) ? 1 : 0;
    }
  } else if (r->mode == 1 || r->mode == 3) {
    std::vector<int> ids;
    std::vector<const float*> uv;
    std::vector<int32_t> N;
    std::vector<const int32_t*> smp;
    for (int s = tid; s < r->S; s += r->threads) {
      const float* u = 0; int32_t n = 0; const int32_t* sp = 0;
      r->last_ok[s] = 0;
      if (r->monos[s]->batchPrepare(&u, &n, &sp)) { ids.push_back(s); uv.push_back(u); N.push_back(n); smp.push_back(sp); }
      r->last_matches[s] = r->monos[s]->getNumberOfMatches();
    }
    if (!ids.empty()) {
      const int nj = (int)ids.size();
      std::vector<double> F(9 * (size_t)nj);
      std::vector<int32_t> ninl(nj), best(nj);
      std::vector<std::vector<uint8_t> > masks(nj);
      std::vector<uint8_t*> mptr(nj);
      for (int j = 0; j < nj; j++) { masks[j].resize(N[j]); mptr[j] = masks[j].data(); }
      visocu_ctx* ctx = b->context();
      const VisualOdometryMono::parameters mp = to_cpp(&r->params);
      if (visocu_ransac_F(ctx, nj, uv.data(), N.data(), smp.data(), mp.ransac_iters, mp.inlier_threshold, F.data(), mptr.data(),
                          ninl.data(), best.data(), 0, 0) == VISOCU_OK) {
        // pose recovery: the two GPU stages (four triangulations per sequence, ground-plane vote) as one batched call
        // each for all of the worker's sequences
        std::vector<int> alive;
        for (int j = 0; j < nj; j++)
          if (r->monos[ids[j]]->poseStageA(&F[9 * (size_t)j], mptr[j])) alive.push_back(ids[j]);
        if (!alive.empty()) {
          const int na = (int)alive.size();
          std::vector<const float*> tuv(na); std::vector<int32_t> tN(na), tsol(na, 4);
          std::vector<const double*> tP1(na), tP2(na); std::vector<double*> tX(na); std::vector<int32_t*> tfront(na);
          for (int a = 0; a < na; a++) {
            VisualOdometryMono::PoseRequest& q = r->monos[alive[a]]->poseRequest();
            tuv[a] = q.uv.data(); tN[a] = q.N; tP1[a] = q.P1; tP2[a] = q.P2; tX[a] = q.X.data(); tfront[a] = q.n_front;
          }
          std::vector<int> alive2;
          if (visocu_triangulate_batch(ctx, na, tuv.data(), tN.data(), tP1.data(), tP2.data(), tsol.data(), tX.data(), tfront.data()) == VISOCU_OK)
            for (int a = 0; a < na; a++)
              if (r->monos[alive[a]]->poseStageB()) alive2.push_back(alive[a]);
          if (!alive2.empty()) {
            const int nb = (int)alive2.size();
            std::vector<const double*> pd(nb); std::vector<int32_t> pn(nb), pbest(nb, 0); std::vector<double> pth(nb), pw(nb);
            for (int a = 0; a < nb; a++) {
              VisualOdometryMono::PoseRequest& q = r->monos[alive2[a]]->poseRequest();
              pd[a] = q.d.data(); pn[a] = (int32_t)q.d.size(); pth[a] = q.threshold; pw[a] = q.weight;
            }
            if (visocu_best_plane_batch(ctx, nb, pd.data(), pn.data(), pth.data(), pw.data(), pbest.data()) == VISOCU_OK)
              for (int a = 0; a < nb; a++) r->last_ok[alive2[a]] = r->monos[alive2[a]]->poseStageC(pbest[a]) ? 1 : 0;
          }
        }
      }
    }
  } else {
    int k = 0;
    for (int s = tid; s < r->S; s += r->threads, k++) {
      Matcher& m = b->sequence(k);
      if (bucket) m.bucketFeatures(r->bucket_max, r->bucket_w, r->bucket_h);
      r->last_matches[s] = (int32_t)m.matches(2).size();
      r->last_ok[s] = 1;
    }
  }
  if (r->mode == 3 || r->mode == 4) runner_sfm(r, tid);
  if (r->disp_on) runner_disparity(r, tid);
  for (int s = tid; s < r->S; s += r->threads) {
    if (n_matches_out) n_matches_out[s] = r->last_matches[s];
    if (ok_out) ok_out[s] = r->last_ok[s];
  }
}

void runner_push(Runner* r, int tid, const uint8_t* const* imgs, const uint8_t* const* imgs2, const int32_t* dims, int on_device) {
  uint32_t d[3] = {(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]};
  std::vector<const uint8_t*> i1, i2;
  for (int s = tid; s < r->S; s += r->threads) { i1.push_back(imgs[s]); if (imgs2) i2.push_back(imgs2[s]); }
  if (r->mode == 3 || r->mode == 4) {              // each sequence's replace flag, as the facades pass it
    std::unique_ptr<bool[]> replace(new bool[i1.size()]);
    size_t k = 0;
    for (int s = tid; s < r->S; s += r->threads) replace[k++] = r->sfms[s]->replace;
    r->batches[tid]->pushBack(i1.data(), r->mode == 4 ? i2.data() : 0, d, replace.get(), on_device != 0);
    return;
  }
  r->batches[tid]->pushBack(i1.data(), imgs2 ? i2.data() : 0, d, false, on_device != 0);
}

// Steps of modes 3 and 4 never take the pipelined path: a step's push needs the previous step's outcome (the replace flag).
bool runner_pipelined(Runner* r, int tid, const uint8_t* const* imgs2) {
  return !imgs2 && r->mode != 3 && r->mode != 4 && r->batches[tid]->stepAvailable(r->method);
}

// one frame for every sequence of worker `tid`, synchronously
void runner_advance(Runner* r, int tid, const uint8_t* const* imgs, const uint8_t* const* imgs2, const int32_t* dims, int on_device,
                    int bucket, int32_t* n_matches_out, int32_t* ok_out) {
  MatcherBatch* b = r->batches[tid];
  if (runner_pipelined(r, tid, imgs2)) {
    uint32_t d[3] = {(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]};
    std::vector<const uint8_t*> i1;
    for (int s = tid; s < r->S; s += r->threads) i1.push_back(imgs[s]);
    while (b->stepsInFlight() > 0) b->stepCollect();
    if (b->stepSubmit(i1.data(), d, on_device != 0)) b->stepCollect();
  } else {
    runner_push(r, tid, imgs, imgs2, dims, on_device);
    if (r->mode == 2 || r->mode == 4) {
      std::vector<const Matrix*> pred;                 // quad matching with each sequence's motion, as process() does
      for (int s = tid; s < r->S; s += r->threads) pred.push_back(r->stereos[s]->predictedMotion());
      b->matchFeatures(r->method, pred.data());
    } else {
      b->matchFeatures(r->method);
    }
  }
  runner_post(r, tid, bucket, n_matches_out, ok_out);
}

template <class F> void run_workers(int threads, F work) {
  if (threads == 1) { work(0); return; }
  std::vector<std::thread> pool;
  for (int t = 0; t < threads; t++) pool.emplace_back(work, t);
  for (std::thread& t : pool) t.join();
}
}  // namespace

namespace {
Runner* runner_new(int device, int n_sequences, int threads, int mode, int method, const Matcher::parameters& match) {
  Runner* r = new Runner();
  r->device = device; r->S = n_sequences; r->threads = std::max(1, std::min(threads, n_sequences)); r->mode = mode; r->method = method;
  visob::set_device(device);
  for (int t = 0; t < r->threads; t++) {
    int n = 0;
    for (int s = t; s < n_sequences; s += r->threads) n++;
    r->batches.push_back(new MatcherBatch(match, n));
  }
  r->last_matches.assign(n_sequences, 0);
  r->last_ok.assign(n_sequences, 0);
  return r;
}
}  // namespace

VISOB_API void* visob_runner_create(int device, int n_sequences, int threads, int mode, int method, const MonoParamsC* p) {
  Runner* r = runner_new(device, n_sequences, threads, mode, method, p->match);
  r->params = *p;
  r->bucket_max = p->bucket_max_features; r->bucket_w = (float)p->bucket_width; r->bucket_h = (float)p->bucket_height;
  if (mode == 1) {
    // one odometry object per sequence, running on its sequence of the worker's batch
    for (int s = 0; s < n_sequences; s++) {
      MonoAccess* vo = new MonoAccess(to_cpp(p));
      vo->adoptMatcher(&r->batches[s % r->threads]->sequence(s / r->threads));
      r->monos.push_back(vo);
    }
  }
  return r;
}
// Stereo odometry (mode 2): one VisualOdometryStereo per sequence.  A step pushes the left and right images of every
// sequence, runs quad matching with each sequence's previous motion where it has one, and per worker ONE
// visocu_stereo_motion for the sequences with enough matches; steps are synchronous (imgs2 is required).
VISOB_API void* visob_runner_create_stereo(int device, int n_sequences, int threads, const StereoParamsC* p) {
  Runner* r = runner_new(device, n_sequences, threads, 2, 2, p->match);
  r->sparams = *p;
  r->bucket_max = p->bucket_max_features; r->bucket_w = (float)p->bucket_width; r->bucket_h = (float)p->bucket_height;
  for (int s = 0; s < n_sequences; s++) {
    VisualOdometryStereo* vo = new VisualOdometryStereo(to_cpp(p));
    vo->adoptMatcher(&r->batches[s % r->threads]->sequence(s / r->threads));
    r->stereos.push_back(vo);
  }
  return r;
}
// Structure from motion (mode 3): per sequence what StructureFromMotion keeps - a VisualOdometryMono on its sequence of the
// worker's batch, the accumulated pose, the first-frame and replace flags and a Reconstruction with the facade's calibration
// and constants (point type 0, min track length 2, 30 m, 3 degrees).  A step pushes every sequence with its replace flag,
// runs flow matching and the mono odometry stages, and per worker ONE visocu_recon_update for the sequences whose frame is
// ok.  Each sequence's points stay in a device store on its worker's context.  Steps are synchronous.
VISOB_API void* visob_runner_create_sfm(int device, int n_sequences, int threads, const MonoParamsC* p) {
  Runner* r = (Runner*)visob_runner_create(device, n_sequences, threads, 1, 0, p);
  r->mode = 3;
  for (int s = 0; s < n_sequences; s++) {
    SfmState* q = new SfmState();
    q->recon.setCalibration(p->f, p->cu, p->cv);
    r->sfms.push_back(q);
  }
  return r;
}
// Stereo structure from motion (mode 4): per sequence a VisualOdometryStereo on its sequence of the worker's batch, as in
// mode 2, and what StructureFromMotionStereo keeps besides it, as in mode 3.  A step pushes the left and right images of
// every sequence with its replace flag, runs quad matching with each sequence's previous motion, per worker ONE
// visocu_stereo_motion and then ONE visocu_recon_update.  Steps are synchronous and need right images.
VISOB_API void* visob_runner_create_stereo_sfm(int device, int n_sequences, int threads, const StereoParamsC* p) {
  Runner* r = (Runner*)visob_runner_create_stereo(device, n_sequences, threads, p);
  r->mode = 4;
  for (int s = 0; s < n_sequences; s++) {
    SfmState* q = new SfmState();
    q->recon.setCalibration(p->f, p->cu, p->cv);
    r->sfms.push_back(q);
  }
  return r;
}
VISOB_API void visob_runner_destroy(void* h) {
  Runner* r = (Runner*)h;
  for (int s = 0; s < (int)r->disp_buf.size(); s++)
    if (r->disp_buf[s]) visocu_device_free(r->batches[s % r->threads]->context(), r->disp_buf[s]);
  for (int s = 0; s < (int)r->sfms.size(); s++) {
    if (r->sfms[s]->store) visocu_recon_store_destroy(r->batches[s % r->threads]->context(), r->sfms[s]->store);
    delete r->sfms[s];
  }
  for (MonoAccess* m : r->monos) delete m;
  for (VisualOdometryStereo* m : r->stereos) delete m;
  for (MatcherBatch* b : r->batches) delete b;
  delete r;
}
// imgs / imgs2: S pointers (imgs2 may be null for mono / flow).  on_device: pointers are device memory.
// bucket: apply bucketFeatures after matching (mode 0).  Returns wall seconds spent in the step; -1 for a mode-4 step
// without right images (nothing is pushed or written).
// Raw camera images for every mode: what setRectification does for each sequence's objects (MatcherBatch, the odometry's
// calibration, the reconstruction's projection).  Stereo modes (2, 4) need r->n_cams = 2.  1 = done; 0 = refused, with
// nothing changed: after the first step, or a rectification the mode cannot take.
VISOB_API int visob_runner_set_rectification(void* h, const Rectification* rc) {
  Runner* r = (Runner*)h;
  const bool stereo = r->mode == 2 || r->mode == 4;
  if (r->started || rc->n_cams < 0 || rc->n_cams > 2 || (stereo && rc->n_cams != 2)) return 0;
  for (MatcherBatch* b : r->batches) b->setRectification(*rc);
  for (MonoAccess* m : r->monos) m->setRectification(*rc);
  for (VisualOdometryStereo* m : r->stereos) m->setRectification(*rc);
  if (rc->n_cams > 0) {
    const visocu_camera& c = rc->cams[0];
    r->params.f = c.f; r->params.cu = c.cu; r->params.cv = c.cv;
    r->sparams.f = c.f; r->sparams.cu = c.cu; r->sparams.cv = c.cv;
    if (stereo) r->sparams.base = rc->base;
    for (SfmState* q : r->sfms) q->recon.setCalibration(c.f, c.cu, c.cv);
  }
  return 1;
}
// Dense disparity for the stereo modes (2, 4): with p, every following step computes each sequence's disparity map
// (visocu_disparity, one call per worker) into a device buffer of the runner; null turns it off.  1 = done, 0 = refused
// (another mode, or parameters outside the ranges of visocu_disparity).
VISOB_API int visob_runner_set_disparity(void* h, const visocu_sgm_params* p) {
  Runner* r = (Runner*)h;
  if (r->mode != 2 && r->mode != 4) return 0;
  if (!p) { r->disp_on = false; return 1; }
  if (visocu_sgm_check(p) != VISOCU_OK) return 0;
  r->disp_params = *p;
  r->disp_on = true;
  r->disp_buf.resize(r->S, nullptr); r->disp_w.resize(r->S, 0); r->disp_h.resize(r->S, 0); r->disp_valid.resize(r->S, 0);
  return 1;
}
// the sequence's disparity map of the last step in device memory (w x h int16, 1/16 pixel, -1 = invalid), valid until
// the next step: 0, or -1 when the feature is off, for another mode, a bad sequence or a step without a map
VISOB_API int visob_runner_device_disparity(void* h, int seq, const int16_t** d_map, int32_t* w, int32_t* ht) {
  Runner* r = (Runner*)h;
  if (!r->disp_on || seq < 0 || seq >= r->S || !d_map || !w || !ht || !r->disp_valid[seq]) return -1;
  *d_map = r->disp_buf[seq]; *w = r->disp_w[seq]; *ht = r->disp_h[seq];
  return 0;
}
VISOB_API double visob_runner_step(void* h, const uint8_t* const* imgs, const uint8_t* const* imgs2, const int32_t* dims,
                                   int on_device, int bucket, int32_t* n_matches_out, int32_t* ok_out) {
  Runner* r = (Runner*)h;
  if (r->mode == 4 && !imgs2) return -1.0;
  r->started = true;
  auto t0 = std::chrono::steady_clock::now();
  run_workers(r->threads, [&](int tid) {
    visob::set_device(r->device);
    runner_advance(r, tid, imgs, imgs2, dims, on_device, bucket, n_matches_out, ok_out);
  });
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}
// K steps without a barrier between them: worker t walks its sequences (t, t + threads, ...) through all K frames.
// imgs / imgs2: K x S pointers, step-major.  n_matches_out / ok_out (K x S, optional) receive per-pair results.  -1 as
// visob_runner_step.
VISOB_API double visob_runner_run(void* h, int n_steps, const uint8_t* const* imgs, const uint8_t* const* imgs2, const int32_t* dims,
                                  int on_device, int bucket, int32_t* n_matches_out, int32_t* ok_out) {
  Runner* r = (Runner*)h;
  if (r->mode == 4 && !imgs2) return -1.0;
  r->started = true;
  auto t0 = std::chrono::steady_clock::now();
  run_workers(r->threads, [&](int tid) {
    visob::set_device(r->device);
    MatcherBatch* b = r->batches[tid];
    if (!runner_pipelined(r, tid, imgs2)) {
      for (int k = 0; k < n_steps; k++)
        runner_advance(r, tid, imgs + (size_t)k * r->S, imgs2 ? imgs2 + (size_t)k * r->S : 0, dims, on_device, bucket,
                       n_matches_out ? n_matches_out + (size_t)k * r->S : 0, ok_out ? ok_out + (size_t)k * r->S : 0);
      return;
    }
    // Pipelined: up to `depth` steps of the worker's sequences are in flight.  Step k is submitted (push of frame k and
    // its matching against frame k - 1: one submission, replayed as a graph); then the oldest step is collected if the
    // window is full, and its host stages (bucketing, odometry) run while the GPU works on the younger steps.  Every
    // step's results are complete when the call returns.
    const int depth = visob::pipeline_depth();
    uint32_t d[3] = {(uint32_t)dims[0], (uint32_t)dims[1], (uint32_t)dims[2]};
    std::vector<const uint8_t*> i1;
    while (b->stepsInFlight() > 0) b->stepCollect();
    int collected = 0;
    auto collect_one = [&]() {
      b->stepCollect();
      runner_post(r, tid, bucket, n_matches_out ? n_matches_out + (size_t)collected * r->S : 0, ok_out ? ok_out + (size_t)collected * r->S : 0);
      collected++;
    };
    for (int k = 0; k < n_steps; k++) {
      i1.clear();
      for (int s = tid; s < r->S; s += r->threads) i1.push_back(imgs[(size_t)k * r->S + s]);
      if (!b->stepSubmit(i1.data(), d, on_device != 0)) break;
      if (b->stepsInFlight() >= depth) collect_one();
    }
    while (b->stepsInFlight() > 0) collect_one();
  });
  return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}
VISOB_API int visob_runner_get_matches(void* h, int seq, void* out, int cap) {
  Runner* r = (Runner*)h;
  if (seq < 0 || seq >= r->S) return -1;
  if (r->mode == 1 || r->mode == 3) return copy_matches(r->monos[seq]->usedMatches(), out, cap);
  if (r->mode == 2 || r->mode == 4) return copy_matches(r->stereos[seq]->usedMatches(), out, cap);
  return copy_matches(r->matcher_of(seq).matches(2), out, cap);
}
VISOB_API void visob_runner_get_motion(void* h, int seq, double* out16) {
  Runner* r = (Runner*)h;
  if (r->mode == 0 || seq < 0 || seq >= r->S) return;
  Matrix T = r->mode == 2 || r->mode == 4 ? r->stereos[seq]->getMotion() : r->monos[seq]->getMotion();
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) out16[4 * i + j] = T.val[i][j];
}
// inlier indices of the last motion estimate (odometry modes); -1 for mode 0 or a bad sequence
VISOB_API int visob_runner_get_inliers(void* h, int seq, int32_t* out, int cap) {
  Runner* r = (Runner*)h;
  if (r->mode == 0 || seq < 0 || seq >= r->S) return -1;
  std::vector<int32_t> in = r->mode == 2 || r->mode == 4 ? r->stereos[seq]->getInlierIndices() : r->monos[seq]->getInlierIndices();
  if (out) memcpy(out, in.data(), sizeof(int32_t) * (size_t)std::min((int)in.size(), cap));
  return (int)in.size();
}
// structure-from-motion modes (3 and 4): the sequence's reconstructed points (x, y, z per point; returns the count, -1 for
// another mode or a bad sequence) and its accumulated pose (first camera -> current camera)
VISOB_API int visob_runner_get_points(void* h, int seq, float* out3, int cap) {
  Runner* r = (Runner*)h;
  if ((r->mode != 3 && r->mode != 4) || seq < 0 || seq >= r->S) return -1;
  const visocu_recon_store* store = r->sfms[seq]->store;
  if (!store) return 0;
  const float* d = 0; int64_t n = 0;
  visocu_recon_store_points(store, &d, &n);
  const int64_t count = std::min<int64_t>(n, std::max(cap, 0));
  visocu_ctx* ctx = r->batches[seq % r->threads]->context();
  if (count > 0 && visocu_recon_store_read(ctx, store, 0, count, out3) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    return -1;
  }
  return (int)n;
}
// the same points in device memory of the runner's GPU (x, y, z floats per point), valid until the next step: 0, or -1 for
// another mode or a bad sequence; null and 0 before the sequence's first step
VISOB_API int visob_runner_device_points(void* h, int seq, const float** d_xyz, int64_t* n) {
  Runner* r = (Runner*)h;
  if ((r->mode != 3 && r->mode != 4) || seq < 0 || seq >= r->S || !d_xyz || !n) return -1;
  *d_xyz = 0; *n = 0;
  if (r->sfms[seq]->store) visocu_recon_store_points(r->sfms[seq]->store, d_xyz, n);
  return 0;
}
VISOB_API void visob_runner_get_pose(void* h, int seq, double* out16) {
  Runner* r = (Runner*)h;
  if ((r->mode != 3 && r->mode != 4) || seq < 0 || seq >= r->S) return;
  const Matrix& T = r->sfms[seq]->Tr_total;
  for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) out16[4 * i + j] = T.val[i][j];
}
VISOB_API void visob_runner_transfer_bytes(void* h, uint64_t* h2d, uint64_t* d2h) {
  Runner* r = (Runner*)h;
  uint64_t a = 0, b = 0, x = 0, y = 0;
  for (MatcherBatch* m : r->batches) if (m->context() && visocu_transfer_bytes(m->context(), &x, &y) == 0) { a += x; b += y; }
  *h2d = a; *d2h = b;
}
VISOB_API void visob_runner_outlier_stats(void* h, uint64_t* out8) {
  Runner* r = (Runner*)h;
  uint64_t one[8];
  for (int k = 0; k < 8; k++) out8[k] = 0;
  for (MatcherBatch* m : r->batches)
    if (m->context() && visocu_outlier_stats(m->context(), one) == 0)
      for (int k = 0; k < 8; k++) out8[k] += one[k];
}
VISOB_API void visob_runner_node_stats(void* h, uint64_t* out2) {
  Runner* r = (Runner*)h;
  uint64_t one[2];
  out2[0] = out2[1] = 0;
  for (MatcherBatch* m : r->batches)
    if (m->context() && visocu_node_stats(m->context(), one) == 0) { out2[0] += one[0]; out2[1] += one[1]; }
}
VISOB_API uint64_t visob_runner_launches(void* h) {
  Runner* r = (Runner*)h;
  uint64_t total = 0, n = 0;
  for (MatcherBatch* m : r->batches) if (m->context() && visocu_launch_count(m->context(), &n) == 0) total += n;
  return total;
}
