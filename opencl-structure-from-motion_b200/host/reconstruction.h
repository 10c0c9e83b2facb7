// Sparse 3-D reconstruction from monocular feature tracks, with the reference's interface
// (viso/reconstruction.h:40-67): feed it the flow matches of every frame pair and the egomotion, it links matches into
// tracks (via the feature indices i1p -> i1c), and when a track ends it triangulates the point, refines it by
// Gauss-Newton over all observations and keeps it if it passes the type / distance / ray-angle tests.
// Cost: every finished track needs a 4x4 SVD and up to 22 Gauss-Newton updates over as many as 6 observations; with
// 1 000 - 3 000 matches per frame that is milliseconds per update on one core.  update() runs it on the host; callers with
// many sequences split it: batchPrepare (the bookkeeping), ONE visocu_recon_points for the finished tracks of all of them
// (include/visocu.h), batchFinish (SURVEY.md 8f rank 4).  Callers that keep the points in device stores use
// batchPrepareTracks and ONE visocu_recon_update, which also moves the stored points and appends the kept ones.
// Own layout: frames carry absolute numbers instead of the reference's frames_ago counters and raw pointers; tracks
// live in a vector that is compacted in order, which preserves the reference's output order of points.
#ifndef VISOB_RECONSTRUCTION_H
#define VISOB_RECONSTRUCTION_H
#include <deque>
#include <vector>
#include "matcher.h"
#include "matrix.h"
#include "point3d.h"
#include "visocu.h"

Point3d affineTransform(const Matrix& M, const Point3d& p);      // rows 0..2 of M applied to (p, 1)  (matrix.cpp:37-44)

class Reconstruction {
public:
  Reconstruction();
  ~Reconstruction();

  // intrinsics (fu = fv = f); must be called once.  Also fixes the camera -> road transform used by the point types
  // (pitch -0.08 rad, height 1.6 m: reconstruction.cpp:37-48).
  void setCalibration(FLOAT f, FLOAT cu, FLOAT cv);

  // p_matched: flow matches of the newest frame pair; Tr: motion previous -> current camera coordinates.
  // point_type: 0 everything, 1 road and above, 2 only above the road; min_track_length in frames;
  // max_dist in metres from the camera; min_angle between the first and last viewing ray in degrees.
  void update(std::vector<Matcher::p_match> p_matched, Matrix Tr, int32_t point_type = 1, int32_t min_track_length = 2,
              double max_dist = 30, double min_angle = 2);

  // points of all finished tracks, in current camera coordinates
  const std::vector<Point3d>& getPoints() { return points; }

  // update() in two halves around the evaluation of the finished tracks.  batchPrepare does all of update()'s bookkeeping
  // (stored points moved into the new camera frame, frame window, tracks linked, tracks shorter than min_track_length
  // dropped) and returns the job of the tracks that ended with this frame, in order: the window's frame table (oldest first,
  // the newest camera last) and the tracks.  The job points into this object and stays valid until the next batchPrepare.
  // batchFinish takes its results (visocu_recon_points' status and xyz, or hostEval's) and appends the kept points.
  const visocu_recon_job& batchPrepare(const std::vector<Matcher::p_match>& p_matched, Matrix Tr, int32_t point_type = 1,
                                       int32_t min_track_length = 2, double max_dist = 30, double min_angle = 2);
  void batchFinish(const int32_t* status, const float* xyz);
  // batchPrepare without moving the stored points: for callers that keep the points elsewhere (a device store,
  // visocu_recon_update) and move them there with Tr.  batchPrepare is the move followed by this.
  const visocu_recon_job& batchPrepareTracks(const std::vector<Matcher::p_match>& p_matched, Matrix Tr, int32_t point_type = 1,
                                             int32_t min_track_length = 2, double max_dist = 30, double min_angle = 2);
  const visocu_recon_job& batchJob() const { return job; }
  // the host functions (initPoint, pointType, refinePoint, pointDistance, rayAngle) on every track of the prepared job
  void hostEval(int32_t* status, float* xyz) const;

private:
  struct Obs { float u, v; };
  struct Frame {
    Matrix fwd, inv, proj;      // frame -> current camera, its inverse, K * inv[0:3, 0:4]
    int64_t id;                 // absolute frame number
    int32_t track_count;        // live tracks that started here
  };
  struct Track {
    std::vector<Obs> pixels;
    int64_t first_id;
    int32_t last_idx;
    bool refreshed;
  };
  // A track anchored at frame U has 6 observations by update U + 4 and ends at U + 5 at the latest, and frames nobody's
  // track starts in are popped from the front first: the window never holds more than max_track_length frames.
  static const unsigned max_track_length = 6;

  Frame& frame(int64_t id) { return frames[(size_t)(id - frames.front().id)]; }
  // the host functions on one track of the prepared job (window indices: frame 0 = job.frames[0])
  bool initPoint(const visocu_recon_track& t, Point3d& p) const;
  bool refinePoint(const visocu_recon_track& t, Point3d& p) const;
  int32_t pointType(const visocu_recon_track& t, const Point3d& p) const;
  double pointDistance(const visocu_recon_track& t, const Point3d& p) const;
  double rayAngle(const visocu_recon_track& t, const Point3d& p) const;

  Matrix K, Tr_cam_road;
  std::vector<Track> tracks;
  std::vector<Point3d> points;
  std::deque<Frame> frames;
  int64_t next_id;
  // the prepared job: frame table, finished tracks, parameters
  std::vector<visocu_recon_frame> job_frames;
  std::vector<visocu_recon_track> job_tracks;
  visocu_recon_job job;
};
#endif
