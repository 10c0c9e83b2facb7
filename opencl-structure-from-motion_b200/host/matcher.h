// Matcher with the reference's public interface (viso/matcher.h:37-136): same parameters struct and defaults,
// same p_match layout, same pushBack / matchFeatures / bucketFeatures / getMatches / getGain signatures and
// error behaviour, so it is a drop-in for libviso2's feature front end.  What runs where:
//   GPU (through include/visocu.h): image copy into the 16-byte stride, half-resolution image, 5x5 filters,
//       both non-maximum-suppression passes, descriptors, bin index, SAD circle matching (flow and quad),
//       pixel and sub-pixel refinement.
//   host (this class): ring-buffer bookkeeping, computePriorStatistics, removeOutliers (own exact Delaunay
//       triangulation + support vote), bucketFeatures, getGain.
// The Tr_delta-guided search of quad matching (matcher.cpp:1112-1138) runs on the GPU as well.
#ifndef VISOB_MATCHER_H
#define VISOB_MATCHER_H
#include <stdint.h>
#include <stdlib.h>
#include <vector>

#include "matrix.h"
#include "rectify.h"
#include "visocu.h"

struct visocu_ctx;

class Matcher {
public:
  struct parameters {
    int32_t nms_n;                   // non-max-suppression: min. distance between maxima (in pixels)
    int32_t nms_tau;                 // non-max-suppression: interest point peakiness threshold
    int32_t match_binsize;           // matching bin width/height (affects efficiency only)
    int32_t match_radius;            // matching radius (du/dv in pixels)
    int32_t match_disp_tolerance;    // dv tolerance for stereo matches (in pixels)
    int32_t outlier_disp_tolerance;  // outlier removal: disparity tolerance (in pixels)
    int32_t outlier_flow_tolerance;  // outlier removal: flow tolerance (in pixels)
    int32_t multi_stage;             // 0=disabled,1=multistage matching (denser and faster)
    int32_t half_resolution;         // 0=disabled,1=match at half resolution, refine at full resolution
    int32_t refinement;              // refinement (0=none,1=pixel,2=subpixel)
    double f, cu, cv, base;          // calibration (only for match prediction)
    parameters() {
      nms_n = 3; nms_tau = 50; match_binsize = 50; match_radius = 200; match_disp_tolerance = 2;
      outlier_disp_tolerance = 5; outlier_flow_tolerance = 5; multi_stage = 1; half_resolution = 1; refinement = 1;
      f = 1; cu = 0; cv = 0; base = 1;
    }
  };

  Matcher(parameters param);
  ~Matcher();

  void setIntrinsics(double f, double cu, double cv, double base) {
    param.f = f; param.cu = cu; param.cv = cv; param.base = base;
  }

  struct p_match {
    float u1p, v1p; int32_t i1p;
    float u2p, v2p; int32_t i2p;
    float u1c, v1c; int32_t i1c;
    float u2c, v2c; int32_t i2c;
    p_match() {}
    p_match(float u1p, float v1p, int32_t i1p, float u2p, float v2p, int32_t i2p,
            float u1c, float v1c, int32_t i1c, float u2c, float v2c, int32_t i2c)
        : u1p(u1p), v1p(v1p), i1p(i1p), u2p(u2p), v2p(v2p), i2p(i2p),
          u1c(u1c), v1c(v1c), i1c(i1c), u2c(u2c), v2c(v2c), i2c(i2c) {}
  };

  // dims = {width, height, bytes per line}; the images are only read during the call
  void pushBack(uint8_t* I1, uint8_t* I2, uint32_t* dims, const bool replace);
  void pushBack(uint8_t* I1, uint32_t* dims, const bool replace) { pushBack(I1, 0, dims, replace); }
  // method: 0 = flow, 1 = stereo, 2 = quad matching
  void matchFeatures(int32_t method, Matrix* Tr_delta = 0);
  void bucketFeatures(int32_t max_features, float bucket_width, float bucket_height);
  std::vector<Matcher::p_match> getMatches() { return p_matched_2; }
  float getGain(std::vector<int32_t> inliers);

  // ---- extensions (not in the reference) ----
  // Raw camera images: after setRectification(r) with r.n_cams > 0, pushBack and pushBackDevice take images of
  // r.src_w x r.src_h (bytes per line >= r.src_w) and resample them on the GPU into r.out_w x r.out_h rectified images, the
  // left one with map 0 and the right one with map 1 (host/rectify.h); everything after the push sees the rectified
  // images.  r.n_cams = 0 returns to plain pushes.  Allowed before the first push only: afterwards it returns false and
  // changes nothing (as it does for more than 2 cameras).
  bool setRectification(const Rectification& r);
  // Dense disparity of the current stereo pair (left against right image of the last push, visocu_disparity): out
  // receives w x h int16 in 1/16 pixel (-1 = invalid), row stride w; host memory, or device memory of this matcher's GPU
  // with on_device.  False, with a message on cerr, after a mono push or when the device call fails.
  bool computeDisparity(const visocu_sgm_params& p, int16_t* out, bool on_device);
  // the device frames and the (rectified) size of the current stereo pair; false after a mono push or a failed one
  bool stereoPair(int32_t* left, int32_t* right, int32_t* w, int32_t* h) const;
  // same as pushBack, but the images already live in device memory of this matcher's GPU
  void pushBackDevice(const uint8_t* d_I1, const uint8_t* d_I2, uint32_t* dims, const bool replace);
  visocu_ctx* context() { return ctx; }
  // bucketFeatures shuffles with the same generator as the reference's std::random_shuffle (glibc rand()), but the
  // state is owned by this object: no process-wide lock, and sharded runs are reproducible.  Default state = rand()
  // without srand; VisualOdometry reseeds with 0 exactly where the reference calls srand(0) (viso.cpp:35).
  void seedShuffle(unsigned seed);
  // stage access for parity tests: 1 = pass-1 list after removeOutliers, 2 = getMatches()
  const std::vector<p_match>& matches(int stage) const { return stage == 1 ? p_matched_1 : p_matched_2; }
  int32_t featureCount(int which) { syncCounts(); return which >= 0 && which < 8 ? n_feat[which] : 0; }   // 1p1 2p1 1c1 2c1 1p2 2p2 1c2 2c2
  // host stages, usable on their own (used by the batch runner and the tests)
  struct range { float u_min[4], u_max[4], v_min[4], v_max[4]; };
  void computePriorStatistics(std::vector<p_match>& p_matched, int32_t method);
  void removeOutliers(std::vector<p_match>& p_matched, int32_t method);
  const std::vector<range>& priorRanges() const { return ranges; }

private:
  friend class MatcherBatch;
  void push(const uint8_t* I1, const uint8_t* I2, uint32_t* dims, bool replace, bool on_device);
  // stage functions shared by the stand-alone path and MatcherBatch
  void useSharedContext(visocu_ctx* shared, int32_t first_frame, int32_t w, int32_t h);
  bool pushPrepare(const uint8_t* I1, const uint8_t* I2, uint32_t* dims, bool replace, int32_t* frames);
  void pushFinish(bool ok, bool stereo, const int32_t* ns, const int32_t* nd);
  bool matchBegin(int32_t method);
  void matchAfterPass1(int32_t method);
  void matchAfterPass2(int32_t method);
  int refineMode() const;
  bool lazyCounts() const;               // push without reading the record counts back (n_feat = -1 until somebody needs them)
  void syncCounts();
  int32_t queryCount(int pass, int32_t method) const;
  bool ensureContext(int32_t w, int32_t h);
  // with rectification: dims must be the raw size (else false, with the reference's message); out = the output dims
  bool rectifiedDims(const uint32_t* dims, uint32_t* out) const;
  bool fetchImage(int which, std::vector<uint8_t>& out);
  bool matching(int pass, std::vector<p_match>& out, int32_t method, bool use_prior, int refine);
  // both passes of multi-stage flow matching as one submission (visocu_match_fused) for a group of matchers on one context
  static bool fusedAvailable(const Matcher& m, int32_t method);
  static void fusedMatch(visocu_ctx* ctx, const std::vector<Matcher*>& group, int32_t method);
  static void takeFused(Matcher* m, bool ok, const int32_t* counts, const visocu_pmatch* l1, int32_t n1, int32_t d1,
                        const visocu_pmatch* l2, int32_t n2, int32_t d2, int32_t method, int compact);

  parameters param;
  int32_t margin;
  visocu_ctx* ctx;
  bool owns_ctx;
  int32_t slot_base;                     // first device frame of this matcher inside its context
  int device;
  int32_t cfg_w, cfg_h;
  Rectification rect;                    // rect.n_cams = 0: plain pushes
  bool started;                          // a push has been prepared: the rectification is fixed
  // ring buffer: frame slots of the context.  slot[0] = previous left, [1] = previous right, [2] = current left,
  // [3] = current right (-1 = empty)
  int32_t slot[4];
  int32_t n_feat[8];
  int32_t dims_p[3], dims_c[3];
  std::vector<uint8_t> I1p, I1c;         // host copies for getGain (matcher.cpp:286-324), fetched from the device lazily
  bool have_I1p, have_I1c;
  std::vector<p_match> p_matched_1, p_matched_2;
  std::vector<range> ranges;
  bool has_tr;
  bool ro_done[2];                  // removeOutliers of the pass already ran on the device
  double tr_rows[12];
  struct random_data rnd_data;
  char rnd_state[128];
};

// Extension (not in the reference): S independent sequences that share one context, so that every GPU stage is ONE
// batched launch for all of them.  sequence(i) is an ordinary Matcher (bucketFeatures, getMatches, getGain ...); do
// not call its pushBack / matchFeatures directly.
class MatcherBatch {
public:
  MatcherBatch(Matcher::parameters param, int32_t n_sequences);
  ~MatcherBatch();
  // one image (and optionally one right image) per sequence; dims as for Matcher::pushBack
  void pushBack(const uint8_t* const* I1, const uint8_t* const* I2, uint32_t* dims, bool replace, bool on_device = false);
  // the same with a replace flag per sequence (Matcher::pushBack's replace: the new image takes the place of the current one)
  void pushBack(const uint8_t* const* I1, const uint8_t* const* I2, uint32_t* dims, const bool* replace, bool on_device);
  // tr_delta (optional, one entry per sequence, null = no prediction): the previous motion of each sequence for the
  // motion-predicted quad search, as Matcher::matchFeatures(2, Tr_delta).  The sequences share one calibration (setIntrinsics).
  void matchFeatures(int32_t method, const Matrix* const* tr_delta = nullptr);
  // Pipelined stepping for callers that walk many frames (the sequence runner): stepSubmit pushes one new frame per sequence
  // and enqueues its flow matching against the previous frame - one submission, nothing is waited for -, stepCollect waits
  // for the OLDEST submitted step and puts its matches into the sequences (getMatches, bucketFeatures ... then refer to that
  // step).  Up to three steps may be in flight: consecutive steps use different lanes of the context and a ring of four
  // frames per sequence, and a step that repeats is replayed as a CUDA graph.  Host images of a step must stay valid and
  // unchanged until that step has been collected (pinned ones are copied asynchronously).  Do not mix with pushBack /
  // matchFeatures.
  bool stepAvailable(int32_t method) const;
  bool stepSubmit(const uint8_t* const* I1, uint32_t* dims, bool on_device);
  bool stepCollect();
  // Matcher::setRectification for all sequences (the shared context holds the maps): before the first push or step only
  bool setRectification(const Rectification& r);
  int32_t stepsInFlight() const { return (int32_t)(k_submit - k_collect); }
  int32_t size() const { return (int32_t)seq.size(); }
  Matcher& sequence(int32_t i) { return *seq[i]; }
  visocu_ctx* context() { return ctx; }

private:
  bool ensure(int32_t w, int32_t h);
  bool matchPass(const std::vector<int32_t>& active, int pass, int32_t method, bool use_prior, int refine);
  int32_t step_dims[3];
  Rectification rect;
  bool started;
  int64_t k_submit, k_collect;                          // steps submitted / collected so far (stepSubmit / stepCollect)
  std::vector<Matcher*> seq;
  visocu_ctx* ctx;
  int device;
  int32_t width, height;
};

#endif
