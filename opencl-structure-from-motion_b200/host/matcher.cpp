// Host side of the feature front end.  See matcher.h for the split between GPU and host work.
// Reference behaviour restated here (paths relative to /root/reference/viso):
//   constructor ........................ matcher.cpp:38-62     pushBack ............ matcher.cpp:95-181
//   matchFeatures ...................... matcher.cpp:183-241   bucketFeatures ...... matcher.cpp:243-284
//   getGain ............................ matcher.cpp:286-324   computePriorStatistics matcher.cpp:734-868
//   removeOutliers ..................... matcher.cpp:1207-1377
#include "matcher.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <memory>

#include "delaunay.h"
#include "device.h"
#include "visocu.h"

using std::vector;

namespace visob {
// optional per-stage wall-clock accounting of the host layer (bench.py --host-timing); seconds, summed over threads
std::atomic<long long> g_stage_ns[8];
std::atomic<long long> g_stage_calls[8];
struct StageTimer {
  int id; std::chrono::steady_clock::time_point t0;
  explicit StageTimer(int id) : id(id), t0(std::chrono::steady_clock::now()) {}
  ~StageTimer() {
    g_stage_ns[id] += std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
    g_stage_calls[id]++;
  }
};
// Matcher::removeOutliers runs on the device behind the matching kernels unless VISOB_HOST_OUTLIERS=1 (the host
// implementation in delaunay.cpp stays the path for lists the device declines: too long, or duplicate positions)
bool device_outliers() {
  static const bool on = [] { const char* e = getenv("VISOB_HOST_OUTLIERS"); return !(e && e[0] == '1'); }();
  return on;
}
static std::atomic<int> g_depth(-1);
void set_pipeline_depth(int depth) { g_depth = depth < 1 ? 1 : (depth > 3 ? 3 : depth); }
int pipeline_depth() {
  int v = g_depth.load();
  if (v < 0) { const char* e = getenv("VISOB_DEPTH"); v = e ? atoi(e) : 3; v = v < 1 ? 1 : (v > 3 ? 3 : v); g_depth = v; }
  return v;
}
static thread_local int t_device = 0;
void set_device(int device) { t_device = device; }
int current_device() { return t_device; }
}  // namespace visob

static_assert(sizeof(Matcher::p_match) == sizeof(visocu_pmatch), "p_match layout");
static_assert(sizeof(Matcher::range) == sizeof(visocu_range), "range layout");
static_assert(sizeof(Matcher::parameters) == sizeof(visocu_params), "parameters layout");

Matcher::Matcher(parameters param) : param(param), ctx(0), owns_ctx(true), slot_base(0), cfg_w(0), cfg_h(0), have_I1p(false), have_I1c(false), has_tr(false) {
  ro_done[0] = ro_done[1] = false;
  margin = 5 + 1;
  if (param.half_resolution) this->param.match_radius /= 2;     // matcher.cpp:59-60
  device = visob::current_device();
  for (int k = 0; k < 4; k++) slot[k] = -1;
  for (int k = 0; k < 8; k++) n_feat[k] = 0;
  for (int k = 0; k < 3; k++) dims_p[k] = dims_c[k] = 0;
  memset(&rect, 0, sizeof rect);
  started = false;
  memset(&rnd_data, 0, sizeof rnd_data);
  memset(rnd_state, 0, sizeof rnd_state);
  initstate_r(1, rnd_state, sizeof rnd_state, &rnd_data);     // the state rand() starts from
}

void Matcher::seedShuffle(unsigned seed) { srandom_r(seed, &rnd_data); }

bool Matcher::lazyCounts() const {
  static const bool on = [] { const char* e = getenv("VISOB_LAZY"); return !(e && e[0] == '0'); }();
  static const bool fused = [] { const char* e = getenv("VISOB_FUSED"); return !(e && e[0] == '0'); }();
  return on && fused && param.multi_stage && refineMode() != 2 && visob::device_outliers();
}

// record counts that were not read back at push time (-1): fetch them from the device
void Matcher::syncCounts() {
  int32_t frames[4], which[4], n = 0;
  for (int k = 0; k < 4; k++)
    if (slot[k] >= 0 && (n_feat[k] < 0 || n_feat[4 + k] < 0)) { frames[n] = slot[k]; which[n] = k; n++; }
  if (n == 0 || !ctx) return;
  int32_t ns[4], nd[4];
  if (visocu_frame_counts(ctx, n, frames, ns, nd) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    for (int i = 0; i < n; i++) { ns[i] = 0; nd[i] = 0; }
  }
  for (int i = 0; i < n; i++) { n_feat[which[i]] = ns[i]; n_feat[4 + which[i]] = nd[i]; }
}

Matcher::~Matcher() {
  if (ctx && owns_ctx) visocu_destroy(ctx);
}

void Matcher::useSharedContext(visocu_ctx* shared, int32_t first_frame, int32_t w, int32_t h) {
  if (ctx && owns_ctx) visocu_destroy(ctx);
  ctx = shared; owns_ctx = false; slot_base = first_frame; cfg_w = w; cfg_h = h;
  for (int k = 0; k < 4; k++) slot[k] = -1;
  for (int k = 0; k < 8; k++) n_feat[k] = 0;
}

bool Matcher::ensureContext(int32_t w, int32_t h) {
  if (!owns_ctx) {
    if (w == cfg_w && h == cfg_h) return true;
    std::cerr << "ERROR: Image dimension mismatch!" << std::endl;      // a shared context is configured once for one image size
    return false;
  }
  if (!ctx) {
    if (visocu_create(device, &ctx) != VISOCU_OK) {
      std::cerr << "ERROR: " << visocu_last_error(0) << std::endl;
      ctx = 0;
      return false;
    }
  }
  if (w != cfg_w || h != cfg_h) {
    visocu_params vp;
    memcpy(&vp, &param, sizeof vp);
    if (visocu_configure(ctx, &vp, w, h, 4) != VISOCU_OK) {
      std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
      return false;
    }
    if (rect.n_cams > 0 && visocu_set_rectification(ctx, rect.n_cams, rect.cams, rect.src_w, rect.src_h) != VISOCU_OK) {
      std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
      return false;
    }
    cfg_w = w; cfg_h = h;
    for (int k = 0; k < 4; k++) slot[k] = -1;        // features of another image size cannot be matched
    for (int k = 0; k < 8; k++) n_feat[k] = 0;
    have_I1p = have_I1c = false;
  }
  return true;
}

bool Matcher::setRectification(const Rectification& r) {
  if (started || r.n_cams < 0 || r.n_cams > 2) return false;
  rect = r;
  cfg_w = cfg_h = 0;                                 // the next push configures the context and sets the maps
  return true;
}

bool Matcher::rectifiedDims(const uint32_t* dims, uint32_t* out) const {
  if ((int32_t)dims[0] != rect.src_w || (int32_t)dims[1] != rect.src_h || (int32_t)dims[2] < rect.src_w) {
    std::cerr << "ERROR: Image dimension mismatch!" << std::endl;
    return false;
  }
  out[0] = (uint32_t)rect.out_w; out[1] = (uint32_t)rect.out_h; out[2] = (uint32_t)rect.out_w;
  return true;
}

void Matcher::pushBack(uint8_t* I1, uint8_t* I2, uint32_t* dims, const bool replace) { push(I1, I2, dims, replace, false); }
void Matcher::pushBackDevice(const uint8_t* d_I1, const uint8_t* d_I2, uint32_t* dims, const bool replace) { push(d_I1, d_I2, dims, replace, true); }

void Matcher::push(const uint8_t* I1, const uint8_t* I2, uint32_t* dims, bool replace, bool on_device) {
  visob::StageTimer timer(0);
  int32_t frames[2];
  uint32_t od[3];
  const bool rectify = rect.n_cams > 0;
  if (rectify && !rectifiedDims(dims, od)) return;
  if (!pushPrepare(I1, I2, rectify ? od : dims, replace, frames)) return;
  const uint8_t* imgs[2] = {I1, I2};
  const int32_t cams[2] = {0, 1};
  int32_t ns[2] = {-1, -1}, nd[2] = {-1, -1};
  const int nimg = I2 ? 2 : 1;
  // flow matching of a monocular sequence goes through the fused call, which needs no record counts on the host: the
  // push then returns without waiting for the GPU (the counts are fetched lazily if somebody asks, syncCounts)
  const bool lazy = lazyCounts() && !I2;
  const int32_t bpl = (int32_t)dims[2], where = on_device ? 1 : 0;
  const bool ok = (rectify ? visocu_push_frames_rectified(ctx, nimg, frames, imgs, cams, bpl, where, lazy ? 0 : ns, lazy ? 0 : nd)
                           : visocu_push_frames(ctx, nimg, frames, imgs, bpl, where, lazy ? 0 : ns, lazy ? 0 : nd)) == VISOCU_OK;
  if (!ok) std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
  pushFinish(ok, I2 != 0, ns, nd);
}

// ring-buffer bookkeeping of pushBack (matcher.cpp:108-160); frames[] receives the device frames of the new images
bool Matcher::pushPrepare(const uint8_t* I1, const uint8_t* I2, uint32_t* dims, bool replace, int32_t* frames) {
  const int32_t width = dims[0], height = dims[1], bpl = dims[2];
  if (width <= 0 || height <= 0 || bpl < width || I1 == 0) {
    std::cerr << "ERROR: Image dimension mismatch!" << std::endl;
    return false;
  }
  if (!ensureContext(width, height)) return false;
  started = true;
  if (!replace) {
    // current -> previous: the device frames swap roles, nothing is copied
    std::swap(slot[0], slot[2]);
    std::swap(slot[1], slot[3]);
    for (int k = 0; k < 2; k++) { n_feat[0 + k] = n_feat[2 + k]; n_feat[4 + k] = n_feat[6 + k]; }
    I1p.swap(I1c);
    have_I1p = have_I1c;
    for (int k = 0; k < 3; k++) dims_p[k] = dims_c[k];
  }
  dims_c[0] = width; dims_c[1] = height; dims_c[2] = width + 15 - (width - 1) % 16;
  // pick device frames for the new current images: reuse the ones just vacated (or never used)
  bool used[4] = {false, false, false, false};
  if (slot[0] >= 0) used[slot[0] - slot_base] = true;
  if (slot[1] >= 0) used[slot[1] - slot_base] = true;
  int32_t fresh[2], nf = 0;
  for (int k = 0; k < 4 && nf < 2; k++) if (!used[k]) fresh[nf++] = slot_base + k;
  slot[2] = fresh[0];
  slot[3] = I2 ? fresh[1] : -1;
  frames[0] = slot[2]; frames[1] = slot[3];
  return true;
}

void Matcher::pushFinish(bool ok, bool stereo, const int32_t* ns, const int32_t* nd) {
  if (!ok) {
    slot[2] = slot[3] = -1;
    n_feat[2] = n_feat[3] = n_feat[6] = n_feat[7] = 0;
    return;
  }
  n_feat[2] = ns[0]; n_feat[6] = nd[0];
  n_feat[3] = stereo ? ns[1] : 0; n_feat[7] = stereo ? nd[1] : 0;
  // getGain needs the two left images on the host (matcher.cpp:286-324); they are fetched from the device on demand
  have_I1c = false;
}

bool Matcher::stereoPair(int32_t* left, int32_t* right, int32_t* w, int32_t* h) const {
  if (!ctx || slot[2] < 0 || slot[3] < 0) return false;
  *left = slot[2]; *right = slot[3]; *w = cfg_w; *h = cfg_h;
  return true;
}

bool Matcher::computeDisparity(const visocu_sgm_params& p, int16_t* out, bool on_device) {
  int32_t l, r, w, h;
  if (!stereoPair(&l, &r, &w, &h)) {
    std::cerr << "ERROR: computeDisparity needs a stereo pair (the last push was mono or failed)" << std::endl;
    return false;
  }
  if (visocu_disparity(ctx, 1, &l, &r, &p, &out, on_device ? 1 : 0) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    return false;
  }
  return true;
}

// padded copy of a left image (previous or current) from the device frame it lives in
bool Matcher::fetchImage(int which, vector<uint8_t>& out) {
  const int32_t f = slot[which];
  if (f < 0 || !ctx) return false;
  int32_t d3[3];
  if (visocu_get_plane(ctx, f, 4, 0, 0, d3) != VISOCU_OK) return false;
  out.resize((size_t)d3[2] * d3[1]);
  return visocu_get_plane(ctx, f, 4, out.data(), out.size(), d3) == VISOCU_OK;
}

bool Matcher::matching(int pass, vector<p_match>& out, int32_t method, bool use_prior, int refine) {
  visob::StageTimer timer(1 + pass);
  visocu_quad q = {slot[0], slot[1], slot[2], slot[3]};
  const int32_t nq = queryCount(pass, method);
  out.resize((size_t)nq + 1);
  visocu_pmatch* optr = reinterpret_cast<visocu_pmatch*>(out.data());
  const visocu_range* rptr = reinterpret_cast<const visocu_range*>(ranges.data());
  int32_t cap = nq + 1, n = 0;
  const double* tptr = tr_rows;
  int32_t done = 0;
  int rc = visocu_match(ctx, 1, &q, method, pass, use_prior ? 1 : 0, use_prior ? &rptr : 0, (has_tr && method == 2) ? &tptr : 0, refine,
                        &optr, &cap, &n, visob::device_outliers() ? &done : 0);
  ro_done[pass] = done != 0;
  if (rc != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    out.clear();
    return false;
  }
  out.resize(n);
  return true;
}

void Matcher::matchFeatures(int32_t method, Matrix* Tr_delta) {
  has_tr = false;
  if (!fusedAvailable(*this, method)) syncCounts();
  if (!matchBegin(method)) return;
  // motion-predicted search (quad matching only, matcher.cpp:1112-1138): rows 0..2 of Tr_delta go to the kernel
  if (Tr_delta && method == 2 && Tr_delta->m >= 3 && Tr_delta->n >= 4) {
    has_tr = true;
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 4; c++) tr_rows[4 * r + c] = Tr_delta->val[r][c];
    visocu_params vp;
    memcpy(&vp, &param, sizeof vp);
    visocu_set_intrinsics(ctx, vp.f, vp.cu, vp.cv, vp.base);      // setIntrinsics may have been called after the first push
  }
  const int refine = refineMode();
  if (fusedAvailable(*this, method)) {
    fusedMatch(ctx, vector<Matcher*>(1, this), method);
    return;
  }
  p_matched_1.clear();
  p_matched_2.clear();
  if (param.multi_stage) {
    if (!matching(0, p_matched_1, method, false, 0)) return;
    matchAfterPass1(method);
    if (!matching(1, p_matched_2, method, true, refine)) return;
  } else {
    if (!matching(1, p_matched_2, method, false, refine)) return;
  }
  matchAfterPass2(method);
}

// Flow matching with both passes, the outlier removal of both and the prior statistics in between on the device, one
// submission and one wait per call.  VISOB_FUSED=0 keeps the pass-by-pass path (host prior statistics).
bool Matcher::fusedAvailable(const Matcher& m, int32_t method) {
  static const bool on = [] { const char* e = getenv("VISOB_FUSED"); return !(e && e[0] == '0'); }();
  return on && method == 0 && m.param.multi_stage && m.refineMode() != 2 && visob::device_outliers() && !m.has_tr;
}

void Matcher::fusedMatch(visocu_ctx* ctx, const vector<Matcher*>& group, int32_t method) {
  visob::StageTimer timer(2);
  const size_t n = group.size();
  vector<visocu_quad> quads(n);
  vector<const visocu_pmatch*> l1(n), l2(n);
  vector<visocu_range*> rp(n);
  vector<int32_t> n1(n, 0), n2(n, 0), d1(n, 0), d2(n, 0), counts(4 * n, 0);
  for (size_t k = 0; k < n; k++) {
    Matcher* m = group[k];
    quads[k] = visocu_quad{m->slot[0], m->slot[1], m->slot[2], m->slot[3]};
    const float bs = (float)m->param.match_binsize;
    const size_t nbin = (size_t)ceil((float)m->dims_c[0] / bs) * (size_t)ceil((float)m->dims_c[1] / bs);
    m->ranges.resize(nbin);
    rp[k] = reinterpret_cast<visocu_range*>(m->ranges.data());
  }
  int32_t compact = 0;
  const int rc = visocu_match_fused(ctx, (int32_t)n, quads.data(), group[0]->refineMode(), l1.data(), n1.data(), d1.data(),
                                    l2.data(), n2.data(), d2.data(), rp.data(), counts.data(), &compact);
  if (rc != VISOCU_OK) std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
  for (size_t k = 0; k < n; k++) takeFused(group[k], rc == VISOCU_OK, &counts[4 * k], l1[k], n1[k], d1[k], l2[k], n2[k], d2[k], method, compact);
}

// results of a fused call for one matcher
void Matcher::takeFused(Matcher* m, bool ok, const int32_t* counts, const visocu_pmatch* l1, int32_t n1, int32_t d1,
                        const visocu_pmatch* l2, int32_t n2, int32_t d2, int32_t method, int compact) {
  if (!ok) { m->p_matched_1.clear(); m->p_matched_2.clear(); m->ro_done[0] = m->ro_done[1] = false; return; }
  // the record counts arrive with the results (the frames were pushed without reading them back)
  m->n_feat[0] = counts[0]; m->n_feat[4] = counts[1];
  m->n_feat[2] = counts[2]; m->n_feat[6] = counts[3];
  // the reference returns from matchFeatures without touching its match lists if a needed feature set is empty
  // (matcher.cpp:190-212); the kernels matched nothing in that case
  if (m->n_feat[0] == 0 || m->n_feat[2] == 0 || m->n_feat[4] == 0 || m->n_feat[6] == 0) return;
  const p_match* a1 = reinterpret_cast<const p_match*>(l1);
  const p_match* a2 = reinterpret_cast<const p_match*>(l2);
  if (a1) m->p_matched_1.assign(a1, a1 + n1); else m->p_matched_1.clear();     // not delivered (sequence runner): nobody reads it
  if (compact == 0) {
    m->p_matched_2.assign(a2, a2 + n2);
  } else if (compact == 2) {
    // three words per match: whole-pixel coordinates and feature indices in 16 bits each
    const uint32_t* h = reinterpret_cast<const uint32_t*>(l2);
    m->p_matched_2.resize((size_t)n2);
    for (int32_t i = 0; i < n2; i++) {
      p_match& o = m->p_matched_2[i];
      const uint32_t a = h[3 * i], b = h[3 * i + 1], c = h[3 * i + 2];
      o.u1p = (float)(a & 0xFFFFu); o.v1p = (float)(a >> 16); o.i1p = (int32_t)(c & 0xFFFFu);
      o.u2p = -1; o.v2p = -1; o.i2p = -1;
      o.u1c = (float)(b & 0xFFFFu); o.v1c = (float)(b >> 16); o.i1c = (int32_t)(c >> 16);
      o.u2c = -1; o.v2c = -1; o.i2c = -1;
    }
  } else {
    // six words per flow match crossed PCIe: (u1p, v1p, i1p, u1c, v1c, i1c); the fields of the right images are -1
    struct Half { float u, v; int32_t i; };
    const Half* h = reinterpret_cast<const Half*>(l2);
    m->p_matched_2.resize((size_t)n2);
    for (int32_t i = 0; i < n2; i++) {
      p_match& o = m->p_matched_2[i];
      o.u1p = h[2 * i].u; o.v1p = h[2 * i].v; o.i1p = h[2 * i].i;
      o.u2p = -1; o.v2p = -1; o.i2p = -1;
      o.u1c = h[2 * i + 1].u; o.v1c = h[2 * i + 1].v; o.i1c = h[2 * i + 1].i;
      o.u2c = -1; o.v2c = -1; o.i2c = -1;
    }
  }
  m->ro_done[0] = d1 != 0;
  m->ro_done[1] = d2 != 0;
  if (!m->ro_done[0]) {
    // the device declined the first list (too long, degenerate): the second pass ran on ranges of nothing - redo it
    // pass by pass for this matcher
    m->matchAfterPass1(method);
    if (!m->matching(1, m->p_matched_2, method, true, m->refineMode())) return;
  }
  m->matchAfterPass2(method);
}

// sanity checks of matcher.cpp:190-212: silently keep the old matches if a needed set is empty
bool Matcher::matchBegin(int32_t method) {
  const int32_t* n1 = n_feat;       // sparse: 1p 2p 1c 2c
  const int32_t* n2 = n_feat + 4;   // dense
  if (method == 0) {
    if (n2[0] == 0 || n2[2] == 0) return false;
    if (param.multi_stage && (n1[0] == 0 || n1[2] == 0)) return false;
  } else if (method == 1) {
    if (n2[2] == 0 || n2[3] == 0) return false;
    if (param.multi_stage && (n1[2] == 0 || n1[3] == 0)) return false;
  } else {
    if (n2[0] == 0 || n2[1] == 0 || n2[2] == 0 || n2[3] == 0) return false;
    if (param.multi_stage && (n1[0] == 0 || n1[1] == 0 || n1[2] == 0 || n1[3] == 0)) return false;
  }
  return true;
}

int Matcher::refineMode() const { return param.refinement <= 0 ? 0 : (param.refinement == 1 ? 1 : 2); }

int32_t Matcher::queryCount(int pass, int32_t method) const {
  const int32_t base = pass == 0 ? 0 : 4;
  return method == 2 ? n_feat[base + 0] : n_feat[base + 2];
}

// host stages between the two matching passes (matcher.cpp:223-226) and after the second (matcher.cpp:232)
void Matcher::matchAfterPass1(int32_t method) {
  if (!ro_done[0]) removeOutliers(p_matched_1, method);
  computePriorStatistics(p_matched_1, method);
}
void Matcher::matchAfterPass2(int32_t method) {
  if (!ro_done[1]) removeOutliers(p_matched_2, method);
}

void Matcher::bucketFeatures(int32_t max_features, float bucket_width, float bucket_height) {
  float u_max = 0, v_max = 0;
  for (const p_match& m : p_matched_2) {
    if (m.u1c > u_max) u_max = m.u1c;
    if (m.v1c > v_max) v_max = m.v1c;
  }
  const int32_t cols = (int32_t)floor(u_max / bucket_width) + 1, rows = (int32_t)floor(v_max / bucket_height) + 1;
  vector<vector<p_match> > buckets((size_t)cols * rows);
  for (const p_match& m : p_matched_2) {
    const int32_t u = (int32_t)floor(m.u1c / bucket_width), v = (int32_t)floor(m.v1c / bucket_height);
    buckets[(size_t)v * cols + u].push_back(m);
  }
  p_matched_2.clear();
  for (vector<p_match>& b : buckets) {
    // std::random_shuffle of the reference (matcher.cpp:270) restated: libstdc++ swaps element i with element
    // rand() % (i + 1); rand() is glibc's additive-feedback generator, reproduced here by random_r on this object's state
    for (size_t i = 1; i < b.size(); i++) {
      int32_t r = 0;
      random_r(&rnd_data, &r);
      const size_t j = (size_t)r % (i + 1);
      if (i != j) std::swap(b[i], b[j]);
    }
    int32_t k = 0;
    for (const p_match& m : b) {
      p_matched_2.push_back(m);
      if (++k >= max_features) break;
    }
  }
}

static float window_mean(const vector<uint8_t>& I, int32_t bpl, int32_t u_min, int32_t u_max, int32_t v_min, int32_t v_max) {
  float mean = 0;
  for (int32_t v = v_min; v <= v_max; v++)
    for (int32_t u = u_min; u <= u_max; u++) mean += (float)I[(size_t)v * bpl + u];
  return mean / (float)((u_max - u_min + 1) * (v_max - v_min + 1));
}

float Matcher::getGain(vector<int32_t> inliers) {
  if (slot[0] < 0 || slot[2] < 0 || p_matched_2.empty() || inliers.empty()) return 1;
  if (!have_I1p) have_I1p = fetchImage(0, I1p);
  if (!have_I1c) have_I1c = fetchImage(2, I1c);
  if (!have_I1p || !have_I1c) return 1;
  const int32_t ws = 3;
  float gain = 0;
  int32_t num = 0;
  auto clampi = [](int32_t x, int32_t hi) { return std::min(std::max(x, 0), hi); };
  for (int32_t idx : inliers) {
    if (idx >= (int32_t)p_matched_2.size()) continue;
    const p_match& m = p_matched_2[idx];
    // note: the reference clamps to dims_p[0] / dims_p[1] (one past the last pixel) for both images
    const float mp = window_mean(I1p, dims_p[2], clampi((int32_t)m.u1p - ws, dims_p[0]), clampi((int32_t)m.u1p + ws, dims_p[0]),
                                 clampi((int32_t)m.v1p - ws, dims_p[1] - 1), clampi((int32_t)m.v1p + ws, dims_p[1] - 1));
    const float mc = window_mean(I1c, dims_c[2], clampi((int32_t)m.u1c - ws, dims_p[0]), clampi((int32_t)m.u1c + ws, dims_p[0]),
                                 clampi((int32_t)m.v1c - ws, dims_p[1] - 1), clampi((int32_t)m.v1c + ws, dims_p[1] - 1));
    if (mp > 10) { gain += mc / mp; num++; }
  }
  return num > 0 ? gain / (float)num : 1;
}

void Matcher::computePriorStatistics(vector<p_match>& p_matched, int32_t method) {
  visob::StageTimer timer(3);
  const float bs = (float)param.match_binsize;
  const int32_t ub = (int32_t)ceil((float)dims_c[0] / bs), vb = (int32_t)ceil((float)dims_c[1] / bs);
  const int32_t nbin = ub * vb, stages = method == 2 ? 4 : 2, nd = stages * 2;
  // running min / max of the displacements seen in the 3x3 bin neighbourhood of every match
  vector<float> lo((size_t)nbin * 8, 1000000.f), hi((size_t)nbin * 8, -1000000.f);
  vector<uint8_t> seen(nbin, 0);
  for (const p_match& m : p_matched) {
    float d[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    float ru, rv;
    if (method == 0) {
      d[0] = m.u1p - m.u1c; d[1] = m.v1p - m.v1c; d[2] = m.u1c - m.u1p; d[3] = m.v1c - m.v1p;
      ru = m.u1c; rv = m.v1c;
    } else if (method == 1) {
      d[0] = m.u2c - m.u1c; d[2] = m.u1c - m.u2c;
      ru = m.u1c; rv = m.v1c;
    } else {
      d[0] = m.u2p - m.u1p; d[2] = m.u2c - m.u2p; d[3] = m.v2c - m.v2p; d[4] = m.u1c - m.u2c;
      d[6] = m.u1p - m.u1c; d[7] = m.v1p - m.v1c;
      ru = m.u1p; rv = m.v1p;
    }
    const int32_t cu = (int32_t)floor(ru / bs), cv = (int32_t)floor(rv / bs);
    const int32_t u0 = std::min(std::max(cu - 1, 0), ub - 1), u1 = std::min(std::max(cu + 1, 0), ub - 1);
    const int32_t v0 = std::min(std::max(cv - 1, 0), vb - 1), v1 = std::min(std::max(cv + 1, 0), vb - 1);
    for (int32_t v = v0; v <= v1; v++)
      for (int32_t u = u0; u <= u1; u++) {
        const size_t b = (size_t)v * ub + u;
        seen[b] = 1;
        for (int32_t i = 0; i < nd; i++) {
          if (d[i] < lo[b * 8 + i]) lo[b * 8 + i] = d[i];
          if (d[i] > hi[b * 8 + i]) hi[b * 8 + i] = d[i];
        }
      }
  }
  ranges.assign(nbin, range());
  for (int32_t b = 0; b < nbin; b++) {
    float dmin[8], dmax[8];
    for (int32_t i = 0; i < 8; i++) {
      dmin[i] = seen[b] ? lo[(size_t)b * 8 + i] : (float)(-param.match_radius);
      dmax[i] = seen[b] ? hi[(size_t)b * 8 + i] : (float)(+param.match_radius);
    }
    range r;
    memset(&r, 0, sizeof r);
    for (int32_t i = 0; i < stages; i++) {
      for (int32_t a = 0; a < 2; a++) {                // widen to at least 20 pixels (matcher.cpp:845-854)
        const float span = dmax[i * 2 + a] - dmin[i * 2 + a];
        if (span < 20) {
          const float grow = ceil((20 - span) / 2);
          dmin[i * 2 + a] -= grow;
          dmax[i * 2 + a] += grow;
        }
      }
      r.u_min[i] = dmin[i * 2 + 0]; r.u_max[i] = dmax[i * 2 + 0];
      r.v_min[i] = dmin[i * 2 + 1]; r.v_max[i] = dmax[i * 2 + 1];
    }
    ranges[b] = r;
  }
}

void Matcher::removeOutliers(vector<p_match>& p_matched, int32_t method) {
  const int32_t n = (int32_t)p_matched.size();
  if (n <= 3) return;
  visob::StageTimer timer(n < 2000 ? 4 : 5);
  static thread_local vector<int32_t> x, y, edges, support;
  x.resize(n); y.resize(n);
  for (int32_t i = 0; i < n; i++) { x[i] = (int32_t)p_matched[i].u1c; y[i] = (int32_t)p_matched[i].v1c; }
  // lists beyond the device path as a whole (3840x2160 frames): the nodes of the triangulation's tree that fit the device
  // kernel are built there, the merges above them and the vote here (delaunay.cpp build_on_device)
  static const bool device_nodes = [] { const char* e = getenv("VISOB_DEVICE_NODES"); return !(e && e[0] == '0'); }();
  visob::delaunay_use_device(visob::device_outliers() && device_nodes ? ctx : nullptr);
  visob::delaunay_edges(x.data(), y.data(), n, edges);
  visob::delaunay_use_device(nullptr);
  support.assign(n, 0);
  const float flow_tol = (float)param.outlier_flow_tolerance, disp_tol = (float)param.outlier_disp_tolerance;
  // float arithmetic throughout, as in the reference (matcher.cpp:1273-1349: float flows, fabs on floats).  What an edge
  // compares is computed once per match (the same float subtractions), so that the vote walks three small arrays instead
  // of the 48-byte records
  static thread_local vector<float> fu, fv, fd;
  fu.resize(n); fv.resize(n); fd.resize(n);
  for (int32_t i = 0; i < n; i++) {
    const p_match& a = p_matched[i];
    fu[i] = a.u1c - a.u1p; fv[i] = a.v1c - a.v1p;
    fd[i] = method == 1 ? a.u1c - a.u2c : a.u1p - a.u2p;
  }
  auto edge_ok = [&](int32_t a, int32_t b) -> bool {
    if (method == 0) return fabsf(fu[a] - fu[b]) + fabsf(fv[a] - fv[b]) < flow_tol;
    if (method == 1) return fabsf(fd[a] - fd[b]) < disp_tol;
    return fabsf(fd[a] - fd[b]) < disp_tol && fabsf(fu[a] - fu[b]) + fabsf(fv[a] - fv[b]) < flow_tol;
  };
  // the reference votes per triangle edge (matcher.cpp:1259-1362): an edge shared by two triangles counts twice
  for (size_t e = 0; e + 2 < edges.size(); e += 3) {
    const int32_t a = edges[e], b = edges[e + 1], t = edges[e + 2];
    if (edge_ok(a, b)) { support[a] += t; support[b] += t; }
  }
  int32_t k = 0;
  for (int32_t i = 0; i < n; i++)
    if (support[i] >= 4) p_matched[k++] = p_matched[i];
  p_matched.resize(k);
}


// ---------------------------------------------------------------------------------------------------------------------
// MatcherBatch: S independent sequences on ONE context.  Every GPU stage is issued once for all sequences (the C-ABI is
// batched: one launch per kernel covers all S frames / pairs), the host stages run per sequence in between.  The result
// of every sequence is identical to what a stand-alone Matcher produces.
MatcherBatch::MatcherBatch(Matcher::parameters param, int32_t n_sequences) : k_submit(0), k_collect(0), ctx(0), width(0), height(0) {
  for (int32_t s = 0; s < n_sequences; s++) seq.push_back(new Matcher(param));
  device = visob::current_device();
  memset(&rect, 0, sizeof rect);
  started = false;
}

bool MatcherBatch::setRectification(const Rectification& r) {
  if (started || r.n_cams < 0 || r.n_cams > 2) return false;
  for (Matcher* m : seq) m->setRectification(r);     // the sequences check the raw dims and see the rectified ones
  rect = r;
  width = height = 0;                                // the next push configures the context and sets the maps
  return true;
}

MatcherBatch::~MatcherBatch() {
  for (Matcher* m : seq) delete m;
  if (ctx) visocu_destroy(ctx);
}

bool MatcherBatch::ensure(int32_t w, int32_t h) {
  if (ctx && w == width && h == height) return true;
  if (!ctx && visocu_create(device, &ctx) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(0) << std::endl;
    ctx = 0;
    return false;
  }
  visocu_params vp;
  memcpy(&vp, &seq[0]->param, sizeof vp);
  if (visocu_configure(ctx, &vp, w, h, 4 * (int32_t)seq.size()) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    return false;
  }
  if (rect.n_cams > 0 && visocu_set_rectification(ctx, rect.n_cams, rect.cams, rect.src_w, rect.src_h) != VISOCU_OK) {
    std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
    return false;
  }
  width = w; height = h;
  started = true;
  for (size_t s = 0; s < seq.size(); s++) seq[s]->useSharedContext(ctx, 4 * (int32_t)s, w, h);
  return true;
}

void MatcherBatch::pushBack(const uint8_t* const* I1, const uint8_t* const* I2, uint32_t* dims, bool replace, bool on_device) {
  std::unique_ptr<bool[]> flags(new bool[seq.size()]);
  for (size_t s = 0; s < seq.size(); s++) flags[s] = replace;
  pushBack(I1, I2, dims, flags.get(), on_device);
}

void MatcherBatch::pushBack(const uint8_t* const* I1, const uint8_t* const* I2, uint32_t* dims, const bool* replace, bool on_device) {
  visob::StageTimer timer(0);
  uint32_t od[3];
  const bool rectify = rect.n_cams > 0;
  if (rectify) {
    if (!seq[0]->rectifiedDims(dims, od)) return;
  } else if ((int32_t)dims[0] <= 0 || (int32_t)dims[1] <= 0 || dims[2] < dims[0]) {
    std::cerr << "ERROR: Image dimension mismatch!" << std::endl;
    return;
  }
  const int32_t bpl = (int32_t)dims[2];
  if (rectify) dims = od;                            // the sequences see the rectified images
  if (!ensure((int32_t)dims[0], (int32_t)dims[1])) return;
  const size_t S = seq.size();
  vector<int32_t> frames, owner, cams;
  vector<const uint8_t*> imgs;
  for (size_t s = 0; s < S; s++) {
    int32_t f[2];
    const uint8_t* i2 = I2 ? I2[s] : 0;
    if (!seq[s]->pushPrepare(I1[s], i2, dims, replace[s], f)) continue;
    frames.push_back(f[0]); imgs.push_back(I1[s]); owner.push_back((int32_t)s); cams.push_back(0);
    if (i2) { frames.push_back(f[1]); imgs.push_back(i2); owner.push_back((int32_t)s); cams.push_back(1); }
  }
  if (frames.empty()) return;
  vector<int32_t> ns(frames.size(), -1), nd(frames.size(), -1);
  const bool lazy = seq[0]->lazyCounts() && !I2;           // see Matcher::push
  const int32_t nf = (int32_t)frames.size(), where = on_device ? 1 : 0;
  const bool ok = (rectify ? visocu_push_frames_rectified(ctx, nf, frames.data(), imgs.data(), cams.data(), bpl, where, lazy ? 0 : ns.data(),
                                                          lazy ? 0 : nd.data())
                           : visocu_push_frames(ctx, nf, frames.data(), imgs.data(), bpl, where, lazy ? 0 : ns.data(),
                                                lazy ? 0 : nd.data())) == VISOCU_OK;
  if (!ok) std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
  for (size_t k = 0; k < frames.size();) {
    const int32_t s = owner[k];
    const bool stereo = k + 1 < frames.size() && owner[k + 1] == s;
    seq[s]->pushFinish(ok, stereo, &ns[k], &nd[k]);
    k += stereo ? 2 : 1;
  }
}

bool MatcherBatch::matchPass(const vector<int32_t>& active, int pass, int32_t method, bool use_prior, int refine) {
  visob::StageTimer timer(1 + pass);
  const size_t n = active.size();
  vector<visocu_quad> quads(n);
  vector<visocu_pmatch*> outs(n);
  vector<const visocu_range*> rptr(n);
  vector<const double*> tptr(n, 0);
  vector<int32_t> cap(n), cnt(n), done(n, 0);
  bool any_tr = false;
  for (size_t k = 0; k < n; k++) {
    Matcher* m = seq[active[k]];
    vector<Matcher::p_match>& out = pass == 0 ? m->p_matched_1 : m->p_matched_2;
    const int32_t nq = m->queryCount(pass, method);
    out.resize((size_t)nq + 1);
    quads[k] = visocu_quad{m->slot[0], m->slot[1], m->slot[2], m->slot[3]};
    outs[k] = reinterpret_cast<visocu_pmatch*>(out.data());
    rptr[k] = reinterpret_cast<const visocu_range*>(m->ranges.data());
    cap[k] = nq + 1;
    if (m->has_tr && method == 2) { tptr[k] = m->tr_rows; any_tr = true; }
  }
  const int rc = visocu_match(ctx, (int32_t)n, quads.data(), method, pass, use_prior ? 1 : 0, use_prior ? rptr.data() : 0,
                              any_tr ? tptr.data() : 0, refine, outs.data(), cap.data(), cnt.data(), visob::device_outliers() ? done.data() : 0);
  if (rc != VISOCU_OK) std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
  for (size_t k = 0; k < n; k++) {
    Matcher* m = seq[active[k]];
    m->ro_done[pass] = rc == VISOCU_OK && done[k] != 0;
    (pass == 0 ? m->p_matched_1 : m->p_matched_2).resize(rc == VISOCU_OK ? cnt[k] : 0);
  }
  return rc == VISOCU_OK;
}

void MatcherBatch::matchFeatures(int32_t method, const Matrix* const* tr_delta) {
  if (!ctx) return;
  vector<int32_t> active;
  // per-sequence motion prediction of quad matching, as Matcher::matchFeatures(2, Tr_delta) does for one sequence; the
  // sequences share the context and with it the calibration, which is taken from the first sequence that predicts
  const Matcher* calib = 0;
  for (size_t s = 0; s < seq.size(); s++) {
    Matcher* m = seq[s];
    const Matrix* T = tr_delta ? tr_delta[s] : 0;
    m->has_tr = T && method == 2 && T->m >= 3 && T->n >= 4;
    if (!m->has_tr) continue;
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 4; c++) m->tr_rows[4 * r + c] = T->val[r][c];
    if (!calib) calib = m;
  }
  if (calib) visocu_set_intrinsics(ctx, calib->param.f, calib->param.cu, calib->param.cv, calib->param.base);
  const bool fused = Matcher::fusedAvailable(*seq[0], method) && seq.size() <= 128;
  for (size_t s = 0; s < seq.size(); s++) {
    if (!fused) seq[s]->syncCounts();
    if (seq[s]->matchBegin(method)) active.push_back((int32_t)s);
  }
  if (active.empty()) return;
  const Matcher::parameters& p = seq[0]->param;
  const int refine = seq[0]->refineMode();
  if (fused) {
    vector<Matcher*> group;
    for (int32_t s : active) group.push_back(seq[s]);
    Matcher::fusedMatch(ctx, group, method);
    return;
  }
  for (int32_t s : active) { seq[s]->p_matched_1.clear(); seq[s]->p_matched_2.clear(); }
  if (p.multi_stage) {
    if (!matchPass(active, 0, method, false, 0)) return;
    for (int32_t s : active) seq[s]->matchAfterPass1(method);
    if (!matchPass(active, 1, method, true, refine)) return;
  } else {
    if (!matchPass(active, 1, method, false, refine)) return;
  }
  for (int32_t s : active) seq[s]->matchAfterPass2(method);
}

// ---- pipelined stepping (see matcher.h)
bool MatcherBatch::stepAvailable(int32_t method) const {
  return method == 0 && !seq.empty() && seq[0]->lazyCounts() && (int32_t)seq.size() <= 128;
}

bool MatcherBatch::stepSubmit(const uint8_t* const* I1, uint32_t* dims, bool on_device) {
  // host images of a step stay valid until the step is collected (the runner's contract): mode 2 of visocu_push_frames
  visob::StageTimer timer(0);
  uint32_t od[3];
  const bool rectify = rect.n_cams > 0;
  if (rectify) {
    if (!seq[0]->rectifiedDims(dims, od)) return false;
  } else if ((int32_t)dims[0] <= 0 || (int32_t)dims[1] <= 0 || dims[2] < dims[0]) {
    std::cerr << "ERROR: Image dimension mismatch!" << std::endl;
    return false;
  }
  const int32_t bpl = (int32_t)dims[2];
  if (rectify) dims = od;
  if (!ensure((int32_t)dims[0], (int32_t)dims[1])) return false;
  if (k_submit - k_collect >= 3) return false;                       // the fourth frame of the ring is still being read
  const size_t S = seq.size();
  const int64_t k = k_submit;
  const int lane = (int)(k & 3);
  if (visocu_set_lane(ctx, lane) != VISOCU_OK) { std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl; return false; }
  // frame k of sequence s lives in slot 4 s + (k & 3): four consecutive frames stay alive
  vector<int32_t> frames(S), cams(S, 0);
  vector<visocu_quad> quads(S);
  for (size_t s = 0; s < S; s++) {
    frames[s] = 4 * (int32_t)s + lane;
    quads[s] = visocu_quad{4 * (int32_t)s + (int)((k + 3) & 3), -1, frames[s], -1};
    if (!I1[s]) { std::cerr << "ERROR: Image dimension mismatch!" << std::endl; return false; }
  }
  const int32_t where = on_device ? 1 : 2;
  bool ok = (rectify ? visocu_push_frames_rectified(ctx, (int32_t)S, frames.data(), I1, cams.data(), bpl, where, 0, 0)
                     : visocu_push_frames(ctx, (int32_t)S, frames.data(), I1, bpl, where, 0, 0)) == VISOCU_OK;
  if (ok && k > 0)
    ok = visocu_match_fused_submit(ctx, (int32_t)S, quads.data(), seq[0]->refineMode(), 0, (int)((k + 3) & 3)) == VISOCU_OK;
  if (!ok) std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
  visocu_set_lane(ctx, 4);
  if (!ok) return false;
  for (int c = 0; c < 3; c++) step_dims[c] = (int32_t)dims[c];
  k_submit++;
  return true;
}

bool MatcherBatch::stepCollect() {
  if (k_collect >= k_submit) return false;
  visob::StageTimer timer(2);
  const size_t S = seq.size();
  const int64_t k = k_collect++;
  const int lane = (int)(k & 3), prev = (int)((k + 3) & 3);
  for (size_t s = 0; s < S; s++) {
    Matcher* m = seq[s];
    // the sequence now refers to the pair (frame k - 1, frame k)
    m->slot[0] = k > 0 ? 4 * (int32_t)s + prev : -1; m->slot[1] = -1;
    m->slot[2] = 4 * (int32_t)s + lane; m->slot[3] = -1;
    for (int c = 0; c < 3; c++) { m->dims_p[c] = k > 0 ? step_dims[c] : 0; m->dims_c[c] = step_dims[c]; }
    m->dims_c[2] = step_dims[0] + 15 - (step_dims[0] - 1) % 16;
    if (k > 0) m->dims_p[2] = m->dims_c[2];
    m->have_I1p = m->have_I1c = false;
    m->n_feat[1] = m->n_feat[3] = m->n_feat[5] = m->n_feat[7] = 0;
  }
  if (k == 0) {                                                       // only a push: nothing to collect but its counts
    for (size_t s = 0; s < S; s++) { Matcher* m = seq[s]; m->n_feat[0] = m->n_feat[4] = 0; m->n_feat[2] = m->n_feat[6] = -1; }
    return true;
  }
  if (visocu_set_lane(ctx, lane) != VISOCU_OK) return false;
  vector<const visocu_pmatch*> l1(S), l2(S);
  vector<int32_t> n1(S, 0), n2(S, 0), d1(S, 0), d2(S, 0), counts(4 * S, 0);
  int32_t compact = 0;
  const int rc = visocu_match_fused_collect(ctx, l1.data(), n1.data(), d1.data(), l2.data(), n2.data(), d2.data(), 0, counts.data(), &compact);
  if (rc != VISOCU_OK) std::cerr << "ERROR: " << visocu_last_error(ctx) << std::endl;
  visocu_set_lane(ctx, 4);                                            // fall-backs and odometry calls run on their own lane
  for (size_t s = 0; s < S; s++) Matcher::takeFused(seq[s], rc == VISOCU_OK, &counts[4 * s], l1[s], n1[s], d1[s], l2[s], n2[s], d2[s], 0, compact);
  return rc == VISOCU_OK;
}
