// Reconstruction of finished feature tracks: linear triangulation, point type, Gauss-Newton refinement, distance and
// ray-angle tests for the tracks of many Reconstruction::update calls at once.
//
// What it reproduces (host/reconstruction.cpp, which restates the reference reconstruction.cpp:50-343):
//   initPoint ....... null vector of the 4x4 system built from the first observation in the track's first frame and the
//                     last observation in the NEWEST frame; w rounded to float, fails if |w| < 1e-10; point in float
//   pointType ....... on the initial point: both end cameras at z > 1 (else -1), then the road height of the point in the
//                     newest camera: > 0.5 -> 0, > -1 -> 1, else 2; the track is dropped if the type < point_type
//   refinePoint ..... observation k predicted with the projection of frame first + k; c^2 < 1e-10 fails; the 3x3 normal
//                     equations summed over the 2 n_obs rows in the host's order, solved as Matrix::solve does (full
//                     pivoting, eps 1e-20); the point stays in float between updates; converged when all three updates
//                     are below 1e-5, failed after 22 updates
//   pointDistance ... to the centre of the frame half way along the track, < max_dist
//   rayAngle ........ acos(|cos|) in degrees between the rays from the first and the newest centre (1000 if a ray is
//                     degenerate), > min_angle
//
// Design: one thread per track, FP64.  A track is a short strictly sequential chain (a Jacobi null vector, at most 22
// tiny solves); tracks are independent.  Jobs are concatenated: thread i finds its job by a binary search over the jobs'
// first track.  The frames of a job are read through the cache (every track of the job reads the same few frames).  The
// 3x3 elimination runs on the thread's own column of shared memory (pivot rows and columns are dynamic indices).
// Floating-point contract: nvcc contracts to FMA, as the host build does in its own places; results agree with the host
// to rounding and are not bit-identical to it (the null vector also comes from a different algorithm).
#include "visocu_internal.cuh"
#include <cstring>

namespace {

constexpr int RECON_THREADS = 128;
constexpr int MAX_FRAMES = 8;
constexpr int MAX_OBS = 6;
constexpr int MAX_UPDATES = 22;          // refinePoint: `iter > 20` after each update
constexpr double SOLVE_EPS = 1e-20;      // Matrix::solve default

enum { KEPT = 0, INIT_FAILED = 1, TYPE_BELOW = 2, REFINE_FAILED = 3, TOO_FAR = 4, ANGLE_TOO_SMALL = 5 };

struct ReconJobDev {
  const visocu_recon_frame* frames;
  const visocu_recon_track* tracks;
  int4* out;                             // per track: status, then x, y, z as float bits
  double cam_road[12];
  double max_dist, min_angle;
  int first_track, n_tracks, point_type, n_frames;
};

// affineTransform (host/reconstruction.cpp): rows 0..2 of M applied to (p, 1), accumulated in double, rounded to float
__device__ __forceinline__ float3 affine(const double* M, float3 p) {
  return make_float3((float)(p.x * M[0] + p.y * M[1] + p.z * M[2] + M[3]),
                     (float)(p.x * M[4] + p.y * M[5] + p.z * M[6] + M[7]),
                     (float)(p.x * M[8] + p.y * M[9] + p.z * M[10] + M[11]));
}

__global__ void __launch_bounds__(RECON_THREADS) k_recon(const ReconJobDev* __restrict__ jobs, int n_jobs, int n_total) {
  __shared__ double sA[9 * RECON_THREADS], sb[3 * RECON_THREADS];
  const int i = blockIdx.x * RECON_THREADS + threadIdx.x;
  if (i >= n_total) return;
  int lo = 0, hi = n_jobs - 1;                       // last job whose first track is <= i (empty jobs are skipped over)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].first_track <= i) lo = mid; else hi = mid - 1;
  }
  const ReconJobDev& J = jobs[lo];
  const visocu_recon_track t = J.tracks[i - J.first_track];
  const visocu_recon_frame* F = J.frames;
  const int newest = J.n_frames - 1, f0 = t.first;
  const int last = t.n_obs - 1;
  int status = KEPT;
  float3 p = make_float3(0.f, 0.f, 0.f);

  // ---- initPoint
  {
    const double* P1 = F[f0].proj;
    const double* P2 = F[newest].proj;
    const double au = t.u[0], av = t.v[0];
    const double bu = last == 1 ? t.u[1] : (last == 2 ? t.u[2] : (last == 3 ? t.u[3] : (last == 4 ? t.u[4] : t.u[5])));
    const double bv = last == 1 ? t.v[1] : (last == 2 ? t.v[2] : (last == 3 ? t.v[3] : (last == 4 ? t.v[4] : t.v[5])));
    double g[4][4], X[4];
#pragma unroll
    for (int c = 0; c < 4; c++) {
      g[c][0] = P1[8 + c] * au - P1[c];
      g[c][1] = P1[8 + c] * av - P1[4 + c];
      g[c][2] = P2[8 + c] * bu - P2[c];
      g[c][3] = P2[8 + c] * bv - P2[4 + c];
    }
    jacobi_null_vector4(g, X);
    const float w = (float)X[3];
    if (fabsf(w) < 1e-10) status = INIT_FAILED;
    else p = make_float3((float)(X[0] / (double)w), (float)(X[1] / (double)w), (float)(X[2] / (double)w));
  }

  // ---- pointType on the initial point
  if (status == KEPT) {
    const float3 x1c = affine(F[f0].inv, p);
    const float3 x2c = affine(F[newest].inv, p);
    const float3 x2r = affine(J.cam_road, x2c);
    const int type = (x1c.z <= 1 || x2c.z <= 1) ? -1 : (x2r.y > 0.5 ? 0 : (x2r.y > -1 ? 1 : 2));
    if (type < J.point_type) status = TYPE_BELOW;
  }

  // ---- refinePoint
  if (status == KEPT) {
    double* A = sA + threadIdx.x;
    double* b = sb + threadIdx.x;
    bool done = false;
    for (int it = 0; it < MAX_UPDATES && !done && status == KEPT; it++) {
      double Jr[2 * MAX_OBS][3], res[2 * MAX_OBS];
#pragma unroll
      for (int k = 0; k < MAX_OBS; k++) {                 // unrolled: Jr and res stay in registers
        if (k > last) break;
        const double* P = F[f0 + k].proj;
        const double a = P[0] * p.x + P[1] * p.y + P[2] * p.z + P[3];
        const double bb = P[4] * p.x + P[5] * p.y + P[6] * p.z + P[7];
        const double c = P[8] * p.x + P[9] * p.y + P[10] * p.z + P[11];
        const double cc = c * c;
        if (cc < 1e-10) { status = REFINE_FAILED; break; }
#pragma unroll
        for (int j = 0; j < 3; j++) {
          Jr[2 * k][j] = (P[j] * c - P[8 + j] * a) / cc;
          Jr[2 * k + 1][j] = (P[4 + j] * c - P[8 + j] * bb) / cc;
        }
        res[2 * k] = t.u[k] - a / c;
        res[2 * k + 1] = t.v[k] - bb / c;
      }
      if (status != KEPT) break;
#pragma unroll
      for (int m = 0; m < 3; m++) {
#pragma unroll
        for (int n = 0; n < 3; n++) {
          double s = 0;
#pragma unroll
          for (int r = 0; r < 2 * MAX_OBS; r++) if (r <= 2 * last + 1) s += Jr[r][m] * Jr[r][n];
          A[(3 * m + n) * RECON_THREADS] = s;
        }
        double s = 0;
#pragma unroll
        for (int r = 0; r < 2 * MAX_OBS; r++) if (r <= 2 * last + 1) s += Jr[r][m] * res[r];
        b[m * RECON_THREADS] = s;
      }
      if (!gj_solve<3>(A, b, RECON_THREADS, SOLVE_EPS)) { status = REFINE_FAILED; break; }
      const double dx = b[0], dy = b[RECON_THREADS], dz = b[2 * RECON_THREADS];
      p.x = (float)(p.x + dx); p.y = (float)(p.y + dy); p.z = (float)(p.z + dz);
      done = fabs(dx) < 1e-5 && fabs(dy) < 1e-5 && fabs(dz) < 1e-5;
    }
    if (status == KEPT && !done) status = REFINE_FAILED;
    if (status == REFINE_FAILED) p = make_float3(0.f, 0.f, 0.f);
  }

  // ---- pointDistance, rayAngle
  if (status == KEPT) {
    const double* cm = F[newest - (J.n_frames - f0) / 2].center;
    const double dx = cm[0] - p.x, dy = cm[1] - p.y, dz = cm[2] - p.z;
    if (!(sqrt(dx * dx + dy * dy + dz * dz) < J.max_dist)) status = TOO_FAR;
  }
  if (status == KEPT) {
    const double* c1 = F[f0].center;
    const double* c2 = F[newest].center;
    const double pt[3] = {p.x, p.y, p.z};
    double v1[3], v2[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { v1[k] = c1[k] - pt[k]; v2[k] = c2[k] - pt[k]; }
    const double n1 = sqrt(v1[0] * v1[0] + v1[1] * v1[1] + v1[2] * v1[2]);
    const double n2 = sqrt(v2[0] * v2[0] + v2[1] * v2[1] + v2[2] * v2[2]);
    double angle = 1000;
    if (!(n1 < 1e-10 || n2 < 1e-10)) {
      double dot = 0;
#pragma unroll
      for (int k = 0; k < 3; k++) dot += (v1[k] / n1) * (v2[k] / n2);
      angle = acos(fabs(dot)) * 180.0 / M_PI;
    }
    if (!(angle > J.min_angle)) status = ANGLE_TOO_SMALL;
  }
  J.out[i - J.first_track] = make_int4(status, __float_as_int(p.x), __float_as_int(p.y), __float_as_int(p.z));
}

}  // namespace

// Shared with recon_store.cu (visocu_recon_update): the checks, the upload image and the launch of k_recon.
int visocu_recon_check(visocu_ctx* ctx, const char* what, int32_t n_jobs, const visocu_recon_job* jobs, int32_t* const* status,
                       float* const* xyz, size_t* n_tracks_total, size_t* n_frames_total) {
  size_t n_total = 0, nf = 0;
  for (int j = 0; j < n_jobs; j++) {
    const visocu_recon_job& J = jobs[j];
    if (J.n_frames < 1 || J.n_frames > MAX_FRAMES || !J.frames || J.n_tracks < 0)
      return visocu_set_error(ctx, VISOCU_EINVAL, "%s job %d: bad frame table or track count", what, j);
    if (J.n_tracks > 0 && (!J.tracks || (status && !status[j]) || (xyz && !xyz[j])))
      return visocu_set_error(ctx, VISOCU_EINVAL, "%s job %d: null pointer", what, j);
    for (int k = 0; k < J.n_tracks; k++) {
      const visocu_recon_track& t = J.tracks[k];
      if (t.n_obs < 2 || t.n_obs > MAX_OBS || t.first < 0 || t.first > J.n_frames - t.n_obs)   // no overflow: n_obs <= 6
        return visocu_set_error(ctx, VISOCU_EINVAL, "%s job %d track %d: observations outside the window", what, j, k);
    }
    n_total += (size_t)J.n_tracks;
    nf += (size_t)J.n_frames;
  }
  if (n_total > (size_t)INT32_MAX / 2) return visocu_set_error(ctx, VISOCU_EINVAL, "%s: too many tracks", what);
  *n_tracks_total = n_total;
  *n_frames_total = nf;
  return VISOCU_OK;
}

// bytes of k_recon's inputs: job descriptors, frame tables, tracks, each part 256-byte aligned
size_t visocu_recon_stage_bytes(int32_t n_jobs, size_t n_frames_total, size_t n_tracks_total) {
  const size_t o_frames = align_up(sizeof(ReconJobDev) * n_jobs, 256);
  const size_t o_tracks = align_up(o_frames + sizeof(visocu_recon_frame) * n_frames_total, 256);
  return o_tracks + sizeof(visocu_recon_track) * n_tracks_total;
}

// writes k_recon's inputs into `pin`, the host image of the device bytes at `dev`; job j's results go to out + its first
// track.  first_track (n_jobs entries, optional) receives each job's first track.
void visocu_recon_stage(int32_t n_jobs, const visocu_recon_job* jobs, size_t n_frames_total, uint8_t* pin, uint8_t* dev, int4* out,
                        int32_t* first_track) {
  const size_t o_frames = align_up(sizeof(ReconJobDev) * n_jobs, 256);
  const size_t o_tracks = align_up(o_frames + sizeof(visocu_recon_frame) * n_frames_total, 256);
  ReconJobDev* hj = (ReconJobDev*)pin;
  size_t fo = 0, to = 0;
  for (int j = 0; j < n_jobs; j++) {
    const visocu_recon_job& J = jobs[j];
    ReconJobDev& d = hj[j];
    d.frames = (const visocu_recon_frame*)(dev + o_frames) + fo;
    d.tracks = (const visocu_recon_track*)(dev + o_tracks) + to;
    d.out = out + to;
    memcpy(d.cam_road, J.cam_road, sizeof d.cam_road);
    d.max_dist = J.max_dist; d.min_angle = J.min_angle;
    d.first_track = (int)to; d.n_tracks = J.n_tracks; d.point_type = J.point_type; d.n_frames = J.n_frames;
    if (first_track) first_track[j] = (int32_t)to;
    memcpy(pin + o_frames + sizeof(visocu_recon_frame) * fo, J.frames, sizeof(visocu_recon_frame) * J.n_frames);
    if (J.n_tracks) memcpy(pin + o_tracks + sizeof(visocu_recon_track) * to, J.tracks, sizeof(visocu_recon_track) * J.n_tracks);
    fo += (size_t)J.n_frames; to += (size_t)J.n_tracks;
  }
}

int visocu_recon_launch(visocu_ctx* ctx, const uint8_t* dev, int32_t n_jobs, size_t n_tracks_total) {
  k_recon<<<(unsigned)((n_tracks_total + RECON_THREADS - 1) / RECON_THREADS), RECON_THREADS, 0, ctx->stream>>>(
      (const ReconJobDev*)dev, n_jobs, (int)n_tracks_total);
  CU_LAUNCH_CHECK(ctx);
  return VISOCU_OK;
}

extern "C" int visocu_recon_points(visocu_ctx* ctx, int32_t n_jobs, const visocu_recon_job* jobs, int32_t* const* status,
                                   float* const* xyz) {
  if (!ctx) return VISOCU_EINVAL;
  if (n_jobs < 0 || (n_jobs > 0 && (!jobs || !status || !xyz))) return visocu_set_error(ctx, VISOCU_EINVAL, "bad recon_points arguments");
  // every job is checked before anything is enqueued or written
  size_t n_total = 0, n_frames_total = 0;
  int rc = visocu_recon_check(ctx, "recon_points", n_jobs, jobs, status, xyz, &n_total, &n_frames_total);
  if (rc) return rc;
  if (n_total == 0) return VISOCU_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  // Upload: job descriptors, frame tables, tracks (ONE copy).  Read-back: 16 bytes per track (ONE copy).
  const size_t up_bytes = visocu_recon_stage_bytes(n_jobs, n_frames_total, n_total);
  const size_t o_out = align_up(up_bytes, 256);
  const size_t back_bytes = 16 * n_total;
  if ((rc = visocu_ensure_scratch(ctx, o_out + back_bytes))) return rc;
  if ((rc = visocu_ensure_pinned(ctx, o_out + back_bytes))) return rc;
  uint8_t* sb = (uint8_t*)ctx->scratch;
  uint8_t* pin = (uint8_t*)ctx->pinned;
  std::vector<int32_t> first((size_t)n_jobs);
  visocu_recon_stage(n_jobs, jobs, n_frames_total, pin, sb, (int4*)(sb + o_out), first.data());
  CU_COPY(ctx, sb, pin, up_bytes, cudaMemcpyHostToDevice);
  if ((rc = visocu_recon_launch(ctx, sb, n_jobs, n_total))) return rc;
  CU_COPY(ctx, pin + o_out, sb + o_out, back_bytes, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  const int32_t* res = (const int32_t*)(pin + o_out);
  for (int j = 0; j < n_jobs; j++) {
    for (int k = 0; k < jobs[j].n_tracks; k++) {
      const int32_t* r = res + 4 * (size_t)(first[j] + k);
      status[j][k] = r[0];
      memcpy(xyz[j] + 3 * (size_t)k, r + 1, 12);
    }
  }
  return VISOCU_OK;
}
