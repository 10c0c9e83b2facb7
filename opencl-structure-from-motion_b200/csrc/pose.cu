// Pose-recovery helpers of monocular odometry that follow the RANSAC step (SURVEY.md 8f rank 2).
//
// What it reproduces (reference paths relative to /root/reference/viso):
//   VisualOdometryMono::triangulateChieral ... viso_mono.cpp:394-431  (N independent 4x4 null-vector problems per (R|t))
//   VisualOdometryMono::findBestPlane ........ viso_mono.cpp:74-98    (O(n^2) Gaussian vote; the reference's OpenCL
//                                              offload is plane_calc_sums, kernels/plane_and_inliers.cl:142-162, float32)
// Here both run in FP64.  The triangulation does all four (R|t) candidates of EtoRt (viso_mono.cpp:347-392) in one
// launch, one thread per (candidate, match): a 4x4 one-sided Jacobi in registers replaces Matrix::svd.
#include "visocu_internal.cuh"
#include <cstring>

namespace {

struct TriJob {
  const float4* uv;      // N x (u1p, v1p, u1c, v1c) in pixels
  double* X;             // n_sol x 4 x N
  int32_t* n_front;      // n_sol
  int N, n_sol;
  double P1[12];
  double P2[4][12];
};

__global__ void __launch_bounds__(128) k_triangulate(const TriJob* __restrict__ jobs) {
  const TriJob& job = jobs[blockIdx.z];
  const int i = blockIdx.x * 128 + threadIdx.x, sol = blockIdx.y;
  if (sol >= job.n_sol) return;
  int front = 0;
  if (i < job.N) {
    const float4 m = job.uv[i];
    const double* P1 = job.P1;
    const double* P2 = job.P2[sol];
    // J rows (viso_mono.cpp:411-416); g[c][r] = column c of J
    double g[4][4];
#pragma unroll
    for (int c = 0; c < 4; c++) {
      g[c][0] = P1[8 + c] * (double)m.x - P1[c];
      g[c][1] = P1[8 + c] * (double)m.y - P1[4 + c];
      g[c][2] = P2[8 + c] * (double)m.z - P2[c];
      g[c][3] = P2[8 + c] * (double)m.w - P2[4 + c];
    }
    double X[4];
    jacobi_null_vector4(g, X);
    double* out = job.X + (size_t)sol * 4 * job.N;
#pragma unroll
    for (int r = 0; r < 4; r++) out[(size_t)r * job.N + i] = X[r];
    // points in front of both cameras (viso_mono.cpp:421-427)
    const double a = P1[8] * X[0] + P1[9] * X[1] + P1[10] * X[2] + P1[11] * X[3];
    const double b = P2[8] * X[0] + P2[9] * X[1] + P2[10] * X[2] + P2[11] * X[3];
    front = (a * X[3] > 0 && b * X[3] > 0) ? 1 : 0;
  }
  const unsigned bal = __ballot_sync(0xFFFFFFFFu, front);
  if ((threadIdx.x & 31) == 0 && bal) atomicAdd(&job.n_front[sol], __popc(bal));
}

// one warp per candidate i: sum_j exp(-(d_j - d_i)^2 w) with a fixed lane-strided + butterfly summation order
// (deterministic; differs from the reference's sequential order only in rounding).  Candidates need d_i > threshold.
struct PlaneJob { const double* d; double* sums; double threshold, weight; int n, pad; };

__global__ void __launch_bounds__(256) k_plane_sums(const PlaneJob* __restrict__ jobs) {
  const PlaneJob J = jobs[blockIdx.y];
  const double* d = J.d; double* sums = J.sums;
  const int n = J.n; const double threshold = J.threshold, weight = J.weight;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= n) return;
  const double di = d[i];
  if (!(di > threshold)) {
    if (lane == 0) sums[i] = -1.0;          // marks "not a candidate"
    return;
  }
  double sum = 0;
  for (int j = lane; j < n; j += 32) {
    const double dist = d[j] - di;
    sum += exp(-dist * dist * weight);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
  if (lane == 0) sums[i] = sum;
}

}  // namespace

extern "C" int visocu_triangulate_batch(visocu_ctx* ctx, int32_t n_jobs, const float* const* uv, const int32_t* N, const double* const* P1,
                                        const double* const* P2, const int32_t* n_sol, double* const* X, int32_t* const* n_front) {
  if (!ctx || n_jobs <= 0 || n_jobs > VISO_MAX_BATCH || !uv || !N || !P1 || !P2 || !n_sol || !X || !n_front)
    return ctx ? visocu_set_error(ctx, VISOCU_EINVAL, "bad triangulate arguments") : VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  // one upload (job descriptors + coordinates), one launch, one read-back (points + counters), pinned staging
  std::vector<TriJob> hj(n_jobs);
  std::vector<size_t> o_uv(n_jobs), o_X(n_jobs), o_cnt(n_jobs);
  size_t off = align_up(sizeof(TriJob) * n_jobs, 256);
  int maxN = 0, maxsol = 0;
  for (int j = 0; j < n_jobs; j++) {
    if (!uv[j] || !P1[j] || !P2[j] || !X[j] || !n_front[j] || N[j] <= 0 || n_sol[j] < 1 || n_sol[j] > 4)
      return visocu_set_error(ctx, VISOCU_EINVAL, "bad triangulate job %d", j);
    o_uv[j] = off; off += align_up((size_t)N[j] * 16, 256);
    if (N[j] > maxN) maxN = N[j];
    if (n_sol[j] > maxsol) maxsol = n_sol[j];
  }
  const size_t up_bytes = off;
  for (int j = 0; j < n_jobs; j++) {
    o_X[j] = off; off += align_up((size_t)n_sol[j] * 4 * N[j] * 8, 256);
    o_cnt[j] = off; off += 256;
  }
  int rc = visocu_ensure_scratch(ctx, off);
  if (rc) return rc;
  if ((rc = visocu_ensure_pinned(ctx, off))) return rc;
  uint8_t* sb = (uint8_t*)ctx->scratch;
  uint8_t* pin = (uint8_t*)ctx->pinned;
  for (int j = 0; j < n_jobs; j++) {
    TriJob& job = hj[j];
    job.uv = (const float4*)(sb + o_uv[j]); job.X = (double*)(sb + o_X[j]); job.n_front = (int32_t*)(sb + o_cnt[j]);
    job.N = N[j]; job.n_sol = n_sol[j];
    memcpy(job.P1, P1[j], sizeof job.P1);
    memcpy(job.P2, P2[j], sizeof(double) * 12 * n_sol[j]);
    memcpy(pin + o_uv[j], uv[j], (size_t)N[j] * 16);
  }
  memcpy(pin, hj.data(), sizeof(TriJob) * n_jobs);
  CU_COPY(ctx, sb, pin, up_bytes, cudaMemcpyHostToDevice);
  CU_TRY(ctx, cudaMemsetAsync(sb + up_bytes, 0, off - up_bytes, ctx->stream));
  k_triangulate<<<dim3((maxN + 127) / 128, maxsol, n_jobs), 128, 0, ctx->stream>>>((const TriJob*)sb);
  CU_LAUNCH_CHECK(ctx);
  CU_COPY(ctx, pin + up_bytes, sb + up_bytes, off - up_bytes, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  for (int j = 0; j < n_jobs; j++) {
    memcpy(X[j], pin + o_X[j], (size_t)n_sol[j] * 4 * N[j] * 8);
    memcpy(n_front[j], pin + o_cnt[j], (size_t)n_sol[j] * 4);
  }
  return VISOCU_OK;
}

extern "C" int visocu_triangulate(visocu_ctx* ctx, const float* uv, int32_t N, const double* P1, const double* P2, int32_t n_sol,
                                  double* X, int32_t* n_front) {
  if (!ctx || !uv || !P1 || !P2 || !X || !n_front || N <= 0 || n_sol < 1 || n_sol > 4) return ctx ? visocu_set_error(ctx, VISOCU_EINVAL, "bad triangulate arguments") : VISOCU_EINVAL;
  return visocu_triangulate_batch(ctx, 1, &uv, &N, &P1, &P2, &n_sol, &X, &n_front);
}

extern "C" int visocu_best_plane_batch(visocu_ctx* ctx, int32_t n_jobs, const double* const* d, const int32_t* n, const double* threshold,
                                       const double* weight, int32_t* best_idx) {
  if (!ctx || n_jobs <= 0 || n_jobs > VISO_MAX_BATCH || !d || !n || !threshold || !weight || !best_idx)
    return ctx ? visocu_set_error(ctx, VISOCU_EINVAL, "bad best_plane arguments") : VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  std::vector<PlaneJob> hj(n_jobs);
  std::vector<size_t> o_d(n_jobs), o_s(n_jobs);
  size_t off = align_up(sizeof(PlaneJob) * n_jobs, 256);
  int maxn = 0;
  for (int j = 0; j < n_jobs; j++) {
    if (!d[j] || n[j] <= 0) return visocu_set_error(ctx, VISOCU_EINVAL, "bad best_plane job %d", j);
    o_d[j] = off; off += align_up((size_t)n[j] * 8, 256);
    if (n[j] > maxn) maxn = n[j];
  }
  const size_t up_bytes = off;
  for (int j = 0; j < n_jobs; j++) { o_s[j] = off; off += align_up((size_t)n[j] * 8, 256); }
  int rc = visocu_ensure_scratch(ctx, off);
  if (rc) return rc;
  if ((rc = visocu_ensure_pinned(ctx, off))) return rc;
  uint8_t* sb = (uint8_t*)ctx->scratch;
  uint8_t* pin = (uint8_t*)ctx->pinned;
  for (int j = 0; j < n_jobs; j++) {
    hj[j].d = (const double*)(sb + o_d[j]); hj[j].sums = (double*)(sb + o_s[j]);
    hj[j].threshold = threshold[j]; hj[j].weight = weight[j]; hj[j].n = n[j]; hj[j].pad = 0;
    memcpy(pin + o_d[j], d[j], (size_t)n[j] * 8);
  }
  memcpy(pin, hj.data(), sizeof(PlaneJob) * n_jobs);
  CU_COPY(ctx, sb, pin, up_bytes, cudaMemcpyHostToDevice);
  k_plane_sums<<<dim3((maxn + 7) / 8, n_jobs), 256, 0, ctx->stream>>>((const PlaneJob*)sb);
  CU_LAUNCH_CHECK(ctx);
  CU_COPY(ctx, pin + up_bytes, sb + up_bytes, off - up_bytes, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  for (int j = 0; j < n_jobs; j++) {
    // arg-max with the reference's rule: strictly larger wins, so the first maximum is kept; index 0 if no candidate
    const double* sums = (const double*)(pin + o_s[j]);
    double best_sum = 0;
    int32_t best = 0;
    for (int32_t i = 0; i < n[j]; i++)
      if (sums[i] > best_sum) { best_sum = sums[i]; best = i; }
    best_idx[j] = best;
  }
  return VISOCU_OK;
}

extern "C" int visocu_best_plane(visocu_ctx* ctx, const double* d, int32_t n, double threshold, double weight, int32_t* best_idx) {
  if (!ctx || !d || !best_idx || n <= 0) return ctx ? visocu_set_error(ctx, VISOCU_EINVAL, "bad best_plane arguments") : VISOCU_EINVAL;
  return visocu_best_plane_batch(ctx, 1, &d, &n, &threshold, &weight, best_idx);
}
