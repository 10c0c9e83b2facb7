// Stereo odometry motion estimate: 3-point RANSAC over Gauss-Newton fits and the final refinement on all inliers.
//
// What it reproduces (host/viso_stereo.cpp, which restates the reference viso_stereo.cpp:42-316):
//   back-projection ...... d = max(u1p - u2p, 0.0001f) in float, X, Y, Z in double
//   hypothesis k ......... Gauss-Newton from tr = 0 on the 12 rows of sample k, step 1, eps 1e-6, at most 22 updates
//   updateParameters ..... normal equations J^T J x = J^T r, solved by Matrix::solve (host/matrix.cpp:249-285:
//                          Gauss-Jordan, full pivoting, '>=' pivot rule, FAILED if |pivot| < 1e-20); a FAILED
//                          hypothesis is not scored
//   getInlier ............ unweighted sum over u1c, v1c, u2c, v2c of (observe - predict)^2 < threshold^2
//   winner ............... earliest hypothesis whose count is strictly greater than the running best (start 0)
//   final refinement ..... Gauss-Newton on all inliers of the winner (>= 6), eps 1e-8, at most 102 updates; ok only
//                          if it ends CONVERGED
//
// Design:
//   k_hyp     one thread per hypothesis.  The chain is short and strictly sequential (trig, 12 Jacobian rows, a 6x6
//             elimination with data-dependent pivots), so there is nothing to share between lanes; the normal
//             equations are accumulated row by row in registers, the elimination runs on the thread's own column of
//             shared memory (pivot rows and columns are dynamic indices, which registers cannot take).
//   k_score   one thread per match, hypotheses' R | t streamed through shared memory, counts by warp ballot and
//             integer shared / global atomics (order-independent, so deterministic) - the pattern of k_score in
//             ransac.cu.
//   k_finish  one CTA per job: arg-max, inlier mask, then the refinement.  Every update is a block reduction of the
//             21 + 6 sums of the normal equations over the inliers with a fixed tree (warp shuffles, then the warps'
//             partials in warp order): a call is bit-identical from run to run.
// Floating-point contract: FP64 throughout; nvcc contracts to FMA, so results agree with the host to rounding and are
// not bit-identical to it (the sums of the refinement are also ordered differently).
#include "visocu_internal.cuh"
#include <cstring>

namespace {

constexpr int HYP_THREADS = 64;
constexpr int SCORE_THREADS = 256;
constexpr int SCORE_TILE = 64;          // hypotheses staged in shared memory per scoring step
constexpr int FINISH_THREADS = 256;
constexpr int HYP_MAX_UPDATES = 22;     // viso_stereo.cpp:44-47: `iter++ > 20` after each update
constexpr int FINAL_MAX_UPDATES = 102;  // viso_stereo.cpp:57-61: `iter++ > 100`
constexpr double SOLVE_EPS = 1e-20;     // Matrix::solve default

struct StereoJob {
  const visocu_pmatch* m;   // N records
  const int32_t* samples;   // iters x 3
  double* tr_all;           // iters x 6
  double* Rt_all;           // iters x 12 (R row-major, then t)
  int32_t* counts;          // iters (-1 = Gauss-Newton failed)
  uint8_t* mask;            // N
  double* out;              // tr6 [0..5], then int32 ok, n_inliers, best_iter at byte 48
  int N;
};

struct Calib { double f, cu, cv, base, thr2; int iters, reweighting; };

enum { UPDATED = 0, FAILED = 1, CONVERGED = 2 };

// 3-D point of a match in the previous left camera (viso_stereo.cpp:30-35 here): the disparity in float
__device__ __forceinline__ void back_project(const visocu_pmatch& m, const Calib& c, double& X, double& Y, double& Z) {
  const float dd = __fsub_rn(m.u1p, m.u2p);
  const float d = dd < 0.0001f ? 0.0001f : dd;                        // std::max(dd, 0.0001f)
  X = ((double)m.u1p - c.cu) * c.base / (double)d;
  Y = ((double)m.v1p - c.cv) * c.base / (double)d;
  Z = c.f * c.base / (double)d;
}

// R = Rx(rx) Ry(ry) Rz(rz) (viso_stereo.cpp:116-119 here) and, if wanted, its derivatives w.r.t. the three angles
struct Pose { double R[9], dR[27], t[3]; };

__device__ __forceinline__ void make_pose(const double* tr, Pose& p, bool derivatives) {
  double sx, cx, sy, cy, sz, cz;
  sincos(tr[0], &sx, &cx); sincos(tr[1], &sy, &cy); sincos(tr[2], &sz, &cz);
  p.R[0] = +cy * cz;                p.R[1] = -cy * sz;                p.R[2] = +sy;
  p.R[3] = +sx * sy * cz + cx * sz; p.R[4] = -sx * sy * sz + cx * cz; p.R[5] = -sx * cy;
  p.R[6] = -cx * sy * cz + sx * sz; p.R[7] = +cx * sy * sz + sx * cz; p.R[8] = +cx * cy;
  p.t[0] = tr[3]; p.t[1] = tr[4]; p.t[2] = tr[5];
  if (!derivatives) return;
  double* D = p.dR;
  D[0] = 0;                         D[1] = 0;                         D[2] = 0;
  D[3] = +cx * sy * cz - sx * sz;   D[4] = -cx * sy * sz - sx * cz;   D[5] = -cx * cy;
  D[6] = +sx * sy * cz + cx * sz;   D[7] = -sx * sy * sz + cx * cz;   D[8] = -sx * cy;
  D += 9;
  D[0] = -sy * cz;                  D[1] = +sy * sz;                  D[2] = +cy;
  D[3] = +sx * cy * cz;             D[4] = -sx * cy * sz;             D[5] = +sx * sy;
  D[6] = -cx * cy * cz;             D[7] = +cx * cy * sz;             D[8] = -cx * sy;
  D += 9;
  D[0] = -cy * sz;                  D[1] = -cy * cz;                  D[2] = 0;
  D[3] = -sx * sy * sz + cx * cz;   D[4] = -sx * sy * cz - cx * sz;   D[5] = 0;
  D[6] = +cx * sy * sz + sx * cz;   D[7] = +cx * sy * cz - sx * sz;   D[8] = 0;
}

// Adds the four rows of one match to the normal equations: A (upper triangle, 21 entries row by row) and B
// (viso_stereo.cpp:88-99 and 130-161 here: the same expressions, rows in the order u1c, v1c, u2c, v2c).
template <class P>
__device__ __forceinline__ void accumulate(const P& p, const Calib& c, double Xp, double Yp, double Zp, const visocu_pmatch& m,
                                           double (&A)[21], double (&B)[6]) {
  const double X1c = p.R[0] * Xp + p.R[1] * Yp + p.R[2] * Zp + p.t[0];
  const double Y1c = p.R[3] * Xp + p.R[4] * Yp + p.R[5] * Zp + p.t[1];
  const double Z1c = p.R[6] * Xp + p.R[7] * Yp + p.R[8] * Zp + p.t[2];
  const double o[4] = {(double)m.u1c, (double)m.v1c, (double)m.u2c, (double)m.v2c};
  double weight = 1.0;
  if (c.reweighting) weight = 1.0 / (fabs(o[0] - c.cu) / fabs(c.cu) + 0.05);
  const double X2c = X1c - c.base;
  const double zz = Z1c * Z1c;
  // derivative of the point in current left coordinates w.r.t. the three angles (the translations give unit vectors)
  double Pd[3][3];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    const double* D = p.dR + 9 * j;
    Pd[j][0] = D[0] * Xp + D[1] * Yp + D[2] * Zp;
    Pd[j][1] = D[3] * Xp + D[4] * Yp + D[5] * Zp;
    Pd[j][2] = D[6] * Xp + D[7] * Yp + D[8] * Zp;
  }
  const double pr[4] = {c.f * X1c / Z1c + c.cu, c.f * Y1c / Z1c + c.cv, c.f * X2c / Z1c + c.cu, c.f * Y1c / Z1c + c.cv};
#pragma unroll
  for (int r = 0; r < 4; r++) {
    // row r: u1c (X1c, Xd), v1c (Y1c, Yd), u2c (X2c, Xd), v2c (Y1c, Yd)
    const int ax = (r & 1) ? 1 : 0;
    const double Pc = r == 0 ? X1c : (r == 2 ? X2c : Y1c);
    double J[6];
#pragma unroll
    for (int j = 0; j < 6; j++) {
      const double Ad = j < 3 ? Pd[j][ax] : (double)(j - 3 == ax);
      const double Zd = j < 3 ? Pd[j][2] : (double)(j == 5);
      J[j] = weight * c.f * (Ad * Z1c - Pc * Zd) / zz;
    }
    const double res = weight * (o[r] - pr[r]);
    int k = 0;
#pragma unroll
    for (int a = 0; a < 6; a++) {
#pragma unroll
      for (int b = a; b < 6; b++) A[k++] += J[a] * J[b];
      B[a] += J[a] * res;
    }
  }
}

// getInlier (viso_stereo.cpp:69-81 here): unweighted squared reprojection error over the four coordinates
__device__ __forceinline__ bool is_inlier(const double* Rt, const Calib& c, double Xp, double Yp, double Zp, const float4 o) {
  const double X1c = Rt[0] * Xp + Rt[1] * Yp + Rt[2] * Zp + Rt[9];
  const double Y1c = Rt[3] * Xp + Rt[4] * Yp + Rt[5] * Zp + Rt[10];
  const double Z1c = Rt[6] * Xp + Rt[7] * Yp + Rt[8] * Zp + Rt[11];
  const double X2c = X1c - c.base;
  const double p0 = c.f * X1c / Z1c + c.cu, p1 = c.f * Y1c / Z1c + c.cv, p2 = c.f * X2c / Z1c + c.cu, p3 = c.f * Y1c / Z1c + c.cv;
  double e = 0;
  double q = (double)o.x - p0; e += q * q;
  q = (double)o.y - p1; e += q * q;
  q = (double)o.z - p2; e += q * q;
  q = (double)o.w - p3; e += q * q;
  return e < c.thr2;
}

// Matrix::solve restated (host/matrix.cpp:249-285) for the 6x6 system A x = b, A and b at stride `s` (element (r, k) of
// A at A[(6 r + k) s]).  The solution replaces b; A is destroyed.  The final column unscrambling of the reference only
// concerns the inverse left in A, not the solution, and is omitted.  `used` keeps the reference's counters (4 bits per
// column): with NaN entries no pivot passes the '>=' test and column 0 is chosen again, so a counter can exceed 1.
__device__ __forceinline__ bool gj_solve6(double* A, double* b, int s) {
  unsigned used = 0;
  for (int step = 0; step < 6; step++) {
    double big = 0;
    int pr = 0, pc = 0;
    for (int r = 0; r < 6; r++) {
      if (((used >> (4 * r)) & 15u) == 1u) continue;
      for (int cc = 0; cc < 6; cc++)
        if (((used >> (4 * cc)) & 15u) == 0u && fabs(A[(6 * r + cc) * s]) >= big) { big = fabs(A[(6 * r + cc) * s]); pr = r; pc = cc; }
    }
    used += 1u << (4 * pc);
    if (pr != pc) {
      for (int k = 0; k < 6; k++) { const double x = A[(6 * pr + k) * s]; A[(6 * pr + k) * s] = A[(6 * pc + k) * s]; A[(6 * pc + k) * s] = x; }
      const double x = b[pr * s]; b[pr * s] = b[pc * s]; b[pc * s] = x;
    }
    if (fabs(A[(6 * pc + pc) * s]) < SOLVE_EPS) return false;
    const double piv = 1.0 / A[(6 * pc + pc) * s];
    A[(6 * pc + pc) * s] = 1;
    for (int k = 0; k < 6; k++) A[(6 * pc + k) * s] *= piv;
    b[pc * s] *= piv;
    for (int r = 0; r < 6; r++) {
      if (r == pc) continue;
      const double f = A[(6 * r + pc) * s];
      A[(6 * r + pc) * s] = 0;
      for (int k = 0; k < 6; k++) A[(6 * r + k) * s] -= A[(6 * pc + k) * s] * f;
      b[r * s] -= b[pc * s] * f;
    }
  }
  return true;
}

// normal equations (21 + 6 sums) -> solve -> tr update (updateParameters, viso_stereo.cpp:83-107 here)
__device__ __forceinline__ int gn_update(const double (&A)[21], const double (&B)[6], double* sA, double* sb, int s, double* tr,
                                         double eps) {
  int k = 0;
#pragma unroll
  for (int a = 0; a < 6; a++) {
#pragma unroll
    for (int b = a; b < 6; b++) { sA[(6 * a + b) * s] = A[k]; sA[(6 * b + a) * s] = A[k]; k++; }
    sb[a * s] = B[a];
  }
  if (!gj_solve6(sA, sb, s)) return FAILED;
  bool converged = true;
#pragma unroll
  for (int m = 0; m < 6; m++) {
    const double x = sb[m * s];
    tr[m] += 1.0 * x;
    if (fabs(x) > eps) converged = false;
  }
  return converged ? CONVERGED : UPDATED;
}

__global__ void __launch_bounds__(HYP_THREADS) k_hyp(const StereoJob* jobs, Calib c) {
  const StereoJob& J = jobs[blockIdx.y];
  const int h = blockIdx.x * HYP_THREADS + threadIdx.x;
  __shared__ double sA[36 * HYP_THREADS], sb[6 * HYP_THREADS];
  if (h >= c.iters) return;
  double P[3][3];
  visocu_pmatch M[3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    M[k] = J.m[J.samples[3 * h + k]];
    back_project(M[k], c, P[k][0], P[k][1], P[k][2]);
  }
  double tr[6] = {0, 0, 0, 0, 0, 0};
  int res = UPDATED;
  for (int it = 0; it < HYP_MAX_UPDATES && res == UPDATED; it++) {
    Pose p;
    make_pose(tr, p, true);
    double A[21], B[6];
#pragma unroll
    for (int k = 0; k < 21; k++) A[k] = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) B[k] = 0;
#pragma unroll
    for (int k = 0; k < 3; k++) accumulate(p, c, P[k][0], P[k][1], P[k][2], M[k], A, B);
    res = gn_update(A, B, sA + threadIdx.x, sb + threadIdx.x, HYP_THREADS, tr, 1e-6);
  }
  Pose p;
  make_pose(tr, p, false);
#pragma unroll
  for (int k = 0; k < 6; k++) J.tr_all[(size_t)h * 6 + k] = tr[k];
#pragma unroll
  for (int k = 0; k < 9; k++) J.Rt_all[(size_t)h * 12 + k] = p.R[k];
#pragma unroll
  for (int k = 0; k < 3; k++) J.Rt_all[(size_t)h * 12 + 9 + k] = p.t[k];
  J.counts[h] = res == FAILED ? -1 : 0;
}

__device__ __forceinline__ float4 observed(const visocu_pmatch& m) { return make_float4(m.u1c, m.v1c, m.u2c, m.v2c); }

__global__ void __launch_bounds__(SCORE_THREADS) k_score(const StereoJob* jobs, Calib c) {
  const StereoJob& J = jobs[blockIdx.z];
  if ((int)blockIdx.x * SCORE_THREADS >= J.N) return;
  __shared__ double sRt[SCORE_TILE * 12];
  __shared__ int sFail[SCORE_TILE], sCnt[SCORE_TILE];
  const int i = blockIdx.x * SCORE_THREADS + threadIdx.x;
  const bool live = i < J.N;
  double X = 0, Y = 0, Z = 0;
  float4 o = make_float4(0, 0, 0, 0);
  if (live) { const visocu_pmatch m = J.m[i]; back_project(m, c, X, Y, Z); o = observed(m); }
  for (int h0 = blockIdx.y * SCORE_TILE; h0 < c.iters; h0 += gridDim.y * SCORE_TILE) {
    const int nh = min(SCORE_TILE, c.iters - h0);
    __syncthreads();
    for (int k = threadIdx.x; k < nh * 12; k += SCORE_THREADS) sRt[k] = J.Rt_all[(size_t)h0 * 12 + k];
    if (threadIdx.x < nh) { sFail[threadIdx.x] = J.counts[h0 + threadIdx.x] < 0; sCnt[threadIdx.x] = 0; }
    __syncthreads();
    for (int h = 0; h < nh; h++) {
      if (sFail[h]) continue;                                         // FAILED: not scored (uniform branch)
      const bool in = live && is_inlier(sRt + 12 * h, c, X, Y, Z, o);
      const unsigned b = __ballot_sync(0xFFFFFFFFu, in);
      if ((threadIdx.x & 31) == 0 && b) atomicAdd(&sCnt[h], __popc(b));
    }
    __syncthreads();
    if (threadIdx.x < nh && sCnt[threadIdx.x]) atomicAdd(&J.counts[h0 + threadIdx.x], sCnt[threadIdx.x]);
  }
}

// Sum of x over the block, the same value on every thread; the tree is fixed (deterministic)
__device__ __forceinline__ void block_sums(double* v, int n, double* red, int tid) {
  const int lane = tid & 31, wid = tid >> 5;
  for (int k = 0; k < n; k++) {
    double x = v[k];
#pragma unroll
    for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, o);
    if (lane == 0) red[k * (FINISH_THREADS / 32) + wid] = x;
  }
  __syncthreads();
  for (int k = 0; k < n; k++) {
    double s = 0;
#pragma unroll
    for (int w = 0; w < FINISH_THREADS / 32; w++) s += red[k * (FINISH_THREADS / 32) + w];
    v[k] = s;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(FINISH_THREADS) k_finish(const StereoJob* jobs, Calib c) {
  const StereoJob& J = jobs[blockIdx.x];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  __shared__ long long s_best[FINISH_THREADS / 32];
  __shared__ int s_cnt[FINISH_THREADS / 32];
  __shared__ double s_red[27 * (FINISH_THREADS / 32)];
  __shared__ double s_Rt[12], s_tr[6], s_A[36], s_b[6];
  __shared__ Pose s_pose;
  __shared__ int s_bestk, s_res;

  // ---- arg-max: largest count, earliest hypothesis on ties; a count of 0 (or a failed fit) never wins
  long long key = 0;
  for (int k = tid; k < c.iters; k += FINISH_THREADS) {
    const int n = J.counts[k];
    const long long cand = n > 0 ? ((long long)n << 32) | (unsigned)(0x7FFFFFFF - k) : 0;
    key = cand > key ? cand : key;
  }
  for (int o = 16; o; o >>= 1) { const long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o); key = other > key ? other : key; }
  if (lane == 0) s_best[wid] = key;
  __syncthreads();
  if (tid == 0) {
    long long b = 0;
    for (int k = 0; k < FINISH_THREADS / 32; k++) b = s_best[k] > b ? s_best[k] : b;
    const int bestk = b == 0 ? -1 : 0x7FFFFFFF - (int)(b & 0xFFFFFFFF);
    s_bestk = bestk;
    for (int k = 0; k < 12; k++) s_Rt[k] = bestk >= 0 ? J.Rt_all[(size_t)bestk * 12 + k] : 0.0;
    for (int k = 0; k < 6; k++) s_tr[k] = bestk >= 0 ? J.tr_all[(size_t)bestk * 6 + k] : 0.0;
  }
  __syncthreads();
  const int bestk = s_bestk;

  // ---- inlier mask of the winner (none without a winner)
  int cnt = 0;
  for (int i = tid; i < J.N; i += FINISH_THREADS) {
    bool in = false;
    if (bestk >= 0) {
      const visocu_pmatch m = J.m[i];
      double X, Y, Z;
      back_project(m, c, X, Y, Z);
      in = is_inlier(s_Rt, c, X, Y, Z, observed(m));
    }
    J.mask[i] = (uint8_t)in;
    cnt += in;
  }
  for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, o);
  if (lane == 0) s_cnt[wid] = cnt;
  __syncthreads();
  int n_inl = 0;
  for (int w = 0; w < FINISH_THREADS / 32; w++) n_inl += s_cnt[w];

  // ---- final refinement on all inliers (viso_stereo.cpp:54-66 here)
  int ok = 0;
  if (n_inl >= 6) {
    for (int it = 0; it < FINAL_MAX_UPDATES; it++) {
      if (tid == 0) make_pose(s_tr, s_pose, true);
      __syncthreads();
      double A[21], B[6];
#pragma unroll
      for (int k = 0; k < 21; k++) A[k] = 0;
#pragma unroll
      for (int k = 0; k < 6; k++) B[k] = 0;
      for (int i = tid; i < J.N; i += FINISH_THREADS) {
        if (!J.mask[i]) continue;
        const visocu_pmatch m = J.m[i];
        double X, Y, Z;
        back_project(m, c, X, Y, Z);
        accumulate(s_pose, c, X, Y, Z, m, A, B);
      }
      double v[27];
#pragma unroll
      for (int k = 0; k < 21; k++) v[k] = A[k];
#pragma unroll
      for (int k = 0; k < 6; k++) v[21 + k] = B[k];
      block_sums(v, 27, s_red, tid);
      if (tid == 0) {
#pragma unroll
        for (int k = 0; k < 21; k++) A[k] = v[k];
#pragma unroll
        for (int k = 0; k < 6; k++) B[k] = v[21 + k];
        s_res = gn_update(A, B, s_A, s_b, 1, s_tr, 1e-8);
      }
      __syncthreads();
      if (s_res != UPDATED) break;
    }
    ok = s_res == CONVERGED;
  }
  if (tid == 0) {
    for (int k = 0; k < 6; k++) J.out[k] = ok ? s_tr[k] : 0.0;
    int32_t* w = (int32_t*)(J.out + 6);
    w[0] = ok; w[1] = n_inl; w[2] = bestk;
  }
}

}  // namespace

extern "C" int visocu_stereo_motion(visocu_ctx* ctx, int32_t n_jobs, const visocu_pmatch* const* matches, const int32_t* N,
                                    const int32_t* const* samples, const visocu_stereo_params* p, double* tr6, int32_t* ok,
                                    uint8_t* const* inlier_mask, int32_t* n_inliers, int32_t* best_iter,
                                    int32_t* const* counts, double* const* tr_all) {
  if (!ctx) return VISOCU_EINVAL;
  if (n_jobs <= 0 || !matches || !N || !samples || !p || !tr6 || !ok || p->ransac_iters <= 0)
    return visocu_set_error(ctx, VISOCU_EINVAL, "bad stereo_motion arguments");
  const int iters = p->ransac_iters;
  // every job is checked before anything is enqueued or written
  for (int j = 0; j < n_jobs; j++) {
    const int n = N[j];
    if (n < 6 || !matches[j] || !samples[j]) return visocu_set_error(ctx, VISOCU_EINVAL, "stereo_motion job %d: need >= 6 matches", j);
    for (int k = 0; k < iters * 3; k++)
      if (samples[j][k] < 0 || samples[j][k] >= n) return visocu_set_error(ctx, VISOCU_EINVAL, "stereo_motion job %d: sample index out of range", j);
  }
  const Calib c{p->f, p->cu, p->cv, p->base, p->inlier_threshold * p->inlier_threshold, iters, p->reweighting};
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  for (int start = 0; start < n_jobs; start += VISO_MAX_BATCH) {
    const int nb = n_jobs - start < VISO_MAX_BATCH ? n_jobs - start : VISO_MAX_BATCH;
    std::vector<StereoJob> hj(nb);
    // Upload: job descriptors, match records, sample tables (ONE copy).  Read-back: a 64-byte result slot per job
    // followed by the masks (ONE copy).  Per-hypothesis tables stay on the device unless a test asks for them.
    std::vector<size_t> o_m(nb), o_smp(nb), o_mask(nb), o_hyp(nb);
    size_t off = align_up(sizeof(StereoJob) * nb, 256);
    for (int j = 0; j < nb; j++) {
      const int n = N[start + j];
      hj[j].N = n;
      o_m[j] = off; off += align_up((size_t)n * sizeof(visocu_pmatch), 256);
      o_smp[j] = off; off += align_up((size_t)iters * 12, 256);
    }
    const size_t up_bytes = off;
    const size_t o_back = off;
    off += (size_t)64 * nb;
    for (int j = 0; j < nb; j++) { o_mask[j] = off; off += align_up((size_t)hj[j].N, 16); }
    const size_t back_bytes = off - o_back;
    off = align_up(off, 256);
    const size_t hyp_stride = align_up((size_t)iters * (6 + 12) * 8 + (size_t)iters * 4, 256);
    for (int j = 0; j < nb; j++) { o_hyp[j] = off; off += hyp_stride; }
    int rc = visocu_ensure_scratch(ctx, off);
    if (rc) return rc;
    const size_t p_back = align_up(up_bytes, 256);
    if ((rc = visocu_ensure_pinned(ctx, p_back + back_bytes))) return rc;
    uint8_t* sb = (uint8_t*)ctx->scratch;
    uint8_t* pin = (uint8_t*)ctx->pinned;
    for (int j = 0; j < nb; j++) {
      const int n = hj[j].N;
      uint8_t* hyp = sb + o_hyp[j];
      hj[j].m = (const visocu_pmatch*)(sb + o_m[j]); hj[j].samples = (const int32_t*)(sb + o_smp[j]);
      hj[j].tr_all = (double*)hyp; hj[j].Rt_all = (double*)(hyp + (size_t)iters * 48);
      hj[j].counts = (int32_t*)(hyp + (size_t)iters * 144);
      hj[j].mask = sb + o_mask[j]; hj[j].out = (double*)(sb + o_back + (size_t)64 * j);
      memcpy(pin + o_m[j], matches[start + j], (size_t)n * sizeof(visocu_pmatch));
      memcpy(pin + o_smp[j], samples[start + j], (size_t)iters * 12);
    }
    memcpy(pin, hj.data(), sizeof(StereoJob) * nb);
    CU_COPY(ctx, sb, pin, up_bytes, cudaMemcpyHostToDevice);
    const StereoJob* dj = (const StereoJob*)sb;
    int maxN = 0;
    for (int j = 0; j < nb; j++) maxN = hj[j].N > maxN ? hj[j].N : maxN;
    k_hyp<<<dim3((iters + HYP_THREADS - 1) / HYP_THREADS, nb), HYP_THREADS, 0, ctx->stream>>>(dj, c);
    CU_LAUNCH_CHECK(ctx);
    const int ty = (iters + SCORE_TILE - 1) / SCORE_TILE;
    k_score<<<dim3((maxN + SCORE_THREADS - 1) / SCORE_THREADS, ty, nb), SCORE_THREADS, 0, ctx->stream>>>(dj, c);
    CU_LAUNCH_CHECK(ctx);
    k_finish<<<nb, FINISH_THREADS, 0, ctx->stream>>>(dj, c);
    CU_LAUNCH_CHECK(ctx);
    CU_COPY(ctx, pin + p_back, sb + o_back, back_bytes, cudaMemcpyDeviceToHost);
    for (int j = 0; j < nb; j++) {                  // optional per-hypothesis tables (tests): straight to the caller
      if (counts && counts[start + j])
        CU_COPY(ctx, counts[start + j], hj[j].counts, (size_t)iters * 4, cudaMemcpyDeviceToHost);
      if (tr_all && tr_all[start + j])
        CU_COPY(ctx, tr_all[start + j], hj[j].tr_all, (size_t)iters * 48, cudaMemcpyDeviceToHost);
    }
    CU_TRY(ctx, visocu_stream_wait(ctx));
    for (int j = 0; j < nb; j++) {
      const uint8_t* slot = pin + p_back + (size_t)64 * j;
      memcpy(tr6 + 6 * (size_t)(start + j), slot, 48);
      const int32_t* w = (const int32_t*)(slot + 48);
      ok[start + j] = w[0];
      if (n_inliers) n_inliers[start + j] = w[1];
      if (best_iter) best_iter[start + j] = w[2];
      if (inlier_mask && inlier_mask[start + j]) memcpy(inlier_mask[start + j], pin + p_back + (o_mask[j] - o_back), (size_t)hj[j].N);
    }
  }
  return VISOCU_OK;
}
