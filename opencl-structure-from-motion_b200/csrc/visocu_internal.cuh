// Internal declarations shared by the CUDA translation units behind include/visocu.h.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <functional>
#include <string>
#include <vector>
#include "visocu.h"

#define VISO_MARGIN 6            // Matcher::margin, reference matcher.cpp:56
#define VISO_MAX_BATCH 128       // frames / jobs per launch (larger batches are split by the host code)

// Device pointers of one frame slot (everything Matcher keeps per image in its ring buffer, matcher.h:232-241).
struct FrameDev {
  uint8_t *img, *half, *du, *dv, *du_full, *dv_full;
  uint32_t* codes[2];      // per NMS cell: 4 bytes (one per class) = (di<<4|dj) of the kept extremum or 0xFF
  int32_t*  blk[2];        // per 512-cell chunk: number of records it emits (ordered compaction)
  int32_t*  rec[2];        // 12 x int32 records, pass 0 = sparse, 1 = dense
  int32_t*  bin_start[2];  // 4*ub*vb + 1 offsets into bin_ent
  int32_t*  bin_cursor[2]; // scratch for the scatter
  int2*     bin_ent[2];    // (u | v<<16, feature index), grouped by bin
  int32_t*  counts;        // [0..1] record counts, [2] overflow flag
};

struct Geometry {
  int w, h, bpl;           // full resolution, bpl = 16-byte stride (matcher.cpp:158-160)
  int wm, hm, bplm;        // matching resolution (== full unless half_resolution, matcher.cpp:630-634)
  int half, scale;
  int first_pass;          // 0 if multi_stage (sparse + dense) else 1 (dense only)
  int n[2], ncx[2], ncy[2], cap[2];
  int tau;
  int binsize, ub, vb, nbins;
  int radius, disp_tol;
};

struct SlotList { int n; int s[VISO_MAX_BATCH]; };

#define VISO_TILE_LEVELS 3
// one tile configuration of the fused filter+NMS kernel (csrc/features.cu: TileCfg) and its TMA descriptor
struct visocu_tile { alignas(64) CUtensorMap tmap; alignas(64) CUtensorMap tmap_full; alignas(8) unsigned char cfg[160]; void* tables = nullptr; };

// state of a matching call whose outlier removal runs on the second stream (visocu_match_deferred / _collect)
struct visocu_deferred {
  bool pending = false;
  int nb = 0;
  uint8_t* pin_words = nullptr; uint8_t* pin_lists = nullptr;   // pinned: 16 result words per job, staged lists
  const uint8_t* dev_lists = nullptr; size_t ostride = 0;       // device: survivor lists, uniform stride
  const int32_t* dev_words = nullptr;                           // device: the 16 result words per job
  const void* dev_jobs = nullptr;                               // device: the MatchJob array of the pass
};

// Everything a step in flight needs for itself: a context has VISO_LANES of these, so that several push + match steps
// (of the same sequences, on consecutive frames) can be in flight at once without sharing a stream, scratch memory or
// a result area.  visocu_set_lane swaps one of them into the context's working fields of the same names.
#define VISO_LANES 6            // 0: default; 0..3: pipelined steps (lane = step & 3); 4: synchronous fall-backs and odometry calls
struct visocu_graph { cudaGraphExec_t exec = nullptr; uint64_t key = 0; int seen = 0; };
struct visocu_lane {
  cudaStream_t stream = nullptr;
  void* scratch = nullptr; size_t scratch_bytes = 0;
  void* scratch2 = nullptr; size_t scratch2_bytes = 0;
  void* pinned = nullptr; size_t pinned_bytes = 0;
  void* pinned2 = nullptr; size_t pinned2_bytes = 0;
  visocu_deferred part[2];
  void* d_ranges = nullptr; size_t d_ranges_bytes = 0; void* pin_ranges = nullptr;
  void* deliver = nullptr; void* deliver_dev = nullptr; size_t deliver_bytes = 0;
  void* deliver2 = nullptr; size_t deliver2_bytes = 0;
  volatile uint32_t* wait_flag = nullptr; void* wait_flag_dev = nullptr; uint32_t wait_seq = 0;
  int32_t* counts_stage = nullptr;
  uint8_t* img_stage = nullptr; size_t img_stage_bytes = 0;
  const uint8_t** src_table = nullptr; const uint8_t** src_table_pin = nullptr;   // image pointers of a push (device / pinned copy)
  cudaEvent_t ev_push = nullptr;       // recorded behind the feature kernels of the lane's last push
  visocu_graph g_push, g_match;        // the two halves of a step, captured once their shape repeats
  bool fused_pending = false; int fused_n = 0; bool fused_ranges = false, fused_list1 = false; uint32_t fused_seq = 0;
  std::vector<visocu_quad> fused_jobs;  // the submitted, not yet collected fused call of the lane
  bool created = false;
};

struct visocu_ctx {
  int device = 0;
  int sm_count = 0, cc_major = 0, cc_minor = 0;
  char name[64] = {0};
  cudaStream_t stream = nullptr;
  int lane = 0;                      // the lane whose resources are in the working fields below
  visocu_lane lanes[VISO_LANES];     // parked lanes (the entry of the current lane is stale)
  int use_graphs = 1;                // VISOCU_GRAPHS=0: always enqueue kernel by kernel
  int in_step = 0;                   // > 0 while a (replayable) step is being enqueued: buffer growth does not drop the graphs
  bool fused_pending = false; int fused_n = 0; bool fused_ranges = false, fused_list1 = false; uint32_t fused_seq = 0;   // per lane, see VISO_LANE_FIELDS
  std::vector<visocu_quad> fused_jobs;
  int ro_bound_seen[2] = {0, 0};
  int ro_bound[2] = {-1, -1};        // longest match list seen per pass (shared-memory size of the outlier kernel in lazy mode)
  int ro_threads = 0;                // outlier kernel: threads per list, 0 = by batch size (VISOCU_RO_THREADS, read by visocu_configure)
  int ro_warp = 1;                   // outlier kernel: a warp per top-level merge; 0 = one thread (VISOCU_RO_WARP)
  const uint8_t** src_table = nullptr; const uint8_t** src_table_pin = nullptr;
  cudaEvent_t ev_push = nullptr;
  visocu_graph g_push, g_match;
  visocu_deferred part[2];           // the two passes of a fused call (visocu_match_fused)
  void* deliver2 = nullptr; size_t deliver2_bytes = 0;        // pinned landing area of the lists when they are too large for that
  void* deliver = nullptr; void* deliver_dev = nullptr; size_t deliver_bytes = 0;     // mapped pinned memory the last kernel of a fused call writes the results to
  void* d_ranges = nullptr; size_t d_ranges_bytes = 0; void* pin_ranges = nullptr;   // prior ranges computed on the device between the passes
  void* scratch2 = nullptr; size_t scratch2_bytes = 0;
  void* pinned2 = nullptr;  size_t pinned2_bytes = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  volatile uint32_t* wait_flag = nullptr; void* wait_flag_dev = nullptr; uint32_t wait_seq = 0;   // see visocu_stream_wait
  cudaEvent_t ev_sync = nullptr;     // blocking-sync event: host threads sleep instead of spinning while the GPU works
  std::string err;
  bool configured = false;
  visocu_params param{};
  Geometry g{};
  int n_frames = 0;
  void* pool = nullptr;
  size_t pool_bytes = 0;
  std::vector<FrameDev> frames_h;
  FrameDev* frames_d = nullptr;
  std::vector<int32_t> h_counts;     // 2 per frame, host mirror (valid after a push that synchronised)
  std::vector<uint8_t> frame_valid;
  // scratch for matching / ransac, grown on demand
  void* scratch = nullptr; size_t scratch_bytes = 0;
  void* pinned = nullptr;  size_t pinned_bytes = 0;
  int32_t* counts_stage = nullptr;   // device: 4 int32 per frame of the last feature launch (one read-back per push)
  uint8_t* img_stage = nullptr; size_t img_stage_bytes = 0;   // contiguous landing area for host images
  uint64_t launches = 0;
  visocu_tile tiles[VISO_TILE_LEVELS];   // tile configurations, largest first (visocu_make_tensor_map)
  int n_tiles = 0;
  size_t frame_stride = 0;           // bytes between the pool blocks of consecutive frame slots
  int use_tma = 0;
  int fused_half = 0;                // half-resolution mode runs as one fused kernel (full-resolution tile staged by TMA)
  int pinv_ready = 0;                // paraboloid pseudo-inverse uploaded to constant memory (sub-pixel refinement)
  uint64_t h2d_bytes = 0, d2h_bytes = 0;   // host<->device traffic issued by this context
  int profile = 0;                   // time the fused filter+NMS launches with events (visocu_profile)
  cudaEvent_t pev0 = nullptr, pev1 = nullptr;
  double filter_ms = 0; uint64_t filter_launches = 0, filter_frames = 0;
  uint64_t* d_stats = nullptr;       // [0] SAD candidates, [1] entries scanned
  uint64_t h_stats[2] = {0, 0};
  uint64_t ro_node_calls = 0, ro_nodes = 0;   // visocu_delaunay_subtrees: large lists, nodes built for them
  uint64_t ro_ns[4] = {0, 0, 0, 0}, ro_jobs = 0, ro_declined = 0, ro_reason[4] = {0, 0, 0, 0}, ro_declined_n = 0;   // device outlier removal: phase times (VISOCU_RO_STATS)
  std::vector<visocu_recon_store*> stores;   // device point stores alive on this context (csrc/recon_store.cu)
  // rectification maps (csrc/rectify.cu): per camera 2 int32 per output pixel, on the device and a host copy
  int rect_n = 0, rect_src_w = 0, rect_src_h = 0;
  int2* rect_map[2] = {nullptr, nullptr};
  std::vector<int32_t> rect_host[2];
};

int visocu_set_error(visocu_ctx* ctx, int code, const char* fmt, ...);
cudaError_t visocu_stream_wait(visocu_ctx* ctx);                 // enqueue a completion word on the lane's stream and wait for it
cudaError_t visocu_stream_signal(visocu_ctx* ctx, uint32_t* seq_out);
cudaError_t visocu_stream_wait_seq(visocu_ctx* ctx, uint32_t seq);
void visocu_drop_graphs(visocu_ctx* ctx);
void visocu_drop_lane_graphs(visocu_ctx* ctx);               // of the current lane
int visocu_use_lane(visocu_ctx* ctx, int lane);                  // swap the lane's resources into the working fields
int visocu_ensure_scratch(visocu_ctx* ctx, size_t bytes);
int visocu_ensure_pinned(visocu_ctx* ctx, size_t bytes);
int visocu_run_or_replay(visocu_ctx* ctx, visocu_graph& g, uint64_t key, const std::function<int()>& enqueue);

#define CU_TRY(ctx, expr)                                                                        \
  do {                                                                                           \
    cudaError_t e__ = (expr);                                                                    \
    if (e__ != cudaSuccess)                                                                      \
      return visocu_set_error((ctx), VISOCU_ECUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr, \
                              cudaGetErrorString(e__));                                          \
  } while (0)

// async copy on the context's stream with byte accounting (bench.py reports h2d / d2h bytes per step)
#define CU_COPY(ctx, dst, src, bytes, kind)                                                   \
  do {                                                                                        \
    if ((kind) == cudaMemcpyHostToDevice) (ctx)->h2d_bytes += (uint64_t)(bytes);               \
    else if ((kind) == cudaMemcpyDeviceToHost) (ctx)->d2h_bytes += (uint64_t)(bytes);          \
    CU_TRY((ctx), cudaMemcpyAsync((dst), (src), (bytes), (kind), (ctx)->stream));             \
  } while (0)

#define CU_LAUNCH_CHECK(ctx)                  \
  do {                                        \
    (ctx)->launches++;                        \
    CU_TRY((ctx), cudaGetLastError());        \
  } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Matrix::solve restated (host/matrix.cpp:249-285) for the N x N system A x = b (N <= 8), A and b at stride `s` (element
// (r, k) of A at A[(N r + k) s]).  The solution replaces b; A is destroyed.  The final column unscrambling of the reference
// only concerns the inverse left in A, not the solution, and is omitted.  `used` keeps the reference's counters (4 bits per
// column): with NaN entries no pivot passes the '>=' test and column 0 is chosen again, so a counter can exceed 1.
template <int N>
__device__ __forceinline__ bool gj_solve(double* A, double* b, int s, double eps) {
  unsigned used = 0;
  for (int step = 0; step < N; step++) {
    double big = 0;
    int pr = 0, pc = 0;
    for (int r = 0; r < N; r++) {
      if (((used >> (4 * r)) & 15u) == 1u) continue;
      for (int cc = 0; cc < N; cc++)
        if (((used >> (4 * cc)) & 15u) == 0u && fabs(A[(N * r + cc) * s]) >= big) { big = fabs(A[(N * r + cc) * s]); pr = r; pc = cc; }
    }
    used += 1u << (4 * pc);
    if (pr != pc) {
      for (int k = 0; k < N; k++) { const double x = A[(N * pr + k) * s]; A[(N * pr + k) * s] = A[(N * pc + k) * s]; A[(N * pc + k) * s] = x; }
      const double x = b[pr * s]; b[pr * s] = b[pc * s]; b[pc * s] = x;
    }
    if (fabs(A[(N * pc + pc) * s]) < eps) return false;
    const double piv = 1.0 / A[(N * pc + pc) * s];
    A[(N * pc + pc) * s] = 1;
    for (int k = 0; k < N; k++) A[(N * pc + k) * s] *= piv;
    b[pc * s] *= piv;
    for (int r = 0; r < N; r++) {
      if (r == pc) continue;
      const double f = A[(N * r + pc) * s];
      A[(N * r + pc) * s] = 0;
      for (int k = 0; k < N; k++) A[(N * r + k) * s] -= A[(N * pc + k) * s] * f;
      b[r * s] -= b[pc * s] * f;
    }
  }
  return true;
}

// Null vector of a 4x4 system of rank 3 (the linear triangulation of two views) by a one-sided Jacobi in registers, in
// place of Matrix::svd: g[c][r] = column c of the matrix; X receives the right singular vector of the smallest singular
// value (unit length, sign arbitrary).  g is destroyed.
__device__ __forceinline__ void jacobi_null_vector4(double (&g)[4][4], double (&X)[4]) {
  double v[4][4];
#pragma unroll
  for (int c = 0; c < 4; c++)
#pragma unroll
    for (int r = 0; r < 4; r++) v[c][r] = r == c ? 1.0 : 0.0;
  double total = 0;
#pragma unroll
  for (int c = 0; c < 4; c++)
#pragma unroll
    for (int k = 0; k < 4; k++) total = fma(g[c][k], g[c][k], total);
  const double tiny = 1e-28 * total;      // columns this small are numerically null (J has rank 3): leave them alone
  for (int sweep = 0; sweep < 40; sweep++) {
    bool rotated = false;
#pragma unroll
    for (int p = 0; p < 3; p++)
#pragma unroll
      for (int q = p + 1; q < 4; q++) {
        double alpha = 0, beta = 0, gamma = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) { alpha = fma(g[p][k], g[p][k], alpha); beta = fma(g[q][k], g[q][k], beta); gamma = fma(g[p][k], g[q][k], gamma); }
        if (alpha > tiny && beta > tiny && fabs(gamma) > 1e-15 * sqrt(alpha * beta)) {
          const double zeta = (beta - alpha) / (2.0 * gamma);
          const double t = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
          const double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
#pragma unroll
          for (int k = 0; k < 4; k++) {
            const double a = g[p][k], b = g[q][k];
            g[p][k] = c * a - s * b; g[q][k] = s * a + c * b;
            const double va = v[p][k], vb = v[q][k];
            v[p][k] = c * va - s * vb; v[q][k] = s * va + c * vb;
          }
          rotated = true;
        }
      }
    if (!rotated) break;
  }
  double nrm[4];
#pragma unroll
  for (int c = 0; c < 4; c++) { nrm[c] = 0; for (int k = 0; k < 4; k++) nrm[c] = fma(g[c][k], g[c][k], nrm[c]); }
  int js = 0;
#pragma unroll
  for (int c = 1; c < 4; c++) if (nrm[c] < nrm[js]) js = c;
#pragma unroll
  for (int r = 0; r < 4; r++) X[r] = js == 0 ? v[0][r] : (js == 1 ? v[1][r] : (js == 2 ? v[2][r] : v[3][r]));
}

// cells of Matcher::nonMaximumSuppression along one axis: origins n+margin+k(n+1) < len-n-margin (matcher.cpp:344-345)
__host__ __device__ static inline int viso_cell_count(int len, int n) {
  int s = len - 2 * n - 2 * VISO_MARGIN;
  return s > 0 ? (s + n) / (n + 1) : 0;
}

// launchers implemented in the kernel translation units
int visocu_launch_features(visocu_ctx* ctx, const SlotList& sl);
int visocu_make_tensor_map(visocu_ctx* ctx, size_t frame_stride_bytes);
void visocu_free_tiles(visocu_ctx* ctx);
int visocu_make_half_image(visocu_ctx* ctx, int frame);
// k_recon's checks, upload image and launch (csrc/recon.cu), shared by visocu_recon_points and visocu_recon_update
int visocu_recon_check(visocu_ctx* ctx, const char* what, int32_t n_jobs, const visocu_recon_job* jobs, int32_t* const* status,
                       float* const* xyz, size_t* n_tracks_total, size_t* n_frames_total);
size_t visocu_recon_stage_bytes(int32_t n_jobs, size_t n_frames_total, size_t n_tracks_total);
void visocu_recon_stage(int32_t n_jobs, const visocu_recon_job* jobs, size_t n_frames_total, uint8_t* pin, uint8_t* dev, int4* out,
                        int32_t* first_track);
int visocu_recon_launch(visocu_ctx* ctx, const uint8_t* dev, int32_t n_jobs, size_t n_tracks_total);
void visocu_free_recon_stores(visocu_ctx* ctx);                // visocu_destroy: the stores still alive
// csrc/rectify.cu: the maps go with visocu_configure and visocu_destroy; the gather kernel replaces k_repitch in a push
struct CamList { int32_t c[VISO_MAX_BATCH]; };
void visocu_free_rectification(visocu_ctx* ctx);
void visocu_launch_rectify(visocu_ctx* ctx, const SlotList& sl, const CamList& cams, int bpl_in);
