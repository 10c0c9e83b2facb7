// Device point store of Reconstruction (include/visocu.h: visocu_recon_store_*, visocu_recon_update).
//
// Reconstruction keeps every point it has reconstructed in the coordinates of the current camera, so each update moves ALL
// stored points into the new camera frame (host/reconstruction.cpp, batchPrepare) before it appends the points of the
// tracks that ended.  On the host that move costs O(points so far) per frame and grows with the length of the drive.  Here
// the points stay in HBM and one call does the whole device half of an update for many sequences:
//   k_recon_move ..... every point of every store in the call, in place; one CTA per chunk of MOVE_CHUNK points of one
//                      store (the chunk table is built on the host from the counts it knows).  24 algorithmic bytes per
//                      point (12 read, 12 written), loaded and stored as 3 float4 per 4 points; bandwidth bound.  On one
//                      B200 (1000 W power limit), 23.5 M points (565 MB of traffic) took 93.7 us: 6.0 TB/s, 78 % of the
//                      7.7 TB/s data-sheet HBM bandwidth (profiles/bench_sfm_long.py, DESIGN.md section 7).
//   k_recon .......... the evaluation of the finished tracks, unchanged (csrc/recon.cu)
//   k_recon_append ... one CTA per job: order-preserving compaction of the status-0 points of k_recon's results behind the
//                      store's current end; the CTA's count is the job's kept count
// A call is one upload (job descriptors, frame tables, tracks, transforms, chunk table, append table), at most these three
// launches and one read-back (kept counts, plus status and points when asked for), and waits at the end.
#include "visocu_internal.cuh"
#include <algorithm>
#include <cstring>

struct visocu_recon_store {
  visocu_ctx* ctx;
  float* d;              // x, y, z per point
  int64_t n, cap;        // points stored, points allocated
};

namespace {

constexpr int MOVE_THREADS = 256;
constexpr int64_t MOVE_CHUNK = 4096;   // points per CTA; a multiple of 4, so every chunk starts 16-byte aligned
constexpr int APPEND_THREADS = 256;

struct MoveChunk { float* xyz; int32_t count, job; };
struct AppendJob { const int4* res; float* dst; int32_t n_tracks, pad; };

// One row of affineTransform (host/reconstruction.cpp) with the host's rounding.  The host library is built with
// g++ -O3 -march=x86-64-v3, and GCC contracts C++ by default (-ffp-contract=fast); its code for every row is
//   vmulsd y*m1 ; vfmadd x*m0 + t ; vfmadd z*m2 + t ; vaddsd t + m3 ; vcvtsd2ss
// (rows 0 and 1 as the packed forms of the same instructions), on the float coordinates widened to double.  The same
// sequence with explicit rounding intrinsics gives the same bytes whatever nvcc would contract on its own.
__device__ __forceinline__ float affine_row(const double* m, double x, double y, double z) {
  double t = __dmul_rn(y, m[1]);
  t = __fma_rn(x, m[0], t);
  t = __fma_rn(z, m[2], t);
  t = __dadd_rn(t, m[3]);
  return __double2float_rn(t);
}

__device__ __forceinline__ void move3(const double* M, float& x, float& y, float& z) {
  const double px = x, py = y, pz = z;
  x = affine_row(M, px, py, pz);
  y = affine_row(M + 4, px, py, pz);
  z = affine_row(M + 8, px, py, pz);
}

__global__ void __launch_bounds__(MOVE_THREADS) k_recon_move(const MoveChunk* __restrict__ chunks, const double* __restrict__ tr) {
  __shared__ double M[12];
  const MoveChunk c = chunks[blockIdx.x];
  if (threadIdx.x < 12) M[threadIdx.x] = tr[12 * c.job + threadIdx.x];
  __syncthreads();
  float4* v = reinterpret_cast<float4*>(c.xyz);
  const int n4 = c.count >> 2;
  for (int g = threadIdx.x; g < n4; g += MOVE_THREADS) {       // 4 points = 48 bytes = 3 float4
    float4 a = v[3 * g], b = v[3 * g + 1], e = v[3 * g + 2];
    move3(M, a.x, a.y, a.z);
    move3(M, a.w, b.x, b.y);
    move3(M, b.z, b.w, e.x);
    move3(M, e.y, e.z, e.w);
    v[3 * g] = a; v[3 * g + 1] = b; v[3 * g + 2] = e;
  }
  const int i = 4 * n4 + (int)threadIdx.x;                      // the store's last 1 - 3 points
  if (i < c.count) move3(M, c.xyz[3 * i], c.xyz[3 * i + 1], c.xyz[3 * i + 2]);
}

__global__ void __launch_bounds__(APPEND_THREADS) k_recon_append(const AppendJob* __restrict__ jobs, int32_t* __restrict__ kept) {
  __shared__ int warp_kept[APPEND_THREADS / 32];
  const AppendJob J = jobs[blockIdx.x];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int base = 0;
  for (int t0 = 0; t0 < J.n_tracks; t0 += APPEND_THREADS) {
    const int i = t0 + (int)threadIdx.x;
    int4 r = make_int4(1, 0, 0, 0);
    if (i < J.n_tracks) r = J.res[i];
    const unsigned ballot = __ballot_sync(0xffffffffu, r.x == 0);
    if (lane == 0) warp_kept[warp] = __popc(ballot);
    __syncthreads();
    int at = base, total = 0;
#pragma unroll
    for (int w = 0; w < APPEND_THREADS / 32; w++) {
      at += w < warp ? warp_kept[w] : 0;
      total += warp_kept[w];
    }
    if (r.x == 0) {
      at += __popc(ballot & ((1u << lane) - 1u));
      J.dst[3 * (size_t)at] = __int_as_float(r.y);
      J.dst[3 * (size_t)at + 1] = __int_as_float(r.z);
      J.dst[3 * (size_t)at + 2] = __int_as_float(r.w);
    }
    __syncthreads();
    base += total;
  }
  if (threadIdx.x == 0) kept[blockIdx.x] = base;
}

bool owned(const visocu_ctx* ctx, const visocu_recon_store* s) {
  return std::find(ctx->stores.begin(), ctx->stores.end(), s) != ctx->stores.end();
}

// Store memory is stream-ordered (cudaMallocAsync / cudaFreeAsync on the lane's stream): cudaFree would wait for the whole
// device, i.e. stall every other worker's stream each time one sequence's store grows.
// Room for `need` points: a new buffer of twice the capacity (again until it fits), a stream-ordered copy of the stored
// points and the old buffer freed behind it.  VISOCU_ECAPACITY if the allocation fails.
int reserve(visocu_ctx* ctx, visocu_recon_store* s, int64_t need) {
  if (need <= s->cap) return VISOCU_OK;
  int64_t cap = std::max<int64_t>(s->cap, 1);
  while (cap < need) cap *= 2;
  void* d = nullptr;
  if (cudaMallocAsync(&d, (size_t)cap * 12, ctx->stream) != cudaSuccess) {
    cudaGetLastError();
    return visocu_set_error(ctx, VISOCU_ECAPACITY, "recon store: no device memory for %lld points", (long long)cap);
  }
  if (s->n) CU_TRY(ctx, cudaMemcpyAsync(d, s->d, (size_t)s->n * 12, cudaMemcpyDeviceToDevice, ctx->stream));
  if (s->d) CU_TRY(ctx, cudaFreeAsync(s->d, ctx->stream));
  s->d = (float*)d; s->cap = cap;
  return VISOCU_OK;
}

}  // namespace

void visocu_free_recon_stores(visocu_ctx* ctx) {
  for (visocu_recon_store* s : ctx->stores) {
    if (s->d) cudaFreeAsync(s->d, ctx->stream);
    delete s;
  }
  ctx->stores.clear();
}

extern "C" int visocu_recon_store_create(visocu_ctx* ctx, int64_t initial_capacity, visocu_recon_store** out) {
  if (!ctx) return VISOCU_EINVAL;
  if (!out || initial_capacity < 0 || initial_capacity > ((int64_t)1 << 40))
    return visocu_set_error(ctx, VISOCU_EINVAL, "recon_store_create: bad arguments");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  visocu_recon_store* s = new visocu_recon_store{ctx, nullptr, 0, 0};
  if (reserve(ctx, s, initial_capacity) != VISOCU_OK) {
    delete s;
    return VISOCU_ECAPACITY;
  }
  ctx->stores.push_back(s);
  *out = s;
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}

extern "C" int visocu_recon_store_destroy(visocu_ctx* ctx, visocu_recon_store* store) {
  if (!ctx) return VISOCU_EINVAL;
  if (!store || !owned(ctx, store)) return visocu_set_error(ctx, VISOCU_EINVAL, "recon_store_destroy: not a store of this context");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ctx->stores.erase(std::find(ctx->stores.begin(), ctx->stores.end(), store));
  const cudaError_t e = store->d ? cudaFreeAsync(store->d, ctx->stream) : cudaSuccess;
  delete store;
  CU_TRY(ctx, e);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}

extern "C" int visocu_recon_store_append(visocu_ctx* ctx, visocu_recon_store* store, const float* xyz, int64_t n) {
  if (!ctx) return VISOCU_EINVAL;
  if (!store || store->ctx != ctx || n < 0 || n > ((int64_t)1 << 40) || (n > 0 && !xyz))
    return visocu_set_error(ctx, VISOCU_EINVAL, "recon_store_append: bad arguments");
  if (n == 0) return VISOCU_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  int rc = reserve(ctx, store, store->n + n);
  if (rc) return rc;
  CU_COPY(ctx, store->d + 3 * store->n, xyz, (size_t)n * 12, cudaMemcpyHostToDevice);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  store->n += n;
  return VISOCU_OK;
}

extern "C" int visocu_recon_store_read(visocu_ctx* ctx, const visocu_recon_store* store, int64_t first, int64_t count, float* xyz) {
  if (!ctx) return VISOCU_EINVAL;
  if (!store || store->ctx != ctx || first < 0 || count < 0 || first > store->n || count > store->n - first || (count > 0 && !xyz))
    return visocu_set_error(ctx, VISOCU_EINVAL, "recon_store_read: bad arguments");
  if (count == 0) return VISOCU_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_COPY(ctx, xyz, store->d + 3 * first, (size_t)count * 12, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}

extern "C" int visocu_recon_store_points(const visocu_recon_store* store, const float** d_xyz, int64_t* n) {
  if (!store || !d_xyz || !n) return VISOCU_EINVAL;
  *d_xyz = store->d;
  *n = store->n;
  return VISOCU_OK;
}

extern "C" int visocu_recon_update(visocu_ctx* ctx, int32_t n_jobs, visocu_recon_store* const* stores, const double* const* tr12,
                                   const visocu_recon_job* jobs, int32_t* n_kept, int32_t* const* status, float* const* xyz) {
  if (!ctx) return VISOCU_EINVAL;
  if (n_jobs < 0 || (n_jobs > 0 && (!stores || !tr12 || !jobs))) return visocu_set_error(ctx, VISOCU_EINVAL, "bad recon_update arguments");
  // every argument is checked before anything is enqueued or written
  for (int j = 0; j < n_jobs; j++) {
    if (!stores[j] || stores[j]->ctx != ctx || !tr12[j])
      return visocu_set_error(ctx, VISOCU_EINVAL, "recon_update job %d: null transform, or no store of this context", j);
  }
  {
    std::vector<const visocu_recon_store*> sorted(stores, stores + n_jobs);
    std::sort(sorted.begin(), sorted.end());
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end())
      return visocu_set_error(ctx, VISOCU_EINVAL, "recon_update: a store appears twice");
  }
  size_t n_total = 0, n_frames_total = 0;
  int rc = visocu_recon_check(ctx, "recon_update", n_jobs, jobs, status, xyz, &n_total, &n_frames_total);
  if (rc) return rc;
  size_t n_chunks = 0;
  for (int j = 0; j < n_jobs; j++) n_chunks += (size_t)((stores[j]->n + MOVE_CHUNK - 1) / MOVE_CHUNK);
  if (n_kept) for (int j = 0; j < n_jobs; j++) n_kept[j] = 0;
  if (n_total == 0 && n_chunks == 0) return VISOCU_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));

  // Upload: k_recon's inputs, transforms, chunk table, append table (ONE copy).  Read-back: the kept counts, then 16 bytes
  // per track if status or points are wanted (ONE copy).
  const bool want = status || xyz;
  const size_t o_tr = align_up(n_total ? visocu_recon_stage_bytes(n_jobs, n_frames_total, n_total) : 0, 256);
  const size_t o_chunks = align_up(o_tr + 96 * (size_t)n_jobs, 256);
  const size_t o_append = align_up(o_chunks + sizeof(MoveChunk) * n_chunks, 256);
  const size_t up_bytes = o_append + sizeof(AppendJob) * (size_t)n_jobs;
  const size_t o_kept = align_up(up_bytes, 256);
  const size_t o_out = align_up(o_kept + 4 * (size_t)n_jobs, 256);
  const size_t end = o_out + 16 * n_total;
  if ((rc = visocu_ensure_scratch(ctx, end))) return rc;
  if ((rc = visocu_ensure_pinned(ctx, end))) return rc;
  uint8_t* sb = (uint8_t*)ctx->scratch;
  uint8_t* pin = (uint8_t*)ctx->pinned;

  // capacity first (kept points <= tracks): the move then runs on the grown buffers
  bool grown = true;
  for (int j = 0; j < n_jobs && grown; j++) {
    rc = reserve(ctx, stores[j], stores[j]->n + jobs[j].n_tracks);
    if (rc == VISOCU_ECAPACITY) grown = false;
    else if (rc) { cudaStreamSynchronize(ctx->stream); return rc; }
  }
  const bool eval = grown && n_total > 0;

  std::vector<int32_t> first((size_t)n_jobs);
  if (n_total) visocu_recon_stage(n_jobs, jobs, n_frames_total, pin, sb, (int4*)(sb + o_out), first.data());
  MoveChunk* ch = (MoveChunk*)(pin + o_chunks);
  AppendJob* ap = (AppendJob*)(pin + o_append);
  size_t c = 0;
  for (int j = 0; j < n_jobs; j++) {
    visocu_recon_store* s = stores[j];
    memcpy(pin + o_tr + 96 * (size_t)j, tr12[j], 96);
    for (int64_t p = 0; p < s->n; p += MOVE_CHUNK) ch[c++] = MoveChunk{s->d + 3 * p, (int32_t)std::min<int64_t>(MOVE_CHUNK, s->n - p), j};
    ap[j] = AppendJob{(const int4*)(sb + o_out) + first[j], s->d + 3 * s->n, jobs[j].n_tracks, 0};
  }
  CU_COPY(ctx, sb, pin, up_bytes, cudaMemcpyHostToDevice);
  if (n_chunks) {
    k_recon_move<<<(unsigned)n_chunks, MOVE_THREADS, 0, ctx->stream>>>((const MoveChunk*)(sb + o_chunks), (const double*)(sb + o_tr));
    CU_LAUNCH_CHECK(ctx);
  }
  if (eval) {
    if ((rc = visocu_recon_launch(ctx, sb, n_jobs, n_total))) return rc;
    k_recon_append<<<(unsigned)n_jobs, APPEND_THREADS, 0, ctx->stream>>>((const AppendJob*)(sb + o_append), (int32_t*)(sb + o_kept));
    CU_LAUNCH_CHECK(ctx);
    CU_COPY(ctx, pin + o_kept, sb + o_kept, (want ? end : o_out) - o_kept, cudaMemcpyDeviceToHost);
  }
  CU_TRY(ctx, visocu_stream_wait(ctx));
  if (!grown) return VISOCU_ECAPACITY;           // the message was set by reserve
  if (!eval) return VISOCU_OK;
  const int32_t* kept = (const int32_t*)(pin + o_kept);
  const int32_t* res = (const int32_t*)(pin + o_out);
  for (int j = 0; j < n_jobs; j++) {
    stores[j]->n += kept[j];
    if (n_kept) n_kept[j] = kept[j];
    for (int k = 0; k < jobs[j].n_tracks; k++) {
      const int32_t* r = res + 4 * (size_t)(first[j] + k);
      if (status) status[j][k] = r[0];
      if (xyz) memcpy(xyz[j] + 3 * (size_t)k, r + 1, 12);
    }
  }
  return VISOCU_OK;
}
