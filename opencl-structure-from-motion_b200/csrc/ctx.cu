// Context, frame pool and host<->device transport behind include/visocu.h.
// Replaces the reference's OpenCL::Container / Buffer<T> runtime (viso/opencl_wrapper.hh:19-166,
// viso/opencl_wrapper.cpp:66-164) with one CUDA stream per context and a pre-carved device pool.
#include "visocu_internal.cuh"
#include <cstdarg>
#include <cstdio>
#include <sched.h>
#include <time.h>
#include <cstring>
#include <cmath>
#include <cstdlib>
#include <functional>

static thread_local std::string g_create_error;

int visocu_set_error(visocu_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf; else g_create_error = buf;
  return code;
}

// Host-side wait for the context's stream.  Several host threads share the GPU (one context each), and there may be more
// of them than cores.  The default wait costs no driver call while it waits: a stream memory operation
// (cuStreamWriteValue32) stores a sequence number into pinned host memory when the stream reaches it, and the thread
// polls that word, yielding the core between polls - the driver's lock stays free for the threads that are launching
// work, and a waiting thread does not keep a runnable one off its core.  VISOCU_WAIT=sync falls back to
// cudaStreamSynchronize (spinning inside the driver), VISOCU_BLOCKING_SYNC=1 to a blocking event.
namespace {
typedef CUresult (*WriteValueFn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
WriteValueFn write_value_fn() {
  static WriteValueFn fn = [] {
    const char* e = getenv("VISOCU_WAIT");
    if (e && e[0] == 's') return (WriteValueFn) nullptr;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return (WriteValueFn) nullptr;
    return (WriteValueFn)p;
  }();
  return fn;
}
}  // namespace

// the host-visible completion word of the current lane's stream: enqueue only
cudaError_t visocu_stream_signal(visocu_ctx* ctx, uint32_t* seq_out) {
  WriteValueFn wv = write_value_fn();
  if (!wv || !ctx->wait_flag || ctx->ev_sync) { *seq_out = 0; return cudaSuccess; }
  const uint32_t seq = ++ctx->wait_seq;
  if (wv((CUstream)ctx->stream, (CUdeviceptr)(uintptr_t)ctx->wait_flag_dev, seq, 0) != CUDA_SUCCESS) { *seq_out = 0; return cudaSuccess; }
  *seq_out = seq;
  return cudaSuccess;
}

// wait until the completion word shows seq (0: fall back to a synchronising call)
cudaError_t visocu_stream_wait_seq(visocu_ctx* ctx, uint32_t seq) {
  cudaStream_t st = ctx->stream;
  if (ctx->ev_sync) {
    cudaError_t e = cudaEventRecord(ctx->ev_sync, st);
    return e != cudaSuccess ? e : cudaEventSynchronize(ctx->ev_sync);
  }
  if (seq == 0 || !ctx->wait_flag) return cudaStreamSynchronize(st);
  // VISOCU_WAIT_SLEEP_US=n (set by callers that run more worker threads than they have cores): after a short
  // spin the thread sleeps n microseconds between polls, so that it does not take half of a shared core away from
  // a worker that has host work to do
  static const int sleep_us = [] { const char* e = getenv("VISOCU_WAIT_SLEEP_US"); return e ? atoi(e) : 0; }();
  volatile uint32_t* flag = ctx->wait_flag;
  unsigned spins = 0;
  while ((int32_t)(*flag - seq) < 0) {
    if ((++spins & 0x3FFF) == 0) {                 // now and then: did the stream die?
      cudaError_t e = cudaStreamQuery(st);
      if (e != cudaSuccess && e != cudaErrorNotReady) return e;
    }
    if (sleep_us > 0 && spins > 64) {
      struct timespec ts = {0, (long)sleep_us * 1000L};
      nanosleep(&ts, nullptr);
    } else {
      sched_yield();
    }
  }
  return cudaSuccess;
}

cudaError_t visocu_stream_wait(visocu_ctx* ctx) {
  uint32_t seq = 0;
  visocu_stream_signal(ctx, &seq);
  return visocu_stream_wait_seq(ctx, seq);
}

// ---- lanes
static cudaError_t make_wait_flag(volatile uint32_t** flag, void** dev) {
  void* f = nullptr;
  *flag = nullptr; *dev = nullptr;
  if (cudaHostAlloc(&f, 64, cudaHostAllocMapped) == cudaSuccess) {
    memset(f, 0, 64);
    void* d = nullptr;
    if (cudaHostGetDevicePointer(&d, f, 0) == cudaSuccess) { *flag = (volatile uint32_t*)f; *dev = d; }
    else cudaFreeHost(f);
  }
  cudaGetLastError();
  return cudaSuccess;
}

#define VISO_LANE_FIELDS(X) X(stream) X(scratch) X(scratch_bytes) X(scratch2) X(scratch2_bytes) X(pinned) X(pinned_bytes) X(pinned2) \
  X(pinned2_bytes) X(d_ranges) X(d_ranges_bytes) X(pin_ranges) X(deliver) X(deliver_dev) X(deliver_bytes) X(deliver2) X(deliver2_bytes) \
  X(wait_flag) X(wait_flag_dev) X(wait_seq) X(counts_stage) X(img_stage) X(img_stage_bytes) X(src_table) X(src_table_pin) X(ev_push) \
  X(g_push) X(g_match) X(fused_pending) X(fused_n) X(fused_ranges) X(fused_list1) X(fused_seq) X(fused_jobs)

int visocu_use_lane(visocu_ctx* ctx, int lane) {
  if (lane < 0 || lane >= VISO_LANES) return visocu_set_error(ctx, VISOCU_EINVAL, "lane %d out of range", lane);
  if (lane == ctx->lane) return VISOCU_OK;
  visocu_lane& out = ctx->lanes[ctx->lane];
  visocu_lane& in = ctx->lanes[lane];
#define X(f) out.f = ctx->f;
  VISO_LANE_FIELDS(X)
#undef X
  out.part[0] = ctx->part[0]; out.part[1] = ctx->part[1];
  out.created = true;
  if (!in.created) {
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaStreamCreateWithFlags(&in.stream, cudaStreamNonBlocking));
    make_wait_flag(&in.wait_flag, &in.wait_flag_dev);
    in.created = true;
  }
#define X(f) ctx->f = in.f;
  VISO_LANE_FIELDS(X)
#undef X
  ctx->part[0] = in.part[0]; ctx->part[1] = in.part[1];
  ctx->lane = lane;
  return VISOCU_OK;
}
extern "C" int visocu_set_lane(visocu_ctx* ctx, int32_t lane) { return ctx ? visocu_use_lane(ctx, lane) : VISOCU_EINVAL; }

static void destroy_graph(visocu_graph& g) { if (g.exec) cudaGraphExecDestroy(g.exec); g = visocu_graph(); }
static void free_lane_resources(visocu_ctx* ctx) {     // of the lane in the working fields
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  destroy_graph(ctx->g_push); destroy_graph(ctx->g_match);
  if (ctx->scratch) cudaFree(ctx->scratch);
  if (ctx->scratch2) cudaFree(ctx->scratch2);
  if (ctx->d_ranges) cudaFree(ctx->d_ranges);
  if (ctx->pin_ranges) cudaFreeHost(ctx->pin_ranges);
  if (ctx->deliver) cudaFreeHost(ctx->deliver);
  if (ctx->deliver2) cudaFreeHost(ctx->deliver2);
  if (ctx->pinned2) cudaFreeHost(ctx->pinned2);
  if (ctx->img_stage) cudaFree(ctx->img_stage);
  if (ctx->counts_stage) cudaFree(ctx->counts_stage);
  if (ctx->src_table) cudaFree((void*)ctx->src_table);
  if (ctx->src_table_pin) cudaFreeHost((void*)ctx->src_table_pin);
  if (ctx->wait_flag) cudaFreeHost((void*)ctx->wait_flag);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->ev_push) cudaEventDestroy(ctx->ev_push);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = nullptr; ctx->scratch = ctx->scratch2 = ctx->d_ranges = ctx->pin_ranges = ctx->deliver = ctx->deliver2 = nullptr;
  ctx->pinned = ctx->pinned2 = nullptr; ctx->img_stage = nullptr; ctx->counts_stage = nullptr; ctx->wait_flag = nullptr;
  ctx->src_table = ctx->src_table_pin = nullptr; ctx->ev_push = nullptr;
  ctx->scratch_bytes = ctx->scratch2_bytes = ctx->pinned_bytes = ctx->pinned2_bytes = ctx->d_ranges_bytes = ctx->deliver_bytes = 0;
  ctx->deliver2_bytes = ctx->img_stage_bytes = 0;
}
void visocu_drop_lane_graphs(visocu_ctx* ctx) { destroy_graph(ctx->g_push); destroy_graph(ctx->g_match); }
// graphs bake frame pointers and sizes: a re-configuration drops them on every lane
void visocu_drop_graphs(visocu_ctx* ctx) {
  destroy_graph(ctx->g_push); destroy_graph(ctx->g_match);
  for (int l = 0; l < VISO_LANES; l++) { destroy_graph(ctx->lanes[l].g_push); destroy_graph(ctx->lanes[l].g_match); }
}

extern "C" const char* visocu_last_error(const visocu_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int visocu_create(int device, visocu_ctx** out) {
  if (!out) return VISOCU_EINVAL;
  *out = nullptr;
  // One context = one stream, and a process may drive many of them (one per host worker).  With the default of 8 hardware
  // work queues, streams share queues and a long kernel at the head of one stream stalls the kernels of its queue
  // neighbours; CUDA_DEVICE_MAX_CONNECTIONS=32 removes that (flow bench: 13.9 k -> 23.2 k pairs/s).  That variable is
  // process-wide and only read when CUDA initialises, so it is the APPLICATION's to set (bench.py does, before anything
  // touches CUDA; include/visocu.h says so); the library does not modify its host's environment.
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0)
    return visocu_set_error(nullptr, VISOCU_ENODEVICE, "no CUDA device (%s); this library has no CPU fallback",
                            e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (device < 0 || device >= ndev) return visocu_set_error(nullptr, VISOCU_EINVAL, "device %d out of range (%d devices)", device, ndev);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
    return visocu_set_error(nullptr, VISOCU_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return visocu_set_error(nullptr, VISOCU_ENODEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only", device, prop.major, prop.minor);
  visocu_ctx* ctx = new visocu_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount; ctx->cc_major = prop.major; ctx->cc_minor = prop.minor;
  snprintf(ctx->name, sizeof ctx->name, "%s", prop.name);
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess ||
      (e = cudaMalloc(&ctx->d_stats, 2 * sizeof(uint64_t))) != cudaSuccess) {
    visocu_set_error(nullptr, VISOCU_ECUDA, "context setup: %s", cudaGetErrorString(e));
    visocu_destroy(ctx);             // releases whatever was created before the failure
    return VISOCU_ECUDA;
  }
  cudaMemset(ctx->d_stats, 0, 2 * sizeof(uint64_t));
  make_wait_flag(&ctx->wait_flag, &ctx->wait_flag_dev);      // completion word of visocu_stream_wait: pinned, mapped, written by the stream itself
  ctx->lanes[0].created = true;
  if (const char* e = getenv("VISOCU_GRAPHS")) ctx->use_graphs = e[0] != '0';
  // VISOCU_BLOCKING_SYNC=1: waiting host threads sleep (for runs with more worker threads than cores)
  if (const char* e = getenv("VISOCU_BLOCKING_SYNC"))
    if (e[0] == '1') cudaEventCreateWithFlags(&ctx->ev_sync, cudaEventBlockingSync | cudaEventDisableTiming);
  *out = ctx;
  return VISOCU_OK;
}

static void free_pool(visocu_ctx* ctx) {
  if (ctx->pool) cudaFree(ctx->pool);
  if (ctx->frames_d) cudaFree(ctx->frames_d);
  ctx->pool = nullptr; ctx->frames_d = nullptr; ctx->configured = false;
  visocu_free_tiles(ctx);
  visocu_free_rectification(ctx);
  visocu_drop_graphs(ctx);
}

extern "C" void visocu_destroy(visocu_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (int l = 0; l < VISO_LANES; l++)
    if (l == ctx->lane || ctx->lanes[l].created) { if (visocu_use_lane(ctx, l) == VISOCU_OK && ctx->stream) cudaStreamSynchronize(ctx->stream); }
  if (getenv("VISOCU_RO_STATS") && (ctx->ro_jobs || ctx->ro_declined)) {
    const double nj = ctx->ro_jobs ? (double)ctx->ro_jobs : 1.0;
    fprintf(stderr, "[outliers] %llu lists on the device, mean us: sort %.1f partition %.1f build %.1f vote %.1f; declined %llu "
            "(too long %llu, duplicates %llu, guard %llu; mean length %.0f)\n",
            (unsigned long long)ctx->ro_jobs, 1e-3 * ctx->ro_ns[0] / nj, 1e-3 * ctx->ro_ns[1] / nj, 1e-3 * ctx->ro_ns[2] / nj,
            1e-3 * ctx->ro_ns[3] / nj, (unsigned long long)ctx->ro_declined, (unsigned long long)ctx->ro_reason[1],
            (unsigned long long)ctx->ro_reason[2], (unsigned long long)ctx->ro_reason[3],
            ctx->ro_declined ? (double)ctx->ro_declined_n / (double)ctx->ro_declined : 0.0);
  }
  visocu_free_recon_stores(ctx);
  for (int l = 0; l < VISO_LANES; l++)
    if (l == ctx->lane || ctx->lanes[l].created) { if (visocu_use_lane(ctx, l) == VISOCU_OK) free_lane_resources(ctx); }
  free_pool(ctx);
  if (ctx->d_stats) cudaFree(ctx->d_stats);
  if (ctx->pev0) cudaEventDestroy(ctx->pev0);
  if (ctx->pev1) cudaEventDestroy(ctx->pev1);
  if (ctx->ev_sync) cudaEventDestroy(ctx->ev_sync);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  delete ctx;
}

extern "C" int visocu_device_info(const visocu_ctx* ctx, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, char* name64) {
  if (!ctx) return VISOCU_EINVAL;
  if (sm_count) *sm_count = ctx->sm_count;
  if (cc_major) *cc_major = ctx->cc_major;
  if (cc_minor) *cc_minor = ctx->cc_minor;
  if (name64) memcpy(name64, ctx->name, 64);
  return VISOCU_OK;
}

int visocu_ensure_scratch(visocu_ctx* ctx, size_t bytes) {
  if (!ctx->in_step && (ctx->g_push.exec || ctx->g_match.exec)) visocu_drop_lane_graphs(ctx);   // the graphs replay copies out of these buffers
  if (bytes <= ctx->scratch_bytes) return VISOCU_OK;
  CU_TRY(ctx, visocu_stream_wait(ctx));
  if (ctx->scratch) cudaFree(ctx->scratch);
  ctx->scratch = nullptr; ctx->scratch_bytes = 0;
  size_t want = align_up(bytes + bytes / 4, 1 << 20);
  CU_TRY(ctx, cudaMalloc(&ctx->scratch, want));
  ctx->scratch_bytes = want;
  return VISOCU_OK;
}

int visocu_ensure_pinned(visocu_ctx* ctx, size_t bytes) {
  if (!ctx->in_step && (ctx->g_push.exec || ctx->g_match.exec)) visocu_drop_lane_graphs(ctx);
  if (bytes <= ctx->pinned_bytes) return VISOCU_OK;
  CU_TRY(ctx, visocu_stream_wait(ctx));
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  ctx->pinned = nullptr; ctx->pinned_bytes = 0;
  size_t want = align_up(bytes + bytes / 4, 1 << 16);
  CU_TRY(ctx, cudaMallocHost(&ctx->pinned, want));
  ctx->pinned_bytes = want;
  return VISOCU_OK;
}

// bytes per line rounded up to 16 (reference matcher.cpp:158-160)
static int viso_bpl(int w) { return w + 15 - (w - 1) % 16; }

extern "C" int visocu_configure(visocu_ctx* ctx, const visocu_params* p, int32_t width, int32_t height, int32_t n_frames) {
  if (!ctx || !p) return VISOCU_EINVAL;
  if (width <= 0 || height <= 0 || n_frames <= 0) return visocu_set_error(ctx, VISOCU_EINVAL, "bad dims %dx%d / %d frames", width, height, n_frames);
  if (p->nms_n < 1 || p->nms_n > 14) return visocu_set_error(ctx, VISOCU_EINVAL, "nms_n=%d outside the supported range 1..14", p->nms_n);
  if (p->match_binsize < 1) return visocu_set_error(ctx, VISOCU_EINVAL, "match_binsize must be positive");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  for (int l = 0; l < VISO_LANES; l++) if (ctx->lanes[l].created && l != ctx->lane && ctx->lanes[l].stream) cudaStreamSynchronize(ctx->lanes[l].stream);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  free_pool(ctx);
  ctx->param = *p;
  ctx->ro_bound[0] = ctx->ro_bound[1] = -1;
  // outlier kernel shape (experiments and tests): VISOCU_RO_THREADS=256|512|1024 threads per list, VISOCU_RO_WARP=0 one
  // thread per top-level merge.  Read per configure, so that one process can run every variant.
  ctx->ro_threads = 0;
  if (const char* e = getenv("VISOCU_RO_THREADS")) { const int t = atoi(e); if (t == 256 || t == 512 || t == 1024) ctx->ro_threads = t; }
  ctx->ro_warp = 1;
  if (const char* e = getenv("VISOCU_RO_WARP")) if (e[0] == '0') ctx->ro_warp = 0;
  Geometry& g = ctx->g;
  g.w = width; g.h = height; g.bpl = viso_bpl(width);
  g.half = p->half_resolution ? 1 : 0;
  g.scale = g.half ? 2 : 1;
  if (g.half) { g.wm = width / 2; g.hm = height / 2; g.bplm = g.wm > 0 ? viso_bpl(g.wm) : 16; }   // matcher.cpp:630-634
  else        { g.wm = width; g.hm = height; g.bplm = g.bpl; }
  g.first_pass = p->multi_stage ? 0 : 1;
  // sparse-pass neighbourhood (matcher.cpp:684-688)
  int ns = p->nms_n * 3;
  if (ns > 10) ns = p->nms_n > 10 ? p->nms_n : 10;
  g.n[0] = ns; g.n[1] = p->nms_n;
  g.tau = p->nms_tau;
  for (int k = 0; k < 2; k++) {
    g.ncx[k] = viso_cell_count(g.wm, g.n[k]);
    g.ncy[k] = viso_cell_count(g.hm, g.n[k]);
    g.cap[k] = 4 * g.ncx[k] * g.ncy[k] + 32;
  }
  g.binsize = p->match_binsize;
  g.ub = (int)ceilf((float)width / (float)p->match_binsize);     // matcher.cpp:973-975 (full-resolution dims_c)
  g.vb = (int)ceilf((float)height / (float)p->match_binsize);
  g.nbins = 4 * g.ub * g.vb;
  g.radius = p->match_radius; g.disp_tol = p->match_disp_tolerance;
  if (g.ub > 4095 || g.vb > 4095 || width > 8191 * g.scale || height > 8191 * g.scale || g.cap[0] > (1 << 24) || g.cap[1] > (1 << 24))
    return visocu_set_error(ctx, VISOCU_EINVAL, "image, bin grid or feature capacity too large for the packed match keys (24-bit feature index)");

  // carve one pool
  size_t plane_f = align_up((size_t)g.bpl * g.h + 64, 256), plane_m = align_up((size_t)g.bplm * g.hm + 64, 256);
  size_t per = 0;
  auto take = [&](size_t bytes) { size_t o = per; per += align_up(bytes, 256); return o; };
  size_t o_img = take(plane_f), o_half = g.half ? take(plane_m) : 0, o_du = take(plane_m), o_dv = take(plane_m);
  size_t o_duf = g.half ? take(plane_f) : 0, o_dvf = g.half ? take(plane_f) : 0;
  size_t o_codes[2], o_blk[2], o_rec[2], o_bs[2], o_bc[2], o_be[2];
  for (int k = 0; k < 2; k++) {
    size_t cells = (size_t)g.ncx[k] * g.ncy[k];
    o_codes[k] = take((cells + 1) * 4);
    o_blk[k] = take((cells / 512 + 2) * 4);
    o_rec[k] = take((size_t)g.cap[k] * 48);
    o_bs[k] = take((size_t)(g.nbins + 1) * 4);
    o_bc[k] = take((size_t)(g.nbins + 1) * 4);
    o_be[k] = take((size_t)g.cap[k] * 8);
  }
  size_t o_cnt = take(64);
  ctx->pool_bytes = per * (size_t)n_frames;
  CU_TRY(ctx, cudaMalloc(&ctx->pool, ctx->pool_bytes));
  CU_TRY(ctx, cudaMemsetAsync(ctx->pool, 0, ctx->pool_bytes, ctx->stream));
  ctx->frames_h.assign(n_frames, FrameDev());
  for (int f = 0; f < n_frames; f++) {
    uint8_t* base = (uint8_t*)ctx->pool + per * (size_t)f;
    FrameDev& F = ctx->frames_h[f];
    F.img = base + o_img; F.half = g.half ? base + o_half : nullptr;
    F.du = base + o_du; F.dv = base + o_dv;
    F.du_full = g.half ? base + o_duf : nullptr; F.dv_full = g.half ? base + o_dvf : nullptr;
    for (int k = 0; k < 2; k++) {
      F.codes[k] = (uint32_t*)(base + o_codes[k]); F.blk[k] = (int32_t*)(base + o_blk[k]);
      F.rec[k] = (int32_t*)(base + o_rec[k]); F.bin_start[k] = (int32_t*)(base + o_bs[k]);
      F.bin_cursor[k] = (int32_t*)(base + o_bc[k]); F.bin_ent[k] = (int2*)(base + o_be[k]);
    }
    F.counts = (int32_t*)(base + o_cnt);
  }
  CU_TRY(ctx, cudaMalloc(&ctx->frames_d, sizeof(FrameDev) * (size_t)n_frames));
  CU_COPY(ctx, ctx->frames_d, ctx->frames_h.data(), sizeof(FrameDev) * (size_t)n_frames, cudaMemcpyHostToDevice);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  ctx->n_frames = n_frames;
  {
    int rc = visocu_make_tensor_map(ctx, per);
    if (rc) return rc;
  }
  ctx->h_counts.assign((size_t)n_frames * 2, 0);
  ctx->frame_valid.assign(n_frames, 0);
  ctx->configured = true;
  return VISOCU_OK;
}

extern "C" int visocu_set_intrinsics(visocu_ctx* ctx, double f, double cu, double cv, double base) {
  if (!ctx) return VISOCU_EINVAL;
  ctx->param.f = f; ctx->param.cu = cu; ctx->param.cv = cv; ctx->param.base = base;
  return VISOCU_OK;
}
extern "C" int visocu_sync(visocu_ctx* ctx) {
  if (!ctx) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}
extern "C" int visocu_timer_start(visocu_ctx* ctx) {
  if (!ctx) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  return VISOCU_OK;
}
extern "C" int visocu_timer_stop(visocu_ctx* ctx, float* ms) {
  if (!ctx || !ms) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  CU_TRY(ctx, cudaEventSynchronize(ctx->ev1));
  CU_TRY(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  return VISOCU_OK;
}
extern "C" int visocu_host_alloc(visocu_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaMallocHost(out, bytes));
  return VISOCU_OK;
}
extern "C" int visocu_host_free(visocu_ctx* ctx, void* p) {
  if (!ctx) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaFreeHost(p));
  return VISOCU_OK;
}
extern "C" int visocu_device_alloc(visocu_ctx* ctx, size_t bytes, void** out) {
  if (!ctx || !out) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaMalloc(out, bytes));
  return VISOCU_OK;
}
extern "C" int visocu_device_free(visocu_ctx* ctx, void* p) {
  if (!ctx) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaFree(p));
  return VISOCU_OK;
}
extern "C" int visocu_memcpy_h2d(visocu_ctx* ctx, void* dst, const void* src, size_t bytes) {
  if (!ctx) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_COPY(ctx, dst, src, bytes, cudaMemcpyHostToDevice);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}
extern "C" int visocu_transfer_bytes(const visocu_ctx* ctx, uint64_t* h2d, uint64_t* d2h) {
  if (!ctx) return VISOCU_EINVAL;
  if (h2d) *h2d = ctx->h2d_bytes;
  if (d2h) *d2h = ctx->d2h_bytes;
  return VISOCU_OK;
}
extern "C" int visocu_profile(visocu_ctx* ctx, int32_t enable) {
  if (!ctx) return VISOCU_EINVAL;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (enable && !ctx->pev0) { CU_TRY(ctx, cudaEventCreate(&ctx->pev0)); CU_TRY(ctx, cudaEventCreate(&ctx->pev1)); }
  ctx->profile = enable ? 1 : 0;
  ctx->filter_ms = 0; ctx->filter_launches = 0; ctx->filter_frames = 0;
  return VISOCU_OK;
}
extern "C" int visocu_profile_read(const visocu_ctx* ctx, double* filter_ms, uint64_t* launches, uint64_t* frames) {
  if (!ctx) return VISOCU_EINVAL;
  if (filter_ms) *filter_ms = ctx->filter_ms;
  if (launches) *launches = ctx->filter_launches;
  if (frames) *frames = ctx->filter_frames;
  return VISOCU_OK;
}
extern "C" int visocu_outlier_stats(const visocu_ctx* ctx, uint64_t* out8) {
  if (!ctx || !out8) return VISOCU_EINVAL;
  out8[0] = ctx->ro_jobs; out8[1] = ctx->ro_declined;
  out8[2] = ctx->ro_reason[1]; out8[3] = ctx->ro_reason[2]; out8[4] = ctx->ro_reason[3];
  out8[5] = ctx->ro_ns[0] + ctx->ro_ns[1]; out8[6] = ctx->ro_ns[2]; out8[7] = ctx->ro_ns[3];
  return VISOCU_OK;
}

extern "C" int visocu_node_stats(const visocu_ctx* ctx, uint64_t* out2) {
  if (!ctx || !out2) return VISOCU_EINVAL;
  out2[0] = ctx->ro_node_calls; out2[1] = ctx->ro_nodes;
  return VISOCU_OK;
}

extern "C" int visocu_launch_count(const visocu_ctx* ctx, uint64_t* n) {
  if (!ctx || !n) return VISOCU_EINVAL;
  *n = ctx->launches;
  return VISOCU_OK;
}

// Row-wise copy of a batch of images into the 16-byte-stride frame planes (matcher.cpp:163-175); pad columns stay zero.
// One launch for all frames of a push: a source row starts at any byte, a destination word is assembled from four bytes.
__global__ void __launch_bounds__(256) k_repitch(Geometry g, const FrameDev* frames, SlotList sl, const uint8_t* const* table, int bpl_in) {
  // The source rows have any alignment (1241 bytes per line): every lane loads the aligned word that holds its first byte,
  // the neighbour's word arrives by shuffle, and a funnel shift lines the four pixels up - one request per warp and 128 bytes
  const uint8_t* __restrict__ src = table[blockIdx.y];
  uint8_t* dst = frames[sl.s[blockIdx.y]].img;
  const int wpr = g.bpl >> 2, total = wpr * g.h, lane = threadIdx.x & 31;
  for (int base = blockIdx.x * 256 + (threadIdx.x & ~31); base < total; base += gridDim.x * 256) {
    const int idx = base + lane;
    const bool in = idx < total;
    const int y = in ? idx / wpr : 0, x = in ? 4 * (idx - y * wpr) : 0;
    const int nb = in ? min(4, g.w - x) : 0;                        // pixels of this word inside the image (<= 0: padding)
    const uintptr_t p = (uintptr_t)(src + (size_t)y * bpl_in + x);
    const uint32_t* wp = (const uint32_t*)(p & ~(uintptr_t)3);
    const int a = (int)(p & 3);
    const uint32_t w0 = nb > 0 ? wp[0] : 0u;
    uint32_t w1 = __shfl_down_sync(0xFFFFFFFFu, w0, 1);
    const uintptr_t next = __shfl_down_sync(0xFFFFFFFFu, (unsigned long long)(nb > 0 ? (uintptr_t)wp : 0), 1);      // 0: that lane loaded nothing
    const bool need1 = nb > 0 && a + nb > 4;                        // some wanted byte lies in the following word
    if (need1 && (lane == 31 || next != (uintptr_t)(wp + 1))) w1 = wp[1];     // row ends, padding neighbours, the warp's last lane
    if (in) {
      uint32_t v = a ? __funnelshift_r(w0, w1, 8 * a) : w0;
      v = nb >= 4 ? v : (nb > 0 ? v & (0xFFFFFFFFu >> (8 * (4 - nb))) : 0u);
      *(uint32_t*)(dst + (size_t)y * g.bpl + x) = v;
    }
  }
}

static int check_frames(visocu_ctx* ctx, int32_t n, const int32_t* frames) {
  if (!ctx->configured) return visocu_set_error(ctx, VISOCU_ESTATE, "context not configured");
  if (n <= 0 || !frames) return visocu_set_error(ctx, VISOCU_EINVAL, "empty frame list");
  for (int i = 0; i < n; i++)
    if (frames[i] < 0 || frames[i] >= ctx->n_frames) return visocu_set_error(ctx, VISOCU_EINVAL, "frame %d out of range", frames[i]);
  return VISOCU_OK;
}

extern "C" int visocu_frame_counts(visocu_ctx* ctx, int32_t n, const int32_t* frames, int32_t* n_sparse, int32_t* n_dense) {
  if (!ctx) return VISOCU_EINVAL;
  int rc = check_frames(ctx, n, frames);
  if (rc) return rc;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((rc = visocu_ensure_pinned(ctx, (size_t)n * 16))) return rc;
  int32_t* stage = (int32_t*)ctx->pinned;
  for (int i = 0; i < n; i++)
    CU_COPY(ctx, stage + 4 * i, ctx->frames_h[frames[i]].counts, 16, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  for (int i = 0; i < n; i++) {
    if (stage[4 * i + 2]) return visocu_set_error(ctx, VISOCU_ECAPACITY, "feature list of frame %d overflowed", frames[i]);
    ctx->h_counts[2 * (size_t)frames[i] + 0] = stage[4 * i + 0];
    ctx->h_counts[2 * (size_t)frames[i] + 1] = stage[4 * i + 1];
    if (n_sparse) n_sparse[i] = stage[4 * i + 0];
    if (n_dense) n_dense[i] = stage[4 * i + 1];
  }
  return VISOCU_OK;
}

// Run `enqueue` on the lane's stream, or replay it as a CUDA graph once the same call (same key) has been seen twice: the
// first time buffers get their final size, the second time the stream is captured, from then on one graph launch replaces
// the individual launches and copies.  Everything `enqueue` does must depend on the key only.
static int run_or_replay_impl(visocu_ctx* ctx, visocu_graph& g, uint64_t key, const std::function<int()>& enqueue, const char** what);
int visocu_run_or_replay(visocu_ctx* ctx, visocu_graph& g, uint64_t key, const std::function<int()>& enqueue) {
  static const bool dbg = getenv("VISOCU_GRAPH_DEBUG") != nullptr;
  if (!dbg) { const char* w; return run_or_replay_impl(ctx, g, key, enqueue, &w); }
  struct timespec a, b; clock_gettime(CLOCK_MONOTONIC, &a);
  const char* what = "?";
  const int rc = run_or_replay_impl(ctx, g, key, enqueue, &what);
  clock_gettime(CLOCK_MONOTONIC, &b);
  fprintf(stderr, "[graph] lane %d %s %s key %016llx %.1f us\n", ctx->lane, &g == &ctx->g_push ? "push " : "match", what, (unsigned long long)key,
          (b.tv_sec - a.tv_sec) * 1e6 + (b.tv_nsec - a.tv_nsec) * 1e-3);
  return rc;
}
static int run_or_replay_impl(visocu_ctx* ctx, visocu_graph& g, uint64_t key, const std::function<int()>& enqueue, const char** what) {
  *what = "plain";
  if (!ctx->use_graphs || ctx->profile) return enqueue();
  if (g.key != key) { destroy_graph(g); g.key = key; }
  if (g.exec) {
    *what = "replay";
    CU_TRY(ctx, cudaGraphLaunch(g.exec, ctx->stream));
    ctx->launches += (uint64_t)g.seen;                   // kernels inside the graph
    return VISOCU_OK;
  }
  if (g.seen == 0) { g.seen = 1; return enqueue(); }
  if (g.seen < 0) return enqueue();                      // capture failed before: stay with plain launches
  const uint64_t l0 = ctx->launches;
  *what = "capture";
  CU_TRY(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
  const int rc = enqueue();
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
  if (rc != VISOCU_OK || e != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    g.seen = -1;
    ctx->launches = l0;
    *what = "capture-failed";
    return rc != VISOCU_OK ? rc : enqueue();
  }
  const int kernels = (int)(ctx->launches - l0);
  cudaGraphExec_t exec = nullptr;
  const cudaError_t e2 = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e2 != cudaSuccess) { cudaGetLastError(); g.seen = -1; ctx->launches = l0; return enqueue(); }
  g.exec = exec; g.seen = kernels;
  CU_TRY(ctx, cudaGraphLaunch(g.exec, ctx->stream));
  return VISOCU_OK;
}

static uint64_t hash_words(uint64_t h, const void* data, size_t bytes) {
  const uint8_t* p = (const uint8_t*)data;
  for (size_t i = 0; i < bytes; i++) { h ^= p[i]; h *= 1099511628211ull; }
  return h;
}

// One batch (at most VISO_MAX_BATCH frames) of a push: host images cross PCIe as ONE contiguous transfer each into a staging
// area (a pitched host-to-device copy of 376 unaligned 1241-byte rows is several times slower than the 0.47 MB it moves);
// then, graph-able: the table of source pointers, the re-pitch kernel and the feature kernels.  cams (or null): the push is
// rectifying, image i is a raw image of the maps' source size and k_rectify resamples it with map cams->c[i] in place of
// the re-pitch.
static int push_batch(visocu_ctx* ctx, const SlotList& sl, const uint8_t* const* imgs, const CamList* cams, int32_t bpl_in, int32_t on_device) {
  const Geometry& g = ctx->g;
  int rc;
  const int w_in = cams ? ctx->rect_src_w : g.w, h_in = cams ? ctx->rect_src_h : g.h;
  const size_t stage_stride = align_up((size_t)bpl_in * h_in, 256);
  const bool direct = !cams && on_device != 1 && bpl_in == g.bpl;  // already in the frame layout: straight into the frame planes
  bool async_pinned = false;                              // on_device = 0: the caller may reuse its buffers when the call returns
  if (on_device != 1 && !direct) {
    const size_t want = stage_stride * (size_t)sl.n;
    if (want > ctx->img_stage_bytes) {
      CU_TRY(ctx, visocu_stream_wait(ctx));
      visocu_drop_lane_graphs(ctx);
      if (ctx->img_stage) cudaFree(ctx->img_stage);
      ctx->img_stage = nullptr; ctx->img_stage_bytes = 0;
      CU_TRY(ctx, cudaMalloc(&ctx->img_stage, want));
      ctx->img_stage_bytes = want;
    }
  }
  if (!ctx->src_table) {
    CU_TRY(ctx, cudaMalloc((void**)&ctx->src_table, sizeof(void*) * VISO_MAX_BATCH));
    CU_TRY(ctx, cudaMallocHost((void**)&ctx->src_table_pin, sizeof(void*) * VISO_MAX_BATCH));
  }
  if (!ctx->counts_stage) CU_TRY(ctx, cudaMalloc(&ctx->counts_stage, VISO_MAX_BATCH * 16));
  if (!ctx->ev_push) CU_TRY(ctx, cudaEventCreateWithFlags(&ctx->ev_push, cudaEventDisableTiming));
  for (int i = 0; i < sl.n; i++) {
    if (!imgs[i]) return visocu_set_error(ctx, VISOCU_EINVAL, "null image %d", i);
    const int f = sl.s[i];
    if (on_device == 1) {
      ctx->src_table_pin[i] = imgs[i];
    } else {
      // pinned host memory is copied asynchronously (pageable memory is staged by the driver before the copy call returns)
      // (on_device = 2: the caller keeps the images valid until the step is collected, nothing to wait for.  Letting the
      // layout kernel read pinned images in place over PCIe instead of copying them was tried: e2e 54 k -> 38 k pairs/s)
      bool pinned = false;
      if (on_device == 0) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, imgs[i]) == cudaSuccess) pinned = at.type == cudaMemoryTypeHost;
        else cudaGetLastError();
      }
      if (direct) {
        CU_COPY(ctx, ctx->frames_h[f].img, imgs[i], (size_t)bpl_in * g.h, cudaMemcpyHostToDevice);
      } else {
        uint8_t* stage = ctx->img_stage + (size_t)i * stage_stride;
        CU_COPY(ctx, stage, imgs[i], (size_t)bpl_in * (h_in - 1) + w_in, cudaMemcpyHostToDevice);
        ctx->src_table_pin[i] = stage;
      }
      if (pinned) async_pinned = true;
    }
    ctx->frame_valid[f] = 1;
  }
  uint64_t key = hash_words(1469598103934665603ull, &sl.n, sizeof(int));
  key = hash_words(key, sl.s, sizeof(int) * (size_t)sl.n);
  key = hash_words(key, &bpl_in, sizeof bpl_in);
  key = hash_words(key, &direct, sizeof direct);
  if (cams) {                                             // the maps and their source size are fixed between two set calls
    const uint8_t rect = 1;
    key = hash_words(key, &rect, 1);
    key = hash_words(key, cams->c, sizeof(int32_t) * (size_t)sl.n);
  }
  ctx->in_step++;
  rc = visocu_run_or_replay(ctx, ctx->g_push, key, [&]() -> int {
    if (!direct) {
      CU_TRY(ctx, cudaMemcpyAsync((void*)ctx->src_table, (const void*)ctx->src_table_pin, sizeof(void*) * (size_t)sl.n, cudaMemcpyHostToDevice, ctx->stream));
      if (cams) {
        visocu_launch_rectify(ctx, sl, *cams, bpl_in);
      } else {
        int gx = (g.bpl / 4 * g.h + 255) / 256; if (gx > 64) gx = 64;
        k_repitch<<<dim3(gx, sl.n), 256, 0, ctx->stream>>>(g, ctx->frames_d, sl, ctx->src_table, bpl_in);
      }
      CU_LAUNCH_CHECK(ctx);
    }
    return visocu_launch_features(ctx, sl);
  });
  ctx->in_step--;
  if (rc) return rc;
  CU_TRY(ctx, cudaEventRecord(ctx->ev_push, ctx->stream));
  if (async_pinned) CU_TRY(ctx, visocu_stream_wait(ctx));            // "read only during the call" also for pinned sources
  return VISOCU_OK;
}

// cam (or null): a rectifying push, image k resampled with map cam[k]; the caller has checked cam and bpl_in
static int push_frames(visocu_ctx* ctx, int32_t n, const int32_t* frames, const uint8_t* const* imgs, const int32_t* cam,
                       int32_t bpl_in, int32_t on_device, int32_t* n_sparse, int32_t* n_dense) {
  int rc;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  for (int start = 0; start < n; start += VISO_MAX_BATCH) {
    SlotList sl;
    CamList cl;
    sl.n = n - start < VISO_MAX_BATCH ? n - start : VISO_MAX_BATCH;
    for (int i = 0; i < sl.n; i++) sl.s[i] = frames[start + i];
    if (cam) for (int i = 0; i < sl.n; i++) cl.c[i] = cam[start + i];
    if ((rc = push_batch(ctx, sl, imgs + start, cam ? &cl : nullptr, bpl_in, on_device))) return rc;
    if (!n_sparse && !n_dense) {
      // Lazy mode: nobody asked for the record counts, so nothing is read back and nothing is waited for.  The matching
      // call that follows takes the counts from device memory (visocu_match_fused) or fetches them (visocu_frame_counts).
      for (int i = 0; i < sl.n; i++) { ctx->h_counts[2 * (size_t)sl.s[i]] = -1; ctx->h_counts[2 * (size_t)sl.s[i] + 1] = -1; }
      continue;
    }
    // the caller wants the record counts: one small read-back per launch
    if ((rc = visocu_ensure_pinned(ctx, (size_t)sl.n * 16))) return rc;
    int32_t* stage = (int32_t*)ctx->pinned;
    CU_COPY(ctx, stage, ctx->counts_stage, (size_t)sl.n * 16, cudaMemcpyDeviceToHost);
    CU_TRY(ctx, visocu_stream_wait(ctx));
    for (int i = 0; i < sl.n; i++) {
      const int f = sl.s[i];
      if (stage[4 * i + 2]) return visocu_set_error(ctx, VISOCU_ECAPACITY, "feature list of frame %d overflowed", f);
      ctx->h_counts[2 * (size_t)f + 0] = stage[4 * i + 0];
      ctx->h_counts[2 * (size_t)f + 1] = stage[4 * i + 1];
      if (n_sparse) n_sparse[start + i] = stage[4 * i + 0];
      if (n_dense) n_dense[start + i] = stage[4 * i + 1];
    }
  }
  return VISOCU_OK;
}

extern "C" int visocu_push_frames(visocu_ctx* ctx, int32_t n, const int32_t* frames, const uint8_t* const* imgs,
                                  int32_t bpl_in, int32_t on_device, int32_t* n_sparse, int32_t* n_dense) {
  if (!ctx) return VISOCU_EINVAL;
  int rc = check_frames(ctx, n, frames);
  if (rc) return rc;
  if (!imgs) return visocu_set_error(ctx, VISOCU_EINVAL, "null image list");
  const Geometry& g = ctx->g;
  if (bpl_in < g.w) return visocu_set_error(ctx, VISOCU_EINVAL, "bytes per line %d < width %d", bpl_in, g.w);   // matcher.cpp:103
  return push_frames(ctx, n, frames, imgs, nullptr, bpl_in, on_device, n_sparse, n_dense);
}

extern "C" int visocu_push_frames_rectified(visocu_ctx* ctx, int32_t n, const int32_t* frames, const uint8_t* const* imgs,
                                            const int32_t* cam, int32_t bpl_in, int32_t on_device, int32_t* n_sparse, int32_t* n_dense) {
  if (!ctx) return VISOCU_EINVAL;
  int rc = check_frames(ctx, n, frames);
  if (rc) return rc;
  if (!imgs || !cam) return visocu_set_error(ctx, VISOCU_EINVAL, "null image or camera list");
  if (ctx->rect_n == 0) return visocu_set_error(ctx, VISOCU_ESTATE, "no rectification maps on this context (visocu_set_rectification)");
  for (int i = 0; i < n; i++)
    if (cam[i] < 0 || cam[i] >= ctx->rect_n) return visocu_set_error(ctx, VISOCU_EINVAL, "camera %d of image %d out of range (%d maps)", cam[i], i, ctx->rect_n);
  if (bpl_in < ctx->rect_src_w) return visocu_set_error(ctx, VISOCU_EINVAL, "bytes per line %d < raw width %d", bpl_in, ctx->rect_src_w);
  return push_frames(ctx, n, frames, imgs, cam, bpl_in, on_device, n_sparse, n_dense);
}

extern "C" int visocu_get_features(visocu_ctx* ctx, int32_t frame, int32_t pass, int32_t* out12, int32_t cap, int32_t* n_out) {
  if (!ctx) return VISOCU_EINVAL;
  int rc = check_frames(ctx, 1, &frame);
  if (rc) return rc;
  if (pass < 0 || pass > 1) return visocu_set_error(ctx, VISOCU_EINVAL, "pass must be 0 or 1");
  if (!ctx->frame_valid[frame]) return visocu_set_error(ctx, VISOCU_ESTATE, "frame %d holds no features", frame);
  if (ctx->h_counts[2 * (size_t)frame] < 0) { if ((rc = visocu_frame_counts(ctx, 1, &frame, nullptr, nullptr))) return rc; }
  int32_t n = ctx->h_counts[2 * (size_t)frame + pass];
  if (n_out) *n_out = n;
  if (!out12) return VISOCU_OK;
  if (cap < n) return visocu_set_error(ctx, VISOCU_ECAPACITY, "need room for %d records", n);
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if (n > 0) CU_COPY(ctx, out12, ctx->frames_h[frame].rec[pass], (size_t)n * 48, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}

extern "C" int visocu_get_plane(visocu_ctx* ctx, int32_t frame, int32_t which, uint8_t* out, size_t cap, int32_t* dims3) {
  if (!ctx) return VISOCU_EINVAL;
  int rc = check_frames(ctx, 1, &frame);
  if (rc) return rc;
  const Geometry& g = ctx->g;
  const FrameDev& F = ctx->frames_h[frame];
  const uint8_t* src = nullptr;
  int w = g.wm, h = g.hm, bpl = g.bplm;
  switch (which) {
    case 0: src = F.du; break;
    case 1: src = F.dv; break;
    case 2: src = F.du_full; w = g.w; h = g.h; bpl = g.bpl; break;
    case 3: src = F.dv_full; w = g.w; h = g.h; bpl = g.bpl; break;
    case 4: src = F.img; w = g.w; h = g.h; bpl = g.bpl; break;
    case 5: src = F.half; if (src && ctx->fused_half) { int rc2 = visocu_make_half_image(ctx, frame); if (rc2) return rc2; } break;
    default: return visocu_set_error(ctx, VISOCU_EINVAL, "unknown plane %d", which);
  }
  if (!src) return visocu_set_error(ctx, VISOCU_ESTATE, "plane %d does not exist in this configuration", which);
  if (dims3) { dims3[0] = w; dims3[1] = h; dims3[2] = bpl; }
  if (!out) return VISOCU_OK;
  size_t bytes = (size_t)bpl * h;
  if (cap < bytes) return visocu_set_error(ctx, VISOCU_ECAPACITY, "plane needs %zu bytes", bytes);
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_COPY(ctx, out, src, bytes, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}
