// Rectification of raw camera images behind include/visocu.h: the per-camera maps (built on the host by host/rectify.cpp,
// kept in HBM) and k_rectify, which takes k_repitch's place in a rectifying push.
#include "visocu_internal.cuh"
#include "../host/rectify.h"

#include <cstring>

namespace {
struct RectMaps { const int2* m[2]; int src_w, src_h; };
}  // namespace

// One launch for all frames of a push, with k_repitch's shape: blockIdx.y = frame, table[] = its raw image (device copy or
// the caller's device pointer), one 32-bit word of 4 output pixels per thread.  Each pixel reads its map entry (x, y in
// 1/32 pixel, already clamped to the raw image) and interpolates the 2x2 neighbourhood in integers; the right and lower
// neighbours are clamped to the last column and row.  Pad columns up to bpl are written as zero, as k_repitch writes them.
// The map (8 B per pixel) dominates the traffic: 3.7 MB per camera at 1241x376, read by every frame of the push from L2.
__global__ void __launch_bounds__(256) k_rectify(Geometry g, const FrameDev* frames, SlotList sl, CamList cams, RectMaps maps,
                                                 const uint8_t* const* table, int bpl_in) {
  const uint8_t* __restrict__ src = table[blockIdx.y];
  const int2* __restrict__ map = cams.c[blockIdx.y] ? maps.m[1] : maps.m[0];
  uint8_t* dst = frames[sl.s[blockIdx.y]].img;
  const int wpr = g.bpl >> 2, total = wpr * g.h;
  const int xm = maps.src_w - 1, ym = maps.src_h - 1;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int y = idx / wpr, x0 = 4 * (idx - y * wpr);
    const int2* row = map + (size_t)y * g.w;
    uint32_t word = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int x = x0 + k;
      if (x < g.w) {
        const int2 e = __ldg(row + x);
        const int ix = e.x >> 5, iy = e.y >> 5, fx = e.x & 31, fy = e.y & 31;
        const int ix1 = min(ix + 1, xm);
        const uint8_t* r0 = src + (size_t)iy * bpl_in;
        const uint8_t* r1 = src + (size_t)min(iy + 1, ym) * bpl_in;
        const int p00 = r0[ix], p01 = r0[ix1], p10 = r1[ix], p11 = r1[ix1];
        const int v = ((32 - fx) * (32 - fy) * p00 + fx * (32 - fy) * p01 + (32 - fx) * fy * p10 + fx * fy * p11 + 512) >> 10;
        word |= (uint32_t)v << (8 * k);
      }
    }
    *(uint32_t*)(dst + (size_t)y * g.bpl + x0) = word;
  }
}

void visocu_launch_rectify(visocu_ctx* ctx, const SlotList& sl, const CamList& cams, int bpl_in) {
  const Geometry& g = ctx->g;
  RectMaps maps = {{ctx->rect_map[0], ctx->rect_map[1]}, ctx->rect_src_w, ctx->rect_src_h};
  int gx = (g.bpl / 4 * g.h + 255) / 256;
  if (gx > 256) gx = 256;
  k_rectify<<<dim3(gx, sl.n), 256, 0, ctx->stream>>>(g, ctx->frames_d, sl, cams, maps, ctx->src_table, bpl_in);
}

void visocu_free_rectification(visocu_ctx* ctx) {
  for (int k = 0; k < 2; k++) {
    if (ctx->rect_map[k]) cudaFree(ctx->rect_map[k]);
    ctx->rect_map[k] = nullptr;
    std::vector<int32_t>().swap(ctx->rect_host[k]);
  }
  ctx->rect_n = ctx->rect_src_w = ctx->rect_src_h = 0;
}

extern "C" int visocu_set_rectification(visocu_ctx* ctx, int32_t n_cams, const visocu_camera* cams, int32_t src_w, int32_t src_h) {
  if (!ctx) return VISOCU_EINVAL;
  if (!ctx->configured) return visocu_set_error(ctx, VISOCU_ESTATE, "context not configured");
  if (n_cams < 0 || n_cams > 2) return visocu_set_error(ctx, VISOCU_EINVAL, "%d cameras: at most 2", n_cams);
  if (n_cams > 0 && !cams) return visocu_set_error(ctx, VISOCU_EINVAL, "null camera list");
  const Geometry& g = ctx->g;
  std::vector<int32_t> host[2];
  for (int k = 0; k < n_cams; k++) {
    const char* why = "";
    host[k].resize(2 * (size_t)g.w * g.h);
    if (!visob::rectifyMap(cams[k], src_w, src_h, g.w, g.h, host[k].data(), &why))
      return visocu_set_error(ctx, VISOCU_EINVAL, "camera %d: %s", k, why);
  }
  // pushes in flight on any lane may still read the old maps, and the push graphs bake their addresses
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  for (int l = 0; l < VISO_LANES; l++) if (ctx->lanes[l].created && l != ctx->lane && ctx->lanes[l].stream) cudaStreamSynchronize(ctx->lanes[l].stream);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  visocu_drop_graphs(ctx);
  visocu_free_rectification(ctx);
  for (int k = 0; k < n_cams; k++) {
    const size_t bytes = host[k].size() * sizeof(int32_t);
    CU_TRY(ctx, cudaMalloc((void**)&ctx->rect_map[k], bytes));
    CU_TRY(ctx, cudaMemcpy(ctx->rect_map[k], host[k].data(), bytes, cudaMemcpyHostToDevice));
    ctx->rect_host[k].swap(host[k]);
  }
  ctx->rect_n = n_cams;
  ctx->rect_src_w = n_cams ? src_w : 0;
  ctx->rect_src_h = n_cams ? src_h : 0;
  return VISOCU_OK;
}

extern "C" int visocu_get_rectify_map(visocu_ctx* ctx, int32_t cam, int32_t* out, size_t cap) {
  if (!ctx || !out) return VISOCU_EINVAL;
  if (cam < 0 || cam >= ctx->rect_n) return visocu_set_error(ctx, VISOCU_EINVAL, "camera %d out of range (%d maps)", cam, ctx->rect_n);
  const std::vector<int32_t>& m = ctx->rect_host[cam];
  if (cap < m.size()) return visocu_set_error(ctx, VISOCU_ECAPACITY, "the map needs %zu entries", m.size());
  memcpy(out, m.data(), m.size() * sizeof(int32_t));
  return VISOCU_OK;
}
