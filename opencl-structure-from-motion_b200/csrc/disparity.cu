// Dense stereo disparity behind include/visocu.h: semi-global matching (Hirschmueller 2008) on the full-resolution images
// of pushed frame slots.  Census 9x7 per image, Hamming costs computed on the fly from the census words (no cost volume),
// 4 or 8 path recurrences summed into S (uint16), then winner, uniqueness, left-right check and sub-pixel offset in one
// pass over S.  oracle/sgm_oracle.c states the same algorithm in plain C; the device is bit-identical to it.
//
// Launches per group of at most VISO_MAX_BATCH pairs: k_census, k_sgm_rows, k_sgm_cols, [k_sgm_diag, k_sgm_antidiag],
// k_sgm_select.  Scratch per pair: census 2 w h 8 B, S w h D 2 B (and w h 2 B of output for host destinations).
#include "visocu_internal.cuh"

namespace {

constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr int BIG = 1 << 14;           // "no neighbour" in the path minimum; BIG + P1 stays far above any L

struct PairList { int l[VISO_MAX_BATCH], r[VISO_MAX_BATCH]; };
struct OutList { int16_t* p[VISO_MAX_BATCH]; };
struct Dims { int w, h, bpl; };

// K uint16 of one lane in one vector access (K = D / 32 disparities per lane: 4, 8 or 16 bytes)
template <int K> struct alignas(2 * K) U16K { uint16_t v[K]; };

// One thread per pixel; grid z = 2 x pairs (left, right).  Bit b set when the neighbour is darker than the centre, the
// neighbours in row-major order of (dy, dx), dy in [-3, 3], dx in [-4, 4], centre skipped; coordinates clamped.
__global__ void __launch_bounds__(256) k_census(const FrameDev* frames, PairList pl, Dims g, uint64_t* cen) {
  const int k = blockIdx.z >> 1, side = blockIdx.z & 1;
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
  if (x >= g.w || y >= g.h) return;
  const uint8_t* __restrict__ img = frames[side ? pl.r[k] : pl.l[k]].img;
  const int c = img[(size_t)y * g.bpl + x];
  uint64_t bits = 0;
  int b = 0;
#pragma unroll
  for (int dy = -3; dy <= 3; dy++) {
    const uint8_t* row = img + (size_t)min(max(y + dy, 0), g.h - 1) * g.bpl;
#pragma unroll
    for (int dx = -4; dx <= 4; dx++) {
      if (dx == 0 && dy == 0) continue;
      bits |= (uint64_t)(__ldg(row + min(max(x + dx, 0), g.w - 1)) < c) << b;
      b++;
    }
  }
  cen[((size_t)blockIdx.z * g.h + y) * g.w + x] = bits;
}

// One warp walks one line of n pixels from (x0, y0) in steps (sx, sy), then back from the far end.  Lane l holds
// d = l K .. l K + K - 1; M comes from a warp reduction, the d +- 1 neighbours across lanes from two shuffles.  The next
// pixel's census words and S are loaded before the current pixel is computed (within a pass only: pass 1 reads the S
// that pass 0 wrote).  INIT: pass 0 writes S instead of adding to it (the first path of a call).
template <int K, bool INIT>
__device__ __forceinline__ void sgm_line(const uint64_t* __restrict__ cenL, const uint64_t* __restrict__ cenR, uint16_t* S,
                                         int w, int x0, int y0, int sx, int sy, int n, int p1, int p2) {
  constexpr int D = 32 * K;
  const int lane = threadIdx.x & 31, d0 = lane * K;
  for (int pass = 0; pass < 2; pass++) {
    const int dx = pass ? -sx : sx, dy = pass ? -sy : sy;
    int x = pass ? x0 + (n - 1) * sx : x0, y = pass ? y0 + (n - 1) * sy : y0;
    const bool write_only = INIT && pass == 0;
    uint64_t cl, cr[K];
    U16K<K> sv;
    auto load = [&](int xx, int yy, uint64_t& l, uint64_t (&r)[K], U16K<K>& s) {
      const size_t pix = (size_t)yy * w + xx;
      l = cenL[pix];
#pragma unroll
      for (int j = 0; j < K; j++) r[j] = xx - d0 - j >= 0 ? cenR[pix - d0 - j] : 0;
      if (!write_only) s = *(const U16K<K>*)(S + pix * D + d0);
    };
    load(x, y, cl, cr, sv);
    int Lp[K], Mp = 0;
    for (int i = 0; i < n; i++) {
      uint64_t ncl = 0, ncr[K];
      U16K<K> nsv;
      if (i + 1 < n) load(x + dx, y + dy, ncl, ncr, nsv);
      int L[K];
      if (i == 0) {
#pragma unroll
        for (int j = 0; j < K; j++) L[j] = x - d0 - j >= 0 ? __popcll(cl ^ cr[j]) : 62;
      } else {
        const int lo = __shfl_up_sync(FULL, Lp[K - 1], 1), hi = __shfl_down_sync(FULL, Lp[0], 1);
#pragma unroll
        for (int j = 0; j < K; j++) {
          const int c = x - d0 - j >= 0 ? __popcll(cl ^ cr[j]) : 62;
          const int dm = j > 0 ? Lp[j - 1] : (lane > 0 ? lo : BIG);
          const int dp = j < K - 1 ? Lp[j + 1] : (lane < 31 ? hi : BIG);
          L[j] = c + min(min(Lp[j], Mp + p2), min(dm, dp) + p1) - Mp;
        }
      }
      int m = L[0];
#pragma unroll
      for (int j = 1; j < K; j++) m = min(m, L[j]);
      Mp = (int)__reduce_min_sync(FULL, (unsigned)m);
      U16K<K> o;
#pragma unroll
      for (int j = 0; j < K; j++) { o.v[j] = (uint16_t)(write_only ? L[j] : sv.v[j] + L[j]); Lp[j] = L[j]; }
      *(U16K<K>*)(S + ((size_t)y * w + x) * D + d0) = o;
      if (i + 1 < n) {
        x += dx; y += dy;
        cl = ncl; sv = nsv;
#pragma unroll
        for (int j = 0; j < K; j++) cr[j] = ncr[j];
      }
    }
  }
}

// The lines of one direction pair: blockIdx.y = pair, 4 warps (lines) per block.
//   KIND 0: rows, (1, 0) and (-1, 0) (first path: writes S);  1: columns, (0, 1) and (0, -1);
//   2: diagonals x - y = c, (1, 1) and (-1, -1);  3: anti-diagonals x + y = c, (-1, 1) and (1, -1).
template <int K, int KIND>
__device__ __forceinline__ void sgm_lines(const uint64_t* cen, uint16_t* S, Dims g, int p1, int p2) {
  const int line = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int w = g.w, h = g.h;
  const int nlines = KIND == 0 ? h : (KIND == 1 ? w : w + h - 1);
  if (line >= nlines) return;
  const size_t plane = (size_t)w * h;
  const uint64_t* cenL = cen + 2 * plane * blockIdx.y;
  uint16_t* Sk = S + plane * (32 * K) * blockIdx.y;
  int x0, y0, sx, sy, n;
  if (KIND == 0)      { x0 = 0; y0 = line; sx = 1; sy = 0; n = w; }
  else if (KIND == 1) { x0 = line; y0 = 0; sx = 0; sy = 1; n = h; }
  else if (KIND == 2) { const int c = line - (h - 1); x0 = max(c, 0); y0 = max(-c, 0); sx = 1; sy = 1; n = min(w - x0, h - y0); }
  else                { y0 = max(0, line - (w - 1)); x0 = line - y0; sx = -1; sy = 1; n = min(x0 + 1, h - y0); }
  sgm_line<K, KIND == 0>(cenL, cenL + plane, Sk, w, x0, y0, sx, sy, n, p1, p2);
}

template <int K> __global__ void __launch_bounds__(128) k_sgm_rows(const uint64_t* cen, uint16_t* S, Dims g, int p1, int p2) { sgm_lines<K, 0>(cen, S, g, p1, p2); }
template <int K> __global__ void __launch_bounds__(128) k_sgm_cols(const uint64_t* cen, uint16_t* S, Dims g, int p1, int p2) { sgm_lines<K, 1>(cen, S, g, p1, p2); }
template <int K> __global__ void __launch_bounds__(128) k_sgm_diag(const uint64_t* cen, uint16_t* S, Dims g, int p1, int p2) { sgm_lines<K, 2>(cen, S, g, p1, p2); }
template <int K> __global__ void __launch_bounds__(128) k_sgm_antidiag(const uint64_t* cen, uint16_t* S, Dims g, int p1, int p2) { sgm_lines<K, 3>(cen, S, g, p1, p2); }

__device__ __forceinline__ int floor_div(int a, int b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }   // b > 0

// One block per (row, pair), one warp per pixel: d* = the smallest d of min S (key S << 9 | d), uniqueness and sub-pixel
// offset; the right map dR(x') = the smallest d of min S(x' + d, y, d) collects in shared memory by atomicMin on the same
// keys.  After a barrier, the left-right check and one coalesced row of int16 output.  Shared memory: 8 w bytes.
template <int K>
__global__ void __launch_bounds__(256) k_sgm_select(const uint16_t* S, Dims g, visocu_sgm_params a, OutList out) {
  constexpr int D = 32 * K;
  extern __shared__ uint32_t sm[];
  const int w = g.w, y = blockIdx.x, lane = threadIdx.x & 31, d0 = lane * K;
  uint32_t* rmin = sm;
  int32_t* val = (int32_t*)(sm + w);
  const bool lr = a.lr_max_diff >= 0;
  for (int i = threadIdx.x; i < w; i += blockDim.x) rmin[i] = 0xFFFFFFFFu;
  __syncthreads();
  const uint16_t* row = S + ((size_t)blockIdx.y * g.h + y) * w * D;
  for (int x = threadIdx.x >> 5; x < w; x += blockDim.x >> 5) {
    const U16K<K> s = *(const U16K<K>*)(row + (size_t)x * D + d0);
    uint32_t key = 0xFFFFFFFFu;
#pragma unroll
    for (int j = 0; j < K; j++) key = min(key, (uint32_t)s.v[j] << 9 | (uint32_t)(d0 + j));
    key = __reduce_min_sync(FULL, key);
    const int ds = (int)(key & 511), smin = (int)(key >> 9);
    int m2 = BIG, sa = 0, sc = 0;
#pragma unroll
    for (int j = 0; j < K; j++) {
      const int d = d0 + j;
      if (abs(d - ds) > 1) m2 = min(m2, (int)s.v[j]);
      if (d == ds - 1) sa = s.v[j];
      if (d == ds + 1) sc = s.v[j];
    }
    m2 = (int)__reduce_min_sync(FULL, (unsigned)m2);
    sa = (int)__reduce_add_sync(FULL, (unsigned)sa);
    sc = (int)__reduce_add_sync(FULL, (unsigned)sc);
    if (lr) {
#pragma unroll
      for (int j = 0; j < K; j++)
        if (x - d0 - j >= 0) atomicMin(&rmin[x - d0 - j], (uint32_t)s.v[j] << 9 | (uint32_t)(d0 + j));
    }
    if (lane == 0) {
      int v = 16 * ds;
      if (a.subpixel && ds > 0 && ds < D - 1) {
        const int den = sa + sc - 2 * smin;
        if (den > 0) v += floor_div(16 * (sa - sc) + den, 2 * den);
      }
      val[x] = 100 * smin > a.uniqueness * m2 ? -1 : (ds << 16 | v);
    }
  }
  __syncthreads();
  int16_t* o = out.p[blockIdx.y] + (size_t)y * w;
  for (int x = threadIdx.x; x < w; x += blockDim.x) {
    const int e = val[x];
    int v = -1;
    if (e >= 0) {
      const int ds = e >> 16;
      v = e & 0xFFFF;
      if (lr && (x - ds < 0 || abs((int)(rmin[x - ds] & 511) - ds) > a.lr_max_diff)) v = -1;
    }
    o[x] = (int16_t)v;
  }
}

template <int K>
int launch_group(visocu_ctx* ctx, const PairList& pl, int nb, const visocu_sgm_params& p, uint64_t* cen, uint16_t* S, const OutList& ol) {
  const Geometry& G = ctx->g;
  const Dims g{G.w, G.h, G.bpl};
  cudaStream_t st = ctx->stream;
  k_census<<<dim3((g.w + 31) / 32, (g.h + 7) / 8, 2 * nb), dim3(32, 8), 0, st>>>(ctx->frames_d, pl, g, cen);
  CU_LAUNCH_CHECK(ctx);
  k_sgm_rows<K><<<dim3((g.h + 3) / 4, nb), 128, 0, st>>>(cen, S, g, p.p1, p.p2);
  CU_LAUNCH_CHECK(ctx);
  k_sgm_cols<K><<<dim3((g.w + 3) / 4, nb), 128, 0, st>>>(cen, S, g, p.p1, p.p2);
  CU_LAUNCH_CHECK(ctx);
  if (p.paths == 8) {
    k_sgm_diag<K><<<dim3((g.w + g.h + 2) / 4, nb), 128, 0, st>>>(cen, S, g, p.p1, p.p2);
    CU_LAUNCH_CHECK(ctx);
    k_sgm_antidiag<K><<<dim3((g.w + g.h + 2) / 4, nb), 128, 0, st>>>(cen, S, g, p.p1, p.p2);
    CU_LAUNCH_CHECK(ctx);
  }
  const size_t smem = (size_t)8 * g.w;
  if (smem > 48 * 1024) CU_TRY(ctx, cudaFuncSetAttribute(k_sgm_select<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_sgm_select<K><<<dim3(g.h, nb), 256, smem, st>>>(S, g, p, ol);
  CU_LAUNCH_CHECK(ctx);
  return VISOCU_OK;
}

}  // namespace

extern "C" int visocu_sgm_check(const visocu_sgm_params* p) {
  if (!p) return VISOCU_EINVAL;
  const int D = p->max_disp;
  const bool ok = (D == 64 || D == 128 || D == 256) && (p->paths == 4 || p->paths == 8) && p->p1 >= 1 && p->p1 < p->p2 && p->p2 <= 150 &&
                  p->uniqueness >= 0 && p->uniqueness <= 100 && p->lr_max_diff >= -1 && p->lr_max_diff <= D &&
                  (p->subpixel == 0 || p->subpixel == 1);
  return ok ? VISOCU_OK : VISOCU_EINVAL;
}

extern "C" int visocu_disparity(visocu_ctx* ctx, int32_t n_pairs, const int32_t* left, const int32_t* right,
                                const visocu_sgm_params* p, int16_t* const* out, int32_t out_on_device) {
  if (!ctx) return VISOCU_EINVAL;
  if (!p) return visocu_set_error(ctx, VISOCU_EINVAL, "null disparity parameters");
  const int D = p->max_disp;
  if (visocu_sgm_check(p) != VISOCU_OK)
    return visocu_set_error(ctx, VISOCU_EINVAL, "disparity parameters out of range (max_disp %d, paths %d, p1 %d, p2 %d, uniqueness %d, "
                            "lr_max_diff %d, subpixel %d)", D, p->paths, p->p1, p->p2, p->uniqueness, p->lr_max_diff, p->subpixel);
  if (n_pairs < 0) return visocu_set_error(ctx, VISOCU_EINVAL, "n_pairs %d < 0", n_pairs);
  if (out_on_device != 0 && out_on_device != 1) return visocu_set_error(ctx, VISOCU_EINVAL, "out_on_device must be 0 or 1");
  if (n_pairs > 0 && (!left || !right || !out)) return visocu_set_error(ctx, VISOCU_EINVAL, "null pair or output list");
  if (!ctx->configured) return visocu_set_error(ctx, VISOCU_ESTATE, "context not configured");
  for (int k = 0; k < n_pairs; k++) {
    if (left[k] < 0 || left[k] >= ctx->n_frames || right[k] < 0 || right[k] >= ctx->n_frames)
      return visocu_set_error(ctx, VISOCU_EINVAL, "pair %d: frame (%d, %d) out of range", k, left[k], right[k]);
    if (!out[k]) return visocu_set_error(ctx, VISOCU_EINVAL, "pair %d: null output", k);
  }
  for (int k = 0; k < n_pairs; k++)
    if (!ctx->frame_valid[left[k]] || !ctx->frame_valid[right[k]])
      return visocu_set_error(ctx, VISOCU_ESTATE, "pair %d: frame (%d, %d) was never pushed", k, left[k], right[k]);
  if (n_pairs == 0) return VISOCU_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  // the frames may have been pushed on another lane: start behind the last push of every other lane
  for (int l = 0; l < VISO_LANES; l++)
    if (l != ctx->lane && ctx->lanes[l].created && ctx->lanes[l].ev_push) CU_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->lanes[l].ev_push, 0));
  const Geometry& g = ctx->g;
  const size_t plane = (size_t)g.w * g.h;
  const int groups = (n_pairs + VISO_MAX_BATCH - 1) / VISO_MAX_BATCH;
  const int nmax = n_pairs < VISO_MAX_BATCH ? n_pairs : VISO_MAX_BATCH;
  const size_t cen_bytes = align_up(2 * plane * 8, 256), s_bytes = align_up(plane * D * 2, 256), o_bytes = align_up(plane * 2, 256);
  int rc = visocu_ensure_scratch(ctx, (size_t)nmax * (cen_bytes + s_bytes + (out_on_device ? 0 : o_bytes)));
  if (rc) return rc;
  uint8_t* sb = (uint8_t*)ctx->scratch;
  uint64_t* cen = (uint64_t*)sb;
  uint16_t* S = (uint16_t*)(sb + nmax * cen_bytes);
  int16_t* ob = (int16_t*)(sb + nmax * (cen_bytes + s_bytes));
  for (int gi = 0; gi < groups; gi++) {
    const int start = gi * VISO_MAX_BATCH, nb = n_pairs - start < VISO_MAX_BATCH ? n_pairs - start : VISO_MAX_BATCH;
    PairList pl;
    OutList ol;
    for (int k = 0; k < nb; k++) {
      pl.l[k] = left[start + k]; pl.r[k] = right[start + k];
      ol.p[k] = out_on_device ? out[start + k] : ob + (size_t)k * (o_bytes / 2);
    }
    rc = D == 64 ? launch_group<2>(ctx, pl, nb, *p, cen, S, ol)
                 : (D == 128 ? launch_group<4>(ctx, pl, nb, *p, cen, S, ol) : launch_group<8>(ctx, pl, nb, *p, cen, S, ol));
    if (rc) return rc;
    if (!out_on_device)
      for (int k = 0; k < nb; k++) CU_COPY(ctx, out[start + k], ol.p[k], plane * 2, cudaMemcpyDeviceToHost);
  }
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}
