// Post-filters of disparity maps behind include/visocu.h (visocu_disparity, visocu_disparity_filter): the masked 3x3
// median and speckle removal by connected components.  oracle/disp_filter_oracle.c states both in plain C; the
// device is bit-identical to it.
//
// Speckles: block-based union-find (Playne & Hawick 2018, Allegretti et al. 2019).  A label is the index of a pixel in the
// group's label array (map k starts at k w h, so two maps never join); every label points at a pixel of the same component
// with an index no larger than its own, and a root points at itself.  The tile pass and the merge both link the larger
// root under the smaller with atomicMin and retry with whatever the atomic returned, which gives the same partition
// whatever order the atomics land in; each component's root ends as its smallest index.
//
// Launches per group of at most VISO_MAX_BATCH maps: [k_disp_median3], [k_speckle_local, k_speckle_merge,
// k_speckle_count], k_speckle_apply (it stores the median's result when speckle removal is off).  Scratch per map:
// labels 4 w h, counts 4 w h, median output 2 w h bytes.
#include "visocu_internal.cuh"

namespace {

constexpr int TW = 32, TH = 32;        // speckle tile, one thread per pixel
constexpr int BIG16 = 0x7FFF;          // an invalid or clipped median sample: above every disparity
constexpr unsigned FULL = 0xFFFFFFFFu;

struct MapList { int16_t* p[VISO_MAX_BATCH]; };

__device__ __forceinline__ bool joined(int a, int b, int r16) { return a >= 0 && b >= 0 && abs(a - b) <= r16; }

// volatile: other threads of the launch move roots while this one walks
__device__ __forceinline__ int find_root(const int* L, int i) {
  int p = ((const volatile int*)L)[i];
  while (p != i) { i = p; p = ((const volatile int*)L)[i]; }
  return i;
}

// link the roots of a and b, the larger under the smaller; an atomicMin that finds its target no longer a root has moved
// that target under min(old parent, a), and the walk continues with the old parent
__device__ void unite(int* L, int a, int b) {
  while (true) {
    a = find_root(L, a); b = find_root(L, b);
    if (a == b) return;
    if (a > b) { const int t = a; a = b; b = t; }
    const int old = atomicMin(&L[b], a);
    if (old == b) return;
    b = old;
  }
}

__device__ __forceinline__ void cswap(int& a, int& b) { const int lo = min(a, b); b = max(a, b); a = lo; }

// One thread per pixel; grid z = map.  Clipped samples and invalid ones sort above every value (BIG16), so the n valid
// ones come first and the lower median is entry (n - 1) / 2 of the sorted nine.
__global__ void __launch_bounds__(256) k_disp_median3(MapList src, int16_t* dst, int w, int h) {
  const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y, k = blockIdx.z;
  if (x >= w || y >= h) return;
  const int16_t* __restrict__ m = src.p[k];
  const int c = __ldg(m + (size_t)y * w + x);
  int out = c;                                         // an invalid pixel stays as it is
  if (c >= 0) {
    int v[9], n = 0;
#pragma unroll
    for (int dy = -1; dy <= 1; dy++)
#pragma unroll
      for (int dx = -1; dx <= 1; dx++) {
        const int xx = x + dx, yy = y + dy;
        const int e = xx >= 0 && xx < w && yy >= 0 && yy < h ? __ldg(m + (size_t)yy * w + xx) : -1;
        n += e >= 0;
        v[(dy + 1) * 3 + dx + 1] = e >= 0 ? e : BIG16;
      }
#pragma unroll
    for (int round = 0; round < 9; round++)          // odd-even transposition: 9 rounds sort 9 values
#pragma unroll
      for (int i = round & 1; i + 1 < 9; i += 2) cswap(v[i], v[i + 1]);
    const int r = (n - 1) >> 1;
#pragma unroll
    for (int j = 0; j < 5; j++)                        // n <= 9: r <= 4; constant indices keep v in registers
      if (j == r) out = v[j];
  }
  dst[(size_t)k * w * h + (size_t)y * w + x] = (int16_t)out;
}

// One CTA per TW x TH tile of one map (grid z = map), one warp per tile row.  Within a row, every pixel points at the start
// of its run of joined pixels (ballot of the left joins, no atomics); the vertical joins then unite runs in shared memory,
// skipping a join that the pixel to the left already implies (both pixels joined up and the two upper pixels joined:
// Hennequin et al. 2018).  Then a pre-count of each tile component at its root (one shared atomic per root and warp), and
// every pixel's label = its tile root as an index of the group's arrays.  cnt receives the component's pixel count in the
// tile at the tile root and 0 everywhere else (other pixels, invalid pixels).
__global__ void __launch_bounds__(TW * TH) k_speckle_local(MapList src, int* lab, int* cnt, int w, int h, int r16) {
  static_assert(TW == 32, "one warp per tile row");
  __shared__ int L[TW * TH], V[TW * TH], N[TW * TH];
  __shared__ unsigned LJ[TH];
  const int tx = threadIdx.x, ty = threadIdx.y, i = ty * TW + tx;
  const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH, x = x0 + tx, y = y0 + ty;
  const bool in = x < w && y < h;
  const int v = in ? src.p[blockIdx.z][(size_t)y * w + x] : -1;
  const bool jl = joined(v, __shfl_up_sync(FULL, v, 1), r16) && tx > 0;
  const unsigned lj = __ballot_sync(FULL, jl);
  // bits 0..tx of ~lj mark run starts (bit 0 always); the run of tx starts at the highest of them
  L[i] = ty * TW + 31 - __clz(~lj & (FULL >> (31 - tx)));
  V[i] = v; N[i] = 0;
  if (tx == 0) LJ[ty] = lj;
  __syncthreads();
  const bool ju = ty > 0 && joined(v, V[i - TW], r16);
  const unsigned uj = __ballot_sync(FULL, ju);
  if (ju && !(jl && (uj >> (tx - 1) & 1) && (LJ[ty - 1] >> tx & 1))) unite(L, i, i - TW);
  __syncthreads();
  const int r = find_root(L, i);
  const unsigned same = __match_any_sync(FULL, v >= 0 ? r : -1 - tx);
  if (v >= 0 && tx == __ffs(same) - 1) atomicAdd(&N[r], __popc(same));
  __syncthreads();
  if (!in) return;
  const size_t base = (size_t)blockIdx.z * w * h;
  const size_t g = base + (size_t)y * w + x;
  lab[g] = (int)(base + (size_t)(y0 + r / TW) * w + x0 + r % TW);
  cnt[g] = r == i ? N[i] : 0;
}

// One thread per 4-neighbour pair across a tile border: nvx h pairs (x, y) - (x + 1, y) at the vertical borders, then
// nhy w pairs (x, y) - (x, y + 1) at the horizontal ones.  Grid y = map.
__global__ void __launch_bounds__(256) k_speckle_merge(MapList src, int* lab, int w, int h, int r16, int nvx, int nhy) {
  const int t = blockIdx.x * 256 + threadIdx.x, nv = nvx * h;
  int x, y, x2, y2;
  if (t < nv) {
    y = t / nvx; x = (t % nvx + 1) * TW - 1; x2 = x + 1; y2 = y;
  } else {
    const int u = t - nv;
    if (u >= nhy * w) return;
    x = u % w; y = (u / w + 1) * TH - 1; x2 = x; y2 = y + 1;
  }
  const int16_t* __restrict__ m = src.p[blockIdx.y];
  const int a = (size_t)y * w + x, b = (size_t)y2 * w + x2;
  if (!joined(m[a], m[b], r16)) return;
  const int base = blockIdx.y * w * h;
  unite(lab, base + a, base + b);
}

// One thread per pixel (grid y = map); only tile roots (cnt > 0) act: they add their tile count into their component's
// root and point straight at it, so every pixel then reaches its root in two steps.
__global__ void __launch_bounds__(256) k_speckle_count(int* lab, int* cnt, int plane) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= plane) return;
  const int g = blockIdx.y * plane + i;
  const int c = cnt[g];
  if (c == 0) return;
  const int r = find_root(lab, g);
  if (r != g) { atomicAdd(&cnt[r], c); lab[g] = r; }
}

// One thread per pixel (grid y = map): dst = src, or -1 where speckle removal (size > 0) finds a component of at most
// `size` pixels.  src and dst may be the same maps.
__global__ void __launch_bounds__(256) k_speckle_apply(MapList src, MapList dst, const int* lab, const int* cnt, int plane, int size) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= plane) return;
  const int k = blockIdx.y;
  int v = src.p[k][i];
  if (v >= 0 && size > 0) {
    const int g = k * plane + i;
    if (cnt[lab[lab[g]]] <= size) v = -1;
  }
  dst.p[k][i] = (int16_t)v;
}

}  // namespace

size_t visocu_disp_filter_scratch(int n_maps, size_t plane) { return align_up((size_t)n_maps * plane * 10, 256); }

int visocu_disp_filter_group(visocu_ctx* ctx, int nb, int16_t* const* maps, int w, int h, int median, int speckle_size,
                             int speckle_range, void* scratch) {
  if (!median && !speckle_size) return VISOCU_OK;
  cudaStream_t st = ctx->stream;
  const int plane = w * h;
  int* lab = (int*)scratch;
  int* cnt = lab + (size_t)nb * plane;
  int16_t* buf = (int16_t*)(cnt + (size_t)nb * plane);
  MapList dst, src;
  for (int k = 0; k < nb; k++) { dst.p[k] = maps[k]; src.p[k] = median ? buf + (size_t)k * plane : maps[k]; }
  if (median) {
    k_disp_median3<<<dim3((w + 31) / 32, (h + 7) / 8, nb), dim3(32, 8), 0, st>>>(dst, buf, w, h);
    CU_LAUNCH_CHECK(ctx);
  }
  const int r16 = 16 * speckle_range;
  if (speckle_size) {
    const int nvx = (w + TW - 1) / TW - 1, nhy = (h + TH - 1) / TH - 1;
    k_speckle_local<<<dim3((w + TW - 1) / TW, (h + TH - 1) / TH, nb), dim3(TW, TH), 0, st>>>(src, lab, cnt, w, h, r16);
    CU_LAUNCH_CHECK(ctx);
    const int pairs = nvx * h + nhy * w;
    k_speckle_merge<<<dim3((pairs + 255) / 256 > 0 ? (pairs + 255) / 256 : 1, nb), 256, 0, st>>>(src, lab, w, h, r16, nvx, nhy);
    CU_LAUNCH_CHECK(ctx);
    k_speckle_count<<<dim3((plane + 255) / 256, nb), 256, 0, st>>>(lab, cnt, plane);
    CU_LAUNCH_CHECK(ctx);
  }
  k_speckle_apply<<<dim3((plane + 255) / 256, nb), 256, 0, st>>>(src, dst, lab, cnt, plane, speckle_size);
  CU_LAUNCH_CHECK(ctx);
  return VISOCU_OK;
}

extern "C" int visocu_disparity_filter(visocu_ctx* ctx, int32_t n_maps, int16_t* const* maps, int32_t w, int32_t h,
                                       int32_t on_device, int32_t median, int32_t speckle_size, int32_t speckle_range) {
  if (!ctx) return VISOCU_EINVAL;
  if (n_maps < 0) return visocu_set_error(ctx, VISOCU_EINVAL, "n_maps %d < 0", n_maps);
  if (w < 1 || h < 1 || (int64_t)w * h > VISOCU_DISP_FILTER_MAX_PIXELS)
    return visocu_set_error(ctx, VISOCU_EINVAL, "map size %d x %d outside [1, %d] pixels", w, h, VISOCU_DISP_FILTER_MAX_PIXELS);
  if (on_device != 0 && on_device != 1) return visocu_set_error(ctx, VISOCU_EINVAL, "on_device must be 0 or 1");
  if ((median != 0 && median != 1) || speckle_size < 0 || speckle_range < 0 || speckle_range > 256)
    return visocu_set_error(ctx, VISOCU_EINVAL, "filter parameters out of range (median %d, speckle_size %d, speckle_range %d)",
                            median, speckle_size, speckle_range);
  if (n_maps > 0 && !maps) return visocu_set_error(ctx, VISOCU_EINVAL, "null map list");
  for (int k = 0; k < n_maps; k++)
    if (!maps[k]) return visocu_set_error(ctx, VISOCU_EINVAL, "map %d: null", k);
  if (n_maps == 0 || (!median && !speckle_size)) return VISOCU_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t plane = (size_t)w * h;
  const int nmax = n_maps < VISO_MAX_BATCH ? n_maps : VISO_MAX_BATCH;
  const size_t f_bytes = visocu_disp_filter_scratch(nmax, plane), m_bytes = align_up(plane * 2, 256);
  int rc = visocu_ensure_scratch(ctx, f_bytes + (on_device ? 0 : nmax * m_bytes));
  if (rc) return rc;
  uint8_t* stage = (uint8_t*)ctx->scratch + f_bytes;
  for (int start = 0; start < n_maps; start += VISO_MAX_BATCH) {
    const int nb = n_maps - start < VISO_MAX_BATCH ? n_maps - start : VISO_MAX_BATCH;
    int16_t* dm[VISO_MAX_BATCH];
    for (int k = 0; k < nb; k++) {
      dm[k] = on_device ? maps[start + k] : (int16_t*)(stage + k * m_bytes);
      if (!on_device) CU_COPY(ctx, dm[k], maps[start + k], plane * 2, cudaMemcpyHostToDevice);
    }
    rc = visocu_disp_filter_group(ctx, nb, dm, w, h, median, speckle_size, speckle_range, ctx->scratch);
    if (rc) return rc;
    if (!on_device)
      for (int k = 0; k < nb; k++) CU_COPY(ctx, maps[start + k], dm[k], plane * 2, cudaMemcpyDeviceToHost);
  }
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}
