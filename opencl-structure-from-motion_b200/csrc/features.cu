// Feature front end: fused 5x5 filters + both non-maximum-suppression passes, ordered compaction with the
// 32-byte descriptor gather, and the (class, v_bin, u_bin) bin index.
//
// What it reproduces (reference paths relative to /root/reference/viso):
//   filter::sobel5x5 / blob5x5 / checkerboard5x5 .......... filter.cpp:316-365 (semantics restated in SURVEY.md 9.3)
//   Matcher::createHalfResolutionImage ..................... matcher.cpp:630-647
//   Matcher::nonMaximumSuppression, sparse + dense pass .... matcher.cpp:330-431, 684-694
//   Matcher::computeDescriptors + record packing ........... matcher.cpp:433-477, 707-731
//   Matcher::createIndexVector ............................. matcher.cpp:870-890
// None of it is a translation of the reference's SSE row/column passes or its integral image: the blob and
// checkerboard responses never leave the SM (they live in shared memory only), the NMS neighbourhood test is
// reduced to "window extreme == cell extreme", and the output order (cell-column-major, then class) is
// rebuilt with a deterministic scan instead of push_back.
#include "visocu_internal.cuh"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

namespace {

constexpr int CELLS_PER_BLOCK = 512;
constexpr int MAX_FILTER_THREADS = 512;

// ----------------------------------------------------------------------------------------------------------
// half-resolution image: 2x2 box mean, truncating (matcher.cpp:636-647).  One thread = 4 output pixels.
__global__ void k_half_image(Geometry g, const FrameDev* frames, SlotList sl) {
  const FrameDev F = frames[sl.s[blockIdx.z]];
  int wx = blockIdx.x * blockDim.x + threadIdx.x;        // output word index along the row
  int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (y >= g.hm || wx * 4 >= g.bplm) return;
  const uint8_t* r0 = F.img + (size_t)(2 * y) * g.bpl + 8 * wx;
  const uint8_t* r1 = r0 + g.bpl;
  uint32_t out = 0;
  if (8 * wx + 7 < g.bpl) {
    uint2 a = *(const uint2*)r0, b = *(const uint2*)r1;
    uint32_t aw[2] = {a.x, a.y}, bw[2] = {b.x, b.y};
#pragma unroll
    for (int k = 0; k < 4; k++) {
      uint32_t wa = aw[k >> 1] >> (16 * (k & 1)), wb = bw[k >> 1] >> (16 * (k & 1));
      uint32_t s = (wa & 255) + ((wa >> 8) & 255) + (wb & 255) + ((wb >> 8) & 255);
      uint32_t px = (4 * wx + k < g.wm) ? (s >> 2) : 0;    // pad columns stay zero
      out |= px << (8 * k);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 4; k++) {
      int x = 4 * wx + k;
      uint32_t px = 0;
      if (x < g.wm) px = ((uint32_t)r0[2 * k] + r0[2 * k + 1] + r1[2 * k] + r1[2 * k + 1]) >> 2;
      out |= px << (8 * k);
    }
  }
  *(uint32_t*)(F.half + (size_t)y * g.bplm + 4 * wx) = out;
}

// ----------------------------------------------------------------------------------------------------------
// Packed filter arithmetic.  A thread owns one 32-bit word (4 pixels b0..b3) of an image row and walks down the rows
// with a 5-row register window.  Everything is computed on two 16-bit lanes per register, (b0,b2) and (b1,b3) of the
// word; every intermediate is kept non-negative by a bias, so plain 32-bit adds, subtracts and multiplies by small
// constants never carry between the lanes (ptxas spreads them over the FMA pipe as IMAD and the ALU pipe as IADD3).
constexpr int BIAS_F1 = 6375;    // 25 * 255: f1 + BIAS_F1 >= 0
constexpr int BIAS_F2 = 2040;    //  8 * 255
#define K2(v) ((uint32_t)(v) | ((uint32_t)(v) << 16))   /* the same constant in both 16-bit lanes */

// the six tap vectors of word C with neighbours L and R: t[k] = pixels (x-2+k, x+k) for x = b0, i.e.
// (l2,b0) (l3,b1) (b0,b2) (b1,b3) (b2,r0) (b3,r1); lane pair A = pixels (b0,b2) uses t[0..4], B = (b1,b3) uses t[1..5]
__device__ __forceinline__ void taps6(uint32_t L, uint32_t C, uint32_t R, uint32_t t[6]) {
  const uint32_t s2a = __funnelshift_r(L, C, 16);          // bytes l2 l3 b0 b1
  const uint32_t s2b = __funnelshift_r(C, R, 16);          // bytes b2 b3 r0 r1
  t[0] = s2a & 0x00FF00FFu;
  t[1] = __byte_perm(s2a, 0, 0x4341);
  t[2] = C & 0x00FF00FFu;
  t[3] = __byte_perm(C, 0, 0x4341);
  t[4] = s2b & 0x00FF00FFu;
  t[5] = __byte_perm(s2b, 0, 0x4341);
}

__device__ __forceinline__ uint32_t lds32(uint32_t addr) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr)); return v; }
__device__ __forceinline__ uint2 lds64(uint32_t addr) { uint2 v; asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr)); return v; }
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t x) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(addr), "r"(x) : "memory"); }
__device__ __forceinline__ void sts64(uint32_t addr, uint32_t x, uint32_t y) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(addr), "r"(x), "r"(y) : "memory"); }

// Sobel walker: du = ((1,4,6,4,1)^T x (1,2,0,-2,-1)) >> 7 + 128, dv = ((1,2,0,-2,-1)^T x (1,4,6,4,1)) >> 7 + 128
// (filter.cpp:316-324).  The sums are formed at twice their scale with a bias of 32768, so the result byte is simply the
// high byte of each 16-bit lane and one PRMT assembles the four pixels of the output word.
// col: shared-memory address of word L of the first row needed (two rows above the first output row); IWB: bytes per
// row of the image tile.  Writes rows [gy0, gy0 + nrow) of word column gx to the planes du / dv (stride bpl).
__device__ __forceinline__ void walk_sobel(uint32_t col, int IWB, int nrow, int gy0, int gx, int bpl, int himg,
                                           uint8_t* __restrict__ du, uint8_t* __restrict__ dv) {
  uint32_t hd[5][2], ha[5][2];
#define SOB_HROW(S) {                                                                           \
    uint32_t t[6]; taps6(lds32(col), lds32(col + 4), lds32(col + 8), t); col += IWB;              \
    _Pragma("unroll") for (int k = 0; k < 2; k++) {                                               \
      hd[S][k] = (t[k] + 2 * t[k + 1] + K2(765)) - (t[k + 4] + 2 * t[k + 3]);      /* (1,2,0,-2,-1) + 765 */ \
      ha[S][k] = (t[k] + t[k + 4]) + 4 * (t[k + 1] + t[k + 3]) + 6 * t[k + 2];     /* (1,4,6,4,1) */          \
    } }
  SOB_HROW(0) SOB_HROW(1) SOB_HROW(2) SOB_HROW(3)
  uint8_t* pu = du + (size_t)gy0 * bpl + gx;
  uint8_t* pv = dv + (size_t)gy0 * bpl + gx;
  uint8_t* const pu0 = pu; uint8_t* const pv0 = pv;
  for (int r5 = 0; r5 < nrow; r5 += 5) {
#define SOB_STEP(PH)                                                                                              \
    if (r5 + PH < nrow) {                                                                                         \
      constexpr int s0 = PH % 5, s1 = (PH + 1) % 5, s2 = (PH + 2) % 5, s3 = (PH + 3) % 5, s4 = (PH + 4) % 5;      \
      SOB_HROW(s4)                                                                                                \
      uint32_t u2[2], v2[2];                                                                                      \
      _Pragma("unroll") for (int k = 0; k < 2; k++) {                                                             \
        u2[k] = 2 * (hd[s0][k] + hd[s4][k]) + 8 * (hd[s1][k] + hd[s3][k]) + 12 * hd[s2][k] + K2(8288);            \
        v2[k] = 2 * ((ha[s0][k] + K2(4080)) - ha[s4][k]) + 4 * ((ha[s1][k] + K2(4080)) - ha[s3][k]) + K2(8288);   \
      }                                                                                                           \
      *(uint32_t*)pu = __byte_perm(u2[0], u2[1], 0x7351); pu += bpl;                                              \
      *(uint32_t*)pv = __byte_perm(v2[0], v2[1], 0x7351); pv += bpl;                                              \
    }
    SOB_STEP(0) SOB_STEP(1) SOB_STEP(2) SOB_STEP(3) SOB_STEP(4)
#undef SOB_STEP
  }
#undef SOB_HROW
  // image border (filter.cpp:185-186 and the pad columns): the two outermost rows and columns read 128.  The same
  // thread stored the words above, so these stores land after them.
  if (gy0 < 2 || gy0 + nrow > himg - 2 || gx == 0 || gx == bpl - 4) {
    for (int r = 0; r < nrow; r++) {
      const int gy = gy0 + r;
      if (gy < 2 || gy > himg - 3) { *(uint32_t*)(pu0 + r * bpl) = 0x80808080u; *(uint32_t*)(pv0 + r * bpl) = 0x80808080u; }
      else if (gx == 0) { *(uint16_t*)(pu0 + r * bpl) = 0x8080; *(uint16_t*)(pv0 + r * bpl) = 0x8080; }
      if (gx == bpl - 4 && gy >= 2 && gy <= himg - 3) { *(uint16_t*)(pu0 + r * bpl + 2) = 0x8080; *(uint16_t*)(pv0 + r * bpl + 2) = 0x8080; }
    }
  }
}

// Blob / checkerboard walker: f1 = -box5 + 2 box3 + 7 centre (filter.cpp:343-365), f2 = (1,1,0,-1,-1)^T x (1,1,0,-1,-1)
// (filter.cpp:331-336), stored biased (BIAS_F1 / BIAS_F2) as int16 rows of FS samples in shared memory.
// col as above; out1 / out2: shared-memory addresses of the first output row of this word (4 samples = 8 bytes, 8-byte
// aligned); FSB: bytes per row of the response planes.
__device__ __forceinline__ void walk_blob_checker(uint32_t col, int IWB, int nrow, uint32_t out1, uint32_t out2, int FSB) {
  uint32_t h1[5][2], h3[5][2], hc[5][2], pc[5][2];
#define BC_HROW(S) {                                                                            \
    uint32_t t[6]; taps6(lds32(col), lds32(col + 4), lds32(col + 8), t); col += IWB;              \
    _Pragma("unroll") for (int k = 0; k < 2; k++) {                                               \
      h3[S][k] = t[k + 1] + t[k + 2] + t[k + 3];                                                  \
      h1[S][k] = h3[S][k] + t[k] + t[k + 4];                                                      \
      hc[S][k] = (t[k] + t[k + 1] + K2(510)) - (t[k + 3] + t[k + 4]);             /* (1,1,0,-1,-1) + 510 */   \
      pc[S][k] = t[k + 2];                                                                        \
    } }
  BC_HROW(0) BC_HROW(1) BC_HROW(2) BC_HROW(3)
  for (int r5 = 0; r5 < nrow; r5 += 5) {
#define BC_STEP(PH)                                                                                               \
    if (r5 + PH < nrow) {                                                                                         \
      constexpr int s0 = PH % 5, s1 = (PH + 1) % 5, s2 = (PH + 2) % 5, s3 = (PH + 3) % 5, s4 = (PH + 4) % 5;      \
      BC_HROW(s4)                                                                                                 \
      uint32_t f1[2], f2[2];                                                                                      \
      _Pragma("unroll") for (int k = 0; k < 2; k++) {                                                             \
        const uint32_t b3 = h3[s1][k] + h3[s2][k] + h3[s3][k];                                                    \
        const uint32_t b5 = h1[s0][k] + h1[s1][k] + h1[s2][k] + h1[s3][k] + h1[s4][k];                            \
        f1[k] = (7 * pc[s2][k] + 2 * b3 + K2(BIAS_F1)) - b5;                                                      \
        f2[k] = (hc[s0][k] + hc[s1][k] + K2(BIAS_F2)) - (hc[s3][k] + hc[s4][k]);                                  \
      }                                                                                                           \
      sts64(out1, __byte_perm(f1[0], f1[1], 0x5410), __byte_perm(f1[0], f1[1], 0x7632)); out1 += FSB;             \
      sts64(out2, __byte_perm(f2[0], f2[1], 0x5410), __byte_perm(f2[0], f2[1], 0x7632)); out2 += FSB;             \
    }
    BC_STEP(0) BC_STEP(1) BC_STEP(2) BC_STEP(3) BC_STEP(4)
#undef BC_STEP
  }
#undef BC_HROW
}

// full-resolution Sobel planes only (the *_full planes of matcher.cpp:676 used by the refinement), half-resolution mode:
// the same walker on words loaded from global memory through a small shared-memory tile.
constexpr int SF_TW = 256, SF_TH = 32;                      // core pixels of one CTA
__global__ void __launch_bounds__(256) k_sobel_full(Geometry g, const FrameDev* frames, SlotList sl) {
  __shared__ uint32_t simg[(SF_TH + 4) * (SF_TW / 4 + 2)];
  const FrameDev F = frames[sl.s[blockIdx.z]];
  const int x0 = blockIdx.x * SF_TW, y0 = blockIdx.y * SF_TH;
  constexpr int IW = SF_TW / 4 + 2;
  for (int idx = threadIdx.x; idx < (SF_TH + 4) * IW; idx += 256) {
    const int ly = idx / IW, lw = idx - ly * IW;
    const int gx = x0 - 4 + 4 * lw, gy = y0 - 2 + ly;
    uint32_t v = 0;
    if (gy >= 0 && gy < g.h && gx >= 0 && gx < g.bpl) v = __ldg((const uint32_t*)(F.img + (size_t)gy * g.bpl + gx));
    simg[idx] = v;
  }
  __syncthreads();
  // 64 word columns x 4 row segments of 8 rows
  const int wcol = threadIdx.x & 63, seg = threadIdx.x >> 6;
  const int gx = x0 + 4 * wcol, gy0 = y0 + 8 * seg;
  if (gx >= g.bpl || gy0 >= g.h) return;
  walk_sobel((uint32_t)__cvta_generic_to_shared(simg + (8 * seg) * IW + wcol), 4 * IW, min(8, g.h - gy0), gy0, gx, g.bpl, g.h, F.du_full, F.dv_full);
}

// ----------------------------------------------------------------------------------------------------------
// Tiling of the fused kernel.  Tiles are aligned to the cell grid of the NMS pass with the larger neighbourhood (the
// sparse pass when multi_stage): a tile owns kx x ky of its cells, which lie completely inside the tile, so the response
// planes need a halo of only n samples to the left / top and max(n, 2 n_other) to the right / bottom.  Cells of the
// other pass belong to the tile that contains their origin.  du / dv are written for the 4-aligned pixel range of the
// tile; first and last tiles extend to the image borders.  Everything that depends on the tile index along one axis is
// computed once on the host (AxisTile tables in device memory): the kernel does no division to find its ranges.
struct TileCfg {
  int nA, stepA, orgA;     // the aligning pass: n, n + 1, n + margin
  int extR;                // response halo to the right / bottom of the tile's cell range
  int kx, ky, ntx, nty, TWn, THn;
  int NWf, FS, FH;         // response planes in shared memory: words (4 samples) per row, samples per row, rows
  int IS, IH;              // image tile: bytes per row (multiple of 16), rows
  int max_cells;           // owned cells of one tile, both passes
  int threads;
  // fused half-resolution mode: the full-resolution tile is staged in P parts of HP half-resolution rows (SR = 2 HP + 4
  // full-resolution rows) by nbox TMA boxes of BW bytes per row (two boxes overlap so that no word column straddles them)
  int fused, HP, P, SR, nbox, BW, segF;
  unsigned img_bytes, f_bytes, smem;
  const struct AxisTile* xt;   // ntx entries
  const struct AxisTile* yt;   // nty entries
};

struct AxisTile {          // one axis of one tile
  int own_lo, own_hi;      // cells with origin in [own_lo, own_hi) belong to the tile
  int f_lo, f_hi;          // response samples computed into shared memory: [f_lo, f_hi), f_lo 4-aligned along x
  int v_hi, fill_hi;       // samples in [v_hi, fill_hi) lie beyond the last valid one (len - margin - 1): set to the neutral value
  int d_lo, d_hi;          // du / dv samples written
  int i_lo, i_hi;          // image samples needed (along x: i_lo 16-byte aligned)
  int klo[2], nk[2];       // owned cells of the two passes along this axis
  float inv_nk[2];         // 1 / nk (x axis: cell index -> column, row)
  int nwa, nwb;            // x axis: word columns of the Sobel / response range
  float inv_nwa, inv_nwb;
  int df_lo, df_hi;        // fused half-resolution mode: full-resolution du / dv samples written along this axis
  int nwF; float inv_nwF;  // x axis: their word columns
  int segA, segB, nsA, nsB;   // y axis: rows per Sobel / response walker and number of row segments
};

__host__ __device__ inline void tile_range(const TileCfg& t, int idx, int ntiles, int len, int len_pad, bool xaxis, AxisTile& r) {
  const int TN = xaxis ? t.TWn : t.THn;
  const int n0 = t.orgA + TN * idx;
  const bool first = idx == 0, last = idx == ntiles - 1;
  r.own_lo = first ? 0 : n0;
  r.own_hi = last ? 0x3FFFFFFF : n0 + TN;
  int f_lo = first ? VISO_MARGIN : n0 - t.nA;
  int f_hi = len - VISO_MARGIN;
  if (!last && n0 + TN + t.extR < f_hi) f_hi = n0 + TN + t.extR;
  int d_lo = first ? 0 : n0, d_hi = last ? len_pad : n0 + TN;
  if (xaxis) { f_lo &= ~3; d_lo &= ~3; if (!last) d_hi &= ~3; }
  if (d_lo > len_pad) d_lo = len_pad;
  if (d_hi > len_pad) d_hi = len_pad;
  if (f_hi < f_lo) f_hi = f_lo;
  if (xaxis) f_hi = f_lo + ((f_hi - f_lo + 3) & ~3);
  r.f_lo = f_lo; r.f_hi = f_hi; r.d_lo = d_lo; r.d_hi = d_hi;
  // Windows are clamped at len - 1 - margin (matcher.cpp:383-384).  Instead of clamping, the samples behind that line are
  // given the response 0, which is never strictly better than a candidate (|candidate| >= tau >= 1): the scans need no
  // border case.  They read up to n + 1 samples past the last valid one.
  r.v_hi = f_hi; r.fill_hi = f_hi;
  if (f_hi >= len - VISO_MARGIN && f_hi > f_lo) { r.v_hi = len - VISO_MARGIN; r.fill_hi = len - VISO_MARGIN + t.nA + 1; if (r.fill_hi < f_hi) r.fill_hi = f_hi; }
  if (xaxis) r.fill_hi = f_lo + ((r.fill_hi - f_lo + 3) & ~3);
  int lo = d_lo < f_lo ? d_lo : f_lo, hi = d_hi > f_hi ? d_hi : f_hi;
  if (d_hi <= d_lo) { lo = f_lo; hi = f_hi; }
  if (f_hi <= f_lo) { lo = d_lo; hi = d_hi; }
  if (xaxis) { r.i_lo = (lo - 4) & ~15; r.i_hi = hi + 4; }
  else { r.i_lo = lo - 2; r.i_hi = hi + 2; }
}

// owned cell range of pass p along one axis: cells k with origin org + k * step in [own_lo, own_hi), k < ncells
inline void owned_cells(const AxisTile& r, int n, int ncells, int& klo, int& nk) {
  const int step = n + 1, org = n + VISO_MARGIN;
  int a = r.own_lo - org; klo = a > 0 ? (a + step - 1) / step : 0;
  int khi = ncells;
  if (r.own_hi < 0x3FFFFFFF) { int b = r.own_hi - org; khi = b > 0 ? (b + step - 1) / step : 0; if (khi > ncells) khi = ncells; }
  nk = khi > klo ? khi - klo : 0;
}

// atomicAdd on a shared-memory word (the generic form costs a dozen instructions when the compiler cannot see the
// address space)
__device__ __forceinline__ int atom_add_shared(int* p, int v) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  int old;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
  return old;
}

// q = a / d for 0 <= a < 2^20 with inv = 1.0f / d: (a + 0.5) / d is at least 0.5 / d away from an integer, far more than
// the rounding error of the float product
__device__ __forceinline__ int fast_div(int a, float inv) { return __float2int_rz(((float)a + 0.5f) * inv); }

__device__ __forceinline__ bool mbar_wait_or_trap(uint32_t bar, uint32_t phase) {
  const long long t0 = clock64();
  for (;;) {
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(phase) : "memory");
    if (done) return true;
    if (clock64() - t0 > 2000000000LL) __trap();           // about one second: never hang the GPU on a TMA mistake
  }
}

// ---- phase 3a: cell extremes as keys (value << 16 | position), position = (dx << 4 | dy) for the minimum and its
// complement for the maximum, so that "first extreme in column-major order" (matcher.cpp:356-379) falls out of min / max.
// A row of the cell is read as 32-bit words (two samples each); the key of the low sample is w * 65536 + pos (an IMAD on
// the FMA pipe), the key of the high sample (w & 0xFFFF0000) | pos (a LOP3 on the ALU pipe).
struct Keys4 { uint32_t k[4]; };      // 0 = f1 min, 1 = f1 max, 2 = f2 min, 3 = f2 max

template <int N1, bool ODD, int ROWS>
__device__ __forceinline__ void cell_keys_rows(const uint32_t* r1, const uint32_t* r2, int FSW, int nrows, Keys4& K) {
  // r1 / r2: word holding sample i0 (ODD: in its high half) of the first row, planes f1 / f2; positions are relative
  // to this row (dy = 0 .. nrows - 1).  Words are fetched in pairs (64-bit loads) when the first word is 8-byte aligned.
  constexpr int NW = (N1 + (ODD ? 1 : 0) + 1) / 2;
  constexpr int NWP = (NW + 1) & ~1;
  const bool aligned = (((uintptr_t)r1) & 7) == 0;
#pragma unroll
  for (int rr = 0; rr < ROWS; rr++) {
    if (rr < nrows) {
      uint32_t a[NWP], b[NWP];
      if (aligned) {
#pragma unroll
        for (int j = 0; j < NWP; j += 2) {
          const uint2 va = *(const uint2*)(r1 + rr * FSW + j), vb = *(const uint2*)(r2 + rr * FSW + j);
          a[j] = va.x; a[j + 1] = va.y; b[j] = vb.x; b[j + 1] = vb.y;
        }
      } else {
#pragma unroll
        for (int j = 0; j < NW; j++) { a[j] = r1[rr * FSW + j]; b[j] = r2[rr * FSW + j]; }
      }
#pragma unroll
      for (int j = 0; j < NW; j++) {
        const int dx_lo = 2 * j - (ODD ? 1 : 0), dx_hi = dx_lo + 1;
        if (dx_lo >= 0 && dx_lo < N1) {
          const uint32_t p = (uint32_t)((dx_lo << 4) | rr);
          K.k[0] = min(K.k[0], a[j] * 65536u + p); K.k[1] = max(K.k[1], a[j] * 65536u + (p ^ 0xFFu));
          K.k[2] = min(K.k[2], b[j] * 65536u + p); K.k[3] = max(K.k[3], b[j] * 65536u + (p ^ 0xFFu));
        }
        if (dx_hi >= 0 && dx_hi < N1) {
          const uint32_t p = (uint32_t)((dx_hi << 4) | rr);
          K.k[0] = min(K.k[0], (a[j] & 0xFFFF0000u) | p); K.k[1] = max(K.k[1], (a[j] & 0xFFFF0000u) | (p ^ 0xFFu));
          K.k[2] = min(K.k[2], (b[j] & 0xFFFF0000u) | p); K.k[3] = max(K.k[3], (b[j] & 0xFFFF0000u) | (p ^ 0xFFu));
        }
      }
    }
  }
}

// any cell size: one 16-bit load per sample
__device__ __forceinline__ void cell_keys_generic(const int16_t* q1, const int16_t* q2, int FS, int n1, int nrows, Keys4& K) {
  for (int dj = 0; dj < nrows; dj++)
    for (int di = 0; di < n1; di++) {
      const uint32_t p = (uint32_t)((di << 4) | dj);
      const uint32_t v1 = (uint32_t)(uint16_t)q1[dj * FS + di] << 16, v2 = (uint32_t)(uint16_t)q2[dj * FS + di] << 16;
      K.k[0] = min(K.k[0], v1 | p); K.k[1] = max(K.k[1], v1 | (p ^ 0xFFu));
      K.k[2] = min(K.k[2], v2 | p); K.k[3] = max(K.k[3], v2 | (p ^ 0xFFu));
    }
}

// ---- window test (matcher.cpp:383-427): a candidate survives iff nothing in its clamped (2n+1)^2 window is strictly
// better; positions inside the cell can never be strictly better than the cell extreme, so the reference's cell
// exclusion is implied.  A window row is read as n+1 32-bit words (two samples each); of the 2n+2 samples exactly one
// lies outside the window (the low half of the first word or the high half of the last) and is neutralised by a mask.
// Rows are combined with packed 16-bit min3 / max3 (VIMNMX3.U16x2) before the masks are applied.
template <int N1, bool IS_MIN>
__device__ __forceinline__ bool rows_better(const uint32_t* r0, const uint32_t* r1, const uint32_t* r2, int nw, uint32_t m_first, uint32_t m_last, uint32_t target2) {
  uint32_t acc;
  if (N1 > 0) {
    uint32_t x[N1 > 0 ? N1 : 1];
#pragma unroll
    for (int j = 0; j < N1; j++) x[j] = IS_MIN ? __vimin3_u16x2(r0[j], r1[j], r2[j]) : __vimax3_u16x2(r0[j], r1[j], r2[j]);
    if (IS_MIN) { x[0] |= m_first; x[N1 - 1] |= m_last; } else { x[0] &= ~m_first; x[N1 - 1] &= ~m_last; }
    acc = x[0];
#pragma unroll
    for (int j = 1; j + 1 < N1; j += 2) acc = IS_MIN ? __vimin3_u16x2(acc, x[j], x[j + 1]) : __vimax3_u16x2(acc, x[j], x[j + 1]);
    if ((N1 & 1) == 0) acc = IS_MIN ? __vminu2(acc, x[N1 - 1]) : __vmaxu2(acc, x[N1 - 1]);
  } else {
    acc = IS_MIN ? 0xFFFFFFFFu : 0u;
    for (int j = 0; j < nw; j++) {
      uint32_t x = IS_MIN ? __vimin3_u16x2(r0[j], r1[j], r2[j]) : __vimax3_u16x2(r0[j], r1[j], r2[j]);
      if (j == 0) x = IS_MIN ? (x | m_first) : (x & ~m_first);
      if (j == nw - 1) x = IS_MIN ? (x | m_last) : (x & ~m_last);
      acc = IS_MIN ? __vminu2(acc, x) : __vmaxu2(acc, x);
    }
  }
  return (IS_MIN ? __vminu2(acc, target2) : __vmaxu2(acc, target2)) != target2;
}

// windows clamped at the right or bottom image border (last cell columns / rows only): plain scan
__device__ __noinline__ bool slow_keep(const int16_t* sf, int FS, int ex, int ey, int n, int xhi, int yhi, uint32_t val, bool is_min) {
  const int xe = min(ex + n, xhi), ye = min(ey + n, yhi);
  for (int j2 = ey - n; j2 <= ye; j2++)
    for (int i2 = ex - n; i2 <= xe; i2++) {
      const uint32_t v = (uint16_t)sf[j2 * FS + i2];
      if (is_min ? v < val : v > val) return false;
    }
  return true;
}

struct NmsArgs {
  const int16_t* sf1; const int16_t* sf2;   // response planes (sf2 = sf1 + FH * FS)
  int FS;
  uint32_t* codes;         // one word per owned cell of this pass
  uint32_t* queue[2];      // candidates that passed the quick test: [0] minima, [1] maxima
  int* qn;                 // their counters (two ints)
  int n, ncell, nk; float inv_nk;
  int cx0, cy0;            // plane coordinates of the first owned cell's origin
  int xhi, yhi, tau;
};

// Cell extremes, tau test and quick window test (the three rows around the extreme, where most candidates die) of all
// owned cells of one pass.  G lanes per cell: one for small cells; two for cells of six or more rows, the upper rows on
// the even lane and the lower rows on the odd one, f1 classes tested by the even lane and f2 classes by the odd one.
// Survivors of the quick test are queued (warp-aggregated) for phase 3b.
template <int N1>
__device__ __forceinline__ void nms_cells(const NmsArgs& A, int item, unsigned lane) {
  const int n = A.n, n1 = n + 1, FS = A.FS, FSW = FS >> 1;
  const bool two = n1 >= 6;
  const int half_rows = (n1 + 1) >> 1;
  constexpr int ROWS = N1 >= 6 ? (N1 + 1) / 2 : N1;
  const unsigned lt = (1u << lane) - 1u;                             // whole warps take part in the shuffles and ballots
  const uint32_t* sfw = (const uint32_t*)A.sf1;
  {
    const int cell = two ? item >> 1 : item, tt = two ? item & 1 : 0;
    const bool live = cell < A.ncell;
    const int ll = live ? fast_div(cell, A.inv_nk) : 0, kk = live ? cell - ll * A.nk : 0;
    const int i0 = A.cx0 + kk * n1, j0 = A.cy0 + ll * n1;
    Keys4 K = {{0xFFFFFFFFu, 0u, 0xFFFFFFFFu, 0u}};
    const int row_lo = two ? tt * half_rows : 0, nrows = two ? (tt ? n1 - half_rows : half_rows) : n1;
    if (live) {
      const uint32_t* r1 = (const uint32_t*)(A.sf1 + (j0 + row_lo) * FS) + (i0 >> 1);
      const uint32_t* r2 = (const uint32_t*)(A.sf2 + (j0 + row_lo) * FS) + (i0 >> 1);
      if (N1 > 0) {
        constexpr int NC = N1 > 0 ? N1 : 1;
        if (i0 & 1) cell_keys_rows<NC, true, ROWS>(r1, r2, FSW, nrows, K);
        else cell_keys_rows<NC, false, ROWS>(r1, r2, FSW, nrows, K);
      } else {
        cell_keys_generic(A.sf1 + (j0 + row_lo) * FS + i0, A.sf2 + (j0 + row_lo) * FS + i0, FS, n1, nrows, K);
      }
      // positions are relative to row_lo: shift them to the cell (dy is the low nibble; complemented for maxima)
      K.k[0] += row_lo; K.k[2] += row_lo; K.k[1] -= row_lo; K.k[3] -= row_lo;
    }
    if (two) {
      K.k[0] = min(K.k[0], __shfl_xor_sync(0xFFFFFFFFu, K.k[0], 1)); K.k[1] = max(K.k[1], __shfl_xor_sync(0xFFFFFFFFu, K.k[1], 1));
      K.k[2] = min(K.k[2], __shfl_xor_sync(0xFFFFFFFFu, K.k[2], 1)); K.k[3] = max(K.k[3], __shfl_xor_sync(0xFFFFFFFFu, K.k[3], 1));
    }
    // a single lane tests the four classes one after the other; a lane pair tests two classes each (the even lane
    // those of f1, the odd lane those of f2), minima in the first round and maxima in the second
    uint32_t code = 0xFFFFFFFFu;
#pragma unroll
    for (int u = 0; u < 4; u++) {
      if (!(two && u >= 2)) {
        const bool is_min = (u & 1) == 0;
        const int plane = two ? tt : u >> 1;
        const int c = two ? 2 * tt + u : u;
        const uint32_t key = two ? (tt ? K.k[2 + (u & 1)] : K.k[u & 1]) : K.k[u];
        const uint32_t val = key >> 16, pos = is_min ? (key & 0xFFu) : ((key & 0xFFu) ^ 0xFFu);
        const int bias = plane ? BIAS_F2 : BIAS_F1;
        bool cand = live && (is_min ? (int)val <= bias - A.tau : (int)val >= bias + A.tau);
        bool push = false;
        uint32_t ent = 0;
        if (cand) {
          const int ex = i0 + (int)(pos >> 4), ey = j0 + (int)(pos & 15), xs = ex - n;
          const int16_t* sf = plane ? A.sf2 : A.sf1;
          if (A.tau < 1 && (ex + n > A.xhi || ey + n > A.yhi)) {
            cand = slow_keep(sf, FS, ex, ey, n, A.xhi, A.yhi, val, is_min);    // the neutral border needs tau >= 1
          } else {
            const uint32_t* mid = (const uint32_t*)(sf + ey * FS) + (xs >> 1);
            const uint32_t m_first = (xs & 1) ? 0x0000FFFFu : 0u, m_last = (xs & 1) ? 0u : 0xFFFF0000u;
            const uint32_t target2 = val | (val << 16);
            const bool better = is_min ? rows_better<N1, true>(mid - FSW, mid, mid + FSW, n1, m_first, m_last, target2)
                                       : rows_better<N1, false>(mid - FSW, mid, mid + FSW, n1, m_first, m_last, target2);
            if (better) cand = false;
            else if (n > 1) { push = true; ent = (uint32_t)(mid - sfw) | ((uint32_t)(xs & 1) << 16) | ((uint32_t)(4 * cell + c) << 17); }
          }
        }
        if (cand) code = (code & ~(0xFFu << (8 * c))) | (pos << (8 * c));
        const unsigned m = __ballot_sync(0xFFFFFFFFu, push);
        if (m) {
          int base = 0;
          const int leader = __ffs(m) - 1;
          if ((int)lane == leader) base = atom_add_shared(A.qn + (u & 1), __popc(m));
          base = __shfl_sync(0xFFFFFFFFu, base, leader);
          if (push) A.queue[u & 1][base + __popc(m & lt)] = ent;
        }
          }
    }
    if (live) {
      if (!two) A.codes[cell] = code;
      else ((uint16_t*)(A.codes + cell))[tt] = (uint16_t)(tt ? code >> 16 : code);
    }
  }
}

// ---- phase 3b: the remaining rows (distance 2 .. n above and below the extreme) of the queued candidates
template <int N1, bool IS_MIN>
__device__ __forceinline__ void finish_scans(const NmsArgs& A, const uint32_t* queue, int nq, int q) {
  const int n = A.n, FSW = A.FS >> 1;
  const uint32_t* sfw = (const uint32_t*)A.sf1;
  uint8_t* codeb = (uint8_t*)A.codes;
  if (q < nq) {
    const uint32_t ent = queue[q];
    const uint32_t* rowc = sfw + (ent & 0xFFFFu);
    const uint32_t parity = (ent >> 16) & 1u;
    const uint32_t m_first = parity ? 0x0000FFFFu : 0u, m_last = parity ? 0u : 0xFFFF0000u;
    const uint32_t val = ((const uint16_t*)rowc)[parity + n];
    const uint32_t target2 = val | (val << 16);
    bool better = false;
    for (int r = 2; r <= n && !better; r++) {
      const uint32_t* up = rowc - r * FSW;
      const uint32_t* dn = rowc + r * FSW;
      better = rows_better<N1, IS_MIN>(up, dn, dn, n + 1, m_first, m_last, target2);
    }
    if (better) codeb[ent >> 17] = 0xFF;
  }
}

__device__ __forceinline__ void nms_pass(const NmsArgs& A, int item, unsigned lane) {
  switch (A.n + 1) {
    case 3: nms_cells<3>(A, item, lane); break;
    case 4: nms_cells<4>(A, item, lane); break;
    case 7: nms_cells<7>(A, item, lane); break;
    case 10: nms_cells<10>(A, item, lane); break;
    default: nms_cells<0>(A, item, lane); break;
  }
}
// kind 0: minima, 1: maxima
__device__ __forceinline__ void finish_pass(const NmsArgs& A, int kind, int nq, int q) {
  const uint32_t* queue = A.queue[kind];
  switch (A.n + 1) {
    case 3: if (kind) finish_scans<3, false>(A, queue, nq, q); else finish_scans<3, true>(A, queue, nq, q); break;
    case 4: if (kind) finish_scans<4, false>(A, queue, nq, q); else finish_scans<4, true>(A, queue, nq, q); break;
    case 7: if (kind) finish_scans<7, false>(A, queue, nq, q); else finish_scans<7, true>(A, queue, nq, q); break;
    case 10: if (kind) finish_scans<10, false>(A, queue, nq, q); else finish_scans<10, true>(A, queue, nq, q); break;
    default: if (kind) finish_scans<0, false>(A, queue, nq, q); else finish_scans<0, true>(A, queue, nq, q); break;
  }
}

// Warp-granular dynamic scheduling: the warps of a CTA take chunks of 32 work items from a shared counter, expensive
// chunks first, so that no warp waits long at the barrier that ends a phase.
__device__ __forceinline__ int next_chunk(int* counter, unsigned lane) {
  int c = 0;
  if (lane == 0) c = atom_add_shared(counter, 1);
  return __shfl_sync(0xFFFFFFFFu, c, 0);
}

// ----------------------------------------------------------------------------------------------------------
// Fused kernel.  One CTA = one tile of one image (TileCfg above).
//   phase 1  one elected thread issues a TMA tile load (cp.async.bulk.tensor.3d, zero fill outside the image) of the
//            image tile into shared memory; everybody waits on the mbarrier.
//   phase 2  register-window filters: Sobel walkers write du / dv (one coalesced 32-bit store per word and row),
//            blob / checkerboard walkers write the biased responses f1 / f2 to shared memory only.
//   phase 3  NMS of both passes on the responses: cell extremes as keys, tau test, quick window test (3a), the rest of
//            the windows of the survivors (3b), then one code word per owned cell (4 bytes = position of the kept
//            extreme of each class or 0xFF) to global memory (3c).  The candidate queues reuse the image tile.
__global__ void __launch_bounds__(MAX_FILTER_THREADS, 2)
k_filter_nms(const __grid_constant__ Geometry g, const FrameDev* frames, const __grid_constant__ SlotList sl, const __grid_constant__ TileCfg t,
             const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_full, int use_tma) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int slot = sl.s[blockIdx.z];
  const FrameDev F = frames[slot];
  const int tid = threadIdx.x, T = blockDim.x;
  const AxisTile& X = t.xt[blockIdx.x];
  const AxisTile& Y = t.yt[blockIdx.y];
  const int FS = t.FS, IS = t.IS, IH = t.IH, IW = IS >> 2;
  uint8_t* simg = smem;
  int16_t* sf1 = (int16_t*)(smem + t.img_bytes);
  int16_t* sf2 = sf1 + (size_t)t.FH * FS;
  uint64_t* s_bar = (uint64_t*)(smem + t.img_bytes + t.f_bytes);
  int* s_qn = (int*)(s_bar + 2);                          // four candidate counters, two chunk counters
  uint32_t* s_code = (uint32_t*)(s_qn + 8);
  const int x_ilo = X.i_lo, y_ilo = Y.i_lo;

  // ---- phase 1
  if (tid < 8) s_qn[tid] = 0;
  if (t.fused) {
    // Half-resolution mode, fused: the FULL-resolution tile comes in by TMA, part by part, into the (still unused) response
    // plane area.  Sobel walkers write du_full / dv_full from it (matcher.cpp:676), and the 2x2 box mean of
    // createHalfResolutionImage (matcher.cpp:636-647) goes straight into the image tile that the phases below work on:
    // the half-resolution image never exists in global memory.
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(s_bar);
    const uint32_t stage0 = (uint32_t)__cvta_generic_to_shared(sf1);
    const uint32_t simg_sa = (uint32_t)__cvta_generic_to_shared(simg);
    const unsigned lane = tid & 31;
    const int SR = t.SR, BW = t.BW;
    const int fx0 = 2 * x_ilo;                              // full-resolution column of staging byte 0
    const int xr = t.nbox == 2 ? 2 * IS - BW : 0;           // first column of the right box, relative to fx0
    const uint32_t part_bytes = (uint32_t)(t.nbox * BW * SR);   // one staging buffer; two of them alternate
    const uint32_t part_stride = (part_bytes + 127u) & ~127u;   // TMA destinations are 128-byte aligned
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar + 8));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // part p goes to buffer p & 1 and signals mbarrier p & 1; the load of part p + 1 is in flight while part p is worked on
    auto load_part = [&](int p) {
      const uint32_t dst = stage0 + (uint32_t)(p & 1) * part_stride, b = bar + 8u * (uint32_t)(p & 1);
      const int fy = 2 * (y_ilo + p * t.HP) - 2;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(b), "r"(part_bytes) : "memory");
      asm volatile(
          "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
          :: "r"(dst), "l"(&tmap_full), "r"(fx0), "r"(fy), "r"(slot), "r"(b) : "memory");
      if (t.nbox == 2)
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
            :: "r"(dst + (uint32_t)(BW * SR)), "l"(&tmap_full), "r"(fx0 + xr), "r"(fy), "r"(slot), "r"(b) : "memory");
    };
    if (tid == 0) { load_part(0); if (t.P > 1) load_part(1); }
    for (int p = 0; p < t.P; p++) {
      const int hr0 = p * t.HP, hr1 = min(hr0 + t.HP, IH);  // half-resolution rows of the image tile formed by this part
      const int fy0 = 2 * (y_ilo + hr0) - 2;                // first staged full-resolution row
      const uint32_t stage = stage0 + (uint32_t)(p & 1) * part_stride;
      const uint32_t right = stage + (uint32_t)(BW * SR) - (uint32_t)xr;
      mbar_wait_or_trap(bar + 8u * (uint32_t)(p & 1), (uint32_t)((p >> 1) & 1));
      // full-resolution Sobel rows of this part
      const int ry0 = max(Y.df_lo, 2 * (y_ilo + hr0)), ry1 = min(Y.df_hi, 2 * (y_ilo + hr1));
      const int nrF = max(ry1 - ry0, 0), nsF = (nrF + t.segF - 1) / t.segF;
      const int nitem = X.nwF * nsF, ncW = (nitem + 31) >> 5;
      const int nmean = (hr1 - hr0) * IW, ncB = (nmean + 127) >> 7;
      for (int c = next_chunk(s_qn + 6 + (p & 1), lane); c < ncW + ncB; c = next_chunk(s_qn + 6 + (p & 1), lane)) {
        if (c < ncW) {
          const int item = 32 * c + (int)lane;
          if (item < nitem) {
            const int sg = fast_div(item, X.inv_nwF), j = item - sg * X.nwF;
            const int gx = X.df_lo + 4 * j, gy0 = ry0 + sg * t.segF;
            const int b = gx - fx0;                          // byte column in the staged rows
            const uint32_t base = (t.nbox == 2 && b + 8 > BW) ? right : stage;
            walk_sobel(base + (uint32_t)((gy0 - 2 - fy0) * BW + b - 4), BW, min(t.segF, ry1 - gy0), gy0, gx, g.bpl, g.h, F.du_full, F.dv_full);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; k++) {
            const int idx = 128 * (c - ncW) + 32 * k + (int)lane;
            if (idx < nmean) {
              const int hr = fast_div(idx, 1.0f / (float)IW), w = idx - hr * IW;
              const int b8 = 8 * w;
              const uint32_t base = (t.nbox == 2 && b8 + 8 > BW) ? right : stage;
              const uint32_t a = base + (uint32_t)((2 * hr + 2) * BW + b8);
              const uint2 r0 = lds64(a), r1 = lds64(a + (uint32_t)BW);
              // pairs of horizontal neighbours as 16-bit lanes, rows added, truncating division by four
              const uint32_t s0 = (r0.x & 0x00FF00FFu) + ((r0.x >> 8) & 0x00FF00FFu) + (r1.x & 0x00FF00FFu) + ((r1.x >> 8) & 0x00FF00FFu);
              const uint32_t s1 = (r0.y & 0x00FF00FFu) + ((r0.y >> 8) & 0x00FF00FFu) + (r1.y & 0x00FF00FFu) + ((r1.y >> 8) & 0x00FF00FFu);
              uint32_t out = __byte_perm((s0 >> 2) & 0x00FF00FFu, (s1 >> 2) & 0x00FF00FFu, 0x6420);
              const int gxh = x_ilo + 4 * w, gyh = y_ilo + hr0 + hr;
              if (gyh >= g.hm) out = 0;
              else if (gxh + 3 >= g.wm) out = gxh >= g.wm ? 0u : out & (0xFFFFFFFFu >> (8 * (gxh + 4 - g.wm)));   // pad columns stay zero
              sts32(simg_sa + (uint32_t)((hr0 + hr) * IS + 4 * w), out);
            }
          }
        }
      }
      if (tid == 0) s_qn[6 + ((p + 1) & 1)] = 0;            // chunk counter of the next part (idle since the part before this one)
      __syncthreads();
      if (tid == 0 && p + 2 < t.P) load_part(p + 2);        // this buffer is free again
    }
  } else if (use_tma) {
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(s_bar);
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(simg);
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
      const uint32_t bytes = (uint32_t)(IH * IS);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
      asm volatile(
          "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
          :: "r"(dst), "l"(&tmap), "r"(x_ilo), "r"(y_ilo), "r"(slot), "r"(bar) : "memory");
    }
    mbar_wait_or_trap(bar, 0);
  } else {
    const uint8_t* __restrict__ I = g.half ? F.half : F.img;
    for (int idx = tid; idx < IH * IW; idx += T) {
      const int ly = idx / IW, lw = idx - ly * IW;
      const int gx = x_ilo + 4 * lw, gy = y_ilo + ly;
      uint32_t v = 0;
      if (gy >= 0 && gy < g.hm && gx >= 0 && gx < g.bplm) v = __ldg((const uint32_t*)(I + (size_t)gy * g.bplm + gx));
      *(uint32_t*)(simg + ly * IS + 4 * lw) = v;
    }
    __syncthreads();
  }

  // ---- phase 2: work items = (word column, row segment) of the Sobel range, then of the response range
  {
    const int nwa = X.nwa, nwb = X.nwb, nrb = Y.f_hi - Y.f_lo;
    const int na = nwa * Y.nsA, nb = nwb * Y.nsB;
    const int na32 = (na + 31) & ~31;                       // response walkers start on a warp boundary: no warp runs both kinds
    const uint32_t img_sa = (uint32_t)__cvta_generic_to_shared(simg), f1_sa = (uint32_t)__cvta_generic_to_shared(sf1);
    const uint32_t f2_sa = f1_sa + (uint32_t)(t.FH * FS * 2);
    for (int item = tid; item < na32 + nb; item += T) {
      if (item < na32) {
        if (item >= na) continue;
        const int sg = fast_div(item, X.inv_nwa), j = item - sg * nwa;
        const int gx = X.d_lo + 4 * j, gy0 = Y.d_lo + sg * Y.segA;
        const uint32_t col = img_sa + (uint32_t)((gy0 - 2 - y_ilo) * IS + (gx - x_ilo) - 4);
        walk_sobel(col, IS, min(Y.segA, Y.d_hi - gy0), gy0, gx, g.bplm, g.hm, F.du, F.dv);
      } else {
        const int it = item - na32;
        const int sg = fast_div(it, X.inv_nwb), j = it - sg * nwb;
        const int gx = X.f_lo + 4 * j, ly0 = sg * Y.segB, gy0 = Y.f_lo + ly0;
        const uint32_t col = img_sa + (uint32_t)((gy0 - 2 - y_ilo) * IS + (gx - x_ilo) - 4);
        const uint32_t o = (uint32_t)((ly0 * FS + 4 * j) * 2);
        walk_blob_checker(col, IS, min(Y.segB, nrb - ly0), f1_sa + o, f2_sa + o, 2 * FS);
      }
    }
  }
  __syncthreads();
  if (X.fill_hi > X.v_hi || Y.fill_hi > Y.v_hi) {           // tiles at the right / bottom image border only
    const int vw = X.v_hi - X.f_lo, fw = X.fill_hi - X.f_lo, vr = Y.v_hi - Y.f_lo, fr = Y.fill_hi - Y.f_lo;
    const int ncol = fw - vw;
    for (int idx = tid; idx < fr * ncol; idx += T) {        // columns behind the last valid one, all rows
      const int row = idx / ncol, c = vw + idx - row * ncol;
      sf1[row * FS + c] = BIAS_F1; sf2[row * FS + c] = BIAS_F2;
    }
    for (int idx = tid; idx < (fr - vr) * vw; idx += T) {   // rows below the last valid one
      const int row = vr + idx / vw, c = idx % vw;
      sf1[row * FS + c] = BIAS_F1; sf2[row * FS + c] = BIAS_F2;
    }
    __syncthreads();
  }

  // ---- phase 3
  {
    NmsArgs A[2];
    int ncell_total = 0;
    uint32_t* qbase = (uint32_t*)simg;                    // the image tile is dead: its memory holds the candidate queues
#pragma unroll
    for (int p = 0; p < 2; p++) {
      NmsArgs& a = A[p];
      const int n = g.n[p], org = n + VISO_MARGIN;
      a.sf1 = sf1; a.sf2 = sf2; a.FS = FS;
      a.n = n; a.nk = X.nk[p]; a.inv_nk = X.inv_nk[p];
      a.ncell = p < g.first_pass ? 0 : X.nk[p] * Y.nk[p];
      a.codes = s_code + ncell_total;
      a.queue[0] = qbase; a.queue[1] = qbase + 2 * a.ncell; qbase += 4 * a.ncell;
      a.qn = s_qn + 2 * p;
      a.cx0 = org + X.klo[p] * (n + 1) - X.f_lo; a.cy0 = org + Y.klo[p] * (n + 1) - Y.f_lo;
      a.xhi = g.wm - 1 - VISO_MARGIN - X.f_lo; a.yhi = g.hm - 1 - VISO_MARGIN - Y.f_lo;    // window clamps, plane coordinates
      a.tau = g.tau;
      ncell_total += a.ncell;
    }
    const unsigned lane = tid & 31;
    {
      // 3a: chunks of the sparse pass (two lanes per cell if its cells have six or more rows) first, then the dense pass
      const int g0 = g.n[0] + 1 >= 6 ? 2 : 1, g1 = g.n[1] + 1 >= 6 ? 2 : 1;
      const int nc0 = (A[0].ncell * g0 + 31) >> 5, nc1 = (A[1].ncell * g1 + 31) >> 5;
      for (int c = next_chunk(s_qn + 4, lane); c < nc0 + nc1; c = next_chunk(s_qn + 4, lane)) {
        if (c < nc0) nms_pass(A[0], 32 * c + lane, lane);
        else nms_pass(A[1], 32 * (c - nc0) + lane, lane);
      }
    }
    __syncthreads();
    {
      // 3b: chunks of the four candidate queues
      const int q0 = s_qn[0], q1 = s_qn[1], q2 = s_qn[2], q3 = s_qn[3];
      const int e0 = (q0 + 31) >> 5, e1 = e0 + ((q1 + 31) >> 5), e2 = e1 + ((q2 + 31) >> 5), e3 = e2 + ((q3 + 31) >> 5);
      for (int c = next_chunk(s_qn + 5, lane); c < e3; c = next_chunk(s_qn + 5, lane)) {
        if (c < e0) finish_pass(A[0], 0, q0, 32 * c + lane);
        else if (c < e1) finish_pass(A[0], 1, q1, 32 * (c - e0) + lane);
        else if (c < e2) finish_pass(A[1], 0, q2, 32 * (c - e1) + lane);
        else finish_pass(A[1], 1, q3, 32 * (c - e2) + lane);
      }
    }
    __syncthreads();

    // 3c: code words to global memory, cell-column-major
    for (int idx = tid; idx < ncell_total; idx += T) {
      const bool second = idx >= A[0].ncell;
      const int cell = second ? idx - A[0].ncell : idx;
      const int nkp = second ? A[1].nk : A[0].nk;
      const int ll = fast_div(cell, second ? A[1].inv_nk : A[0].inv_nk), kk = cell - ll * nkp;
      uint32_t* dst = second ? F.codes[1] : F.codes[0];
      dst[(size_t)((second ? X.klo[1] : X.klo[0]) + kk) * (second ? g.ncy[1] : g.ncy[0]) + ((second ? Y.klo[1] : Y.klo[0]) + ll)] = s_code[idx];
    }
  }
}

// ----------------------------------------------------------------------------------------------------------
// ordered compaction, step 1: records emitted per chunk of CELLS_PER_BLOCK cells (cells in column-major order)
__device__ __forceinline__ int code_count(uint32_t code) {
  return ((code & 0xFFu) != 0xFFu) + ((code & 0xFF00u) != 0xFF00u) + ((code & 0xFF0000u) != 0xFF0000u) + ((code >> 24) != 0xFFu);
}

__global__ void __launch_bounds__(CELLS_PER_BLOCK) k_cell_count(Geometry g, const FrameDev* frames, SlotList sl) {
  const int p = blockIdx.y;
  if (p < g.first_pass) return;
  const FrameDev F = frames[sl.s[blockIdx.z]];
  const int ncells = g.ncx[p] * g.ncy[p];
  const int nchunk = (ncells + CELLS_PER_BLOCK - 1) / CELLS_PER_BLOCK;
  if ((int)blockIdx.x >= nchunk) return;
  const int c = blockIdx.x * CELLS_PER_BLOCK + threadIdx.x;
  int cnt = c < ncells ? code_count(F.codes[p][c]) : 0;
  __shared__ int wsum[CELLS_PER_BLOCK / 32];
  for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xFFFFFFFFu, cnt, o);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x < 32) {
    int v = threadIdx.x < CELLS_PER_BLOCK / 32 ? wsum[threadIdx.x] : 0;
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if (threadIdx.x == 0) F.blk[p][blockIdx.x] = v;
  }
}

// descriptor sample offsets (matcher.cpp:445-476): 16 (du,dv) pairs
__constant__ int8_t c_desc_ox[16] = {-3, -3, -1, -1, 3, 3, 1, 1, -1, -1, 1, 1, -5, -5, 5, 5};
__constant__ int8_t c_desc_oy[16] = {-1, 1, -1, 1, -1, 1, -1, 1, -5, 5, -5, 5, -3, 3, -3, 3};

// step 2: chunk base = sum of earlier chunks, block scan, then one warp per record gathers the 32 descriptor
// bytes (one byte per lane), packs them to words with shuffles and stores the 48-byte record with 12 lanes.
__global__ void __launch_bounds__(CELLS_PER_BLOCK) k_emit_records(Geometry g, const FrameDev* frames, SlotList sl) {
  const int p = blockIdx.y;
  if (p < g.first_pass) return;
  const FrameDev F = frames[sl.s[blockIdx.z]];
  const int ncells = g.ncx[p] * g.ncy[p];
  const int nchunk = (ncells + CELLS_PER_BLOCK - 1) / CELLS_PER_BLOCK;
  if ((int)blockIdx.x >= nchunk) {
    if (nchunk == 0 && blockIdx.x == 0 && threadIdx.x == 0) F.counts[p] = 0;
    return;
  }
  __shared__ int wsum[CELLS_PER_BLOCK / 32];
  __shared__ int s_base, s_total;
  __shared__ uint32_t s_list[4 * CELLS_PER_BLOCK];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;

  // base of this chunk
  int acc = 0;
  for (int b = tid; b < (int)blockIdx.x; b += CELLS_PER_BLOCK) acc += F.blk[p][b];
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
  if (lane == 0) wsum[wid] = acc;
  __syncthreads();
  if (tid < 32) {
    int v = tid < CELLS_PER_BLOCK / 32 ? wsum[tid] : 0;
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if (tid == 0) s_base = v;
  }
  __syncthreads();

  // exclusive scan of the per-cell counts
  const int c = blockIdx.x * CELLS_PER_BLOCK + tid;
  const uint32_t code = c < ncells ? F.codes[p][c] : 0xFFFFFFFFu;
  const int cnt = code_count(code);
  int incl = cnt;
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
  if (lane == 31) wsum[wid] = incl;
  __syncthreads();
  if (tid < 32) {
    int v = tid < CELLS_PER_BLOCK / 32 ? wsum[tid] : 0, s = v;
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xFFFFFFFFu, s, o); if (lane >= o) s += t; }
    if (tid < CELLS_PER_BLOCK / 32) wsum[tid] = s - v;
    if (tid == CELLS_PER_BLOCK / 32 - 1) s_total = s;
  }
  __syncthreads();
  int off = wsum[wid] + incl - cnt;
  if (cnt) {
    const int n = g.n[p];
    const int k = c / g.ncy[p], l = c - k * g.ncy[p];
    const int i = n + VISO_MARGIN + k * (n + 1), j = n + VISO_MARGIN + l * (n + 1);
#pragma unroll
    for (int cls = 0; cls < 4; cls++) {
      uint32_t b = (code >> (8 * cls)) & 0xFFu;
      if (b != 0xFFu) s_list[off++] = (uint32_t)(i + (b >> 4)) | ((uint32_t)(j + (b & 15)) << 13) | ((uint32_t)cls << 26);
    }
  }
  __syncthreads();
  const int total = s_total, base = s_base;
  if (blockIdx.x == nchunk - 1 && tid == 0) {
    int all = base + total;
    if (all > g.cap[p]) { F.counts[2] = 1; all = g.cap[p]; }
    F.counts[p] = all;
  }
  // four records per warp and round: the byte gathers of a round are independent loads in flight together
  constexpr int NWARP = CELLS_PER_BLOCK / 32, UNR = 4;
  const int s = lane >> 1;
  const uint8_t* plane = (lane & 1) ? F.dv : F.du;
  const int ox = c_desc_ox[s], oy = c_desc_oy[s];
  const int limit = min(total, g.cap[p] - base);
  for (int e0 = wid; e0 < limit; e0 += NWARP * UNR) {
    uint32_t ent[UNR], byte[UNR];
#pragma unroll
    for (int k = 0; k < UNR; k++) {
      const int e = e0 + k * NWARP;
      ent[k] = e < limit ? s_list[e] : s_list[e0];
      const int u = ent[k] & 0x1FFF, v = (ent[k] >> 13) & 0x1FFF;
      byte[k] = plane[(size_t)(v + oy) * g.bplm + u + ox];
    }
#pragma unroll
    for (int k = 0; k < UNR; k++) {
      const int e = e0 + k * NWARP;
      const int u = ent[k] & 0x1FFF, v = (ent[k] >> 13) & 0x1FFF, cls = ent[k] >> 26;
      uint32_t w = byte[k] << (8 * (lane & 3));
      w |= __shfl_xor_sync(0xFFFFFFFFu, w, 1);
      w |= __shfl_xor_sync(0xFFFFFFFFu, w, 2);
      const uint32_t dw = __shfl_sync(0xFFFFFFFFu, w, ((lane - 4) & 7) * 4);
      if (lane < 12 && e < limit) {
        int32_t out;
        if (lane == 0) out = u * g.scale; else if (lane == 1) out = v * g.scale; else if (lane == 2) out = 0;
        else if (lane == 3) out = cls; else out = (int32_t)dw;
        F.rec[p][(size_t)(base + e) * 12 + lane] = out;
      }
    }
  }
}

// ----------------------------------------------------------------------------------------------------------
// bin index (createIndexVector, matcher.cpp:870-890): counting sort of the records by (class, v_bin, u_bin).
// The order inside a bin is not the reference's (ascending index); the matcher compares complete
// (cost, u_bin, v_bin, index) keys instead, which reproduces the reference's first-minimum rule exactly.
__global__ void __launch_bounds__(1024) k_build_bins(Geometry g, const FrameDev* frames, SlotList sl) {
  const int p = blockIdx.y;
  if (p < g.first_pass) return;
  const FrameDev F = frames[sl.s[blockIdx.z]];
  const int tid = threadIdx.x;
  const int n = F.counts[p];
  int32_t* start = F.bin_start[p];
  int32_t* cursor = F.bin_cursor[p];
  const int32_t* rec = F.rec[p];
  for (int b = tid; b <= g.nbins; b += 1024) cursor[b] = 0;
  __syncthreads();
  const float bs = (float)g.binsize;
  auto bin_of = [&](int u, int v, int c) {
    int ubin = min((int)floorf((float)u / bs), g.ub - 1);
    int vbin = min((int)floorf((float)v / bs), g.vb - 1);
    return (c * g.vb + vbin) * g.ub + ubin;
  };
  for (int i = tid; i < n; i += 1024) {
    int4 hdr = *(const int4*)(rec + (size_t)i * 12);
    atomicAdd(&cursor[bin_of(hdr.x, hdr.y, hdr.w)], 1);
  }
  __syncthreads();
  // exclusive scan of the histogram, 1024 bins per round with a running carry
  __shared__ int wsum[32];
  __shared__ int s_carry;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int b0 = 0; b0 <= g.nbins; b0 += 1024) {
    const int b = b0 + tid;
    const int v = b < g.nbins ? cursor[b] : 0;
    int incl = v;
    const int lane = tid & 31, wid = tid >> 5;
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) wsum[wid] = incl;
    __syncthreads();
    if (tid < 32) {
      int w = wsum[tid], s = w;
      for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xFFFFFFFFu, s, o); if (lane >= o) s += t; }
      wsum[tid] = s - w;
    }
    __syncthreads();
    const int excl = s_carry + wsum[wid] + incl - v;
    if (b <= g.nbins) { start[b] = excl; cursor[b] = excl; }
    __syncthreads();
    if (tid == 1023) s_carry = excl + v;
    __syncthreads();
  }
  for (int i = tid; i < n; i += 1024) {
    int4 hdr = *(const int4*)(rec + (size_t)i * 12);
    int pos = atomicAdd(&cursor[bin_of(hdr.x, hdr.y, hdr.w)], 1);
    F.bin_ent[p][pos] = make_int2(hdr.x | (hdr.y << 16), i);
  }
}

// record counts (and the overflow flag) of the frames of one launch, gathered for a single read-back
__global__ void k_gather_counts(const FrameDev* frames, SlotList sl, int32_t* out) {
  const int i = threadIdx.x;
  if (i < sl.n) {
    const int32_t* c = frames[sl.s[i]].counts;
    out[4 * i] = c[0]; out[4 * i + 1] = c[1]; out[4 * i + 2] = c[2]; out[4 * i + 3] = 0;
  }
}

}  // namespace

// ----------------------------------------------------------------------------------------------------------
// host side: tile configurations, tensor maps, launch
namespace {

// kx x ky aligning-pass cells per tile; fills the configuration and the two per-axis tables (host copies); returns false
// if the configuration does not fit (TMA box, shared memory, packed queue entries)
bool make_tile_cfg(const Geometry& g, int kx, int ky, int threads, bool fused, TileCfg& t, std::vector<AxisTile>& xt, std::vector<AxisTile>& yt) {
  memset(&t, 0, sizeof t);
  const int pa = g.first_pass;                              // the aligning pass: sparse when multi_stage (n[0] >= n[1])
  t.nA = g.n[pa]; t.stepA = t.nA + 1; t.orgA = t.nA + VISO_MARGIN;
  t.extR = t.nA;
  if (pa == 0 && 2 * g.n[1] > t.extR) t.extR = 2 * g.n[1];
  t.kx = kx; t.ky = ky; t.TWn = kx * t.stepA; t.THn = ky * t.stepA;
  t.ntx = g.ncx[pa] > 0 ? (g.ncx[pa] + kx - 1) / kx : (g.bplm - t.orgA + t.TWn - 1) / t.TWn;
  t.nty = g.ncy[pa] > 0 ? (g.ncy[pa] + ky - 1) / ky : (g.hm - t.orgA + t.THn - 1) / t.THn;
  if (t.ntx < 1) t.ntx = 1;
  if (t.nty < 1) t.nty = 1;
  xt.assign(t.ntx, AxisTile()); yt.assign(t.nty, AxisTile());
  int nwf = 1, is = 16, fh = 1, ih = 1, nwa_max = 1, nwf_alloc = 1;
  int cells_x[2] = {0, 0}, cells_y[2] = {0, 0};
  for (int a = 0; a < t.ntx; a++) {
    AxisTile& X = xt[a];
    memset(&X, 0, sizeof X);
    tile_range(t, a, t.ntx, g.wm, g.bplm, true, X);
    // fused half-resolution mode: the last tile also writes the full-resolution pad columns up to bpl (> 2 bplm if w is odd)
    if (fused && a == t.ntx - 1 && X.i_hi < (g.bpl + 1) / 2 + 4) X.i_hi = (g.bpl + 1) / 2 + 4;
    X.nwa = (X.d_hi - X.d_lo) / 4; X.nwb = (X.f_hi - X.f_lo) / 4;
    nwf_alloc = std::max(nwf_alloc, (X.fill_hi - X.f_lo) / 4);
    X.inv_nwa = 1.0f / (float)std::max(X.nwa, 1); X.inv_nwb = 1.0f / (float)std::max(X.nwb, 1);
    nwf = std::max(nwf, X.nwb);
    is = std::max(is, (int)align_up((size_t)(X.i_hi - X.i_lo), 16));
    nwa_max = std::max(nwa_max, X.nwa);
    for (int p = 0; p < 2; p++) {
      if (p >= g.first_pass) owned_cells(X, g.n[p], g.ncx[p], X.klo[p], X.nk[p]);
      X.inv_nk[p] = 1.0f / (float)std::max(X.nk[p], 1);
      cells_x[p] = std::max(cells_x[p], X.nk[p]);
    }
  }
  for (int b = 0; b < t.nty; b++) {
    AxisTile& Y = yt[b];
    memset(&Y, 0, sizeof Y);
    tile_range(t, b, t.nty, g.hm, g.hm, false, Y);
    fh = std::max(fh, Y.fill_hi - Y.f_lo);
    ih = std::max(ih, Y.i_hi - Y.i_lo);
    for (int p = 0; p < 2; p++) {
      if (p >= g.first_pass) owned_cells(Y, g.n[p], g.ncy[p], Y.klo[p], Y.nk[p]);
      Y.inv_nk[p] = 1.0f / (float)std::max(Y.nk[p], 1);
      cells_y[p] = std::max(cells_y[p], Y.nk[p]);
    }
  }
  // rows per walker: as short as possible (more walkers) while one round of the threads covers the whole tile
  for (int b = 0; b < t.nty; b++) {
    AxisTile& Y = yt[b];
    const int nra = std::max(Y.d_hi - Y.d_lo, 0), nrb = std::max(Y.f_hi - Y.f_lo, 0);
    Y.nsA = nra > 0 ? 1 : 0; Y.nsB = nrb > 0 ? 1 : 0;
    for (int s = 8; s <= std::max(nra, nrb); s++) {
      const int na = (nra + s - 1) / s, nb = (nrb + s - 1) / s;
      if (((nwa_max * na + 31) & ~31) + nwf * nb <= threads) { Y.nsA = na; Y.nsB = nb; break; }
    }
    Y.segA = Y.nsA ? (nra + Y.nsA - 1) / Y.nsA : 1;
    Y.segB = Y.nsB ? (nrb + Y.nsB - 1) / Y.nsB : 1;
  }
  t.NWf = nwf_alloc; t.FS = 4 * nwf_alloc; t.FH = fh; t.IS = is; t.IH = ih;
  t.max_cells = cells_x[0] * cells_y[0] + cells_x[1] * cells_y[1];
  t.threads = threads;
  // the image tile doubles as the candidate queues of phase 3 (four entries of 4 bytes per cell at most)
  t.img_bytes = (unsigned)align_up(std::max((size_t)t.IS * t.IH, (size_t)16 * t.max_cells), 128);
  t.f_bytes = (unsigned)align_up((size_t)2 * t.FH * t.FS * sizeof(int16_t) + 16, 16);
  t.smem = t.img_bytes + t.f_bytes + 16 + 32 + (unsigned)t.max_cells * 4 + 16;
  if (fused) {
    // full-resolution staging inside the response plane area: two overlapping boxes of 256 bytes per row cover 2 IS <= 480
    if (2 * t.IS > 480) return false;
    t.fused = 1;
    t.nbox = 2 * t.IS > 256 ? 2 : 1;
    t.BW = t.nbox == 2 ? 256 : 2 * t.IS;
    const int rows_fit = (int)(t.f_bytes / (unsigned)(2 * t.nbox * t.BW));     // two staging buffers
    // at least 4 half-resolution rows per part: the response plane area of a small tile is enlarged to hold them
    const int hp = std::max(std::min((rows_fit - 4) / 2, 126), 4);
    t.P = (t.IH + hp - 1) / hp;
    t.HP = (t.IH + t.P - 1) / t.P;
    t.SR = 2 * t.HP + 4;
    // the second buffer starts on the next 128-byte boundary (a TMA destination must be 128-byte aligned)
    t.f_bytes = std::max(t.f_bytes, 2 * (unsigned)align_up((size_t)t.nbox * t.BW * t.SR, 128));
    t.smem = t.img_bytes + t.f_bytes + 16 + 32 + (unsigned)t.max_cells * 4 + 16;
    int nwF_max = 1;
    for (int a = 0; a < t.ntx; a++) {
      AxisTile& X = xt[a];
      X.df_lo = 2 * X.d_lo; X.df_hi = a == t.ntx - 1 ? g.bpl : 2 * X.d_hi;
      X.nwF = std::max(X.df_hi - X.df_lo, 0) / 4; X.inv_nwF = 1.0f / (float)std::max(X.nwF, 1);
      nwF_max = std::max(nwF_max, X.nwF);
    }
    for (int b = 0; b < t.nty; b++) { AxisTile& Y = yt[b]; Y.df_lo = 2 * Y.d_lo; Y.df_hi = b == t.nty - 1 ? g.h : 2 * Y.d_hi; }
    // rows per full-resolution Sobel walker: one round of the threads covers a part
    t.segF = 2 * t.HP;
    for (int sg = 8; sg < 2 * t.HP; sg++)
      if (nwF_max * ((2 * t.HP + sg - 1) / sg) <= threads) { t.segF = sg; break; }
  }
  return t.IS <= 256 && t.IH <= 256 && t.smem <= 227 * 1024 && (size_t)t.FH * t.FS <= 65535 && t.max_cells <= 8191;
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// TMA descriptor of the matching-resolution image plane of every frame slot: a 3-D tensor (bytes per line, rows,
// frame slots) with the tile's box; out-of-bounds elements are filled with zeros, which is what the filters expect
// outside the image.
int encode_tile_map(visocu_ctx* ctx, const TileCfg& t, CUtensorMap* out, bool full) {
  const Geometry& g = ctx->g;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  CU_TRY(ctx, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return visocu_set_error(ctx, VISOCU_ECUDA, "cuTensorMapEncodeTiled is not available");
  const FrameDev& F0 = ctx->frames_h[0];
  // full: the full-resolution image planes with the staging box of the fused half-resolution mode
  void* base = (g.half && !full) ? (void*)F0.half : (void*)F0.img;
  const cuuint64_t dims[3] = {(cuuint64_t)(full ? g.bpl : g.bplm), (cuuint64_t)(full ? g.h : g.hm), (cuuint64_t)ctx->n_frames};
  const cuuint64_t strides[2] = {(cuuint64_t)(full ? g.bpl : g.bplm), (cuuint64_t)ctx->frame_stride};
  const cuuint32_t box[3] = {(cuuint32_t)(full ? t.BW : t.IS), (cuuint32_t)(full ? t.SR : t.IH), 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = ((EncodeFn)fn)(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return visocu_set_error(ctx, VISOCU_ECUDA, "cuTensorMapEncodeTiled failed with %d", (int)r);
  return VISOCU_OK;
}

}  // namespace

// Tile configurations of a context: up to VISO_TILE_LEVELS sizes, largest first.  Large tiles have the smallest halo
// (best throughput when a launch has many frames), small tiles give a launch of a few frames enough CTAs to spread
// over the GPU.  VISOCU_TILE="kx,ky,threads" pins one configuration (experiments).
void visocu_free_tiles(visocu_ctx* ctx) {
  for (int c = 0; c < VISO_TILE_LEVELS; c++) {
    if (ctx->tiles[c].tables) cudaFree(ctx->tiles[c].tables);
    ctx->tiles[c].tables = nullptr;
  }
  ctx->n_tiles = 0;
}

int visocu_make_tensor_map(visocu_ctx* ctx, size_t frame_stride_bytes) {
  const Geometry& g = ctx->g;
  ctx->frame_stride = frame_stride_bytes;
  ctx->use_tma = 1;
  if (const char* env = getenv("VISOCU_TMA")) if (env[0] == '0') ctx->use_tma = 0;    // debugging switch: stage the tile with plain loads
  const int stepA = g.n[g.first_pass] + 1;
  // VISOCU_FUSED_HALF=0: half-resolution mode with separate kernels for the half image and the full-resolution Sobel planes
  bool fused = g.half && ctx->use_tma;
  if (const char* env = getenv("VISOCU_FUSED_HALF")) if (env[0] == '0') fused = false;
  ctx->fused_half = fused ? 1 : 0;
  // upper limits of the tile size per level (aligning-pass cells); the cells of the image are then spread evenly over the
  // tiles so that no tile row or column is nearly empty.  Fused half-resolution mode: 2 IS <= 480 limits the width.
  const int pa = g.first_pass;
  auto balanced = [](int ncells, int kmax) { kmax = std::max(kmax, 1); if (ncells <= 0) return kmax; const int nt = (ncells + kmax - 1) / kmax; return (ncells + nt - 1) / nt; };
  int cand[VISO_TILE_LEVELS][3] = {{balanced(g.ncx[pa], (fused ? 190 : 210) / stepA), balanced(g.ncy[pa], (fused ? 80 : 60) / stepA), 512},
                                   {balanced(g.ncx[pa], 100 / stepA), balanced(g.ncy[pa], 60 / stepA), fused ? 384 : 512},
                                   {balanced(g.ncx[pa], 100 / stepA), balanced(g.ncy[pa], 30 / stepA), 256}};
  int ncand = VISO_TILE_LEVELS;
  if (const char* env = getenv("VISOCU_TILE")) {
    int kx = 0, ky = 0, th = 0;
    if (sscanf(env, "%d,%d,%d", &kx, &ky, &th) == 3 && kx > 0 && ky > 0 && th >= 32 && th <= MAX_FILTER_THREADS && th % 32 == 0) {
      cand[0][0] = kx; cand[0][1] = ky; cand[0][2] = th; ncand = 1;
    }
  }
  visocu_free_tiles(ctx);
  for (int c = 0; c < ncand; c++) {
    int kx = std::max(cand[c][0], 1), ky = std::max(cand[c][1], 1);
    TileCfg t;
    std::vector<AxisTile> xt, yt;
    bool ok = make_tile_cfg(g, kx, ky, cand[c][2], fused, t, xt, yt);
    while (!ok && (kx > 1 || ky > 1)) {                     // shrink until the box and the shared memory fit
      if (kx >= ky && kx > 1) kx = (kx + 1) / 2; else ky = (ky + 1) / 2;
      ok = make_tile_cfg(g, kx, ky, cand[c][2], fused, t, xt, yt);
    }
    if (!ok) continue;
    visocu_tile& slot = ctx->tiles[ctx->n_tiles];
    static_assert(sizeof(TileCfg) <= sizeof(slot.cfg), "TileCfg storage");
    // per-axis tables: x entries then y entries in one device block
    const size_t nb = sizeof(AxisTile) * (xt.size() + yt.size());
    CU_TRY(ctx, cudaMalloc(&slot.tables, nb));
    std::vector<AxisTile> both(xt);
    both.insert(both.end(), yt.begin(), yt.end());
    CU_TRY(ctx, cudaMemcpy(slot.tables, both.data(), nb, cudaMemcpyHostToDevice));
    t.xt = (const AxisTile*)slot.tables; t.yt = t.xt + xt.size();
    memcpy(slot.cfg, &t, sizeof t);
    ctx->n_tiles++;
    if (ctx->use_tma) { int rc = encode_tile_map(ctx, t, &slot.tmap, false); if (rc) return rc; }
    if (t.fused) { int rc = encode_tile_map(ctx, t, &slot.tmap_full, true); if (rc) return rc; }
  }
  if (ctx->n_tiles == 0) return visocu_set_error(ctx, VISOCU_EINVAL, "no tile configuration fits %dx%d with nms_n = %d", g.wm, g.hm, g.n[1]);
  return VISOCU_OK;
}

// the half-resolution image of one frame, for visocu_get_plane (the fused path never writes it)
int visocu_make_half_image(visocu_ctx* ctx, int frame) {
  const Geometry& g = ctx->g;
  if (!g.half) return VISOCU_OK;
  SlotList sl; sl.n = 1; sl.s[0] = frame;
  dim3 bh(32, 8), gh((g.bplm / 4 + 31) / 32, (g.hm + 7) / 8, 1);
  k_half_image<<<gh, bh, 0, ctx->stream>>>(g, ctx->frames_d, sl);
  CU_LAUNCH_CHECK(ctx);
  return VISOCU_OK;
}

// the largest tiles that still give a launch of n frames about one CTA per SM; else the smallest
static int pick_tile_level(const visocu_ctx* ctx, int n) {
  for (int c = 0; c < ctx->n_tiles; c++) {
    TileCfg t; memcpy(&t, ctx->tiles[c].cfg, sizeof t);
    if ((long long)t.ntx * t.nty * n >= ctx->sm_count) return c;
  }
  return ctx->n_tiles - 1;
}

extern "C" int visocu_tile_levels(const visocu_ctx* ctx, int32_t n_launch, int32_t* n_levels, int32_t* out5, int32_t* pick) {
  if (!ctx || !ctx->configured || n_launch < 1 || n_launch > VISO_MAX_BATCH) return VISOCU_EINVAL;
  if (n_levels) *n_levels = ctx->n_tiles;
  for (int c = 0; c < ctx->n_tiles && out5; c++) {
    TileCfg t; memcpy(&t, ctx->tiles[c].cfg, sizeof t);
    const int32_t v[5] = {t.kx, t.ky, t.ntx, t.nty, t.threads};
    memcpy(out5 + 5 * c, v, sizeof v);
  }
  if (pick) *pick = pick_tile_level(ctx, n_launch);
  return VISOCU_OK;
}

int visocu_launch_features(visocu_ctx* ctx, const SlotList& sl) {
  const Geometry& g = ctx->g;
  cudaStream_t st = ctx->stream;
  if (g.half && !ctx->fused_half) {
    dim3 bh(32, 8), gh((g.bplm / 4 + 31) / 32, (g.hm + 7) / 8, sl.n);
    k_half_image<<<gh, bh, 0, st>>>(g, ctx->frames_d, sl);
    CU_LAUNCH_CHECK(ctx);
    dim3 gs((g.bpl + SF_TW - 1) / SF_TW, (g.h + SF_TH - 1) / SF_TH, sl.n);
    k_sobel_full<<<gs, 256, 0, st>>>(g, ctx->frames_d, sl);
    CU_LAUNCH_CHECK(ctx);
  }
  {
    const int pick = pick_tile_level(ctx, sl.n);
    TileCfg t; memcpy(&t, ctx->tiles[pick].cfg, sizeof t);
    // opt in to large dynamic shared memory once per device (the attribute belongs to the function on a device, not
    // to a context: several contexts with different tile shapes share it)
    {
      static std::mutex mtx;
      static bool done[64] = {false};
      std::lock_guard<std::mutex> lock(mtx);
      if (!done[ctx->device & 63]) {
        CU_TRY(ctx, cudaFuncSetAttribute(k_filter_nms, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        done[ctx->device & 63] = true;
      }
    }
    dim3 grid(t.ntx, t.nty, sl.n);
    if (ctx->profile) CU_TRY(ctx, cudaEventRecord(ctx->pev0, st));
    k_filter_nms<<<grid, t.threads, t.smem, st>>>(g, ctx->frames_d, sl, t, ctx->tiles[pick].tmap, ctx->tiles[pick].tmap_full, ctx->use_tma);
    CU_LAUNCH_CHECK(ctx);
    if (ctx->profile) {
      // profiling mode only: this synchronises the stream after every fused launch
      float ms = 0;
      CU_TRY(ctx, cudaEventRecord(ctx->pev1, st));
      CU_TRY(ctx, cudaEventSynchronize(ctx->pev1));
      CU_TRY(ctx, cudaEventElapsedTime(&ms, ctx->pev0, ctx->pev1));
      ctx->filter_ms += ms; ctx->filter_launches++; ctx->filter_frames += sl.n;
    }
  }
  int maxchunk = 1;
  for (int p = g.first_pass; p < 2; p++) {
    int c = (g.ncx[p] * g.ncy[p] + CELLS_PER_BLOCK - 1) / CELLS_PER_BLOCK;
    if (c > maxchunk) maxchunk = c;
  }
  dim3 gc(maxchunk, 2, sl.n);
  k_cell_count<<<gc, CELLS_PER_BLOCK, 0, st>>>(g, ctx->frames_d, sl);
  CU_LAUNCH_CHECK(ctx);
  k_emit_records<<<gc, CELLS_PER_BLOCK, 0, st>>>(g, ctx->frames_d, sl);
  CU_LAUNCH_CHECK(ctx);
  dim3 gb(1, 2, sl.n);
  k_build_bins<<<gb, 1024, 0, st>>>(g, ctx->frames_d, sl);
  CU_LAUNCH_CHECK(ctx);
  if (ctx->counts_stage) {
    k_gather_counts<<<1, VISO_MAX_BATCH, 0, st>>>(ctx->frames_d, sl, ctx->counts_stage);
    CU_LAUNCH_CHECK(ctx);
  }
  return VISOCU_OK;
}
