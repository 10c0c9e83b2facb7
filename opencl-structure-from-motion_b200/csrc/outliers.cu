// Outlier removal on the device (Matcher::removeOutliers, reference matcher.cpp:1207-1377; SURVEY.md 8f rank 1).
//
// The reference triangulates the current-image positions of all matches (Triangle, "zQB") and keeps a match if at
// least four of its triangle edges agree in flow / disparity.  The Delaunay triangulation of pixel coordinates is full
// of co-circular point sets, so WHICH triangulation comes out is a property of the algorithm: divide and conquer with
// alternating cuts and Triangle's tie-breaking.  host/delaunay.cpp restates that algorithm with exact integer
// predicates; this file runs the same algorithm on the GPU, one CTA per match list, everything in shared memory:
//   1. bitonic sort of (x, y) keys, duplicate detection, second sort for the (y, x) order;
//   2. the partition tree (halves by rank, alternating axes) level by level with block-wide stable partitions;
//   3. the divide-and-conquer build bottom-up: all subtrees of one depth are merged concurrently, one thread per
//      merge, on a 16-bit quad-edge structure with per-subtree free lists; the top levels are single threads walking
//      the seam at shared-memory latency while the other CTAs of the batch keep the SMs busy;
//   4. support vote per triangle edge with shared-memory atomics, order-preserving compaction of the survivors.
// Duplicate positions (Triangle triangulates one point per position, the one its randomised quicksort leaves first) are
// resolved before the kernel runs by replaying that sort on the host (ro_resolve_duplicates below); the kernel gets one
// flag per match.  A list that does not fit (more than about 5700 points in 227 KB), has coordinates above 8191 (the
// 32-bit predicates), fewer than four distinct positions, or trips an internal guard is handed back unchanged with a
// non-zero status, and the host runs the identical algorithm (host/delaunay.cpp) on it.
#include "visocu_internal.cuh"
#include "outliers.cuh"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <type_traits>
#include <utility>
#include <vector>

namespace {

// Threads per CTA: a template parameter of the kernel.  1024 threads of 64 registers own every register of their SM: the
// shortest chain for one list (sorts, partitions and the lower merge levels are block-wide), but no other kernel can use
// the SM while one lane walks the seams of the top merges.  Batched launches therefore run with fewer threads per list
// (visocu_launch_remove_outliers) and leave the rest of the SM to the kernels of the other streams.
constexpr int NIL = 0xFFFF;
constexpr uint16_t DEAD = 0xFFFF;

__host__ __device__ inline int ro_edge_capacity(int n) { return (int)(3.04f * (float)n) + 64; }
__host__ __device__ inline size_t ro_smem_bytes(int n) {
  return (((size_t)12 * ro_edge_capacity(n) + 15) & ~(size_t)15) + (size_t)4 * n + 16;
}

struct Mesh {
  // per half-edge: next / previous around the origin (counter-clockwise), origin vertex.  Three separate arrays that never
  // alias: with __restrict__ the compiler may hoist the loads of one above the stores to another
  uint16_t* __restrict__ nx; uint16_t* __restrict__ pv; uint16_t* __restrict__ og;
  const uint32_t* __restrict__ pt;   // x | y << 16 per vertex
  int* bump; int ecap; volatile int* fail;
  int guard;                   // remaining loop iterations of this thread before it gives up

  __device__ __forceinline__ int org(int e) const { return og[e]; }
  __device__ __forceinline__ int dest(int e) const { return og[e ^ 1]; }
  __device__ __forceinline__ int onext(int e) const { return nx[e]; }
  __device__ __forceinline__ int oprev(int e) const { return pv[e]; }
  __device__ __forceinline__ int lnext(int e) const { return pv[e ^ 1]; }
  __device__ __forceinline__ int rprev(int e) const { return nx[e ^ 1]; }
  __device__ __forceinline__ int px(int v) const { return (int)(pt[v] & 0xFFFFu); }
  __device__ __forceinline__ int py(int v) const { return (int)(pt[v] >> 16); }
  __device__ __forceinline__ bool tick() { return --guard >= 0; }    // false once this thread's loop budget is used up
  // Predicates in 32-bit arithmetic with 64-bit products only where needed: exact for coordinates below 8192 (checked
  // when the keys are built; larger images go to the host).  > 0 iff a, b, c make a left turn
  __device__ __forceinline__ int ccw(int a, int b, int c) const { return ccw_pts(pt[a], pt[b], pt[c]); }
  // > 0 iff d lies strictly inside the circle through a, b, c (counter-clockwise)
  __device__ __forceinline__ long long incircle(int a, int b, int c, int d) const { return incircle_pts(pt[a], pt[b], pt[c], pt[d]); }
  static __device__ __forceinline__ int ccw_pts(uint32_t A, uint32_t B, uint32_t C) {
    const int cx = (int)(C & 0xFFFF), cy = (int)(C >> 16);
    const int ax = (int)(A & 0xFFFF) - cx, ay = (int)(A >> 16) - cy;
    const int bx = (int)(B & 0xFFFF) - cx, by = (int)(B >> 16) - cy;
    return ax * by - ay * bx;                                        // |.| < 2^27
  }
  static __device__ __forceinline__ long long incircle_pts(uint32_t A, uint32_t B, uint32_t C, uint32_t D) {
    const int dx = (int)(D & 0xFFFF), dy = (int)(D >> 16);
    const int adx = (int)(A & 0xFFFF) - dx, ady = (int)(A >> 16) - dy;
    const int bdx = (int)(B & 0xFFFF) - dx, bdy = (int)(B >> 16) - dy;
    const int cdx = (int)(C & 0xFFFF) - dx, cdy = (int)(C >> 16) - dy;
    const int al = adx * adx + ady * ady, bl = bdx * bdx + bdy * bdy, cl = cdx * cdx + cdy * cdy;     // < 2^27
    return (long long)al * (bdx * cdy - cdx * bdy) + (long long)bl * (cdx * ady - adx * cdy) + (long long)cl * (adx * bdy - bdx * ady);
  }
};

// free edges of a subtree: singly linked through nx[] of the even half-edge
struct FreeList { int head, tail; };

// W (here and below): the whole warp runs the function on one subtree, every lane with the same arguments and the same
// loads and stores (same addresses, same values), so that merge() can spread the geometric tests of a step over lanes.
// Only the edge counter must be bumped once.
template <bool W>
__device__ __forceinline__ int make_edge(Mesh& m, FreeList& fl, int a, int b) {
  int e;
  if (fl.head != NIL) {
    e = fl.head;
    fl.head = (e == fl.tail) ? NIL : m.nx[e];
  } else {
    int k = 0;
    if (!W || (threadIdx.x & 31) == 0) k = atomicAdd(m.bump, 1);
    if (W) k = __shfl_sync(0xFFFFFFFFu, k, 0);
    if (k >= m.ecap) { *m.fail = 1; e = 0; } else e = 2 * k;
  }
  m.nx[e] = (uint16_t)e; m.pv[e] = (uint16_t)e; m.og[e] = (uint16_t)a;
  m.nx[e + 1] = (uint16_t)(e + 1); m.pv[e + 1] = (uint16_t)(e + 1); m.og[e + 1] = (uint16_t)b;
  return e;
}
// put the isolated half-edge e right after x in the ring around x's origin
__device__ __forceinline__ void insert_after(Mesh& m, int x, int e) {
  const int n = m.nx[x];
  m.nx[e] = (uint16_t)n; m.pv[e] = (uint16_t)x;
  m.pv[n] = (uint16_t)e; m.nx[x] = (uint16_t)e;
}
__device__ __forceinline__ void unlink(Mesh& m, int e) {
  const int n = m.nx[e], p = m.pv[e];
  m.nx[p] = (uint16_t)n; m.pv[n] = (uint16_t)p;
}
// new edge from dest(a) to org(b) so that a, the new edge and b share their left face
template <bool W>
__device__ __forceinline__ int connect(Mesh& m, FreeList& fl, int a, int b) {
  const int e = make_edge<W>(m, fl, m.dest(a), m.org(b));
  insert_after(m, m.lnext(a), e);
  insert_after(m, b, e ^ 1);
  return e;
}
__device__ __forceinline__ void remove_edge(Mesh& m, FreeList& fl, int e) {
  unlink(m, e); unlink(m, e ^ 1);
  e &= ~1;
  m.og[e] = DEAD; m.og[e + 1] = DEAD;
  if (fl.head == NIL) { fl.head = fl.tail = e; } else { m.nx[e] = (uint16_t)fl.head; fl.head = e; }
}

struct Handles { int ldo, rdo; };   // ccw hull edge out of the leftmost vertex, cw hull edge out of the rightmost

// Merge of two triangulations separated by a vertical (axis 0) or horizontal (axis 1) line; the same steps, tests and
// tie-breaking as merge() in host/delaunay.cpp.
//
// A step of the seam walk is a chain of dependent shared-memory loads followed by up to four orientation and three
// in-circle tests on six points, then the stores of the new edge: a few hundred dependent instructions of one thread.  At
// the top levels of the tree, where there are no more subtrees than warps, the warp owns the merge (W): all lanes chase
// the pointers together (broadcast loads), lanes 0-4 evaluate one test each on points handed out by shuffles, and ballots
// bring the outcomes back.  The candidate loops that follow a deletion stay sequential (most steps delete nothing).
template <bool W>
__device__ Handles merge(Mesh& m, FreeList& fl, Handles L, Handles R, int axis) {
  int ldo = L.ldo, ldi = L.rdo, rdi = R.ldo, rdo = R.rdo;
  if (axis == 1) {
    while (m.py(m.dest(ldo)) < m.py(m.org(ldo)) && m.tick()) ldo = m.rprev(ldo);
    while (m.py(m.dest(m.onext(ldi))) > m.py(m.org(ldi)) && m.tick()) ldi = m.onext(ldi) ^ 1;
    while (m.py(m.dest(rdi)) < m.py(m.org(rdi)) && m.tick()) rdi = m.rprev(rdi);
    while (m.py(m.dest(m.onext(rdo))) > m.py(m.org(rdo)) && m.tick()) rdo = m.onext(rdo) ^ 1;
  }
  bool changed;
  do {
    changed = false;
    if (m.ccw(m.org(ldi), m.dest(ldi), m.org(rdi)) > 0) { ldi = m.lnext(ldi); changed = true; }
    if (m.ccw(m.dest(rdi), m.org(rdi), m.org(ldi)) > 0) { rdi = m.rprev(rdi); changed = true; }
  } while (changed && m.tick());
  int basel = connect<W>(m, fl, rdi ^ 1, ldi);
  if (m.org(ldi) == m.org(ldo)) ldo = basel ^ 1;
  if (m.org(rdi) == m.org(rdo)) rdo = basel;
  while (m.tick()) {
    const int lowerright = m.org(basel), lowerleft = m.dest(basel);
    int lcand = m.onext(basel ^ 1), rcand = m.oprev(basel);
    int upperleft = m.dest(lcand), upperright = m.dest(rcand);
    // The first test of the left and of the right candidate loop read disjoint parts of the mesh (the left loop only
    // touches edges of the left triangulation and the ring of lowerleft, the right loop the mirror image), and most
    // steps delete nothing.  Both first tests are therefore evaluated up front, before any store, so that their load
    // chains overlap; the loops below continue from the second candidate on.
    const int lnx0 = m.onext(lcand), rnx0 = m.oprev(rcand);
    const int lapex0 = m.dest(lnx0), rapex0 = m.dest(rnx0);
    bool leftfinished, rightfinished, ldel0, rdel0, right_first = false;
    if (W) {
      // points 0..5 = lowerleft, lowerright, upperleft, upperright, left apex, right apex, one per lane; the tables hold,
      // per lane (4 bits each), which of them are the arguments of its tests:
      //   lane 0: ccw(UL, LL, LR)   lane 1: ccw(UR, LL, LR)   lane 2: ccw(LL, UL, LA), incircle(LL, LR, UL, LA)
      //   lane 3: ccw(LR, RA, UR), incircle(LL, LR, UR, RA)   lane 4: incircle(UL, LL, LR, UR)
      const int lane = threadIdx.x & 31;
      int myv = rapex0;
      myv = lane == 4 ? lapex0 : myv; myv = lane == 3 ? upperright : myv; myv = lane == 2 ? upperleft : myv;
      myv = lane == 1 ? lowerright : myv; myv = lane == 0 ? lowerleft : myv;
      const uint32_t myp = m.pt[myv];
      const int sh = 4 * min(lane, 7);
#define RO_PICK(table) __shfl_sync(0xFFFFFFFFu, myp, (int)(((table) >> sh) & 7u))
      const uint32_t P = RO_PICK(0x01032u), Q = RO_PICK(0x05200u), R = RO_PICK(0x03411u);
      const uint32_t A = RO_PICK(0x20000u), B = RO_PICK(0x01100u), C = RO_PICK(0x13200u), D = RO_PICK(0x35400u);
#undef RO_PICK
      const unsigned cpos = __ballot_sync(0xFFFFFFFFu, Mesh::ccw_pts(P, Q, R) > 0);
      const unsigned ipos = __ballot_sync(0xFFFFFFFFu, Mesh::incircle_pts(A, B, C, D) > 0);
      leftfinished = !(cpos & 1u); rightfinished = !(cpos & 2u);
      ldel0 = !leftfinished && lnx0 != (basel ^ 1) && (cpos & 4u) && (ipos & 4u);
      rdel0 = !rightfinished && rnx0 != basel && (cpos & 8u) && (ipos & 8u);
      right_first = (ipos & 16u) != 0;                 // valid while neither candidate changes
    } else {
      leftfinished = m.ccw(upperleft, lowerleft, lowerright) <= 0;
      rightfinished = m.ccw(upperright, lowerleft, lowerright) <= 0;
      ldel0 = !leftfinished && lnx0 != (basel ^ 1) && m.ccw(lowerleft, upperleft, lapex0) > 0 &&
              m.incircle(lowerleft, lowerright, upperleft, lapex0) > 0;
      rdel0 = !rightfinished && rnx0 != basel && m.ccw(lowerright, rapex0, upperright) > 0 &&
              m.incircle(lowerleft, lowerright, upperright, rapex0) > 0;
    }
    if (leftfinished && rightfinished) break;
    if (ldel0) {
      remove_edge(m, fl, lcand);
      lcand = lnx0; upperleft = lapex0;
      while (m.tick()) {
        const int nx = m.onext(lcand);
        if (nx == (basel ^ 1)) break;
        const int apex = m.dest(nx);
        if (m.ccw(lowerleft, upperleft, apex) <= 0) break;
        if (m.incircle(lowerleft, lowerright, upperleft, apex) <= 0) break;
        remove_edge(m, fl, lcand);
        lcand = nx; upperleft = apex;
      }
    }
    if (rdel0) {
      remove_edge(m, fl, rcand);
      rcand = rnx0; upperright = rapex0;
      while (m.tick()) {
        const int nx = m.oprev(rcand);
        if (nx == basel) break;
        const int apex = m.dest(nx);
        if (m.ccw(lowerright, apex, upperright) <= 0) break;
        if (m.incircle(lowerleft, lowerright, upperright, apex) <= 0) break;
        remove_edge(m, fl, rcand);
        rcand = nx; upperright = apex;
      }
    }
    bool right = leftfinished;
    if (!leftfinished && !rightfinished)
      right = (W && !ldel0 && !rdel0) ? right_first : m.incircle(upperleft, lowerleft, lowerright, upperright) > 0;
    if (right) basel = connect<W>(m, fl, rcand, basel ^ 1);
    else basel = connect<W>(m, fl, basel ^ 1, lcand ^ 1);
    if (W) __syncwarp();
  }
  if (axis == 1) {
    while (m.px(m.dest(m.oprev(ldo))) < m.px(m.org(ldo)) && m.tick()) ldo = m.oprev(ldo) ^ 1;
    while (m.px(m.dest(rdo)) > m.px(m.org(rdo)) && m.tick()) rdo = m.lnext(rdo);
  }
  return Handles{ldo, rdo};
}

// two or three vertices, consecutive numbers starting at v, sorted by x
template <bool W>
__device__ Handles leaf(Mesh& m, FreeList& fl, int v, int n) {
  if (n == 2) {
    const int a = make_edge<W>(m, fl, v, v + 1);
    return Handles{a, a ^ 1};
  }
  const int a = make_edge<W>(m, fl, v, v + 1);
  const int b = make_edge<W>(m, fl, v + 1, v + 2);
  insert_after(m, b, a ^ 1);
  const int area = m.ccw(v, v + 1, v + 2);
  if (area == 0) return Handles{a, b ^ 1};
  const int c = connect<W>(m, fl, b, a);
  if (area > 0) return Handles{a, b ^ 1};
  return Handles{c ^ 1, c};
}

// exclusive prefix sum over the block of one value per thread; total returned to every thread
template <int RO_THREADS>
__device__ __forceinline__ int block_scan(int v, int* s_warp, int& total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
  __syncthreads();                                   // s_warp may still be read from the previous call
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  int base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < RO_THREADS / 32; w++) { const int s = s_warp[w]; if (w < wid) base += s; tot += s; }
  total = tot;
  return base + incl - v;
}

__device__ __forceinline__ bool edge_agrees(const visocu_pmatch& a, const visocu_pmatch& b, int method, float flow_tol, float disp_tol) {
  // float arithmetic, operation by operation as matcher.cpp:1267-1349 (no contraction possible: no multiplications)
  if (method == 0)
    return __fadd_rn(fabsf(__fsub_rn(__fsub_rn(a.u1c, a.u1p), __fsub_rn(b.u1c, b.u1p))),
                     fabsf(__fsub_rn(__fsub_rn(a.v1c, a.v1p), __fsub_rn(b.v1c, b.v1p)))) < flow_tol;
  if (method == 1) return fabsf(__fsub_rn(__fsub_rn(a.u1c, a.u2c), __fsub_rn(b.u1c, b.u2c))) < disp_tol;
  return fabsf(__fsub_rn(__fsub_rn(a.u1p, a.u2p), __fsub_rn(b.u1p, b.u2p))) < disp_tol &&
         __fadd_rn(fabsf(__fsub_rn(__fsub_rn(a.u1c, a.u1p), __fsub_rn(b.u1c, b.u1p))),
                   fabsf(__fsub_rn(__fsub_rn(a.v1c, a.v1p), __fsub_rn(b.v1c, b.v1p)))) < flow_tol;
}

// copy 48-byte records src[list[i]] -> dst[i], 12 lanes per record
template <int RO_THREADS>
__device__ __forceinline__ void copy_records(visocu_pmatch* dst, const visocu_pmatch* src, const int32_t* list, int n) {
  const int32_t* s = (const int32_t*)src;
  int32_t* d = (int32_t*)dst;
  for (int idx = threadIdx.x; idx < 12 * n; idx += RO_THREADS) {
    const int i = idx / 12, w = idx - 12 * i;
    d[idx] = s[12 * (size_t)list[i] + w];
  }
}

template <int RO_THREADS>
__global__ void __launch_bounds__(RO_THREADS, 1024 / RO_THREADS)
k_remove_outliers(const RoJob* __restrict__ jobs, int method, float flow_tol, float disp_tol, int smem_bytes, int warp_merges) {
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ int s_warp[RO_THREADS / 32];
  __shared__ int s_bump, s_fail, s_flag, s_more;
  const RoJob J = jobs[blockIdx.x];
  const int tid = threadIdx.x;
  auto now = []() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; };
  const unsigned long long t_start = now();
  const int n_in = *J.n_in;
  int32_t* src = J.idx;                              // global scratch: list position -> record index (after the keep flags)

  // ---- 0. records that survived the sub-pixel refinement (order preserved)
  const bool pts_mode = J.pts_in != nullptr;         // vertices given as points: every one takes part
  const int axis0 = J.axis0;
  int n = 0;
  if (pts_mode) {
    n = n_in;
  } else {
    const int per = (n_in + RO_THREADS - 1) / RO_THREADS;
    const int i0 = min(tid * per, n_in), i1 = min(i0 + per, n_in);
    int cnt = 0;
    for (int i = i0; i < i1; i++) cnt += (!J.keep_in || J.keep_in[i]) ? 1 : 0;
    int total;
    int off = block_scan<RO_THREADS>(cnt, s_warp, total);
    n = total;
    for (int i = i0; i < i1; i++) if (!J.keep_in || J.keep_in[i]) src[off++] = i;
  }
  if (tid == 0) { s_bump = 0; s_fail = 0; s_flag = 0; }
  __syncthreads();

  // capacity of this launch's shared memory: 12 E bytes of half-edges and 4 n of points.  A triangulation of n points
  // has fewer than 3 n edges and the free lists recycle every deleted one, so E = 3.04 n + 64 is enough in practice
  // (measured peak 2.98 n); running out trips the guard and hands the list to the host.
  const int ecap = ro_edge_capacity(n);
  const size_t need = ro_smem_bytes(n);
  const int nl = n;                                  // list length; n becomes the number of mesh vertices (distinct positions)
  if (n <= 3 || n > 0x7FF0 || need > (size_t)smem_bytes) {
    // nothing to vote on (matcher.cpp:1210-1211), or too large for the device path: hand the list over unchanged
    if (!pts_mode) copy_records<RO_THREADS>(J.out, J.in, src, n);
    if (tid == 0) { J.result[0] = n; J.result[1] = (n <= 3 && !pts_mode) ? 0 : 1; J.result[2] = 0; J.result[3] = n; }
    return;
  }

  // ---- shared-memory layout
  uint16_t* he_nx = (uint16_t*)smem;
  uint16_t* he_pv = he_nx + 2 * ecap;
  uint16_t* he_og = he_pv + 2 * ecap;
  uint32_t* pts = (uint32_t*)(smem + (((size_t)12 * ecap + 15) & ~(size_t)15));
  // hull handles and free lists of the subtrees (indexed by first vertex / 2) are touched twice per merge: global scratch
  uint16_t* h_l = J.hnd;
  uint16_t* h_r = h_l + (n / 2 + 2);
  uint16_t* f_h = h_r + (n / 2 + 2);
  uint16_t* f_t = f_h + (n / 2 + 2);
  // temporaries of steps 1 and 2 live in the half-edge area
  int npad = 1;
  while (npad < n) npad <<= 1;
  unsigned long long* keys = (unsigned long long*)smem;                    // npad keys
  uint16_t* ax = (uint16_t*)(keys + npad);                                  // by x-rank: x, y, list position
  uint16_t* ay = ax + n;
  uint16_t* ain = ay + n;
  uint16_t* la = ain + n;                                                   // three list buffers (x order, y order, spare)
  uint16_t* lb = la + n;
  uint16_t* lc = lb + n;
  uint16_t* nlo = lc + n;                                                   // partition node of every list position
  uint16_t* nsz = nlo + n;
  uint16_t* pre = nsz + n;                                                  // prefix sums of the side bits
  uint8_t* side = (uint8_t*)(pre + n + 1);
  // (8 npad + 19 n + 2 <= 12 ecap because npad < 2 n)

  // Bitonic merge sort of keys[0, m), ascending.  Every compare-exchange puts the smaller key at the lower index (the
  // first step of each merge pairs i with its mirror image in the block), so the elements beyond m can stay virtual
  // "+infinity" padding: pairs that reach past m are skipped, and the work follows m, not the next power of two.
  auto bitonic = [&](int m) {
    for (int k = 2; k <= npad; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int t = tid; t < (npad >> 1); t += RO_THREADS) {
          const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));              // element with bit j clear
          const int p = (j == (k >> 1)) ? (i ^ (k - 1)) : (i | j);
          if (p < m) {
            const unsigned long long a = keys[i], b = keys[p];
            if (a > b) { keys[i] = b; keys[p] = a; }
          }
        }
        __syncthreads();
      }
  };

  // ---- 1. order by (x, y); positions are the truncated coordinates in the current left image (matcher.cpp:1230-1233)
  // (records the duplicate resolution excluded get the padding key: they are no vertices, collect no votes and drop out)
  if (tid == 0) s_more = 0;
  for (int i = tid; i < npad; i += RO_THREADS) {
    unsigned long long key = ~0ull;
    if (i < nl && (pts_mode || !J.rep || J.rep[src[i]])) {
      int x, y;
      if (pts_mode) { const uint32_t p = J.pts_in[i]; x = (int)(p & 0xFFFFu); y = (int)(p >> 16); }
      else { const visocu_pmatch& r = J.in[src[i]]; x = (int)r.u1c; y = (int)r.v1c; }
      if (x < 0 || y < 0 || x > 8191 || y > 8191) s_fail = 1;        // range of the 32-bit predicates
      key = ((unsigned long long)(unsigned)x << 40) | ((unsigned long long)(unsigned)y << 16) | (unsigned)i;
    }
    keys[i] = key;
  }
  __syncthreads();
  bitonic(nl);
  for (int i = tid; i < npad; i += RO_THREADS)
    if (keys[i] != ~0ull && (i + 1 == npad || keys[i + 1] == ~0ull)) s_more = i + 1;     // number of vertices
  __syncthreads();
  for (int i = tid; i < s_more; i += RO_THREADS) {
    const unsigned long long key = keys[i];
    if (i > 0 && (keys[i - 1] >> 16) == (key >> 16)) s_flag = 1;           // two vertices on one pixel
    ax[i] = (uint16_t)(key >> 40); ay[i] = (uint16_t)(key >> 16);
    ain[i] = (uint16_t)key;
  }
  __syncthreads();
  if (s_fail) {
    if (!pts_mode) copy_records<RO_THREADS>(J.out, J.in, src, nl);
    if (tid == 0) { J.result[0] = nl; J.result[1] = 1; J.result[2] = 0; J.result[3] = nl; }
    return;
  }
  if (s_flag) {
    // Two vertices on one pixel: the caller did not resolve the duplicates (ro_resolve_duplicates) - Triangle's choice
    // among them depends on its randomised quicksort, which is replayed on the host, not here.
    if (!pts_mode) copy_records<RO_THREADS>(J.out, J.in, src, nl);
    if (tid == 0) { J.result[0] = nl; J.result[1] = 2; J.result[2] = 0; J.result[3] = nl; }
    return;
  }
  n = s_more;                                        // number of vertices (records that take part)
  if (n <= 3) {
    if (!pts_mode) copy_records<RO_THREADS>(J.out, J.in, src, nl);
    if (tid == 0) { J.result[0] = nl; J.result[1] = 3; J.result[2] = 0; J.result[3] = nl; }
    return;
  }
  for (int i = tid; i < npad; i += RO_THREADS)
    keys[i] = i < n ? ((unsigned long long)ay[i] << 40) | ((unsigned long long)ax[i] << 16) | (unsigned)i : ~0ull;
  __syncthreads();
  bitonic(n);
  const unsigned long long t_sorted = now();
  uint16_t* xl = la; uint16_t* yl = lb; uint16_t* spare = lc;
  for (int i = tid; i < n; i += RO_THREADS) { xl[i] = (uint16_t)i; yl[i] = (uint16_t)keys[i]; nlo[i] = 0; nsz[i] = (uint16_t)n; }
  __syncthreads();

  // ---- 2. partition tree: halves by rank along the node's axis, the other list distributed stably
  int depth = 0;
  {
    const int per = (n + RO_THREADS - 1) / RO_THREADS;
    const int i0 = min(tid * per, n), i1 = min(i0 + per, n);
    for (;; depth++) {
      const int axis = (depth + axis0) & 1;
      uint16_t* from = axis == 0 ? xl : yl;
      uint16_t* other = axis == 0 ? yl : xl;
      if (tid == 0) s_more = 0;
      for (int i = i0; i < i1; i++) {
        const int sz = nsz[i];
        if (sz > 3) side[from[i]] = (uint8_t)((i - nlo[i]) >= (sz >> 1));
      }
      __syncthreads();
      int cnt = 0;
      for (int i = i0; i < i1; i++) cnt += (nsz[i] > 3) ? side[other[i]] : 0;
      int total;
      int run = block_scan<RO_THREADS>(cnt, s_warp, total);
      for (int i = i0; i < i1; i++) { pre[i] = (uint16_t)run; run += (nsz[i] > 3) ? side[other[i]] : 0; }
      if (i1 == n && i0 < n) pre[n] = (uint16_t)run;
      __syncthreads();
      bool more = false;
      for (int i = i0; i < i1; i++) {
        const int sz = nsz[i], lo = nlo[i];
        const int id = other[i];
        if (sz > 3) {
          const int div = sz >> 1;
          const int ones = pre[i] - pre[lo];
          const int s = side[id];
          spare[s ? lo + div + ones : lo + (i - lo - ones)] = (uint16_t)id;
        } else {
          spare[i] = (uint16_t)id;
        }
      }
      __syncthreads();                               // every pre[lo] has been read
      for (int i = i0; i < i1; i++) {
        const int sz = nsz[i], lo = nlo[i];
        if (sz > 3) {
          const int div = sz >> 1;
          if (i - lo < div) { nsz[i] = (uint16_t)div; } else { nlo[i] = (uint16_t)(lo + div); nsz[i] = (uint16_t)(sz - div); }
          if (nsz[i] > 3) more = true;
        }
      }
      if (more) s_more = 1;
      // the distributed list replaces `other`
      if (axis == 0) { uint16_t* t = yl; yl = spare; spare = t; } else { uint16_t* t = xl; xl = spare; spare = t; }
      __syncthreads();
      if (!s_more) break;
      __syncthreads();                               // s_more is reset at the top of the next round
    }
  }
  const int maxdepth = depth + 1;                    // nodes of depth maxdepth are all leaves
  // vertices renumbered in partition order: every subtree owns a contiguous range.  The point array lies behind the
  // half-edge area, which still holds the temporaries read here.
  for (int i = tid; i < n; i += RO_THREADS) {
    const int id = xl[i];
    pts[i] = (uint32_t)ax[id] | ((uint32_t)ay[id] << 16);
    J.vert[i] = ain[id];                             // vertex -> list position
  }
  for (int i = tid; i < n / 2 + 2; i += RO_THREADS) { f_h[i] = NIL; f_t[i] = NIL; }
  __syncthreads();

  // ---- 3. build, deepest level first; one thread per subtree of the level
  const unsigned long long t_part = now();
  Mesh m;
  m.nx = he_nx; m.pv = he_pv; m.og = he_og; m.pt = pts; m.bump = &s_bump; m.ecap = ecap; m.fail = &s_fail;
  m.guard = 64 * ecap;
  unsigned long long t_level = now();
  for (int d = maxdepth; d >= 0; d--) {
    // one subtree of the level: its vertex range from the index, leaf or merge, handles and free list stored
    auto subtree = [&](int j, auto warp_wide) {
      constexpr bool W = decltype(warp_wide)::value;
      int lo = 0, sz = n;
      for (int t = d - 1; t >= 0; t--) {
        if (sz <= 3) return;                         // the node does not exist: an ancestor is a leaf
        const int div = sz >> 1;
        if ((j >> t) & 1) { lo += div; sz -= div; } else { sz = div; }
      }
      FreeList fl{NIL, NIL};
      Handles h;
      if (sz <= 3) {
        h = leaf<W>(m, fl, lo, sz);
      } else {
        const int div = sz >> 1;
        const int sl = lo >> 1, sr = (lo + div) >> 1;
        fl.head = f_h[sl]; fl.tail = f_t[sl];
        if (f_h[sr] != NIL) {
          if (fl.head == NIL) { fl.head = f_h[sr]; fl.tail = f_t[sr]; }
          else { m.nx[fl.tail] = f_h[sr]; fl.tail = f_t[sr]; }
        }
        h = merge<W>(m, fl, Handles{h_l[sl], h_r[sl]}, Handles{h_l[sr], h_r[sr]}, (d + axis0) & 1);
      }
      if (m.guard < 0) s_fail = 1;
      if (!W || (tid & 31) == 0) {
        h_l[lo >> 1] = (uint16_t)h.ldo; h_r[lo >> 1] = (uint16_t)h.rdo;
        f_h[lo >> 1] = (uint16_t)fl.head; f_t[lo >> 1] = (uint16_t)fl.tail;
      }
    };
    if (warp_merges && (1 << d) <= RO_THREADS / 32) {
      // no more subtrees than warps: a warp per merge, the tests of a seam step spread over its lanes (merge<true>)
      if ((tid >> 5) < (1 << d)) {
        m.guard = __reduce_min_sync(0xFFFFFFFFu, m.guard);            // one loop budget for the warp: uniform control flow
        subtree(tid >> 5, std::true_type());
      }
    } else {
      // Threads of a warp that run different merges take turns (the merges diverge completely), so the subtrees of a
      // level are dealt to the warps first: 32 or fewer subtrees run on 32 different warps, one lane each.
      for (int j = (tid & 31) * (RO_THREADS / 32) + (tid >> 5); j < (1 << d); j += RO_THREADS) subtree(j, std::false_type());
    }
    __syncthreads();
    if (tid == 0 && d < 7) { const unsigned long long t = now(); J.result[9 + d] = (int32_t)(t - t_level); t_level = t; }
    else if (tid == 0) t_level = now();
    if (s_fail) break;
  }
  if (s_fail) {
    if (!pts_mode) copy_records<RO_THREADS>(J.out, J.in, src, nl);
    if (tid == 0) { J.result[0] = nl; J.result[1] = 3; J.result[2] = s_bump; J.result[3] = nl; }
    return;
  }

  if (J.mesh_out) {
    // triangulation only: the mesh in the caller's numbering, deleted edges and the unused tail marked, the hull handles
    const int nh = 2 * min(s_bump, ecap), hb = J.he_base, vb = J.v_base;
    for (int e = tid; e < 2 * ecap; e += RO_THREADS) {
      int4 rec = make_int4(hb + e, hb + e, -1, 0);
      if (e < nh) {
        const int o = he_og[e];
        if (o != DEAD) rec = make_int4(hb + he_nx[e], hb + he_pv[e], vb + o, (int)pts[o]);
      }
      J.mesh_out[e] = rec;
    }
    if (tid == 0) {
      J.result[0] = n; J.result[1] = 0; J.result[2] = s_bump; J.result[3] = nl; J.result[4] = hb + h_l[0]; J.result[5] = hb + h_r[0];
    }
    return;
  }

  // ---- 4. half-edges of the unbounded face, support vote, compaction
  const unsigned long long t_built = now();
  if (tid == 0) {
    const int start = h_r[0];
    int e = start, guard = 4 * ecap;
    do { he_og[e] |= 0x8000; e = m.lnext(e); } while (e != start && --guard > 0);
    if (guard <= 0) s_fail = 1;
  }
  __syncthreads();
  if (s_fail) {
    if (!pts_mode) copy_records<RO_THREADS>(J.out, J.in, src, nl);
    if (tid == 0) { J.result[0] = nl; J.result[1] = 3; J.result[2] = s_bump; J.result[3] = nl; }
    return;
  }
  // The ring pointers of the mesh are no longer needed.  Their arrays now hold, per list position, the vote counter and
  // the quantities the vote compares (flow / disparity of the match, computed once with the reference's float
  // operations, matcher.cpp:1267-1349), and per vertex its list position: the vote itself touches shared memory only.
  unsigned int* support = (unsigned int*)he_nx;                       // nl words
  float* q_d = (float*)he_nx + nl;                                    // disparity (methods 1 and 2), nl words <= rest of he_nx
  float* q_u = (float*)he_pv;                                         // flow u, flow v (methods 0 and 2)
  float* q_v = q_u + nl;
  uint16_t* vpos = (uint16_t*)(q_v + nl);                             // 8 nl + 2 n bytes <= 12 ecap / ... of he_pv
  const bool vote_in_smem = (size_t)8 * nl <= (size_t)4 * ecap && (size_t)8 * nl + (size_t)2 * n <= (size_t)4 * ecap;
  for (int i = tid; i < nl; i += RO_THREADS) {
    support[i] = 0;
    if (vote_in_smem) {
      const visocu_pmatch& r = J.in[src[i]];
      q_u[i] = __fsub_rn(r.u1c, r.u1p); q_v[i] = __fsub_rn(r.v1c, r.v1p);
      q_d[i] = method == 1 ? __fsub_rn(r.u1c, r.u2c) : __fsub_rn(r.u1p, r.u2p);
    }
  }
  if (vote_in_smem)
    for (int i = tid; i < n; i += RO_THREADS) vpos[i] = (uint16_t)J.vert[i];
  __syncthreads();
  const int nedge = min(s_bump, ecap);
  for (int k = tid; k < nedge; k += RO_THREADS) {
    const int o0 = he_og[2 * k], o1 = he_og[2 * k + 1];
    if (o0 == DEAD || o1 == DEAD) continue;
    // an edge with a triangle on both sides votes twice (the reference votes per triangle, matcher.cpp:1259-1362)
    const int t = ((o0 & 0x8000) ? 0 : 1) + ((o1 & 0x8000) ? 0 : 1);
    if (t == 0) continue;
    int pa, pb;
    bool agree;
    if (vote_in_smem) {
      pa = vpos[o0 & 0x7FFF]; pb = vpos[o1 & 0x7FFF];
      const bool flow_ok = __fadd_rn(fabsf(__fsub_rn(q_u[pa], q_u[pb])), fabsf(__fsub_rn(q_v[pa], q_v[pb]))) < flow_tol;
      const bool disp_ok = fabsf(__fsub_rn(q_d[pa], q_d[pb])) < disp_tol;
      agree = method == 0 ? flow_ok : (method == 1 ? disp_ok : (disp_ok && flow_ok));
    } else {
      pa = J.vert[o0 & 0x7FFF]; pb = J.vert[o1 & 0x7FFF];
      agree = edge_agrees(J.in[src[pa]], J.in[src[pb]], method, flow_tol, disp_tol);
    }
    if (agree) {
      atomicAdd(&support[pa], (unsigned)t);
      atomicAdd(&support[pb], (unsigned)t);
    }
  }
  __syncthreads();
  {
    const int per = (nl + RO_THREADS - 1) / RO_THREADS;
    const int i0 = min(tid * per, nl), i1 = min(i0 + per, nl);
    int cnt = 0;
    for (int i = i0; i < i1; i++) cnt += support[i] >= 4u ? 1 : 0;
    int total;
    int off = block_scan<RO_THREADS>(cnt, s_warp, total);
    // compacted index list in place of src (entries only move towards the front, chunk by chunk behind a barrier)
    int32_t* kept = J.vert;                          // the vertex map is no longer needed
    __syncthreads();
    for (int i = i0; i < i1; i++) if (support[i] >= 4u) kept[off++] = src[i];
    __syncthreads();
    copy_records<RO_THREADS>(J.out, J.in, kept, total);
    if (tid == 0) {
      J.result[0] = total; J.result[1] = 0; J.result[2] = s_bump; J.result[3] = nl;
      // phase times in nanoseconds (sort, partition, build, vote + compaction): read by profiles/profile_outliers.py
      const unsigned long long t_end = now();
      J.result[4] = (int32_t)(t_sorted - t_start); J.result[5] = (int32_t)(t_part - t_sorted);
      J.result[6] = (int32_t)(t_built - t_part); J.result[7] = (int32_t)(t_end - t_built);
    }
  }
}

// positions of all records of a list for the host-side duplicate resolution
__global__ void k_outlier_keys(const RoJob* __restrict__ jobs, uint32_t* keys, int stride) {
  const RoJob J = jobs[blockIdx.y];
  const int n = *J.n_in;
  uint32_t* out = keys + (size_t)blockIdx.y * stride;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    uint32_t k = 0xFFFFFFFFu;
    if (!J.keep_in || J.keep_in[i]) {
      const int x = (int)J.in[i].u1c, y = (int)J.in[i].v1c;
      if (x >= 0 && y >= 0 && x <= 0xFFFF && y <= 0xFFFF) k = ((uint32_t)x << 16) | (uint32_t)y;
    }
    out[i] = k;
  }
}

}  // namespace

int visocu_launch_remove_outliers(visocu_ctx* ctx, const RoJob* jobs_dev, int n_jobs, int method, int max_records, cudaStream_t stream) {
  // shared memory for the largest list of the launch, at most the 227 KB a CTA can have
  size_t smem = ro_smem_bytes(max_records);
  const size_t smem_max = 227 * 1024 - 256;          // the kernel also has a few static shared variables
  if (smem > smem_max) smem = smem_max;
  if (smem < 16 * 1024) smem = 16 * 1024;
  {
    static std::mutex mtx;
    static bool done[64] = {false};
    std::lock_guard<std::mutex> lock(mtx);
    if (!done[ctx->device & 63]) {
      CU_TRY(ctx, cudaFuncSetAttribute(k_remove_outliers<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
      CU_TRY(ctx, cudaFuncSetAttribute(k_remove_outliers<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
      CU_TRY(ctx, cudaFuncSetAttribute(k_remove_outliers<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
      done[ctx->device & 63] = true;
    }
  }
  // one or two lists (a stand-alone Matcher): the shortest chain; batches: the smaller footprint
  const int threads = ctx->ro_threads ? ctx->ro_threads : (n_jobs <= 2 ? 1024 : 512);
  const int warp = ctx->ro_warp;
  const float ft = (float)ctx->param.outlier_flow_tolerance, dt = (float)ctx->param.outlier_disp_tolerance;
  if (threads >= 1024) k_remove_outliers<1024><<<n_jobs, 1024, smem, stream>>>(jobs_dev, method, ft, dt, (int)smem, warp);
  else if (threads >= 512) k_remove_outliers<512><<<n_jobs, 512, smem, stream>>>(jobs_dev, method, ft, dt, (int)smem, warp);
  else k_remove_outliers<256><<<n_jobs, 256, smem, stream>>>(jobs_dev, method, ft, dt, (int)smem, warp);
  CU_LAUNCH_CHECK(ctx);
  return VISOCU_OK;
}

extern "C" int visocu_remove_outliers(visocu_ctx* ctx, int32_t n_jobs, int32_t method, visocu_pmatch* const* inout, const int32_t* n,
                                      int32_t* n_out, int32_t* status) {
  if (!ctx) return VISOCU_EINVAL;
  if (!ctx->configured) return visocu_set_error(ctx, VISOCU_ESTATE, "context not configured");
  if (n_jobs <= 0 || !inout || !n || !n_out || !status) return visocu_set_error(ctx, VISOCU_EINVAL, "bad outlier removal arguments");
  if (method < 0 || method > 2) return visocu_set_error(ctx, VISOCU_EINVAL, "method %d not supported", method);
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  std::vector<RoJob> hj(n_jobs);
  std::vector<size_t> o_in(n_jobs), o_out(n_jobs), o_idx(n_jobs), o_vert(n_jobs), o_res(n_jobs), o_hnd(n_jobs), o_rep(n_jobs);
  std::vector<std::vector<uint8_t> > reps(n_jobs);
  size_t off = align_up(sizeof(RoJob) * n_jobs, 256);
  int maxn = 0;
  for (int j = 0; j < n_jobs; j++) {
    if (n[j] < 0) return visocu_set_error(ctx, VISOCU_EINVAL, "job %d has a negative count", j);
    const size_t cnt = (size_t)n[j] + 1;
    if (n[j] > maxn) maxn = n[j];
    o_in[j] = off; off += align_up(cnt * 48, 256);
    o_out[j] = off; off += align_up(cnt * 48, 256);
    o_idx[j] = off; off += align_up(cnt * 4, 256);
    o_vert[j] = off; off += align_up(cnt * 4, 256);
    o_hnd[j] = off; off += align_up((cnt / 2 + 2) * 8, 256);
    o_rep[j] = off; off += align_up(cnt, 256);
    o_res[j] = off; off += 256;
  }
  int rc = visocu_ensure_scratch(ctx, off);
  if (rc) return rc;
  if ((rc = visocu_ensure_pinned(ctx, align_up(sizeof(RoJob) * n_jobs, 256) + (size_t)n_jobs * 64))) return rc;
  uint8_t* sb = (uint8_t*)ctx->scratch;
  uint8_t* pin = (uint8_t*)ctx->pinned;
  for (int j = 0; j < n_jobs; j++) {
    RoJob& J = hj[j];
    J.in = (const visocu_pmatch*)(sb + o_in[j]); J.keep_in = nullptr; J.out = (visocu_pmatch*)(sb + o_out[j]);
    J.result = (int32_t*)(sb + o_res[j]); J.n_in = J.result + 8;   // [9..15]: times of the top merge levels
    J.idx = (int32_t*)(sb + o_idx[j]); J.vert = (int32_t*)(sb + o_vert[j]); J.hnd = (uint16_t*)(sb + o_hnd[j]);
    if (n[j] > 0) CU_COPY(ctx, sb + o_in[j], inout[j], (size_t)n[j] * 48, cudaMemcpyHostToDevice);
    J.rep = nullptr;
    if (n[j] > 3) {
      std::vector<uint32_t> keys((size_t)n[j]);
      for (int i = 0; i < n[j]; i++) {
        const int x = (int)inout[j][i].u1c, y = (int)inout[j][i].v1c;
        keys[i] = (x >= 0 && y >= 0 && x <= 0xFFFF && y <= 0xFFFF) ? ((uint32_t)x << 16) | (uint32_t)y : 0xFFFFFFFFu;
      }
      reps[j].resize((size_t)n[j]);
      if (ro_resolve_duplicates(keys.data(), n[j], reps[j].data())) {
        CU_COPY(ctx, sb + o_rep[j], reps[j].data(), (size_t)n[j], cudaMemcpyHostToDevice);
        J.rep = sb + o_rep[j];
      }
    }
    CU_COPY(ctx, (void*)J.n_in, &n[j], 4, cudaMemcpyHostToDevice);
  }
  memcpy(pin, hj.data(), sizeof(RoJob) * n_jobs);
  CU_COPY(ctx, sb, pin, sizeof(RoJob) * n_jobs, cudaMemcpyHostToDevice);
  if ((rc = visocu_launch_remove_outliers(ctx, (const RoJob*)sb, n_jobs, method, maxn, ctx->stream))) return rc;
  int32_t* pin_res = (int32_t*)(pin + align_up(sizeof(RoJob) * n_jobs, 256));
  for (int j = 0; j < n_jobs; j++) CU_COPY(ctx, pin_res + 16 * j, hj[j].result, 64, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  for (int j = 0; j < n_jobs; j++) {
    n_out[j] = pin_res[16 * j]; status[j] = pin_res[16 * j + 1];
    if (getenv("VISOCU_RO_STATS") && j == 0)
      fprintf(stderr, "[outliers] n=%d kept=%d status=%d edges=%d (%.2f n) ns: sort %d partition %d build %d vote %d\n", n[j], pin_res[0], pin_res[1],
              pin_res[2], n[j] ? (double)pin_res[2] / n[j] : 0.0, pin_res[4], pin_res[5], pin_res[6], pin_res[7]),
      fprintf(stderr, "[outliers] merge levels 0..6 (ns): %d %d %d %d %d %d %d\n", pin_res[9], pin_res[10], pin_res[11], pin_res[12], pin_res[13], pin_res[14], pin_res[15]);
    if (status[j] == 0 && n_out[j] > 0) CU_COPY(ctx, inout[j], hj[j].out, (size_t)n_out[j] * 48, cudaMemcpyDeviceToHost);
  }
  CU_TRY(ctx, visocu_stream_wait(ctx));
  return VISOCU_OK;
}

extern "C" int32_t visocu_delaunay_edge_capacity(int32_t n_vertices) { return n_vertices > 0 ? ro_edge_capacity(n_vertices) : 0; }

// Nodes of a larger divide-and-conquer Delaunay triangulation built on the device, one CTA each (see include/visocu.h)
extern "C" int visocu_delaunay_subtrees(visocu_ctx* ctx, const uint32_t* pts, int32_t n_pts, int32_t n_jobs, const int32_t* first,
                                        const int32_t* count, const int32_t* axis, int32_t extra_halfedges, int32_t** mesh,
                                        int32_t* mesh_first, int32_t* n_halfedges, const int32_t** vert, const int32_t** result) {
  if (!ctx) return VISOCU_EINVAL;
  if (!ctx->configured) return visocu_set_error(ctx, VISOCU_ESTATE, "context not configured");
  if (!pts || n_pts <= 0 || n_jobs <= 0 || !first || !count || !axis || extra_halfedges < 0 || !mesh || !mesh_first || !n_halfedges || !vert || !result)
    return visocu_set_error(ctx, VISOCU_EINVAL, "bad subtree arguments");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  // device: jobs | points | vertex maps | result words | handles scratch | meshes      host (pinned): jobs | result words | vertex maps | meshes + room
  size_t n_he = 0;
  int maxn = 0;
  for (int j = 0; j < n_jobs; j++) {
    if (first[j] < 0 || count[j] < 4 || count[j] > 0x7FF0 || (int64_t)first[j] + count[j] > n_pts)
      return visocu_set_error(ctx, VISOCU_EINVAL, "subtree %d: range [%d, +%d) not inside %d points or size out of range", j, first[j], count[j], n_pts);
    mesh_first[j] = (int32_t)n_he;
    n_he += 2 * (size_t)ro_edge_capacity(count[j]);
    if (count[j] > maxn) maxn = count[j];
  }
  if (n_he + (size_t)extra_halfedges > 0x7FFFFFF0u) return visocu_set_error(ctx, VISOCU_EINVAL, "too many half-edges");
  const size_t d_jobs = 0, d_pts = align_up(sizeof(RoJob) * n_jobs, 256), d_vert = d_pts + align_up((size_t)4 * n_pts, 256);
  const size_t d_res = d_vert + align_up((size_t)4 * n_pts, 256), d_hnd = d_res + (size_t)64 * n_jobs;
  const size_t d_mesh = d_hnd + align_up((size_t)8 * ((size_t)n_pts / 2 + 2 * (size_t)n_jobs), 256), d_end = d_mesh + 16 * n_he;
  const size_t h_res = align_up(sizeof(RoJob) * n_jobs, 256), h_vert = h_res + (size_t)64 * n_jobs, h_mesh = h_vert + align_up((size_t)4 * n_pts, 256);
  const size_t h_end = h_mesh + 16 * (n_he + (size_t)extra_halfedges);
  int rc = visocu_ensure_scratch(ctx, d_end);
  if (rc) return rc;
  if ((rc = visocu_ensure_pinned(ctx, h_end))) return rc;
  uint8_t* sb = (uint8_t*)ctx->scratch;
  uint8_t* pin = (uint8_t*)ctx->pinned;
  RoJob* hj = (RoJob*)pin;
  int32_t* hres = (int32_t*)(pin + h_res);
  size_t hnd_off = 0;
  for (int j = 0; j < n_jobs; j++) {
    RoJob J;
    memset(&J, 0, sizeof J);
    J.result = (int32_t*)(sb + d_res) + 16 * j; J.n_in = J.result + 8;
    J.vert = (int32_t*)(sb + d_vert) + first[j];
    J.hnd = (uint16_t*)(sb + d_hnd) + hnd_off; hnd_off += 4 * ((size_t)count[j] / 2 + 2);
    J.pts_in = (const uint32_t*)(sb + d_pts) + first[j];
    J.mesh_out = (int4*)(sb + d_mesh) + mesh_first[j];
    J.axis0 = axis[j] & 1; J.he_base = mesh_first[j]; J.v_base = first[j];
    hj[j] = J;
    memset(hres + 16 * j, 0, 64);
    hres[16 * j + 1] = -1; hres[16 * j + 8] = count[j];
  }
  CU_COPY(ctx, sb + d_jobs, pin, sizeof(RoJob) * n_jobs, cudaMemcpyHostToDevice);
  CU_COPY(ctx, sb + d_res, hres, (size_t)64 * n_jobs, cudaMemcpyHostToDevice);
  CU_COPY(ctx, sb + d_pts, pts, (size_t)4 * n_pts, cudaMemcpyHostToDevice);
  if ((rc = visocu_launch_remove_outliers(ctx, (const RoJob*)(sb + d_jobs), n_jobs, 0, maxn, ctx->stream))) return rc;
  CU_COPY(ctx, hres, sb + d_res, (size_t)64 * n_jobs, cudaMemcpyDeviceToHost);
  CU_COPY(ctx, pin + h_vert, sb + d_vert, (size_t)4 * n_pts, cudaMemcpyDeviceToHost);
  CU_COPY(ctx, pin + h_mesh, sb + d_mesh, 16 * n_he, cudaMemcpyDeviceToHost);
  CU_TRY(ctx, visocu_stream_wait(ctx));
  ctx->ro_node_calls++;
  for (int j = 0; j < n_jobs; j++) if (hres[16 * j + 1] == 0) ctx->ro_nodes++;
  *mesh = (int32_t*)(pin + h_mesh); *n_halfedges = (int32_t)n_he; *vert = (const int32_t*)(pin + h_vert); *result = hres;
  return VISOCU_OK;
}

int visocu_launch_outlier_keys(visocu_ctx* ctx, const RoJob* jobs_dev, int n_jobs, uint32_t* keys_dev, int stride) {
  int gx = (stride + 255) / 256; if (gx > 64) gx = 64;
  k_outlier_keys<<<dim3(gx, n_jobs), 256, 0, ctx->stream>>>(jobs_dev, keys_dev, stride);
  CU_LAUNCH_CHECK(ctx);
  return VISOCU_OK;
}

// Triangle's vertexsort (a randomised quicksort: Hoare partition, pivot index from x' = (1366 x + 150889) mod 714025
// starting at 1, scaled to the subarray length) replayed on the positions in list order; the first of every run of equal
// positions is the point Triangle triangulates, the others it ignores (they collect no votes and are removed).
bool ro_resolve_duplicates(const uint32_t* keys, int n_records, uint8_t* rep) {
  static thread_local std::vector<uint32_t> kk, seen_words;
  static thread_local std::vector<int32_t> rec;
  kk.clear(); rec.clear();
  for (int i = 0; i < n_records; i++)
    if (keys[i] != 0xFFFFFFFFu) { kk.push_back(keys[i]); rec.push_back(i); }
  const int n = (int)kk.size();
  // any position taken twice?  (open-addressing hash set, a few n entries: stays in the cache)
  size_t cap = 64;
  while (cap < (size_t)4 * n) cap <<= 1;
  seen_words.assign(cap, 0xFFFFFFFFu);
  bool dup = false;
  for (int i = 0; i < n && !dup; i++) {
    const uint32_t k = kk[i];
    size_t h = ((size_t)k * 2654435761u) & (cap - 1);
    while (seen_words[h] != 0xFFFFFFFFu) {
      if (seen_words[h] == k) { dup = true; break; }
      h = (h + 1) & (cap - 1);
    }
    seen_words[h] = k;
  }
  if (!dup) return false;
  // elements: position in the high word (what the sort compares), index into rec[] in the low word
  static thread_local std::vector<unsigned long long> el;
  el.resize((size_t)n + 1);
  for (int i = 0; i < n; i++) el[i] = ((unsigned long long)kk[i] << 32) | (unsigned)i;
  el[n] = ~0ull;
  unsigned seed = 1;
  static thread_local std::vector<std::pair<int, int> > stack;
  stack.clear();
  stack.push_back(std::make_pair(0, n));
  while (!stack.empty()) {
    const int lo = stack.back().first, len = stack.back().second;
    stack.pop_back();
    if (len < 2) continue;
    unsigned long long* v = el.data() + lo;
    if (len == 2) {
      if ((v[0] >> 32) > (v[1] >> 32)) std::swap(v[0], v[1]);
      continue;
    }
    seed = (seed * 1366u + 150889u) % 714025u;
    const unsigned long long pkey = v[seed / (714025u / (unsigned)len + 1u)] >> 32;
    int left = -1, right = len;
    while (left < right) {
      do { left++; } while (left <= right && (v[left] >> 32) < pkey);
      do { right--; } while (left <= right && (v[right] >> 32) > pkey);
      if (left < right) std::swap(v[left], v[right]);
    }
    if (right < len - 2) stack.push_back(std::make_pair(lo + right + 1, len - right - 1));    // taken second
    if (left > 1) stack.push_back(std::make_pair(lo, left));                                   // taken first
  }
  // A record without a key (position outside 0..65535, e.g. a negative coordinate) stays a vertex, so that the kernel's
  // range check sees it and hands the list to the host, which triangulates any coordinates.  Left out, it would collect
  // no votes and be dropped with status 0.  Records the sub-pixel refinement dropped have no key either, but they never
  // reach the kernel's list.
  for (int i = 0; i < n_records; i++) rep[i] = keys[i] == 0xFFFFFFFFu ? 1 : 0;
  for (int i = 0; i < n; i++)
    if (i == 0 || (el[i] >> 32) != (el[i - 1] >> 32)) rep[rec[(size_t)(el[i] & 0xFFFFFFFFu)]] = 1;
  return true;
}
