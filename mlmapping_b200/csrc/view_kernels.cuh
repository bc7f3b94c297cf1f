// Candidate-view gain (mlm_view_gain; no reference counterpart): per pose of a pinhole depth sensor, the target cells
// (unknown, or frontier) in its frustum, and how many of them it sees through free space.  The spec is in
// include/mlmap_b200.h ("candidate-view gain"); oracle/oracle_views.cpp and tests/view_spec.py restate it, and the records
// agree bit for bit.
//
//   k_view_setup  one thread per view: T_sw, the origin and the status (the pose algebra of the frame path, exact_math.cuh),
//                 a conservative cell AABB of the frustum clipped to the view's box, and the number of subbox-aligned
//                 tiles that cover it; initialises the view's record
//   k_view_scan   one CTA: inclusive scan of the per-view tile counts (64-bit), so every (view, tile) item has an index
//   k_view_tiles  grid-stride over the items, one CTA per item: a tile that lies wholly outside one face of the frustum is
//                 skipped; else one hash probe for the tile's subbox, then the threads go over its cells with the exact
//                 frustum and target tests, and walk the line of sight (ray_walk) for targets only.  All threads of a
//                 CTA walk from one origin towards neighbouring cells, so the walks share their subboxes in L1 / L2.
//                 Counts go through a warp reduction and one integer atomic per warp, so they do not depend on the order
//                 threads run in.
#pragma once
#include "ray_kernels.cuh"

namespace mlm {

constexpr int kViewFrontier = 1;   // MLM_VIEW_FRONTIER
constexpr int kViewInflated = 2;   // MLM_VIEW_INFLATED
constexpr int kViewInvalid = -2;   // MLM_VIEW_INVALID
constexpr int kViewMaxCells = 256; // max_depth and the far corners' lateral offsets are at most 256 * d_sub
constexpr int kViewTileThreads = 256;
constexpr int kViewScanThreads = 1024;

struct ViewSensor {  // memory layout of mlm_view_sensor
  double fx, fy, cx, cy;
  int cols, rows;
  double min_depth, max_depth;
};

struct __align__(16) ViewGain {  // memory layout of mlm_view_gain_record
  int status, n_target, n_visible, pad;
};
static_assert(sizeof(ViewGain) == 16, "mlm_view_gain_record is 16 bytes");

struct __align__(16) ViewSetup {  // one view, from k_view_setup
  HQuat q;            // T_sw = T_ws.inverse()
  double t[3];
  double o[3];        // origin T_ws.t
  int co[3];          // cell(o)
  int lo[3], hi[3];   // inclusive cell AABB of the frustum, clipped to the box
  int glo[3], gdim[3];  // the tiles: subboxes glo .. glo + gdim - 1
};

// rule 3 on sensor coordinates p: depth range, then the pixel rectangle with the project_depth pixel centres
__device__ __forceinline__ bool view_in_frustum(const ViewSensor &S, const double p[3]) {
  if (!(p[2] >= S.min_depth && p[2] <= S.max_depth)) return false;
  const double u = (p[0] / p[2]) * S.fx + S.cx;
  const double v = (p[1] / p[2]) * S.fy + S.cy;
  return u >= -0.5 && u < (double)S.cols - 0.5 && v >= -0.5 && v < (double)S.rows - 0.5;
}

// p = T_sw * x (Sophus SE3 * Vector3: rotate, then add the translation)
__device__ __forceinline__ void view_to_sensor(const HQuat &q, const double t[3], const double x[3], double p[3]) {
  h_rotate(q, x, p);
#pragma unroll
  for (int k = 0; k < 3; k++) p[k] = p[k] + t[k];
}

__global__ void __launch_bounds__(256) k_view_setup(MapParams P, HPose T_bs, ViewSensor S, const double *T_wb,
                                                    const int *boxes, size_t n, ViewSetup *setup,
                                                    unsigned long long *tiles, ViewGain *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double p7[7];
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 7; k++) {
    p7[k] = T_wb[7 * i + k];
    ok = ok && isfinite(p7[k]);
  }
  // rule 1: the squared norm as h_normalized forms it
  const double n2 = (p7[4] * p7[4] + p7[6] * p7[6]) + (p7[5] * p7[5] + p7[3] * p7[3]);
  ok = ok && n2 > 0.0 && isfinite(n2);
  ViewSetup V = {};
  unsigned long long cnt = 0;
  const double d = P.d_sub;
  if (ok) {
    const HPose Tws = h_compose(h_pose_from7(p7), T_bs);
    const HPose Tsw = h_inverse(Tws);
    V.q = Tsw.q;
    double mn[3], mx[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      V.t[k] = Tsw.t[k];
      V.o[k] = Tws.t[k];
      ok = ray_cell(V.o[k], d, V.co[k]) && ok;
      mn[k] = mx[k] = V.o[k];
    }
    // the frustum lies in the pyramid of the origin and the four far corners; one cell of margin covers the rounding
    // of these corners and of the cell-centre tests
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const double uc = (j & 1) ? (double)S.cols - 0.5 : -0.5, vc = (j & 2) ? (double)S.rows - 0.5 : -0.5;
      const double s[3] = {((uc - S.cx) / S.fx) * S.max_depth, ((vc - S.cy) / S.fy) * S.max_depth, S.max_depth};
      double w[3];
      view_to_sensor(Tws.q, Tws.t, s, w);
#pragma unroll
      for (int k = 0; k < 3; k++) {
        mn[k] = fmin(mn[k], w[k]);
        mx[k] = fmax(mx[k], w[k]);
      }
    }
    bool empty = false;
#pragma unroll
    for (int k = 0; k < 3; k++) {
      V.lo[k] = (int)floor(mn[k] / d) - 1;
      V.hi[k] = (int)floor(mx[k] / d) + 1;
      if (boxes) {
        const int blo = boxes[6 * i + k], bhi = boxes[6 * i + 3 + k];
        ok = ok && blo <= bhi;
        V.lo[k] = max(V.lo[k], blo);
        V.hi[k] = min(V.hi[k], bhi);
      }
      empty = empty || V.lo[k] > V.hi[k];
    }
    if (ok && !empty) {
      cnt = 1;
#pragma unroll
      for (int k = 0; k < 3; k++) {
        V.glo[k] = floor_div(V.lo[k], P.n);
        V.gdim[k] = floor_div(V.hi[k], P.n) - V.glo[k] + 1;
        cnt *= (unsigned long long)V.gdim[k];
      }
    }
  }
  if (!ok) cnt = 0;
  setup[i] = V;
  tiles[i] = cnt;
  out[i] = ViewGain{ok ? 0 : kViewInvalid, 0, 0, 0};
}

// inclusive scan of a[0..n) in place, one CTA of kViewScanThreads
__global__ void __launch_bounds__(kViewScanThreads) k_view_scan(unsigned long long *a, size_t n) {
  __shared__ unsigned long long s_warp[kViewScanThreads / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned long long carry = 0;
  for (size_t base = 0; base < n; base += kViewScanThreads) {
    const size_t i = base + threadIdx.x;
    unsigned long long v = i < n ? a[i] : 0ull;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    if (lane == 31) s_warp[w] = v;
    __syncthreads();
    if (w == 0) {
      unsigned long long s = s_warp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += t;
      }
      s_warp[lane] = s;
    }
    __syncthreads();
    v += carry + (w > 0 ? s_warp[w - 1] : 0ull);
    if (i < n) a[i] = v;
    carry += s_warp[kViewScanThreads / 32 - 1];
    __syncthreads();
  }
}

// The tile [a, b] (cell centres) lies wholly outside the frustum: all 8 corners of the box of its cell centres beyond one
// face by more than 2 cells, so no rounding of the per-cell test can bring a centre back in.  Skipping it changes no count.
__device__ __forceinline__ bool view_tile_outside(const ViewSensor &S, const ViewSetup &V, const int a[3], const int b[3],
                                                  double d) {
  // side planes through the origin: u >= -0.5 <=> fx * p_x - (-0.5 - cx) * p_z >= 0 for p_z > 0 (likewise the others)
  const double al = -0.5 - S.cx, ar = (double)S.cols - 0.5 - S.cx, at = -0.5 - S.cy, ab = (double)S.rows - 0.5 - S.cy;
  const double m = 2.0 * d;
  const double ml = m * sqrt(S.fx * S.fx + al * al), mr = m * sqrt(S.fx * S.fx + ar * ar);
  const double mt = m * sqrt(S.fy * S.fy + at * at), mb = m * sqrt(S.fy * S.fy + ab * ab);
  bool near = true, far = true, left = true, right = true, top = true, bottom = true;
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const double x[3] = {((double)((j & 1) ? b[0] : a[0]) + 0.5) * d, ((double)((j & 2) ? b[1] : a[1]) + 0.5) * d,
                         ((double)((j & 4) ? b[2] : a[2]) + 0.5) * d};
    double p[3];
    view_to_sensor(V.q, V.t, x, p);
    near = near && p[2] < S.min_depth - m;
    far = far && p[2] > S.max_depth + m;
    left = left && S.fx * p[0] - al * p[2] < -ml;
    right = right && S.fx * p[0] - ar * p[2] > mr;
    top = top && S.fy * p[1] - at * p[2] < -mt;
    bottom = bottom && S.fy * p[1] - ab * p[2] > mb;
  }
  return near || far || left || right || top || bottom;
}

template <bool kFrontier, bool kInflated>
__global__ void __launch_bounds__(kViewTileThreads) k_view_tiles(MapParams P, DeviceBuffers D, ViewSensor S,
                                                                 const ViewSetup *setup, const unsigned long long *incl,
                                                                 size_t n, ViewGain *out) {
  __shared__ ViewSetup sV;
  __shared__ int s_skip;
  const unsigned long long total = incl[n - 1];
  const double d = P.d_sub;
  const int nn = P.n;
  for (unsigned long long item = blockIdx.x; item < total; item += gridDim.x) {
    // the view of the item: the first v with incl[v] > item (every thread searches the same entries: broadcast loads)
    size_t lo = 0, hi = n - 1;
    while (lo < hi) {
      const size_t mid = (lo + hi) >> 1;
      if (incl[mid] > item) hi = mid;
      else lo = mid + 1;
    }
    const size_t v = lo;
    const unsigned long long tile = item - (v ? incl[v - 1] : 0ull);
    __syncthreads();  // the previous item is done with sV
    if (threadIdx.x < sizeof(ViewSetup) / 16)
      reinterpret_cast<uint4 *>(&sV)[threadIdx.x] = reinterpret_cast<const uint4 *>(setup + v)[threadIdx.x];
    __syncthreads();
    const int tx = (int)(tile % (unsigned)sV.gdim[0]);
    const unsigned long long tyz = tile / (unsigned)sV.gdim[0];
    const int g[3] = {sV.glo[0] + tx, sV.glo[1] + (int)(tyz % (unsigned)sV.gdim[1]),
                      sV.glo[2] + (int)(tyz / (unsigned)sV.gdim[1])};
    int a[3], b[3], m[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      a[k] = max(g[k] * nn, sV.lo[k]);
      b[k] = min(g[k] * nn + nn - 1, sV.hi[k]);
      m[k] = b[k] - a[k] + 1;
    }
    if (threadIdx.x == 0) s_skip = view_tile_outside(S, sV, a, b, d);
    __syncthreads();
    if (s_skip) continue;
    // the tile's subbox, probed once: its state bytes, and its frontier words (live blocks only)
    uint32_t slot;
    const int blk = ht_find_slot(P, D, g, slot);
    SubboxView tv = {&g_ray_unknown_cell, &g_ray_unknown_cell, 0};
    const uint32_t *front = nullptr;
    if (blk >= 0) {
      tv.occ = D.pool_occ + (size_t)blk * P.cell_stride;
      front = D.pool_front + (size_t)blk * P.front_words;
      tv.mask = ~0;
    } else if (blk == kBlockCollapsed) {
      tv.occ = D.col_occ + slot;
    }
    int n_target = 0, n_visible = 0;
    const int cells = m[0] * m[1] * m[2];
    for (int j = threadIdx.x; j < cells; j += kViewTileThreads) {
      const int c[3] = {a[0] + j % m[0], a[1] + (j / m[0]) % m[1], a[2] + j / (m[0] * m[1])};
      const double x[3] = {((double)c[0] + 0.5) * d, ((double)c[1] + 0.5) * d, ((double)c[2] + 0.5) * d};
      double p[3];
      view_to_sensor(sV.q, sV.t, x, p);
      if (!view_in_frustum(S, p)) continue;
      const int sub = ((c[2] - g[2] * nn) * nn + (c[1] - g[1] * nn)) * nn + (c[0] - g[0] * nn);
      bool target;
      if (kFrontier) {
        target = front && ((__ldg(front + (sub >> 5)) >> (sub & 31)) & 1u);
      } else {
        const char st = __ldg(tv.occ + (sub & tv.mask));
        target = st != 'f' && st != 'o';
      }
      if (!target) continue;
      n_target++;
      // rule 5: from o to the centre, every cell before c FREE (and not inflated with kInflated)
      int w[3] = {sV.co[0], sV.co[1], sV.co[2]};
      long long steps = 0;
#pragma unroll
      for (int k = 0; k < 3; k++) steps += c[k] > w[k] ? c[k] - w[k] : w[k] - c[k];
      bool seen = false;
      double t_enter;
      ray_walk(P, D, sV.o, x, w, c, steps, t_enter, [&](const SubboxView &view, int s, int left) {
        if (left == 0) {
          seen = true;
          return true;
        }
        char st;
        return view_blocks<kInflated>(view, s, st) || st != 'f';
      });
      n_visible += seen ? 1 : 0;
    }
    n_target = __reduce_add_sync(0xffffffffu, n_target);
    n_visible = __reduce_add_sync(0xffffffffu, n_visible);
    if ((threadIdx.x & 31) == 0 && n_target) {
      atomicAdd(&out[v].n_target, n_target);
      if (n_visible) atomicAdd(&out[v].n_visible, n_visible);
    }
  }
}

}  // namespace mlm
