// Batched ray casting through the map (mlm_cast_rays; no reference counterpart: the reference answers only point
// queries).  Exact voxel traversal of segments from[i] -> to[i]: the first blocking cell, and how many free / unknown
// cells the segment crosses before it.  The spec is in include/mlmap_b200.h ("batched queries"); oracle/oracle_rays.cpp
// (orc_cast_rays) and tests/raycast_spec.py restate it, and the records agree bit for bit.
//
// One thread per segment.  The walk keeps the subbox it is in in registers (pool block, collapsed state or absence) and
// the cell's position inside it, so a step needs no integer division and probes the hash table only when it wraps
// into the next subbox (about once every subbox_n steps); a cell costs one byte load (two with the inflated layer).
#pragma once
#include "query_kernels.cuh"

namespace mlm {

constexpr int kRayInflated = 1;                // MLM_RAY_INFLATED
constexpr int kRayInvalid = -2;                // MLM_RAY_INVALID
constexpr double kRayMaxQuot = 1073741824.0;   // |p / d_sub| < 2^30
constexpr long long kRayMaxCells = 1 << 20;    // |e - c|_1 <= 2^20
__device__ char g_ray_unknown_cell = 'u';      // what a cell of an absent subbox reads

struct __align__(16) RayHit {  // memory layout of mlm_ray_hit
  int status;
  int cell[3];
  int n_free, n_unknown;
  double t;
};
static_assert(sizeof(RayHit) == 32, "mlm_ray_hit is 32 bytes");

// cell of one coordinate: floor of the IEEE quotient (get_subbox_id's floor(pt / d_sub)), the canonical cell; the id-0
// quirk of locate_cell for point queries does not apply.  False for a non-finite p or |p / d| >= 2^30.
__device__ __forceinline__ bool ray_cell(double p, double d, int &c) {
  const double q = p / d;
  if (!(fabs(q) < kRayMaxQuot)) return false;
  c = (int)floor(q);
  return true;
}

// A subbox as a byte pointer per layer and an index mask: pool block (mask ~0: cell `sub`), collapsed (occupancy: its
// element 0; inflation: an unknown byte, so it never blocks by inflation) or absent (both read an unknown byte).  The ray
// walk and the ESDF gather (esdf_kernels.cuh) read cells through it, so the two agree on the blocking rule.
struct SubboxView {
  const char *occ, *inf;
  int mask;
};
__device__ __forceinline__ SubboxView subbox_view(const MapParams &P, const DeviceBuffers &D, const int g[3]) {
  uint32_t slot;
  const int blk = ht_find_slot(P, D, g, slot);
  SubboxView v = {&g_ray_unknown_cell, &g_ray_unknown_cell, 0};
  if (blk >= 0) {
    v.occ = D.pool_occ + (size_t)blk * P.cell_stride;
    v.inf = D.pool_inf + (size_t)blk * P.cell_stride;
    v.mask = ~0;
  } else if (blk == kBlockCollapsed) {
    v.occ = D.col_occ + slot;
  }
  return v;
}
// the spec's rule 3: `st` is the cell's state byte; with kInflated the inflation layer blocks too
template <bool kInflated>
__device__ __forceinline__ bool view_blocks(const SubboxView &v, int sub, char &st) {
  st = __ldg(v.occ + (sub & v.mask));
  return st == 'o' || (kInflated && __ldg(v.inf + (sub & v.mask)) == 'o');
}

// t of the next cell boundary on one axis, recomputed from the integer cell (no accumulation)
__device__ __forceinline__ double ray_next_t(int c, int s, double d, double from, double inv) {
  return ((double)(c + (s > 0 ? 1 : 0)) * d - from) * inv;
}

// The DDA of the spec's rule 2 from the point f in cell c to the point e_w in cell e, `total` = |e - c|_1 steps.  visit(view,
// sub, left) sees every cell of the walk in order (its subbox, its index there, the steps still to go) and returns true to
// stop; it must stop when left == 0.  On return c is the last cell visited and t_enter its entry t.  Rays stop at the
// first blocking cell (cast_ray), views at the first non-free cell before the target (view_kernels.cuh).
template <class Visit>
__device__ __forceinline__ void ray_walk(const MapParams &P, const DeviceBuffers &D, const double f[3], const double e_w[3],
                                         int c[3], const int e[3], long long total, double &t_enter, Visit visit) {
  int rem[3], s[3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const long long dl = (long long)e[k] - c[k];
    s[k] = dl > 0 ? 1 : (dl < 0 ? -1 : 0);
  }
  double inv[3], t[3];
  int g[3], loc[3];
  const double d = P.d_sub;
  const int n = P.n;
  const int stride[3] = {1, n, n * n};
  int sub = 0;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    rem[k] = e[k] > c[k] ? e[k] - c[k] : c[k] - e[k];
    inv[k] = rem[k] > 0 ? 1.0 / (e_w[k] - f[k]) : 0.0;
    t[k] = rem[k] > 0 ? ray_next_t(c[k], s[k], d, f[k], inv[k]) : 0.0;
    g[k] = floor_div(c[k], n);
    loc[k] = c[k] - g[k] * n;
    sub += loc[k] * stride[k];
  }
  // The current subbox (SubboxView): every step does the same one or two loads whatever kind of subbox it is in.
  SubboxView view = subbox_view(P, D, g);
  int left = (int)total;
  t_enter = 0.0;
  for (;;) {
    if (visit(view, sub, left)) break;
    // the axis whose boundary comes first among those with steps left; ties go to x, then y, then z
    int ax = -1;
    double tb = 0.0;
#pragma unroll
    for (int k = 0; k < 3; k++)
      if (rem[k] > 0 && (ax < 0 || t[k] < tb)) {
        ax = k;
        tb = t[k];
      }
    t_enter = tb;
    left--;
    // the step, as selects rather than one branch per axis (lanes of a warp step along different axes)
    int ca = 0, sa = 0, la = 0, stra = 0;
    double fa = 0.0, ia = 0.0;
#pragma unroll
    for (int k = 0; k < 3; k++)
      if (k == ax) {
        c[k] += s[k];
        rem[k]--;
        loc[k] += s[k];
        ca = c[k];
        sa = s[k];
        la = loc[k];
        stra = stride[k];
        fa = f[k];
        ia = inv[k];
      }
    const double tn = ray_next_t(ca, sa, d, fa, ia);
#pragma unroll
    for (int k = 0; k < 3; k++)
      if (k == ax) t[k] = tn;
    sub += sa * stra;
    if (la == n || la < 0) {  // wrapped into the next subbox along the axis (about once every n steps)
#pragma unroll
      for (int k = 0; k < 3; k++)
        if (k == ax) {
          loc[k] = la < 0 ? n - 1 : 0;
          g[k] += sa;
        }
      sub -= sa * n * stra;
      view = subbox_view(P, D, g);
    }
  }
}

template <bool kInflated>
__device__ __forceinline__ RayHit cast_ray(const MapParams &P, const DeviceBuffers &D, const double *a, const double *b) {
  RayHit r = {kRayInvalid, {0, 0, 0}, 0, 0, 0.0};
  const double f[3] = {a[0], a[1], a[2]};
  const double e_w[3] = {b[0], b[1], b[2]};
  const double d = P.d_sub;
  int c[3], e[3];
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    ok = ray_cell(f[k], d, c[k]) && ok;
    ok = ray_cell(e_w[k], d, e[k]) && ok;
  }
  if (!ok) return r;
  long long total = 0;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const long long dl = (long long)e[k] - c[k];
    total += dl < 0 ? -dl : dl;
  }
  if (total > kRayMaxCells) return r;
  int n_free = 0, n_unknown = 0, status = 0;
  double t_enter;
  ray_walk(P, D, f, e_w, c, e, total, t_enter, [&](const SubboxView &view, int sub, int left) {
    char st;
    if (view_blocks<kInflated>(view, sub, st)) {
      status = 0;  // MLM_OCCUPIED
      return true;
    }
    n_free += st == 'f' ? 1 : 0;
    n_unknown += st == 'f' ? 0 : 1;
    if (left == 0) {
      status = 1;  // MLM_FREE
      return true;
    }
    return false;
  });
  r.status = status;
  r.cell[0] = c[0];
  r.cell[1] = c[1];
  r.cell[2] = c[2];
  r.n_free = n_free;
  r.n_unknown = n_unknown;
  r.t = t_enter > 0.0 ? (t_enter < 1.0 ? t_enter : 1.0) : 0.0;  // clamp to [0, 1]; -0 and NaN give 0
  return r;
}

// from / to: n x 3 doubles; out: n records.  Each warp stages its 32 records (1 KiB) in shared memory and stores them
// as 64 contiguous 16-byte words.
template <bool kInflated>
__global__ void __launch_bounds__(256) k_cast_rays(MapParams P, DeviceBuffers D, const double *from, const double *to,
                                                   size_t n, RayHit *out) {
  __shared__ uint4 s_rec[2 * 256];
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  RayHit r = {kRayInvalid, {0, 0, 0}, 0, 0, 0.0};
  if (i < n) r = cast_ray<kInflated>(P, D, from + 3 * i, to + 3 * i);
  const unsigned long long tb = (unsigned long long)__double_as_longlong(r.t);
  s_rec[2 * threadIdx.x] = make_uint4((uint32_t)r.status, (uint32_t)r.cell[0], (uint32_t)r.cell[1], (uint32_t)r.cell[2]);
  s_rec[2 * threadIdx.x + 1] = make_uint4((uint32_t)r.n_free, (uint32_t)r.n_unknown, (uint32_t)tb, (uint32_t)(tb >> 32));
  __syncwarp();
  const int lane = threadIdx.x & 31, w0 = threadIdx.x & ~31;
  const size_t first = (size_t)blockIdx.x * blockDim.x + w0;  // first record of this warp
  uint4 *o4 = reinterpret_cast<uint4 *>(out);
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const int k = 32 * j + lane;
    if (first + (k >> 1) < n) o4[2 * first + k] = s_rec[2 * w0 + k];
  }
}

}  // namespace mlm
