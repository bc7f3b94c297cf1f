// Per-frame map update kernels (sm_100a).  Replaces, on the GPU, the reference's
//   mlmap::project_depth            src/mlmap.cpp:311-349            -> k_project_depth
//   awareness::input_pc_pose        src/map_awareness.cpp:173-282    -> k_project_* + k_column
//   awareness::update_hits          src/map_awareness.cpp:135-171    -> k_column (contributions + ordered fold)
//   local::input_pc_pose_direct     src/map_local.cpp:143-207        -> k_column (staging) + k_submaps + k_fuse
//   local::allocate_ram             include/map_local.h:215-231      -> k_submaps
// Design notes are in DESIGN.md; every arithmetic step that decides an index or a float result
// follows SURVEY Appendix A exactly (IEEE, no FMA contraction: this TU is built with -fmad=false).
#pragma once
#include "exact_math.cuh"
#include "types.cuh"

namespace mlm {

// ---- small helpers -------------------------------------------------------------------------------

// x86-64 cvttsd2si semantics (what the g++-compiled reference does for static_cast<int>(double)):
// NaN / out-of-range -> INT_MIN ("integer indefinite").
__device__ __forceinline__ int cvt_trunc_x86(double x) {
  if (!(x > -2147483649.0 && x < 2147483648.0)) return (int)0x80000000;
  return __double2int_rz(x);
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// static_cast<int>(round(v)) for |v| < 2^31: std::round is half-away-from-zero.  v - trunc(v) is exact,
// so this equals the libm result bit for bit (falls back to cvt_trunc_x86(round(v)) outside the range).
__device__ __forceinline__ int round_to_int_x86(double v) {
  if (!(v > -2147483000.0 && v < 2147483000.0)) return cvt_trunc_x86(round(v));
  int zi = __double2int_rz(v);
  double frac = v - (double)zi;
  if (frac >= 0.5) zi++;
  else if (frac <= -0.5) zi--;
  return zi;
}

// warp-aggregated counter increment; returns this thread's slot
__device__ __forceinline__ int agg_inc(int *ctr) {
  unsigned mask = __activemask();
  int leader = __ffs(mask) - 1;
  int res = 0;
  if (lane_id() == leader) res = atomicAdd(ctr, __popc(mask));
  res = __shfl_sync(mask, res, leader);
  return res + __popc(mask & ((1u << lane_id()) - 1));
}

__device__ __forceinline__ int floor_div(int a, int b) {
  int q = a / b, r = a - q * b;
  return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q;
}

// fast_atan / fast_atan2, reference include/map_awareness.h:86-118
__device__ __forceinline__ double ref_fast_atan(double x) { return x * (45 - (x - 1) * (14 + 3.83 * x)); }
__device__ __forceinline__ double ref_fast_atan2(double y, double x) {
  const double deg2rad = M_PI / 180;  // "M_PI / 180 * (...)" associates as (M_PI/180) * (...)
  double input = y / x;
  double a_input = fabs(input);
  double res;
  if (a_input > 1) {
    res = copysign(deg2rad * (90 - ref_fast_atan(1 / a_input)), input);
  } else {
    res = copysign(deg2rad * ref_fast_atan(a_input), input);
  }
  if (x > 0) return res;
  if (y >= 0) return res + M_PI;
  return res - M_PI;
}

// floor(fl(p / d)) without paying for an IEEE division on every call.  qa = p * fl(1/d) differs from the
// correctly rounded quotient fl(p/d) by less than 4e-16 relative, so when qa is not within 1e-15 relative
// of an integer both have the same floor; otherwise (lattice points, cell borders) the true division
// decides.  The result is therefore always exactly what the reference's division + floor gives.
__device__ __forceinline__ double floor_quot_exact(double p, double d, double inv_d) {
  const double qa = p * inv_d;
  double f = floor(qa);
  const double eps = fabs(qa) * 1e-15;
  if (!(qa - f > eps && (f + 1.0) - qa > eps)) f = floor(p / d);  // also taken for NaN / inf
  return f;
}

// get_global_idx + get_subbox_id, reference include/map_local.h:148-152,167-173.
// sub-index components outside [0,n) hit unordered_map::operator[] on a missing key -> id 0.
struct CellRef {
  int g[3];   // subbox (global) index
  int sub;    // cell id inside the subbox
  int c[3];   // canonical global cell coordinate g*n + xyz(sub)
};
__device__ __forceinline__ CellRef locate_cell(const MapParams &P, double px, double py, double pz) {
  CellRef r;
  double p[3] = {px, py, pz};
  int loc[3];
  bool ok = true;
#pragma unroll
  for (int a = 0; a < 3; a++) {
    r.g[a] = cvt_trunc_x86(floor_quot_exact(p[a], P.d_glb, P.inv_d_glb));
    double l = floor_quot_exact(p[a], P.d_sub, P.inv_d_sub) - (double)(r.g[a] * P.n);
    loc[a] = cvt_trunc_x86(l);
    ok = ok && loc[a] >= 0 && loc[a] < P.n;
  }
  if (!ok) loc[0] = loc[1] = loc[2] = 0;
  r.sub = (loc[2] * P.n + loc[1]) * P.n + loc[0];
#pragma unroll
  for (int a = 0; a < 3; a++) r.c[a] = r.g[a] * P.n + loc[a];
  return r;
}

__device__ __forceinline__ int lvg_index(const MapParams &P, const FrameParams &F, const CellRef &r) {
  int lx = r.c[0] - F.lvg_base[0], ly = r.c[1] - F.lvg_base[1], lz = r.c[2] - F.lvg_base[2];
  if ((unsigned)lx >= (unsigned)P.lvg_dim_xy || (unsigned)ly >= (unsigned)P.lvg_dim_xy ||
      (unsigned)lz >= (unsigned)P.lvg_dim_z)
    return -1;
  return (lz * P.lvg_dim_xy + ly) * P.lvg_dim_xy + lx;
}
__device__ __forceinline__ int lsg_index(const MapParams &P, const FrameParams &F, const int g[3]) {
  int lx = g[0] - F.lsg_base[0], ly = g[1] - F.lsg_base[1], lz = g[2] - F.lsg_base[2];
  if ((unsigned)lx >= (unsigned)P.lsg_dim_xy || (unsigned)ly >= (unsigned)P.lsg_dim_xy ||
      (unsigned)lz >= (unsigned)P.lsg_dim_z)
    return -1;
  return (lz * P.lsg_dim_xy + ly) * P.lsg_dim_xy + lx;
}

// raycasting_z_over_rho, reference src/map_awareness.cpp:64-71 and :252-259 (same expression)
__device__ __forceinline__ double ray_rate(const MapParams &P, int rho, int z) {
  return rho > 0 ? (double)(z - P.n_below) / ((double)rho * 1.0) : 0.0;
}

// 63-bit packing of a subbox index for the device hash table
__device__ __forceinline__ bool pack_glb(const int g[3], uint64_t &key) {
  const int lim = 1 << 20;
  if (g[0] < -lim || g[0] >= lim || g[1] < -lim || g[1] >= lim || g[2] < -lim || g[2] >= lim) return false;
  key = ((uint64_t)(uint32_t)(g[0] + lim) << 42) | ((uint64_t)(uint32_t)(g[1] + lim) << 21) |
        (uint64_t)(uint32_t)(g[2] + lim);
  return true;
}
__device__ __forceinline__ void unpack_glb(uint64_t key, int g[3]) {
  const int lim = 1 << 20;
  g[0] = (int)((key >> 42) & 0x1fffff) - lim;
  g[1] = (int)((key >> 21) & 0x1fffff) - lim;
  g[2] = (int)(key & 0x1fffff) - lim;
}
__device__ __forceinline__ uint32_t ht_hash(uint64_t k) {  // splitmix64 finaliser
  k ^= k >> 30;
  k *= 0xbf58476d1ce4e5b9ull;
  k ^= k >> 27;
  k *= 0x94d049bb133111ebull;
  k ^= k >> 31;
  return (uint32_t)k;
}
// sharded maps: the rank that owns subbox g (every rank computes the same hash)
__device__ __forceinline__ int subbox_owner(const int g[3], int world) {
  uint64_t key;
  if (world <= 1 || !pack_glb(g, key)) return 0;
  const uint32_t hsh = ht_hash(key);
  return (world & (world - 1)) == 0 ? (int)(hsh & (uint32_t)(world - 1)) : (int)(hsh % (uint32_t)world);
}
// lookup that also reports the hash slot (collapsed subboxes keep their element 0 in per-slot arrays)
__device__ __forceinline__ int ht_find_slot(const MapParams &P, const DeviceBuffers &D, const int g[3], uint32_t &slot_out) {
  uint64_t key;
  slot_out = 0;
  if (!pack_glb(g, key)) return -1;
  uint32_t slot = ht_hash(key) & P.ht_mask;
  for (uint32_t probe = 0; probe <= P.ht_mask; probe++) {
    uint64_t k = D.ht_key[slot];
    if (k == key) {
      slot_out = slot;
      return D.ht_val[slot];
    }
    if (k == kEmptyKey) return -1;
    slot = (slot + 1) & P.ht_mask;
  }
  return -1;
}
// read-only lookup of a subbox: returns pool block (>=0), or -1 if absent
__device__ __forceinline__ int ht_find(const MapParams &P, const DeviceBuffers &D, const int g[3]) {
  uint64_t key;
  if (!pack_glb(g, key)) return -1;
  uint32_t slot = ht_hash(key) & P.ht_mask;
  for (uint32_t probe = 0; probe <= P.ht_mask; probe++) {
    uint64_t k = D.ht_key[slot];
    if (k == key) return D.ht_val[slot];
    if (k == kEmptyKey) return -1;
    slot = (slot + 1) & P.ht_mask;
  }
  return -1;
}

// ---- K1: projection + transform + cylindrical index ------------------------------------------------
// One thread per point.  Output: a RayRecord per castable / inside point (in point order) and the
// per-phi-column histogram used to group the records by column.
__device__ __forceinline__ void point_to_record(const MapParams &P, const FrameParams &F, double xs, double ys,
                                                double zs, uint32_t t, RayRecord &rec, int &inside_out,
                                                int &cast_out) {
  // p_l = T_ls * p_s : Eigen Quaternion::_transformVector then + translation (se3.cpp:91-95)
  const double qw = F.q_ls[0], qx = F.q_ls[1], qy = F.q_ls[2], qz = F.q_ls[3];
  double uvx = qy * zs - qz * ys;
  double uvy = qz * xs - qx * zs;
  double uvz = qx * ys - qy * xs;
  uvx += uvx;
  uvy += uvy;
  uvz += uvz;
  double cx = qy * uvz - qz * uvy;
  double cy = qz * uvx - qx * uvz;
  double cz = qx * uvy - qy * uvx;
  double x = ((xs + qw * uvx) + cx) + F.t_ls[0];
  double y = ((ys + qw * uvy) + cy) + F.t_ls[1];
  double z = ((zs + qw * uvz) + cz) + F.t_ls[2];
  // xyz2RhoPhiZwithBoderCheck, src/map_awareness.cpp:84-107
  double rho = sqrt(x * x + y * y);
  // static_cast<int>(x / d) truncates; rho and the wrapped phi are >= 0 (or NaN -> exact path), so trunc == floor
  int rho_idx = cvt_trunc_x86(floor_quot_exact(rho, P.dRho, P.inv_dRho));
  double phi = ref_fast_atan2(y, x);
  if (phi < 0) phi += 2 * M_PI;
  int phi_idx = phi >= 0 ? cvt_trunc_x86(floor_quot_exact(phi, P.dPhi, P.inv_dPhi)) : cvt_trunc_x86(phi / P.dPhi);
  double zz = z - P.z_border_min;
  int z_idx = cvt_trunc_x86(floor_quot_exact(zz, P.dZ, P.inv_dZ));
  bool can = rho_idx >= 0 && phi_idx >= 0 && phi_idx < P.nPhi;
  bool inside = can && z_idx >= 0 && rho_idx < P.nRho && z_idx < P.nZ;
  bool cast = can && P.visibility_check;
  inside_out = inside;
  cast_out = cast;
  if (inside || cast) {
    rec.rho = rho_idx;
    rec.z = z_idx;
    rec.phi_flags = (uint32_t)phi_idx | (inside ? kRecInside : 0u);
    rec.t = t;
  }
}

// Guarded fast path of point_to_record.  Only the three integer indices of a point reach the map, so the
// point is first located with cheap arithmetic (FMA transform in double, then float sqrt / division /
// polynomial): the float values are within 1e-6 relative of what the reference's double chain yields, and
// an index is accepted only when its value (in cells) is farther than a 1000x larger guard band from the
// next integer, where truncation cannot differ.  Anything inside a guard band, on the x == 0 quirk of
// fast_atan2 or not finite is left to the exact path.  Returns false when the exact path has to run.
__device__ __forceinline__ bool point_to_record_fast(const MapParams &P, const FrameParams &F, double xs, double ys,
                                                     double zs, uint32_t t, RayRecord &rec, int &inside_out,
                                                     int &cast_out) {
  const double qw = F.q_ls[0], qx = F.q_ls[1], qy = F.q_ls[2], qz = F.q_ls[3];
  double uvx = __fma_rn(qy, zs, -(qz * ys));
  double uvy = __fma_rn(qz, xs, -(qx * zs));
  double uvz = __fma_rn(qx, ys, -(qy * xs));
  uvx += uvx;
  uvy += uvy;
  uvz += uvz;
  const double x = __fma_rn(qw, uvx, xs) + __fma_rn(qy, uvz, -(qz * uvy)) + F.t_ls[0];
  const double y = __fma_rn(qw, uvy, ys) + __fma_rn(qz, uvx, -(qx * uvz)) + F.t_ls[1];
  const double z = __fma_rn(qw, uvz, zs) + __fma_rn(qx, uvy, -(qy * uvx)) + F.t_ls[2];
  const float xf = (float)x, yf = (float)y, zf = (float)(z - P.z_border_min);
  const float ax = fabsf(xf), ay = fabsf(yf);
  if (!(ax > 1e-30f) || !(ax < 1e6f) || !(ay < 1e6f) || !(fabsf(zf) < 1e6f)) return false;  // x == 0 quirk, NaN, huge
  const float rho_c = sqrtf(xf * xf + yf * yf) * P.fast_inv_dRho;
  const float z_c = zf * P.fast_inv_dZ;
  const bool steep = ay > ax;
  const float tq = steep ? ax / ay : ay / ax;                       // a_input or 1 / a_input, in [0, 1]
  const float f = tq * (45.0f - (tq - 1.0f) * (14.0f + 3.83f * tq));  // fast_atan, degrees
  float deg = steep ? 90.0f - f : f;
  if ((yf < 0.0f) != (xf < 0.0f)) deg = -deg;                        // copysign(., y / x)
  if (!(xf > 0.0f)) deg += yf >= 0.0f ? 180.0f : -180.0f;
  if (deg < 0.0f) deg += 360.0f;
  const float phi_c = deg * P.fast_deg2cell;
  // guard bands: 1e-3 cells + 4e-6 relative (float chain error < 1e-6 relative)
  const float rr = rintf(rho_c), zr = rintf(z_c), pr = rintf(phi_c);
  if (fabsf(rho_c - rr) < 1e-3f + 4e-6f * rho_c || fabsf(z_c - zr) < 1e-3f + 4e-6f * fabsf(z_c) ||
      fabsf(phi_c - pr) < 1e-3f + 4e-6f * phi_c)
    return false;
  const int rho_idx = (int)rho_c, phi_idx = (int)phi_c, z_idx = (int)floorf(z_c);
  const bool can = phi_idx < P.nPhi;  // rho_idx, phi_idx >= 0 by construction
  const bool inside = can && z_idx >= 0 && rho_idx < P.nRho && z_idx < P.nZ;
  const bool cast = can && P.visibility_check;
  inside_out = inside;
  cast_out = cast;
  if (inside || cast) {
    rec.rho = rho_idx;
    rec.z = z_idx;
    rec.phi_flags = (uint32_t)phi_idx | (inside ? kRecInside : 0u);
    rec.t = t;
  }
  return true;
}

// CTA-wide exclusive scan of data[0,n) in shared memory (in place); returns the total.
// Each thread scans a contiguous slice, slices are combined with warp shuffles.
__device__ __forceinline__ int block_exclusive_scan(int *data, int n, int *s_warp /*[33]*/) {
  const int nt = blockDim.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = nt >> 5;
  const int per = (n + nt - 1) / nt;
  const int beg = min(tid * per, n), end = min(beg + per, n);
  int sum = 0;
  for (int i = beg; i < end; i++) sum += data[i];
  int incl = sum;
#pragma unroll
  for (int ofs = 1; ofs < 32; ofs <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, incl, ofs);
    if (lane >= ofs) incl += t;
  }
  if (lane == 31) s_warp[w] = incl;
  __syncthreads();
  if (w == 0) {
    int sv = lane < nw ? s_warp[lane] : 0, si = sv;
#pragma unroll
    for (int ofs = 1; ofs < 32; ofs <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, si, ofs);
      if (lane >= ofs) si += t;
    }
    if (lane < nw) s_warp[lane] = si - sv;
    if (lane == 31) s_warp[32] = si;
  }
  __syncthreads();
  int run = s_warp[w] + incl - sum;
  for (int i = beg; i < end; i++) {
    int v = data[i];
    data[i] = run;
    run += v;
  }
  __syncthreads();
  return s_warp[32];
}

// kMode: 0 = sensor-frame points (xyz doubles), 1 = full depth image (every pixel, row-major),
//        2 = sampled depth pixels: input is uint2 {pixel index, raw depth} in sampling order (src/mlmap.cpp:321-346)
// One CTA owns a tile of F.tile_pts consecutive points (a multiple of 32); warp w owns a run of consecutive
// 32-point rounds of the tile (at most kProjMaxPts, 64-byte depth-row loads each),
// so "point order" inside the tile is (warp, round, lane) and everything that has to follow point order is
// warp-local except one exclusive scan over the warps.
constexpr int kProjThreads = 512;                    // stand-alone k_project launch
constexpr int kProjMaxPts = 4;                       // upper bound of rounds per warp: tile_pts <= 128 * warps
__host__ __device__ inline size_t project_smem_bytes(int nCol, int threads) { return (size_t)(threads / 32 + 3) * nCol * sizeof(int); }

// work column of a record: its phi column, or (phi, side) when the columns are split at the sensor row
__device__ __forceinline__ int work_column(const MapParams &P, const RayRecord &rc) {
  const int phi = (int)(rc.phi_flags & kRecPhiMask);
  return P.split ? (phi << 1) | (rc.z >= P.n_below ? 1 : 0) : phi;
}

template <int kMode>
__device__ __forceinline__ void project_tile(const MapParams &P, DeviceBuffers &D, const FrameParams &F, const int tile,
                                             int *s_proj) {
  // shared: [warps][W] per-warp counts -> exclusive prefix over warps, [W] totals, [W] offsets, [W] contribution bounds,
  // where W is the span of work columns this tile touches (indices are relative to a per-tile base, modulo nCol,
  // so a tile that straddles phi = 0 still has a short span); sized for the worst case W = nCol
  __shared__ int s_cnt[3];
  __shared__ int s_warp[33];
  __shared__ int s_base, s_rmin, s_rmax;
  const int nCol = P.nCol;  // work columns: phi, or (phi, side of the sensor row) when the columns are split
  const int N = F.n_total;
  const int nthreads = blockDim.x, nwarps = nthreads >> 5;
  // the tile's 32-point rounds are dealt to the warps in order, as evenly as they go (<= kProjMaxPts each)
  const int rounds = F.tile_pts >> 5;
  const int r0 = (int)(((long long)(threadIdx.x >> 5) * rounds) / nwarps), r1 = (int)(((long long)((threadIdx.x >> 5) + 1) * rounds) / nwarps);
  const int pts = r1 - r0;
  const int tile0 = tile * F.tile_pts;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (P.split && tile == 0) {
    // the one miss-bitmap row both half columns of a phi write (atomicOr in k_column) starts the frame empty
    for (int i = tid; i < P.nPhi * P.words_per_row; i += nthreads) {
      const int ph = i / P.words_per_row;
      D.miss_bitmap[(size_t)ph * P.col_words + P.n_below * P.words_per_row + (i - ph * P.words_per_row)] = 0;
    }
  }
  if (tile0 >= N) return;  // the grid is sized for cfg.max_points (graph replay)
  if (tid < 3) s_cnt[tid] = 0;
  if (tid == 0) {
    s_base = -1;
    s_rmin = 0x7fffffff;
    s_rmax = -1;
  }
  const void *input = F.input;
  const int cols = F.cols;
  const uint32_t cols_magic = F.cols_magic;
  const int cols_shift = F.cols_shift;
  const int warp0 = tile0 + r0 * 32;
  // ---- the points of this thread: projection, transform, cylindrical index (independent chains) ----
  RayRecord rec[kProjMaxPts];
  int n_valid = 0, n_inside = 0, n_cast = 0;
#pragma unroll
  for (int j = 0; j < kProjMaxPts; j++) {
    const int i = warp0 + j * 32 + lane;
    rec[j].rho = 0;
    rec[j].z = 0;
    rec[j].t = (uint32_t)i;
    rec[j].phi_flags = 0xffffffffu;
    if (j < pts && i < N) {
      double xs = 0, ys = 0, zs = 0;
      if (kMode != 0) {
        // project_depth, src/mlmap.cpp:329-346 (kMode 1: every pixel, v outer / u inner; kMode 2: the sampled pixels)
        int pix = i;
        uint16_t raw;
        if (kMode == 1) {
          raw = __ldg(reinterpret_cast<const uint16_t *>(input) + i);
        } else {
          const uint2 sp = __ldg(reinterpret_cast<const uint2 *>(input) + i);
          pix = (int)sp.x;
          raw = (uint16_t)sp.y;
        }
        if (raw != 0) {
          // row / column of the pixel by multiply-high (host-built magic, exact for pixel indices < 2^31)
          const int v = cols_magic ? (int)(__umulhi((uint32_t)pix, cols_magic) >> cols_shift) : pix / cols, u = pix - v * cols;
          const double depth = (double)(int)raw * P.inv_factor;
          const double du = (double)__fsub_rn((float)u, P.cx) * depth, dv = (double)__fsub_rn((float)v, P.cy) * depth;
          zs = depth;
          int inside = 0, cast = 0;
          if (!point_to_record_fast(P, F, du * P.inv_fx, dv * P.inv_fy, zs, (uint32_t)i, rec[j], inside, cast)) {
            xs = du / (double)P.fx;  // the reference's own operation order
            ys = dv / (double)P.fy;
            point_to_record(P, F, xs, ys, zs, (uint32_t)i, rec[j], inside, cast);
          }
          n_valid++;
          n_inside += inside;
          n_cast += cast;
        }
      } else {
        const double *xyz = reinterpret_cast<const double *>(input);
        xs = xyz[3 * (size_t)i];
        ys = xyz[3 * (size_t)i + 1];
        zs = xyz[3 * (size_t)i + 2];
        int inside = 0, cast = 0;
        if (!point_to_record_fast(P, F, xs, ys, zs, (uint32_t)i, rec[j], inside, cast))
          point_to_record(P, F, xs, ys, zs, (uint32_t)i, rec[j], inside, cast);
        n_valid++;
        n_inside += inside;
        n_cast += cast;
      }
    }
  }
  __syncthreads();
  // span of the touched work columns, relative to the column of some record of the tile
  int col[kProjMaxPts];
  bool any = false;
#pragma unroll
  for (int j = 0; j < kProjMaxPts; j++) {
    col[j] = rec[j].phi_flags != 0xffffffffu ? work_column(P, rec[j]) : -1;
    any = any || col[j] >= 0;
  }
  if (any && s_base < 0) {
    int c0 = -1;
#pragma unroll
    for (int j = kProjMaxPts - 1; j >= 0; j--) c0 = col[j] >= 0 ? col[j] : c0;
    atomicCAS(&s_base, -1, c0);
  }
  __syncthreads();
  const int base = s_base;
  const int half = nCol >> 1;
  {
    int rlo = 0x7fffffff, rhi = -1;
#pragma unroll
    for (int j = 0; j < kProjMaxPts; j++)
      if (col[j] >= 0) {
        int r = col[j] - base + half;  // in (-nCol/2 .. 3*nCol/2)
        r = r < 0 ? r + nCol : (r >= nCol ? r - nCol : r);
        col[j] = r;
        rlo = min(rlo, r);
        rhi = max(rhi, r);
      }
    rlo = __reduce_min_sync(0xffffffffu, rlo);
    rhi = __reduce_max_sync(0xffffffffu, rhi);
    if (lane == 0 && rhi >= 0) {
      atomicMin(&s_rmin, rlo);
      atomicMax(&s_rmax, rhi);
    }
  }
  __syncthreads();
  const int rmin = s_rmin;
  const int W = s_rmax >= 0 ? s_rmax - rmin + 1 : 0;
  int *s_hist = s_proj + nwarps * W;
  int *s_off = s_hist + W;
  int *s_bnd = s_off + W;
  for (int i = tid; i < (nwarps + 3) * W; i += nthreads) s_proj[i] = 0;
  // directory row of this tile: zero outside the span (the span itself is written at the end)
  uint32_t *dir = D.rec_dir + (size_t)tile * nCol;
  if (W < nCol) {
    if ((nCol & 3) == 0) {
      uint4 *d4 = reinterpret_cast<uint4 *>(dir);
      for (int i = tid; i < (nCol >> 2); i += nthreads) d4[i] = make_uint4(0, 0, 0, 0);
    } else {
      for (int i = tid; i < nCol; i += nthreads) dir[i] = 0;
    }
  }
  __syncthreads();
  // ---- run-length merge + stable rank inside the warp's points ----
  // Consecutive points (in input order) that land in the same awareness cell contribute the same
  // (key, odd) list back to back, so for every key their contributions are adjacent in the key's
  // insertion sequence.  One record with a repeat count is therefore exact for the ordered fold, the
  // first-insert stamps and the (idempotent) ray walk.  Runs are cut at the 32-point rounds and at
  // points without a record.
  int *s_mine = s_proj + warp * W;
  int rank[kProjMaxPts];
#pragma unroll
  for (int j = 0; j < kProjMaxPts; j++) {
    rank[j] = 0;
    if (j >= pts) continue;  // warp-uniform: this warp owns fewer rounds
    const bool has = rec[j].phi_flags != 0xffffffffu;
    const int p_rho = __shfl_up_sync(0xffffffffu, rec[j].rho, 1);
    const int p_z = __shfl_up_sync(0xffffffffu, rec[j].z, 1);
    const uint32_t p_pf = __shfl_up_sync(0xffffffffu, rec[j].phi_flags, 1);
    const bool same = has && lane > 0 && p_pf == rec[j].phi_flags && p_rho == rec[j].rho && p_z == rec[j].z;
    const unsigned sames = __ballot_sync(0xffffffffu, same);
    if (has && !same) {
      const unsigned follow = lane < 31 ? (sames >> (lane + 1)) : 0u;
      const int m = 1 + (__ffs(~follow) - 1);  // consecutive followers that repeat this cell
      rec[j].phi_flags |= (uint32_t)m << kRecCountShift;
      // upper bound of the hit contributions of this record: 1 + 2*min(K(rho), nRho-1-rho)
      if (rec[j].phi_flags & kRecInside)
        atomicAdd(&s_bnd[col[j] - rmin], 1 + 2 * min(__ldg(&P.k_reach[rec[j].rho]), P.nRho - 1 - rec[j].rho));
    } else {
      rec[j].phi_flags = 0xffffffffu;
    }
    // stable rank of the record among the warp's records of the same column (rounds are in point order)
    const bool holds = rec[j].phi_flags != 0xffffffffu;
    const int myphi = holds ? col[j] - rmin : -1 - lane;
    const unsigned peers = __match_any_sync(0xffffffffu, myphi);
    const int before = __popc(peers & ((1u << lane) - 1));
    rank[j] = holds ? s_mine[myphi] + before : 0;
    __syncwarp();
    if (holds && before == 0) s_mine[myphi] += __popc(peers);
    __syncwarp();
  }
  // CTA-level counters
  for (int ofs = 16; ofs > 0; ofs >>= 1) {
    n_valid += __shfl_xor_sync(0xffffffffu, n_valid, ofs);
    n_inside += __shfl_xor_sync(0xffffffffu, n_inside, ofs);
    n_cast += __shfl_xor_sync(0xffffffffu, n_cast, ofs);
  }
  if (lane == 0) {
    if (n_valid) atomicAdd(&s_cnt[0], n_valid);
    if (n_inside) atomicAdd(&s_cnt[1], n_inside);
    if (n_cast) atomicAdd(&s_cnt[2], n_cast);
  }
  __syncthreads();
  // per touched column: exclusive prefix over the warps (warp order == point order) and the tile's total
  for (int p = tid; p < W; p += nthreads) {
    int run = 0;
    for (int w = 0; w < nwarps; w++) {
      const int c = s_proj[w * W + p];
      s_proj[w * W + p] = run;
      run += c;
    }
    s_hist[p] = run;
    s_off[p] = run;
    int c = p + rmin + base - half;  // back to the work column
    c = c < 0 ? c + nCol : (c >= nCol ? c - nCol : c);
    if (run) atomicAdd(&D.phi_hist[c], run);
    if (s_bnd[p]) atomicAdd(&D.phi_bound[c], s_bnd[p]);
  }
  __syncthreads();
  block_exclusive_scan(s_off, W, s_warp);
  // The tile's records are written grouped by work column into its own kProjTile-slot window of rec_lin,
  // with one directory word per (tile, column): offset << 16 | count.  k_column gathers from there.
#pragma unroll
  for (int j = 0; j < kProjMaxPts; j++)
    if (rec[j].phi_flags != 0xffffffffu) {
      const int p = col[j] - rmin;
      D.rec_lin[(size_t)tile0 + s_off[p] + s_mine[p] + rank[j]] = rec[j];
    }
  for (int p = tid; p < W; p += nthreads) {
    int c = p + rmin + base - half;
    c = c < 0 ? c + nCol : (c >= nCol ? c - nCol : c);
    dir[c] = ((uint32_t)s_off[p] << 16) | (uint32_t)s_hist[p];
  }
  if (tid == 0) {
    FrameCounters *fc = D.fc[F.parity];
    if (s_cnt[0]) atomicAdd(&fc->n_points, s_cnt[0]);
    if (s_cnt[1]) atomicAdd(&fc->n_inside, s_cnt[1]);
    if (s_cnt[2]) atomicAdd(&fc->n_cast, s_cnt[2]);
  }
}

template <int kMode>
__global__ void __launch_bounds__(kProjThreads) k_project(MapParams P, DeviceBuffers D, FrameParams F) {
  extern __shared__ int s_proj_dyn[];
  project_tile<kMode>(P, D, F, (int)blockIdx.x, s_proj_dyn);  // the grid is sized for cfg.max_points (graph replay)
}

// ---- K2: one CTA per phi column ------------------------------------------------------------------------
// (a) expand inside records into hit contributions (update_hits), (b) sort them by (cell, insert
// time), (c) fold each cell's contributions in insertion order (update_odds_hashmap), emit the
// distinct hit keys with their first-insert stamps and stage them in the frame-local voxel grid,
// (d) warp-cooperative ray walks into a shared-memory miss bitmap, (e) stage the distinct miss
// cells in the voxel grid.
constexpr int kColThreads = 1024;
constexpr int kColWarps = kColThreads / 32;
constexpr int kRadixBits = 8;
constexpr int kRadixDigits = 1 << kRadixBits;
constexpr int kCellBits = 20;
constexpr int kHalf = kColThreads / 2;  // threads per half-CTA group in k_column's overlapped phases
constexpr int kLongChain = 32;  // contributions per cell from which the fold claims the cell early
constexpr int kMapCap = 4096;  // records per column addressed through the shared-memory index map

// contribution key:  [.. : 12+kbits] cell in column | [12+kbits-1 : 12] record index k in the column
// (records are in point order) | [11:7] substep | [6:0] run length.  Contributions are generated in
// insertion order (k, substep), so a STABLE sort by cell alone yields every cell's insertion sequence.
__device__ __forceinline__ uint64_t contrib_key(int cell, int k, int substep, int reps, int cell_shift) {
  return ((uint64_t)(uint32_t)cell << cell_shift) | ((uint64_t)(uint32_t)k << 12) | ((uint64_t)substep << 7) | (uint64_t)reps;
}

// One stable LSD radix pass over 8 key bits for the whole CTA (src -> dst), keys in shared or
// global memory.  Warp w owns a contiguous chunk; cnt[digit*W + w] after the exclusive scan is the
// output cursor of (digit, warp), so order inside a digit is (warp, position) = input order.
constexpr int kCntStride = kColWarps + 1;                 // +1: (digit, warp) counters of one warp hit 32 banks
constexpr int kCntTotal = kRadixDigits * kCntStride;
constexpr int kCntPerThread = (kCntTotal + kColThreads - 1) / kColThreads;
__device__ __forceinline__ void radix_pass(const uint64_t *src, uint64_t *dst, int n, int shift, int bits, uint32_t *cnt,
                                           uint32_t *warp_sums) {
  const int W = kColWarps, w = threadIdx.x >> 5, lane = lane_id(), tid = threadIdx.x;
  const int chunk = (((n + W - 1) / W) + 31) & ~31;
  const int beg = min(w * chunk, n), end = min(beg + chunk, n);
  const int digits = 1 << bits;                 // <= kRadixDigits; narrower passes clear and scan fewer counters
  const int total = digits * kCntStride;
  for (int i = tid; i < total; i += kColThreads) cnt[i] = 0;
  __syncthreads();
  for (int i = beg + lane; i < end; i += 32)
    atomicAdd(&cnt[(int)((src[i] >> shift) & (digits - 1)) * kCntStride + w], 1u);
  __syncthreads();
  // exclusive scan over the counters in (digit, warp) order: kCntPerThread consecutive entries per thread
  uint32_t v[kCntPerThread], sum = 0;
#pragma unroll
  for (int e = 0; e < kCntPerThread; e++) {
    const int idx = kCntPerThread * tid + e;
    v[e] = idx < total ? cnt[idx] : 0u;
    sum += v[e];
  }
  uint32_t incl = sum;
#pragma unroll
  for (int ofs = 1; ofs < 32; ofs <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, incl, ofs);
    if (lane >= ofs) incl += t;
  }
  if (lane == 31) warp_sums[w] = incl;
  __syncthreads();
  if (w == 0) {
    uint32_t sv = lane < W ? warp_sums[lane] : 0, si = sv;
#pragma unroll
    for (int ofs = 1; ofs < 32; ofs <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, si, ofs);
      if (lane >= ofs) si += t;
    }
    if (lane < W) warp_sums[lane] = si - sv;
  }
  __syncthreads();
  uint32_t run = warp_sums[w] + incl - sum;
#pragma unroll
  for (int e = 0; e < kCntPerThread; e++) {
    const int idx = kCntPerThread * tid + e;
    if (idx < total) cnt[idx] = run;
    run += v[e];
  }
  __syncthreads();
  for (int base = beg; base < end; base += 32) {
    const int i = base + lane;
    const bool ok = i < end;
    const uint64_t key = ok ? src[i] : 0;
    const int d = ok ? (int)((key >> shift) & (digits - 1)) : kRadixDigits + lane;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & ((1u << lane) - 1));
    if (ok) dst[cnt[d * kCntStride + w] + rank] = key;
    __syncwarp();
    if (ok && rank == 0) cnt[d * kCntStride + w] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
}

// ---- resolve / allocate a subbox touched this frame (allocate_ram, include/map_local.h:215-231) ----
// Hash find-or-insert and, for a new subbox, a pop from the free stack.  Blocks on the free stack are
// always in the initial state ('u','u',0.f) — they are initialised when the pool is created and when a
// block is returned — so allocation writes nothing.  Safe to run from many threads at once (one per subbox).
__device__ __forceinline__ void resolve_one(const MapParams &P, const FrameParams &F, DeviceBuffers &D, FrameCounters *fc,
                                            const int ls, const bool rearm_flag) {
  int block = -3;
  int lx = ls % P.lsg_dim_xy, ly = (ls / P.lsg_dim_xy) % P.lsg_dim_xy, lz = ls / (P.lsg_dim_xy * P.lsg_dim_xy);
  int g[3] = {lx + F.lsg_base[0], ly + F.lsg_base[1], lz + F.lsg_base[2]};
  uint64_t key;
  if (!pack_glb(g, key)) {
    fc->error = kErrRange;
  } else {
    uint32_t slot = ht_hash(key) & P.ht_mask;
    bool done = false;
    for (uint32_t probe = 0; probe <= P.ht_mask && !done; probe++) {
      uint64_t k = __ldcg(&D.ht_key[slot]);
      if (k == kEmptyKey) {
        unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long *>(&D.ht_key[slot]),
                                           (unsigned long long)kEmptyKey, (unsigned long long)key);
        if (old == kEmptyKey) {
          int top = atomicSub(D.free_top, 1) - 1;
          if (top < 0) {
            atomicAdd(D.free_top, 1);
            D.ht_val[slot] = -3;  // key stays so the table is consistent; the subbox is unusable
            fc->error = kErrPool;
          } else {
            block = D.free_stack[top];
            D.ht_val[slot] = block;
            atomicAdd(&fc->n_new_blocks, 1);
          }
          done = true;
          break;
        }
        k = (uint64_t)old;
      }
      if (k == key) {
        block = __ldcg(&D.ht_val[slot]);
        // a subbox created while the pool was exhausted stays without a block: every frame that touches it again
        // reports the exhaustion (its updates are dropped), not only the frame that hit it first
        if (block == kBlockUnusable) fc->error = kErrPool;
        done = true;
        break;
      }
      slot = (slot + 1) & P.ht_mask;
    }
    if (!done) fc->error = kErrPool;
  }
  D.lsg_block[ls] = block;
  if (rearm_flag) D.lsg_flag[ls] = 0;
}
// all subboxes on the frame's touched list, one per thread of the given stride
__device__ __forceinline__ void resolve_subboxes(const MapParams &P, const FrameParams &F, DeviceBuffers &D,
                                                 FrameCounters *fc, int first, int stride) {
  const int n = *reinterpret_cast<volatile int *>(&fc->n_touched_sub);
  for (int i = first; i < n; i += stride) resolve_one(P, F, D, fc, __ldcg(&D.touched_sub[i]), true);
}

__device__ __forceinline__ void touch_subbox(const MapParams &P, const FrameParams &F, DeviceBuffers &D,
                                             FrameCounters *fc, const int g[3]) {
  int ls = lsg_index(P, F, g);
  if (ls < 0) {
    fc->error = kErrInternal;
    return;
  }
  if (__ldcg(&D.lsg_flag[ls]) == 0) {
    if (atomicExch(&D.lsg_flag[ls], 1) == 0) {
      int pos = atomicAdd(&fc->n_touched_sub, 1);
      D.touched_sub[pos] = ls;
      // k_frame: the first toucher resolves the subbox on the spot (no resolve phase, one device barrier less);
      // the flag stays up for the rest of the frame and is rearmed by the fusion's tail
      if (F.inline_resolve) resolve_one(P, F, D, fc, ls, false);
    }
  }
}

// Ray walk toward the axis, reference src/map_awareness.cpp:243-275, split in two so that the scalar
// part (rate division + range clamp, once per ray) runs one ray per LANE, and only the marking of
// the <= nRho-2 cells runs one ray per WARP.
struct WalkStart {
  double rate;
  int rho, z;  // start cell after the clamp of :261-265
};
__device__ __forceinline__ WalkStart walk_prepare(const MapParams &P, int rho, int z) {
  WalkStart ws;
  ws.rate = (rho < P.nRho && z >= 0 && z < P.nZ) ? __ldg(&P.rate_table[z * P.nRho + rho]) : ray_rate(P, rho, z);
  if (rho >= P.nRho) {
    z = round_to_int_x86((double)z - (double)(rho - P.nRho + 1) * ws.rate);
    rho = P.nRho - 1;
  }
  ws.rho = rho;
  ws.z = z;
  return ws;
}
// All 32 lanes cooperate on one ray: lane l owns rho step r = 32*w + l; lanes that land in the same
// z row merge into one shared-memory atomicOr (warp-aggregated by __match_any_sync).
__device__ __forceinline__ void walk_mark(const MapParams &P, uint32_t *s_miss, double rate, int rho, int z,
                                          uint32_t *stamp_col, uint32_t t) {
  const int lane = lane_id();
  const double zd = (double)z;
  const int w_top = (rho - 1) >> 5;
  double diff = (double)(rho - (w_top << 5) - lane);  // rho - r for r = 32*w + lane; +32 (exact) per step down
  for (int w = w_top; w >= 0; --w, diff += 32.0) {
    const int r = (w << 5) + lane;
    bool valid = r >= 1 && r <= rho - 1;
    // |v| < 2^31 on every valid lane of a sane ray; round_to_int_x86 handles the rest exactly as x86 would
    const int zc = round_to_int_x86(zd - diff * rate);
    valid = valid && zc >= 0 && zc < P.nZ;
    // exploration mode: first-insert stamp of the miss cell = (point stamp, step along the ray: r = rho-1 first)
    if (stamp_col && valid) atomicMin(&stamp_col[zc * P.nRho + r], t * (uint32_t)P.nRho + (uint32_t)(rho - 1 - r));
    // zc is monotone along the ray, so the lanes of one z row are consecutive: one shuffle + ballot finds the
    // runs, the first lane of a run owns its mask, and the atomic is skipped when the bits are already there
    const int key = valid ? zc : -1;
    const int prev = __shfl_up_sync(0xffffffffu, key, 1);
    const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || key != prev);
    if (valid && (lane == 0 || key != prev)) {
      const unsigned rest = lane < 31 ? heads >> (lane + 1) : 0u;
      const int len = rest ? __ffs(rest) : 32 - lane;
      const unsigned mask = (len >= 32 ? 0xffffffffu : ((1u << len) - 1u)) << lane;
      uint32_t *wp = &s_miss[zc * P.words_per_row + w];
      if ((*reinterpret_cast<volatile uint32_t *>(wp) & mask) != mask) atomicOr(wp, mask);
    }
  }
}
// one prepared ray per lane (need = this lane has one); the warp marks them one after the other
__device__ __forceinline__ void walk_batch(const MapParams &P, uint32_t *s_miss, bool need, int rho, int z,
                                           uint32_t *stamp_col = nullptr, uint32_t t = 0) {
  WalkStart ws;
  ws.rate = 0.0;
  ws.rho = 0;
  ws.z = 0;
  if (need) ws = walk_prepare(P, rho, z);
  unsigned todo = __ballot_sync(0xffffffffu, need);
  while (todo) {
    const int src = __ffs(todo) - 1;
    todo &= todo - 1;
    const double rate = __shfl_sync(0xffffffffu, ws.rate, src);
    const int r0 = __shfl_sync(0xffffffffu, ws.rho, src);
    const int z0 = __shfl_sync(0xffffffffu, ws.z, src);
    const uint32_t t0 = __shfl_sync(0xffffffffu, t, src);
    walk_mark(P, s_miss, rate, r0, z0, stamp_col, t0);
  }
}

// named barrier over `count` threads (the two half-CTA groups of k_column use ids 1 and 2; 0 is __syncthreads)
__device__ __forceinline__ void group_bar(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// CTA-wide compaction of the set bits of bm[w0,w1) into list (entries = word*32 + bit), any order.
__device__ __forceinline__ void compact_bits(const uint32_t *bm, int w0, int w1, uint32_t *list, int *counter, int warp,
                                             int nwarps) {
  const int lane = lane_id();
  for (int wi = w0 + warp; wi < w1; wi += nwarps) {
    const uint32_t bits = bm[wi];
    if (!bits) continue;
    int base = 0;
    if (lane == 0) base = atomicAdd(counter, __popc(bits));
    base = __shfl_sync(0xffffffffu, base, 0);
    if ((bits >> lane) & 1u) list[base + __popc(bits & ((1u << lane) - 1))] = ((uint32_t)wi << 5) | (uint32_t)lane;
  }
}

// bytes of k_column's shared memory in front of the two key buffers
__host__ __device__ inline size_t col_smem_prefix_bytes(int col_words, int nRho, int nCol) {
  return (((size_t)2 * col_words + kCntTotal + kColWarps + (size_t)kOddsRows * nRho + nRho + kMapCap) * 4 + (size_t)nCol * 2 + 15) & ~(size_t)15;
}

#ifdef MLM_PHASE_TIMING
#define MLM_PHASE(i) do { __syncthreads(); if (threadIdx.x == 0) D.debug_cycles[vc * 16 + (i)] = clock64(); } while (0)
#define MLM_PHASE_G(i, leader) do { if (threadIdx.x == (leader)) D.debug_cycles[vc * 16 + (i)] = clock64(); } while (0)
#define MLM_WALL(i) do { if (threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); D.debug_cycles[vc * 16 + (i)] = (long long)t_; } } while (0)
// per-CTA timeline of the fused frame (rows nCol + blockIdx.x of the debug buffer)
#define MLM_FRAME_WALL(i) do { if (threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); D.debug_cycles[(P.nCol + blockIdx.x) * 16 + (i)] = (long long)t_; } } while (0)
#else
#define MLM_FRAME_WALL(i) do { } while (0)
#define MLM_WALL(i) do { } while (0)
#define MLM_PHASE(i) do { } while (0)
#define MLM_PHASE_G(i, leader) do { } while (0)
#endif

// One work item (a phi column or one of its halves), start to finish, by the whole CTA.
// exploration mode, split layouts: first-insert stamp of a miss-list entry whose cell lies in the sensor row, once every
// column of the frame has walked (the stamp is the minimum over the walks of both halves of the column)
constexpr uint32_t kMissStampPending = 0xffffffffu;
__device__ __forceinline__ void miss_finalize_body(const MapParams &P, DeviceBuffers &D, const FrameParams &F) {
  if (!P.explore || !P.split) return;
  const FrameCounters *fc = D.fc[F.parity];
  const int n = __ldcg(&fc->n_miss_list);
  const int per_z = P.nRho * P.nPhi;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
    if (__ldcg(&D.miss_t[j]) != kMissStampPending) continue;
    const int idx = __ldcg(&D.miss_idx[j]);                       // mapIdx = (z * nPhi + phi) * nRho + r
    const int z = idx / per_z, rem = idx - z * per_z;
    const int phi = rem / P.nRho, r = rem - phi * P.nRho;
    const uint32_t st = __ldcg(&D.miss_stamp[((size_t)phi * P.nZ + z) * P.nRho + r]);
    D.miss_t[j] = st;
    atomicMin(&D.act_miss[F.parity][__ldcg(&D.miss_bucket[j])], st);
  }
}

// item < nCol: work column `item`; item >= nCol (split layouts only): the two halves of phi column item - nCol worked as
// ONE whole column (the queue merges the lightest columns when there are more active halves than CTAs: a second round of
// items costs more than the few larger ones).  The halves feed disjoint hit cells, so concatenating their records is exact.
__device__ __forceinline__ void column_item(const MapParams &P, DeviceBuffers &D, const FrameParams &F, const int item,
                                            unsigned char *s_raw) {
  FrameCounters *fc = D.fc[F.parity];
  uint32_t *act = D.act[F.parity];
  // work column: a phi column, or one of its two halves (records below / at-or-above the sensor row n_below)
  const bool merged = P.split && item >= P.nCol;
  const int phi = merged ? item - P.nCol : (P.split ? item >> 1 : item);
  const int side = (P.split && !merged) ? (item & 1) : -1;
  const int vc = merged ? 2 * phi : item;   // first (or only) work column of the item
  const int vc2 = merged ? vc + 1 : -1;
  // miss-bitmap rows this CTA owns outright, and the one row (n_below) both halves mark: rays of either half
  // end at the sensor row, so that row goes to global memory with atomicOr and whoever sets a bit first stages it
  const int z_own_lo = side == 1 ? P.n_below + 1 : 0;
  const int z_own_hi = side == 0 ? P.n_below : P.nZ;
  const int z_shared = side >= 0 ? P.n_below : -1;
  const int tid = threadIdx.x;
  const int n_c = D.phi_hist[vc] + (merged ? D.phi_hist[vc2] : 0);
  uint32_t *g_miss = D.miss_bitmap + (size_t)phi * P.col_words;
  MLM_PHASE(15);
  MLM_WALL(13);
  // shared memory: [miss bitmap][end-cell bitmap][radix counters][warp sums][odds table][k_reach][record index map][keys A][keys B]
  uint32_t *s_miss = reinterpret_cast<uint32_t *>(s_raw);
  uint32_t *s_end = s_miss + P.col_words;
  uint32_t *s_cnt = s_end + P.col_words;
  uint32_t *s_wsum = s_cnt + kCntTotal;
  float *s_odds = reinterpret_cast<float *>(s_wsum + kColWarps);
  int *s_reach = reinterpret_cast<int *>(s_odds + kOddsRows * P.nRho);
  int *s_map = s_reach + P.nRho;
  uint64_t *s_keys = reinterpret_cast<uint64_t *>(s_raw + col_smem_prefix_bytes(P.col_words, P.nRho, P.nCol));
  // exploration mode: per-column stamp arrays (earliest point stamp per end cell, first-insert stamp per miss cell)
  uint32_t *end_t_col = P.explore ? D.end_t + (size_t)phi * P.nZ * P.nRho : nullptr;
  uint32_t *stamp_col = P.explore ? D.miss_stamp + (size_t)phi * P.nZ * P.nRho : nullptr;
  if (P.explore) {
    // rows of this item.  Split layouts: the end cells of the sensor row belong to the upper half; the miss stamps of that
    // row are written by the walks of BOTH halves, so nobody resets them here (frame_finish leaves them reset)
    const int e_lo = side == 1 ? P.n_below : z_own_lo;
    for (int i = e_lo * P.nRho + tid; i < z_own_hi * P.nRho; i += blockDim.x) end_t_col[i] = 0xffffffffu;
    for (int i = z_own_lo * P.nRho + tid; i < z_own_hi * P.nRho; i += blockDim.x)
      if (!P.split || i < P.n_below * P.nRho || i >= (P.n_below + 1) * P.nRho) stamp_col[i] = 0xffffffffu;
  }
  // ---- locate this column's records in the per-CTA windows k_project wrote (replaces a scatter pass):
  // s_map[k] = index into rec_lin of the column's k-th record
  __shared__ int s_warp[33];
  __shared__ int s_off;
  const int bound_c = D.phi_bound[vc] + (merged ? D.phi_bound[vc2] : 0);   // upper bound of this item's hit contributions
  const bool in_smem = bound_c <= P.sort_cap_smem;       // sort buffer in shared memory, else global spill (slow, exact)
  const bool big = n_c > P.map_cap;                      // more records than the shared-memory index map holds
  int off = 0;
  if (big || !in_smem) {
    // rare: first slot of this column in the global spill / record areas = records of the columns before it
    int part = 0;
    for (int p = tid; p < vc; p += blockDim.x) part += D.phi_hist[p];
    for (int ofs = 16; ofs > 0; ofs >>= 1) part += __shfl_xor_sync(0xffffffffu, part, ofs);
    if (tid == 0) s_off = 0;
    __syncthreads();
    if (lane_id() == 0 && part) atomicAdd(&s_off, part);
    __syncthreads();
    off = s_off;
  }
  {
    const int nb = (F.n_total + F.tile_pts - 1) / F.tile_pts;   // tiles of the projection
    const int per = (nb + (int)blockDim.x - 1) / (int)blockDim.x;
    const int b0 = min(tid * per, nb), b1 = min(b0 + per, nb);
    uint32_t dsave[4], dsave2[4];
    int mine = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      dsave[q] = 0;
      dsave2[q] = 0;
      if (b0 + q < b1) {
        dsave[q] = __ldcg(&D.rec_dir[(size_t)(b0 + q) * P.nCol + vc]);
        mine += (int)(dsave[q] & 0xffffu);
        if (merged) {
          dsave2[q] = __ldcg(&D.rec_dir[(size_t)(b0 + q) * P.nCol + vc2]);
          mine += (int)(dsave2[q] & 0xffffu);
        }
      }
    }
    for (int b = b0 + 4; b < b1; b++) {
      mine += (int)(__ldcg(&D.rec_dir[(size_t)b * P.nCol + vc]) & 0xffffu);
      if (merged) mine += (int)(__ldcg(&D.rec_dir[(size_t)b * P.nCol + vc2]) & 0xffffu);
    }
    // exclusive scan of `mine` over threads (thread order == CTA order)
    int incl = mine;
    const int lane = lane_id(), w = tid >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int ofs = 1; ofs < 32; ofs <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, incl, ofs);
      if (lane >= ofs) incl += t;
    }
    if (lane == 31) s_warp[w] = incl;
    __syncthreads();
    if (w == 0) {
      int sv = lane < nw ? s_warp[lane] : 0, si = sv;
#pragma unroll
      for (int ofs = 1; ofs < 32; ofs <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, si, ofs);
        if (lane >= ofs) si += t;
      }
      if (lane < nw) s_warp[lane] = si - sv;
    }
    __syncthreads();
    int dst = s_warp[w] + incl - mine;
    for (int b = b0; b < b1; b++) {
      for (int half = 0; half < (merged ? 2 : 1); half++) {
        const int col = half ? vc2 : vc;
        const uint32_t d = b - b0 < 4 ? (half ? dsave2[b - b0] : dsave[b - b0]) : __ldcg(&D.rec_dir[(size_t)b * P.nCol + col]);
        const int c = (int)(d & 0xffffu);
        const int src = b * F.tile_pts + (int)(d >> 16);
        for (int r = 0; r < c; r++) {
          if (big) D.rec_col[off + dst + r] = D.rec_lin[src + r];  // oversized column: materialise the records
          else s_map[dst + r] = src + r;
        }
        dst += c;
      }
    }
  }
  __syncthreads();
  const RayRecord *recs = big ? D.rec_col + off : D.rec_lin;
#define REC_AT(i) recs[big ? (i) : s_map[i]]
  MLM_PHASE(0);

  __shared__ int s_nk;
  __shared__ int s_nmiss;
  __shared__ int s_nhead;
  __shared__ int s_nlist;
  for (int i = tid; i < 2 * P.col_words; i += blockDim.x) s_miss[i] = 0;
  if (tid == 0) {
    s_nk = 0;
    s_nmiss = 0;
    s_nhead = 0;
  }
  __syncthreads();
  uint64_t *keys = in_smem ? s_keys : D.col_scratch + (size_t)2 * off * P.contrib_per_point;
  uint64_t *keys_alt = in_smem ? s_keys + P.sort_cap_smem : keys + (size_t)n_c * P.contrib_per_point;
  int kbits = 1;
  while ((1 << kbits) < n_c) kbits++;
  const int cell_shift = 12 + kbits;
  const int cell_sentinel = 1 << P.cell_bits;  // sorts behind every real cell
  __syncthreads();

  MLM_PHASE(1);
  // (a) contributions, update_hits src/map_awareness.cpp:135-171.  Record k of the column (point order)
  // owns a fixed window of 1 + 2*min(K(rho), nRho-1-rho) slots at the prefix sum of the windows before
  // it, so the contribution array is generated in insertion order (k, substep); neighbours that fall
  // outside the z range leave a sentinel.
  int *s_pos = reinterpret_cast<int *>(keys_alt);
  for (int i = tid; i < n_c; i += blockDim.x) {
    const RayRecord rc = REC_AT(i);
    s_pos[i] = (rc.phi_flags & kRecInside) ? 1 + 2 * min(s_reach[rc.rho], P.nRho - 1 - rc.rho) : 0;
  }
  __syncthreads();
  const int n_k = block_exclusive_scan(s_pos, n_c, s_warp);  // == bound_c
  for (int i = tid; i < n_c; i += blockDim.x) {
    const RayRecord rc = REC_AT(i);
    if (!(rc.phi_flags & kRecInside)) continue;
    const int rho = rc.rho, z = rc.z;
    const int reps = (int)((rc.phi_flags >> kRecCountShift) & kRecCountMask);
    if (P.visibility_check) atomicOr(&s_end[z * P.words_per_row + (rho >> 5)], 1u << (rho & 31));
    if (P.explore) atomicMin(&end_t_col[z * P.nRho + rho], rc.t);
    const int dmax = min(s_reach[rho], P.nRho - 1 - rho);
    int pos = s_pos[i];
    const int c0 = z * P.nRho + rho;
    keys[pos++] = contrib_key(c0, i, 0, reps, cell_shift);
    // z rows of the neighbour contributions: (int)round(z +/- d*rate), tabulated per end cell by the host
    const short2 *dzr = P.dz_table + (size_t)c0 * P.maxK - 1;
    for (int d = 1; d <= dmax; d++) {
      const short2 e = __ldg(&dzr[d]);
      const int zp = e.x, zm = e.y;
      keys[pos++] = contrib_key(zp >= 0 ? zp * P.nRho + rho + d : cell_sentinel, i, 2 * d - 1, reps, cell_shift);
      keys[pos++] = contrib_key(zm >= 0 ? zm * P.nRho + rho - d : cell_sentinel, i, 2 * d, reps, cell_shift);
    }
  }
  __syncthreads();

  MLM_PHASE(2);
  // (b) stable LSD radix sort by cell only: bits [cell_shift, cell_shift + cell_bits + 1)
  {
    // cell_bits + 1 key bits (the sentinel sorts last) in the fewest passes of equal width
    const int sort_bits = P.cell_bits + 1;
    const int passes = (sort_bits + kRadixBits - 1) / kRadixBits;
    const int pass_bits = (sort_bits + passes - 1) / passes;
    const int hi_bit = cell_shift + sort_bits;
    for (int shift = cell_shift; shift < hi_bit; shift += pass_bits) {
      radix_pass(keys, keys_alt, n_k, shift, pass_bits, s_cnt, s_wsum);
      uint64_t *t = keys;
      keys = keys_alt;
      keys_alt = t;
    }
  }
  const uint64_t k_mask = (1ull << kbits) - 1;

  MLM_PHASE(3);
  // From here the CTA works as two halves with their own named barriers: warps 0-15 detect the cell
  // segments, fold them and stage the hit keys; warps 16-31 run the ray walks (which only need the
  // records and the end-cell bitmap).  They meet again before the miss staging.
  const int nFold = kHalf;  // an adaptive split (768/256 by contributions per record) was measured: no gain at CFG-A, slower LiDAR scans
  const int nWalk = kColThreads - nFold;
  if (tid < nFold) {
    // (c1) ordered list of segment heads (first contribution of every distinct cell) and a compact decode
    // of every contribution, both in the idle ping-pong buffer:
    //   s_head[h]  = index into keys of the h-th cell's first contribution
    //   s_dec[i]   = odds-table index (25 bits) | run length - 1 (5 bits, bits 25..29) | last-of-cell (bit 30);
    //                after the fold, s_dec[s_head[h]] holds the folded probability bits of cell h
    uint32_t *s_head = reinterpret_cast<uint32_t *>(keys_alt);
    uint32_t *s_dec = s_head + n_k;
    {
      // one pass, heads compacted in any order (the fold and the staging do not care which thread gets which cell)
      const int lane = lane_id();
      for (int base = tid & ~31; base < n_k; base += nFold) {
        const int i = base + lane;
        bool head = false;
        if (i < n_k) {
          const uint64_t ki = keys[i];
          const int cell = (int)(ki >> cell_shift);
          if (cell != cell_sentinel) {
            head = i == 0 || (int)(keys[i - 1] >> cell_shift) != cell;
            const bool last = i + 1 >= n_k || (int)(keys[i + 1] >> cell_shift) != cell;
            int zq = (int)__umulhi((uint32_t)cell, P.nRho_magic);
            int rk = cell - zq * P.nRho;
            if (rk >= P.nRho) rk -= P.nRho;  // never taken for cell < 2^20, nRho < 2^12; kept for safety
            const int sstep = (int)((ki >> 7) & 31);
            const int d = sstep == 0 ? 0 : ((sstep & 1) ? (sstep + 1) >> 1 : -(sstep >> 1));
            const uint32_t oi = (uint32_t)((kDiffRange + d) * P.nRho + (rk - d));
            s_dec[i] = oi | ((uint32_t)((ki & 127) - 1) << 25) | (last ? (1u << 30) : 0u);
          }
        }
        const unsigned hb = __ballot_sync(0xffffffffu, head);
        if (hb) {
          int pos = 0;
          if (lane == 0) pos = atomicAdd(&s_nhead, __popc(hb));
          pos = __shfl_sync(0xffffffffu, pos, 0);
          if (head) s_head[pos + __popc(hb & ((1u << lane) - 1))] = (uint32_t)i;
        }
      }
    }
    group_bar(1, nFold);
    MLM_PHASE_G(4, 0);
    // (c2) update_odds_hashmap fold, one thread per distinct cell (static: head h -> thread h, so the
    // lanes of a warp stay in one loop).  The chain p <- 1-(1-p)(1-odd) is inherently ordered; it is
    // flattened over (contribution, repeat) so that a lane never waits for another lane's run length,
    // the next contribution is fetched one step ahead, and a lane leaves as soon as p saturates at 1
    // (1 - (1-1)*(1-odd) == 1 for every later contribution).
    {
      const int n_head = s_nhead;
      // dense, static assignment (head h -> thread h).  With few warps in flight every dependent
      // instruction costs ~5 cycles, so the loop is written for instruction count: a tight 3-op repeat
      // loop per contribution, entries pre-decoded (s_dec), the next entry and its odds fetched ahead.
      auto fold_chain = [&](const uint32_t *heads, uint32_t *dec) {
        for (int h = tid; h < n_head; h += nFold) {
          const int i0 = (int)heads[h];
          int i = i0;
          uint32_t e = dec[i];
          float p = s_odds[e & 0x1ffffffu];  // first insert: hit_idx_odds_hashmap[key] = odd
          int reps = (int)((e >> 25) & 31);  // remaining repeats of the first contribution
          float c1 = __fsub_rn(1.0f, p);     // (1 - odd)
          for (;;) {
            const bool last = (e >> 30) & 1u;
            // next entry and its (1 - odd), independent of p
            const uint32_t en = last ? 0u : dec[i + 1];
            const float c1n = __fsub_rn(1.0f, s_odds[en & 0x1ffffffu]);
            for (int r = 0; r < reps; r++) p = __fsub_rn(1.0f, __fmul_rn(__fsub_rn(1.0f, p), c1));
            if (last || p == 1.0f) break;    // p == 1: 1 - (1-1)*(1-odd) == 1 for every later contribution
            e = en;
            c1 = c1n;
            reps = (int)((e >> 25) & 31) + 1;
            i++;
          }
          dec[i0] = __float_as_uint(p);
        }
      };
      if (in_smem) {
        // same buffers, but addressed through the shared-memory window so the loads are LDS, not generic LD
        uint32_t *sh = reinterpret_cast<uint32_t *>(keys_alt == s_keys ? s_keys : s_keys + P.sort_cap_smem);
        fold_chain(sh, sh + n_k);
      } else {
        fold_chain(s_head, s_dec);
      }
    }
    group_bar(1, nFold);
    MLM_PHASE_G(5, 0);
    {
      const int n_head = s_nhead;
      int base_idx = 0;
      if (tid == 0) s_nk = atomicAdd(&fc->n_hit, n_head);  // one global reservation per column
      group_bar(1, nFold);
      base_idx = s_nk;
      for (int k = tid; k < n_head; k += nFold) {
        const uint64_t k0 = keys[s_head[k]];
        const int cell = (int)(k0 >> cell_shift);
        const int zk = cell / P.nRho, rk = cell - zk * P.nRho;
        // first-insert stamp of the key: point stamp t of the record * 32 + substep
        const uint32_t stamp = (REC_AT((int)((k0 >> 12) & k_mask)).t << 5) | (uint32_t)((k0 >> 7) & 31);
        const int idx = base_idx + k;
        if (idx >= P.max_hits) {
          fc->error = kErrCapacity;
          continue;
        }
        D.hit_key[idx] = (zk * P.nPhi + phi) * P.nRho + rk;  // mapIdx, map_awareness.h:81-84
        D.hit_p[idx] = __uint_as_float(s_dec[s_head[k]]);
        D.hit_t[idx] = stamp;
        // bucket activation stamp (libstdc++ iteration order, SURVEY Appendix B)
        const uint32_t bucket = libstdcxx_bucket_fast(vector_hash3(rk, phi, zk), F.bucket_count, F.bucket_c64);
        D.hit_bucket[idx] = bucket;
        atomicMin(&act[bucket], stamp);
        // p_w = T_wa * centre  (identity rotation: one add per axis), src/map_local.cpp:151
        double2 cxy = __ldg(&P.centre_xy[phi * P.nRho + rk]);
        CellRef cr = locate_cell(P, cxy.x + F.t_wa[0], cxy.y + F.t_wa[1], __ldg(&P.centre_z[zk]) + F.t_wa[2]);
        int lv = lvg_index(P, F, cr);
        if (lv < 0) {
          fc->error = kErrInternal;
          D.hit_next[idx] = kLvgEmpty;
          continue;
        }
        int old = atomicExch(&D.lvg[lv].x, idx);
        D.hit_next[idx] = old;
        // sharded staging: voxels of subboxes another rank owns go to their own list (the push kernel sends them away),
        // the others are staged exactly as on one GPU
        const bool remote = F.stage_only && subbox_owner(cr.g, F.shard_world) != F.shard_rank;
        if (old == kLvgEmpty) {
          if (!remote) {
            int tp = agg_inc(&fc->n_touched);
            if (tp < P.max_touched) D.touched[tp] = (uint32_t)lv | kTouchedHitTag; else fc->error = kErrCapacity;
          } else {
            int tp = agg_inc(&fc->n_touched_remote);
            if (tp < P.max_touched) D.touched_remote[tp] = (uint32_t)lv | kTouchedHitTag; else fc->error = kErrCapacity;
          }
        }
        if (!remote) touch_subbox(P, F, D, fc, cr.g);
      }
    }
    group_bar(1, nFold);
    MLM_PHASE_G(8, 0);
  } else {
    // scratch of the walk group: the radix counters are idle now -> [hash set of outside rays][end-cell list]
    uint32_t *s_hash = s_cnt;
    const int hcap = 4096;
    uint32_t *s_list = s_cnt + hcap;
    const int list_cap = kCntTotal - hcap;
    const int words_per_chunk = max(1, list_cap >> 5);   // a chunk of words can never overflow the list
    const int gt = tid - nFold;                          // thread index inside the walk group

    // (d) ray walks, src/map_awareness.cpp:241-275
    if (P.visibility_check) {
      const int warp = gt >> 5, nwarps = nWalk >> 5;
      // distinct inside end cells: each walks once (the walk depends only on (rho,phi,z))
      for (int w0 = 0; w0 < P.col_words; w0 += words_per_chunk) {
        if (gt == 0) s_nlist = 0;
        group_bar(2, nWalk);
        compact_bits(s_end, w0, min(w0 + words_per_chunk, P.col_words), s_list, &s_nlist, warp, nwarps);
        group_bar(2, nWalk);
        const int n_list = s_nlist;
        // entry (it*32 + lane)*nwarps + warp: every warp gets the same share of the list
        for (int it = 0; it * 32 * nwarps < n_list; it++) {
          const int k = (it * 32 + lane_id()) * nwarps + warp;
          int rho = 0, z = 0;
          if (k < n_list) {
            const uint32_t e = s_list[k];
            const int wi = (int)(e >> 5), wr = wi - (wi / P.words_per_row) * P.words_per_row;
            z = wi / P.words_per_row;
            rho = (wr << 5) + (int)(e & 31);
          }
          walk_batch(P, s_miss, k < n_list, rho, z, stamp_col,
                     (P.explore && k < n_list) ? end_t_col[z * P.nRho + rho] : 0u);
        }
        group_bar(2, nWalk);
      }
      // castable points outside the awareness range walk from the clamped cell (:261-265).  Records
      // with identical (rho,z) repeat the same walk: drop them through a small shared-memory set
      // (walks are idempotent, so a missed duplicate only costs time).
      for (int i = gt; i < hcap; i += nWalk) s_hash[i] = 0xffffffffu;
      group_bar(2, nWalk);
      MLM_PHASE_G(9, nFold);
      for (int it = 0; it * 32 * nwarps < n_c; it++) {
        const int i = (it * 32 + lane_id()) * nwarps + warp;
        RayRecord rc;
        rc.phi_flags = kRecInside;
        if (i < n_c) rc = REC_AT(i);
        bool need = !(rc.phi_flags & kRecInside);
        if (need && !P.explore && rc.rho < 65536 && rc.z >= -32768 && rc.z < 32768) {
          const uint32_t key = ((uint32_t)rc.rho << 16) | (uint32_t)(rc.z + 32768);
          uint32_t slot = (key * 2654435761u) >> 7;
          for (int probe = 0; probe < 8; probe++) {
            slot &= (uint32_t)(hcap - 1);
            uint32_t old = atomicCAS(&s_hash[slot], 0xffffffffu, key);
            if (old == 0xffffffffu) break;
            if (old == key) {
              need = false;
              break;
            }
            slot++;
          }
        }
        walk_batch(P, s_miss, need, rc.rho, rc.z, stamp_col, rc.t);
      }
      group_bar(2, nWalk);
      MLM_PHASE_G(12, nFold);
    }
  }
#ifdef MLM_PHASE_TIMING
#endif
  __syncthreads();

  MLM_PHASE(6);
  // (e) distinct miss cells -> voxel grid staging (one cell per thread); bitmap to global for export.
  // The sorted keys are dead now: the key area is the scratch for the compacted cell list.
  // First key buffer: the compacted cell list of a chunk; second: the voxels the chunk touches first, which go to
  // the frame's touched list with ONE global reservation per chunk (a per-voxel append would put a contended
  // same-address atomic with return on every thread's dependent chain).
  uint32_t *s_list = reinterpret_cast<uint32_t *>(s_keys);
  uint32_t *s_tout = s_list + P.sort_cap_smem * 2;
  __shared__ int s_tcnt, s_tbase, s_rcnt, s_rbase, s_mbase;
  const int list_cap = P.sort_cap_smem * 2;            // 32-bit entries in one key buffer
  const int words_per_chunk = max(1, list_cap >> 5);   // a chunk of words can never overflow the list
  for (int wi = z_own_lo * P.words_per_row + tid; wi < z_own_hi * P.words_per_row; wi += blockDim.x) g_miss[wi] = s_miss[wi];
  if (z_shared >= 0) {
    // cells of the shared row: only the half that sets a bit first keeps it for the staging below
    if (tid < P.words_per_row) {
      const int wi = z_shared * P.words_per_row + tid;
      const uint32_t mine = s_miss[wi];
      if (mine) s_miss[wi] = mine & ~atomicOr(&g_miss[wi], mine);
    }
    __syncthreads();
  }
  const int stage_w0 = min(z_own_lo, z_shared >= 0 ? z_shared : z_own_lo) * P.words_per_row;
  const int stage_w1 = max(z_own_hi, z_shared + 1) * P.words_per_row;
  for (int w0 = stage_w0; w0 < stage_w1; w0 += words_per_chunk) {
    if (tid == 0) {
      s_nk = 0;
      s_tcnt = 0;
      s_rcnt = 0;
    }
    __syncthreads();
    compact_bits(s_miss, w0, min(w0 + words_per_chunk, stage_w1), s_list, &s_nk, tid >> 5, (int)blockDim.x >> 5);
    __syncthreads();
    const int n_list = s_nk;
    if (P.explore) {
      // the chunk's miss cells take a contiguous run of the frame's miss list: ONE reservation per chunk (an atomic per
      // warp on the list's counter, from every CTA, serialises at that address for tens of microseconds per frame)
      if (tid == 0) s_mbase = n_list ? atomicAdd(&fc->n_miss_list, n_list) : 0;
      __syncthreads();
    }
    for (int k = tid; k < n_list; k += blockDim.x) {
      const uint32_t e = s_list[k];
      const int wi = (int)(e >> 5), z = wi / P.words_per_row, wr = wi - z * P.words_per_row;
      const int r = (wr << 5) + (int)(e & 31);
      double2 cxy = __ldg(&P.centre_xy[phi * P.nRho + r]);
      CellRef cr = locate_cell(P, cxy.x + F.t_wa[0], cxy.y + F.t_wa[1], __ldg(&P.centre_z[z]) + F.t_wa[2]);
      int lv = lvg_index(P, F, cr);
      if (P.explore) {
        // per-frame miss list for the ordered exploration passes
        const int idx_cell = (z * P.nPhi + phi) * P.nRho + r;  // mapIdx
        // split layouts: a cell of the sensor row gets its stamp from the walks of both halves, and the other half may
        // still be walking: the entry stays pending until miss_finalize_body (after all columns)
        const bool pending = P.split && z == P.n_below;
        const uint32_t st = pending ? kMissStampPending : stamp_col[z * P.nRho + r];
        const uint32_t bkt = (uint32_t)idx_cell % F.bucket_count_miss;   // identity hash of the size_t key
        if (!pending) atomicMin(&D.act_miss[F.parity][bkt], st);
        const int j = s_mbase + k;
        D.miss_idx[j] = idx_cell;
        D.miss_lv[j] = lv < 0 ? 0 : lv;   // (lv < 0 fails the frame below; the slot stays well-formed)
        D.miss_t[j] = st;
        D.miss_bucket[j] = bkt;
      }
      if (lv < 0) {
        fc->error = kErrInternal;
        continue;
      }
      int old = atomicAdd(&D.lvg[lv].y, 1);
      const bool remote = F.stage_only && subbox_owner(cr.g, F.shard_world) != F.shard_rank;
      if (old == 0) {
        // voxels that stay fill the chunk's list from the front, voxels of other ranks' subboxes from the back
        if (!remote) s_tout[agg_inc(&s_tcnt)] = (uint32_t)lv;
        else s_tout[list_cap - 1 - agg_inc(&s_rcnt)] = (uint32_t)lv;
      }
      if (!remote) touch_subbox(P, F, D, fc, cr.g);
    }
    __syncthreads();
    const int n_t = s_tcnt, n_r = s_rcnt;
    if (tid == 0) {
      s_nmiss += n_list;
      if (n_t) s_tbase = atomicAdd(&fc->n_touched, n_t);
    }
    if (tid == 32 && n_r) s_rbase = atomicAdd(&fc->n_touched_remote, n_r);
    __syncthreads();
    if (n_t) {
      const int tb = s_tbase;
      if (tb + n_t > P.max_touched) fc->error = kErrCapacity;
      for (int i = tid; i < n_t && tb + i < P.max_touched; i += blockDim.x) D.touched[tb + i] = s_tout[i];
    }
    if (n_r) {
      const int rb = s_rbase;
      if (rb + n_r > P.max_touched) fc->error = kErrCapacity;
      for (int i = tid; i < n_r && rb + i < P.max_touched; i += blockDim.x) D.touched_remote[rb + i] = s_tout[list_cap - 1 - i];
    }
    __syncthreads();
  }
  MLM_PHASE(7);
  MLM_WALL(14);
#ifdef MLM_PHASE_TIMING
  if (tid == 0) { D.debug_cycles[vc * 16 + 10] = n_c; D.debug_cycles[vc * 16 + 11] = n_k; }
#endif
  if (tid == 0 && s_nmiss) atomicAdd(&fc->n_miss, s_nmiss);
}

// weight of a work column for the longest-first queue (records dominate the walks, contributions the fold)
__device__ __forceinline__ int column_weight(const DeviceBuffers &D, int vc) { return 4 * D.phi_hist[vc] + D.phi_bound[vc]; }

// Persistent kernel: one CTA per SM pulls work columns, heaviest first, from a queue every CTA derives
// identically (stable counting sort of the per-column weights k_project accumulated), so a depth camera's
// ~80 lit columns (160 halves) spread over all SMs instead of one SM per column.
// The CTA's copies of the odds table and k_reach in shared memory (frame-independent).  The fused frames load them
// while they wait at the barrier behind the projection, whose shared memory they overlap.
__device__ __forceinline__ void load_col_tables(const MapParams &P, unsigned char *s_raw) {
  float *s_odds = reinterpret_cast<float *>(s_raw) + 2 * P.col_words + kCntTotal + kColWarps;
  int *s_reach = reinterpret_cast<int *>(s_odds + kOddsRows * P.nRho);
  for (int i = threadIdx.x; i < kOddsRows * P.nRho; i += blockDim.x) s_odds[i] = __ldg(&P.odds_table[i]);
  for (int i = threadIdx.x; i < P.nRho; i += blockDim.x) s_reach[i] = __ldg(&P.k_reach[i]);
}

__device__ __forceinline__ void column_phase(const MapParams &P, DeviceBuffers &D, const FrameParams &F, unsigned char *s_raw,
                                             bool tables_loaded = false) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  __shared__ int s_item, s_wmax, s_nactive, s_nq;
  __shared__ int s_mh[64];   // merge histogram (below)
  // shared memory: [miss bitmap][end-cell bitmap][radix counters][warp sums][odds table][k_reach][record index map][queue order][keys A][keys B]
  uint16_t *s_order = reinterpret_cast<uint16_t *>(reinterpret_cast<int *>(s_raw) + 2 * P.col_words + kCntTotal + kColWarps +
                                                   kOddsRows * P.nRho + P.nRho + kMapCap);
  uint64_t *s_keys = reinterpret_cast<uint64_t *>(s_raw + col_smem_prefix_bytes(P.col_words, P.nRho, P.nCol));
  if (!tables_loaded) load_col_tables(P, s_raw);
  if (tid < 64) s_mh[tid] = 0;
  if (tid == 0) {
    s_wmax = 0;
    s_nactive = 0;
    s_nq = 0;
  }
  __syncthreads();
  MLM_FRAME_WALL(13);  // tables loaded
  // per work column: records (0 = idle this frame or cast by another rank) and queue weight, loaded once
  int *s_nrec = reinterpret_cast<int *>(s_keys);          // [nCol]; the key buffers are idle until the first item
  int *s_wgt = s_nrec + P.nCol;
  const bool sorted = P.nCol <= P.sort_cap_smem;  // 2 ints per column fit the first key buffer, the keys the second
  auto not_mine = [&](int vc) {
    const int phi = P.split ? vc >> 1 : vc;
    return F.shard_world > 1 && (phi % F.shard_world) != F.shard_rank;  // another rank casts this column
  };
  if (sorted) {
    int my_active = 0;
    for (int vc = tid; vc < P.nCol; vc += blockDim.x) {
      const int n = not_mine(vc) ? 0 : D.phi_hist[vc];
      const int w = n > 0 ? column_weight(D, vc) : 0;
      s_nrec[vc] = n;
      s_wgt[vc] = w;
      if (n > 0) {
        my_active++;
        atomicMax(&s_wmax, w);
      }
    }
    if (my_active) atomicAdd(&s_nactive, my_active);
  }
  __syncthreads();
  MLM_FRAME_WALL(14);  // weights loaded (slots 13-15: the column prologue; 9-12 are k_frame_explore's)
  // More active halves than CTAs would mean another round of items, and even the lightest item costs ~15 us of
  // barrier-separated phases: work the lightest columns whole instead (both halves as ONE item), as many as it takes to
  // get down to one item per CTA.  The heavy columns stay split: the heaviest item bounds the phase.
  // s_nrec afterwards: > 0 half item, < 0 merged item (even slot, -records), kCovered odd slot of a merged column, 0 idle.
  constexpr int kCovered = (int)0x80000000;
  if (sorted && P.split && s_nactive > (int)gridDim.x) {
    __shared__ int s_T, s_need, s_below;
    __shared__ int s_wc[32];
    int sh2 = 0;
    while (((2 * s_wmax) >> sh2) > 63) sh2++;
    for (int phi = tid; phi < P.nPhi; phi += blockDim.x)
      if (s_nrec[2 * phi] > 0 && s_nrec[2 * phi + 1] > 0) atomicAdd(&s_mh[(s_wgt[2 * phi] + s_wgt[2 * phi + 1]) >> sh2], 1);
    __syncthreads();
    if (warp == 0) {
      // one warp over the 64 buckets (two per lane), prefix sums by shuffles
      const int m0 = s_mh[2 * lane], m1 = s_mh[2 * lane + 1];
      int cum = m0 + m1;
#pragma unroll
      for (int ofs = 1; ofs < 32; ofs <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, cum, ofs);
        if (lane >= ofs) cum += t;
      }
      const int c2 = __shfl_sync(0xffffffffu, cum, 31);                 // columns with both halves active
      // Down to one item per CTA when that is possible, else every column whole: with more than one round the total work
      // decides, and a whole column costs less than its two halves.  Measured on CFG-C (360 lit columns, 148 CTAs): all
      // whole 175 us; a mix that fills the rounds exactly 193 us; whole except the columns 1.4x heavier than average
      // 199 us; all halves 210 us.  With 2 ranks (180 columns each): 120 / 135 / 123 us.
      const int need = min(c2, s_nactive - (int)gridDim.x);
      // threshold bucket T: the first whose cumulative count reaches `need` (none when need <= 0)
      const int cum0 = cum - m1;                                          // through bucket 2 * lane
      const unsigned hit = __ballot_sync(0xffffffffu, need > 0 && cum >= need);
      const int L = hit ? __ffs(hit) - 1 : 0;
      const int cum0_L = __shfl_sync(0xffffffffu, cum0, L), m0_L = __shfl_sync(0xffffffffu, m0, L);
      if (lane == 0) {
        const bool first = cum0_L >= need;
        s_T = hit ? (first ? 2 * L : 2 * L + 1) : -1;
        s_below = hit ? (first ? cum0_L - m0_L : cum0_L) : 0;             // candidates in the buckets below T
        s_need = need;
      }
    }
    __syncthreads();
    // exactly `need` columns: every candidate below the threshold bucket, and of the threshold bucket itself the first
    // ones in column order (columns of a LiDAR scan weigh alike: a whole bucket would merge the heavy ones too, and the
    // heaviest item bounds the phase).  Rank in column order: ballots inside a warp, per-warp counts across warps.
    const int T = s_T;
    const int take = s_need - s_below;                                    // how many of bucket T to merge (T < 0: none at all)
    int merged_here = 0, run = 0;
    for (int base = 0; base < P.nPhi; base += blockDim.x) {
      const int phi = base + tid;
      const bool both = phi < P.nPhi && s_nrec[2 * phi] > 0 && s_nrec[2 * phi + 1] > 0;
      const int w = both ? s_wgt[2 * phi] + s_wgt[2 * phi + 1] : 0;
      const int bkt = w >> sh2;
      const unsigned at_t = __ballot_sync(0xffffffffu, both && bkt == T);
      if (lane == 0) s_wc[warp] = __popc(at_t);
      __syncthreads();
      int wsum = lane < (int)(blockDim.x >> 5) ? s_wc[lane] : 0;          // inclusive scan of the warp counts
#pragma unroll
      for (int ofs = 1; ofs < 32; ofs <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wsum, ofs);
        if (lane >= ofs) wsum += t;
      }
      const int rank = run + (warp ? __shfl_sync(0xffffffffu, wsum, warp - 1) : 0) + __popc(at_t & ((1u << lane) - 1));
      run += __shfl_sync(0xffffffffu, wsum, 31);
      if (both && (bkt < T || (bkt == T && rank < take))) {
        s_wgt[2 * phi] = w;
        s_nrec[2 * phi] = -(s_nrec[2 * phi] + s_nrec[2 * phi + 1]);
        s_nrec[2 * phi + 1] = kCovered;
        merged_here++;
        atomicMax(&s_wmax, w);
      }
      __syncthreads();                                                    // s_wc is rewritten by the next chunk
    }
    if (merged_here) atomicSub(&s_nactive, merged_here);
    __syncthreads();
  }
  MLM_FRAME_WALL(15);  // merge done
  auto is_active = [&](int vc) { return sorted ? s_nrec[vc] != 0 : (D.phi_hist[vc] > 0 && !not_mine(vc)); };
  // idle work columns: their own rows of the miss bitmap are empty this frame (spread over the CTAs)
  for (int vc = blockIdx.x; vc < P.nCol; vc += gridDim.x) {
    if (is_active(vc)) continue;
    const int phi = P.split ? vc >> 1 : vc, side = P.split ? (vc & 1) : -1;
    const int z_lo = side == 1 ? P.n_below + 1 : 0, z_hi = side == 0 ? P.n_below : P.nZ;
    uint32_t *g_miss = D.miss_bitmap + (size_t)phi * P.col_words;
    for (int i = z_lo * P.words_per_row + tid; i < z_hi * P.words_per_row; i += blockDim.x) g_miss[i] = 0;
  }
  // queue order: active work columns by descending weight bucket, ties by column index (deterministic, so
  // every CTA holds the same list); one 7-bit radix pass over (63 - bucket | column)
  int n_active = 0;
  if (sorted) {
    n_active = s_nactive;
    int sh = 0;
    while ((s_wmax >> sh) > 63) sh++;
    // one distinct 32-bit key per item, (63 - bucket, column, merged): its rank among the items' keys is its queue position
    // (by bucket, then column).  The items are few (about one per CTA), so counting the smaller keys costs less than a
    // radix pass over every column with its block-wide barriers.
    uint32_t *q_key = reinterpret_cast<uint32_t *>(s_keys + P.sort_cap_smem);   // second key buffer (16-byte aligned)
    for (int vc = tid; vc < P.nCol; vc += blockDim.x) {
      const int nr = s_nrec[vc];
      if (nr != 0 && nr != kCovered)
        q_key[agg_inc(&s_nq)] = ((uint32_t)(63 - (s_wgt[vc] >> sh)) << 24) | ((uint32_t)vc << 1) | (nr < 0 ? 1u : 0u);
    }
    if (tid < 3) q_key[n_active + tid] = 0xffffffffu;      // pad to whole uint4s (never smaller than a key)
    __syncthreads();
    const uint4 *q4 = reinterpret_cast<const uint4 *>(q_key);
    for (int i = tid; i < n_active; i += blockDim.x) {
      const uint32_t k = q_key[i];
      int rank = 0;
      for (int j = 0; j < (n_active + 3) >> 2; j++) {
        const uint4 q = q4[j];
        rank += (q.x < k) + (q.y < k) + (q.z < k) + (q.w < k);
      }
      const int vc = (int)((k >> 1) & 0x7fffffu);
      s_order[rank] = (uint16_t)((k & 1u) ? P.nCol + (vc >> 1) : vc);
    }
  } else {
    n_active = P.nCol;  // more work columns than the sort scratch holds: plain column order, idle ones skipped below
  }
  MLM_FRAME_WALL(7);  // queue ready
  bool first_round = true;
  for (;;) {
    __syncthreads();  // the previous item is done with shared memory; s_order is in place
    // the first item of every CTA needs no ticket: items [0, gridDim) are dealt by block index, the queue continues after them
    if (tid == 0) s_item = first_round ? (int)blockIdx.x : atomicAdd(D.col_queue, 1) + (int)gridDim.x;
    first_round = false;
    __syncthreads();
    const int item = s_item;
    if (item >= n_active) break;
    const int vc = sorted ? (int)s_order[item] : item;
    if (!sorted && !is_active(vc)) continue;
    column_item(P, D, F, vc, s_raw);
  }
}

__global__ void __launch_bounds__(kColThreads, 1) k_column(MapParams P, DeviceBuffers D, FrameParams F) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  FrameCounters *fc = D.fc[F.parity];
  const int tid = threadIdx.x;
  __shared__ int s_last;
  column_phase(P, D, F, s_raw);
  // the last CTA to run dry resolves the touched subboxes for k_fuse and rearms the queue
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(D.col_ticket, 1) == (int)gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    if (tid == 0) {
      *D.col_ticket = 0;
      *D.col_queue = 0;
    }
    __threadfence();
    if (!F.stage_only) resolve_subboxes(P, F, D, fc, threadIdx.x, blockDim.x);
  }
}

// libstdc++ _Prime_rehash_policy growth chain (SURVEY Appendix B), mirrored by the host in mlmap_capi.cu
constexpr int kBucketChainLen = 24;
__device__ __constant__ uint32_t c_bucket_chain[kBucketChainLen] = {
    1,      13,     29,      59,      127,     257,      541,      1109,     2357,     5087,     10273,   20753,
    42043,  85229,  172933,  351061,  712697,  1447153,  2938679,  5967347,  12117689, 24607243, 49969847, 101473717};

// frame counters -> mapped pinned host memory (zero-copy store; visible to the host after the stream sync)
__device__ __forceinline__ void publish_counters(const DeviceBuffers &D, FrameCounters *fc, uint32_t frame_seq = 0) {
  // called by one whole warp: lane i moves word i (independent L2 reads and PCIe writes, not a serial chain)
  const int lane = threadIdx.x & 31;
  const int n = (int)(sizeof(FrameCounters) / sizeof(int)) - 1;   // all words but the sequence number
  for (int i = lane; i < n; i += 32) reinterpret_cast<volatile int *>(D.host_fc)[i] = __ldcg(reinterpret_cast<const int *>(fc) + i);
  // the sequence number goes last, behind a system-scope fence: a host that polls it (instead of waiting for the stream
  // to drain) finds the counters of that frame complete
  __syncwarp();
  if (lane == 0 && frame_seq) {
    __threadfence_system();
    *reinterpret_cast<volatile uint32_t *>(&D.host_fc->seq) = frame_seq;
  }
}

// ---- K5: clamped log-odds fusion, one thread per touched cell (map_local.cpp:147-207) ---------------
constexpr int kFuseLocal = 16;
// a frame that crosses a libstdc++ rehash leaves the device untouched after staging: every CTA takes a ticket so that the
// last one can rearm the launch-scoped counters safely, flags the frame and hands the counters to the host
__device__ __forceinline__ void frame_bail(const DeviceBuffers &D, FrameCounters *fc, const FrameParams &F) {
  __shared__ int s_ovf_last;
  if (threadIdx.x == 0) {
    s_ovf_last = atomicAdd(D.fuse_ticket, 1) == (int)gridDim.x - 1;
    if (s_ovf_last) {
      *D.fuse_ticket = 0;
      *D.grid_bar = 0;
      fc->overflow = 1;
      __threadfence();
    }
  }
  __syncthreads();
  if (s_ovf_last && threadIdx.x < 32) publish_counters(D, fc, F.frame_seq);
}

__device__ __forceinline__ void frame_finish(const MapParams &P, DeviceBuffers &D, const FrameParams &F, FrameCounters *fc, int n_hit_frame);

// kPhase 0: hits then misses (normal mode).  Exploration mode splits the pass so that update_observation can
// look at the neighbours' state between them: kPhase 1 = hits only (LVG left intact), kPhase 2 = misses only.
template <int kPhase, bool kFinish = true>
__device__ __forceinline__ void fuse_body(const MapParams &P, DeviceBuffers &D, const FrameParams &F) {
  if (F.skip_flag && __ldcg(F.skip_flag)) return;  // sharded scan that needs the rehash path: nothing may be consumed yet
  FrameCounters *fc = D.fc[F.parity];
  const uint32_t *act = D.act[F.parity];
  const int n_hit_frame = fc->n_hit;
  // a frame that crosses a libstdc++ rehash needs the slow ordering pass first (host re-launches)
  if (kPhase == 0 && F.order_mode == 0 && n_hit_frame > (int)F.bucket_count) {
    frame_bail(D, fc, F);
    return;
  }
  const int n = min(fc->n_touched, P.max_touched);
  const int dxy = P.lvg_dim_xy;
  const unsigned long long kClaimed64 = (unsigned long long)(uint32_t)kLvgClaimed;  // {head = claimed, miss = 0}
  const unsigned long long kEmpty64 = (unsigned long long)(uint32_t)kLvgEmpty;      // {head = empty,   miss = 0}
  int my_touched = 0, my_obs = 0;
  // entries are dealt warp by warp round-robin over the CTAs: every SM gets its share of the dependent chains
  // (with contiguous blocks only the first ~40 % of the SMs had work: 82.6 -> 76.6 us per CFG-A frame)
  const int fw_ = (int)(threadIdx.x >> 5), fl_ = (int)(threadIdx.x & 31);
  for (int i = ((fw_ * (int)gridDim.x + (int)blockIdx.x) << 5) + fl_; i < n; i += (int)gridDim.x * (int)blockDim.x) {
    const uint32_t e = D.touched[i];
    if (e == 0xffffffffu) continue;  // sharded ingest: a record whose voxel was staged by an earlier record
    const int lv = (int)(e & ~kTouchedHitTag);
    // subbox of this cell (independent of the claim below, so its load overlaps the atomic)
    int c[3], g[3], sub;
    {
      // lv -> (x, y, z) of the voxel grid and the subbox split, all by multiply-high (no integer division on this path)
      const int lz = (int)fast_div((uint32_t)lv, P.dxy2_mul, P.dxy2_shift);
      const int rem = lv - lz * dxy * dxy;
      const int ly = (int)fast_div((uint32_t)rem, P.dxy_mul, P.dxy_shift);
      c[0] = rem - ly * dxy + F.lvg_base[0];
      c[1] = ly + F.lvg_base[1];
      c[2] = lz + F.lvg_base[2];
      int l[3];
      for (int a = 0; a < 3; a++) {
        g[a] = fast_floor_div(c[a], P.n, P.n_mul, P.n_shift);
        l[a] = c[a] - g[a] * P.n;
      }
      sub = (l[2] * P.n + l[1]) * P.n + l[0];
    }
    const int ls = lsg_index(P, F, g);
    const int block = ls >= 0 ? __ldcg(&D.lsg_block[ls]) : -3;
    // A cell with both hits and misses appears twice in the touched list.  The first thread to swap in
    // the claimed marker owns the cell (and gets head + miss count in one 64-bit exchange); the other
    // one only restores the empty marker.
    unsigned long long *slot = reinterpret_cast<unsigned long long *>(&D.lvg[lv]);
    int head, mc;
    bool counted_by_hits = false;  // kPhase 2: the hits-only phase already counted this cell as touched
    if (kPhase == 1) {
      // hits-only phase: only the hit entry of a cell works, and the staging stays for the miss phase
      if (!(e & kTouchedHitTag)) continue;
      head = D.lvg[lv].x;
      mc = 0;
    } else {
      const unsigned long long old = atomicExch(slot, kClaimed64);
      head = (int)(uint32_t)old;
      mc = (int)(old >> 32);
      if (head == kLvgClaimed) {
        *slot = kEmpty64;
        continue;
      }
      if (!(head != kLvgEmpty && mc > 0)) *slot = kEmpty64;  // single entry: restore ourselves
      if (kPhase == 2) {
        counted_by_hits = head != kLvgEmpty;
        head = kLvgEmpty;  // hits were applied by the hits-only phase
        D.lvg_tkey[lv] = 0ull;
      }
    }
    if (block < 0) continue;  // collapsed subbox (allocate_ram false) or pool error
    const size_t addr = (size_t)block * P.cell_stride + sub;
    float lo = D.pool_lo[addr];
    char occ = D.pool_occ[addr];
    if (!counted_by_hits) my_touched++;
    bool became_o = false, became_f = false;

    // hits in the reference's unordered_map iteration order: descending (bucket activation, insert stamp).
    // Up to 4 hits per cell are ordered in registers; longer lists use selection by repeated traversal.
    if (head != kLvgEmpty) {
      uint64_t st0 = 0, st1 = 0, st2 = 0, st3 = 0;
      float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
      int cnt = 0;
      // one walk over the list: only the next-pointer load is on the dependent chain, the node's stamp and
      // probability loads overlap the following hop; entries 4..15 wait in a local array
      uint64_t ls[kFuseLocal];
      float lp[kFuseLocal];
      for (int h = head; h != kLvgEmpty; h = D.hit_next[h]) {
        if (cnt < kFuseLocal) {
          const uint64_t st = ((uint64_t)act[D.hit_bucket[h]] << 32) | D.hit_t[h];
          const float ph = D.hit_p[h];
          if (cnt == 0) { st0 = st; p0 = ph; }
          else if (cnt == 1) { st1 = st; p1 = ph; }
          else if (cnt == 2) { st2 = st; p2 = ph; }
          else if (cnt == 3) { st3 = st; p3 = ph; }
          else { ls[cnt] = st; lp[cnt] = ph; }
        }
        cnt++;
      }
      auto apply_hit = [&](float ph) {  // src/map_local.cpp:157-171
        if (lo < P.lo_max) {
          lo = __fadd_rn(lo, logit_f(ph, P.log10f_fma));
          lo = lo > P.lo_max ? P.lo_max : lo;
        }
        if (lo > P.lo_sh && occ != 'o') {
          occ = 'o';
          my_obs++;
          became_o = true;
        }
      };
      if (cnt <= 4) {
        // descending sorting network on (stamp, p); unused slots have stamp 0 and sink to the end
#define MLM_CSWAP(sa, pa, sb, pb) if (sa < sb) { uint64_t ts = sa; sa = sb; sb = ts; float tp = pa; pa = pb; pb = tp; }
        MLM_CSWAP(st0, p0, st1, p1) MLM_CSWAP(st2, p2, st3, p3) MLM_CSWAP(st0, p0, st2, p2)
        MLM_CSWAP(st1, p1, st3, p3) MLM_CSWAP(st1, p1, st2, p2)
#undef MLM_CSWAP
        apply_hit(p0);
        if (cnt > 1) apply_hit(p1);
        if (cnt > 2) apply_hit(p2);
        if (cnt > 3) apply_hit(p3);
      } else if (cnt <= kFuseLocal) {
        // 5..16 hits (near walls, where several thin cylindrical cells share a voxel): insertion sort of the
        // collected entries by stamp, applied in descending order
        ls[0] = st0; lp[0] = p0;
        ls[1] = st1; lp[1] = p1;
        ls[2] = st2; lp[2] = p2;
        ls[3] = st3; lp[3] = p3;
        for (int m = 1; m < cnt; m++) {
          const uint64_t st = ls[m];
          const float ph = lp[m];
          int j = m;
          while (j > 0 && ls[j - 1] < st) {
            ls[j] = ls[j - 1];
            lp[j] = lp[j - 1];
            j--;
          }
          ls[j] = st;
          lp[j] = ph;
        }
        for (int k = 0; k < cnt; k++) apply_hit(lp[k]);
      } else {
        uint64_t prev = ~0ull;
        for (int k = 0; k < cnt; k++) {
          uint64_t best = 0;
          int hb = -1;
          for (int q = head; q != kLvgEmpty; q = D.hit_next[q]) {
            const uint64_t st = ((uint64_t)act[D.hit_bucket[q]] << 32) | D.hit_t[q];
            if (st < prev && (hb < 0 || st > best)) {
              best = st;
              hb = q;
            }
          }
          prev = best;
          apply_hit(D.hit_p[hb]);
        }
      }
    }
    // misses: every miss cell mapping here applies the same step (src/map_local.cpp:188-203)
    for (int k = 0; k < mc; k++) {
      bool changed = false;
      if (lo >= P.lo_min) {
        float nl = __fadd_rn(lo, P.lo_miss);
        nl = nl < P.lo_min ? P.lo_min : nl;
        changed = nl != lo;
        lo = nl;
      }
      if (lo < P.lo_sh && occ != 'f') {
        occ = 'f';
        changed = true;
        became_f = true;
      }
      if (!changed) break;  // fixed point: the remaining identical steps are no-ops
    }
    D.pool_lo[addr] = lo;
    D.pool_occ[addr] = occ;
    // frontier.erase(subbox_id) on either transition (src/map_local.cpp:167-168,200-201)
    if (P.explore && (became_o || became_f))
      atomicAnd(&D.pool_front[(size_t)block * P.front_words + (sub >> 5)], ~(1u << (sub & 31)));
  }
  // counters: warp shuffle, then shared memory, then ONE global atomic per CTA and counter (thousands of same-address
  // atomics, one per warp, are paid for at a few ns each at the kernel's end)
  __shared__ int s_ctr[2];
  if (threadIdx.x < 2) s_ctr[threadIdx.x] = 0;
  __syncthreads();
  for (int ofs = 16; ofs > 0; ofs >>= 1) {
    my_touched += __shfl_xor_sync(0xffffffffu, my_touched, ofs);
    my_obs += __shfl_xor_sync(0xffffffffu, my_obs, ofs);
  }
  if (lane_id() == 0) {
    if (my_touched) atomicAdd(&s_ctr[0], my_touched);
    if (my_obs) atomicAdd(&s_ctr[1], my_obs);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_ctr[0]) atomicAdd(&fc->n_touched_voxels, s_ctr[0]);
    if (s_ctr[1]) atomicAdd(&fc->obs_delta, s_ctr[1]);
  }
  if (kPhase == 1 || !kFinish) return;  // the miss phase finishes the frame (the fused exploration frame: after its release pass)
  frame_finish(P, D, F, fc, n_hit_frame);
}

// end of a frame: counters to the host, launch-scoped counters rearmed, the NEXT frame's scratch reset
__device__ __forceinline__ void frame_finish(const MapParams &P, DeviceBuffers &D, const FrameParams &F, FrameCounters *fc, int n_hit_frame) {
  if (blockIdx.x == 0 && threadIdx.x == 0) fc->fused = 1;
  // the last block to get here publishes the frame counters to the host (no memcpy node in the graph)
  {
    __shared__ int s_is_last;
    __threadfence();
    __syncthreads();
    MLM_FRAME_WALL(8);
    if (threadIdx.x == 0) s_is_last = atomicAdd(D.fuse_ticket, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (s_is_last && threadIdx.x < 32) {
      if (threadIdx.x == 0) {
        *D.fuse_ticket = 0;
        *D.grid_bar = 0;  // every CTA of a k_frame launch is past its last barrier once it has taken a ticket
        fc->fused = 1;
        __threadfence();
      }
      __syncwarp();
      publish_counters(D, fc, F.frame_seq);
    }
  }

  // ---- reset of the NEXT frame's scratch (double-buffered, nothing below is read by this launch) ----
  {
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    // bucket count the hit map will have at the start of the next frame (clear() keeps the buckets)
    uint32_t B = F.bucket_count;
    const uint32_t n_hit = (uint32_t)n_hit_frame;
    if (n_hit > 0 && B == 1) B = 13;
    for (int c = 0; c + 1 < kBucketChainLen && n_hit > B; c++)
      if (c_bucket_chain[c] == B) B = c_bucket_chain[c + 1];
    uint32_t *act_next = D.act[F.parity ^ 1];
    for (uint32_t i = gtid; i < B; i += nth) act_next[i] = 0xffffffffu;
    if (P.explore) {
      uint32_t Bm = F.bucket_count_miss;
      const uint32_t n_miss = (uint32_t)fc->n_miss_list;
      if (n_miss > 0 && Bm == 1) Bm = 13;
      for (int c = 0; c + 1 < kBucketChainLen && n_miss > Bm; c++)
        if (c_bucket_chain[c] == Bm) Bm = c_bucket_chain[c + 1];
      uint32_t *am = D.act_miss[F.parity ^ 1];
      for (uint32_t i = gtid; i < Bm; i += nth) am[i] = 0xffffffffu;
    }
    if (F.inline_resolve) {
      const int nts = fc->n_touched_sub;
      for (int i = gtid; i < nts; i += nth) D.lsg_flag[__ldcg(&D.touched_sub[i])] = 0;
    }
    for (int i = gtid; i < P.nCol; i += nth) {
      D.phi_hist[i] = 0;
      D.phi_bound[i] = 0;
    }
    if (P.explore && P.split)   // miss stamps of the sensor row (both halves of a column write them; this frame is done with them)
      for (int i = gtid; i < P.nPhi * P.nRho; i += nth) {
        const int phi = i / P.nRho, r = i - phi * P.nRho;
        D.miss_stamp[((size_t)phi * P.nZ + P.n_below) * P.nRho + r] = 0xffffffffu;
      }
    if (gtid < (int)(sizeof(FrameCounters) / sizeof(int))) reinterpret_cast<int *>(D.fc[F.parity ^ 1])[gtid] = 0;
  }
}

template <int kPhase>
__global__ void __launch_bounds__(256) k_fuse(MapParams P, DeviceBuffers D, FrameParams F) {
  fuse_body<kPhase>(P, D, F);
}

// ---- the whole frame as ONE cooperative launch: projection tiles, work columns, subbox resolve, fusion ----
// One CTA per SM stays resident through the four phases; device-wide barriers replace three kernel
// boundaries (each boundary costs a drain, a launch and a ramp-up that together outweigh the phase's own
// tail on a ~70 us frame).  The barrier is a monotone counter in global memory: arrive with a release
// add, spin on an acquire load; the last CTA through k_fuse's completion ticket rearms it.
// Split in arrive / wait so that a CTA can do work that does not depend on the other CTAs in between.
__device__ __forceinline__ void grid_arrive(int *counter) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1);
  }
}
__device__ __forceinline__ void grid_wait(int *counter, int target) {
  if (threadIdx.x == 0) {
    int v;
    do {
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    } while (v < target);
    __threadfence();
  }
  __syncthreads();
}
__device__ __forceinline__ void grid_barrier(int *counter, int target) {
  grid_arrive(counter);
  grid_wait(counter, target);
}

template <int kMode>
__global__ void __launch_bounds__(kColThreads, 1) k_frame(MapParams P, DeviceBuffers D, FrameParams F) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  const int G = (int)gridDim.x;
  MLM_FRAME_WALL(0);
  // (1) projection: tile t of F.tile_pts points -> CTA t % G
  {
    const int n_tiles = (F.n_total + F.tile_pts - 1) / F.tile_pts;
    for (int t = blockIdx.x; t < max(n_tiles, 1); t += G) {
      project_tile<kMode>(P, D, F, t, reinterpret_cast<int *>(s_raw));
      __syncthreads();
    }
  }
  MLM_FRAME_WALL(1);
  grid_arrive(D.grid_bar);
  load_col_tables(P, s_raw);   // the projection is done with shared memory (the loop's last barrier)
  grid_wait(D.grid_bar, G);
  MLM_FRAME_WALL(2);
  // (2) work columns (awareness update + staging into the frame-local voxel grid)
  column_phase(P, D, F, s_raw, true);
  MLM_FRAME_WALL(3);
  grid_barrier(D.grid_bar, 2 * G);
  MLM_FRAME_WALL(4);
  MLM_FRAME_WALL(5);
  // (3) the touched subboxes were resolved / allocated by their first toucher (F.inline_resolve)
  if (blockIdx.x == 0 && threadIdx.x == 0) *D.col_queue = 0;
  // (4) clamped log-odds fusion, next frame's resets, counters to the host
  fuse_body<0>(P, D, F);
  MLM_FRAME_WALL(6);
}

}  // namespace mlm
