// Batched point queries, box fill, inflation and map export kernels.  Replaces the reference's
//   mlmap::getOccupancy / getOdd / getOddGrad / getInflateOccupancy   include/mlmap.h:142-295
//   mlmap::setFree_map_in_bound                                        src/mlmap.cpp:388-407
// One thread per query; the subbox hash table and pool blocks are read-only here.
#pragma once
#include "frame_kernels.cuh"

namespace mlm {

// logit_inv, include/mlmap.h:40: pow(10, x) / (1 + pow(10, x)) in double, returned as float.  10^x through exp10
// (1 ulp in double, a third of pow's instructions).  Moving 10^x by one double ulp either way changes the float result
// for no float x with 2^-28 <= |x| <= 64 (tests/test_query_grad_host.py scans every one; below 2^-28 the odd is 0.5),
// so getOdd equals glibc's bit for bit wherever exp10 keeps its documented bound
__device__ __forceinline__ float logit_inv_f(float lo) {
  double y = exp10((double)lo);
  return (float)(y / (1 + y));
}

// getOdd(glb, sub), include/mlmap.h:227-235
__device__ __forceinline__ float odd_at(const MapParams &P, const DeviceBuffers &D, const int g[3], int sub) {
  uint32_t slot;
  int block = ht_find_slot(P, D, g, slot);
  if (block == kBlockCollapsed) return logit_inv_f(D.col_lo[slot]);  // log_odds.size() == 1 -> element 0
  if (block < 0) return 0.5f;
  return logit_inv_f(D.pool_lo[(size_t)block * P.cell_stride + sub]);
}

__device__ __forceinline__ int occupancy_at(const MapParams &P, const DeviceBuffers &D, double x, double y,
                                            double z) {  // include/mlmap.h:170-193
  CellRef c = locate_cell(P, x, y, z);
  uint32_t slot;
  int block = ht_find_slot(P, D, c.g, slot);
  char res;
  if (block == kBlockCollapsed) res = D.col_occ[slot];  // occupancy.size() == 1 -> element 0
  else if (block < 0) return -1;
  else res = D.pool_occ[(size_t)block * P.cell_stride + c.sub];
  return res == 'o' ? 0 : (res == 'f' ? 1 : -1);
}

__global__ void __launch_bounds__(256) k_get_occupancy(MapParams P, DeviceBuffers D, const double *pos, size_t n,
                                                       int *out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = occupancy_at(P, D, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
}

// getOccupancy(pos, inflate): 19-point stencil, include/mlmap.h:142-169 (short-circuit order kept
// only as far as the result is concerned: any OCCUPIED probe -> OCCUPIED)
__global__ void __launch_bounds__(256) k_get_occupancy_inflate(MapParams P, DeviceBuffers D, const double *pos,
                                                               size_t n, float inflate, int *out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x = pos[3 * i], y = pos[3 * i + 1], z = pos[3 * i + 2];
  const double f = (double)inflate, m = (double)(-inflate);
  const double off[19][3] = {{0, 0, 0}, {0, 0, f}, {0, 0, m}, {0, f, 0}, {0, m, 0}, {f, 0, 0}, {m, 0, 0},
                             {m, f, 0}, {m, m, 0}, {f, f, 0}, {f, m, 0}, {0, m, f}, {0, m, m}, {0, f, f},
                             {0, f, m}, {m, 0, f}, {m, 0, m}, {f, 0, f}, {f, 0, m}};
  int res = 1;
  for (int k = 0; k < 19; k++) {
    if (occupancy_at(P, D, x + off[k][0], y + off[k][1], z + off[k][2]) == 0) {
      res = 0;
      break;
    }
  }
  out[i] = res;
}

__global__ void __launch_bounds__(256) k_get_inflate_occupancy(MapParams P, DeviceBuffers D, const double *pos,
                                                               size_t n, int *out) {  // mlmap.h:195-211
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  CellRef c = locate_cell(P, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
  int block = ht_find(P, D, c.g);
  int r = -1;
  if (block >= 0 && D.pool_inf[(size_t)block * P.cell_stride + c.sub] == 'o') r = 0;
  out[i] = r;
}

__global__ void __launch_bounds__(256) k_get_odd(MapParams P, DeviceBuffers D, const double *pos, size_t n,
                                                 float *out) {  // mlmap.h:213-225
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  CellRef c = locate_cell(P, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]);
  out[i] = odd_at(P, D, c.g, c.sub);
}

// getOdd(const Vec3I &glb_id, size_t subbox_id), include/mlmap.h:227-235
__global__ void __launch_bounds__(256) k_get_odd_at(MapParams P, DeviceBuffers D, const int *glb3, const int *sub, size_t n, float *out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int g[3] = {glb3[3 * i], glb3[3 * i + 1], glb3[3 * i + 2]};
  out[i] = odd_at(P, D, g, sub[i]);
}

// sampled project_depth on a device image (src/mlmap.cpp:321-346): tries[t].x = pixel index of try t (v*cols + u from the
// rand() stream).  A try is executed while fewer than cnt_max valid pixels have been collected; the valid pixels of the
// executed tries are compacted in order into pairs {pixel, raw depth}; info = {points, tries executed}.  One CTA.
__global__ void __launch_bounds__(1024) k_sample_gather(const uint16_t *img, const uint2 *tries, int max_iter, int cnt_max,
                                                        uint2 *pairs, int *info) {
  __shared__ int s_warp[33];
  __shared__ int s_carry, s_tries;
  if (threadIdx.x == 0) {
    s_carry = 0;
    s_tries = -1;
  }
  __syncthreads();
  for (int base = 0; base < max_iter; base += blockDim.x) {
    const int t = base + threadIdx.x;
    unsigned pix = 0;
    uint16_t raw = 0;
    if (t < max_iter) {
      pix = tries[t].x;
      raw = img[pix];
    }
    const int valid = raw != 0 ? 1 : 0;
    // inclusive count of valid pixels up to try t
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int incl = valid;
#pragma unroll
    for (int ofs = 1; ofs < 32; ofs <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, ofs);
      if (lane >= ofs) incl += v;
    }
    if (lane == 31) s_warp[w] = incl;
    __syncthreads();
    if (w == 0) {
      int sv = s_warp[lane], si = sv;
#pragma unroll
      for (int ofs = 1; ofs < 32; ofs <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, si, ofs);
        if (lane >= ofs) si += v;
      }
      s_warp[lane] = si - sv;
      if (lane == 31) s_warp[32] = si;
    }
    __syncthreads();
    const int upto = s_carry + s_warp[w] + incl;   // valid pixels among tries 0..t
    // try t runs iff fewer than cnt_max valid pixels were collected before it
    if (t < max_iter && upto - valid < cnt_max) {
      if (valid) pairs[upto - 1] = make_uint2(pix, (unsigned)raw);
      if (valid && upto == cnt_max) s_tries = t + 1;   // the try that fills the quota is the last one executed
    }
    __syncthreads();
    if (threadIdx.x == 0) s_carry += s_warp[32];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    info[0] = min(s_carry, cnt_max);
    info[1] = s_tries >= 0 ? s_tries : max_iter;
  }
}

// subbox_neighbors row i of cell sub (src/map_local.cpp:78-120): order +z,-z,+y,-y,+x,-x
__device__ __forceinline__ void neighbor_step(const MapParams &P, int dir, int g[3], int &sub) {
  int x = sub % P.n, y = (sub / P.n) % P.n, z = sub / (P.n * P.n);
  int c[3] = {x, y, z};
  const int axis = 2 - (dir >> 1);
  c[axis] += (dir & 1) ? -1 : 1;
  if (c[axis] >= P.n) {
    g[axis] += 1;
    c[axis] = 0;
  } else if (c[axis] < 0) {
    g[axis] -= 1;
    c[axis] = P.n - 1;
  }
  sub = (c[2] * P.n + c[1]) * P.n + c[0];
}

// ---- getOddGrad (include/mlmap.h:237-295) ---------------------------------------------------------------------------
// where the log-odds of a subbox live: base + cell * mul (pool block: one float per cell; collapsed subbox: its single
// element, mul 0; absent subbox: no storage, the reference's getOdd answers 0.5 == logit_inv(0.f))
struct GradSource {
  unsigned long long v;   // address of element 0 (4-byte aligned) | mul in bit 0; 0 = absent
  __device__ __forceinline__ bool present() const { return v != 0; }
};
__device__ __forceinline__ GradSource grad_source_key(const MapParams &P, const DeviceBuffers &D, uint64_t key) {
  GradSource s = {0ull};
  uint32_t slot = ht_hash(key) & P.ht_mask;
  for (uint32_t probe = 0; probe <= P.ht_mask; probe++) {
    const uint64_t k = D.ht_key[slot];
    if (k == key) {
      const int block = D.ht_val[slot];
      if (block >= 0) s.v = reinterpret_cast<unsigned long long>(D.pool_lo + (size_t)block * P.cell_stride) | 1ull;
      else if (block == kBlockCollapsed) s.v = reinterpret_cast<unsigned long long>(D.col_lo + slot);
      return s;
    }
    if (k == kEmptyKey) return s;
    slot = (slot + 1) & P.ht_mask;
  }
  return s;
}
__device__ __forceinline__ GradSource grad_source(const MapParams &P, const DeviceBuffers &D, const int g[3]) {
  uint64_t key;
  if (!pack_glb(g, key)) return GradSource{0ull};
  return grad_source_key(P, D, key);
}
__device__ __forceinline__ float grad_lo(const GradSource &s, int sub) {
  if (!s.present()) return 0.0f;
  const float *base = reinterpret_cast<const float *>(s.v & ~3ull);
  return __ldg(base + ((s.v & 1ull) ? sub : 0));
}

#ifndef MLM_GRAD_MINB
#define MLM_GRAD_MINB 4
#endif
__global__ void __launch_bounds__(256, MLM_GRAD_MINB) k_get_odd_grad(MapParams P, DeviceBuffers D, const double *pos, size_t n,
                                                         int max_iter, double *out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double px = pos[3 * i], py = pos[3 * i + 1], pz = pos[3 * i + 2];
  const CellRef c = locate_cell(P, px, py, pz);
  // The six probes walk along +z,-z,+y,-y,+x,-x (subbox_neighbors row order, src/map_local.cpp:78-120): only the
  // coordinate on the probe's own axis changes.  After k steps probe d sits at cell c_axis +- k of the origin's subbox
  // or, once it has left it, of the neighbouring subbox in that direction.  The neighbours a walk of max_iter steps can
  // reach are looked up ONCE, up front, where the whole warp is converged (a lookup inside the walk runs for the two or
  // three lanes that happen to cross a border at that step); their packed keys differ from the origin's in one field.
  const int lim = 1 << 20;
  uint64_t key0 = 0;
  const bool packed = pack_glb(c.g, key0);
  bool inner = packed;   // all six neighbours have a packed key too
#pragma unroll
  for (int a = 0; a < 3; a++) inner = inner && c.g[a] > -lim && c.g[a] < lim - 1;
  const GradSource src0 = packed ? grad_source_key(P, D, key0) : GradSource{0ull};
  const float lo0 = grad_lo(src0, c.sub);
  const int cxyz[3] = {c.sub % P.n, (c.sub / P.n) % P.n, c.sub / (P.n * P.n)};
  const int stride[3] = {1, P.n, P.n * P.n};
  const bool short_walk = max_iter <= P.n;   // a probe leaves at most one subbox behind
  GradSource nb[6];
  bool any_source = src0.present();
  // per axis usually ONE of the two probes can leave the subbox (both only when max_iter exceeds half a subbox): one
  // lookup site per axis serves whichever direction a lane needs, so the warp runs three lookups, not six half-empty ones
#pragma unroll
  for (int h = 0; h < 3; h++) {   // h = d >> 1: z, y, x
    const int axis = 2 - h;
    const bool reach_p = cxyz[axis] + max_iter >= P.n, reach_m = cxyz[axis] - max_iter < 0;
    nb[2 * h] = GradSource{0ull};
    nb[2 * h + 1] = GradSource{0ull};
    auto neighbour = [&](bool minus) {
      if (inner) {
        const uint64_t step = 1ull << (21 * h);   // pack_glb: x at bit 42, y at 21, z at 0
        return grad_source_key(P, D, minus ? key0 - step : key0 + step);
      }
      int g[3] = {c.g[0], c.g[1], c.g[2]};
      g[axis] += minus ? -1 : 1;
      return grad_source(P, D, g);
    };
    if (reach_p || reach_m) {
      const GradSource s = neighbour(!reach_p);
      if (reach_p) nb[2 * h] = s;
      else nb[2 * h + 1] = s;
      any_source = any_source || s.present();
    }
    if (reach_p && reach_m) {
      nb[2 * h + 1] = neighbour(true);
      any_source = any_source || nb[2 * h + 1].present();
    }
  }
  // log-odds of the six neighbours of round k
  auto load_round = [&](int k, float lo_d[6]) {
#pragma unroll
    for (int d = 0; d < 6; d++) {
      const int axis = 2 - (d >> 1);
      int p = cxyz[axis] + ((d & 1) ? -k : k);
      GradSource s = src0;
      if (p >= P.n || p < 0) {
        if (short_walk) {
          p += (d & 1) ? P.n : -P.n;
          s = nb[d];
        } else {
          const int hops = p >= P.n ? p / P.n : -((-p + P.n - 1) / P.n);   // subboxes left behind
          p -= hops * P.n;
          if (hops == 1 || hops == -1) {
            s = nb[d];
          } else {
            int g[3] = {c.g[0], c.g[1], c.g[2]};
            g[axis] += hops;
            s = grad_source(P, D, g);
          }
        }
      }
      lo_d[d] = grad_lo(s, c.sub + (p - cxyz[axis]) * stride[axis]);
    }
  };
  // A round of the reference visits the six neighbours in order and keeps the first one with the strictly lowest odd
  // below the running minimum; a round that finds one ends the search.  logit_inv is monotone non-decreasing in the
  // log-odds (also after the cast to float), so the round's winner is the neighbour with the lowest log-odds (the first
  // of those), unless an EARLIER neighbour with a slightly higher log-odds rounds to the same float odd; those rare
  // near-ties are settled with their own pow.  Below kNearOne every float log-odds with the same float odd as lo_m lies
  // within kTie of it (tests/test_query_grad_host.py computes the first lo_m where this fails: 5.586); closer to odd 1
  // the float odd's spacing of 2^-24 spans more than kTie of log-odds, and below -30 the odd underflows, so there every
  // earlier direction is checked.  The walk itself compares log-odds only: the first round whose minimum lies below the
  // origin's is the candidate, and its odd is computed AFTER the loop, next to the origin's, where the warp is converged
  // again (a pow inside the loop runs for the few lanes whose search ends in that round, once per round).
  const float kTie = 1e-2f, kNearOne = 5.5f;
  float lo_d[6];
  int m = 0, k = max_iter + 1;
  float lo_m = lo0;
  if (any_source || !short_walk)   // (nothing stored within reach: every probe reads 0.5, like the origin)
  {
    for (k = 1; k <= max_iter; k++) {
      load_round(k, lo_d);
      m = 0;
      lo_m = lo_d[0];
#pragma unroll
      for (int d = 1; d < 6; d++)
        if (lo_d[d] < lo_m) {
          lo_m = lo_d[d];
          m = d;
        }
      if (lo_m < lo0) break;
    }
  }
  const bool cand = k <= max_iter;
  const float ori_odd = logit_inv_f(lo0);
  float min_odd = ori_odd;
  float odd_m = logit_inv_f(cand ? lo_m : lo0);
  int best_d = -1, best_k = 0;
  if (cand) {
    // a lower log-odds that rounds to the origin's odd is not strictly lower: the search goes on (a few queries per million)
    while (!(odd_m < min_odd)) {
      bool found = false;
      for (k = k + 1; k <= max_iter && !found; k++) {
        load_round(k, lo_d);
        m = 0;
        lo_m = lo_d[0];
#pragma unroll
        for (int d = 1; d < 6; d++)
          if (lo_d[d] < lo_m) {
            lo_m = lo_d[d];
            m = d;
          }
        found = lo_m < lo0;
      }
      if (!found) break;
      k--;   // the round that was found
      odd_m = logit_inv_f(lo_m);
    }
    if (odd_m < min_odd) {
      min_odd = odd_m;
      best_d = m;
      best_k = k;
      // earlier directions whose log-odds is a hair above the minimum: same float odd -> the reference keeps the earlier one
#pragma unroll
      for (int d = 0; d < 5; d++)
        if (d < m && (lo_d[d] - lo_m <= kTie || lo_m < -30.0f || lo_m > kNearOne) && lo_d[d] < lo0) {
          if (logit_inv_f(lo_d[d]) == odd_m) {
            best_d = d;
            break;
          }
        }
    }
  }
  double gx = 0.0, gy = 0.0, gz = 0.0;
  if (best_d >= 0) {
    const int axis = 2 - (best_d >> 1);
    int p = cxyz[axis] + ((best_d & 1) ? -best_k : best_k);
    const int hops = p >= P.n ? p / P.n : (p < 0 ? -((-p + P.n - 1) / P.n) : 0);
    p -= hops * P.n;
    int best_g[3] = {c.g[0], c.g[1], c.g[2]};
    best_g[axis] += hops;
    int cb[3] = {cxyz[0], cxyz[1], cxyz[2]};
    cb[axis] = p;
    // subbox_id2xyz_glb_vec (map_local.h:208-213) - pos, times (double)(float)(ori - min)
    const double s = (double)__fsub_rn(ori_odd, min_odd);
    gx = ((((double)best_g[0] * P.d_glb + (double)cb[0] * P.d_sub) + P.d_sub_half) - px) * s;
    gy = ((((double)best_g[1] * P.d_glb + (double)cb[1] * P.d_sub) + P.d_sub_half) - py) * s;
    gz = ((((double)best_g[2] * P.d_glb + (double)cb[2] * P.d_sub) + P.d_sub_half) - pz) * s;
  }
  out[3 * i] = gx;
  out[3 * i + 1] = gy;
  out[3 * i + 2] = gz;
}

// setFree_map_in_bound: the per-axis coordinate sequences are generated on the host by repeated
// "+= d" exactly like the reference loops (src/mlmap.cpp:392-396); one thread per (x,y,z) triple.
__global__ void __launch_bounds__(256) k_set_free(MapParams P, DeviceBuffers D, const double *xs, int nx,
                                                  const double *ys, int ny, const double *zs, int nz) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = (size_t)nx * ny * nz;
  if (i >= total) return;
  int iz = (int)(i % nz), iy = (int)((i / nz) % ny), ix = (int)(i / ((size_t)nz * ny));
  CellRef c = locate_cell(P, xs[ix], ys[iy], zs[iz]);
  int block = ht_find(P, D, c.g);
  if (block < 0) return;
  size_t addr = (size_t)block * P.cell_stride + c.sub;
  D.pool_occ[addr] = 'f';
  D.pool_lo[addr] = 0.f;
}

// ---- inflation layer: mlmap::inflate_map (src/mlmap.cpp:286-309) + inflate_atpos (include/map_local.h:233-264) ----
// The reference walks the (2N+1)^3 window of subboxes around the body in a fixed order (x offset outermost,
// then y, then z).  For every window subbox that exists and is not collapsed it first resets
// inflate_occupancy to 'u', then stamps an L1 ball of radius inflate_n around each 'o' cell whose centre is
// above flate_height; stamps cross subbox borders (allocating the neighbour if needed).  A stamp that lands
// in a window subbox processed LATER is wiped by that subbox's reset, so the net effect is:
//   target cell <- 'o'  iff  some source stamps it and NOT (target subbox is in the window, is processed
//   after the source subbox, and exists when the loop gets to it).
// Subboxes created by a stamp exist from then on (allocate_ram), so they count as "exists when reached".
struct InflateArgs {
  int ct_g[3];   // subbox of ct_pos
  int N;         // inflate_global_n
  int r;         // inflate_n
  double height; // flate_height
};
__device__ __forceinline__ int window_order(const InflateArgs &A, const int g[3]) {
  const int W = 2 * A.N + 1;
  const int ox = g[0] - A.ct_g[0] + A.N, oy = g[1] - A.ct_g[1] + A.N, oz = g[2] - A.ct_g[2] + A.N;
  if ((unsigned)ox >= (unsigned)W || (unsigned)oy >= (unsigned)W || (unsigned)oz >= (unsigned)W) return -1;
  return (ox * W + oy) * W + oz;
}
// pass 1: reset the window subboxes that exist; remember their blocks (win_block[order], -1 = absent)
__global__ void __launch_bounds__(256) k_inflate_reset(MapParams P, DeviceBuffers D, InflateArgs A, int *win_block) {
  const int W = 2 * A.N + 1;
  const int w = blockIdx.x;
  if (w >= W * W * W) return;
  int g[3] = {A.ct_g[0] + w / (W * W) - A.N, A.ct_g[1] + (w / W) % W - A.N, A.ct_g[2] + w % W - A.N};
  const int block = ht_find(P, D, g);
  if (threadIdx.x == 0) win_block[w] = block;
  if (block < 0) return;
  for (int i = threadIdx.x; i < P.cells; i += blockDim.x) D.pool_inf[(size_t)block * P.cell_stride + i] = 'u';
}
// pass 2 (ensure) / pass 3 (stamp): one thread per (window subbox, cell); sources are the 'o' cells above the height
template <bool kStamp>
__global__ void __launch_bounds__(256) k_inflate_sources(MapParams P, DeviceBuffers D, InflateArgs A, const int *win_block,
                                                         int *counters /*[0]=new subboxes, [1]=error*/) {
  const int W = 2 * A.N + 1;
  const int w = blockIdx.x;
  if (w >= W * W * W) return;
  const int block = win_block[w];
  if (block < 0) return;  // absent (or collapsed) when the loop reached it: nothing to scan
  int g[3] = {A.ct_g[0] + w / (W * W) - A.N, A.ct_g[1] + (w / W) % W - A.N, A.ct_g[2] + w % W - A.N};
  for (int it = threadIdx.x; it < P.cells; it += blockDim.x) {
    if (D.pool_occ[(size_t)block * P.cell_stride + it] != 'o') continue;
    const int cx = it % P.n, cy = (it / P.n) % P.n, cz = it / (P.n * P.n);
    // subbox_id2xyz_glb_vec(temp_glb, it)(2) > flate_height
    const double zc = ((double)g[2] * P.d_glb + (double)cz * P.d_sub) + P.d_sub_half;
    if (!(zc > A.height)) continue;
    for (int ox = -A.r; ox <= A.r; ox++)
      for (int oy = -A.r; oy <= A.r; oy++)
        for (int oz = -A.r; oz <= A.r; oz++) {
          if (abs(ox) + abs(oy) + abs(oz) > A.r) continue;
          int t[3] = {cx + ox, cy + oy, cz + oz};
          int tg[3] = {g[0], g[1], g[2]};
          bool expanded = false;
          for (int m = 0; m < 3; m++) {
            if (t[m] >= P.n) {
              tg[m] += 1;
              t[m] -= P.n;
              expanded = true;
            } else if (t[m] < 0) {
              tg[m] -= 1;
              t[m] += P.n;
              expanded = true;
            }
          }
          const int tsub = (t[2] * P.n + t[1]) * P.n + t[0];
          if (!kStamp) {
            // ensure pass: allocate_ram(glb_idx_inflate) for expanded targets (find-or-insert, one winner pops a block)
            if (!expanded) continue;
            uint64_t key;
            if (!pack_glb(tg, key)) {
              counters[1] = kErrRange;
              continue;
            }
            uint32_t slot = ht_hash(key) & P.ht_mask;
            for (uint32_t probe = 0; probe <= P.ht_mask; probe++) {
              uint64_t k = D.ht_key[slot];
              if (k == kEmptyKey) {
                unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long *>(&D.ht_key[slot]),
                                                   (unsigned long long)kEmptyKey, (unsigned long long)key);
                if (old == kEmptyKey) {
                  int top = atomicSub(D.free_top, 1) - 1;
                  if (top < 0) {
                    atomicAdd(D.free_top, 1);
                    D.ht_val[slot] = -3;
                    counters[1] = kErrPool;
                  } else {
                    D.ht_val[slot] = D.free_stack[top];
                    atomicAdd(&counters[0], 1);
                  }
                  break;
                }
                k = (uint64_t)old;
              }
              if (k == key) break;
              slot = (slot + 1) & P.ht_mask;
            }
          } else {
            const int t_order = window_order(A, tg);
            if (expanded && t_order > w) continue;  // the target subbox is reset later in the loop: stamp is wiped
            const int tb = expanded ? ht_find(P, D, tg) : block;
            if (tb < 0) continue;                   // collapsed / unusable subbox: allocate_ram returned false
            D.pool_inf[(size_t)tb * P.cell_stride + tsub] = 'o';
          }
        }
  }
}

// ---- map clouds for consumers (reference src/rviz_vis.cpp:267-327, src/mlmap.cpp:200-284) ----------------------
// Whole-map stream compaction: one warp per hash slot; a live subbox is scanned 16 cells per lane and load, the
// selected cells are ranked inside the warp, space for them is reserved with ONE atomicAdd per warp and round,
// and the points go out as float4 {x, y, z, w} = the memory layout of pcl::PointXYZ (include/common.h:53).
//   kind 0: inflate_occupancy == 'o'  (rviz_vis::pub_global_local_map, the map cloud the reference publishes)
//   kind 1: occupancy == 'o'
//   kind 2: the frontier sets         (rviz_vis::pub_frontier)
// A collapsed subbox holds one element per array, so only its cell 0 can qualify (the reference loops over
// vectors of size 1 there).  Point order is unspecified (the reference's is its unordered_map iteration order).
__device__ __forceinline__ float4 cell_point(const MapParams &P, const int g[3], int sub, float w) {
  const int x = sub % P.n, y = (sub / P.n) % P.n, z = sub / (P.n * P.n);
  // subbox_id2xyz_glb, include/map_local.h:201-206: origin*d_glb + xyz*d_sub + d_sub/2 in double, then float
  return make_float4((float)(((double)g[0] * P.d_glb + (double)x * P.d_sub) + P.d_sub_half),
                     (float)(((double)g[1] * P.d_glb + (double)y * P.d_sub) + P.d_sub_half),
                     (float)(((double)g[2] * P.d_glb + (double)z * P.d_sub) + P.d_sub_half), w);
}
__global__ void __launch_bounds__(256) k_export_cloud(MapParams P, DeviceBuffers D, int kind, float4 *out,
                                                      unsigned long long *counter, unsigned long long cap) {
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t slot = warp; slot <= P.ht_mask; slot += nwarps) {
    const uint64_t k = D.ht_key[slot];
    if (k == kEmptyKey) continue;
    const int block = D.ht_val[slot];
    int g[3];
    unpack_glb(k, g);
    if (block == kBlockCollapsed) {
      const bool sel = kind == 0 ? D.col_inf[slot] == 'o' : (kind == 1 ? D.col_occ[slot] == 'o' : false);
      if (sel && lane == 0) {
        const unsigned long long at = atomicAdd(counter, 1ull);
        if (at < cap) out[at] = cell_point(P, g, 0, 1.0f);
      }
      continue;
    }
    if (block < 0) continue;
    if (kind == 2 && !P.explore) continue;
    const char *src = (kind == 0 ? D.pool_inf : D.pool_occ) + (size_t)block * P.cell_stride;
    for (int c0 = 0; c0 < P.cell_stride; c0 += 32 * 16) {
      const int c = c0 + lane * 16;
      uint32_t m = 0;  // bit i: cell c + i selected
      if (c < P.cell_stride) {
        if (kind == 2) {
          // 16 frontier bits of this lane: cells c .. c+15 live in word c/32, half (c/16)&1
          const uint32_t w = D.pool_front[(size_t)block * P.front_words + (c >> 5)];
          m = (w >> (c & 16)) & 0xffffu;
        } else {
          const uint4 v = *reinterpret_cast<const uint4 *>(src + c);
          const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int q = 0; q < 4; q++)
#pragma unroll
            for (int b = 0; b < 4; b++)
              if (((wv[q] >> (8 * b)) & 0xffu) == (uint32_t)'o') m |= 1u << (4 * q + b);
        }
        if (c + 16 > P.cells) m &= (c < P.cells) ? ((1u << (P.cells - c)) - 1u) : 0u;  // padding cells of the block
      }
      const int cnt = __popc(m);
      int incl = cnt;
#pragma unroll
      for (int ofs = 1; ofs < 32; ofs <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, ofs);
        if (lane >= ofs) incl += t;
      }
      const int total = __shfl_sync(0xffffffffu, incl, 31);
      if (total == 0) continue;
      unsigned long long base = 0;
      if (lane == 0) base = atomicAdd(counter, (unsigned long long)total);
      base = __shfl_sync(0xffffffffu, base, 0) + (unsigned long long)(incl - cnt);
      while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        if (base < cap) out[base] = cell_point(P, g, c + b, 1.0f);
        base++;
      }
    }
  }
}
// Horizontal slice of the odds field (mlmap::visualize_odds, src/mlmap.cpp:200-284): every cell whose centre height
// is within 1e-3 of `height` goes out as {x, y, z, odd} with odd = logit_inv(log_odds) (the reference colours the
// marker by it; its gradient lines are getOddGrad at the same points, available through mlm_get_odd_grad).
__global__ void __launch_bounds__(256) k_export_odds_slice(MapParams P, DeviceBuffers D, double height, float4 *out,
                                                           unsigned long long *counter, unsigned long long cap) {
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t slot = warp; slot <= P.ht_mask; slot += nwarps) {
    const uint64_t k = D.ht_key[slot];
    if (k == kEmptyKey) continue;
    const int block = D.ht_val[slot];
    if (block < 0 && block != kBlockCollapsed) continue;
    int g[3];
    unpack_glb(k, g);
    for (int z = 0; z < P.n; z++) {
      const double pz = ((double)g[2] * P.d_glb + (double)z * P.d_sub) + P.d_sub_half;
      if (!(pz < height + 1e-3 && pz > height - 1e-3)) continue;
      const int layer = P.n * P.n;
      for (int i0 = 0; i0 < layer; i0 += 32) {
        const int i = i0 + lane, sub = z * layer + i;
        const bool sel = i < layer && (block != kBlockCollapsed || sub == 0);
        const unsigned sm = __ballot_sync(0xffffffffu, sel);
        if (!sm) continue;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(counter, (unsigned long long)__popc(sm));
        base = __shfl_sync(0xffffffffu, base, 0) + (unsigned long long)__popc(sm & ((1u << lane) - 1));
        if (sel && base < cap) {
          const float lo = block == kBlockCollapsed ? D.col_lo[slot] : D.pool_lo[(size_t)block * P.cell_stride + sub];
          out[base] = cell_point(P, g, sub, logit_inv_f(lo));
        }
      }
    }
  }
}

// ---- export -----------------------------------------------------------------------------------------
__global__ void k_export_list(MapParams P, DeviceBuffers D, int *out_glb3, int *out_block, int *counter, int cap) {
  uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot > P.ht_mask) return;
  uint64_t k = D.ht_key[slot];
  if (k == kEmptyKey) return;
  int block = D.ht_val[slot];
  if (block < 0 && block != kBlockCollapsed) return;
  int idx = atomicAdd(counter, 1);
  if (idx >= cap) return;
  int g[3];
  unpack_glb(k, g);
  out_glb3[3 * idx] = g[0];
  out_glb3[3 * idx + 1] = g[1];
  out_glb3[3 * idx + 2] = g[2];
  out_block[idx] = block == kBlockCollapsed ? -16 - (int)slot : block;
}
// collapsed subboxes export element 0 and zeros elsewhere (blocks[b] <= -16 encodes the hash slot);
// front (optional) receives the frontier bitmask, cells/8 bytes per subbox rounded to front_words*4
__global__ void k_export_blocks(MapParams P, DeviceBuffers D, const int *blocks, int n, char *occ, char *inf,
                                float *lo, unsigned char *collapsed, uint32_t *front) {
  int b = blockIdx.x;
  if (b >= n) return;
  const int blk = blocks[b];
  const size_t dst = (size_t)b * P.cells;
  if (blk <= -16) {
    const int slot = -(blk + 16);
    for (int i = threadIdx.x; i < P.cells; i += blockDim.x) {
      occ[dst + i] = i == 0 ? D.col_occ[slot] : 0;
      inf[dst + i] = i == 0 ? D.col_inf[slot] : 0;
      lo[dst + i] = i == 0 ? D.col_lo[slot] : 0.f;
    }
    if (threadIdx.x == 0) collapsed[b] = 1;
    if (front)
      for (int w = threadIdx.x; w < P.front_words; w += blockDim.x) front[(size_t)b * P.front_words + w] = 0;
    return;
  }
  const size_t src = (size_t)blk * P.cell_stride;
  for (int i = threadIdx.x; i < P.cells; i += blockDim.x) {
    occ[dst + i] = D.pool_occ[src + i];
    inf[dst + i] = D.pool_inf[src + i];
    lo[dst + i] = D.pool_lo[src + i];
  }
  if (threadIdx.x == 0) collapsed[b] = 0;
  if (front)
    for (int w = threadIdx.x; w < P.front_words; w += blockDim.x)
      front[(size_t)b * P.front_words + w] = P.explore ? D.pool_front[(size_t)blk * P.front_words + w] : 0u;
}
// miss set export: ascending awareness indices from the per-column bitmaps
__global__ void k_export_miss(MapParams P, DeviceBuffers D, unsigned long long *out, int *counter, int cap) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= P.nPhi * P.col_words) return;
  uint32_t bits = D.miss_bitmap[w];
  int phi = w / P.col_words, wi = w - phi * P.col_words;
  int z = wi / P.words_per_row, wr = wi - z * P.words_per_row;
  while (bits) {
    int b = __ffs(bits) - 1;
    bits &= bits - 1;
    int idx = atomicAdd(counter, 1);
    if (idx < cap) out[idx] = (unsigned long long)((z * P.nPhi + phi) * P.nRho + (wr << 5) + b);
  }
}

__global__ void k_debug_log10f(const float *x, size_t n, float *out, int use_fma) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = glibc_log10f_sel(x[i], use_fma);
}

__global__ void k_l2_flush(uint4 *buf, size_t n16, uint32_t v) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n16; i += stride) buf[i] = make_uint4(v, v, v, v);
}

}  // namespace mlm
