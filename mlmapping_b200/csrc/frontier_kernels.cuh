// Frontier clustering (mlm_frontier_clusters; no reference counterpart): connected components of the exploration
// frontier sets, with per-cluster size, key cell, bounds and centroid.  The spec is in include/mlmap_b200.h ("frontier
// clustering"); oracle/oracle_frontier.cpp and tests/frontier_spec.py restate it, and the records agree bit for bit.
//
// The frontier set is addressed through the hash table and the bitmasks alone, with no cell-to-index table:
//   k_fc_count     one warp per hash slot: the subbox's frontier words masked to the box (mword), popcount per slot
//   k_fc_scan      one CTA: exclusive scan of the per-slot counts -> the first list index of each subbox
//   k_fc_index     one warp per slot: the first list index of every frontier word (wbase); a cell's index is then
//                  wbase[word] + popc(bits below it), for its own subbox and for a neighbour's alike
//   k_fc_hook      one warp per slot, a lane per word: the 13 forward neighbours of each cell (3 with CONN6), the 26
//                  neighbour subboxes probed once per subbox into shared memory; lock-free hooking of the larger root
//                  onto the smaller (ECL-CC style), so a component's root is its smallest index
//   k_fc_compress  parent[i] = root of i; clears the per-root accumulators
//   k_fc_reduce    integer atomics per root (count, int64 sums, min / max; then the key among the cells on the lowest
//                  z layer): the result does not depend on the order threads run in
//   k_fc_select    the roots with n_cells >= min_cells, and the extent of their keys
//   k_fc_sort      one CTA: stable LSD radix sort of the kept roots by key in (z, y, x) order (one composite key when
//                  the key extent fits 64 bits, else y/x first and z second)
//   k_fc_records   the records and the root -> cluster index map
//   k_fc_labels    per-cell labels, counted per slot, scanned and written in list order (deterministic)
#pragma once
#include "ray_kernels.cuh"

namespace mlm {

constexpr int kFcConn6 = 1;             // MLM_FRONTIER_CONN6
constexpr int kFcScanThreads = 1024;
constexpr int kFcSortThreads = 1024;

struct __align__(8) FrontierCluster {  // memory layout of mlm_frontier_cluster
  int n_cells;
  int key[3];
  int lo[3], hi[3];
  double centroid[3];
};
static_assert(sizeof(FrontierCluster) == 64, "mlm_frontier_cluster is 64 bytes");

struct FcBox {
  int lo[3], hi[3];  // inclusive cell range (the whole int range without a box)
  int whole;         // 1: no box
};

struct FcScratch {
  uint32_t *mword;        // [pool_blocks * front_words] frontier words masked to the box
  int *wbase;             // [pool_blocks * front_words] list index of the first cell of each word
  int *slot_cnt;          // [ht cap + 1] per-slot counts, scanned in place (the total lands at [ht cap])
  int *parent;            // [cells] union-find forest over list indices
  int *acc_n;             // [cells] per root: cluster size
  unsigned long long *acc_s;  // [3 * cells] per root: coordinate sums (int64, two's complement)
  int *acc_lo, *acc_hi;   // [3 * cells] per root: bounds
  unsigned long long *acc_key;  // [cells] per root: (y - lo_y) << 32 | (x - lo_x) of the smallest cell on z = lo_z
  int *map;               // [cells] root -> cluster index (-1: dropped)
  unsigned long long *sk[2];  // [cells] sort keys (ping-pong)
  int *sv[2];             // [cells] sort values: roots (ping-pong)
  int *counters;          // [0] kept clusters [1] cells of kept clusters [2..7] key min/max (z, y, x) [8] sort result buffer
};

__device__ __forceinline__ bool fc_in_box(const FcBox &B, int x, int y, int z) {
  return B.whole || (x >= B.lo[0] && x <= B.hi[0] && y >= B.lo[1] && y <= B.hi[1] && z >= B.lo[2] && z <= B.hi[2]);
}

// frontier bits of word w of a live block, masked to the cells of the subbox and to the box
__device__ __forceinline__ uint32_t fc_masked_word(const MapParams &P, const DeviceBuffers &D, const FcBox &B, int block,
                                                   const int g[3], int w) {
  uint32_t m = D.pool_front[(size_t)block * P.front_words + w];
  const int first = 32 * w;
  if (first + 32 > P.cells) m &= first < P.cells ? (1u << (P.cells - first)) - 1u : 0u;
  if (B.whole || !m) return m;
  const int n = P.n;
  bool inside = true, outside = false;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const long long a = (long long)g[k] * n, e = a + n - 1;
    inside = inside && a >= B.lo[k] && e <= B.hi[k];
    outside = outside || e < B.lo[k] || a > B.hi[k];
  }
  if (inside) return m;
  if (outside) return 0u;
  uint32_t r = 0, t = m;
  while (t) {
    const int b = __ffs(t) - 1;
    t &= t - 1;
    const int sub = first + b;
    if (fc_in_box(B, g[0] * n + sub % n, g[1] * n + (sub / n) % n, g[2] * n + sub / (n * n))) r |= 1u << b;
  }
  return r;
}

// the live, non-collapsed subbox of a hash slot (false for empty slots, collapsed and unusable subboxes)
__device__ __forceinline__ bool fc_slot_block(const MapParams &P, const DeviceBuffers &D, uint32_t slot, int &block, int g[3]) {
  const uint64_t k = D.ht_key[slot];
  if (k == kEmptyKey) return false;
  block = D.ht_val[slot];
  if (block < 0) return false;
  unpack_glb(k, g);
  return true;
}

__device__ __forceinline__ int fc_warp_exclusive(int v, int &total) {
  const int lane = threadIdx.x & 31;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  total = __shfl_sync(0xffffffffu, incl, 31);
  return incl - v;
}

#define FC_WARP_LOOP                                                                               \
  const int lane = threadIdx.x & 31;                                                               \
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5; \
  for (uint32_t slot = warp; slot <= P.ht_mask; slot += nwarps)

__global__ void __launch_bounds__(256) k_fc_count(MapParams P, DeviceBuffers D, FcBox B, FcScratch S) {
  FC_WARP_LOOP {
    int block, g[3];
    if (!fc_slot_block(P, D, slot, block, g)) {
      if (lane == 0) S.slot_cnt[slot] = 0;
      continue;
    }
    int cnt = 0;
    for (int w = lane; w < P.front_words; w += 32) {
      const uint32_t m = fc_masked_word(P, D, B, block, g, w);
      S.mword[(size_t)block * P.front_words + w] = m;
      cnt += __popc(m);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) S.slot_cnt[slot] = cnt;
  }
}

// exclusive scan of a[0..n) in place, the total into a[n]; one CTA
__global__ void __launch_bounds__(kFcScanThreads) k_fc_scan(int *a, int n) {
  __shared__ int s[kFcScanThreads];
  const int t = threadIdx.x, per = (n + kFcScanThreads - 1) / kFcScanThreads;
  const int i0 = min(t * per, n), i1 = min(i0 + per, n);
  int sum = 0;
  for (int i = i0; i < i1; i++) sum += a[i];
  s[t] = sum;
  for (int o = 1; o < kFcScanThreads; o <<= 1) {
    __syncthreads();
    const int v = t >= o ? s[t - o] : 0;
    __syncthreads();
    s[t] += v;
  }
  __syncthreads();
  int run = s[t] - sum;
  for (int i = i0; i < i1; i++) {
    const int v = a[i];
    a[i] = run;
    run += v;
  }
  if (t == kFcScanThreads - 1) a[n] = s[t];
}

__global__ void __launch_bounds__(256) k_fc_index(MapParams P, DeviceBuffers D, FcScratch S) {
  FC_WARP_LOOP {
    int block, g[3];
    if (!fc_slot_block(P, D, slot, block, g)) continue;
    int run = S.slot_cnt[slot];
    for (int w0 = 0; w0 < P.front_words; w0 += 32) {
      const int w = w0 + lane;
      const size_t at = (size_t)block * P.front_words + w;
      const int c = w < P.front_words ? __popc(S.mword[at]) : 0;
      int total;
      const int ex = fc_warp_exclusive(c, total);
      if (w < P.front_words) {
        S.wbase[at] = run + ex;
        for (int j = 0; j < c; j++) S.parent[run + ex + j] = run + ex + j;
      }
      run += total;
    }
  }
}

// root of x with path halving; parents only decrease, so concurrent halving stays in the same tree
__device__ __forceinline__ int fc_find(volatile int *parent, int x) {
  int cur = parent[x];
  if (cur != x) {
    int next, prev = x;
    while (cur > (next = parent[cur])) {
      parent[prev] = next;
      prev = cur;
      cur = next;
    }
  }
  return cur;
}

__device__ __forceinline__ void fc_union(int *parent, int a, int b) {
  int ra = fc_find(parent, a), rb = fc_find(parent, b);
  while (ra != rb) {
    if (ra < rb) {
      const int old = atomicCAS(parent + rb, rb, ra);
      if (old == rb) break;
      rb = fc_find(parent, old);
    } else {
      const int old = atomicCAS(parent + ra, ra, rb);
      if (old == ra) break;
      ra = fc_find(parent, old);
    }
  }
}

template <bool kConn6>
__global__ void __launch_bounds__(256) k_fc_hook(MapParams P, DeviceBuffers D, FcBox B, FcScratch S) {
  __shared__ int s_nb[8][27];  // pool block of each neighbour subbox (-1: none), per warp
  const int wib = threadIdx.x >> 5;
  const int n = P.n, fw = P.front_words;
  FC_WARP_LOOP {
    int block, g[3];
    if (!fc_slot_block(P, D, slot, block, g)) continue;
    if (lane < 27) {
      const int gn[3] = {g[0] + lane % 3 - 1, g[1] + (lane / 3) % 3 - 1, g[2] + lane / 9 - 1};
      const int b = lane == 13 ? block : ht_find(P, D, gn);
      s_nb[wib][lane] = b >= 0 ? b : -1;
    }
    __syncwarp();
    for (int w = lane; w < fw; w += 32) {
      uint32_t m = S.mword[(size_t)block * fw + w];
      int ia = S.wbase[(size_t)block * fw + w];
      while (m) {
        const int bit = __ffs(m) - 1;
        m &= m - 1;
        const int sub = 32 * w + bit;
        const int lx = sub % n, ly = (sub / n) % n, lz = sub / (n * n);
        for (int o = 0; o < (kConn6 ? 3 : 13); o++) {
          // forward offsets: +x, +y, +z (6-connectivity), or the 13 offsets after (0,0,0) in (z, y, x) order
          const int q = 14 + o;  // 14..26 = the offsets (z, y, x) > (0, 0, 0) of the 3x3x3 cube
          int x = lx + (kConn6 ? (o == 0) : q % 3 - 1), y = ly + (kConn6 ? (o == 1) : (q / 3) % 3 - 1),
              z = lz + (kConn6 ? (o == 2) : q / 9 - 1);
          if (!B.whole) {
            const long long cx = (long long)g[0] * n + x, cy = (long long)g[1] * n + y, cz = (long long)g[2] * n + z;
            if (!(cx >= B.lo[0] && cx <= B.hi[0] && cy >= B.lo[1] && cy <= B.hi[1] && cz >= B.lo[2] && cz <= B.hi[2]))
              continue;
          }
          const int sx = x < 0 ? -1 : (x >= n ? 1 : 0), sy = y < 0 ? -1 : (y >= n ? 1 : 0),
                    sz = z < 0 ? -1 : (z >= n ? 1 : 0);
          x -= sx * n;
          y -= sy * n;
          z -= sz * n;
          const int nb = s_nb[wib][(sz + 1) * 9 + (sy + 1) * 3 + (sx + 1)];
          if (nb < 0) continue;
          const int sb = (z * n + y) * n + x;
          const uint32_t wm = S.mword[(size_t)nb * fw + (sb >> 5)];
          if (!((wm >> (sb & 31)) & 1u)) continue;
          const int ib = S.wbase[(size_t)nb * fw + (sb >> 5)] + __popc(wm & ((1u << (sb & 31)) - 1u));
          fc_union(S.parent, ia, ib);
        }
        ia++;
      }
    }
    __syncwarp();
  }
}

// The walk only reads: a halving store here could write a stale ancestor over an entry another thread has already set
// to its root.
__global__ void __launch_bounds__(256) k_fc_compress(FcScratch S, int total) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const volatile int *parent = S.parent;
    int r = parent[i], next;
    while (r != (next = parent[r])) r = next;
    S.parent[i] = r;
    S.acc_n[i] = 0;
    S.acc_key[i] = ~0ull;
    S.map[i] = -1;
#pragma unroll
    for (int k = 0; k < 3; k++) {
      S.acc_s[3 * i + k] = 0ull;
      S.acc_lo[3 * i + k] = 0x7fffffff;
      S.acc_hi[3 * i + k] = (int)0x80000000;
    }
  }
}

// kPass 0: count, sums, bounds; kPass 1: the key among the cells on the cluster's lowest z layer
template <int kPass>
__global__ void __launch_bounds__(256) k_fc_reduce(MapParams P, DeviceBuffers D, FcScratch S) {
  const int n = P.n, fw = P.front_words;
  FC_WARP_LOOP {
    int block, g[3];
    if (!fc_slot_block(P, D, slot, block, g)) continue;
    for (int w = lane; w < fw; w += 32) {
      uint32_t m = S.mword[(size_t)block * fw + w];
      int i = S.wbase[(size_t)block * fw + w];
      while (m) {
        const int bit = __ffs(m) - 1;
        m &= m - 1;
        const int sub = 32 * w + bit;
        const int c[3] = {g[0] * n + sub % n, g[1] * n + (sub / n) % n, g[2] * n + sub / (n * n)};
        const int r = S.parent[i++];
        if (kPass == 0) {
          atomicAdd(S.acc_n + r, 1);
#pragma unroll
          for (int k = 0; k < 3; k++) {
            atomicAdd(S.acc_s + 3 * r + k, (unsigned long long)(long long)c[k]);
            atomicMin(S.acc_lo + 3 * r + k, c[k]);
            atomicMax(S.acc_hi + 3 * r + k, c[k]);
          }
        } else if (c[2] == S.acc_lo[3 * r + 2]) {
          const unsigned long long yx = ((unsigned long long)(uint32_t)(c[1] - S.acc_lo[3 * r + 1]) << 32) |
                                        (uint32_t)(c[0] - S.acc_lo[3 * r]);
          atomicMin(S.acc_key + r, yx);
        }
      }
    }
  }
}

__device__ __forceinline__ void fc_key(const FcScratch &S, int r, int key[3]) {
  const unsigned long long yx = S.acc_key[r];
  key[0] = (int)((uint32_t)S.acc_lo[3 * r] + (uint32_t)(yx & 0xffffffffu));
  key[1] = (int)((uint32_t)S.acc_lo[3 * r + 1] + (uint32_t)(yx >> 32));
  key[2] = S.acc_lo[3 * r + 2];
}

__global__ void __launch_bounds__(256) k_fc_select(FcScratch S, int total, int min_cells) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    if (S.parent[i] != i || S.acc_n[i] < min_cells) continue;
    const int k = atomicAdd(S.counters, 1);
    atomicAdd(S.counters + 1, S.acc_n[i]);
    S.sv[0][k] = i;
    int key[3];
    fc_key(S, i, key);
#pragma unroll
    for (int a = 0; a < 3; a++) {
      atomicMin(S.counters + 2 + a, key[2 - a]);  // z, y, x
      atomicMax(S.counters + 5 + a, key[2 - a]);
    }
  }
}

// stable LSD radix sort of (sk[cur], sv[cur])[0..m) by bits [0, nbits) of the key, 8 bits per pass; returns the buffer
// holding the result.  Tiles of one element per thread: the rank inside a warp comes from __match_any_sync, the rank
// across warps and tiles from per-warp digit counts in shared memory.
__device__ int fc_radix_sort(const FcScratch &S, int m, int nbits, int cur) {
  __shared__ int s_hist[256], s_run[256];
  __shared__ int s_warp[kFcSortThreads / 32][256];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  for (int shift = 0; shift < nbits; shift += 8) {
    const unsigned long long *ki = S.sk[cur];
    const int *vi = S.sv[cur];
    unsigned long long *ko = S.sk[cur ^ 1];
    int *vo = S.sv[cur ^ 1];
    for (int d = t; d < 256; d += kFcSortThreads) s_hist[d] = 0;
    __syncthreads();
    for (int i = t; i < m; i += kFcSortThreads) atomicAdd(s_hist + (int)((ki[i] >> shift) & 255u), 1);
    __syncthreads();
    if (t == 0) {
      int run = 0;
      for (int d = 0; d < 256; d++) {
        s_run[d] = run;
        run += s_hist[d];
      }
    }
    __syncthreads();
    for (int base = 0; base < m; base += kFcSortThreads) {
      for (int j = t; j < (kFcSortThreads / 32) * 256; j += kFcSortThreads) (&s_warp[0][0])[j] = 0;
      __syncthreads();
      const int i = base + t;
      const bool valid = i < m;
      const unsigned long long key = valid ? ki[i] : 0ull;
      const int dg = valid ? (int)((key >> shift) & 255u) : 256 + lane;  // invalid lanes never match a digit
      const unsigned peers = __match_any_sync(0xffffffffu, dg);
      const int rank = __popc(peers & ((1u << lane) - 1u));
      if (valid && rank == 0) s_warp[wid][dg] = __popc(peers);
      __syncthreads();
      // exclusive prefix over the warps of each digit, tile totals into s_run afterwards
      for (int d = t; d < 256; d += kFcSortThreads) {
        int run = 0;
        for (int w = 0; w < kFcSortThreads / 32; w++) {
          const int c = s_warp[w][d];
          s_warp[w][d] = run;
          run += c;
        }
        s_hist[d] = run;
      }
      __syncthreads();
      if (valid) {
        const int pos = s_run[dg] + s_warp[wid][dg] + rank;
        ko[pos] = key;
        vo[pos] = vi[i];
      }
      __syncthreads();
      for (int d = t; d < 256; d += kFcSortThreads) s_run[d] += s_hist[d];
      __syncthreads();
    }
    cur ^= 1;
  }
  return cur;
}

__device__ __forceinline__ int fc_bits(unsigned v) { return v ? 32 - __clz(v) : 0; }

// one CTA: sort the kept roots by key (z, y, x); counters[8] = the buffer that holds the sorted roots
__global__ void __launch_bounds__(kFcSortThreads) k_fc_sort(FcScratch S) {
  const int m = S.counters[0];
  const int zmin = S.counters[2], ymin = S.counters[3], xmin = S.counters[4];
  const int bz = fc_bits((unsigned)(S.counters[5] - zmin)), by = fc_bits((unsigned)(S.counters[6] - ymin)),
            bx = fc_bits((unsigned)(S.counters[7] - xmin));
  const bool one = bz + by + bx <= 64;
  for (int i = threadIdx.x; i < m; i += kFcSortThreads) {
    int key[3];
    fc_key(S, S.sv[0][i], key);
    const unsigned long long yx = ((unsigned long long)(uint32_t)(key[1] - ymin) << bx) | (uint32_t)(key[0] - xmin);
    S.sk[0][i] = one ? (bz ? ((unsigned long long)(uint32_t)(key[2] - zmin) << (by + bx)) : 0ull) | yx : yx;
  }
  __syncthreads();
  int cur = fc_radix_sort(S, m, one ? bz + by + bx : by + bx, 0);
  if (!one) {  // a stable second pass by z
    __syncthreads();
    for (int i = threadIdx.x; i < m; i += kFcSortThreads) {
      int key[3];
      fc_key(S, S.sv[cur][i], key);
      S.sk[cur][i] = (uint32_t)(key[2] - zmin);
    }
    __syncthreads();
    cur = fc_radix_sort(S, m, bz, cur);
  }
  if (threadIdx.x == 0) S.counters[8] = cur;
}

__global__ void __launch_bounds__(256) k_fc_records(FcScratch S, double d, FrontierCluster *out, size_t cap) {
  const int m = S.counters[0];
  const int *sorted = S.sv[S.counters[8]];
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < m; k += gridDim.x * blockDim.x) {
    const int r = sorted[k];
    S.map[r] = k;
    if ((size_t)k >= cap) continue;
    FrontierCluster c;
    c.n_cells = S.acc_n[r];
    fc_key(S, r, c.key);
#pragma unroll
    for (int a = 0; a < 3; a++) {
      c.lo[a] = S.acc_lo[3 * r + a];
      c.hi[a] = S.acc_hi[3 * r + a];
      // rule 3: ((double)S / (double)n + 0.5) * d_sub, each operation correctly rounded (built with -fmad=false)
      c.centroid[a] = (__ll2double_rn((long long)S.acc_s[3 * r + a]) / (double)c.n_cells + 0.5) * d;
    }
    out[k] = c;
  }
}

// kWrite false: per-slot count of the cells of kept clusters into slot_cnt; true: write them in list order from the
// scanned counts (cells3 / cluster_of hold cell_cap entries)
template <bool kWrite>
__global__ void __launch_bounds__(256) k_fc_labels(MapParams P, DeviceBuffers D, FcScratch S, int *cells3, int *cluster_of,
                                                   size_t cell_cap) {
  const int n = P.n, fw = P.front_words;
  FC_WARP_LOOP {
    int block, g[3];
    if (!fc_slot_block(P, D, slot, block, g)) {
      if (!kWrite && lane == 0) S.slot_cnt[slot] = 0;
      continue;
    }
    int run = kWrite ? S.slot_cnt[slot] : 0;
    for (int w0 = 0; w0 < fw; w0 += 32) {
      const int w = w0 + lane;
      uint32_t m = w < fw ? S.mword[(size_t)block * fw + w] : 0u;
      const int i0 = w < fw ? S.wbase[(size_t)block * fw + w] : 0;
      int cnt = 0, i = i0;
      for (uint32_t t = m; t; t &= t - 1) cnt += S.map[S.parent[i++]] >= 0;
      int total;
      const int ex = fc_warp_exclusive(cnt, total);
      if (kWrite) {
        size_t at = (size_t)run + ex;
        i = i0;
        while (m) {
          const int bit = __ffs(m) - 1;
          m &= m - 1;
          const int k = S.map[S.parent[i++]];
          if (k < 0) continue;
          if (at < cell_cap) {
            const int sub = 32 * w + bit;
            cells3[3 * at] = g[0] * n + sub % n;
            cells3[3 * at + 1] = g[1] * n + (sub / n) % n;
            cells3[3 * at + 2] = g[2] * n + sub / (n * n);
            cluster_of[at] = k;
          }
          at++;
        }
      }
      run += total;
    }
    if (!kWrite && lane == 0) S.slot_cnt[slot] = run;
  }
}

#undef FC_WARP_LOOP

}  // namespace mlm
