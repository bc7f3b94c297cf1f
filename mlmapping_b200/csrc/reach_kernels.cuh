// Reachability field over a box of the map (mlm_reach_*; no reference counterpart): the exact shortest-path cost from a
// set of start cells through traversable cells, 26-connected moves that never cut a corner, integer move costs.  The
// spec is in include/mlmap_b200.h ("reachability field"); oracle/oracle_reach.cpp (Dijkstra) and tests/reach_spec.py
// (scipy) restate it, and the field, the cost queries and the paths agree bit for bit.
//
// Build, on the handle's stream:
//   k_esdf_gather   the distance field's gather: one CTA per subbox meeting the box, one hash probe, a class byte per cell
//                   (free / blocking / unknown, read through SubboxView)
//   k_reach_seed    one thread per distinct source cell: class kCellSource, cost 0; its tile and every tile whose halo
//                   holds it on the first worklist (a source never improves, so no tile pass would announce it)
//   k_reach_solve   one persistent cooperative launch.  The box is cut into 8 x 8 x 8 tiles; a round works the tiles of
//                   its worklist, one CTA per tile (one thread per cell): the tile and a one-cell halo are staged in
//                   shared memory and relaxed to a local fixpoint, improved cells go back to global memory, and each
//                   neighbouring tile that shares an improved boundary cell goes on the next round's worklist.  Rounds
//                   are separated by a device-wide barrier; the launch ends when a round queues nothing.
// Costs are int32 sums of the move weights 1000 / 1414 / 1732, bounded by the budget K <= 2^30 (kReachInf above it), and
// every update is a monotone min of such sums.  Whatever order tiles and threads run in, and whatever (older or newer)
// value a concurrent read sees, a stored value is always the cost of some real path, and a tile is re-queued whenever a
// cell its halo holds improves after it was read (or holds a source); so the launch ends at the unique fixpoint, which is
// the exact minimum.  Every round after the first follows an improvement of some cell, which bounds the round count far
// below the int range of the round numbers; the barrier between rounds is wrap-safe (reach_barrier).
// The path-cost matrix (mlm_reach_matrix) solves one field per start with the same tile pass, the fields of a batch in
// one cooperative launch over (field, tile) work items (k_reach_matrix_seed / _solve / _gather, below).
// Queries are one thread per point; paths one warp per goal, the 26 candidate predecessors on 26 lanes and a ballot for
// the first in the spec's order.
#pragma once
#include "esdf_kernels.cuh"

namespace mlm {

constexpr int kReachInflated = 1;               // MLM_REACH_INFLATED
constexpr int kReachUnknown = 2;                // MLM_REACH_UNKNOWN
constexpr int kReachTile = 8;                   // tile edge in cells
constexpr int kReachHalo = kReachTile + 2;      // the tile with its one-cell halo
constexpr int kReachThreads = kReachTile * kReachTile * kReachTile;  // one thread per cell of a tile
constexpr int kReachInf = 0x7f7f7f7f;           // no path yet (the byte 0x7f, so a memset initialises the field)
constexpr long long kReachMaxBudget = 1ll << 30;
constexpr uint8_t kCellSource = 3;              // a source cell's class after k_reach_seed

struct ReachGrid {
  EsdfGrid box;     // lo, dims, subbox range of the gather, d_sub
  int tiles[3];     // tiles per axis
  int flags;        // MLM_REACH_*
  int budget;       // K
};

// the solve's worklists: mark[t] = the last round t was queued for; list[r & 1] holds round r's tiles and count[r % 3]
// their number (round r clears count[(r + 2) % 3] for round r + 1's queue); bar is the device-wide barrier's counter
struct ReachWork {
  int *mark, *list0, *list1, *count;
  unsigned *bar;
};

// neighbour j = (dz + 1) * 9 + (dy + 1) * 3 + (dx + 1), j = 13 the cell itself; the move cost floor(1000 sqrt(k)) of its
// k non-zero components
__host__ __device__ constexpr int reach_weight(int j) {
  return ((j / 9 != 1) + (j / 3 % 3 != 1) + (j % 3 != 1)) == 1 ? 1000
         : ((j / 9 != 1) + (j / 3 % 3 != 1) + (j % 3 != 1)) == 2 ? 1414 : 1732;
}
// rule 4: the cells a + d' with d'_k in {0, d_k} as bits of the 27 neighbours (the block a move spans)
__host__ __device__ constexpr uint32_t reach_need(int j) {
  uint32_t m = 0;
  for (int a = 0; a < 8; a++) {
    const int dz = (a & 4) ? j / 9 - 1 : 0, dy = (a & 2) ? j / 3 % 3 - 1 : 0, dx = (a & 1) ? j % 3 - 1 : 0;
    m |= 1u << ((dz + 1) * 9 + (dy + 1) * 3 + dx + 1);
  }
  return m;
}

__device__ __forceinline__ bool reach_passable(uint8_t c, int flags) {  // in T or S
  return c == kCellFree || c == kCellSource || (c == kCellUnknown && (flags & kReachUnknown));
}

__device__ __forceinline__ bool reach_cell(const ReachGrid &R, const double *p, int c[3]) {  // cell(p), inside the box
  bool inside = true;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    c[k] = 0;
    inside = ray_cell(p[k], R.box.d, c[k]) && inside;
    inside = inside && c[k] >= R.box.lo[k] && (long long)c[k] - R.box.lo[k] < R.box.dims[k];
  }
  return inside;
}

// queue tile t for round r (once per round)
__device__ __forceinline__ void reach_queue(const ReachWork &W, int t, int r) {
  if (atomicExch(W.mark + t, r) == r) return;
  int *list = (r & 1) ? W.list1 : W.list0;
  list[atomicAdd(W.count + r % 3, 1)] = t;
}

// the tiles whose staged block (the tile and its halo) holds the cell at l in its own tile: bit (dz + 1) * 9 + (dy + 1) * 3
// + (dx + 1) for the tile at offset (dx, dy, dz), bit 13 for the cell's own tile
__device__ __forceinline__ uint32_t reach_halo_tiles(const int l[3]) {
  int lo[3], hi[3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    lo[k] = l[k] == 0 ? -1 : 0;
    hi[k] = l[k] == kReachTile - 1 ? 1 : 0;
  }
  uint32_t m = 0;
  for (int dz = lo[2]; dz <= hi[2]; dz++)
    for (int dy = lo[1]; dy <= hi[1]; dy++)
      for (int dx = lo[0]; dx <= hi[0]; dx++) m |= 1u << ((dz + 1) * 9 + (dy + 1) * 3 + dx + 1);
  return m;
}
// queue for round r the tile at offset j (a bit of reach_halo_tiles) from tile t3, when the box has one there; the work
// item is base + the tile (base = f * tiles for field f of a matrix batch)
__device__ __forceinline__ void reach_queue_near(const ReachGrid &R, const ReachWork &W, const int t3[3], int j, int r,
                                                 int base = 0) {
  const int n3[3] = {t3[0] + j % 3 - 1, t3[1] + j / 3 % 3 - 1, t3[2] + j / 9 - 1};
  if (n3[0] >= 0 && n3[0] < R.tiles[0] && n3[1] >= 0 && n3[1] < R.tiles[1] && n3[2] >= 0 && n3[2] < R.tiles[2])
    reach_queue(W, base + (n3[2] * R.tiles[1] + n3[1]) * R.tiles[0] + n3[0], r);
}

// What a tile pass needs to know of its field beyond the shared class bytes.  The single build marks its sources in the
// class bytes (kCellSource) and its work items are the tiles.  Field f of a matrix batch has its own source cell, which
// is passable in that field only (so the class bytes stay shared), and its work items are f * tiles + t.
struct ReachSingle {
  __device__ __forceinline__ bool source(size_t) const { return false; }
  __device__ __forceinline__ int base() const { return 0; }
};
struct ReachRow {
  int src;    // the box-linear source cell, -1 when the row has none
  int item0;  // f * tiles
  __device__ __forceinline__ bool source(size_t gi) const { return (long long)gi == src; }
  __device__ __forceinline__ int base() const { return item0; }
};

// idx[i]: the box-linear index of a distinct source cell
__global__ void __launch_bounds__(256) k_reach_seed(ReachGrid R, const int *idx, int n, uint8_t *cls, int *cost,
                                                    ReachWork W) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = idx[i], nx = R.box.dims[0], ny = R.box.dims[1];
  cls[c] = kCellSource;
  cost[c] = 0;
  const int x = c % nx, y = (c / nx) % ny, z = c / (nx * ny);
  const int l[3] = {x % kReachTile, y % kReachTile, z % kReachTile};
  const int t3[3] = {x / kReachTile, y / kReachTile, z / kReachTile};
  // its own tile, and the neighbours whose halo holds it: a source keeps cost 0, so no tile pass ever announces it
  const uint32_t m = reach_halo_tiles(l);
  for (int j = 0; j < 27; j++)
    if ((m >> j) & 1) reach_queue_near(R, W, t3, j, 1);
}

// one tile of round r: stage it with its halo, relax to a local fixpoint, store the improved cells, queue the
// neighbours that share an improved boundary cell for round r + 1; cost is the field's own grid
template <class Field>
__device__ __forceinline__ void reach_tile(const ReachGrid &R, const uint8_t *cls, int *cost, const ReachWork &W, int t,
                                           int r, int *s_cost, uint8_t *s_pass, uint32_t &s_touch, const Field &F) {
  const int tid = threadIdx.x;
  const int t3[3] = {t % R.tiles[0], (t / R.tiles[0]) % R.tiles[1], t / (R.tiles[0] * R.tiles[1])};
  const int nx = R.box.dims[0], ny = R.box.dims[1];
  for (int i = tid; i < kReachHalo * kReachHalo * kReachHalo; i += kReachThreads) {
    const int h[3] = {i % kReachHalo, (i / kReachHalo) % kReachHalo, i / (kReachHalo * kReachHalo)};
    bool in = true;
    int g[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      g[k] = t3[k] * kReachTile + h[k] - 1;
      in = in && g[k] >= 0 && g[k] < R.box.dims[k];
    }
    const size_t gi = ((size_t)g[2] * ny + g[1]) * nx + g[0];
    // costs other CTAs store in this launch: read through L2 (ld.cg), never a stale L1 line
    s_cost[i] = in ? __ldcg(cost + gi) : kReachInf;
    s_pass[i] = in && (reach_passable(cls[gi], R.flags) || F.source(gi));
  }
  if (tid == 0) s_touch = 0;
  __syncthreads();
  const int l[3] = {tid % kReachTile, (tid / kReachTile) % kReachTile, tid / (kReachTile * kReachTile)};
  const int me = ((l[2] + 1) * kReachHalo + l[1] + 1) * kReachHalo + l[0] + 1;
  // the moves into this cell that rule 4 allows, as bits of the 27 neighbours (none unless the cell is in T or S)
  uint32_t allowed = 0;
  if (s_pass[me]) {
    uint32_t nb = 0;
#pragma unroll
    for (int j = 0; j < 27; j++)
      nb |= (uint32_t)s_pass[me + ((j / 9 - 1) * kReachHalo + (j / 3 % 3 - 1)) * kReachHalo + (j % 3 - 1)] << j;
#pragma unroll
    for (int j = 0; j < 27; j++)
      if (j != 13 && (nb & reach_need(j)) == reach_need(j)) allowed |= 1u << j;
  }
  const int c0 = s_cost[me];
  int c = c0;
  const int K = R.budget;
  for (;;) {
    bool improved = false;
    if (allowed) {
      int best = c;
#pragma unroll
      for (int j = 0; j < 27; j++) {
        if (j == 13 || !((allowed >> j) & 1)) continue;
        const int v = s_cost[me + ((j / 9 - 1) * kReachHalo + (j / 3 % 3 - 1)) * kReachHalo + (j % 3 - 1)] +
                      reach_weight(j);  // kReachInf + 1732 stays below 2^31
        best = v < best && v <= K ? v : best;
      }
      if (best < c) {
        c = best;
        s_cost[me] = c;
        improved = true;
      }
    }
    if (!__syncthreads_or(improved)) break;
  }
  if (c < c0) {
    cost[((size_t)(t3[2] * kReachTile + l[2]) * ny + t3[1] * kReachTile + l[1]) * nx + t3[0] * kReachTile + l[0]] = c;
    // the neighbouring tiles whose halo holds this cell
    const uint32_t m = reach_halo_tiles(l) & ~(1u << 13);
    if (m) atomicOr(&s_touch, m);
  }
  __syncthreads();
  if (tid < 27 && ((s_touch >> tid) & 1)) reach_queue_near(R, W, t3, tid, r + 1, F.base());
  __syncthreads();  // shared memory is reused by the next tile
}

// The device-wide barrier between rounds: every CTA adds 1 per round, round r waits for r * G arrivals.  Counter and
// target are unsigned and compared through their signed difference, so the wrap of the counter at 2^32 (after 2^32 / G
// rounds) is harmless: the counter is never more than G away from the target a CTA waits for.
__device__ __forceinline__ void reach_barrier(unsigned *counter, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    unsigned v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    } while ((int)(v - target) < 0);
    __threadfence();
  }
  __syncthreads();
}

// the rounds of a solve: work(item, r) for every item of round r's worklist, a device-wide barrier, until a round queues
// nothing
template <class Work>
__device__ __forceinline__ void reach_rounds(const ReachWork &W, Work &&work) {
  const int G = (int)gridDim.x;
  int n_cur = __ldcg(W.count + 1);
  for (int r = 1; n_cur > 0; r++) {
    if (blockIdx.x == 0 && threadIdx.x == 0) W.count[(r + 2) % 3] = 0;  // round r + 1's queue; read in round r - 1
    const int *list = (r & 1) ? W.list1 : W.list0;
    for (int i = blockIdx.x; i < n_cur; i += G) work(__ldcg(list + i), r);
    reach_barrier(W.bar, (unsigned)r * (unsigned)G);
    n_cur = __ldcg(W.count + (r + 1) % 3);  // nobody changes it before the next barrier: every CTA sees the same value
  }
}

// the whole solve as one cooperative launch (every CTA resident, so the barrier cannot deadlock)
__global__ void __launch_bounds__(kReachThreads, 2) k_reach_solve(ReachGrid R, const uint8_t *cls, int *cost,
                                                                  ReachWork W) {
  __shared__ int s_cost[kReachHalo * kReachHalo * kReachHalo];
  __shared__ uint8_t s_pass[kReachHalo * kReachHalo * kReachHalo];
  __shared__ uint32_t s_touch;
  reach_rounds(W, [&](int t, int r) { reach_tile(R, cls, cost, W, t, r, s_cost, s_pass, s_touch, ReachSingle{}); });
}

// rule 6 at point p of the field `cost`
__device__ __forceinline__ double reach_cost_at(const ReachGrid &R, const int *cost, const double *p) {
  int c[3];
  if (!reach_cell(R, p, c)) return __longlong_as_double(0x7ff8000000000000ll);
  const int v = __ldg(cost + esdf_index(R.box, c[0] - R.box.lo[0], c[1] - R.box.lo[1], c[2] - R.box.lo[2]));
  return v == kReachInf ? __longlong_as_double(0x7ff0000000000000ll) : ((double)v / 1000.0) * R.box.d;
}

// rule 6, one thread per point
__global__ void __launch_bounds__(256) k_reach_cost(ReachGrid R, const int *cost, const double *pos, size_t n,
                                                    double *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = reach_cost_at(R, cost, pos + 3 * i);
}

// ---- path-cost matrix (mlm_reach_matrix): one field per start, the fields of a batch solved in one launch ----------
// Field f of a batch owns cost[f * cells ...] and the work items f * tiles + t (marks and worklists sized for all of
// them); the class bytes are gathered once per call and never hold a source.  Each field is exactly the single build's
// field from that one start: the same tile pass (reach_tile), with the field's source passable in its own field only.

// one thread per field: row f's source cell by rule 1 (the host rule of mlm_reach_build, through ray_cell), cost 0, and
// its tile and every tile whose halo holds it on round 1's worklist; src[f] = -1 for a row without a source
__global__ void __launch_bounds__(256) k_reach_matrix_seed(ReachGrid R, const double *starts, int n, size_t cells,
                                                           int tiles, int *src, int *cost, ReachWork W) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= n) return;
  int c[3];
  if (!reach_cell(R, starts + 3 * (size_t)f, c)) {
    src[f] = -1;
    return;
  }
  const int x = c[0] - R.box.lo[0], y = c[1] - R.box.lo[1], z = c[2] - R.box.lo[2];
  const int i = (int)esdf_index(R.box, x, y, z);
  src[f] = i;
  cost[(size_t)f * cells + i] = 0;
  const int l[3] = {x % kReachTile, y % kReachTile, z % kReachTile};
  const int t3[3] = {x / kReachTile, y / kReachTile, z / kReachTile};
  const uint32_t m = reach_halo_tiles(l);
  for (int j = 0; j < 27; j++)
    if ((m >> j) & 1) reach_queue_near(R, W, t3, j, 1, f * tiles);
}

// the solve of every field of a batch as one cooperative launch: the rounds of k_reach_solve over (field, tile) items
__global__ void __launch_bounds__(kReachThreads, 2) k_reach_matrix_solve(ReachGrid R, const uint8_t *cls, int *cost,
                                                                         ReachWork W, const int *src, size_t cells,
                                                                         int tiles) {
  __shared__ int s_cost[kReachHalo * kReachHalo * kReachHalo];
  __shared__ uint8_t s_pass[kReachHalo * kReachHalo * kReachHalo];
  __shared__ uint32_t s_touch;
  reach_rounds(W, [&](int item, int r) {
    const int f = item / tiles;
    reach_tile(R, cls, cost + (size_t)f * cells, W, item - f * tiles, r, s_cost, s_pass, s_touch,
               ReachRow{__ldg(src + f), f * tiles});
  });
}

// rule 6 for every (row, goal) of a batch, one thread each: out[f * n_goals + j] from field f at goals[j]
__global__ void __launch_bounds__(256) k_reach_matrix_gather(ReachGrid R, const int *cost, size_t cells,
                                                             const double *goals, size_t n_goals, size_t n, double *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t f = i / n_goals;
  out[i] = reach_cost_at(R, cost + f * cells, goals + 3 * (i - f * n_goals));
}

// rule 7, one warp per goal: lane j < 26 tests the j-th offset of the spec's order, the ballot's lowest lane wins
__global__ void __launch_bounds__(256) k_reach_paths(ReachGrid R, const uint8_t *cls, const int *cost,
                                                     const double *goals, size_t n, size_t max_cells, int *cells3,
                                                     int *len) {
  const size_t gi = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gi >= n) return;
  int c[3];
  if (!reach_cell(R, goals + 3 * gi, c)) {
    if (lane == 0) len[gi] = -2;
    return;
  }
  const int *dims = R.box.dims;
#pragma unroll
  for (int k = 0; k < 3; k++) c[k] -= R.box.lo[k];
  int v = __ldg(cost + esdf_index(R.box, c[0], c[1], c[2]));
  if (v == kReachInf) {
    if (lane == 0) len[gi] = -1;
    return;
  }
  const int j = lane < 13 ? lane : lane + 1;
  const int d[3] = {j % 3 - 1, j / 3 % 3 - 1, j / 9 - 1};
  const int w = reach_weight(j);
  int *out = cells3 + gi * max_cells * 3;
  int L = 0;
  for (;;) {
    if (lane < 3 && (size_t)L < max_cells)
      out[3 * (size_t)L + lane] = lane == 0 ? c[0] + R.box.lo[0] : (lane == 1 ? c[1] + R.box.lo[1] : c[2] + R.box.lo[2]);
    L++;
    if (v == 0) break;
    bool ok = false;
    if (lane < 26) {
      const int p[3] = {c[0] + d[0], c[1] + d[1], c[2] + d[2]};
      ok = p[0] >= 0 && p[0] < dims[0] && p[1] >= 0 && p[1] < dims[1] && p[2] >= 0 && p[2] < dims[2];
      ok = ok && __ldg(cost + esdf_index(R.box, p[0], p[1], p[2])) == v - w;  // v - w < kReachInf: p reachable
      // the block of the move: p + d' with d'_k in {0, -d_k}, every cell in T or S
      for (int a = 0; a < 8 && ok; a++) {
        const int q[3] = {p[0] - ((a & 1) ? d[0] : 0), p[1] - ((a & 2) ? d[1] : 0), p[2] - ((a & 4) ? d[2] : 0)};
        ok = reach_passable(__ldg(cls + esdf_index(R.box, q[0], q[1], q[2])), R.flags);
      }
    }
    const unsigned b = __ballot_sync(0xffffffffu, ok);
    if (!b) break;  // cannot happen for a fixpoint field; ends the walk rather than spinning
    const int win = __ffs(b) - 1, wj = win < 13 ? win : win + 1;
    c[0] += wj % 3 - 1;
    c[1] += wj / 3 % 3 - 1;
    c[2] += wj / 9 - 1;
    v -= reach_weight(wj);
  }
  if (lane == 0) len[gi] = L;
}

// the exported field: the cost, -1 where unreachable
__global__ void __launch_bounds__(256) k_reach_export(const int *cost, size_t n, int *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const int v = cost[i];
    out[i] = v == kReachInf ? -1 : v;
  }
}

}  // namespace mlm
