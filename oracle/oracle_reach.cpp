// ORACLE — TEST INFRASTRUCTURE ONLY.  Reachability field over a box of the map, mlm_reach_* (no reference counterpart):
// the spec in include/mlmap_b200.h ("reachability field") computed literally over the restatement's observed_group_map:
// cell states looked up one by one (orc_cell_state, the ray spec's rule 3), then Dijkstra with an int64 binary heap over
// the move graph of rule 4; queries and paths follow rules 6 and 7.  Built into its own library, liboracle_reach.so
// (tests/reach_oracle.py), which is the oracle's whole C surface plus orc_cast_rays, the view gain and its crafted-map
// setter (oracle_views.cpp) plus this file; with the reference's flags (-O3, no -march, so no fused multiply-add).
#include "oracle_views.cpp"

#include <limits>
#include <map>
#include <queue>
#include <vector>

namespace {
constexpr int64_t kUnreached = std::numeric_limits<int64_t>::max();
enum : char { kFree = 0, kBlocking = 1, kUnknown = 2 };  // a cell's class, as the tests' raw grids give it

struct OrcReach {
  int lo[3] = {0, 0, 0}, dims[3] = {0, 0, 0};
  double d = 0.0;
  int flags = 0;
  std::vector<char> pass;      // in T or S
  std::vector<int64_t> cost;   // kUnreached: no path within the budget
  size_t index(int x, int y, int z) const { return ((size_t)z * dims[1] + y) * dims[0] + x; }
  bool inside(int x, int y, int z) const {
    return x >= 0 && y >= 0 && z >= 0 && x < dims[0] && y < dims[1] && z < dims[2];
  }
};
std::map<void *, OrcReach> g_reach;  // the field of each oracle handle

int64_t move_cost(int dx, int dy, int dz) {
  const int k = (dx != 0) + (dy != 0) + (dz != 0);
  return k == 1 ? 1000 : (k == 2 ? 1414 : 1732);
}

// rule 4: every cell a + d' with d'_k in {0, d_k} passable (a itself included)
bool allowed(const OrcReach &R, int x, int y, int z, int dx, int dy, int dz) {
  for (int a = 0; a < 8; a++) {
    const int qx = x + ((a & 1) ? dx : 0), qy = y + ((a & 2) ? dy : 0), qz = z + ((a & 4) ? dz : 0);
    if (!R.inside(qx, qy, qz) || !R.pass[R.index(qx, qy, qz)]) return false;
  }
  return true;
}

// rule 2 and 3 over class bytes, then rule 5: Dijkstra from the source cells (box-relative), keys (cost, cell index)
void solve(OrcReach &R, const std::vector<char> &cls, const std::vector<size_t> &sources, int64_t K) {
  const size_t cells = cls.size();
  R.pass.assign(cells, 0);
  for (size_t i = 0; i < cells; i++)
    R.pass[i] = cls[i] == kFree || (cls[i] == kUnknown && (R.flags & MLM_REACH_UNKNOWN));
  for (size_t s : sources) R.pass[s] = 1;
  R.cost.assign(cells, kUnreached);
  using Item = std::pair<int64_t, size_t>;
  std::priority_queue<Item, std::vector<Item>, std::greater<Item>> heap;
  for (size_t s : sources) {
    R.cost[s] = 0;
    heap.push({0, s});
  }
  while (!heap.empty()) {
    const auto [c, i] = heap.top();
    heap.pop();
    if (c != R.cost[i]) continue;
    const int x = (int)(i % R.dims[0]), y = (int)(i / R.dims[0] % R.dims[1]), z = (int)(i / ((size_t)R.dims[0] * R.dims[1]));
    for (int dz = -1; dz <= 1; dz++)
      for (int dy = -1; dy <= 1; dy++)
        for (int dx = -1; dx <= 1; dx++) {
          if (!dx && !dy && !dz) continue;
          if (!allowed(R, x, y, z, dx, dy, dz)) continue;
          const int64_t v = c + move_cost(dx, dy, dz);
          const size_t j = R.index(x + dx, y + dy, z + dz);
          if (v <= K && v < R.cost[j]) {
            R.cost[j] = v;
            heap.push({v, j});
          }
        }
  }
}

// rule 7 for the box-relative cell (x, y, z); returns L
int64_t path(const OrcReach &R, int x, int y, int z, size_t max_cells, int32_t *out) {
  int64_t L = 0;
  for (;;) {
    if ((size_t)L < max_cells) {
      out[3 * L] = x + R.lo[0];
      out[3 * L + 1] = y + R.lo[1];
      out[3 * L + 2] = z + R.lo[2];
    }
    L++;
    const int64_t c = R.cost[R.index(x, y, z)];
    if (c == 0) return L;
    bool found = false;
    for (int dz = -1; dz <= 1 && !found; dz++)
      for (int dy = -1; dy <= 1 && !found; dy++)
        for (int dx = -1; dx <= 1 && !found; dx++) {
          if (!dx && !dy && !dz) continue;
          const int px = x + dx, py = y + dy, pz = z + dz;
          if (!R.inside(px, py, pz) || R.cost[R.index(px, py, pz)] == kUnreached) continue;
          if (!allowed(R, px, py, pz, -dx, -dy, -dz)) continue;
          if (R.cost[R.index(px, py, pz)] + move_cost(dx, dy, dz) != c) continue;
          x = px;
          y = py;
          z = pz;
          found = true;
        }
    if (!found) return -3;  // not a fixpoint: cannot happen
  }
}

bool cell_in_box(const OrcReach &R, const double *p, int c[3]) {
  for (int k = 0; k < 3; k++) {
    if (!orc_ray_cell(p[k], R.d, c[k])) return false;
    c[k] -= R.lo[k];
    if (c[k] < 0 || c[k] >= R.dims[k]) return false;
  }
  return true;
}
}  // namespace

extern "C" {

int orc_reach_build(void *h, const double box_min[3], const double box_max[3], const double *starts, size_t n_starts,
                    double max_dist, int flags, int32_t *n_sources) {
  auto *L = static_cast<orc::mlmap *>(h)->local;
  const double d = L->map_dxyz_obv_sub;
  if (!starts || n_starts == 0 || (flags & ~(MLM_REACH_INFLATED | MLM_REACH_UNKNOWN)) || !std::isfinite(max_dist) ||
      !(max_dist > 0))
    return MLM_ERR_INVALID_ARG;
  OrcReach R;
  R.d = d;
  R.flags = flags;
  long long cells = 1;
  for (int k = 0; k < 3; k++) {
    int a, b;
    if (!orc_ray_cell(box_min[k], d, a) || !orc_ray_cell(box_max[k], d, b) || !(box_min[k] <= box_max[k]))
      return MLM_ERR_INVALID_ARG;
    if ((long long)b - a + 1 > 4096) return MLM_ERR_CAPACITY;
    R.lo[k] = a;
    R.dims[k] = b - a + 1;
    cells *= R.dims[k];
  }
  if (cells > (1ll << 28)) return MLM_ERR_CAPACITY;
  const double Kd = std::floor((max_dist / d) * 1000.0);
  if (!(Kd <= (double)(1ll << 30))) return MLM_ERR_CAPACITY;
  std::vector<char> cls((size_t)cells);
  const bool inflated = (flags & MLM_REACH_INFLATED) != 0;
  for (int z = 0; z < R.dims[2]; z++)
    for (int y = 0; y < R.dims[1]; y++)
      for (int x = 0; x < R.dims[0]; x++) {
        const int c[3] = {R.lo[0] + x, R.lo[1] + y, R.lo[2] + z};
        char st, inf;
        bool front;
        orc_cell_state(L, c, st, inf, front);
        cls[R.index(x, y, z)] = (st == 'o' || (inflated && inf == 'o')) ? kBlocking : (st == 'f' ? kFree : kUnknown);
      }
  std::vector<size_t> sources;
  for (size_t i = 0; i < n_starts; i++) {
    int c[3];
    if (cell_in_box(R, starts + 3 * i, c)) sources.push_back(R.index(c[0], c[1], c[2]));
  }
  std::sort(sources.begin(), sources.end());
  sources.erase(std::unique(sources.begin(), sources.end()), sources.end());
  solve(R, cls, sources, (int64_t)Kd);
  if (n_sources) *n_sources = (int32_t)sources.size();
  g_reach[h] = std::move(R);
  return MLM_OK;
}

void orc_reach_release(void *h) { g_reach.erase(h); }

// the solve alone, for the tests: a dims[0] x dims[1] x dims[2] grid of classes (x fastest; 0 free, 1 blocking, 2
// unknown), n box-relative source cells (those outside are ignored), the budget K; out = the costs, -1 unreachable
void orc_reach_grid(const char *cls, const int32_t dims[3], const int32_t *sources3, size_t n, int64_t K, int flags,
                    int64_t *out) {
  OrcReach R;
  for (int k = 0; k < 3; k++) R.dims[k] = dims[k];
  R.flags = flags;
  const size_t cells = (size_t)dims[0] * dims[1] * dims[2];
  std::vector<size_t> src;
  for (size_t i = 0; i < n; i++) {
    const int32_t *s = sources3 + 3 * i;
    if (R.inside(s[0], s[1], s[2])) src.push_back(R.index(s[0], s[1], s[2]));
  }
  std::sort(src.begin(), src.end());
  src.erase(std::unique(src.begin(), src.end()), src.end());
  solve(R, std::vector<char>(cls, cls + cells), src, K);
  for (size_t i = 0; i < cells; i++) out[i] = R.cost[i] == kUnreached ? -1 : R.cost[i];
}

// rule 6
int orc_reach_cost(void *h, const double *pos, size_t n, double *out) {
  auto f = g_reach.find(h);
  if (f == g_reach.end()) return MLM_ERR_INVALID_ARG;
  const OrcReach &R = f->second;
  for (size_t i = 0; i < n; i++) {
    int c[3];
    if (!cell_in_box(R, pos + 3 * i, c)) {
      out[i] = std::numeric_limits<double>::quiet_NaN();
      continue;
    }
    const int64_t v = R.cost[R.index(c[0], c[1], c[2])];
    out[i] = v == kUnreached ? std::numeric_limits<double>::infinity() : ((double)v / 1000.0) * R.d;
  }
  return MLM_OK;
}

// rule 7
int orc_reach_paths(void *h, const double *goals, size_t n, size_t max_cells, int32_t *cells3, int32_t *len) {
  auto f = g_reach.find(h);
  if (f == g_reach.end()) return MLM_ERR_INVALID_ARG;
  const OrcReach &R = f->second;
  for (size_t i = 0; i < n; i++) {
    int c[3];
    if (!cell_in_box(R, goals + 3 * i, c)) {
      len[i] = -2;
      continue;
    }
    if (R.cost[R.index(c[0], c[1], c[2])] == kUnreached) {
      len[i] = -1;
      continue;
    }
    len[i] = (int32_t)path(R, c[0], c[1], c[2], max_cells, cells3 + i * max_cells * 3);
  }
  return MLM_OK;
}

// mlm_reach_export's layout: the cost, -1 unreachable, x fastest
int orc_reach_export(void *h, int32_t *out, size_t cap, int32_t lo3[3], int32_t dims3[3]) {
  auto f = g_reach.find(h);
  if (f == g_reach.end()) return MLM_ERR_INVALID_ARG;
  const OrcReach &R = f->second;
  for (int k = 0; k < 3; k++) {
    lo3[k] = R.lo[k];
    dims3[k] = R.dims[k];
  }
  if (!out) return MLM_OK;
  if (cap < R.cost.size()) return MLM_ERR_CAPACITY;
  for (size_t i = 0; i < R.cost.size(); i++) out[i] = R.cost[i] == kUnreached ? -1 : (int32_t)R.cost[i];
  return MLM_OK;
}

}  // extern "C"
