// ORACLE — TEST INFRASTRUCTURE ONLY.  Frontier clustering, mlm_frontier_clusters (no reference counterpart): the spec in
// include/mlmap_b200.h ("frontier clustering") computed literally over the restatement's observed_group_map: the
// frontier sets (unordered_set<int> per subbox, no bitmasks) gathered into a set of cells, then a breadth-first search
// per component over the 26 (or 6) neighbours, records by plain loops and a std::sort by key.  Built into its own
// library, liboracle_frontier.so (tests/frontier_oracle.py), which is the oracle's whole C surface plus orc_cast_rays
// (oracle_rays.cpp, for the cell rule) plus this file; with the reference's flags (-O3, no -march, so no fused
// multiply-add).
#include "oracle_rays.cpp"

#include <algorithm>
#include <array>
#include <set>
#include <vector>

namespace {
using Cell = std::array<int, 3>;  // x, y, z
bool zyx_less(const Cell &a, const Cell &b) {
  if (a[2] != b[2]) return a[2] < b[2];
  if (a[1] != b[1]) return a[1] < b[1];
  return a[0] < b[0];
}
struct ZyxLess {
  bool operator()(const Cell &a, const Cell &b) const { return zyx_less(a, b); }
};
}  // namespace

extern "C" int orc_frontier_clusters(void *h, const double *box_min, const double *box_max, int32_t min_cells, int flags,
                                     mlm_frontier_cluster *out, size_t cap, size_t *n_out, int32_t *cells3,
                                     int32_t *cluster_of, size_t cell_cap, size_t *n_cells_out) {
  auto *L = static_cast<orc::mlmap *>(h)->local;
  const double d = L->map_dxyz_obv_sub;
  const int nn = L->subbox_nxyz;
  if (!n_out || (!box_min) != (!box_max) || min_cells < 1 || (flags & ~MLM_FRONTIER_CONN6) || (!out && cap) ||
      ((!cells3 || !cluster_of) && cell_cap))
    return MLM_ERR_INVALID_ARG;
  int lo[3] = {INT32_MIN, INT32_MIN, INT32_MIN}, hi[3] = {INT32_MAX, INT32_MAX, INT32_MAX};
  if (box_min)
    for (int k = 0; k < 3; k++)
      if (!orc_ray_cell(box_min[k], d, lo[k]) || !orc_ray_cell(box_max[k], d, hi[k]) || !(box_min[k] <= box_max[k]))
        return MLM_ERR_INVALID_ARG;
  if (!L->apply_explored_area) return MLM_ERR_UNSUPPORTED;
  // rule 1: F, the frontier cells of the subboxes that hold a full block, inside the box
  std::set<Cell, ZyxLess> F;
  for (auto &kv : L->observed_group_map) {
    if (kv.second.occupancy.size() == 1) continue;  // collapsed
    for (int id : kv.second.frontier) {
      if (id < 0 || id >= (int)L->cell_num_subbox) continue;
      const Cell c = {kv.first[0] * nn + id % nn, kv.first[1] * nn + (id / nn) % nn, kv.first[2] * nn + id / (nn * nn)};
      bool inside = true;
      for (int k = 0; k < 3; k++) inside = inside && c[k] >= lo[k] && c[k] <= hi[k];
      if (inside) F.insert(c);
    }
  }
  // rule 2: components by breadth-first search; F is walked in (z, y, x) order, so the first cell of a component is its key
  const bool conn6 = (flags & MLM_FRONTIER_CONN6) != 0;
  std::set<Cell, ZyxLess> seen;
  std::vector<mlm_frontier_cluster> recs;
  std::vector<std::vector<Cell>> members;
  for (const Cell &start : F) {
    if (seen.count(start)) continue;
    std::vector<Cell> comp = {start};
    seen.insert(start);
    for (size_t q = 0; q < comp.size(); q++) {
      const Cell c = comp[q];
      for (int dz = -1; dz <= 1; dz++)
        for (int dy = -1; dy <= 1; dy++)
          for (int dx = -1; dx <= 1; dx++) {
            const int l1 = std::abs(dx) + std::abs(dy) + std::abs(dz);
            if (l1 == 0 || (conn6 && l1 != 1)) continue;
            const Cell b = {c[0] + dx, c[1] + dy, c[2] + dz};
            if (F.count(b) && !seen.count(b)) {
              seen.insert(b);
              comp.push_back(b);
            }
          }
    }
    if ((int64_t)comp.size() < min_cells) continue;
    // rule 3
    mlm_frontier_cluster r;
    r.n_cells = (int32_t)comp.size();
    Cell key = comp[0];
    int64_t S[3] = {0, 0, 0};
    for (int k = 0; k < 3; k++) r.lo[k] = r.hi[k] = comp[0][k];
    for (const Cell &c : comp) {
      if (zyx_less(c, key)) key = c;
      for (int k = 0; k < 3; k++) {
        r.lo[k] = std::min(r.lo[k], c[k]);
        r.hi[k] = std::max(r.hi[k], c[k]);
        S[k] += c[k];
      }
    }
    for (int k = 0; k < 3; k++) {
      r.key[k] = key[k];
      r.centroid[k] = (((double)S[k] / (double)r.n_cells) + 0.5) * d;
    }
    recs.push_back(r);
    members.push_back(std::move(comp));
  }
  // rule 4: by key in (z, y, x) order
  std::vector<size_t> order(recs.size());
  for (size_t i = 0; i < order.size(); i++) order[i] = i;
  std::sort(order.begin(), order.end(), [&](size_t a, size_t b) {
    return zyx_less({recs[a].key[0], recs[a].key[1], recs[a].key[2]}, {recs[b].key[0], recs[b].key[1], recs[b].key[2]});
  });
  size_t n_cells = 0;
  for (size_t k = 0; k < order.size(); k++) {
    if (k < cap) out[k] = recs[order[k]];
    for (const Cell &c : members[order[k]]) {  // rule 5
      if (n_cells < cell_cap) {
        for (int a = 0; a < 3; a++) cells3[3 * n_cells + a] = c[a];
        cluster_of[n_cells] = (int32_t)k;
      }
      n_cells++;
    }
  }
  *n_out = recs.size();
  if (n_cells_out) *n_cells_out = n_cells;
  return MLM_OK;
}
