// ORACLE — TEST INFRASTRUCTURE ONLY.  Candidate-view gain, mlm_view_gain (no reference counterpart): the spec in
// include/mlmap_b200.h ("candidate-view gain") computed literally over the restatement's observed_group_map: the pose
// algebra of its SE3 (the frame's), every cell of the frustum's AABB tested one by one, and for targets the ray spec's walk
// with one map lookup per visited cell.  Built into its own library, liboracle_views.so (tests/view_oracle.py), which is
// the oracle's whole C surface plus orc_cast_rays (oracle_rays.cpp, for the cell rule) plus this file; with the
// reference's flags (-O3, no -march, so no fused multiply-add).
#include "oracle_rays.cpp"

#include <algorithm>

namespace {
// (state byte, inflation byte) of cell c, as the ray spec's rule 3 reads them; `front` = its frontier bit
void orc_cell_state(orc::local_map *L, const int c[3], char &st, char &inf, bool &front) {
  const int nn = L->subbox_nxyz;
  Vec3I g(orc_floor_div(c[0], nn), orc_floor_div(c[1], nn), orc_floor_div(c[2], nn));
  const int sub = ((c[2] - g[2] * nn) * nn + (c[1] - g[1] * nn)) * nn + (c[0] - g[0] * nn);
  st = 'u';
  inf = 'u';
  front = false;
  auto it = L->observed_group_map.find(g);
  if (it == L->observed_group_map.end()) return;
  if (it->second.occupancy.size() == 1) {
    st = it->second.occupancy[0];
    return;
  }
  st = it->second.occupancy[sub];
  inf = it->second.inflate_occupancy[sub];
  front = it->second.frontier.count(sub) != 0;
}
}  // namespace

// work (may be NULL): {cells of the AABBs tested, cells visited by the line-of-sight walks}
extern "C" int orc_view_gain(void *h, const double *T_wb, size_t n, const mlm_view_sensor *S, const int32_t *boxes,
                             int flags, mlm_view_gain_record *out, int64_t *work) {
  auto *M = static_cast<orc::mlmap *>(h);
  auto *L = M->local;
  const double d = L->map_dxyz_obv_sub;
  if (!S || !out || (!T_wb && n) || (flags & ~(MLM_VIEW_FRONTIER | MLM_VIEW_INFLATED))) return MLM_ERR_INVALID_ARG;
  for (double v : {S->fx, S->fy, S->cx, S->cy, S->min_depth, S->max_depth})
    if (!std::isfinite(v)) return MLM_ERR_INVALID_ARG;
  if (!(S->fx > 0) || !(S->fy > 0) || S->cols < 1 || S->rows < 1 || !(0 <= S->min_depth && S->min_depth < S->max_depth))
    return MLM_ERR_INVALID_ARG;
  const double lim = 256 * d;
  const double hx = std::max(std::fabs((-0.5 - S->cx) / S->fx), std::fabs(((double)S->cols - 0.5 - S->cx) / S->fx));
  const double hy = std::max(std::fabs((-0.5 - S->cy) / S->fy), std::fabs(((double)S->rows - 0.5 - S->cy) / S->fy));
  if (S->max_depth > lim || hx * S->max_depth > lim || hy * S->max_depth > lim) return MLM_ERR_CAPACITY;
  const bool frontier = (flags & MLM_VIEW_FRONTIER) != 0, inflated = (flags & MLM_VIEW_INFLATED) != 0;
  if (frontier && !L->apply_explored_area) return MLM_ERR_UNSUPPORTED;
  int64_t tested = 0, steps = 0;
  for (size_t i = 0; i < n; i++) {
    const double *p = T_wb + 7 * i;
    mlm_view_gain_record r = {MLM_VIEW_INVALID, 0, 0, 0};
    out[i] = r;
    // rule 1
    bool ok = true;
    for (int k = 0; k < 7; k++) ok = ok && std::isfinite(p[k]);
    const double n2 = (p[4] * p[4] + p[6] * p[6]) + (p[5] * p[5] + p[3] * p[3]);
    if (!ok || !(n2 > 0) || !std::isfinite(n2)) continue;
    const SE3 Tws = se3_from_pose7(p) * M->awareness->T_bs;
    const SE3 Tsw = Tws.inverse();
    const Vec3 o = Tws.translation();
    int co[3];
    for (int k = 0; k < 3; k++) ok = orc_ray_cell(o[k], d, co[k]) && ok;
    const int32_t *b = boxes ? boxes + 6 * i : nullptr;
    for (int k = 0; b && k < 3; k++) ok = ok && b[k] <= b[3 + k];
    if (!ok) continue;
    out[i].status = 0;
    // the cells to test: the AABB of the origin and the four far corners, one cell of margin, clipped to the box
    double mn[3] = {o[0], o[1], o[2]}, mx[3] = {o[0], o[1], o[2]};
    for (int j = 0; j < 4; j++) {
      const double uc = (j & 1) ? (double)S->cols - 0.5 : -0.5, vc = (j & 2) ? (double)S->rows - 0.5 : -0.5;
      const Vec3 w = Tws * Vec3(((uc - S->cx) / S->fx) * S->max_depth, ((vc - S->cy) / S->fy) * S->max_depth, S->max_depth);
      for (int k = 0; k < 3; k++) {
        mn[k] = std::min(mn[k], w[k]);
        mx[k] = std::max(mx[k], w[k]);
      }
    }
    int lo[3], hi[3];
    for (int k = 0; k < 3; k++) {
      lo[k] = (int)std::floor(mn[k] / d) - 1;
      hi[k] = (int)std::floor(mx[k] / d) + 1;
      if (b) {
        lo[k] = std::max(lo[k], b[k]);
        hi[k] = std::min(hi[k], b[3 + k]);
      }
    }
    for (int cz = lo[2]; cz <= hi[2]; cz++)
      for (int cy = lo[1]; cy <= hi[1]; cy++)
        for (int cx = lo[0]; cx <= hi[0]; cx++) {
          tested++;
          const int c[3] = {cx, cy, cz};
          const Vec3 x(((double)cx + 0.5) * d, ((double)cy + 0.5) * d, ((double)cz + 0.5) * d);
          const Vec3 q = Tsw * x;  // rule 2
          // rule 3
          if (!(q[2] >= S->min_depth && q[2] <= S->max_depth)) continue;
          const double u = (q[0] / q[2]) * S->fx + S->cx, v = (q[1] / q[2]) * S->fy + S->cy;
          if (!(u >= -0.5 && u < (double)S->cols - 0.5 && v >= -0.5 && v < (double)S->rows - 0.5)) continue;
          // rule 4
          char st, inf;
          bool front;
          orc_cell_state(L, c, st, inf, front);
          if (frontier ? !front : (st == 'f' || st == 'o')) continue;
          out[i].n_target++;
          // rule 5: the ray spec's walk from o to x; every cell before c free (and not inflated)
          int w[3] = {co[0], co[1], co[2]}, rem[3], s[3];
          double inv[3] = {0, 0, 0};
          for (int k = 0; k < 3; k++) {
            rem[k] = std::abs(c[k] - w[k]);
            s[k] = c[k] > w[k] ? 1 : (c[k] < w[k] ? -1 : 0);
            if (rem[k] > 0) inv[k] = 1.0 / (x[k] - o[k]);
          }
          bool visible = true;
          while (rem[0] + rem[1] + rem[2] > 0) {
            steps++;
            char ws, wi;
            bool wf;
            orc_cell_state(L, w, ws, wi, wf);
            if (ws != 'f' || (inflated && wi == 'o')) {
              visible = false;
              break;
            }
            int ax = -1;
            double tb = 0.0;
            for (int k = 0; k < 3; k++) {
              if (rem[k] == 0) continue;
              const double tk = ((double)(w[k] + (s[k] > 0 ? 1 : 0)) * d - o[k]) * inv[k];
              if (ax < 0 || tk < tb) {
                ax = k;
                tb = tk;
              }
            }
            w[ax] += s[ax];
            rem[ax]--;
          }
          if (visible) out[i].n_visible++;
        }
  }
  if (work) {
    work[0] = tested;
    work[1] = steps;
  }
  return MLM_OK;
}

// Replaces the restatement's map with m subboxes given as mlm_export_map / orc_export_frontier lay them out (glb3,
// collapsed flags, occupancy and inflation bytes per cell, frontier bits per cell, log-odds per cell): the crafted maps
// of the tests.  A collapsed subbox keeps element 0 of its occupancy, inflation and log-odds only, and no frontier.
// log_odds may be NULL: every log-odds 0.
extern "C" void orc_view_set_map(void *h, size_t m, const int32_t *glb3, const uint8_t *collapsed, const char *occ,
                                 const char *infl, const uint8_t *front_bits, const float *log_odds) {
  auto *L = static_cast<orc::mlmap *>(h)->local;
  const size_t cells = L->cell_num_subbox, nb = (cells + 7) / 8;
  L->observed_group_map.clear();
  for (size_t i = 0; i < m; i++) {
    auto &sb = L->observed_group_map[Vec3I(glb3[3 * i], glb3[3 * i + 1], glb3[3 * i + 2])];
    const size_t k = collapsed[i] ? 1 : cells;
    sb.occupancy.assign(occ + i * cells, occ + i * cells + k);
    sb.inflate_occupancy.assign(infl + i * cells, infl + i * cells + k);
    if (log_odds)
      sb.log_odds.assign(log_odds + i * cells, log_odds + i * cells + k);
    else
      sb.log_odds.assign(k, 0.0f);
    sb.frontier.clear();
    for (size_t c = 0; !collapsed[i] && c < cells; c++)
      if (front_bits[i * nb + c / 8] >> (c & 7) & 1) sb.frontier.insert((int)c);
  }
}
