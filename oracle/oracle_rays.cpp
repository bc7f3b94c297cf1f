// ORACLE — TEST INFRASTRUCTURE ONLY.  Batched ray casting, mlm_cast_rays (no reference counterpart): the spec in
// include/mlmap_b200.h ("batched queries") walked literally over the restatement's observed_group_map, one lookup per
// visited cell.  Built into its own library, liboracle_rays.so (tests/ray_oracle.py), which is the oracle's whole C
// surface (oracle_capi.cpp) plus orc_cast_rays; with the reference's flags (oracle/Makefile: -std=c++17 -O3, no -march,
// so no fused multiply-add).  Kept out of mlmap_oracle.hpp, which restates reference functions only.
#include "oracle_capi.cpp"

namespace {
bool orc_ray_cell(double p, double d, int &c) {
  const double q = p / d;
  if (!(std::fabs(q) < 1073741824.0)) return false;  // non-finite or |p / d_sub| >= 2^30
  c = (int)std::floor(q);
  return true;
}
int orc_floor_div(int a, int b) {
  int q = a / b, r = a - q * b;
  return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q;
}
}  // namespace

extern "C" void orc_cast_rays(void *h, const double *from, const double *to, size_t n, int flags, mlm_ray_hit *out) {
  auto *L = static_cast<orc::mlmap *>(h)->local;
  const double d = L->map_dxyz_obv_sub;
  const int nn = L->subbox_nxyz;
  const bool inflated = (flags & MLM_RAY_INFLATED) != 0;
  for (size_t i = 0; i < n; i++) {
    const double *f = from + 3 * i, *t = to + 3 * i;
    mlm_ray_hit r = {MLM_RAY_INVALID, {0, 0, 0}, 0, 0, 0.0};
    int c[3] = {0, 0, 0}, e[3] = {0, 0, 0};
    bool ok = true;
    for (int k = 0; k < 3; k++) ok = orc_ray_cell(f[k], d, c[k]) && orc_ray_cell(t[k], d, e[k]) && ok;
    long long total = 0;
    if (ok)
      for (int k = 0; k < 3; k++) total += std::llabs((long long)e[k] - c[k]);
    if (!ok || total > (1 << 20)) {
      out[i] = r;
      continue;
    }
    int rem[3], s[3];
    double inv[3] = {0, 0, 0};
    for (int k = 0; k < 3; k++) {
      rem[k] = std::abs(e[k] - c[k]);
      s[k] = e[k] > c[k] ? 1 : (e[k] < c[k] ? -1 : 0);
      if (rem[k] > 0) inv[k] = 1.0 / (t[k] - f[k]);
    }
    double t_enter = 0.0;
    for (;;) {
      Vec3I g(orc_floor_div(c[0], nn), orc_floor_div(c[1], nn), orc_floor_div(c[2], nn));
      const int sub = ((c[2] - g[2] * nn) * nn + (c[1] - g[1] * nn)) * nn + (c[0] - g[0] * nn);
      char st = 'u';
      bool blocking = false;
      auto it = L->observed_group_map.find(g);
      if (it != L->observed_group_map.end()) {
        if (it->second.occupancy.size() == 1) {
          st = it->second.occupancy[0];
        } else {
          st = it->second.occupancy[sub];
          blocking = inflated && it->second.inflate_occupancy[sub] == 'o';
        }
      }
      if (st == 'o' || blocking) {
        r.status = MLM_OCCUPIED;
        break;
      }
      if (st == 'f') r.n_free++;
      else r.n_unknown++;
      if (rem[0] + rem[1] + rem[2] == 0) {
        r.status = MLM_FREE;
        break;
      }
      int ax = -1;
      double tb = 0.0;
      for (int k = 0; k < 3; k++) {
        if (rem[k] == 0) continue;
        const double tk = ((double)(c[k] + (s[k] > 0 ? 1 : 0)) * d - f[k]) * inv[k];
        if (ax < 0 || tk < tb) {
          ax = k;
          tb = tk;
        }
      }
      c[ax] += s[ax];
      rem[ax]--;
      t_enter = tb;
    }
    for (int k = 0; k < 3; k++) r.cell[k] = c[k];
    r.t = t_enter > 0.0 ? (t_enter < 1.0 ? t_enter : 1.0) : 0.0;
    out[i] = r;
  }
}
