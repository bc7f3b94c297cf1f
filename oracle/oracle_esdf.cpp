// ORACLE — TEST INFRASTRUCTURE ONLY.  Signed distance field over a box of the map, mlm_esdf_* (no reference
// counterpart): the spec in include/mlmap_b200.h ("signed distance field") computed literally over the restatement's
// observed_group_map.  Blocking cells are looked up one by one; the exact squared distances come from a plain separable
// transform (two sweeps along x, then lower envelopes of parabolas along y and z with integer comparisons); values and
// queries follow the stated formulas.  Built into its own library, liboracle_esdf.so (tests/esdf_oracle.py), which is
// the oracle's whole C surface plus orc_cast_rays (oracle_rays.cpp) plus this file; with the reference's flags (-O3, no
// -march, so no fused multiply-add).
#include "oracle_rays.cpp"

#include <limits>
#include <map>
#include <vector>

namespace {
constexpr int64_t kInf = std::numeric_limits<int64_t>::max();

struct OrcEsdf {
  int lo[3] = {0, 0, 0}, dims[3] = {0, 0, 0};
  double d = 0.0;
  std::vector<int64_t> dplus, dminus;  // exact squared distances, kInf for an empty set
  std::vector<double> val;             // rule 4
  size_t index(int x, int y, int z) const { return ((size_t)z * dims[1] + y) * dims[0] + x; }
};
std::map<void *, OrcEsdf> g_esdf;  // the field of each oracle handle

// one line of f (kInf: no site) -> min over q of f(q) + (p - q)^2, by the lower envelope of the parabolas
void envelope(std::vector<int64_t> &f) {
  const int n = (int)f.size();
  std::vector<int64_t> site, out(n, kInf);
  for (int q = 0; q < n; q++) {
    if (f[q] == kInf) continue;
    // drop the top while the new parabola overtakes it no later than the top overtakes the one below it:
    // s(b, c) <= s(a, b) with s(a, b) = ((f_b + b^2) - (f_a + a^2)) / (2 (b - a))
    while (site.size() >= 2) {
      const int64_t a = site[site.size() - 2], b = site.back(), c = q;
      const int64_t nab = (f[b] + b * b) - (f[a] + a * a), nbc = (f[c] + c * c) - (f[b] + b * b);
      if (nbc * (b - a) > nab * (c - b)) break;
      site.pop_back();
    }
    site.push_back(q);
  }
  if (!site.empty()) {
    size_t k = 0;
    for (int p = 0; p < n; p++) {
      // the next parabola is lower at p once p is past the two's intersection: (f_b + b^2) - (f_a + a^2) < 2 p (b - a)
      while (k + 1 < site.size()) {
        const int64_t a = site[k], b = site[k + 1];
        if ((f[b] + b * b) - (f[a] + a * a) >= 2 * (int64_t)p * (b - a)) break;
        k++;
      }
      const int64_t q = site[k];
      out[p] = f[q] + (p - q) * (p - q);
    }
  }
  f.swap(out);
}

// the squared distance of every cell to the nearest cell with mask[c] == want
std::vector<int64_t> squared_edt(const OrcEsdf &E, const std::vector<char> &mask, char want) {
  const int nx = E.dims[0], ny = E.dims[1], nz = E.dims[2];
  std::vector<int64_t> g(mask.size(), kInf);
  for (int z = 0; z < nz; z++)
    for (int y = 0; y < ny; y++) {
      int64_t last = -1;  // two sweeps along x: distance to the nearest such cell on the left, then on the right
      for (int x = 0; x < nx; x++) {
        if (mask[E.index(x, y, z)] == want) last = x;
        if (last >= 0) g[E.index(x, y, z)] = (x - last) * (x - last);
      }
      last = -1;
      for (int x = nx - 1; x >= 0; x--) {
        if (mask[E.index(x, y, z)] == want) last = x;
        if (last >= 0) g[E.index(x, y, z)] = std::min(g[E.index(x, y, z)], (last - x) * (last - x));
      }
    }
  std::vector<int64_t> line;
  for (int z = 0; z < nz; z++)
    for (int x = 0; x < nx; x++) {
      line.resize(ny);
      for (int y = 0; y < ny; y++) line[y] = g[E.index(x, y, z)];
      envelope(line);
      for (int y = 0; y < ny; y++) g[E.index(x, y, z)] = line[y];
    }
  for (int y = 0; y < ny; y++)
    for (int x = 0; x < nx; x++) {
      line.resize(nz);
      for (int z = 0; z < nz; z++) line[z] = g[E.index(x, y, z)];
      envelope(line);
      for (int z = 0; z < nz; z++) g[E.index(x, y, z)] = line[z];
    }
  return g;
}

double clamped(int64_t d2, double d, double max_dist) {
  if (d2 == kInf) return max_dist;
  return std::min(std::sqrt((double)d2) * d, max_dist);
}
}  // namespace

extern "C" {

int orc_esdf_build(void *h, const double box_min[3], const double box_max[3], double max_dist, int flags) {
  auto *L = static_cast<orc::mlmap *>(h)->local;
  const double d = L->map_dxyz_obv_sub;
  const int nn = L->subbox_nxyz;
  if ((flags != 0 && flags != MLM_ESDF_INFLATED) || !std::isfinite(max_dist) || !(max_dist > 0)) return MLM_ERR_INVALID_ARG;
  OrcEsdf E;
  E.d = d;
  long long cells = 1;
  for (int k = 0; k < 3; k++) {
    int a, b;
    if (!orc_ray_cell(box_min[k], d, a) || !orc_ray_cell(box_max[k], d, b) || !(box_min[k] <= box_max[k]))
      return MLM_ERR_INVALID_ARG;
    if ((long long)b - a + 1 > 4096) return MLM_ERR_CAPACITY;
    E.lo[k] = a;
    E.dims[k] = b - a + 1;
    cells *= E.dims[k];
  }
  if (cells > (1ll << 28)) return MLM_ERR_CAPACITY;
  // rule 2, one lookup per cell
  std::vector<char> blocking((size_t)cells, 0);
  const bool inflated = (flags & MLM_ESDF_INFLATED) != 0;
  for (int z = 0; z < E.dims[2]; z++)
    for (int y = 0; y < E.dims[1]; y++)
      for (int x = 0; x < E.dims[0]; x++) {
        const int c[3] = {E.lo[0] + x, E.lo[1] + y, E.lo[2] + z};
        Vec3I g(orc_floor_div(c[0], nn), orc_floor_div(c[1], nn), orc_floor_div(c[2], nn));
        auto it = L->observed_group_map.find(g);
        if (it == L->observed_group_map.end()) continue;
        char st, inf = 'u';
        if (it->second.occupancy.size() == 1) {
          st = it->second.occupancy[0];
        } else {
          const int sub = ((c[2] - g[2] * nn) * nn + (c[1] - g[1] * nn)) * nn + (c[0] - g[0] * nn);
          st = it->second.occupancy[sub];
          inf = it->second.inflate_occupancy[sub];
        }
        blocking[E.index(x, y, z)] = st == 'o' || (inflated && inf == 'o');
      }
  E.dplus = squared_edt(E, blocking, 1);
  E.dminus = squared_edt(E, blocking, 0);
  E.val.resize((size_t)cells);
  for (size_t i = 0; i < (size_t)cells; i++)
    E.val[i] = blocking[i] ? d - clamped(E.dminus[i], d, max_dist) : clamped(E.dplus[i], d, max_dist);
  g_esdf[h] = std::move(E);
  return MLM_OK;
}

void orc_esdf_release(void *h) { g_esdf.erase(h); }

// the transform alone, for the tests: out[c] = squared distance of cell c of a dims[0] x dims[1] x dims[2] grid (x
// fastest) to the nearest cell with mask == want, -1 for none
void orc_esdf_squared(const char *mask, const int32_t dims[3], int want, int64_t *out) {
  OrcEsdf E;
  for (int k = 0; k < 3; k++) E.dims[k] = dims[k];
  const size_t cells = (size_t)dims[0] * dims[1] * dims[2];
  const std::vector<char> m(mask, mask + cells);
  const std::vector<int64_t> g = squared_edt(E, m, (char)want);
  for (size_t i = 0; i < cells; i++) out[i] = g[i] == kInf ? -1 : g[i];
}

// rule 5
int orc_esdf_distance(void *h, const double *pos, size_t n, double *dist, double *grad) {
  auto f = g_esdf.find(h);
  if (f == g_esdf.end()) return MLM_ERR_INVALID_ARG;
  const OrcEsdf &E = f->second;
  const double d = E.d;
  for (size_t i = 0; i < n; i++) {
    const double *p = pos + 3 * i;
    bool inside = true;
    int c[3], i0[3], i1[3];
    double w[3], u[3];
    for (int k = 0; k < 3; k++)
      inside = inside && orc_ray_cell(p[k], d, c[k]) && c[k] >= E.lo[k] && (long long)c[k] - E.lo[k] < E.dims[k];
    if (!inside) {
      dist[i] = std::numeric_limits<double>::quiet_NaN();
      if (grad) grad[3 * i] = grad[3 * i + 1] = grad[3 * i + 2] = 0.0;
      continue;
    }
    for (int k = 0; k < 3; k++) {
      const double q = p[k] / d - 0.5;
      const int ik = (int)std::floor(q);
      w[k] = q - (double)ik;
      u[k] = 1.0 - w[k];
      i0[k] = std::min(std::max(ik - E.lo[k], 0), E.dims[k] - 1);
      i1[k] = std::min(std::max(ik - E.lo[k] + 1, 0), E.dims[k] - 1);
    }
    auto v = [&](int x, int y, int z) { return E.val[E.index(x ? i1[0] : i0[0], y ? i1[1] : i0[1], z ? i1[2] : i0[2])]; };
    const double e00 = v(0, 0, 0) * u[0] + v(1, 0, 0) * w[0], e10 = v(0, 1, 0) * u[0] + v(1, 1, 0) * w[0];
    const double e01 = v(0, 0, 1) * u[0] + v(1, 0, 1) * w[0], e11 = v(0, 1, 1) * u[0] + v(1, 1, 1) * w[0];
    const double f0 = e00 * u[1] + e10 * w[1], f1 = e01 * u[1] + e11 * w[1];
    dist[i] = f0 * u[2] + f1 * w[2];
    if (grad) {
      const double g00 = v(1, 0, 0) - v(0, 0, 0), g01 = v(1, 0, 1) - v(0, 0, 1);
      const double g10 = v(1, 1, 0) - v(0, 1, 0), g11 = v(1, 1, 1) - v(0, 1, 1);
      grad[3 * i] = ((((g00 * u[1]) * u[2] + (g01 * u[1]) * w[2]) + (g10 * w[1]) * u[2]) + (g11 * w[1]) * w[2]) / d;
      grad[3 * i + 1] = ((e10 - e00) * u[2] + (e11 - e01) * w[2]) / d;
      grad[3 * i + 2] = (f1 - f0) / d;
    }
  }
  return MLM_OK;
}

// mlm_esdf_export's layout: (float)v, x fastest
int orc_esdf_export(void *h, float *out, size_t cap, int32_t lo3[3], int32_t dims3[3]) {
  auto f = g_esdf.find(h);
  if (f == g_esdf.end()) return MLM_ERR_INVALID_ARG;
  const OrcEsdf &E = f->second;
  for (int k = 0; k < 3; k++) {
    lo3[k] = E.lo[k];
    dims3[k] = E.dims[k];
  }
  if (!out) return MLM_OK;
  if (cap < E.val.size()) return MLM_ERR_CAPACITY;
  for (size_t i = 0; i < E.val.size(); i++) out[i] = (float)E.val[i];
  return MLM_OK;
}

// for the tests: the double values and the exact D+ / D- (-1 for +inf) in the same layout
int orc_esdf_export_exact(void *h, double *val, int64_t *dplus, int64_t *dminus) {
  auto f = g_esdf.find(h);
  if (f == g_esdf.end()) return MLM_ERR_INVALID_ARG;
  const OrcEsdf &E = f->second;
  for (size_t i = 0; i < E.val.size(); i++) {
    val[i] = E.val[i];
    dplus[i] = E.dplus[i] == kInf ? -1 : E.dplus[i];
    dminus[i] = E.dminus[i] == kInf ? -1 : E.dminus[i];
  }
  return MLM_OK;
}

}  // extern "C"
