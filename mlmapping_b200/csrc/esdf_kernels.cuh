// Signed distance field over a box of the map (mlm_esdf_*; no reference counterpart).  The spec is in
// include/mlmap_b200.h ("signed distance field"); oracle/oracle_esdf.cpp and tests/esdf_spec.py restate it, and the
// grid and the queries agree bit for bit.
//
// Build, four launches on the handle's stream:
//   k_esdf_gather   one CTA per subbox meeting the box: one hash probe, then the blocking byte of each of its cells in the
//                   box, read through the ray walk's SubboxView (the same blocking rule)
//   k_esdf_x        one CTA per x line, staged in shared memory: 1-D distance to the nearest blocking and non-blocking
//                   cell of the line (prefix scans of the last / first index), squared
//   k_esdf_y        one thread per y line, threads over x: lower envelope of parabolas (Felzenszwalb-Huttenlocher), both
//                   channels in one walk over the line
//   k_esdf_z        the same along z, then the cell values (rule 4)
// The envelope compares intersections as int64 cross products (no division), so D+- are exact and do not depend on the
// order threads run in.  Squared distances are int32 (< 2^26 under the size limit), kEsdfInf stands for +inf.
#pragma once
#include "ray_kernels.cuh"

namespace mlm {

constexpr int kEsdfInflated = 1;               // MLM_ESDF_INFLATED
constexpr int kEsdfMaxAxis = 4096;             // N_k <= 4096
constexpr long long kEsdfMaxCells = 1ll << 28; // N_x * N_y * N_z <= 2^28
constexpr int kEsdfInf = 0x7fffffff;           // an empty set's squared distance
constexpr int kEsdfLineThreads = 64;           // threads (x lines) per CTA of k_esdf_y / k_esdf_z

struct EsdfGrid {
  int lo[3];        // first cell of the box
  int dims[3];      // N_x, N_y, N_z
  int glo[3];       // first subbox meeting the box
  int gdims[3];     // subboxes meeting the box per axis
  double d;         // d_sub
  double max_dist;
};

__device__ __forceinline__ size_t esdf_index(const EsdfGrid &G, int x, int y, int z) {
  return ((size_t)z * G.dims[1] + y) * G.dims[0] + x;
}

// blk[cell] = 1 when the cell blocks (rule 2)
template <bool kInflated>
__global__ void __launch_bounds__(256) k_esdf_gather(MapParams P, DeviceBuffers D, EsdfGrid G, uint8_t *blk) {
  __shared__ SubboxView s_view;
  const int b = blockIdx.x;
  const int g[3] = {G.glo[0] + b % G.gdims[0], G.glo[1] + (b / G.gdims[0]) % G.gdims[1],
                    G.glo[2] + b / (G.gdims[0] * G.gdims[1])};
  if (threadIdx.x == 0) s_view = subbox_view(P, D, g);
  const int n = P.n;
  int c0[3], len[3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const int a = g[k] * n, e = a + n - 1, hi = G.lo[k] + G.dims[k] - 1;
    c0[k] = a > G.lo[k] ? a : G.lo[k];
    len[k] = (e < hi ? e : hi) - c0[k] + 1;
  }
  __syncthreads();
  const SubboxView v = s_view;
  const int count = len[0] * len[1] * len[2];
  for (int t = threadIdx.x; t < count; t += blockDim.x) {
    const int x = c0[0] + t % len[0], y = c0[1] + (t / len[0]) % len[1], z = c0[2] + t / (len[0] * len[1]);
    const int sub = ((z - g[2] * n) * n + (y - g[1] * n)) * n + (x - g[0] * n);
    char st;
    blk[esdf_index(G, x - G.lo[0], y - G.lo[1], z - G.lo[2])] = view_blocks<kInflated>(v, sub, st) ? 1 : 0;
  }
}

// One CTA per x line (y, z): .x = squared distance to the nearest blocking cell of the line, .y = to the nearest
// non-blocking one (kEsdfInf when the line has none).  Each thread owns a run of consecutive cells; the last blocking /
// free index before its run and the first after it come from scans over the threads.
__global__ void __launch_bounds__(256) k_esdf_x(EsdfGrid G, const uint8_t *blk, int2 *out) {
  __shared__ uint8_t s_blk[kEsdfMaxAxis];
  __shared__ int2 s_out[kEsdfMaxAxis];
  __shared__ int s_scan[4][256];
  const int nx = G.dims[0], t = threadIdx.x;
  const size_t row = (size_t)blockIdx.x * nx;
  for (int x = t; x < nx; x += 256) s_blk[x] = blk[row + x];
  __syncthreads();
  const int per = (nx + 255) / 256, x0 = t * per, x1 = min(x0 + per, nx);
  const int kNone = 1 << 30;
  int last_b = -1, last_f = -1, first_b = kNone, first_f = kNone;
  for (int x = x0; x < x1; x++) {
    if (s_blk[x]) {
      last_b = x;
      first_b = min(first_b, x);
    } else {
      last_f = x;
      first_f = min(first_f, x);
    }
  }
  s_scan[0][t] = last_b;
  s_scan[1][t] = last_f;
  s_scan[2][t] = first_b;
  s_scan[3][t] = first_f;
  // inclusive scans: max of the last indices from the left, min of the first indices from the right
  for (int off = 1; off < 256; off <<= 1) {
    __syncthreads();
    const int a = t >= off ? s_scan[0][t - off] : -1, b = t >= off ? s_scan[1][t - off] : -1;
    const int c = t + off < 256 ? s_scan[2][t + off] : kNone, d = t + off < 256 ? s_scan[3][t + off] : kNone;
    __syncthreads();
    s_scan[0][t] = max(s_scan[0][t], a);
    s_scan[1][t] = max(s_scan[1][t], b);
    s_scan[2][t] = min(s_scan[2][t], c);
    s_scan[3][t] = min(s_scan[3][t], d);
  }
  __syncthreads();
  // right-hand neighbours first (walking down), then the left-hand ones (walking up) and the minimum of both
  int nb = t < 255 ? s_scan[2][t + 1] : kNone, nf = t < 255 ? s_scan[3][t + 1] : kNone;
  for (int x = x1 - 1; x >= x0; x--) {
    if (s_blk[x]) nb = x;
    else nf = x;
    s_out[x] = make_int2(nb - x, nf - x);  // >= kNone - 4096 when there is none
  }
  int pb = t > 0 ? s_scan[0][t - 1] : -1, pf = t > 0 ? s_scan[1][t - 1] : -1;
  for (int x = x0; x < x1; x++) {
    if (s_blk[x]) pb = x;
    else pf = x;
    const int2 r = s_out[x];
    const int db = min(r.x, pb >= 0 ? x - pb : kNone), df = min(r.y, pf >= 0 ? x - pf : kNone);
    s_out[x] = make_int2(db < kEsdfMaxAxis ? db * db : kEsdfInf, df < kEsdfMaxAxis ? df * df : kEsdfInf);
  }
  __syncthreads();
  for (int x = t; x < nx; x += 256) out[row + x] = s_out[x];
}

// Lower envelope of the parabolas f(q) + (p - q)^2 of one channel, built one site at a time.  The stack lives in global
// scratch at stk[k * stride] (threads over x: coalesced); its top is kept in registers.
struct EsdfEnvelope {
  int2 *stk;   // .x site, .y f(site)
  int top;     // stack height - 1 (-1: empty)
  int2 t;      // the top entry
};

// does the parabola of site b overtake that of site a no later than that of c overtakes b?  (a < b < c; the
// intersection of a and b is ((f_b + b^2) - (f_a + a^2)) / (2 (b - a)); compared as an int64 cross product)
__device__ __forceinline__ bool esdf_hidden(int2 a, int2 b, int2 c) {
  const long long nab = ((long long)b.y + (long long)b.x * b.x) - ((long long)a.y + (long long)a.x * a.x);
  const long long nbc = ((long long)c.y + (long long)c.x * c.x) - ((long long)b.y + (long long)b.x * b.x);
  return nbc * (long long)(b.x - a.x) <= nab * (long long)(c.x - b.x);
}

__device__ __forceinline__ void esdf_push(EsdfEnvelope &e, int q, int f, size_t stride) {
  if (f == kEsdfInf) return;
  const int2 c = make_int2(q, f);
  while (e.top >= 1) {
    const int2 below = e.stk[(size_t)(e.top - 1) * stride];
    if (!esdf_hidden(below, e.t, c)) break;
    e.top--;
    e.t = below;
  }
  if (e.top >= 0) e.stk[(size_t)e.top * stride] = e.t;
  e.top++;
  e.t = c;
}

// the envelope's walk over p = 0, 1, ...: k only moves forward
struct EsdfScan {
  int k;
  int2 cur, next;
};
__device__ __forceinline__ void esdf_scan_begin(EsdfEnvelope &e, EsdfScan &s, size_t stride) {
  if (e.top >= 0) e.stk[(size_t)e.top * stride] = e.t;  // the top joins the stack in memory
  s.k = 0;
  s.cur = e.top >= 0 ? e.stk[0] : make_int2(0, kEsdfInf);
  s.next = e.top >= 1 ? e.stk[stride] : make_int2(0, 0);
}
__device__ __forceinline__ int esdf_scan_value(const EsdfEnvelope &e, EsdfScan &s, int p, size_t stride) {
  if (e.top < 0) return kEsdfInf;
  while (s.k < e.top) {
    const int a = s.cur.y + (p - s.cur.x) * (p - s.cur.x), b = s.next.y + (p - s.next.x) * (p - s.next.x);
    if (b > a) return a;
    s.k++;
    s.cur = s.next;
    if (s.k < e.top) s.next = e.stk[(size_t)(s.k + 1) * stride];
  }
  return s.cur.y + (p - s.cur.x) * (p - s.cur.x);
}

// one line of n cells at in[p * stride] (both channels), the envelopes in stk0 / stk1 at the same offsets; emit(p, D+, D-)
template <typename Emit>
__device__ __forceinline__ void esdf_line(const int2 *in, int2 *stk0, int2 *stk1, size_t stride, int n, Emit emit) {
  EsdfEnvelope e0 = {stk0, -1, make_int2(0, 0)}, e1 = {stk1, -1, make_int2(0, 0)};
  int2 nxt = in[0];
  for (int q = 0; q < n; q++) {
    const int2 f = nxt;
    if (q + 1 < n) nxt = in[(size_t)(q + 1) * stride];  // the next load is in flight during this site's pops
    esdf_push(e0, q, f.x, stride);
    esdf_push(e1, q, f.y, stride);
  }
  EsdfScan s0, s1;
  esdf_scan_begin(e0, s0, stride);
  esdf_scan_begin(e1, s1, stride);
  for (int p = 0; p < n; p++) emit(p, esdf_scan_value(e0, s0, p, stride), esdf_scan_value(e1, s1, p, stride));
}

// y lines: grid (ceil(N_x / 64), N_z)
__global__ void __launch_bounds__(kEsdfLineThreads, 8) k_esdf_y(EsdfGrid G, const int2 *in, int2 *out, int2 *stk) {
  const int x = blockIdx.x * kEsdfLineThreads + threadIdx.x;
  if (x >= G.dims[0]) return;
  const size_t cells = (size_t)G.dims[0] * G.dims[1] * G.dims[2];
  const size_t base = esdf_index(G, x, 0, blockIdx.y), stride = G.dims[0];
  esdf_line(in + base, stk + base, stk + cells + base, stride, G.dims[1],
            [=](int p, int dp, int dm) { out[base + (size_t)p * stride] = make_int2(dp, dm); });
}

// rule 4; kEsdfInf counts as beyond max_dist
__device__ __forceinline__ double esdf_clamped(int d2, double d, double max_dist) {
  if (d2 == kEsdfInf) return max_dist;
  const double r = sqrt((double)d2) * d;
  return r < max_dist ? r : max_dist;
}

// z lines, then the cell values: grid (ceil(N_x / 64), N_y)
__global__ void __launch_bounds__(kEsdfLineThreads, 8) k_esdf_z(EsdfGrid G, const int2 *in, double *val, int2 *stk) {
  const int x = blockIdx.x * kEsdfLineThreads + threadIdx.x;
  if (x >= G.dims[0]) return;
  const size_t cells = (size_t)G.dims[0] * G.dims[1] * G.dims[2];
  const size_t base = esdf_index(G, x, blockIdx.y, 0), stride = (size_t)G.dims[0] * G.dims[1];
  const double d = G.d, md = G.max_dist;
  esdf_line(in + base, stk + base, stk + cells + base, stride, G.dims[2], [=](int p, int dp, int dm) {
    // D+ == 0 exactly for the cells of B
    val[base + (size_t)p * stride] = dp == 0 ? d - esdf_clamped(dm, d, md) : esdf_clamped(dp, d, md);
  });
}

// rule 5, one thread per point
__global__ void __launch_bounds__(256) k_esdf_query(EsdfGrid G, const double *val, const double *pos, size_t n,
                                                    double *dist, double *grad) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double d = G.d;
  double w[3], u[3];
  int i0[3], i1[3];
  bool inside = true;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const double p = pos[3 * i + k];
    int c = 0;
    inside = ray_cell(p, d, c) && inside;
    inside = inside && c >= G.lo[k] && (long long)c - G.lo[k] < G.dims[k];
    const double q = p / d - 0.5;
    const double fq = floor(q);
    const int ik = inside ? (int)fq : G.lo[k];
    w[k] = q - (double)ik;
    u[k] = 1.0 - w[k];
    const int a = ik - G.lo[k], top = G.dims[k] - 1;
    i0[k] = a < 0 ? 0 : (a > top ? top : a);
    i1[k] = a + 1 < 0 ? 0 : (a + 1 > top ? top : a + 1);
  }
  if (!inside) {
    dist[i] = __longlong_as_double(0x7ff8000000000000ll);
    if (grad) grad[3 * i] = grad[3 * i + 1] = grad[3 * i + 2] = 0.0;
    return;
  }
  double v[2][2][2];  // [z][y][x]
#pragma unroll
  for (int z = 0; z < 2; z++)
#pragma unroll
    for (int y = 0; y < 2; y++)
#pragma unroll
      for (int x = 0; x < 2; x++)
        v[z][y][x] = __ldg(val + esdf_index(G, x ? i1[0] : i0[0], y ? i1[1] : i0[1], z ? i1[2] : i0[2]));
  double e[2][2];  // e_yz as [z][y]
#pragma unroll
  for (int z = 0; z < 2; z++)
#pragma unroll
    for (int y = 0; y < 2; y++) e[z][y] = v[z][y][0] * u[0] + v[z][y][1] * w[0];
  const double f0 = e[0][0] * u[1] + e[0][1] * w[1], f1 = e[1][0] * u[1] + e[1][1] * w[1];
  dist[i] = f0 * u[2] + f1 * w[2];
  if (grad) {
    const double g00 = v[0][0][1] - v[0][0][0], g01 = v[1][0][1] - v[1][0][0];
    const double g10 = v[0][1][1] - v[0][1][0], g11 = v[1][1][1] - v[1][1][0];
    grad[3 * i] = ((((g00 * u[1]) * u[2] + (g01 * u[1]) * w[2]) + (g10 * w[1]) * u[2]) + (g11 * w[1]) * w[2]) / d;
    grad[3 * i + 1] = ((e[0][1] - e[0][0]) * u[2] + (e[1][1] - e[1][0]) * w[2]) / d;
    grad[3 * i + 2] = (f1 - f0) / d;
  }
}

__global__ void __launch_bounds__(256) k_esdf_export(const double *val, size_t n, float *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)val[i];
}

}  // namespace mlm
