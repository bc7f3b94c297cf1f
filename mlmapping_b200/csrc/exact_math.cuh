// Bit-exact restatements of the reference's scalar arithmetic for device (and host) code.
// Everything here must evaluate with IEEE round-to-nearest and WITHOUT fused multiply-add
// contraction, because the reference is built by g++ -O3 with no -march (SURVEY Appendix A/C);
// the translation units including this header are compiled with -fmad=false and the
// float/double products whose sum order matters use explicit __f*_rn / __d*_rn intrinsics.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#ifdef __CUDA_ARCH__
#define MLM_HD __host__ __device__ __forceinline__
#else
#define MLM_HD inline
#endif

namespace mlm {

// ---- glibc 2.39 log10f -------------------------------------------------------------------------
// glibc 2.39 sysdeps/ieee754/flt-32/e_log10f.c (fdlibm-derived wrapper) calling the
// table-driven __logf (sysdeps/ieee754/flt-32/e_logf.c + logf_data.c, N=16, 3-term polynomial
// in double).  On x86-64 __logf is an ifunc: with FMA+AVX2 usable the polynomial is contracted
// into fused multiply-adds (sysdeps/x86_64/fpu/multiarch/e_logf.c); otherwise plain mul/add.
// Both evaluation orders below were read off the disassembly of this image's libm.so.6 and
// the constants dumped from its .rodata; tests/ verifies them exhaustively against the box's
// log10f (the reference computes logit() with std::log10(float), include/map_local.h:8).
struct LogfTab { double invc, logc; };
__device__ __constant__ LogfTab c_logf_tab[16] = {
  {0x1.661ec79f8f3bep+0, -0x1.57bf7808caadep-2}, {0x1.571ed4aaf883dp+0, -0x1.2bef0a7c06ddbp-2},
  {0x1.49539f0f010b0p+0, -0x1.01eae7f513a67p-2}, {0x1.3c995b0b80385p+0, -0x1.b31d8a68224e9p-3},
  {0x1.30d190c8864a5p+0, -0x1.6574f0ac07758p-3}, {0x1.25e227b0b8ea0p+0, -0x1.1aa2bc79c8100p-3},
  {0x1.1bb4a4a1a343fp+0, -0x1.a4e76ce8c0e5ep-4}, {0x1.12358f08ae5bap+0, -0x1.1973c5a611cccp-4},
  {0x1.0953f419900a7p+0, -0x1.252f438e10c1ep-5}, {0x1.0000000000000p+0, 0x0.0p+0},
  {0x1.e608cfd9a47acp-1, 0x1.aa5aa5df25984p-5},  {0x1.ca4b31f026aa0p-1, 0x1.c5e53aa362eb4p-4},
  {0x1.b2036576afce6p-1, 0x1.526e57720db08p-3},  {0x1.9c2d163a1aa2dp-1, 0x1.bc2860d224770p-3},
  {0x1.886e6037841edp-1, 0x1.1058bc8a07ee1p-2},  {0x1.767dcf5534862p-1, 0x1.4043057b6ee09p-2}};

// __logf for a normal positive argument (the only case e_log10f.c reaches it with)
template <bool kFma>
__device__ __forceinline__ float glibc_logf_normal(float x) {
  const double Ln2 = 0x1.62e42fefa39efp-1;
  const double A0 = -0x1.00ea348b88334p-2, A1 = 0x1.5575b0be00b6ap-2, A2 = -0x1.ffffef20a4123p-2;
  uint32_t ix = __float_as_uint(x);
  if (ix == 0x3f800000u) return 0.0f;
  uint32_t tmp = ix - 0x3f330000u;
  int i = (tmp >> 19) & 15;
  int k = (int32_t)tmp >> 23;
  uint32_t iz = ix - (tmp & 0xff800000u);
  double invc = c_logf_tab[i].invc, logc = c_logf_tab[i].logc;
  double z = (double)__uint_as_float(iz);
  double y;
  if (kFma) {
    double r = __fma_rn(z, invc, -1.0);
    double y0 = __fma_rn((double)k, Ln2, logc);
    double r2 = __dmul_rn(r, r);
    double q = __fma_rn(A1, r, A2);
    q = __fma_rn(A0, r2, q);
    y = __fma_rn(q, r2, __dadd_rn(y0, r));
  } else {
    double r = __dadd_rn(__dmul_rn(z, invc), -1.0);
    double y0 = __dadd_rn(logc, __dmul_rn((double)k, Ln2));
    double r2 = __dmul_rn(r, r);
    double q = __dadd_rn(__dmul_rn(A1, r), A2);
    q = __dadd_rn(__dmul_rn(A0, r2), q);
    y = __dadd_rn(__dmul_rn(q, r2), __dadd_rn(y0, r));
  }
  return __double2float_rn(y);
}

template <bool kFma>
__device__ __forceinline__ float glibc_log10f(float x) {
  const float two25 = 3.3554432000e+07f;
  const float ivln10 = __uint_as_float(0x3ede5bd9u);
  const float log10_2hi = __uint_as_float(0x3e9a2080u);
  const float log10_2lo = __uint_as_float(0x355427dbu);
  int32_t hx = __float_as_int(x);
  int32_t k = 0;
  if (hx < 0x00800000) {
    if ((hx & 0x7fffffff) == 0) return -__int_as_float(0x7f800000);  // log(+-0) = -inf
    if (hx < 0) return __int_as_float(0x7fc00000);                   // log(-#) = NaN
    k -= 25;
    x = __fmul_rn(x, two25);
    hx = __float_as_int(x);
  }
  if (hx >= 0x7f800000) return __fadd_rn(x, x);
  k += (hx >> 23) - 127;
  int32_t i = ((uint32_t)k & 0x80000000u) >> 31;
  hx = (hx & 0x007fffff) | ((0x7f - i) << 23);
  float y = (float)(k + i);
  float xm = __int_as_float(hx);
  float lf = glibc_logf_normal<kFma>(xm);
  float z = __fadd_rn(__fmul_rn(ivln10, lf), __fmul_rn(y, log10_2lo));
  return __fadd_rn(z, __fmul_rn(y, log10_2hi));
}

__device__ __forceinline__ float glibc_log10f_sel(float x, int use_fma) {
  return use_fma ? glibc_log10f<true>(x) : glibc_log10f<false>(x);
}

// logit(p) = log10f(p / (1 - p)) in float (reference include/map_local.h:8, src/map_local.cpp:159)
__device__ __forceinline__ float logit_f(float p, int use_fma) {
  return glibc_log10f_sel(__fdiv_rn(p, __fsub_rn(1.0f, p)), use_fma);
}

// update_odds_hashmap combine step: 1 - (1 - h) * (1 - odd), all float (map_awareness.h:153)
__device__ __forceinline__ float odds_combine(float h, float odd) {
  return __fsub_rn(1.0f, __fmul_rn(__fsub_rn(1.0f, h), __fsub_rn(1.0f, odd)));
}

// VectorHasher (reference include/map_awareness.h:31-41): int arithmetic; the literal 0x9e3779b9
// is unsigned so the sums are evaluated in unsigned, (hash >> 2) is an arithmetic shift.
MLM_HD int vector_hash3(int a, int b, int c) {
  int h = 3;
  h = (int)((unsigned)h ^ ((unsigned)a + 0x9e3779b9u + ((unsigned)h << 6) + (unsigned)(h >> 2)));
  h = (int)((unsigned)h ^ ((unsigned)b + 0x9e3779b9u + ((unsigned)h << 6) + (unsigned)(h >> 2)));
  h = (int)((unsigned)h ^ ((unsigned)c + 0x9e3779b9u + ((unsigned)h << 6) + (unsigned)(h >> 2)));
  return h;
}
// libstdc++ _Mod_range_hashing on the int hash converted to size_t (sign extension)
MLM_HD uint32_t libstdcxx_bucket(int h, uint32_t bucket_count) {
  return (uint32_t)((uint64_t)(int64_t)h % (uint64_t)bucket_count);
}
// same value with 32-bit arithmetic only: c64 = 2^64 mod bucket_count (host-computed per frame).  For h < 0 the size_t is
// 2^64 - a with a = -h in [1, 2^31], so the bucket is (c64 - a mod B) mod B.
MLM_HD uint32_t libstdcxx_bucket_fast(int h, uint32_t bucket_count, uint32_t c64) {
  if (h >= 0) return (uint32_t)h % bucket_count;
  const uint32_t r = (0u - (uint32_t)h) % bucket_count;
  return c64 >= r ? c64 - r : c64 + (bucket_count - r);
}

// x / d for x < 2^31 by multiply-high; (mul, shift) from make_div_magic on the host; mul == 0 means d == 1
__device__ __forceinline__ uint32_t fast_div(uint32_t x, uint32_t mul, int shift) { return mul ? (__umulhi(x, mul) >> shift) : x; }
// floor(c / n) for |c| < 2^26 and n <= 64: bias into the non-negative range first
__device__ __forceinline__ int fast_floor_div(int c, int n, uint32_t mul, int shift) {
  const int bias_q = 1 << 21;
  return (int)fast_div((uint32_t)(c + n * bias_q), mul, shift) - bias_q;
}

// ---- Sophus/Eigen subset, host and device (reference 3rdPartLib/Sophus/sophus/so3.cpp:42-90, se3.cpp:59-95)
struct HQuat {
  double w, x, y, z;
};
struct HPose {
  HQuat q;
  double t[3];
};
// Evaluation order as Eigen's x86-64 SSE2 build of the reference has it (packets of 2 doubles; CMakeLists.txt:4 sets no
// -march): squaredNorm of the 4 coefficients x,y,z,w adds the two packets first, the quaternion product is the kernel
// of Eigen/src/Geometry/arch/Geometry_SSE.h.  Checked bit for bit against oracle/_ref in tests/test_reference_pin.py.
// The frame path composes its poses on the host, the view gain (view_kernels.cuh) on the device: one definition serves
// both (the device code is built with -fmad=false, so no product is fused into an add there either).
MLM_HD HQuat h_normalized(const HQuat &q) {  // MatrixBase::normalize(): z = squaredNorm(); if (z > 0) coeffs /= sqrt(z)
  double n2 = (q.x * q.x + q.z * q.z) + (q.y * q.y + q.w * q.w);
  if (!(n2 > 0)) return q;
  double n = sqrt(n2);
  return HQuat{q.w / n, q.x / n, q.y / n, q.z / n};
}
MLM_HD HQuat h_mul(const HQuat &a, const HQuat &b) {
  HQuat r;
  r.x = (a.w * b.x + a.y * b.z) - (a.z * b.y - a.x * b.w);
  r.y = (a.w * b.y + a.y * b.w) + (a.z * b.x - a.x * b.z);
  r.z = (a.w * b.z - a.y * b.x) + (a.z * b.w + a.x * b.y);
  r.w = (a.w * b.w - a.y * b.y) - (a.z * b.z + a.x * b.x);
  return r;
}
MLM_HD void h_rotate(const HQuat &q, const double v[3], double out[3]) {  // Eigen _transformVector
  double uvx = q.y * v[2] - q.z * v[1];
  double uvy = q.z * v[0] - q.x * v[2];
  double uvz = q.x * v[1] - q.y * v[0];
  uvx += uvx;
  uvy += uvy;
  uvz += uvz;
  double cx = q.y * uvz - q.z * uvy;
  double cy = q.z * uvx - q.x * uvz;
  double cz = q.x * uvy - q.y * uvx;
  out[0] = v[0] + q.w * uvx + cx;
  out[1] = v[1] + q.w * uvy + cy;
  out[2] = v[2] + q.w * uvz + cz;
}
MLM_HD HPose h_pose_from7(const double p[7]) {  // SE3(SO3(Quaterniond), t): the SO3 ctor normalises
  HPose r;
  r.q = h_normalized(HQuat{p[3], p[4], p[5], p[6]});
  r.t[0] = p[0];
  r.t[1] = p[1];
  r.t[2] = p[2];
  return r;
}
MLM_HD HPose h_compose(const HPose &a, const HPose &b) {  // SE3::operator*
  HPose r = a;
  double rt[3];
  h_rotate(a.q, b.t, rt);
  for (int i = 0; i < 3; i++) r.t[i] = r.t[i] + rt[i];
  r.q = h_normalized(h_mul(a.q, b.q));
  return r;
}
MLM_HD HPose h_inverse(const HPose &a) {  // SE3::inverse
  HPose r;
  r.q = h_normalized(HQuat{a.q.w, -a.q.x, -a.q.y, -a.q.z});
  double nt[3] = {a.t[0] * -1., a.t[1] * -1., a.t[2] * -1.};
  h_rotate(r.q, nt, r.t);
  return r;
}

}  // namespace mlm
