// Von Karman correlation profile evaluated entirely in registers.
//
//   f(q) = (d)^(5/6) K_{5/6}(2 pi d) / lim0,  d = sqrt(q),  lim0 = Gamma(5/6) / (2 pi^(5/6)),  f(0) = 1
//
// This is the scalar function the reference obtains from scipy.special.kv at
// /root/reference/treegp/kernels.py:255-262 (VonKarman, q = r^2 / l^2) and
// :362-368 (AnisotropicVonKarman, q = Mahalanobis distance squared).
//
// Algebra:  with z = 2 pi d,  f = 2^(1/6)/Gamma(5/6) * z^(5/6) K_{5/6}(z).
//   z <  1 : ascending series in u = z^2/4 = pi^2 q:  f = A(u) - u^(5/6) B(u)      (no sqrt of q needed)
//   z >= 1 : f = C_INF * exp(-z) * psi(z), psi = z^(1/3) phi(z) tabulated per binade of z as a
//            polynomial in the mantissa (no cube root, no division, no iteration).
// Tables come from tools/gen_vk_tables.py (mpmath, 60 digits).  Measured error vs mpmath: see
// tests/test_cpu_host.py::test_vk_profile_against_mpmath (a few ulp relative over the whole range).
//
// The header is host+device so the CPU test-suite can exercise exactly this code with gcc/nvcc host
// compilation; the product only ever calls it from device code.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>
#include "vk_tables.h"

#if defined(__CUDACC__)
#define TGP_HD __host__ __device__ __forceinline__
#else
#define TGP_HD static inline
#endif

#define TGP_PI 3.14159265358979323846
#define TGP_PI2 9.86960440108935861883   /* pi^2 */
#define TGP_2PI 6.28318530717958647692

#define TGP_VK_PHI_ROWS (TGP_VK_E_MAX - TGP_VK_E_MIN + 1)
#define TGP_VK_PHI_SIZE (TGP_VK_PHI_ROWS * TGP_VK_PHI_STRIDE)

// Host copy of the phi table (the device copy lives in shared memory, staged by the kernels).
static const double tgp_vk_phi_host[TGP_VK_PHI_SIZE] = TGP_VK_PHI_TABLE;

TGP_HD double tgp_fma(double a, double b, double c) {
#if defined(__CUDA_ARCH__)
  return __fma_rn(a, b, c);
#else
  return fma(a, b, c);
#endif
}

// Ascending-series branch, valid for u = pi^2 q <= 1/4.
TGP_HD double tgp_vk_small(double u) {
  double a, b;
#define TGP_A_TERM(k, c) const double a##k = c;
#define TGP_B_TERM(k, c) const double b##k = c;
  TGP_VK_SER_A(TGP_A_TERM)
  TGP_VK_SER_B(TGP_B_TERM)
#undef TGP_A_TERM
#undef TGP_B_TERM
  static_assert(TGP_VK_NSER == 11, "regenerate: series length changed");
  a = a10;            b = b10;
  a = tgp_fma(a, u, a9);  b = tgp_fma(b, u, b9);
  a = tgp_fma(a, u, a8);  b = tgp_fma(b, u, b8);
  a = tgp_fma(a, u, a7);  b = tgp_fma(b, u, b7);
  a = tgp_fma(a, u, a6);  b = tgp_fma(b, u, b6);
  a = tgp_fma(a, u, a5);  b = tgp_fma(b, u, b5);
  a = tgp_fma(a, u, a4);  b = tgp_fma(b, u, b4);
  a = tgp_fma(a, u, a3);  b = tgp_fma(b, u, b3);
  a = tgp_fma(a, u, a2);  b = tgp_fma(b, u, b2);
  a = tgp_fma(a, u, a1);  b = tgp_fma(b, u, b1);
  a = tgp_fma(a, u, a0);  b = tgp_fma(b, u, b0);
  // u^(5/6) = sqrt(u) * cbrt(u)
  const double p = sqrt(u) * cbrt(u);
  return tgp_fma(-p, b, a);
}

// Large-argument branch, z >= 1.  `phi` points at the TGP_VK_PHI_SIZE-entry table.
TGP_HD double tgp_vk_large(double z, const double* __restrict__ phi) {
  if (z > 746.0) return 0.0;  // exp(-z) underflows to zero in binary64 (denormals end at ~745.13)
  uint64_t bits;
#if defined(__CUDA_ARCH__)
  bits = (uint64_t)__double_as_longlong(z);
#else
  memcpy(&bits, &z, sizeof bits);
#endif
  const int e = (int)(bits >> 52) - 1023;  // z >= 1 so sign = 0, e in [0, 9]
  // mantissa m in [1,2): overwrite the exponent with the bias
  uint64_t mb = (bits & 0x000FFFFFFFFFFFFFull) | 0x3FF0000000000000ull;
  double m;
#if defined(__CUDA_ARCH__)
  m = __longlong_as_double((long long)mb);
#else
  memcpy(&m, &mb, sizeof m);
#endif
  const double s = tgp_fma(2.0, m, -3.0);
  const double* c = phi + (e - TGP_VK_E_MIN) * TGP_VK_PHI_STRIDE;
  double acc = c[TGP_VK_PHI_STRIDE - 1];
#pragma unroll
  for (int k = TGP_VK_PHI_STRIDE - 2; k >= 0; --k) acc = tgp_fma(acc, s, c[k]);
  return TGP_VK_C_INF * exp(-z) * acc;
}

// f(q); q >= 0.  q == 0 returns exactly 1 (reference: kernels.py:260-262, :275, :367, :380).
TGP_HD double tgp_vk_profile(double q, const double* __restrict__ phi) {
  const double u = TGP_PI2 * q;
  if (u < 0.25) return tgp_vk_small(u);
  // fmax guards the one-ulp case where u >= 1/4 but 2 pi sqrt(q) rounds just below 1
  return tgp_vk_large(fmax(TGP_2PI * sqrt(q), 1.0), phi);
}

// df/dq = -2 pi^2 2^(1/6)/Gamma(5/6) z^(-1/6) K_{1/6}(z), z = 2 pi sqrt(q), from the same series and tables as f:
//   u < 1/4 : f = A(u) - u^(5/6) B(u)  ->  df/dq = pi^2 [A'(u) - u^(5/6) (5/6 B(u) / u + B'(u))]
//   z >= 1  : f = C e^-z psi(z), psi a polynomial in s = 2 m - 3 (m the mantissa of z, ds/dz = 2 / 2^e)
//             ->  df/dz = C e^-z (psi' - psi),  df/dq = df/dz 2 pi^2 / z.
// Singular (-inf) at q = 0: the caller gives coincident points no metric derivative.
TGP_HD double tgp_vk_profile_dq(double q, const double* __restrict__ phi) {
  const double u = TGP_PI2 * q;
  if (u < 0.25) {
#define TGP_A_TERM(k, c) const double a##k = c;
#define TGP_B_TERM(k, c) const double b##k = c;
    TGP_VK_SER_A(TGP_A_TERM)
    TGP_VK_SER_B(TGP_B_TERM)
#undef TGP_A_TERM
#undef TGP_B_TERM
    double b = b10, da = 10.0 * a10, db = 10.0 * b10;
    b = tgp_fma(b, u, b9);  da = tgp_fma(da, u, 9.0 * a9);  db = tgp_fma(db, u, 9.0 * b9);
    b = tgp_fma(b, u, b8);  da = tgp_fma(da, u, 8.0 * a8);  db = tgp_fma(db, u, 8.0 * b8);
    b = tgp_fma(b, u, b7);  da = tgp_fma(da, u, 7.0 * a7);  db = tgp_fma(db, u, 7.0 * b7);
    b = tgp_fma(b, u, b6);  da = tgp_fma(da, u, 6.0 * a6);  db = tgp_fma(db, u, 6.0 * b6);
    b = tgp_fma(b, u, b5);  da = tgp_fma(da, u, 5.0 * a5);  db = tgp_fma(db, u, 5.0 * b5);
    b = tgp_fma(b, u, b4);  da = tgp_fma(da, u, 4.0 * a4);  db = tgp_fma(db, u, 4.0 * b4);
    b = tgp_fma(b, u, b3);  da = tgp_fma(da, u, 3.0 * a3);  db = tgp_fma(db, u, 3.0 * b3);
    b = tgp_fma(b, u, b2);  da = tgp_fma(da, u, 2.0 * a2);  db = tgp_fma(db, u, 2.0 * b2);
    b = tgp_fma(b, u, b1);  da = tgp_fma(da, u, a1);        db = tgp_fma(db, u, b1);
    b = tgp_fma(b, u, b0);
    (void)a0;
    const double p = sqrt(u) * cbrt(u);   // u^(5/6)
    return TGP_PI2 * tgp_fma(-p, (5.0 / 6.0) * b / u + db, da);
  }
  const double z = fmax(TGP_2PI * sqrt(q), 1.0);
  if (z > 746.0) return 0.0;
  uint64_t bits;
#if defined(__CUDA_ARCH__)
  bits = (uint64_t)__double_as_longlong(z);
#else
  memcpy(&bits, &z, sizeof bits);
#endif
  const int e = (int)(bits >> 52) - 1023;
  uint64_t mb = (bits & 0x000FFFFFFFFFFFFFull) | 0x3FF0000000000000ull;
  double m;
#if defined(__CUDA_ARCH__)
  m = __longlong_as_double((long long)mb);
#else
  memcpy(&m, &mb, sizeof m);
#endif
  const double s = tgp_fma(2.0, m, -3.0);
  const double* c = phi + (e - TGP_VK_E_MIN) * TGP_VK_PHI_STRIDE;
  double psi = c[TGP_VK_PHI_STRIDE - 1], dpsi = (TGP_VK_PHI_STRIDE - 1) * c[TGP_VK_PHI_STRIDE - 1];
#pragma unroll
  for (int k = TGP_VK_PHI_STRIDE - 2; k >= 1; --k) {
    psi = tgp_fma(psi, s, c[k]);
    dpsi = tgp_fma(dpsi, s, k * c[k]);
  }
  psi = tgp_fma(psi, s, c[0]);
  const double dpsi_dz = dpsi * ldexp(2.0, -e);
  return TGP_VK_C_INF * exp(-z) * (dpsi_dz - psi) * (2.0 * TGP_PI2 / z);
}
