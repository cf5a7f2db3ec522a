// Derivative df/dq of the correlation profiles f(q) of tgp_profile<FAM> (tgp_common.cuh), q = delta^T M delta.
// Host+device, like vk_profile.cuh, so that the CPU test-suite compiles exactly this code with g++.
//   RBF        f = e^(-q/2)                     f' = -f / 2
//   Matern 1/2 f = e^(-sqrt q)                  f' = -e^(-sqrt q) / (2 sqrt q)         (singular at q = 0)
//   Matern 3/2 f = (1 + s) e^-s,  s = sqrt(3q)  f' = -3/2 e^-s
//   Matern 5/2 f = (1 + s + s^2/3) e^-s, s = sqrt(5q)   f' = -5/6 (1 + s) e^-s
//   von Karman tgp_vk_profile_dq                                                       (singular at q = 0)
// The log-likelihood gradient gives pairs with q = 0 no metric derivative (q f'(q) -> 0 there for every family).
#pragma once
#include "../../include/treegp_b200.h"
#include "vk_profile.cuh"

template <int FAM>
TGP_HD double tgp_profile_dq(double q, const double* __restrict__ phi) {
  if (FAM == TGP_FAM_RBF) {
    return -0.5 * exp(-0.5 * q);
  } else if (FAM == TGP_FAM_VONKARMAN) {
    return tgp_vk_profile_dq(q, phi);
  } else if (FAM == TGP_FAM_MATERN12) {
    const double r = sqrt(q);
    return -0.5 * exp(-r) / r;
  } else if (FAM == TGP_FAM_MATERN32) {
    return -1.5 * exp(-sqrt(3.0 * q));
  } else {
    const double s = sqrt(5.0 * q);
    return (-5.0 / 6.0) * (1.0 + s) * exp(-s);
  }
}

// Run-time family dispatch (host tests).
TGP_HD double tgp_profile_dq_family(int family, double q, const double* __restrict__ phi) {
  switch (family) {
    case TGP_FAM_RBF: return tgp_profile_dq<TGP_FAM_RBF>(q, phi);
    case TGP_FAM_VONKARMAN: return tgp_profile_dq<TGP_FAM_VONKARMAN>(q, phi);
    case TGP_FAM_MATERN12: return tgp_profile_dq<TGP_FAM_MATERN12>(q, phi);
    case TGP_FAM_MATERN32: return tgp_profile_dq<TGP_FAM_MATERN32>(q, phi);
    default: return tgp_profile_dq<TGP_FAM_MATERN52>(q, phi);
  }
}
