// Shared device/host helpers for the treegp_b200 CUDA library.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <vector>
#include "../../include/treegp_b200.h"
#include "vk_profile.cuh"

// ---- error plumbing -------------------------------------------------------------------------
void tgp_set_error(const char* fmt, ...);

#define TGP_CHECK_ARG(cond, msg)                                   \
  do {                                                             \
    if (!(cond)) {                                                 \
      tgp_set_error("%s: invalid argument: %s", __func__, msg);    \
      return TGP_ERR_INVALID;                                      \
    }                                                              \
  } while (0)

#define TGP_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      tgp_set_error("%s: %s failed: %s", __func__, #call, cudaGetErrorString(e_));       \
      return TGP_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define TGP_LAUNCH_CHECK()                                                               \
  do {                                                                                   \
    cudaError_t e_ = cudaGetLastError();                                                 \
    if (e_ != cudaSuccess) {                                                             \
      tgp_set_error("%s: kernel launch failed: %s", __func__, cudaGetErrorString(e_));   \
      return TGP_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

static inline int64_t tgp_cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- envelopes ------------------------------------------------------------------------------
// The blocked Cholesky works on TGP_OB-wide block columns, and an envelope (variable-band factor) gives one row end per
// block column: tgp_envelope_block().
constexpr int TGP_OB = 512;

// row_end holds one entry per block column (NULL: no envelope, for the callers that allow it)
static inline bool tgp_envelope_ok(const int64_t* row_end, int64_t nblocks, int64_t N) {
  return row_end == nullptr || nblocks == tgp_cdiv(N, TGP_OB);
}

// Row ends as the factorisation uses them: clamped to [end of the block, N] and made non-decreasing (an envelope never
// shrinks from one block column to the next); N in every block column without row_end.
static inline std::vector<int64_t> tgp_envelope_ends(const int64_t* row_end, int64_t N) {
  std::vector<int64_t> ends((size_t)tgp_cdiv(N, TGP_OB));
  int64_t prev = 0;
  for (size_t b = 0; b < ends.size(); ++b) {
    const int64_t c1 = ((int64_t)b + 1) * TGP_OB < N ? ((int64_t)b + 1) * TGP_OB : N;
    int64_t r = row_end ? row_end[b] : N;
    if (r < prev) r = prev;
    if (r < c1) r = c1;
    if (r > N) r = N;
    ends[b] = prev = r;
  }
  return ends;
}

int tgp_num_sms();

// Per-device "done once" flags: function attributes, symbol addresses and helper streams belong to ONE device, and
// a process may switch devices between calls (the caller follows torch.cuda.current_device()).
constexpr int TGP_MAX_DEVICES = 64;
struct TgpPerDeviceOnce {
  unsigned char done[TGP_MAX_DEVICES] = {};
};
static inline int tgp_current_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= TGP_MAX_DEVICES) d = 0;
  return d;
}
// true the first time it is called for the current device
static inline bool tgp_first_use_on_device(TgpPerDeviceOnce& o) {
  const int d = tgp_current_device();
  if (o.done[d]) return false;
  o.done[d] = 1;
  return true;
}

// ---- kernel descriptor as the device sees it ------------------------------------------------
struct KDesc {
  double amp, m00, m01x2, m11;  // m01x2 = 2*m01
  int family, ndim;
};

static inline KDesc make_kdesc(const tgp_kernel* k) {
  KDesc d;
  d.amp = k->amp;
  d.m00 = k->m00;
  d.m01x2 = 2.0 * k->m01;
  d.m11 = k->m11;
  d.family = k->family;
  d.ndim = k->ndim;
  return d;
}

static inline bool kdesc_ok(const tgp_kernel* k) {
  return k && (k->ndim == 1 || k->ndim == 2) && k->family >= 0 && k->family <= TGP_FAM_MATERN52;
}

#ifdef __CUDACC__
// Correlation profile f(q), q = squared (Mahalanobis) distance.  `phi` is the shared-memory copy of
// the von Karman table (only dereferenced for FAM == TGP_FAM_VONKARMAN).
template <int FAM>
__device__ __forceinline__ double tgp_profile(double q, const double* __restrict__ phi) {
  if (FAM == TGP_FAM_RBF) {
    return exp(-0.5 * q);
  } else if (FAM == TGP_FAM_VONKARMAN) {
    return tgp_vk_profile(q, phi);
  } else if (FAM == TGP_FAM_MATERN12) {
    return exp(-sqrt(q));
  } else if (FAM == TGP_FAM_MATERN32) {
    const double s = sqrt(3.0 * q);
    return (1.0 + s) * exp(-s);
  } else {
    const double s = sqrt(5.0 * q);
    return (1.0 + s + (5.0 / 3.0) * q) * exp(-s);
  }
}

__device__ __forceinline__ double tgp_qform(const KDesc& kd, double dx, double dy) {
  // q = m00 dx^2 + 2 m01 dx dy + m11 dy^2
  return dx * (kd.m00 * dx + kd.m01x2 * dy) + kd.m11 * dy * dy;
}

// Stage the von Karman phi table into shared memory (all threads of the CTA participate).
__device__ __forceinline__ void tgp_stage_phi(double* phi_s, const double* __restrict__ phi_g) {
  for (int i = threadIdx.x; i < TGP_VK_PHI_SIZE; i += blockDim.x) phi_s[i] = phi_g[i];
}
#endif

// Device-resident copy of the phi table (defined in kmat.cu).
const double* tgp_phi_device();

// Dispatch a templated launch on the kernel family.
#define TGP_FAMILY_SWITCH(fam, ...)                                        \
  switch (fam) {                                                           \
    case TGP_FAM_RBF: { constexpr int FAM = TGP_FAM_RBF; __VA_ARGS__; } break;             \
    case TGP_FAM_VONKARMAN: { constexpr int FAM = TGP_FAM_VONKARMAN; __VA_ARGS__; } break; \
    case TGP_FAM_MATERN12: { constexpr int FAM = TGP_FAM_MATERN12; __VA_ARGS__; } break;   \
    case TGP_FAM_MATERN32: { constexpr int FAM = TGP_FAM_MATERN32; __VA_ARGS__; } break;   \
    default: { constexpr int FAM = TGP_FAM_MATERN52; __VA_ARGS__; } break;                 \
  }
