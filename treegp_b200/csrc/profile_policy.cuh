// Profile policies of the tiled kernels (K build, fused mean, gradient contraction): what one pair of points
// contributes.  The kernels are templated on a policy instead of a family:
//   FamilyProfile<FAM>  one term amp * f_FAM(q) -- the statements of the single-term kernels, unchanged;
//   SumProfile          sum_c amp_c f_c(q_c) over up to TGP_MAX_TERMS terms plus a white level on the diagonal of
//                       K(X, X).  The term loop stays rolled (#pragma unroll 1: the von Karman body alone stalls on
//                       instruction fetch when unrolled) and switches on each term's family at run time; the switch
//                       takes the same branch in every thread of the grid, so it does not diverge.
#pragma once
#include "tgp_common.cuh"
#include "profile_dq.cuh"

// Sum descriptor as the device sees it (one kernel parameter).
struct KSumDesc {
  KDesc term[TGP_MAX_TERMS];
  double white;
  int nterms, ndim, any_vk;
};

static inline bool ksum_ok(const tgp_kernel_sum* ks) {
  if (!ks || ks->nterms < 1 || ks->nterms > TGP_MAX_TERMS || (ks->ndim != 1 && ks->ndim != 2)) return false;
  if (!(ks->white >= 0.0) || ks->white == INFINITY) return false;   // NaN fails the first test
  for (int c = 0; c < ks->nterms; ++c)
    if (!kdesc_ok(&ks->term[c]) || ks->term[c].ndim != ks->ndim) return false;
  return true;
}

static inline KSumDesc make_ksumdesc(const tgp_kernel_sum* ks) {
  KSumDesc d = {};
  d.nterms = ks->nterms;
  d.ndim = ks->ndim;
  d.white = ks->white;
  for (int c = 0; c < ks->nterms; ++c) {
    d.term[c] = make_kdesc(&ks->term[c]);
    if (ks->term[c].family == TGP_FAM_VONKARMAN) d.any_vk = 1;
  }
  return d;
}

// Several outputs sharing one kernel: the policy P with nrhs = r columns of alpha (row-major (N, r)), padded to R
// columns where a kernel keeps them in registers or shared memory.  OutputsOf<P>::kR is 1 for a plain policy, and
// OutputsOf<P>::Base the policy of one output.
template <class P, int R>
struct MultiOut : P {
  int nrhs;
};
template <class P>
struct OutputsOf {
  static constexpr int kR = 1;
  using Base = P;
};
template <class P, int R>
struct OutputsOf<MultiOut<P, R>> {
  static constexpr int kR = R;
  using Base = P;
};

#ifdef __CUDACC__
__device__ __forceinline__ double tgp_profile_rt(int family, double q, const double* __restrict__ phi) {
  switch (family) {
    case TGP_FAM_RBF: return tgp_profile<TGP_FAM_RBF>(q, phi);
    case TGP_FAM_VONKARMAN: return tgp_profile<TGP_FAM_VONKARMAN>(q, phi);
    case TGP_FAM_MATERN12: return tgp_profile<TGP_FAM_MATERN12>(q, phi);
    case TGP_FAM_MATERN32: return tgp_profile<TGP_FAM_MATERN32>(q, phi);
    default: return tgp_profile<TGP_FAM_MATERN52>(q, phi);
  }
}

template <int FAM>
struct FamilyProfile {
  static constexpr bool kSum = false;
  static constexpr int kFam = FAM;
  static constexpr bool kHeavy = FAM == TGP_FAM_VONKARMAN;   // long profile body: keep the row loops short
  static constexpr int kPhiSize = FAM == TGP_FAM_VONKARMAN ? TGP_VK_PHI_SIZE : 1;
  KDesc desc;

  __device__ __forceinline__ bool stage_phi() const { return FAM == TGP_FAM_VONKARMAN; }
  __device__ __forceinline__ double weight() const { return desc.amp; }   // folded into the staged alpha

  // K(X, X) at (rg, cg) and (rg, cg + 1), without diag_add
  __device__ __forceinline__ void sym2(double rx, double ry, double cx0, double cy0, double cx1, double cy1,
                                       int64_t rg, int64_t cg, const double* phi_s, double& v0, double& v1) const {
    const double q0 = tgp_qform(desc, rx - cx0, ry - cy0), q1 = tgp_qform(desc, rx - cx1, ry - cy1);
    v0 = desc.amp * tgp_profile<FAM>(q0, phi_s);
    v1 = desc.amp * tgp_profile<FAM>(q1, phi_s);
    if (FAM == TGP_FAM_VONKARMAN) {
      // Reference quirk kept for parity: in K(X,X) the von Karman kernels leave OFF-diagonal entries of
      // coincident points at 0 (pdist == 0 is filtered out and only the diagonal is refilled,
      // kernels.py:253-262 and :360-367); K(X,Y) returns amp there (kernels.py:273-276, :378-381).
      if (q0 == 0.0 && rg != cg) v0 = 0.0;
      if (q1 == 0.0 && rg != cg + 1) v1 = 0.0;
    }
  }

  // K(Xs, X) at two adjacent columns
  __device__ __forceinline__ void cross2(double rx, double ry, double cx0, double cy0, double cx1, double cy1,
                                         const double* phi_s, double& v0, double& v1) const {
    v0 = desc.amp * tgp_profile<FAM>(tgp_qform(desc, rx - cx0, ry - cy0), phi_s);
    v1 = desc.amp * tgp_profile<FAM>(tgp_qform(desc, rx - cx1, ry - cy1), phi_s);
  }

  // several outputs: acc[c] += f(q) pa[., c] for training points i, i + 1 of the staged tile (pa: R columns per point)
  template <int R>
  __device__ __forceinline__ void mean2_multi(double sx, double sy, const double2* pxy, const double* pa, int i,
                                              const double* phi_s, double (&acc0)[R], double (&acc1)[R]) const {
    const double2 p0 = pxy[i], p1 = pxy[i + 1];
    const double f0 = tgp_profile<FAM>(tgp_qform(desc, sx - p0.x, sy - p0.y), phi_s);
    const double f1 = tgp_profile<FAM>(tgp_qform(desc, sx - p1.x, sy - p1.y), phi_s);
#pragma unroll
    for (int c = 0; c < R; ++c) {
      acc0[c] = fma(f0, pa[i * R + c], acc0[c]);
      acc1[c] = fma(f1, pa[(i + 1) * R + c], acc1[c]);
    }
  }

  // gradient contraction: the term a CTA works on, its f, f' and the von Karman rule
  __device__ __forceinline__ const KDesc& grad_term() const { return desc; }
  __device__ __forceinline__ double f(const KDesc&, double q, const double* phi_s) const {
    return tgp_profile<FAM>(q, phi_s);
  }
  __device__ __forceinline__ double fdq(const KDesc&, double q, const double* phi_s) const {
    return tgp_profile_dq<FAM>(q, phi_s);
  }
  __device__ __forceinline__ bool vk(const KDesc&) const { return FAM == TGP_FAM_VONKARMAN; }
  // index of partial column `col` of tile t
  __device__ __forceinline__ int64_t partial(int64_t t, int col) const { return 4 * t + col; }
};

struct SumProfile {
  static constexpr bool kSum = true;
  static constexpr bool kHeavy = true;
  static constexpr int kPhiSize = TGP_VK_PHI_SIZE;
  KSumDesc desc;

  __device__ __forceinline__ bool stage_phi() const { return desc.any_vk != 0; }
  __device__ __forceinline__ double weight() const { return 1.0; }

  __device__ __forceinline__ void sym2(double rx, double ry, double cx0, double cy0, double cx1, double cy1,
                                       int64_t rg, int64_t cg, const double* phi_s, double& v0, double& v1) const {
    v0 = 0.0;
    v1 = 0.0;
#pragma unroll 1
    for (int c = 0; c < desc.nterms; ++c) {
      const KDesc& kd = desc.term[c];
      const double q0 = tgp_qform(kd, rx - cx0, ry - cy0), q1 = tgp_qform(kd, rx - cx1, ry - cy1);
      double f0 = tgp_profile_rt(kd.family, q0, phi_s), f1 = tgp_profile_rt(kd.family, q1, phi_s);
      if (kd.family == TGP_FAM_VONKARMAN) {   // the reference quirk, per von Karman term
        if (q0 == 0.0 && rg != cg) f0 = 0.0;
        if (q1 == 0.0 && rg != cg + 1) f1 = 0.0;
      }
      v0 += kd.amp * f0;
      v1 += kd.amp * f1;
    }
    // WhiteKernel: by index, so that coincident distinct points do not get it
    if (rg == cg) v0 += desc.white;
    if (rg == cg + 1) v1 += desc.white;
  }

  __device__ __forceinline__ void cross2(double rx, double ry, double cx0, double cy0, double cx1, double cy1,
                                         const double* phi_s, double& v0, double& v1) const {
    v0 = 0.0;
    v1 = 0.0;
#pragma unroll 1
    for (int c = 0; c < desc.nterms; ++c) {
      const KDesc& kd = desc.term[c];
      v0 += kd.amp * tgp_profile_rt(kd.family, tgp_qform(kd, rx - cx0, ry - cy0), phi_s);
      v1 += kd.amp * tgp_profile_rt(kd.family, tgp_qform(kd, rx - cx1, ry - cy1), phi_s);
    }
  }

  // acc += sum_c f_c(q_c) (amp_c alpha) for training points i, i + 1 of the staged tile (pa = alpha), term by term
  __device__ __forceinline__ void mean2(double sx, double sy, const double2* pxy, const double* pa, int i,
                                        const double* phi_s, double& acc0, double& acc1) const {
    const double2 p0 = pxy[i], p1 = pxy[i + 1];
    const double a0 = pa[i], a1 = pa[i + 1];
#pragma unroll 1
    for (int c = 0; c < desc.nterms; ++c) {
      const KDesc& kd = desc.term[c];
      acc0 = fma(tgp_profile_rt(kd.family, tgp_qform(kd, sx - p0.x, sy - p0.y), phi_s), kd.amp * a0, acc0);
      acc1 = fma(tgp_profile_rt(kd.family, tgp_qform(kd, sx - p1.x, sy - p1.y), phi_s), kd.amp * a1, acc1);
    }
  }

  // mean2 for R outputs: each term's profile once per pair, applied to every column (pa: R columns per point)
  template <int R>
  __device__ __forceinline__ void mean2_multi(double sx, double sy, const double2* pxy, const double* pa, int i,
                                              const double* phi_s, double (&acc0)[R], double (&acc1)[R]) const {
    const double2 p0 = pxy[i], p1 = pxy[i + 1];
#pragma unroll 1
    for (int c = 0; c < desc.nterms; ++c) {
      const KDesc& kd = desc.term[c];
      const double f0 = tgp_profile_rt(kd.family, tgp_qform(kd, sx - p0.x, sy - p0.y), phi_s);
      const double f1 = tgp_profile_rt(kd.family, tgp_qform(kd, sx - p1.x, sy - p1.y), phi_s);
#pragma unroll
      for (int j = 0; j < R; ++j) {
        acc0[j] = fma(f0, kd.amp * pa[i * R + j], acc0[j]);
        acc1[j] = fma(f1, kd.amp * pa[(i + 1) * R + j], acc1[j]);
      }
    }
  }

  // gradient contraction: blockIdx.y selects the term; partial columns 4 c .. 4 c + 3 per term, 4 nterms = white
  __device__ __forceinline__ const KDesc& grad_term() const { return desc.term[blockIdx.y]; }
  __device__ __forceinline__ double f(const KDesc& kd, double q, const double* phi_s) const {
    return tgp_profile_rt(kd.family, q, phi_s);
  }
  __device__ __forceinline__ double fdq(const KDesc& kd, double q, const double* phi_s) const {
    return tgp_profile_dq_family(kd.family, q, phi_s);
  }
  __device__ __forceinline__ bool vk(const KDesc& kd) const { return kd.family == TGP_FAM_VONKARMAN; }
  __device__ __forceinline__ int64_t partial(int64_t t, int col) const {
    return (int64_t)(4 * desc.nterms + 1) * t + 4 * (int)blockIdx.y + col;
  }
  __device__ __forceinline__ int64_t white_partial(int64_t t) const {
    return (int64_t)(4 * desc.nterms + 1) * t + 4 * desc.nterms;
  }
};
#endif
