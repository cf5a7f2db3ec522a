// Batches of independent problems (tgp_loglike_batch, tgp_predict_mean_batch): the per-problem table the batched
// kernels read, and the launchers that kmat.cu, dense.cu and predict.cu provide to batch.cu.  Every batched kernel
// runs the body of its single-problem twin on one problem's slice, so each problem gets the single call's arithmetic.
#pragma once
#include "tgp_common.cuh"
#include "profile_policy.cuh"

// One problem of a batch, as the device sees it (staged by batch.cu).
struct TgpBatchProb {
  const double* X;       // N x ndim training points
  const double* y;       // N values
  const double* yerr2;   // N diagonal additions
  double* A;             // (N + 1) x ld block of the workspace: K, then L, with y riding along as row N
  double* alpha;         // N: L^-1 y, or K^-1 y after the backward sweep
  const double* Xs;      // M x ndim test points (predict)
  double* mean;          // M (predict)
  int64_t N, M, ld;
};

// Profile class of a problem: its family (one term, and for the K build no white level), or a sum.  This is the
// choice the single entries make (tgp_kmat_sym_sum, tgp_predict_mean_sum), so a batch runs the same kernel bodies.
constexpr int TGP_BATCH_SUM = 5;
constexpr int TGP_BATCH_NCLASS = 6;

#ifdef __CUDACC__
template <class P>
__device__ __forceinline__ P tgp_batch_profile(const KSumDesc& d);
template <>
__device__ __forceinline__ SumProfile tgp_batch_profile<SumProfile>(const KSumDesc& d) { return SumProfile{d}; }
#define TGP_BATCH_FAMILY_PROFILE(F)                                                                        \
  template <>                                                                                            \
  __device__ __forceinline__ FamilyProfile<F> tgp_batch_profile<FamilyProfile<F>>(const KSumDesc& d) {   \
    return FamilyProfile<F>{d.term[0]};                                                                  \
  }
TGP_BATCH_FAMILY_PROFILE(TGP_FAM_RBF)
TGP_BATCH_FAMILY_PROFILE(TGP_FAM_VONKARMAN)
TGP_BATCH_FAMILY_PROFILE(TGP_FAM_MATERN12)
TGP_BATCH_FAMILY_PROFILE(TGP_FAM_MATERN32)
TGP_BATCH_FAMILY_PROFILE(TGP_FAM_MATERN52)
#undef TGP_BATCH_FAMILY_PROFILE
#endif

// All pointers below are device pointers; `list` holds `count` problem indices of profile class `cls`; max_n / max_m
// bound the sizes of those problems.  Nh: host copy of the problem sizes.
int tgp_batch_kmat_sym(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list, int32_t count, int cls,
                       int64_t max_n, cudaStream_t st);
// Cholesky of every problem's block with y riding along as row N (row N then holds L^-1 y); flags: B zeroed words.
int tgp_batch_potrf_rows(const TgpBatchProb* pr, const int64_t* Nh, int32_t B, int32_t* info, unsigned* flags,
                         cudaStream_t st);
// out[3 b ..] = {logL, chi2, logdet} from the factor and alpha, in the order of the single call's reductions.
int tgp_batch_loglike_finish(const TgpBatchProb* pr, int32_t B, int want_alpha, const int32_t* info, double* out,
                             cudaStream_t st);
int tgp_batch_predict_mean(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list, int32_t count, int cls,
                           int64_t max_m, cudaStream_t st);
