// Batches of independent problems (tgp_loglike_batch, tgp_loglike_grad_batch, tgp_predict_mean_batch,
// tgp_predict_var_batch, tgp_loo_batch and the _multi entries): the per-problem
// table the batched kernels read, and the launchers that kmat.cu, dense.cu, selinv.cu and predict.cu provide to
// batch.cu.  Every batched kernel
// runs the body of its single-problem twin on one problem's slice, so each problem gets the single call's arithmetic.
#pragma once
#include "tgp_common.cuh"
#include "profile_policy.cuh"

// One problem of a batch, as the device sees it (staged by batch.cu).
struct TgpBatchProb {
  const double* X;       // N x ndim training points
  const double* y;       // N x r values, row-major
  const double* yerr2;   // N diagonal additions
  double* A;             // (N + r) x ld block of the workspace: K, then L, with output c riding along as row N + c
  double* alpha;         // N x r: L^-1 y, or K^-1 y after the backward sweep
  const double* Xs;      // M x ndim test points (predict)
  double* mean;          // M x r (predict)
  int64_t N, M, ld;
  int64_t r;             // outputs sharing the kernel, the same for every problem of a batch
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
// Cholesky of every problem's block with its r outputs riding along as rows N .. N + r - 1 (which then hold
// L^-1 y); flags: B zeroed words.
int tgp_batch_potrf_rows(const TgpBatchProb* pr, const int64_t* Nh, int32_t B, int64_t r, int32_t* info,
                         unsigned* flags, cudaStream_t st);
// out[3 b ..] = {logL, chi2, logdet} from the factor and alpha, in the order of the single call's reductions
// (tgp_loglike_sum for r = 1, tgp_loglike_multi for r > 1).
int tgp_batch_loglike_finish(const TgpBatchProb* pr, int32_t B, int64_t r, int want_alpha, const int32_t* info,
                             double* out, cudaStream_t st);
int tgp_batch_predict_mean(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list, int32_t count, int cls,
                           int64_t max_m, int r, cudaStream_t st);

// ---- selected inverse of a batch (tgp_loglike_grad_batch) ----------------------------------------------------------
// Step s of a problem with N points handles its block column nb - 1 - s (nb = ceil(N / TGP_OB)), as selinv_run does
// from the last: columns [k, c1 = k + w), m = N - c1 rows below.  False when the problem has no block column left.
struct TgpSelStep {
  int64_t k, w, c1, m;
};
__host__ __device__ inline bool tgp_selinv_step(int64_t N, int s, TgpSelStep& g) {
  const int64_t nb = (N + TGP_OB - 1) / TGP_OB;
  if (s >= nb) return false;
  g.k = (nb - 1 - s) * TGP_OB;
  g.w = N - g.k < TGP_OB ? N - g.k : TGP_OB;
  g.c1 = g.k + g.w;
  g.m = N - g.c1;
  return true;
}

// The 64-wide leaves of trsm_rows_halving on a w-wide block run in order, and the gemm between leaves i and i + 1
// belongs to their lowest common ancestor: the node [o, o + n) of the halving recursion split at o + h.
__host__ __device__ inline void tgp_halving_node(int64_t w, int64_t i, int64_t& o, int64_t& h, int64_t& n) {
  o = 0;
  n = w;
  for (;;) {
    h = ((n / 2 + 63) / 64) * 64;
    const int64_t last_left = (o + h) / 64 - 1;   // the left half's last leaf
    if (i == last_left) return;
    if (i < last_left) {
      n = h;
    } else {
      o += h;
      n -= h;
    }
  }
}

// The DMMA products of one selected-inverse step (selinv_run), in launch order: T^T = W^T L21^T, Z[R, J] = -Z[R, R] T,
// + W^T W, - T^T Z[J, R]; and the gemm between halving leaves `leaf` and leaf + 1 of the -W^T solve.
enum { TGP_SEL_TT = 0, TGP_SEL_ZRJ = 1, TGP_SEL_WTW = 2, TGP_SEL_TZ = 3, TGP_SEL_HALVE = 4 };
// C (M x Nc) -= A B^T with inner dimension Kd; false (nothing to do) where selinv_run launches nothing.
__host__ __device__ inline bool tgp_selinv_gemm_shape(const TgpSelStep& g, int op, int leaf, int64_t& M, int64_t& Nc,
                                                      int64_t& Kd) {
  switch (op) {
    case TGP_SEL_TT: M = g.w; Nc = g.m; Kd = g.w; break;
    case TGP_SEL_ZRJ: M = g.m; Nc = g.w; Kd = g.m; break;
    case TGP_SEL_WTW: M = g.w; Nc = g.w; Kd = g.w; break;
    case TGP_SEL_TZ: M = g.w; Nc = g.w; Kd = g.m; break;
    default: {
      if ((int64_t)leaf + 1 >= (g.w + 63) / 64) return false;
      int64_t o, h, n;
      tgp_halving_node(g.w, leaf, o, h, n);
      M = g.w;
      Nc = n - h;
      Kd = h;
    }
  }
  return M > 0 && Nc > 0 && Kd > 0;
}

// scr: device array of B per-problem scratch blocks (tgp_loglike_grad_sum_work_doubles(N_b, TGP_MAX_TERMS) doubles,
// 16-byte aligned); prob_h, scr_h: host copies of the problem table and of scr.  On exit each problem's block of the
// workspace holds Z = K^-1, mirrored into the upper triangle.
int tgp_batch_selinv(const TgpBatchProb* pr, double* const* scr, const TgpBatchProb* prob_h, double* const* scr_h,
                     int32_t B, cudaStream_t st);
// One halving leaf of the -W^T solve per problem: trsm_panel_kernel's arguments (a 64-wide leaf takes its FULL path)
struct TgpLeafArgs {
  const double* L;
  double* B;
  int64_t ldl, M, ldb;
  int nb;
};
constexpr int TGP_LEAF_GROUP = 256;   // leaves per launch, passed in the parameter bank (10 KB)
struct TgpLeafLaunch {
  TgpLeafArgs a[TGP_LEAF_GROUP];
};
// The launches of a step that dense.cu owns: `n` leaves of one path (host array), and DMMA product `op` of step s.
int tgp_batch_selinv_leaves(const TgpLeafArgs* leaves, int32_t n, bool full, cudaStream_t st);
int tgp_batch_selinv_gemm(const TgpBatchProb* pr, double* const* scr, int32_t B, int s, int op, int leaf,
                          int tiles_n, int64_t tiles, cudaStream_t st);
// ---- predictive variance of a batch (tgp_predict_var_batch) --------------------------------------------------------
// K(Xs_b, X_b) into the pr[b].M x pr[b].ld rows at pr[b].A for the problems `list` (profile class of tgp_kmat_cross_sum).
int tgp_batch_kmat_cross(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list, int32_t count, int cls,
                         int64_t max_n, int64_t max_m, cudaStream_t st);
// One C (M x Nc) -= A B^T with inner dimension Kd per entry, launched as gemm_nt_sub_kernel's tiles.  The entries
// travel in the parameter bank, as the leaves' do: read from global memory they would spill the tile's registers.
struct TgpGemmArgs {
  double* C;
  const double* A;
  const double* B;
  int64_t M, Nc, Kd, ld;   // C, A and B share the row pitch ld
};
constexpr int TGP_GEMM_GROUP = 256;   // entries per launch (14 KB)
struct TgpGemmLaunch {
  TgpGemmArgs a[TGP_GEMM_GROUP];
};
int tgp_batch_gemm(const TgpGemmArgs* entries, int32_t n, cudaStream_t st);   // n entries (host array), all M > 0
// pr[b].mean[m] = prior[b] - sum_n V_b[m, n]^2 for the pr[b].M rows V_b at pr[b].A (var_from_rows_kernel's body).
int tgp_batch_var_rows(const TgpBatchProb* pr, const double* prior, int32_t B, int64_t max_m, cudaStream_t st);

// The contraction of the problems `list` (profile class cls) into their scratch, then one finishing CTA per problem
// writing out[b * TGP_GRAD_BATCH_OUT ..] from ll[3 b ..] = {logL, chi2, logdet}, the tile sums and info.
// r > 1: the contraction of tgp_loglike_grad_multi, w_ij = sum_c alpha_ic alpha_jc - r Z_ij.
int tgp_batch_grad_contract(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list, int32_t count, int cls,
                            double* const* scr, int64_t max_n, int max_terms, int r, cudaStream_t st);
int tgp_batch_grad_finish(const TgpBatchProb* pr, const KSumDesc* kd, double* const* scr, int32_t B,
                          const int32_t* info, const double* ll, double* out, cudaStream_t st);
