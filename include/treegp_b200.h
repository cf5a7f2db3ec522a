/*
 * treegp_b200 -- C ABI of the B200-native GP hot path.
 *
 * The reference (PFLeget/treegp v1.4.1) is pure Python and has no FFI layer; its operator boundary
 * is what `GPInterpolation`, `log_likelihood` and `two_pcf` call into numpy/scipy/TreeCorr.  Each
 * entry point below replaces one of those call sites (cited per function, paths relative to
 * /root/reference).  A maintainer binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (e.g. torch.Tensor.data_ptr()),
 *    FP64 / int64 / int32, C-contiguous row-major, unless a parameter says "host";
 *  - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it and never
 *    synchronise, except where stated;
 *  - return value: 0 on success, negative tgp_status on a usage / CUDA error
 *    (tgp_last_error() gives the text).  There is no CPU fallback anywhere;
 *  - factorisation status follows LAPACK: *info == 0 ok, *info == j > 0 means the leading minor
 *    of order j is not positive definite (host maps this to logL = -inf exactly where
 *    treegp/log_likelihood.py:38-39 does).
 */
#ifndef TREEGP_B200_H
#define TREEGP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TGP_ABI_VERSION 1

typedef enum {
  TGP_OK = 0,
  TGP_ERR_INVALID = -1,   /* bad argument */
  TGP_ERR_CUDA = -2,      /* CUDA runtime error, see tgp_last_error() */
  TGP_ERR_UNSUPPORTED = -3
} tgp_status;

/* Stationary correlation families: K = amp * f(q), q = delta^T M delta (M = inverse metric). */
typedef enum {
  TGP_FAM_RBF = 0,        /* exp(-q/2): sklearn RBF, treegp AnisotropicRBF  (kernels.py:114-126)          */
  TGP_FAM_VONKARMAN = 1,  /* q^(5/12) K_{5/6}(2 pi sqrt q)/lim0: VonKarman / AnisotropicVonKarman
                             (kernels.py:251-277, :358-381)                                               */
  TGP_FAM_MATERN12 = 2,   /* exp(-sqrt q)                           sklearn Matern(nu=0.5)                */
  TGP_FAM_MATERN32 = 3,   /* (1+sqrt(3q)) exp(-sqrt(3q))            sklearn Matern(nu=1.5)                */
  TGP_FAM_MATERN52 = 4    /* (1+sqrt(5q)+5q/3) exp(-sqrt(5q))       sklearn Matern(nu=2.5)                */
} tgp_family;

/* POD lowering of `const * Kernel` trees produced by treegp.kernels.eval_kernel (kernels.py:17-59). */
typedef struct {
  int32_t family;   /* tgp_family */
  int32_t ndim;     /* 1 or 2 */
  double amp;       /* ConstantKernel value (sigma^2); 1.0 if absent */
  double m00, m01, m11; /* symmetric inverse metric; ndim==1 uses m00 only */
} tgp_kernel;

/* POD lowering of a Sum of such terms plus a WhiteKernel level (sklearn `c1 * A + c2 * B + WhiteKernel(w)`):
 * K(X, X)_ij = sum_c amp_c f_c(q_c) + white [i == j];  K(Xs, X) = sum_c amp_c f_c(q_c) (sklearn's WhiteKernel(X, Y)
 * is zero whenever Y is passed).  The von Karman rule of K(X, X) (0 between distinct coincident points) applies per
 * term.  Only term[0 .. nterms-1] is read. */
#define TGP_MAX_TERMS 4
typedef struct {
  int32_t nterms;               /* 1 .. TGP_MAX_TERMS stationary terms */
  int32_t ndim;                 /* 1 or 2; every term's ndim must equal it */
  double white;                 /* WhiteKernel level: diagonal of K(X, X) only; >= 0, 0 if absent */
  tgp_kernel term[TGP_MAX_TERMS];
} tgp_kernel_sum;

int tgp_abi_version(void);
const char* tgp_last_error(void);

/* ---- (1) covariance construction --------------------------------------------------------- */

/* K(X,X) [+ diag(diag_add)] -> out (N x N, leading dimension ld >= N).
 * Replaces kernel.__call__(X) + eye*y_err**2  (gp_interp.py:180, log_likelihood.py:29).
 * X: (N, ndim).  diag_add: N values or NULL.  lower_only != 0 writes only j <= i (what
 * tgp_potrf reads); otherwise the full symmetric matrix. */
int tgp_kmat_sym(const double* X, int64_t N, const tgp_kernel* k /*host*/, const double* diag_add,
                 double* out, int64_t ld, int lower_only, void* stream);

/* K(Xs, X) -> out (M x N, ld >= N).  Replaces kernel.__call__(X2, Y=X1) (gp_interp.py:177). */
int tgp_kmat_cross(const double* Xs, int64_t M, const double* X, int64_t N,
                   const tgp_kernel* k /*host*/, double* out, int64_t ld, void* stream);

/* ---- (2) dense linear algebra -------------------------------------------------------------- */

/* In-place lower Cholesky A = L L^T of the row-major N x N matrix (only j <= i is read or
 * written).  Replaces scipy.linalg.cholesky (gp_interp.py:181,187; log_likelihood.py:30).
 * info: device int32, see header comment. */
int tgp_potrf(double* A, int64_t N, int64_t ld, int32_t* info, void* stream);

/* Same factorisation, carrying `nrows` extra rows stored directly below the matrix (rows N .. N+nrows-1 of
 * the same workspace, N columns each: right-hand sides as rows).  On exit row N+r holds L^-1 y_r -- the
 * forward substitution is done by the factorisation's own panel solves and DMMA updates. */
int tgp_potrf_rows(double* A, int64_t N, int64_t ld, int64_t nrows, int32_t* info, void* stream);

/* Solve L L^T x = b in place for one right-hand side (b: N).  Replaces cho_solve
 * (gp_interp.py:182, log_likelihood.py:31). */
int tgp_potrs_vec(const double* L, int64_t N, int64_t ld, double* b, void* stream);

/* B <- B L^-T for an (M x N) row-major B (each ROW of B is one right-hand side; afterwards row m
 * holds L^-1 b_m).  The building block of cho_solve with many right-hand sides
 * (gp_interp.py:190). */
int tgp_trsm_rows(const double* L, int64_t N, int64_t ld, double* B, int64_t M, int64_t ldb,
                  void* stream);

/* C (M x Nc, ldc) <- C - A (M x Kd, lda) * B^T (B: Nc x Kd, ldb).  Used for HT.dot(v)
 * (gp_interp.py:191) in factored form.  lower_only != 0 updates only tiles with j <= i. */
int tgp_gemm_nt_sub(double* C, int64_t M, int64_t Nc, int64_t ldc, const double* A, int64_t lda,
                    const double* B, int64_t ldb, int64_t Kd, int lower_only, void* stream);

/* out[0] = sum_i 2 log L_ii   (log_likelihood.py:33);  out[1] = y . alpha (log_likelihood.py:32) when
 * y and alpha are non-NULL. out: device double[2]. */
int tgp_logdet_chi2(const double* L, int64_t N, int64_t ld, const double* y, const double* alpha,
                    double* out, void* stream);

/* Whole marginal log-likelihood evaluation (log_likelihood.py:29-37) in one call:
 * work ((N+1) x ld: one extra row carries y through the factorisation) receives K (lower) then L;
 * out: device double[3] = {logL, chi2, logdet}; info as
 * tgp_potrf.  When *info != 0 out[0] is -inf (log_likelihood.py:38-39).
 * want_alpha != 0: alpha (N) receives K^-1 y (both triangular sweeps) and chi2 = y . alpha;
 * want_alpha == 0: alpha receives L^-1 y (forward sweep only) and chi2 = ||L^-1 y||^2 -- the same
 * number without the backward sweep; this is what the hyper-parameter search loop uses. */
int tgp_loglike(const double* X, const double* y, const double* yerr2, int64_t N,
                const tgp_kernel* k /*host*/, double* work, int64_t ld, double* alpha, int want_alpha,
                double* out, int32_t* info, void* stream);

/* ---- (2b) envelope (variable-band) forms of the dense calls ----------------------------------------
 * Same results as the dense calls above for a matrix that is ZERO outside an envelope -- which is what K(X, X) is,
 * to 1e-40 of its amplitude, once the points are sorted along one axis and the kernel's support (tgp_profile_qcut)
 * is short against the field: row i then starts at the first point within the cut-off distance of point i, and a
 * Cholesky factor keeps the envelope of its matrix.  The reference factorises the dense matrix whatever the kernel
 * (gp_interp.py:181, log_likelihood.py:30); these entry points skip the blocks that are zero: N bw^2 flop instead
 * of N^3 / 3 for a band of bw rows.
 * row_end (HOST array, one entry per block of tgp_envelope_block() = 512 columns, nblocks = ceil(N / 512)):
 * the rows [row_end[b], N) of block column b are outside the envelope.  Entries are clamped to
 * [end of the block, N] and made non-decreasing.  Rows outside the envelope are neither read nor written. */
int tgp_envelope_block(void);

/* tgp_potrf_rows restricted to the envelope (nrows extra right-hand-side rows below the matrix, may be 0). */
int tgp_potrf_env(double* A, int64_t N, int64_t ld, const int64_t* row_end /*host*/, int64_t nblocks,
                  int64_t nrows, int32_t* info, void* stream);

/* tgp_trsm_rows for a factor with the envelope row_end: 2 M N bw flop instead of M N^2. */
int tgp_trsm_rows_env(const double* L, int64_t N, int64_t ld, const int64_t* row_end /*host*/, int64_t nblocks,
                      double* B, int64_t M, int64_t ldb, void* stream);

/* tgp_loglike with the factorisation restricted to the envelope (X sorted along the envelope's axis by the
 * caller; y, yerr2 and alpha in the same order). */
int tgp_loglike_env(const double* X, const double* y, const double* yerr2, int64_t N,
                    const tgp_kernel* k /*host*/, double* work, int64_t ld, double* alpha, int want_alpha,
                    double* out, int32_t* info, const int64_t* row_end /*host*/, int64_t nblocks, void* stream);

/* ---- (2c) selected inverse and the analytic log-likelihood gradient ----------------------------------------------
 * The reference fits by L-BFGS-B with a forward-difference gradient (log_likelihood.py:56-57: n_theta + 1
 * factorisations per step); these entries give the exact gradient for about three factorisations' worth of work.
 * scratch: 16-byte aligned device buffer of tgp_selinv_work_doubles(N) doubles. */
int64_t tgp_selinv_work_doubles(int64_t N);

/* In place on a factor L from tgp_potrf / tgp_potrf_env / tgp_loglike[_env] (row-major, ld even >= N): Z = (L L^T)^-1
 * on every entry of the envelope row_end (HOST, as tgp_potrf_env; NULL = dense), written to the lower triangle and
 * mirrored into the upper one.  Entries outside the envelope are neither read nor written. */
int tgp_selinv(double* L, int64_t N, int64_t ld, const int64_t* row_end /*host*/, int64_t nblocks, double* scratch,
               void* stream);

/* tgp_loglike[_env] with want_alpha (alpha = K^-1 y), then tgp_selinv on the factor in `work`, then one contraction:
 * out: device double[7] = {logL, chi2, logdet, d logL / d ln amp, d logL / d m00, d logL / d m01, d logL / d m11}
 * (1-D: the last two are 0).  On exit `work` holds Z inside the envelope.  When *info != 0, out[0] = -inf and the
 * gradient is 0.  Repeated calls give bit-identical results. */
int tgp_loglike_grad(const double* X, const double* y, const double* yerr2, int64_t N,
                     const tgp_kernel* k /*host*/, double* work, int64_t ld, double* alpha, double* out,
                     int32_t* info, const int64_t* row_end /*host*/, int64_t nblocks, double* scratch, void* stream);

/* ---- (2d) sum kernels: the entries above for a tgp_kernel_sum ---------------------------------------------------
 * Same arguments, conventions and results as their single-term twins, with K built from every term and the white
 * level.  A one-term sum with white == 0 runs the single-term kernels (K(Xs, X) and the means: any one-term sum), so
 * it gives bit for bit what the single-term entry gives. */
int tgp_kmat_sym_sum(const double* X, int64_t N, const tgp_kernel_sum* k /*host*/, const double* diag_add,
                     double* out, int64_t ld, int lower_only, void* stream);
int tgp_kmat_cross_sum(const double* Xs, int64_t M, const double* X, int64_t N, const tgp_kernel_sum* k /*host*/,
                       double* out, int64_t ld, void* stream);
/* tgp_loglike (row_end == NULL) or tgp_loglike_env (row_end != NULL). */
int tgp_loglike_sum(const double* X, const double* y, const double* yerr2, int64_t N, const tgp_kernel_sum* k /*host*/,
                    double* work, int64_t ld, double* alpha, int want_alpha, double* out, int32_t* info,
                    const int64_t* row_end /*host*/, int64_t nblocks, void* stream);
/* tgp_loglike_grad for a sum: out: device double[4 + 4 nterms] = {logL, chi2, logdet, then per term c
 * d logL / d (ln amp_c, m00_c, m01_c, m11_c) at out[3 + 4c ..], then d logL / d ln white at out[3 + 4 nterms]
 * (0 when white == 0)}.  scratch: 16-byte aligned, tgp_loglike_grad_sum_work_doubles(N, nterms) doubles. */
int64_t tgp_loglike_grad_sum_work_doubles(int64_t N, int32_t nterms);
int tgp_loglike_grad_sum(const double* X, const double* y, const double* yerr2, int64_t N,
                         const tgp_kernel_sum* k /*host*/, double* work, int64_t ld, double* alpha, double* out,
                         int32_t* info, const int64_t* row_end /*host*/, int64_t nblocks, double* scratch,
                         void* stream);
/* tgp_predict_mean / tgp_predict_mean_trunc for a sum (no white term: it is zero between distinct point sets).
 * The truncated form skips a group only beyond every term's cut-off; the error bound is
 * 1e-40 * sum_c |amp_c| * sum_n |alpha_n|. */
int tgp_predict_mean_sum(const double* Xs, int64_t M, const double* X, int64_t N, const tgp_kernel_sum* k /*host*/,
                         const double* alpha, double* mean, void* stream);
int tgp_predict_mean_trunc_sum(const double* Xs, int64_t M, const double* X, int64_t N,
                               const tgp_kernel_sum* k /*host*/, const double* alpha, double* mean, double* work,
                               void* stream);
/* var[m] = sum_c amp_c + white - || L^-1 K(X, Xs_m) ||^2 (tgp_predict_var; row_end optional as tgp_predict_var_env). */
int tgp_predict_var_sum(const double* Xs, int64_t M, const double* X, int64_t N, const tgp_kernel_sum* k /*host*/,
                        const double* L, int64_t ld, const int64_t* row_end /*host*/, int64_t nblocks, double* work,
                        int64_t chunk, double* var, void* stream);

/* ---- (2e) several outputs sharing one kernel ---------------------------------------------------------------------
 * r fields measured at the same points with the same errors are r independent GPs with one covariance: K + diag(yerr2)
 * is built and factorised once for all of them.  Every (N, r) or (M, r) matrix is row-major (numpy's layout);
 * 1 <= r <= TGP_MAX_RHS.  The kernel is always a tgp_kernel_sum (a single kernel is a one-term sum).  With r == 1
 * each entry gives bit for bit what its single-output twin gives.  Arguments are checked before any CUDA call. */
#define TGP_MAX_RHS 8
/* tgp_loglike_sum for r outputs.  work: (N + r) x ld (r extra rows carry the outputs through the factorisation).
 * alpha: device double[N * r] = K^-1 Y, or L^-1 Y when want_alpha == 0; each column equals the single-output
 * alpha of that column bit for bit.  out: device double[3] = {sum_c logL_c, sum_c chi2_c, logdet}, i.e.
 * logL = -1/2 sum_c y_c^T K^-1 y_c - r/2 ln|K| - r N/2 ln 2 pi; -inf when *info > 0. */
int tgp_loglike_multi(const double* X, const double* Y, int32_t r, const double* yerr2, int64_t N,
                      const tgp_kernel_sum* k /*host*/, double* work, int64_t ld, double* alpha, int want_alpha,
                      double* out, int32_t* info, const int64_t* row_end /*host*/, int64_t nblocks, void* stream);
/* tgp_loglike_grad_sum for r outputs: the gradient of the joint logL, 1/2 tr((sum_c alpha_c alpha_c^T - r K^-1) dK/dp);
 * d / d ln white = 1/2 white (sum_c |alpha_c|^2 - r tr K^-1).  out has the layout of tgp_loglike_grad_sum.
 * scratch: 16-byte aligned, tgp_loglike_grad_multi_work_doubles(N, nterms, r) doubles. */
int64_t tgp_loglike_grad_multi_work_doubles(int64_t N, int32_t nterms, int32_t r);
/* tgp_potrs_vec for r right-hand sides: B holds r rows of N at pitch ld (the factor's ld), solved in place.  Both
 * sweeps stream the factor once for all of them; each row equals its own tgp_potrs_vec result bit for bit. */
int tgp_potrs_multi(const double* L, int64_t N, int64_t ld, double* B, int32_t r, void* stream);
int tgp_loglike_grad_multi(const double* X, const double* Y, int32_t r, const double* yerr2, int64_t N,
                           const tgp_kernel_sum* k /*host*/, double* work, int64_t ld, double* alpha, double* out,
                           int32_t* info, const int64_t* row_end /*host*/, int64_t nblocks, double* scratch,
                           void* stream);
/* mean (M, r) = K(Xs, X) alpha (alpha: (N, r)); each pair's profile is evaluated once for all r outputs.  The
 * truncated form skips what tgp_predict_mean_trunc_sum skips; work: tgp_predict_work_doubles(N) doubles. */
int tgp_predict_mean_multi(const double* Xs, int64_t M, const double* X, int64_t N, const tgp_kernel_sum* k /*host*/,
                           const double* alpha, int32_t r, double* mean, void* stream);
int tgp_predict_mean_trunc_multi(const double* Xs, int64_t M, const double* X, int64_t N,
                                 const tgp_kernel_sum* k /*host*/, const double* alpha, int32_t r, double* mean,
                                 double* work, void* stream);

/* ---- (2f) batches of independent problems ------------------------------------------------------------------------
 * B problems, each with its own points, values, errors and kernel, in one call: every launch of the dense chain
 * (K build, the panel steps of the Cholesky, the reductions) carries all of them, so that a batch of small problems
 * takes about the launch latency of its largest one.  Problem b owns rows [off[b], off[b+1]) of the concatenated
 * X (total x ndim), y, yerr2 and alpha; N_b = off[b+1] - off[b], 1 <= N_b <= TGP_BATCH_MAX_N.  ks[b] is its kernel (a
 * one-term sum for a single kernel); one ndim for the whole batch.  off, soff and ks are HOST arrays; the entries
 * stage them to the device themselves (stream-ordered allocation on `stream`).  Problems never influence one
 * another: a problem's results are the same bit for bit whatever other problems share the batch and in whatever
 * order.  The factorisation is always dense (no envelope).  Arguments are checked before any CUDA call. */
#define TGP_BATCH_MAX_N 4096
/* sum_b (N_b + 1) * ld_b doubles, ld_b = N_b rounded up to even; -1 for invalid B / off. */
int64_t tgp_batch_work_doubles(const int64_t* off /*host*/, int32_t B);
/* tgp_loglike_sum (dense, row_end == NULL) for every problem.  work: tgp_batch_work_doubles doubles, 16-byte aligned;
 * problem b's (N_b + 1) x ld_b block starts at sum_{c < b} (N_c + 1) ld_c and holds on exit what tgp_loglike_sum
 * leaves in its work (the factor in the lower triangle, L^-1 y in row N_b).  yerr2 is required (zeros for none).
 * out: device double[3 B] = {logL, chi2, logdet} per problem, info: device int32[B], each with the meaning of
 * tgp_loglike (logL = -inf for info > 0, NaN for info < 0).  want_alpha == 0: out, info and the factor equal
 * tgp_loglike_sum on that problem alone bit for bit, alpha = L^-1 y.  want_alpha != 0: alpha = K^-1 y from a batched
 * backward sweep (one CTA per problem), which may differ from the single call's sweep in the last bits, and
 * chi2 = y . alpha. */
int tgp_loglike_batch(const double* X, const double* y, const double* yerr2, const int64_t* off /*host*/, int32_t B,
                      const tgp_kernel_sum* ks /*host*/, double* work, double* alpha, int want_alpha, double* out,
                      int32_t* info, void* stream);
/* mean rows [soff[b], soff[b+1]) = K_b(Xs_b, X_b) alpha_b, the full (untruncated) sum of tgp_predict_mean_sum summed
 * in one pass over the training points (soff non-decreasing from 0: a problem may have no test points).  Equal bit
 * for bit to tgp_predict_mean_sum wherever that call runs unsplit (N_b <= 1024 or many test points). */
int tgp_predict_mean_batch(const double* Xs, const int64_t* soff /*host*/, const double* X, const int64_t* off /*host*/,
                           int32_t B, const tgp_kernel_sum* ks /*host*/, const double* alpha, double* mean,
                           void* stream);
/* per-problem scratch of tgp_loglike_grad_batch: sum_b of the single gradient's scratch for N_b with
 * 4 TGP_MAX_TERMS + 1 partial columns (tgp_loglike_grad_sum_work_doubles(N_b, TGP_MAX_TERMS)); problem b's block
 * starts at the sum over c < b.  -1 for invalid B / off. */
int64_t tgp_loglike_grad_batch_work_doubles(const int64_t* off /*host*/, int32_t B);
/* tgp_loglike_grad_sum (dense, row_end == NULL) for every problem of a batch.  Arguments as tgp_loglike_batch, plus
 * scratch (tgp_loglike_grad_batch_work_doubles doubles, 16-byte aligned).
 * out: device double[B * TGP_GRAD_BATCH_OUT].  Problem b's slice has tgp_loglike_grad_sum's layout for ks[b]:
 * {logL, chi2, logdet, 4 derivatives per term, d / d ln white} (one term without white: 4 derivatives, then 0).
 * Unused tail entries are 0.  The gradient is 0 where info_b != 0.  On exit each problem's work block holds Z = K^-1
 * (lower triangle, mirrored into the upper), equal to tgp_selinv on its factor bit for bit, and alpha = K^-1 y as with
 * want_alpha != 0.  So logL, chi2 and logdet are tgp_loglike_batch's, and the gradient agrees with
 * tgp_loglike_grad_sum on that problem alone to the rounding of alpha. */
#define TGP_GRAD_BATCH_OUT (4 + 4 * TGP_MAX_TERMS)
int tgp_loglike_grad_batch(const double* X, const double* y, const double* yerr2, const int64_t* off /*host*/,
                           int32_t B, const tgp_kernel_sum* ks /*host*/, double* work, double* alpha, double* out,
                           int32_t* info, double* scratch, void* stream);

/* ---- (4) predict ----------------------------------------------------------------------------- */

/* mean[m] = sum_n K(Xs_m, X_n) alpha_n without materialising K(Xs, X).
 * Replaces HT = kernel(X2, Y=X1); np.dot(HT, alpha)  (gp_interp.py:177,183). */
int tgp_predict_mean(const double* Xs, int64_t M, const double* X, int64_t N,
                     const tgp_kernel* k /*host*/, const double* alpha, double* mean, void* stream);

/* Same sum with compact-support truncation: groups of 128 training points whose bounding box lies farther
 * than q_cut (f(q_cut) = 1e-40, tgp_profile_qcut) from the bounding box of a block of 256 test points are
 * skipped, which changes mean[m] by at most 1e-40 * sum_n |amp alpha_n|.  Correct for any point order; fast
 * when Xs and X (with alpha) are both stored along a space-filling curve (tgp_hilbert_keys).
 * work: device scratch of tgp_predict_work_doubles(N) doubles (bounding boxes). */
int tgp_predict_mean_trunc(const double* Xs, int64_t M, const double* X, int64_t N,
                           const tgp_kernel* k /*host*/, const double* alpha, double* mean, double* work,
                           void* stream);
int64_t tgp_predict_work_doubles(int64_t N);
/* q beyond which the correlation profile of `family` is below 1e-40. */
double tgp_profile_qcut(int32_t family);

/* var[m] = amp - || L^-1 K(X, Xs_m) ||^2, the diagonal of gp_interp.py:190-191.
 * work: 16-byte aligned device buffer of at least chunk*(N+1) doubles; `chunk` test points are
 * processed at a time (K(Xs_chunk, X) is materialised there, then solved in place on the DMMA pipe). */
int tgp_predict_var(const double* Xs, int64_t M, const double* X, int64_t N,
                    const tgp_kernel* k /*host*/, const double* L, int64_t ld, double* work,
                    int64_t chunk, double* var, void* stream);

/* tgp_predict_var on a factor with a known envelope (tgp_potrf_env / tgp_loglike_env; X in the factor's order). */
int tgp_predict_var_env(const double* Xs, int64_t M, const double* X, int64_t N,
                        const tgp_kernel* k /*host*/, const double* L, int64_t ld, const int64_t* row_end /*host*/,
                        int64_t nblocks, double* work, int64_t chunk, double* var, void* stream);

/* out[m] = uniform mean of y0 over the k grid points nearest to Xq_m (squared Euclidean distance, exact ties
 * towards the lower grid index, values summed in order of increasing distance).  Replaces
 * KNeighborsRegressor(n_neighbors=k).fit(X0, y0).predict(Xq), the mean-function lookup of
 * gp_interp.py:236-238.  Xq: (M, ndim), X0: (n0, ndim), y0: n0.  1 <= k <= min(n0, 16). */
int tgp_knn_mean(const double* Xq, int64_t M, const double* X0, const double* y0, int64_t n0,
                 int32_t ndim, int32_t k, double* out, void* stream);

/* ---- (3) two-point correlation function ------------------------------------------------------ */

typedef enum {
  TGP_BIN_TWOD = 0, /* treecorr bin_type="TwoD", bin_slop=0 (two_pcf.py:297-305) */
  TGP_BIN_LOG = 1   /* treecorr default Log binning in the bin_slop -> 0 limit (two_pcf.py:330-334) */
} tgp_bintype;

/* Brute-force pair binning of one or several catalogues (a bootstrap batch is ncat > 1).
 *
 *  px, py, pk, pw : concatenated point arrays (total = cat_off[ncat]); pk is the scalar field k,
 *                   pw the weights w or NULL (unit weights).
 *  cat_off        : device int64[ncat+1]; catalogue c owns points [cat_off[c], cat_off[c+1]).
 *  max_cat_len    : host upper bound on the catalogue lengths (sizes the launch).
 *  edges          : device double[nbins+1] of decision THRESHOLDS: edges[k] (1 <= k < nbins) is the
 *                   smallest double that the binning formula sends to bin >= k, so that
 *                   bin(v) = #{k in 1..nbins-1 : v >= edges[k]} reproduces the formula bit for bit.
 *                   TwoD additionally needs edges[0] = -inf and edges[nbins] = +inf.
 *  TGP_BIN_TWOD   : with (dx,dy) = p_j - p_i and r2 = dx*dx + dy*dy (un-fused), a pair is kept iff
 *                   r2 != 0, r2 >= min_sep2 and max(|dx|,|dy|) < max_sep; column = bin(dx),
 *                   row = bin(dy), flat index row*nbins + column (nb = nbins^2).  Every unordered
 *                   pair is entered twice, at (dx,dy) and at (-dx,-dy).
 *  TGP_BIN_LOG    : kept iff min_sep2 <= r2 < max_sep^2; index = bin(r2) (nb = nbins); every
 *                   unordered pair entered once.
 *  tile_rank, tile_nranks : multi-GPU sharding -- runs of pair tiles are dealt round-robin; rank
 *                   r of n computes a disjoint subset and the per-rank outputs add up to the
 *                   single-GPU result (counts exactly; FP64 sums up to summation order).
 *  npairs         : device int64[ncat*nb]   pair counts
 *  sumw           : device double[ncat*nb]  sum w_i w_j
 *  sumwkk         : device double[ncat*nb]  sum w_i k_i w_j k_j
 *  sumwr          : device double[ncat*nb]  sum w_i w_j r   (LOG only; may be NULL)
 * Outputs are ACCUMULATED into (the caller zeroes them).  xi = sumwkk / sumw is left to the caller
 * so that multi-GPU partial sums can be all-reduced first.
 *  work           : optional 32-byte aligned device scratch of tgp_pairbin_work_doubles(total, ncat)
 *                   doubles (bounding boxes, sums and sorted copies of the 32-point chunks, filled by a
 *                   pre-pass; for TwoD also the block records and work counters of the two-pass count, see
 *                   below).  NULL: no block forms (TwoD: pair by pair; Log: the boxes are recomputed on the fly);
 *                   the counts are the same.
 * TwoD with work first books the pairs of super-chunks (256 consecutive points) that sit in one bin or vary along
 * one axis only, and decides the 32-point blocks of the super pairs that span at most 2 x 2 bins (the range edge
 * counting as one) in one more kernel.  Then it runs in rounds of this rank's items: a classification pass books the
 * other blocks that sit in one bin and records the rest, then a second kernel processes the recorded blocks.  A round holds at most
 * 2^26 records (1 GiB of `work` at N >= ~4e5; fewer for smaller catalogues), about 8 rounds at N = 1e6. */
int tgp_pairbin(const double* px, const double* py, const double* pk, const double* pw,
                const int64_t* cat_off, int32_t ncat, int64_t max_cat_len, int32_t bin_type,
                const double* edges, int32_t nbins, double min_sep2, double max_sep,
                int32_t tile_rank, int32_t tile_nranks, int64_t* npairs, double* sumw,
                double* sumwkk, double* sumwr, double* work, void* stream);

/* Size (in doubles) of the optional scratch buffer of tgp_pairbin for catalogues of `total_points` points in
 * all (an upper bound on max_cat_len is enough): the chunk records of the pre-pass, the super-chunk records
 * (boxes, sums and sorted copies of 256-point super-chunks, about 48 MB at N = 1e6), a list with room for every
 * pair of super-chunks (16 bytes each: S (S - 1) / 2 entries for S = total_points / 256, about 122 MB at N = 1e6)
 * and the block records of one round, capped at 2^26 records of 16 bytes. */
int64_t tgp_pairbin_work_doubles(int64_t total_points, int32_t ncat);

/* Hilbert-curve keys of 2-D points on a 2^order x 2^order grid over the square
 * [xmin, xmin+extent) x [ymin, ymin+extent).  tgp_pairbin is correct for any point order, but when the
 * catalogue is sorted by this key (torch.argsort on the caller's side) neighbouring points are stored
 * together and the kernel's register-accumulation path applies (no shared-memory atomics in the inner
 * loop).  keys: device int64[n]. */
int tgp_hilbert_keys(const double* x, const double* y, int64_t n, double xmin, double ymin, double extent,
                     int32_t order, int64_t* keys, void* stream);

/* The same keys with the bounding square (xmin, ymin, extent = max side * (1 + 1e-9)) found on the device, so that
 * the caller does not have to read the extrema back in the middle of a call.  scratch32: device scratch of 32 bytes
 * (8-byte aligned). */
int tgp_hilbert_keys_auto(const double* x, const double* y, int64_t n, int32_t order, void* scratch32,
                          int64_t* keys, void* stream);

/* HOST function (no device work): multiplicities of `b` bootstrap resamples of n points, bit-identical to
 * b successive numpy `Generator(PCG64).integers(0, n-1, size=n)` calls -- the draws of resample_bootstrap
 * (two_pcf.py:266,269-281; index n-1 is never drawn).
 *  state : host uint64[6] = {state_hi, state_lo, inc_hi, inc_lo, has_uint32, uinteger} taken from numpy's
 *          `bit_generator.state`; updated on return to the state numpy would be in after the same calls.
 *  pos   : host int64[n] or NULL; draws of point i are counted at column pos[i] (e.g. its rank along the
 *          Hilbert curve, so the multiplicities come out in storage order).
 *  mult  : host uint8[b * n], overwritten.  More than 255 draws of one point -> TGP_ERR_UNSUPPORTED. */
int tgp_bootstrap_multiplicities(uint64_t* state, int64_t n, int64_t b, const int64_t* pos, uint8_t* mult);

/* Bootstrap batch of the TwoD two-point function with the pair geometry shared by all resamples (replaces the loop
 * of two_pcf.py:342-362: n_bootstrap x [resample_bootstrap :269-281 + comp_2pcf :283-328]).  A resample is the BASE
 * catalogue with integer multiplicities; TreeCorr skips the zero-distance pairs between copies of a point, so with
 * a_b[i] = mult[b][i] * w_i and c_b[i] = a_b[i] * z_i the sums over the pairs (i < j) of the base catalogue in a bin
 *     S0 = sum a_i a_j,  S1 = sum (c_i a_j + a_i c_j),  S2 = sum c_i c_j
 * give sumw = S0 and, with delta_b = sum_i mult[b][i] z_i / n (the mean of the resampled values, np.mean(y) of
 * two_pcf.py:297), sumwkk = S2 - delta_b S1 + delta_b^2 S0.
 *  px, py, pz, pw : device double[n], the base catalogue (Hilbert order recommended, see tgp_hilbert_keys); pz the
 *                   field minus ANY fixed constant (e.g. its mean); pw the weights or NULL (unit weights).
 *  mult           : device uint8[nboot * n], resample-major (the layout tgp_bootstrap_multiplicities writes).
 *  edges, nbins, min_sep2, max_sep : as for tgp_pairbin with TGP_BIN_TWOD (same thresholds, same pair rule).
 *  tile_rank, tile_nranks : multi-GPU sharding of the work items; the per-rank `sums` add up.
 *  sums           : device double[tgp_bootbin_sums_doubles(nbins, nboot)] = [2][3][nbins^2][bpad], bpad = nboot
 *                   rounded up to a multiple of 32; OVERWRITTEN: forward-entry sums S0, S1, S2 per bin and resample,
 *                   then corrections for pairs whose mirrored bin is not the mirror image of the forward bin.
 *  delta          : device double[bpad], overwritten (identical on every rank).
 *  work           : device scratch of tgp_bootbin_work_bytes(n, nboot) bytes, 256-byte aligned.
 * tgp_bootbin_xi turns (all-reduced) sums into xi[nboot][nbins^2] = sumwkk / sumw (0 where sumw == 0) and, if
 * sumw_out != NULL, sumw[nboot][nbins^2]. */
int tgp_bootbin_twod(const double* px, const double* py, const double* pz, const double* pw, int64_t n,
                     const uint8_t* mult, int32_t nboot, const double* edges, int32_t nbins, double min_sep2,
                     double max_sep, int32_t tile_rank, int32_t tile_nranks, double* sums, double* delta,
                     void* work, void* stream);
int tgp_bootbin_xi(const double* sums, const double* delta, int32_t nbins, int32_t nboot, double* xi,
                   double* sumw_out, void* stream);
int64_t tgp_bootbin_work_bytes(int64_t n, int32_t nboot);
int64_t tgp_bootbin_sums_doubles(int32_t nbins, int32_t nboot);
/* Diagnostics: blocks per path of all tgp_bootbin_twod launches since the last reset: [0] booked whole, [1] axis
 * sweeps, [2] pair-by-pair blocks, [3] exact per-pair blocks, [4] window flushes, [5] sweeps handed back,
 * [6] wide-window blocks summed bin by bin. */
int tgp_bootbin_stats(unsigned long long* host8 /*host*/, int reset);

/* Pair sums of a VECTOR field's 2-point functions in log-radius bins (E/B diagnostics; replaces the all-pairs numpy
 * loop of utils.py:5-74 and TreeCorr's VVCorrelation of utils.py:110-155 in the bin_slop -> 0 limit).
 *  x, y, vx, vy : n points and the vector field there.
 *  edges        : device double[nbins+1] thresholds on r^2 (treegp_b200.binning.hist_thresholds_r2): edges[k] = h_k^2,
 *                 h_k the smallest double with np.log(h_k) >= bin_edges[k] of the reference's np.histogram call
 *                 (utils.py:52-55; for k = nbins: > instead of >=, the last bin is closed).  A pair with d = z_j - z_i,
 *                 r2 = |d|^2 != 0 goes to bin k = #{0 <= m <= nbins : r2 >= edges[m]} - 1 if that is in [0, nbins).
 *  counts       : device int64[nbins], ACCUMULATED.
 *  sums         : device double[6 * nbins], ACCUMULATED: {ln r, Re(v_i conj v_j), Re(v_i v_j), Im(v_i v_j),
 *                 Re(v_i v_j conj(d)^2 / r2), Im(same)} each over nbins.
 *  amb_pairs    : device int64[2 * amb_cap]: pairs (i, j) whose r2 lies within 1e-14 (relative) of a threshold are
 *                 NOT accumulated -- hypot() of the reference and sqrt(r2) may round to different sides there --
 *                 but listed here for the caller to settle with the reference's own expression.
 *  amb_count    : device int32[1], ACCUMULATED: number of such pairs (may exceed amb_cap: then the list is
 *                 truncated and the caller must retry with a larger one). */
int tgp_vcorr(const double* x, const double* y, const double* vx, const double* vy, int64_t n,
              const double* edges, int32_t nbins, int64_t* counts, double* sums, int64_t* amb_pairs,
              int32_t amb_cap, int32_t* amb_count, void* stream);

/* Batched chi-square of the robust anisotropic fit: for each of `nsets` parameter triples (size, g1, g2) the objective
 * robust_2dfit.chi2 (two_pcf.py:115-148) -- model profile of `family` (TGP_FAM_RBF | TGP_FAM_VONKARMAN) at the P masked
 * bin lags for the correlation-length matrix of (size, g1, g2) (two_pcf.py:12-31), analytic amplitude and offset,
 * chi2 = r^T W r; +inf outside |g| <= 1 or for non-finite parameters.
 *  coord : device double[2 P] (dx, dy) of the masked pixels;  y : device double[P] masked xi;  W : device double[P * P];
 *  params: device double[3 nsets];  out : device double[4 nsets] = {chi2, |amplitude|, offset, 1 if evaluated}. */
int tgp_robust_chi2_batch(const double* coord, const double* y, const double* W, int32_t P, int32_t family,
                          const double* params, int32_t nsets, double* out, void* stream);

/* ---- the exchange step of the sharded pair binning (SURVEY.md section 8b / 8e) ----------------------------------
 * NCCL bound at run time (dlopen); TGP_ERR_UNSUPPORTED if no libnccl can be found.
 *  tgp_comm_unique_id : rank 0 fills 128 bytes that every rank must pass to tgp_comm_init_rank (ship them by any means).
 *  tgp_comm_init_rank : collective over the `nranks` processes (one GPU each, the current device); *comm receives an
 *                       opaque handle.
 *  tgp_allreduce_bins : in-place sum over the ranks of the packed bin buffer that tgp_pairbin filled on each rank:
 *                       `planes` x `per_plane` doubles (plane 0 = the int64 pair counts as raw 8-byte words, then sumw,
 *                       sumwkk[, sumwr], per_plane = ncat * nb).  Plane 0 is reduced as FP64 VALUES (exact below 2^53)
 *                       and converted back, so on return it holds int64 counts again -- identical for any number of
 *                       ranks.  Asynchronous on `stream`. */
int tgp_comm_unique_id(void* id128 /*host, 128 bytes*/);
int tgp_comm_init_rank(const void* id128 /*host*/, int32_t rank, int32_t nranks, void** comm /*host*/);
int tgp_comm_destroy(void* comm);
int tgp_allreduce_bins(void* comm, double* packed, int64_t planes, int64_t per_plane, void* stream);

/* Sticky device-side error word: set (never cleared by the kernels) when an inter-CTA flag wait inside
 * tgp_potrs_vec / tgp_loglike(want_alpha) timed out -- which cannot happen with the cooperative launch those
 * sweeps use, but would otherwise leave unknowns unsolved without any other sign.  Synchronises the device and
 * returns the word (0 = fine, < 0 = the query itself failed); reset != 0 clears it. */
int tgp_device_error(int reset);

/* Points per pair block: 32 (informational). */
int tgp_pairbin_tile(void);

/* Diagnostics: how many pairs (32 x columns per processed block) of all tgp_pairbin launches since the last
 * reset went through each path: host8[0] closed form (whole block in one bin and its mirror image; TwoD: booked by
 * the classification pass, the other slots by the pass over the recorded blocks), [1] one
 * varying axis (one compare pair per pair of points), [2] pair by pair in a 2 x 2 bin window or through the
 * generic path (the diagonal blocks are not tallied), [3] one varying axis answered by a rank query on the
 * chunk's sorted copy (8 probes per row point instead of 32 compares), [4] 2 x 2 bin window with the column-bit
 * and row-bit sums from two such rank queries and only the "both bits" quadrant summed pair by pair, [5] (TwoD)
 * super-chunk pair in one bin, booked whole, [6] (TwoD) super-chunk pair with one varying axis, one rank query per row
 * point on the super-chunk's sorted copy.  The slots are disjoint.  Synchronous. */
int tgp_pairbin_stats(unsigned long long* host8 /*host*/, int reset);

/* Diagnostics: how many super-chunk pairs of all TwoD tgp_pairbin launches since the last reset spanned at most two
 * bins per axis (the range edge counting as one) and had their 32-point blocks decided by the leaf kernel without
 * block records.  Their blocks are tallied in the slots of tgp_pairbin_stats as usual.  Synchronous. */
int tgp_pairbin_super_leaves(unsigned long long* host1 /*host*/, int reset);
/* Diagnostics: how many of those super-chunk pairs were decided per row point against the column super-chunk staged
 * in shared memory (the others went block by block, after a failed mirrored-bit check or when the staged tables do not
 * fit).  Synchronous. */
int tgp_pairbin_super_rows(unsigned long long* host1 /*host*/, int reset);

/* Test and measurement switches of the pair counts (tgp_pairbin_*, tgp_bootbin_twod), not needed for normal use.
 * Any other name is rejected with TGP_ERR_INVALID ("unknown option").
 * "pairbin_block_sums": 0 = every pair of every in-range block is evaluated individually (no block forms);
 * "pairbin_fast_paths": bit mask, default all on; bit 0 = short-cut dispatch of one-axis blocks that fit the open
 * bin window, bit 1 = 2 x 2-window blocks take their marginal sums from rank queries, bit 2 = the pair-by-pair kernel
 * ("pairbin_block_sums" 0) skips the per-pair mirrored-bin check in blocks whose bounding boxes prove it
 * (0 = the general paths only; results are identical either way); "pairbin_record_cap": block records per round of
 * the two-pass TwoD count, at least 256, at most (and <= 0: back to) the default 2^26 -- more, smaller rounds; "bootbin_paths": bit mask of tgp_bootbin_twod,
 * default all on; bit 0 = blocks in one bin booked from chunk sums, bit 1 = window paths (0: every block through the
 * exact per-pair path), bit 2 = axis sweeps, bit 3 = blocks spanning more than 2 x 2 bins summed bin by bin. */
int tgp_set_option(const char* name, int value);

/* ---- measurement helpers --------------------------------------------------------------------- */

/* FP64 micro-peaks used as roofline denominators.  kind 0: DFMA (FP64 FMA pipe), 1: DMMA
 * (mma.sync m8n8k4 f64).  Synchronous.  Writes achieved TFLOP/s to *tflops (host).
 * kind 2 / 3: launch-latency probe -- microseconds per launch of a chain of `iters` dependent empty kernels,
 * plain / with programmatic dependent launch (returned through *tflops). */
int tgp_microbench_fp64(int kind, int iters, double* tflops /*host*/);

#ifdef __cplusplus
}
#endif
#endif /* TREEGP_B200_H */
