// Selected inverse of the covariance inside the envelope of its Cholesky factor, and the analytic gradient of the
// marginal log-likelihood that it makes possible.
//
// tgp_selinv: Z = (L L^T)^-1 on every entry of the envelope of L (the dense matrix when there is no envelope), by the
// blocked Takahashi recurrence.  For the OB-wide block columns J from last to first, R = [end of J, row_end[J]) the
// envelope rows below J, L11 = L[J, J], L21 = L[R, J]:
//   W       = L11^-1                      (stored as -W^T: tgp_trsm_rows on -I, i.e. the DMMA halving solver)
//   T^T     = W^T L21^T                   (gemm_nt_sub into zeroed scratch)
//   Z[R, J] = -Z[R, R] T                  (gemm_nt_sub over L21's storage; Z[R, R] is dense in memory thanks to the
//                                          mirror into the upper triangle, which the kernel build never writes)
//   Z[J, J] = W^T W - T^T Z[R, J]         (two lower-only gemm_nt_sub, the second with B = the mirrored Z[J, R])
// Z[R, R] lies inside the envelope because row_end is non-decreasing, so nothing outside it is read or written.
// Flops: 2 w m^2 + 3 w^2 m + 2 w^3 per block column (w = OB, m = |R|), about twice the factorisation's w m^2 + w^2 m.
//
// tgp_loglike_grad: K build -> factorisation -> both sweeps (alpha = K^-1 y) -> tgp_selinv -> one fused contraction
// over the lower triangle inside the envelope: with w_ij = alpha_i alpha_j - Z_ij and K_ij = a f(q_ij),
//   d logL / d ln a = 1/2 sum_ij w_ij a f(q_ij),   d logL / d m_uv = 1/2 sum_ij w_ij a f'(q_ij) d q_ij / d m_uv.
#include <string.h>
#include <algorithm>
#include "tgp_common.cuh"
#include "profile_dq.cuh"
#include "profile_policy.cuh"
#include "batch.cuh"

extern "C" int tgp_trsm_rows(const double* L, int64_t N, int64_t ld, double* B, int64_t M, int64_t ldb, void* stream);
extern "C" int tgp_gemm_nt_sub(double* C, int64_t M, int64_t Nc, int64_t ldc, const double* A, int64_t lda,
                               const double* B, int64_t ldb, int64_t Kd, int lower_only, void* stream);
extern "C" int tgp_loglike(const double* X, const double* y, const double* yerr2, int64_t N, const tgp_kernel* k,
                           double* work, int64_t ld, double* alpha, int want_alpha, double* out, int32_t* info,
                           void* stream);
extern "C" int tgp_loglike_env(const double* X, const double* y, const double* yerr2, int64_t N, const tgp_kernel* k,
                               double* work, int64_t ld, double* alpha, int want_alpha, double* out, int32_t* info,
                               const int64_t* row_end, int64_t nblocks, void* stream);
extern "C" int tgp_loglike_sum(const double* X, const double* y, const double* yerr2, int64_t N,
                               const tgp_kernel_sum* k, double* work, int64_t ld, double* alpha, int want_alpha,
                               double* out, int32_t* info, const int64_t* row_end, int64_t nblocks, void* stream);
extern "C" int tgp_loglike_multi(const double* X, const double* Y, int32_t r, const double* yerr2, int64_t N,
                                 const tgp_kernel_sum* k, double* work, int64_t ld, double* alpha, int want_alpha,
                                 double* out, int32_t* info, const int64_t* row_end, int64_t nblocks, void* stream);

constexpr int GT = 64;             // contraction tile edge
constexpr int GT_THREADS = 256;

static int64_t even64(int64_t n) { return (n + 1) & ~(int64_t)1; }
static int64_t grad_tiles(int64_t N) {
  const int64_t nt = tgp_cdiv(N, GT);
  return nt * (nt + 1) / 2;
}

// ncols partial sums per contraction tile: 4 for one term, 4 nterms + 1 for a sum
static int64_t grad_work_doubles(int64_t N, int ncols) {
  if (N < 1) N = 1;
  const int64_t selinv = 2 * (int64_t)TGP_OB * TGP_OB + (int64_t)TGP_OB * even64(N);   // -W^T, W^T, T^T
  const int64_t partials = ncols * grad_tiles(N);                           // contraction partial sums
  return (selinv > partials ? selinv : partials) + even64(tgp_cdiv(N, TGP_OB));  // + the device copy of row_end
}

extern "C" int64_t tgp_selinv_work_doubles(int64_t N) { return grad_work_doubles(N, 4); }

extern "C" int64_t tgp_loglike_grad_sum_work_doubles(int64_t N, int32_t nterms) {
  if (nterms < 1 || nterms > TGP_MAX_TERMS) return -1;
  return grad_work_doubles(N, 4 * nterms + 1);
}

// the outputs change the contraction's weights, not its partial sums
extern "C" int64_t tgp_loglike_grad_multi_work_doubles(int64_t N, int32_t nterms, int32_t r) {
  if (r < 1 || r > TGP_MAX_RHS) return -1;
  return tgp_loglike_grad_sum_work_doubles(N, nterms);
}

// ---- small helpers --------------------------------------------------------------------------------------------
// S (n x n, pitch lds) = -I
__global__ void neg_identity_kernel(double* __restrict__ S, int n, int64_t lds) {
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < (int64_t)n * n;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / n, c = idx % n;
    S[r * lds + c] = (r == c) ? -1.0 : 0.0;
  }
}

// D (n x n) = -S
__global__ void negate_kernel(const double* __restrict__ S, double* __restrict__ D, int n, int64_t ld) {
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < (int64_t)n * n;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / n, c = idx % n;
    D[r * ld + c] = -S[r * ld + c];
  }
}

// dst[c][r] = src[r][c] for the rows x cols block src (both with pitch ld).  lower_only: src == dst is a square
// diagonal block whose strict lower triangle is mirrored into its upper triangle (disjoint entries: no race).
// The 32 x 32 tile whose top-left corner is (r0, c0).
__device__ __forceinline__ void mirror_body(const double* __restrict__ src, double* __restrict__ dst, int64_t rows,
                                            int64_t cols, int64_t ld, int lower_only, const int64_t r0,
                                            const int64_t c0) {
  __shared__ double t[32][33];
  if (lower_only && c0 > r0) return;
  const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t r = r0 + ty + 8 * i, c = c0 + tx;
    if (r < rows && c < cols && (!lower_only || c < r)) t[ty + 8 * i][tx] = src[r * ld + c];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t c = c0 + ty + 8 * i, r = r0 + tx;   // write row c of dst, coalesced along r
    if (r < rows && c < cols && (!lower_only || c < r)) dst[c * ld + r] = t[tx][ty + 8 * i];
  }
}

__global__ void __launch_bounds__(256)
mirror_kernel(const double* __restrict__ src, double* __restrict__ dst, int64_t rows, int64_t cols, int64_t ld,
              int lower_only) {
  mirror_body(src, dst, rows, cols, ld, lower_only, (int64_t)blockIdx.y * 32, (int64_t)blockIdx.x * 32);
}

static int mirror_launch(const double* src, double* dst, int64_t rows, int64_t cols, int64_t ld, int lower_only,
                         cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return TGP_OK;
  dim3 grid((unsigned)tgp_cdiv(cols, 32), (unsigned)tgp_cdiv(rows, 32));
  TGP_CHECK_ARG(grid.y <= 65535u, "too many rows for one launch");
  mirror_kernel<<<grid, dim3(32, 8), 0, st>>>(src, dst, rows, cols, ld, lower_only);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

static int check_args_mat(const double* A, int64_t N, int64_t ld) {
  return N <= 0 || ld < N || !A || (ld & 1) || ((uintptr_t)A & 15);
}

static int selinv_run(double* A, int64_t N, int64_t ld, const std::vector<int64_t>& re, double* scratch,
                      cudaStream_t st) {
  void* sv = (void*)st;
  double* NWT = scratch;                          // -W^T, TGP_OB x TGP_OB
  double* WT = scratch + TGP_OB * TGP_OB;         //  W^T, TGP_OB x TGP_OB
  double* TT = scratch + 2 * TGP_OB * TGP_OB;     //  T^T, TGP_OB x ldt
  const int64_t ldt = even64(N);
  const unsigned eg = 2 * (unsigned)tgp_num_sms();
  for (int64_t b = (int64_t)re.size() - 1; b >= 0; --b) {
    const int64_t k = b * TGP_OB, w = (N - k < TGP_OB) ? (N - k) : TGP_OB, c1 = k + w, m = re[(size_t)b] - c1;
    double* Akk = A + k * ld + k;
    double* L21 = A + c1 * ld + k;        // becomes Z[R, J]
    double* ZJR = A + k * ld + c1;        // upper-triangle storage of Z[J, R]
    int rc;
    neg_identity_kernel<<<eg, 256, 0, st>>>(NWT, (int)w, TGP_OB);
    TGP_LAUNCH_CHECK();
    rc = tgp_trsm_rows(Akk, w, ld, NWT, w, TGP_OB, sv);        // rows of -I times L11^-T: -W^T
    if (rc) return rc;
    negate_kernel<<<eg, 256, 0, st>>>(NWT, WT, (int)w, TGP_OB);
    TGP_LAUNCH_CHECK();
    if (m > 0) {
      TGP_CUDA(cudaMemset2DAsync(TT, ldt * sizeof(double), 0, m * sizeof(double), w, st));
      rc = tgp_gemm_nt_sub(TT, w, m, ldt, NWT, TGP_OB, L21, ld, w, 0, sv);          // T^T = W^T L21^T
      if (rc) return rc;
      TGP_CUDA(cudaMemset2DAsync(L21, ld * sizeof(double), 0, w * sizeof(double), m, st));
      rc = tgp_gemm_nt_sub(L21, m, w, ld, A + c1 * ld + c1, ld, TT, ldt, m, 0, sv);  // Z[R, J] = -Z[R, R] T
      if (rc) return rc;
      rc = mirror_launch(L21, ZJR, m, w, ld, 0, st);
      if (rc) return rc;
    }
    TGP_CUDA(cudaMemset2DAsync(Akk, ld * sizeof(double), 0, w * sizeof(double), w, st));
    rc = tgp_gemm_nt_sub(Akk, w, w, ld, NWT, TGP_OB, WT, TGP_OB, w, 1, sv);         // + W^T W
    if (rc) return rc;
    if (m > 0) {
      rc = tgp_gemm_nt_sub(Akk, w, w, ld, TT, ldt, ZJR, ld, m, 1, sv);               // - T^T Z[R, J]
      if (rc) return rc;
    }
    rc = mirror_launch(Akk, Akk, w, w, ld, 1, st);
    if (rc) return rc;
  }
  return TGP_OK;
}

extern "C" int tgp_selinv(double* L, int64_t N, int64_t ld, const int64_t* row_end, int64_t nblocks, double* scratch,
                          void* stream) {
  TGP_CHECK_ARG(!check_args_mat(L, N, ld), "L must be 16-byte aligned with even ld >= N > 0");
  TGP_CHECK_ARG(tgp_envelope_ok(row_end, nblocks, N), "row_end must hold one entry per tgp_envelope_block() columns");
  TGP_CHECK_ARG(scratch && ((uintptr_t)scratch & 15) == 0,
                "scratch: 16-byte aligned buffer of tgp_selinv_work_doubles(N) doubles");
  return selinv_run(L, N, ld, tgp_envelope_ends(row_end, N), scratch, (cudaStream_t)stream);
}

// ---- gradient contraction ---------------------------------------------------------------------------------------
// One CTA per 64 x 64 tile (I >= J) of the lower triangle; tiles whose rows all lie below the envelope of their
// block column write zeros.  Thread: 2 adjacent columns x 8 rows, as the K build (kmat.cu).  Partial sums
// {sum w a f, sum w a f' dx^2, sum w a f' 2 dx dy, sum w a f' dy^2} (off-diagonal pairs twice) per tile; the finishing
// kernel adds the tiles in index order, so the result does not depend on scheduling.
//
// Pairs outside the envelope are dropped, as by the factorisation: their q is at least tgp_profile_qcut, where
// f <= 1e-40 and |f'(q) q| is below (qcut / 2) f(qcut) ~ 2e-38 (RBF, q f' = -q f / 2 at qcut = 185), below
// 1e-36 for the von Karman profile (qcut = 224: |q f'| = pi sqrt(q) K_{1/6}/K_{5/6} f ~ 47 f) and below
// sqrt(q)/2 f, sqrt(3q) f, 5/6 (1 + sqrt(5q)) sqrt(5q) f ~ 1e-37 for the Matern families -- every dropped term is
// below 1e-36 a |w_ij| |dq / dm| / q.
//
// Sums (SumProfile): CTA (t, c) contracts term c of tile t into columns 4 c .. 4 c + 3 of the tile's 4 nterms + 1
// partials; the CTAs of term 0 also sum w_ii = alpha_i^2 - Z_ii over the diagonal, times the white level, into the
// last column (d K / d ln white = white I).
//
// Several outputs (P = MultiOut<..., TGP_MAX_RHS>, nrhs = r columns of alpha): w_ij = sum_c alpha_ic alpha_jc - r Z_ij.
template <class P>
__global__ void __launch_bounds__(GT_THREADS)
grad_contract_kernel(const double* __restrict__ X, int64_t N, P prof, const double* __restrict__ Z, int64_t ld,
                     const double* __restrict__ alpha, const int64_t* __restrict__ re_dev,
                     double* __restrict__ partials, const double* __restrict__ phi_g) {
#include "grad_contract_body.cuh"
}

// out[3 .. 3 + NC - 1] = 1/2 the tile sums of the NC partial columns in tile order; 0 when the factorisation failed
// (out[0] is then -inf already).  NC = 4 for one term, 4 nterms + 1 for a sum.
template <int NC>
__device__ __forceinline__ void grad_finish_body(const double* __restrict__ partials, int64_t ntiles,
                                                 const int32_t* __restrict__ info, double* __restrict__ out) {
  __shared__ double red[32][NC];
  double s[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) s[c] = 0.0;
  for (int64_t t = threadIdx.x; t < ntiles; t += blockDim.x) {
#pragma unroll
    for (int c = 0; c < NC; ++c) s[c] += partials[NC * t + c];
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[c] += __shfl_xor_sync(0xffffffffu, s[c], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int c = 0; c < NC; ++c) red[warp][c] = s[c];
  }
  __syncthreads();
  if (threadIdx.x < NC) {
    double v = 0.0;
    for (int wi = 0; wi < 32; ++wi) v += red[wi][threadIdx.x];
    out[3 + threadIdx.x] = (*info != 0) ? 0.0 : 0.5 * v;
  }
}

template <int NC>
__global__ void __launch_bounds__(1024)
grad_finish_kernel(const double* __restrict__ partials, int64_t ntiles, const int32_t* __restrict__ info,
                   double* __restrict__ out) {
  grad_finish_body<NC>(partials, ntiles, info, out);
}

static int grad_args(const double* X, const double* y, int64_t N, double* work, int64_t ld, const double* alpha,
                     const double* out, const int32_t* info, const int64_t* row_end, int64_t nblocks,
                     const double* scratch) {
  TGP_CHECK_ARG(N > 0 && X && y && alpha && out && info, "null pointer / N");
  TGP_CHECK_ARG(!check_args_mat(work, N, ld), "work must be 16-byte aligned with even ld >= N");
  TGP_CHECK_ARG(tgp_envelope_ok(row_end, nblocks, N), "row_end must hold one entry per tgp_envelope_block() columns");
  TGP_CHECK_ARG(scratch && ((uintptr_t)scratch & 15) == 0,
                "scratch: 16-byte aligned buffer of tgp_selinv_work_doubles(N) doubles");
  TGP_CHECK_ARG(grad_tiles(N) < (1ll << 31), "matrix too large for one launch");
  return TGP_OK;
}

// After the likelihood call (alpha = K^-1 y, the factor in `work`): the selected inverse, then the contraction over
// nterms x tiles CTAs into `ncols` partials per tile, then the finishing kernel.
template <class P>
static int grad_tail(const double* X, int64_t N, const P& prof, int nterms, int ncols, double* work, int64_t ld,
                     const double* alpha, double* out, const int32_t* info, const int64_t* row_end, double* scratch,
                     cudaStream_t st, int nrhs = 1) {
  const int64_t ntiles = grad_tiles(N);
  const std::vector<int64_t> re = tgp_envelope_ends(row_end, N);
  int rc = selinv_run(work, N, ld, re, scratch, st);
  if (rc) return rc;
  // the selected-inverse scratch is free again: tile partials at the front, the envelope at the back
  int64_t* re_dev = nullptr;
  if (row_end) {
    re_dev = reinterpret_cast<int64_t*>(scratch + grad_work_doubles(N, ncols) - even64((int64_t)re.size()));
    TGP_CUDA(cudaMemcpyAsync(re_dev, re.data(), re.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  }
  if (nrhs == 1) {
    grad_contract_kernel<P><<<dim3((unsigned)ntiles, (unsigned)nterms), GT_THREADS, 0, st>>>(
        X, N, prof, work, ld, alpha, re_dev, scratch, tgp_phi_device());
  } else {
    grad_contract_kernel<MultiOut<P, TGP_MAX_RHS>><<<dim3((unsigned)ntiles, (unsigned)nterms), GT_THREADS, 0, st>>>(
        X, N, MultiOut<P, TGP_MAX_RHS>{prof, nrhs}, work, ld, alpha, re_dev, scratch, tgp_phi_device());
  }
  TGP_LAUNCH_CHECK();
  switch (ncols) {
    case 4: grad_finish_kernel<4><<<1, 1024, 0, st>>>(scratch, ntiles, info, out); break;
    case 5: grad_finish_kernel<5><<<1, 1024, 0, st>>>(scratch, ntiles, info, out); break;
    case 9: grad_finish_kernel<9><<<1, 1024, 0, st>>>(scratch, ntiles, info, out); break;
    case 13: grad_finish_kernel<13><<<1, 1024, 0, st>>>(scratch, ntiles, info, out); break;
    default: grad_finish_kernel<4 * TGP_MAX_TERMS + 1><<<1, 1024, 0, st>>>(scratch, ntiles, info, out); break;
  }
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

extern "C" int tgp_loglike_grad(const double* X, const double* y, const double* yerr2, int64_t N, const tgp_kernel* k,
                                double* work, int64_t ld, double* alpha, double* out, int32_t* info,
                                const int64_t* row_end, int64_t nblocks, double* scratch, void* stream) {
  TGP_CHECK_ARG(kdesc_ok(k), "kernel descriptor");
  int rc = grad_args(X, y, N, work, ld, alpha, out, info, row_end, nblocks, scratch);
  if (rc) return rc;
  rc = row_end ? tgp_loglike_env(X, y, yerr2, N, k, work, ld, alpha, 1, out, info, row_end, nblocks, stream)
               : tgp_loglike(X, y, yerr2, N, k, work, ld, alpha, 1, out, info, stream);
  if (rc) return rc;
  const KDesc kd = make_kdesc(k);
  TGP_FAMILY_SWITCH(k->family, return grad_tail(X, N, FamilyProfile<FAM>{kd}, 1, 4, work, ld, alpha, out, info,
                                                row_end, scratch, (cudaStream_t)stream));
  return TGP_OK;
}

// After the likelihood call of a sum: a one-term sum without white runs the single-term contraction (bit for bit the
// single-term entry's gradient, d / d ln white = 0), any other sum its 4 nterms + 1 partial columns.
static int grad_tail_sum(const double* X, int64_t N, const tgp_kernel_sum* k, double* work, int64_t ld,
                         const double* alpha, double* out, const int32_t* info, const int64_t* row_end,
                         double* scratch, cudaStream_t st, int nrhs) {
  if (k->nterms == 1 && k->white == 0.0) {
    TGP_CUDA(cudaMemsetAsync(out + 7, 0, sizeof(double), st));
    const KDesc kd = make_kdesc(&k->term[0]);
    TGP_FAMILY_SWITCH(k->term[0].family, return grad_tail(X, N, FamilyProfile<FAM>{kd}, 1, 4, work, ld, alpha, out,
                                                          info, row_end, scratch, st, nrhs));
    return TGP_OK;
  }
  return grad_tail(X, N, SumProfile{make_ksumdesc(k)}, k->nterms, 4 * k->nterms + 1, work, ld, alpha, out, info,
                   row_end, scratch, st, nrhs);
}

extern "C" int tgp_loglike_grad_sum(const double* X, const double* y, const double* yerr2, int64_t N,
                                    const tgp_kernel_sum* k, double* work, int64_t ld, double* alpha, double* out,
                                    int32_t* info, const int64_t* row_end, int64_t nblocks, double* scratch,
                                    void* stream) {
  TGP_CHECK_ARG(ksum_ok(k), "kernel sum descriptor");
  int rc = grad_args(X, y, N, work, ld, alpha, out, info, row_end, nblocks, scratch);
  if (rc) return rc;
  rc = tgp_loglike_sum(X, y, yerr2, N, k, work, ld, alpha, 1, out, info, row_end, nblocks, stream);
  if (rc) return rc;
  return grad_tail_sum(X, N, k, work, ld, alpha, out, info, row_end, scratch, (cudaStream_t)stream, 1);
}

extern "C" int tgp_loglike_grad_multi(const double* X, const double* Y, int32_t r, const double* yerr2, int64_t N,
                                      const tgp_kernel_sum* k, double* work, int64_t ld, double* alpha, double* out,
                                      int32_t* info, const int64_t* row_end, int64_t nblocks, double* scratch,
                                      void* stream) {
  TGP_CHECK_ARG(r >= 1 && r <= TGP_MAX_RHS, "number of outputs must be 1 .. TGP_MAX_RHS");
  TGP_CHECK_ARG(ksum_ok(k), "kernel sum descriptor");
  int rc = grad_args(X, Y, N, work, ld, alpha, out, info, row_end, nblocks, scratch);
  if (rc) return rc;
  if (r == 1)   // (N, 1) is an N-vector: the single-output entry, bit for bit
    return tgp_loglike_grad_sum(X, Y, yerr2, N, k, work, ld, alpha, out, info, row_end, nblocks, scratch, stream);
  rc = tgp_loglike_multi(X, Y, r, yerr2, N, k, work, ld, alpha, 1, out, info, row_end, nblocks, stream);
  if (rc) return rc;
  return grad_tail_sum(X, N, k, work, ld, alpha, out, info, row_end, scratch, (cudaStream_t)stream, r);
}

// ---- batches of independent problems (tgp_loglike_grad_batch) ---------------------------------------------------
// The selected inverse, contraction and finish above on every problem of a batch: each launch of selinv_run's
// schedule runs its body on a grid of (problem, CTA), step s handling block column nb_b - 1 - s of problem b
// (batch.cuh), so that every problem starts at step 0; CTAs of problems without that launch exit.  The fills and
// mirrors only move values, and the products and the halving solve are the single call's tile bodies (dense.cu), so Z
// is tgp_selinv's bit for bit.

// 0: -W^T = -I, 1: W^T = -(-W^T), 2: T^T = 0, 3: Z[R, J] = 0, 4: Z[J, J] = 0 (the memsets of selinv_run)
enum { SEL_NEG_I = 0, SEL_NEGATE = 1, SEL_ZERO_TT = 2, SEL_ZERO_ZRJ = 3, SEL_ZERO_ZJJ = 4 };
__global__ void __launch_bounds__(256)
selinv_fill_batch_kernel(const TgpBatchProb* __restrict__ pr, double* const* __restrict__ scr, int s, int op) {
  const int b = blockIdx.x;
  TgpSelStep g;
  if (!tgp_selinv_step(pr[b].N, s, g)) return;
  const int64_t ld = pr[b].ld, ldt = (pr[b].N + 1) & ~(int64_t)1;
  double* NWT = scr[b];
  double* dst = NWT;
  int64_t rows = g.w, cols = g.w, pitch = TGP_OB;
  switch (op) {
    case SEL_NEGATE: dst = NWT + TGP_OB * TGP_OB; break;
    case SEL_ZERO_TT: dst = NWT + 2 * TGP_OB * TGP_OB; cols = g.m; pitch = ldt; break;
    case SEL_ZERO_ZRJ: dst = pr[b].A + g.c1 * ld + g.k; rows = g.m; pitch = ld; break;
    case SEL_ZERO_ZJJ: dst = pr[b].A + g.k * ld + g.k; pitch = ld; break;
    default: break;
  }
  for (int64_t idx = blockIdx.y * (int64_t)blockDim.x + threadIdx.x; idx < rows * cols;
       idx += (int64_t)gridDim.y * blockDim.x) {
    const int64_t r = idx / cols, c = idx % cols;
    double v = 0.0;
    if (op == SEL_NEG_I) v = (r == c) ? -1.0 : 0.0;
    else if (op == SEL_NEGATE) v = -NWT[r * TGP_OB + c];
    dst[r * pitch + c] = v;
  }
}

// 0: Z[J, R] = Z[R, J]^T, 1: the upper triangle of Z[J, J].  grid: (problem, row tile * tiles_c + column tile)
__global__ void __launch_bounds__(256)
selinv_mirror_batch_kernel(const TgpBatchProb* __restrict__ pr, int s, int op, int tiles_c) {
  const int b = blockIdx.x;
  TgpSelStep g;
  if (!tgp_selinv_step(pr[b].N, s, g)) return;
  const int64_t ld = pr[b].ld, rows = op == 0 ? g.m : g.w;
  const int64_t r0 = (int64_t)(blockIdx.y / tiles_c) * 32, c0 = (int64_t)(blockIdx.y % tiles_c) * 32;
  if (r0 >= rows || c0 >= g.w) return;
  double* A = pr[b].A;
  if (op == 0) mirror_body(A + g.c1 * ld + g.k, A + g.k * ld + g.c1, rows, g.w, ld, 0, r0, c0);
  else mirror_body(A + g.k * ld + g.k, A + g.k * ld + g.k, rows, g.w, ld, 1, r0, c0);
}

int tgp_batch_selinv(const TgpBatchProb* pr, double* const* scr, const TgpBatchProb* prob_h, double* const* scr_h,
                     int32_t B, cudaStream_t st) {
  std::vector<int64_t> Nh(B);
  int smax = 0;
  for (int32_t b = 0; b < B; ++b) {
    Nh[b] = prob_h[b].N;
    smax = std::max(smax, (int)tgp_cdiv(Nh[b], TGP_OB));
  }
  std::vector<TgpLeafArgs> full, edge;
  auto fill = [&](int s, int op, int64_t elems) -> int {
    if (elems <= 0) return TGP_OK;
    const unsigned ctas = (unsigned)std::min<int64_t>(tgp_cdiv(elems, 256), 64);
    selinv_fill_batch_kernel<<<dim3((unsigned)B, ctas), 256, 0, st>>>(pr, scr, s, op);
    TGP_LAUNCH_CHECK();
    return TGP_OK;
  };
  // the largest launch of product `op` over the problems of step s
  auto gemm = [&](int s, int op, int leaf) -> int {
    int64_t tm = 0, tn = 0;
    for (int32_t b = 0; b < B; ++b) {
      TgpSelStep g;
      int64_t M, Nc, Kd;
      if (!tgp_selinv_step(Nh[b], s, g) || !tgp_selinv_gemm_shape(g, op, leaf, M, Nc, Kd)) continue;
      tm = std::max(tm, tgp_cdiv(M, 128));
      tn = std::max(tn, tgp_cdiv(Nc, 64));
    }
    if (tm == 0) return TGP_OK;
    return tgp_batch_selinv_gemm(pr, scr, B, s, op, leaf, (int)tn, tm * tn, st);
  };
  auto mirror = [&](int s, int op, int64_t rows, int64_t cols) -> int {
    if (rows <= 0 || cols <= 0) return TGP_OK;
    const int64_t tc = tgp_cdiv(cols, 32), tiles = tgp_cdiv(rows, 32) * tc;
    TGP_CHECK_ARG(tiles <= 65535, "too many tiles for one launch");
    selinv_mirror_batch_kernel<<<dim3((unsigned)B, (unsigned)tiles), dim3(32, 8), 0, st>>>(pr, s, op, (int)tc);
    TGP_LAUNCH_CHECK();
    return TGP_OK;
  };
  int rc;
  for (int s = 0; s < smax; ++s) {
    int64_t wmax = 0, mmax = 0;
    for (int32_t b = 0; b < B; ++b) {
      TgpSelStep g;
      if (!tgp_selinv_step(Nh[b], s, g)) continue;
      wmax = std::max(wmax, g.w);
      mmax = std::max(mmax, g.m);
    }
    if ((rc = fill(s, SEL_NEG_I, wmax * wmax))) return rc;
    // -W^T: rows of -I times L11^-T by halving, leaf, gemm, leaf, ..., leaf for every problem
    const int nleaves = (int)tgp_cdiv(wmax, 64);
    for (int i = 0; i < nleaves; ++i) {
      full.clear();
      edge.clear();
      for (int32_t b = 0; b < B; ++b) {   // leaf i of problem b, on the path trsm_panel_launch takes for it
        TgpSelStep g;
        const int64_t c0 = 64 * (int64_t)i;
        if (!tgp_selinv_step(Nh[b], s, g) || g.w <= c0) continue;
        const int64_t ld = prob_h[b].ld;
        const int nb = (int)std::min<int64_t>(g.w - c0, 64);
        (nb == 64 ? full : edge).push_back(
            TgpLeafArgs{prob_h[b].A + (g.k + c0) * ld + g.k + c0, scr_h[b] + c0, ld, g.w, TGP_OB, nb});
      }
      if ((rc = tgp_batch_selinv_leaves(full.data(), (int32_t)full.size(), true, st))) return rc;
      if ((rc = tgp_batch_selinv_leaves(edge.data(), (int32_t)edge.size(), false, st))) return rc;
      if (i + 1 < nleaves && (rc = gemm(s, TGP_SEL_HALVE, i))) return rc;
    }
    if ((rc = fill(s, SEL_NEGATE, wmax * wmax))) return rc;
    if (mmax > 0) {
      if ((rc = fill(s, SEL_ZERO_TT, wmax * mmax))) return rc;
      if ((rc = gemm(s, TGP_SEL_TT, 0))) return rc;
      if ((rc = fill(s, SEL_ZERO_ZRJ, wmax * mmax))) return rc;
      if ((rc = gemm(s, TGP_SEL_ZRJ, 0))) return rc;
      if ((rc = mirror(s, 0, mmax, wmax))) return rc;
    }
    if ((rc = fill(s, SEL_ZERO_ZJJ, wmax * wmax))) return rc;
    if ((rc = gemm(s, TGP_SEL_WTW, 0))) return rc;
    if (mmax > 0 && (rc = gemm(s, TGP_SEL_TZ, 0))) return rc;
    if ((rc = mirror(s, 1, wmax, wmax))) return rc;
  }
  return TGP_OK;
}

// grid: (tile, term, problem of the list); the single call's contraction on each problem, Z in its workspace block and
// the tile partials at the front of its scratch.  The problem's profile is staged in shared memory: the body indexes a
// sum's terms by blockIdx.y, which a copy in registers could only do from the stack.  P = MultiOut<...>: the problem's
// r outputs (alpha N x r), as tgp_loglike_grad_multi contracts them.
template <class P>
__global__ void __launch_bounds__(GT_THREADS)
grad_contract_batch_kernel(const TgpBatchProb* __restrict__ pr, const KSumDesc* __restrict__ descs,
                           const int32_t* __restrict__ list, double* const* __restrict__ scr,
                           const double* __restrict__ phi_g) {
  const int b = list[blockIdx.z];
  const int64_t N = pr[b].N, nt = (N + GT - 1) / GT;
  if ((int64_t)blockIdx.x >= nt * (nt + 1) / 2) return;
  if (P::kSum && (int)blockIdx.y >= descs[b].nterms) return;
  __shared__ P prof_s;   // P holds one descriptor (the sum's, or a family's single term), and for r outputs nrhs
  static_assert((sizeof(prof_s.desc) == sizeof(P) || OutputsOf<P>::kR > 1) && sizeof(prof_s.desc) % 4 == 0,
                "a profile is its descriptor");
  {
    const int* src = reinterpret_cast<const int*>(P::kSum ? (const void*)&descs[b] : (const void*)&descs[b].term[0]);
    int* dst = reinterpret_cast<int*>(&prof_s.desc);
    for (int i = threadIdx.x; i < (int)(sizeof(prof_s.desc) / 4); i += GT_THREADS) dst[i] = src[i];
    if constexpr (OutputsOf<P>::kR > 1) {
      if (threadIdx.x == 0) prof_s.nrhs = (int)pr[b].r;
    }
  }
  __syncthreads();
  const P& prof = prof_s;
  const double* __restrict__ X = pr[b].X;
  const double* __restrict__ Z = pr[b].A;
  const double* __restrict__ alpha = pr[b].alpha;
  const int64_t ld = pr[b].ld;
  const int64_t* __restrict__ re_dev = nullptr;
  double* __restrict__ partials = scr[b];
#include "grad_contract_body.cuh"
}

template <class Q>
static void grad_contract_batch_launch(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list,
                                       double* const* scr, int r, dim3 grid, cudaStream_t st) {
  const double* phi = tgp_phi_device();
  if (r == 1) grad_contract_batch_kernel<Q><<<grid, GT_THREADS, 0, st>>>(pr, kd, list, scr, phi);
  else grad_contract_batch_kernel<MultiOut<Q, TGP_MAX_RHS>><<<grid, GT_THREADS, 0, st>>>(pr, kd, list, scr, phi);
}

int tgp_batch_grad_contract(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list, int32_t count, int cls,
                            double* const* scr, int64_t max_n, int max_terms, int r, cudaStream_t st) {
  const int64_t ntiles = grad_tiles(max_n);
  TGP_CHECK_ARG(ntiles < (1ll << 31), "matrix too large for one launch");
  for (int32_t z0 = 0; z0 < count; z0 += 65535) {   // gridDim.z <= 65535
    const dim3 grid((unsigned)ntiles, (unsigned)max_terms, (unsigned)std::min(count - z0, 65535));
    if (cls == TGP_BATCH_SUM) {
      grad_contract_batch_launch<SumProfile>(pr, kd, list + z0, scr, r, grid, st);
    } else {
      TGP_FAMILY_SWITCH(cls, (grad_contract_batch_launch<FamilyProfile<FAM>>(pr, kd, list + z0, scr, r, grid, st)));
    }
    TGP_LAUNCH_CHECK();
  }
  return TGP_OK;
}

// One CTA per problem: grad_finish_kernel with the single call's NC, then the rest of the problem's output slice.
__global__ void __launch_bounds__(1024)
grad_finish_batch_kernel(const TgpBatchProb* __restrict__ pr, const KSumDesc* __restrict__ kd,
                         double* const* __restrict__ scr, const int32_t* __restrict__ info,
                         const double* __restrict__ ll, double* __restrict__ out) {
  const int b = blockIdx.x;
  const int nterms = kd[b].nterms;
  const int nc = (nterms == 1 && kd[b].white == 0.0) ? 4 : 4 * nterms + 1;   // one term: d / d ln white = 0
  const int64_t nt = (pr[b].N + GT - 1) / GT, ntiles = nt * (nt + 1) / 2;
  double* o = out + (int64_t)b * TGP_GRAD_BATCH_OUT;
  const int tid = threadIdx.x;
  if (tid < 3) o[tid] = ll[3 * (int64_t)b + tid];
  else if (tid >= 3 + nc && tid < TGP_GRAD_BATCH_OUT) o[tid] = 0.0;
  switch (nc) {
    case 4: grad_finish_body<4>(scr[b], ntiles, info + b, o); break;
    case 5: grad_finish_body<5>(scr[b], ntiles, info + b, o); break;
    case 9: grad_finish_body<9>(scr[b], ntiles, info + b, o); break;
    case 13: grad_finish_body<13>(scr[b], ntiles, info + b, o); break;
    default: grad_finish_body<4 * TGP_MAX_TERMS + 1>(scr[b], ntiles, info + b, o); break;
  }
}

int tgp_batch_grad_finish(const TgpBatchProb* pr, const KSumDesc* kd, double* const* scr, int32_t B,
                          const int32_t* info, const double* ll, double* out, cudaStream_t st) {
  grad_finish_batch_kernel<<<(unsigned)B, 1024, 0, st>>>(pr, kd, scr, info, ll, out);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}
