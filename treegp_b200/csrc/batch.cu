// Batches of independent small problems: B likelihood evaluations (tgp_loglike_batch), B likelihoods with their
// gradients (tgp_loglike_grad_batch), B posterior means (tgp_predict_mean_batch), B diagonal predictive variances
// (tgp_predict_var_batch) or B sets of leave-one-out predictions (tgp_loo_batch) per call.  The _multi entries take r
// outputs per problem sharing its kernel, as tgp_loglike_multi does for one problem: they ride through the
// factorisation as r extra rows, and every later step reads them as an N x r row-major block.
//
// A problem of a few hundred to a few thousand points leaves the B200 idle: its factorisation is a chain of small
// launches (8 panel launches and one update per 512 columns, at most ~70 CTAs each), so its time is launch latency.
// Here every launch of that chain carries all B problems: the schedule runs over the panel steps of the largest
// problem, each CTA picks its problem from blockIdx.x and runs the body of the single-problem kernel on that
// problem's slice (kmat.cu, dense.cu, predict.cu), and CTAs of problems without work at that step exit.  So a
// problem's K, factor, logL and info are what tgp_loglike_sum (dense) gives on it alone, bit for bit, whatever else
// shares the batch.  The only new arithmetic is the backward sweep of want_alpha (one CTA per problem and group of
// outputs, below).  The gradient adds the selected inverse, contraction and finish of tgp_loglike_grad_sum in the
// same form (selinv.cu).
#include <string.h>
#include <algorithm>
#include <vector>
#include "tgp_common.cuh"
#include "profile_policy.cuh"
#include "batch.cuh"

#define BATCH_CHECK(cond, msg)                                        \
  do {                                                                \
    if (!(cond)) {                                                    \
      tgp_set_error("%s: invalid argument: %s", fn, msg);             \
      return TGP_ERR_INVALID;                                         \
    }                                                                 \
  } while (0)

static int64_t even_ld(int64_t n) { return (n + 1) & ~(int64_t)1; }

// off: B + 1 offsets from 0, strictly increasing (min_n = 1) or non-decreasing (min_n = 0), steps <= max_n
static int check_offsets(const char* fn, const char* name, const int64_t* off, int32_t B, int64_t min_n,
                         int64_t max_n) {
  char msg[160];
  snprintf(msg, sizeof msg, "%s must be a host array of B + 1 offsets", name);
  BATCH_CHECK(off != nullptr, msg);
  snprintf(msg, sizeof msg, "%s[0] must be 0", name);
  BATCH_CHECK(off[0] == 0, msg);
  for (int32_t b = 0; b < B; ++b) {
    const int64_t n = off[b + 1] - off[b];
    snprintf(msg, sizeof msg, "%s must be %s (problem %d has %lld points)", name,
             min_n > 0 ? "strictly increasing" : "non-decreasing", (int)b, (long long)n);
    BATCH_CHECK(n >= min_n, msg);
    snprintf(msg, sizeof msg, "N_b = %lld of problem %d exceeds TGP_BATCH_MAX_N = %d", (long long)n, (int)b,
             TGP_BATCH_MAX_N);
    BATCH_CHECK(n <= max_n, msg);
  }
  return TGP_OK;
}

static int check_batch(const char* fn, const int64_t* off, int32_t B, const tgp_kernel_sum* ks) {
  BATCH_CHECK(B >= 1, "B must be >= 1");
  const int rc = check_offsets(fn, "off", off, B, 1, TGP_BATCH_MAX_N);
  if (rc) return rc;
  BATCH_CHECK(ks != nullptr, "ks must be a host array of B kernel sum descriptors");
  for (int32_t b = 0; b < B; ++b) {
    BATCH_CHECK(ksum_ok(&ks[b]), "ks: kernel sum descriptor");
    BATCH_CHECK(ks[b].ndim == ks[0].ndim, "ks: every problem must have the same ndim");
  }
  return TGP_OK;
}

static int check_outputs(const char* fn, int32_t r) {
  BATCH_CHECK(r >= 1 && r <= TGP_MAX_RHS, "number of outputs r must be 1 .. TGP_MAX_RHS");
  return TGP_OK;
}

static int64_t work_doubles(const char* fn, const int64_t* off, int32_t B, int32_t r) {
  if (check_outputs(fn, r)) return TGP_ERR_INVALID;
  if (B < 1) {
    tgp_set_error("%s: invalid argument: B must be >= 1", fn);
    return TGP_ERR_INVALID;
  }
  if (check_offsets(fn, "off", off, B, 1, TGP_BATCH_MAX_N)) return TGP_ERR_INVALID;
  int64_t total = 0;
  for (int32_t b = 0; b < B; ++b) {
    const int64_t n = off[b + 1] - off[b];
    total += (n + r) * even_ld(n);
  }
  return total;
}

extern "C" int64_t tgp_batch_work_doubles(const int64_t* off, int32_t B) { return work_doubles(__func__, off, B, 1); }

extern "C" int64_t tgp_batch_multi_work_doubles(const int64_t* off, int32_t B, int32_t r) {
  return work_doubles(__func__, off, B, r);
}

// The per-call device tables: problem descriptors, kernel descriptors, the problem lists of every profile class,
// (for the factorisation) one flag word per problem and the caller's `extra` bytes, in one stream-ordered allocation
// freed on the same stream.
struct BatchTables {
  void* dev = nullptr;
  cudaStream_t st = nullptr;
  TgpBatchProb* pr = nullptr;
  KSumDesc* kd = nullptr;
  int32_t* list = nullptr;
  unsigned* flags = nullptr;
  unsigned char* extra = nullptr;
  int32_t start[TGP_BATCH_NCLASS + 1] = {};   // class c owns list[start[c] .. start[c + 1])
  int64_t max_n[TGP_BATCH_NCLASS] = {}, max_m[TGP_BATCH_NCLASS] = {};
  ~BatchTables() {
    if (dev) cudaFreeAsync(dev, st);
  }
};

static size_t align16(size_t n) { return (n + 15) & ~(size_t)15; }

static int stage_tables(BatchTables& T, const std::vector<TgpBatchProb>& prob, const tgp_kernel_sum* ks,
                        const std::vector<int>& cls, cudaStream_t st,
                        const std::vector<unsigned char>& extra = std::vector<unsigned char>()) {
  const size_t B = prob.size();
  const size_t o_kd = align16(B * sizeof(TgpBatchProb));
  const size_t o_list = o_kd + align16(B * sizeof(KSumDesc));
  const size_t o_flags = o_list + align16(B * sizeof(int32_t));
  const size_t o_extra = o_flags + align16(B * sizeof(unsigned));
  const size_t bytes = o_extra + align16(extra.size());
  std::vector<unsigned char> h(bytes, 0);
  memcpy(h.data(), prob.data(), B * sizeof(TgpBatchProb));
  if (!extra.empty()) memcpy(h.data() + o_extra, extra.data(), extra.size());
  KSumDesc* kd = reinterpret_cast<KSumDesc*>(h.data() + o_kd);
  int32_t* list = reinterpret_cast<int32_t*>(h.data() + o_list);
  for (size_t b = 0; b < B; ++b) kd[b] = make_ksumdesc(&ks[b]);
  int32_t n = 0;
  for (int c = 0; c < TGP_BATCH_NCLASS; ++c) {
    T.start[c] = n;
    for (size_t b = 0; b < B; ++b) {
      if (cls[b] != c) continue;
      list[n++] = (int32_t)b;
      T.max_n[c] = prob[b].N > T.max_n[c] ? prob[b].N : T.max_n[c];
      T.max_m[c] = prob[b].M > T.max_m[c] ? prob[b].M : T.max_m[c];
    }
  }
  T.start[TGP_BATCH_NCLASS] = n;
  T.st = st;
  TGP_CUDA(cudaMallocAsync(&T.dev, bytes, st));
  TGP_CUDA(cudaMemcpyAsync(T.dev, h.data(), bytes, cudaMemcpyHostToDevice, st));   // pageable: staged before return
  unsigned char* d = static_cast<unsigned char*>(T.dev);
  T.pr = reinterpret_cast<TgpBatchProb*>(d);
  T.kd = reinterpret_cast<KSumDesc*>(d + o_kd);
  T.list = reinterpret_cast<int32_t*>(d + o_list);
  T.flags = reinterpret_cast<unsigned*>(d + o_flags);
  T.extra = d + o_extra;
  return TGP_OK;
}

// Y (N x r, row-major) into rows N .. N + r - 1 of every block (to_alpha == 0), or those rows (= L^-1 y after the
// factorisation) into alpha (N x r), as multi_transpose_kernel moves them for one problem.
__global__ void __launch_bounds__(256)
batch_yrow_kernel(const TgpBatchProb* __restrict__ pr, int to_alpha) {
  const TgpBatchProb& p = pr[blockIdx.x];
  double* rows = p.A + p.N * p.ld;
  const int64_t r = p.r;
  for (int64_t i = threadIdx.x; i < p.N; i += blockDim.x) {
    for (int64_t c = 0; c < r; ++c) {
      if (to_alpha) p.alpha[i * r + c] = rows[c * p.ld + i];
      else rows[c * p.ld + i] = p.y[i * r + c];
    }
  }
}

// Backward sweep alpha <- L^-T alpha for G outputs of a problem per CTA (the persistent cooperative sweeps of trsv.cu
// take one problem per launch); grid (problem, group of G outputs).  Blocks of 64 unknowns from the last: the four row
// groups of the CTA form sum_{i >= j1} L[i, j0 + c] x_qi for the block's 64 columns and all G outputs q (each L entry
// is read once per CTA, rows coalesced), then warp q solves the 64 x 64 diagonal block for output q by substitution
// with shuffles.  Each output's arithmetic, and its order, is that of one output alone.  x lives in shared memory,
// G columns of xp >= N doubles: G = 4 and N = 4096 take 128 KB.  The last group of r = 3, 5, 6, 7 has nq < G outputs;
// its unused columns are zeroed, so that the shared sweep loop reads no uninitialised memory, and never written back.
constexpr int BS_THREADS = 256;
constexpr int BS_NB = 64;
static size_t bs_smem(int G, int64_t xp) { return (size_t)(G * xp + BS_NB * (BS_NB + 1) + 4 * G * BS_NB) * 8; }

template <int G>
__global__ void __launch_bounds__(BS_THREADS, 2)
backward_batch_kernel(const TgpBatchProb* __restrict__ pr, int64_t xp) {
  extern __shared__ double bsm[];
  double* x = bsm;                                 // G x xp unknowns
  double* Ld = bsm + G * xp;                       // diagonal block, pitch BS_NB + 1
  double* part = Ld + BS_NB * (BS_NB + 1);         // G x 4 partial sums per column
  const TgpBatchProb& p = pr[blockIdx.x];
  const int N = (int)p.N, r = (int)p.r;            // N <= TGP_BATCH_MAX_N: int indices
  const int64_t ld = p.ld;
  const int q0 = (int)blockIdx.y * G;              // first output of this CTA
  const int nq = r - q0 < G ? r - q0 : G;          // outputs of this CTA
  const double* L = p.A;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = tid & (BS_NB - 1), g = tid / BS_NB;
  for (int q = 0; q < G; ++q) {   // the columns of outputs beyond r (last group) are zeros, swept and never written
    for (int i = tid; i < N; i += BS_THREADS) x[q * xp + i] = q < nq ? p.alpha[(int64_t)i * r + q0 + q] : 0.0;
  }
  __syncthreads();
  for (int j0 = (N - 1) / BS_NB * BS_NB; j0 >= 0; j0 -= BS_NB) {
    const int nb = N - j0 < BS_NB ? N - j0 : BS_NB;
    const int j1 = j0 + nb;
    double s[G];
#pragma unroll
    for (int q = 0; q < G; ++q) s[q] = 0.0;
    if (c < nb) {
#pragma unroll 4
      for (int i = j1 + g; i < N; i += 4) {
        const double l = L[i * ld + j0 + c];
#pragma unroll
        for (int q = 0; q < G; ++q) s[q] = fma(l, x[q * xp + i], s[q]);
      }
    }
#pragma unroll
    for (int q = 0; q < G; ++q) part[(4 * q + g) * BS_NB + c] = s[q];
    for (int idx = tid; idx < BS_NB * BS_NB; idx += BS_THREADS) {
      const int rr = idx / BS_NB, cc = idx % BS_NB;
      Ld[rr * (BS_NB + 1) + cc] = (rr < nb && cc <= rr) ? L[(j0 + rr) * ld + j0 + cc] : 0.0;
    }
    __syncthreads();
    if (warp < nq) {
      // lane owns unknowns j0 + lane (r0) and j0 + 32 + lane (r1) of output `warp`
      double* xq = x + warp * xp;
      const double* pq = part + 4 * warp * BS_NB;
      double r0 = 0.0, r1 = 0.0;
      if (lane < nb)
        r0 = xq[j0 + lane] - (((pq[lane] + pq[BS_NB + lane]) + pq[2 * BS_NB + lane]) + pq[3 * BS_NB + lane]);
      if (lane + 32 < nb) {
        const int l = lane + 32;
        r1 = xq[j0 + l] - (((pq[l] + pq[BS_NB + l]) + pq[2 * BS_NB + l]) + pq[3 * BS_NB + l]);
      }
      for (int i = nb - 1; i >= 0; --i) {
        const double xi = __shfl_sync(0xffffffffu, i < 32 ? r0 : r1, i & 31) / Ld[i * (BS_NB + 1) + i];
        if (lane == (i & 31)) {
          if (i < 32) r0 = xi;
          else r1 = xi;
        }
        if (lane < i) r0 = fma(-Ld[i * (BS_NB + 1) + lane], xi, r0);
        if (lane + 32 < i) r1 = fma(-Ld[i * (BS_NB + 1) + lane + 32], xi, r1);
      }
      if (lane < nb) xq[j0 + lane] = r0;
      if (lane + 32 < nb) xq[j0 + lane + 32] = r1;
    }
    __syncthreads();
  }
  for (int q = 0; q < nq; ++q) {
    for (int i = tid; i < N; i += BS_THREADS) p.alpha[(int64_t)i * r + q0 + q] = x[q * xp + i];
  }
}

// Outputs per CTA of the backward sweep: one CTA reads the factor for up to 4 outputs (x of 4 outputs at N = 4096
// fills 128 KB of shared memory; 8 would not fit).
static int backward_group(int64_t r) { return r == 1 ? 1 : (r == 2 ? 2 : 4); }

template <int G>
static int backward_batch_launch(const TgpBatchProb* pr, int32_t B, int64_t r, int64_t max_n, cudaStream_t st) {
  static TgpPerDeviceOnce attr_once;
  if (tgp_first_use_on_device(attr_once))
    TGP_CUDA(cudaFuncSetAttribute(backward_batch_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)bs_smem(G, TGP_BATCH_MAX_N)));
  const int64_t xp = even_ld(max_n);
  backward_batch_kernel<G><<<dim3((unsigned)B, (unsigned)tgp_cdiv(r, (int64_t)G)), BS_THREADS, bs_smem(G, xp), st>>>(
      pr, xp);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

// The chain of tgp_loglike_batch (r outputs per problem) on checked arguments, with the tables staged into T (plus
// `extra` bytes) and their host copy in prob.  out: 3 B doubles, or nullptr for T.extra's first 3 B doubles.
static int loglike_batch_run(const double* X, const double* y, int32_t r, const double* yerr2, const int64_t* off,
                             int32_t B, const tgp_kernel_sum* ks, double* work, double* alpha, int want_alpha,
                             double* out, int32_t* info, cudaStream_t st, BatchTables& T,
                             std::vector<TgpBatchProb>& prob, const std::vector<unsigned char>& extra) {
  int rc;
  const int ndim = ks[0].ndim;
  prob.assign(B, TgpBatchProb{});
  std::vector<int> cls(B);
  std::vector<int64_t> Nh(B);
  int64_t woff = 0, max_n = 0;
  for (int32_t b = 0; b < B; ++b) {
    const int64_t r0 = off[b], n = off[b + 1] - off[b];
    TgpBatchProb& p = prob[b];
    p = TgpBatchProb{};
    p.X = X + r0 * ndim;
    p.y = y + r0 * r;
    p.yerr2 = yerr2 + r0;
    p.A = work + woff;
    p.alpha = alpha + r0 * r;
    p.N = Nh[b] = n;
    p.ld = even_ld(n);
    p.r = r;
    woff += (n + r) * p.ld;
    max_n = std::max(max_n, n);
    // the K build of tgp_kmat_sym_sum: the single-term kernel for one term without a white level
    cls[b] = (ks[b].nterms == 1 && ks[b].white == 0.0) ? ks[b].term[0].family : TGP_BATCH_SUM;
  }
  rc = stage_tables(T, prob, ks, cls, st, extra);
  if (rc) return rc;
  if (!out) out = reinterpret_cast<double*>(T.extra);
  for (int c = 0; c < TGP_BATCH_NCLASS; ++c) {
    if (T.start[c + 1] == T.start[c]) continue;
    rc = tgp_batch_kmat_sym(T.pr, T.kd, T.list + T.start[c], T.start[c + 1] - T.start[c], c, T.max_n[c], st);
    if (rc) return rc;
  }
  batch_yrow_kernel<<<(unsigned)B, 256, 0, st>>>(T.pr, 0);
  TGP_LAUNCH_CHECK();
  rc = tgp_batch_potrf_rows(T.pr, Nh.data(), B, r, info, T.flags, st);
  if (rc) return rc;
  batch_yrow_kernel<<<(unsigned)B, 256, 0, st>>>(T.pr, 1);
  TGP_LAUNCH_CHECK();
  if (want_alpha) {
    switch (backward_group(r)) {
      case 1: rc = backward_batch_launch<1>(T.pr, B, r, max_n, st); break;
      case 2: rc = backward_batch_launch<2>(T.pr, B, r, max_n, st); break;
      default: rc = backward_batch_launch<4>(T.pr, B, r, max_n, st); break;
    }
    if (rc) return rc;
  }
  return tgp_batch_loglike_finish(T.pr, B, r, want_alpha, info, out, st);
}

static int loglike_batch_entry(const char* fn, const double* X, const double* y, int32_t r, const double* yerr2,
                               const int64_t* off, int32_t B, const tgp_kernel_sum* ks, double* work, double* alpha,
                               int want_alpha, double* out, int32_t* info, void* stream) {
  int rc = check_outputs(fn, r);
  if (rc) return rc;
  rc = check_batch(fn, off, B, ks);
  if (rc) return rc;
  BATCH_CHECK(X && y && yerr2 && work && alpha && out && info, "null pointer (X, y, yerr2, work, alpha, out, info)");
  BATCH_CHECK(((uintptr_t)work & 15) == 0, "work must be 16-byte aligned");
  BatchTables T;
  std::vector<TgpBatchProb> prob;
  return loglike_batch_run(X, y, r, yerr2, off, B, ks, work, alpha, want_alpha, out, info, (cudaStream_t)stream, T,
                           prob, std::vector<unsigned char>());
}

extern "C" int tgp_loglike_batch(const double* X, const double* y, const double* yerr2, const int64_t* off, int32_t B,
                                 const tgp_kernel_sum* ks, double* work, double* alpha, int want_alpha, double* out,
                                 int32_t* info, void* stream) {
  return loglike_batch_entry(__func__, X, y, 1, yerr2, off, B, ks, work, alpha, want_alpha, out, info, stream);
}

extern "C" int tgp_loglike_batch_multi(const double* X, const double* Y, int32_t r, const double* yerr2,
                                       const int64_t* off, int32_t B, const tgp_kernel_sum* ks, double* work,
                                       double* alpha, int want_alpha, double* out, int32_t* info, void* stream) {
  return loglike_batch_entry(__func__, X, Y, r, yerr2, off, B, ks, work, alpha, want_alpha, out, info, stream);
}

extern "C" int64_t tgp_loglike_grad_sum_work_doubles(int64_t N, int32_t nterms);

// Every problem's scratch block is even in length (the selected-inverse part, 2 TGP_OB^2 + TGP_OB even(N), exceeds
// the (4 TGP_MAX_TERMS + 1) partials of N <= TGP_BATCH_MAX_N), so all blocks stay 16-byte aligned.
extern "C" int64_t tgp_loglike_grad_batch_work_doubles(const int64_t* off, int32_t B) {
  const char* fn = __func__;
  if (B < 1) {
    tgp_set_error("%s: invalid argument: B must be >= 1", fn);
    return TGP_ERR_INVALID;
  }
  if (check_offsets(fn, "off", off, B, 1, TGP_BATCH_MAX_N)) return TGP_ERR_INVALID;
  int64_t total = 0;
  for (int32_t b = 0; b < B; ++b) total += tgp_loglike_grad_sum_work_doubles(off[b + 1] - off[b], TGP_MAX_TERMS);
  return total;
}

// The arguments of tgp_loglike_grad_batch and tgp_loo_batch (and their _multi forms), in the order and with the
// messages of the single-output entries: `nonnull` is the caller's null-pointer test, `null_msg` its message.
static int check_selinv_batch(const char* fn, int32_t r, const int64_t* off, int32_t B, const tgp_kernel_sum* ks,
                              bool nonnull, const char* null_msg, const double* work, const double* scratch) {
  int rc = check_outputs(fn, r);
  if (rc) return rc;
  rc = check_batch(fn, off, B, ks);
  if (rc) return rc;
  BATCH_CHECK(nonnull, null_msg);
  BATCH_CHECK(((uintptr_t)work & 15) == 0, "work must be 16-byte aligned");
  BATCH_CHECK(((uintptr_t)scratch & 15) == 0, "scratch must be 16-byte aligned");
  return TGP_OK;
}

// tgp_loglike_batch(want_alpha = 1) and the batched selected inverse on checked arguments.  T.extra holds
// {logL, chi2, logdet} per problem, then the scratch block of every problem (*scr on the device), then `tail`.
static int selinv_batch_run(const double* X, const double* y, int32_t r, const double* yerr2, const int64_t* off,
                            int32_t B, const tgp_kernel_sum* ks, double* work, double* alpha, int32_t* info,
                            double* scratch, cudaStream_t st, BatchTables& T, std::vector<TgpBatchProb>& prob,
                            double* const** scr, const std::vector<unsigned char>& tail = std::vector<unsigned char>()) {
  const size_t o_scr = align16((size_t)B * 3 * sizeof(double));
  const size_t o_tail = align16(o_scr + (size_t)B * sizeof(double*));
  std::vector<unsigned char> extra(o_tail + tail.size(), 0);
  if (!tail.empty()) memcpy(extra.data() + o_tail, tail.data(), tail.size());
  double** scr_h = reinterpret_cast<double**>(extra.data() + o_scr);
  int64_t soff = 0;
  for (int32_t b = 0; b < B; ++b) {
    scr_h[b] = scratch + soff;
    soff += tgp_loglike_grad_sum_work_doubles(off[b + 1] - off[b], TGP_MAX_TERMS);
  }
  int rc = loglike_batch_run(X, y, r, yerr2, off, B, ks, work, alpha, 1, nullptr, info, st, T, prob, extra);
  if (rc) return rc;
  *scr = reinterpret_cast<double* const*>(T.extra + o_scr);
  return tgp_batch_selinv(T.pr, *scr, prob.data(), scr_h, B, st);
}

static int loglike_grad_batch_entry(const char* fn, const double* X, const double* y, int32_t r, const double* yerr2,
                                    const int64_t* off, int32_t B, const tgp_kernel_sum* ks, double* work,
                                    double* alpha, double* out, int32_t* info, double* scratch, void* stream) {
  int rc = check_selinv_batch(fn, r, off, B, ks, X && y && yerr2 && work && alpha && out && info && scratch,
                              "null pointer (X, y, yerr2, work, alpha, out, info, scratch)", work, scratch);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  BatchTables T;
  std::vector<TgpBatchProb> prob;
  double* const* scr = nullptr;
  rc = selinv_batch_run(X, y, r, yerr2, off, B, ks, work, alpha, info, scratch, st, T, prob, &scr);
  if (rc) return rc;
  const double* ll = reinterpret_cast<const double*>(T.extra);
  for (int c = 0; c < TGP_BATCH_NCLASS; ++c) {
    if (T.start[c + 1] == T.start[c]) continue;
    int max_terms = 1;   // a sum's CTAs of terms beyond its own exit
    if (c == TGP_BATCH_SUM) {
      for (int32_t b = 0; b < B; ++b) max_terms = ks[b].nterms > max_terms ? ks[b].nterms : max_terms;
    }
    rc = tgp_batch_grad_contract(T.pr, T.kd, T.list + T.start[c], T.start[c + 1] - T.start[c], c, scr, T.max_n[c],
                                 max_terms, r, st);
    if (rc) return rc;
  }
  return tgp_batch_grad_finish(T.pr, T.kd, scr, B, info, ll, out, st);
}

extern "C" int tgp_loglike_grad_batch(const double* X, const double* y, const double* yerr2, const int64_t* off,
                                      int32_t B, const tgp_kernel_sum* ks, double* work, double* alpha, double* out,
                                      int32_t* info, double* scratch, void* stream) {
  return loglike_grad_batch_entry(__func__, X, y, 1, yerr2, off, B, ks, work, alpha, out, info, scratch, stream);
}

extern "C" int tgp_loglike_grad_batch_multi(const double* X, const double* Y, int32_t r, const double* yerr2,
                                            const int64_t* off, int32_t B, const tgp_kernel_sum* ks, double* work,
                                            double* alpha, double* out, int32_t* info, double* scratch,
                                            void* stream) {
  return loglike_grad_batch_entry(__func__, X, Y, r, yerr2, off, B, ks, work, alpha, out, info, scratch, stream);
}

static int predict_mean_batch_entry(const char* fn, const double* Xs, const int64_t* soff, const double* X,
                                    const int64_t* off, int32_t B, const tgp_kernel_sum* ks, const double* alpha,
                                    int32_t r, double* mean, void* stream) {
  int rc = check_outputs(fn, r);
  if (rc) return rc;
  rc = check_batch(fn, off, B, ks);
  if (rc) return rc;
  rc = check_offsets(fn, "soff", soff, B, 0, INT64_MAX);
  if (rc) return rc;
  BATCH_CHECK(Xs && X && alpha && mean, "null pointer (Xs, X, alpha, mean)");
  cudaStream_t st = (cudaStream_t)stream;
  if (soff[B] == 0) return TGP_OK;
  const int ndim = ks[0].ndim;
  std::vector<TgpBatchProb> prob(B);
  std::vector<int> cls(B);
  for (int32_t b = 0; b < B; ++b) {
    TgpBatchProb& p = prob[b];
    p = TgpBatchProb{};
    p.X = X + off[b] * ndim;
    p.alpha = const_cast<double*>(alpha) + off[b] * r;
    p.N = off[b + 1] - off[b];
    p.Xs = Xs + soff[b] * ndim;
    p.mean = mean + soff[b] * r;
    p.M = soff[b + 1] - soff[b];
    p.r = r;
    // tgp_predict_mean_sum / _multi: the single-term kernel for any one-term sum (no white term in K(Xs, X))
    cls[b] = ks[b].nterms == 1 ? ks[b].term[0].family : TGP_BATCH_SUM;
  }
  BatchTables T;
  rc = stage_tables(T, prob, ks, cls, st);
  if (rc) return rc;
  for (int c = 0; c < TGP_BATCH_NCLASS; ++c) {
    if (T.start[c + 1] == T.start[c] || T.max_m[c] == 0) continue;
    rc = tgp_batch_predict_mean(T.pr, T.kd, T.list + T.start[c], T.start[c + 1] - T.start[c], c, T.max_m[c], r, st);
    if (rc) return rc;
  }
  return TGP_OK;
}

extern "C" int tgp_predict_mean_batch(const double* Xs, const int64_t* soff, const double* X, const int64_t* off,
                                      int32_t B, const tgp_kernel_sum* ks, const double* alpha, double* mean,
                                      void* stream) {
  return predict_mean_batch_entry(__func__, Xs, soff, X, off, B, ks, alpha, 1, mean, stream);
}

extern "C" int tgp_predict_mean_batch_multi(const double* Xs, const int64_t* soff, const double* X,
                                            const int64_t* off, int32_t B, const tgp_kernel_sum* ks,
                                            const double* alpha, int32_t r, double* mean, void* stream) {
  return predict_mean_batch_entry(__func__, Xs, soff, X, off, B, ks, alpha, r, mean, stream);
}

// ---- leave-one-out predictions (tgp_loo_batch) ---------------------------------------------------------------------
// One CTA per problem, in residual space, with the operations of GPInterpolation.loo_predict in the same order:
// mean_ic = y_ic - alpha_ic / Z_ii for each output c, var_i = 1 / Z_ii - yerr2_i once per point; NaN for a problem
// with info != 0.
__global__ void __launch_bounds__(256)
loo_finish_batch_kernel(const TgpBatchProb* __restrict__ pr, const int64_t* __restrict__ off,
                        const int32_t* __restrict__ info, double* __restrict__ mean, double* __restrict__ var) {
  const TgpBatchProb& p = pr[blockIdx.x];
  const int64_t r0 = off[blockIdx.x], r = p.r;
  const bool ok = info[blockIdx.x] == 0;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  for (int64_t i = threadIdx.x; i < p.N; i += blockDim.x) {
    const double z = p.A[i * p.ld + i];
    for (int64_t c = 0; c < r; ++c) mean[(r0 + i) * r + c] = ok ? p.y[i * r + c] - p.alpha[i * r + c] / z : nan;
    var[r0 + i] = ok ? 1.0 / z - p.yerr2[i] : nan;
  }
}

static int loo_batch_entry(const char* fn, const double* X, const double* y, int32_t r, const double* yerr2,
                           const int64_t* off, int32_t B, const tgp_kernel_sum* ks, double* work, double* alpha,
                           double* scratch, double* loo_mean, double* loo_var, int32_t* info, void* stream) {
  int rc = check_selinv_batch(fn, r, off, B, ks,
                              X && y && yerr2 && work && alpha && scratch && loo_mean && loo_var && info,
                              "null pointer (X, y, yerr2, work, alpha, scratch, loo_mean, loo_var, info)", work, scratch);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<unsigned char> tail((size_t)(B + 1) * sizeof(int64_t));   // the offsets, for the finish
  memcpy(tail.data(), off, tail.size());
  BatchTables T;
  std::vector<TgpBatchProb> prob;
  double* const* scr = nullptr;
  rc = selinv_batch_run(X, y, r, yerr2, off, B, ks, work, alpha, info, scratch, st, T, prob, &scr, tail);
  if (rc) return rc;
  const int64_t* off_d = reinterpret_cast<const int64_t*>(reinterpret_cast<const unsigned char*>(scr) +
                                                          align16((size_t)B * sizeof(double*)));
  loo_finish_batch_kernel<<<(unsigned)B, 256, 0, st>>>(T.pr, off_d, info, loo_mean, loo_var);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

extern "C" int tgp_loo_batch(const double* X, const double* y, const double* yerr2, const int64_t* off, int32_t B,
                             const tgp_kernel_sum* ks, double* work, double* alpha, double* scratch, double* loo_mean,
                             double* loo_var, int32_t* info, void* stream) {
  return loo_batch_entry(__func__, X, y, 1, yerr2, off, B, ks, work, alpha, scratch, loo_mean, loo_var, info, stream);
}

extern "C" int tgp_loo_batch_multi(const double* X, const double* Y, int32_t r, const double* yerr2,
                                   const int64_t* off, int32_t B, const tgp_kernel_sum* ks, double* work,
                                   double* alpha, double* scratch, double* loo_mean, double* loo_var, int32_t* info,
                                   void* stream) {
  return loo_batch_entry(__func__, X, Y, r, yerr2, off, B, ks, work, alpha, scratch, loo_mean, loo_var, info, stream);
}

// ---- predictive variance (tgp_predict_var_batch) -------------------------------------------------------------------
// Per pass over `chunk` test points of every problem: K(Xs, X) into each problem's rows of vwork, then V <- V L^-T as
// trsm_rows_blocked (dense) runs it, for all problems in one launch sequence: per 512-wide block column of the largest
// problem the halving solve (leaf, gemm, leaf, ..., the gemm between leaves i and i + 1 shaped by tgp_halving_node) and
// the trailing update V[:, c1:N] -= V[:, k:c1] L[c1:N, k:c1]^T; last the variance of every row.  Every launch runs the
// single-problem body with the single call's operands, so each row gets tgp_predict_var_sum's arithmetic.

// The largest row count per pass the launches accept: the gemm grid (row tiles x column tiles) and the K build's row
// tiles stay within 65535.
static int64_t var_chunk_limit(int64_t max_n) { return std::min<int64_t>(65535 / tgp_cdiv(max_n, 64) * 128, 65535 * 64); }

static int check_var_batch(const char* fn, const int64_t* soff, const int64_t* off, int32_t B, int64_t chunk) {
  BATCH_CHECK(B >= 1, "B must be >= 1");
  int rc = check_offsets(fn, "off", off, B, 1, TGP_BATCH_MAX_N);
  if (rc) return rc;
  rc = check_offsets(fn, "soff", soff, B, 0, INT64_MAX);
  if (rc) return rc;
  BATCH_CHECK(chunk >= 1, "chunk must be >= 1");
  int64_t max_n = 0, max_m = 0;
  for (int32_t b = 0; b < B; ++b) {
    max_n = std::max(max_n, off[b + 1] - off[b]);
    max_m = std::max(max_m, soff[b + 1] - soff[b]);
  }
  char msg[160];
  snprintf(msg, sizeof msg, "chunk = %lld exceeds %lld test points per pass (grid limit for N_b = %lld)",
           (long long)chunk, (long long)var_chunk_limit(max_n), (long long)max_n);
  BATCH_CHECK(std::min(chunk, max_m) <= var_chunk_limit(max_n), msg);
  return TGP_OK;
}

extern "C" int64_t tgp_predict_var_batch_work_doubles(const int64_t* soff, const int64_t* off, int32_t B,
                                                      int64_t chunk) {
  if (check_var_batch(__func__, soff, off, B, chunk)) return TGP_ERR_INVALID;
  int64_t total = 0;
  for (int32_t b = 0; b < B; ++b) total += std::min(soff[b + 1] - soff[b], chunk) * even_ld(off[b + 1] - off[b]);
  return total;
}

struct VarOp {   // one launch of the row solve: the leaves of one halving step, or one gemm
  std::vector<TgpLeafArgs> full, edge;
  std::vector<TgpGemmArgs> gemm;
};

extern "C" int tgp_predict_var_batch(const double* Xs, const int64_t* soff, const double* X, const int64_t* off,
                                     int32_t B, const tgp_kernel_sum* ks, const double* work, double* vwork,
                                     int64_t chunk, double* var, void* stream) {
  const char* fn = __func__;
  int rc = check_var_batch(fn, soff, off, B, chunk);
  if (rc) return rc;
  rc = check_batch(fn, off, B, ks);
  if (rc) return rc;
  BATCH_CHECK(X && work, "null pointer (X, work)");
  BATCH_CHECK(((uintptr_t)work & 15) == 0, "work must be 16-byte aligned");
  if (soff[B] == 0) return TGP_OK;
  BATCH_CHECK(Xs && vwork && var, "null pointer (Xs, vwork, var)");
  BATCH_CHECK(((uintptr_t)vwork & 15) == 0, "vwork must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int ndim = ks[0].ndim;
  std::vector<int> cls(B);
  std::vector<int64_t> Nh(B), ld(B), voff(B), woff(B);
  std::vector<double> prior(B);
  int64_t max_n = 0, max_m = 0, v = 0, w = 0;
  for (int32_t b = 0; b < B; ++b) {
    Nh[b] = off[b + 1] - off[b];
    ld[b] = even_ld(Nh[b]);
    woff[b] = w;
    w += (Nh[b] + 1) * ld[b];
    voff[b] = v;
    v += std::min(soff[b + 1] - soff[b], chunk) * ld[b];
    max_n = std::max(max_n, Nh[b]);
    max_m = std::max(max_m, soff[b + 1] - soff[b]);
    // tgp_kmat_cross_sum: the single-term kernel for any one-term sum (no white term in K(Xs, X))
    cls[b] = ks[b].nterms == 1 ? ks[b].term[0].family : TGP_BATCH_SUM;
    double p = ks[b].white;   // the prior variance in predict_var_impl's order
    for (int c = 0; c < ks[b].nterms; ++c) p += ks[b].term[c].amp;
    prior[b] = p;
  }
  for (int64_t m0 = 0; m0 < max_m; m0 += chunk) {
    std::vector<TgpBatchProb> prob(B);
    std::vector<int64_t> mc(B);
    for (int32_t b = 0; b < B; ++b) {
      TgpBatchProb& p = prob[b];
      p = TgpBatchProb{};
      mc[b] = std::max<int64_t>(0, std::min(soff[b + 1] - soff[b] - m0, chunk));
      p.X = X + off[b] * ndim;
      p.N = Nh[b];
      p.ld = ld[b];
      p.A = vwork + voff[b];
      p.M = mc[b];
      p.Xs = Xs + (soff[b] + (mc[b] ? m0 : 0)) * ndim;
      p.mean = var + soff[b] + (mc[b] ? m0 : 0);
    }
    // the launch sequence of the row solve
    std::vector<VarOp> ops;
    for (int64_t k = 0; k < max_n; k += TGP_OB) {
      int64_t wmax = 0;
      for (int32_t b = 0; b < B; ++b)
        if (mc[b] > 0 && Nh[b] > k) wmax = std::max(wmax, std::min<int64_t>(TGP_OB, Nh[b] - k));
      const int nleaves = (int)tgp_cdiv(wmax, 64);
      for (int i = 0; i < nleaves; ++i) {
        ops.emplace_back();
        const int64_t c0 = 64 * (int64_t)i;
        for (int32_t b = 0; b < B; ++b) {   // leaf i of problem b, on the path trsm_panel_launch takes for it
          const int64_t wb = std::min<int64_t>(TGP_OB, Nh[b] - k);
          if (mc[b] == 0 || wb <= c0) continue;
          const double* L = work + woff[b] + (k + c0) * ld[b] + k + c0;
          double* Vb = prob[b].A + k + c0;
          const int nb = (int)std::min<int64_t>(wb - c0, 64);
          const bool full = nb == 64 && (ld[b] & 1) == 0 && ((uintptr_t)Vb & 15) == 0;
          (full ? ops.back().full : ops.back().edge).push_back(TgpLeafArgs{L, Vb, ld[b], mc[b], ld[b], nb});
        }
        if (i + 1 == nleaves) break;
        ops.emplace_back();
        for (int32_t b = 0; b < B; ++b) {   // B2 -= B1 L21^T on the node [o, o + n) of leaves i and i + 1, split at h
          const int64_t wb = std::min<int64_t>(TGP_OB, Nh[b] - k);
          if (mc[b] == 0 || wb <= 0 || i + 1 >= tgp_cdiv(wb, 64)) continue;
          int64_t o, h, n;
          tgp_halving_node(wb, i, o, h, n);
          const double* Lk = work + woff[b] + k * ld[b] + k;
          double* Vk = prob[b].A + k;
          ops.back().gemm.push_back(TgpGemmArgs{Vk + o + h, Vk + o, Lk + (o + h) * ld[b] + o, mc[b], n - h, h, ld[b]});
        }
      }
      ops.emplace_back();
      const int64_t c1 = k + TGP_OB;
      for (int32_t b = 0; b < B; ++b) {   // V[:, c1:N] -= V[:, k:c1] L[c1:N, k:c1]^T
        if (mc[b] == 0 || Nh[b] <= c1) continue;
        ops.back().gemm.push_back(TgpGemmArgs{prob[b].A + c1, prob[b].A + k, work + woff[b] + c1 * ld[b] + k, mc[b],
                                              Nh[b] - c1, TGP_OB, ld[b]});
      }
    }
    std::vector<unsigned char> extra((size_t)B * sizeof(double));   // the prior variances
    memcpy(extra.data(), prior.data(), extra.size());
    BatchTables T;
    rc = stage_tables(T, prob, ks, cls, st, extra);
    if (rc) return rc;
    for (int c = 0; c < TGP_BATCH_NCLASS; ++c) {
      if (T.start[c + 1] == T.start[c] || T.max_m[c] == 0) continue;
      rc = tgp_batch_kmat_cross(T.pr, T.kd, T.list + T.start[c], T.start[c + 1] - T.start[c], c, T.max_n[c],
                                T.max_m[c], st);
      if (rc) return rc;
    }
    for (const VarOp& op : ops) {
      if ((rc = tgp_batch_gemm(op.gemm.data(), (int32_t)op.gemm.size(), st))) return rc;
      if ((rc = tgp_batch_selinv_leaves(op.full.data(), (int32_t)op.full.size(), true, st))) return rc;
      if ((rc = tgp_batch_selinv_leaves(op.edge.data(), (int32_t)op.edge.size(), false, st))) return rc;
    }
    rc = tgp_batch_var_rows(T.pr, reinterpret_cast<const double*>(T.extra), B,
                            std::min(chunk, max_m - m0), st);
    if (rc) return rc;
  }
  return TGP_OK;
}
