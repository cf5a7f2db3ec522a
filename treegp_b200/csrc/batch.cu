// Batches of independent small problems: B likelihood evaluations (tgp_loglike_batch), B likelihoods with their
// gradients (tgp_loglike_grad_batch) or B posterior means (tgp_predict_mean_batch) per call.
//
// A problem of a few hundred to a few thousand points leaves the B200 idle: its factorisation is a chain of small
// launches (8 panel launches and one update per 512 columns, at most ~70 CTAs each), so its time is launch latency.
// Here every launch of that chain carries all B problems: the schedule runs over the panel steps of the largest
// problem, each CTA picks its problem from blockIdx.x and runs the body of the single-problem kernel on that
// problem's slice (kmat.cu, dense.cu, predict.cu), and CTAs of problems without work at that step exit.  So a
// problem's K, factor, logL and info are what tgp_loglike_sum (dense) gives on it alone, bit for bit, whatever else
// shares the batch.  The only new arithmetic is the backward sweep of want_alpha (one CTA per problem, below).  The
// gradient adds the selected inverse, contraction and finish of tgp_loglike_grad_sum in the same form (selinv.cu).
#include <string.h>
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

extern "C" int64_t tgp_batch_work_doubles(const int64_t* off, int32_t B) {
  const char* fn = __func__;
  if (B < 1) {
    tgp_set_error("%s: invalid argument: B must be >= 1", fn);
    return TGP_ERR_INVALID;
  }
  if (check_offsets(fn, "off", off, B, 1, TGP_BATCH_MAX_N)) return TGP_ERR_INVALID;
  int64_t total = 0;
  for (int32_t b = 0; b < B; ++b) {
    const int64_t n = off[b + 1] - off[b];
    total += (n + 1) * even_ld(n);
  }
  return total;
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

// y into row N of every block (to_alpha == 0), or row N (= L^-1 y after the factorisation) into alpha.
__global__ void __launch_bounds__(256)
batch_yrow_kernel(const TgpBatchProb* __restrict__ pr, int to_alpha) {
  const TgpBatchProb& p = pr[blockIdx.x];
  double* row = p.A + p.N * p.ld;
  for (int64_t i = threadIdx.x; i < p.N; i += blockDim.x) {
    if (to_alpha) p.alpha[i] = row[i];
    else row[i] = p.y[i];
  }
}

// Backward sweep alpha <- L^-T alpha, one CTA per problem (the persistent cooperative sweeps of trsv.cu take one
// problem per launch).  Blocks of 64 unknowns from the last: the four row groups of the CTA form
// sum_{i >= j1} L[i, j0 + c] x_i for the block's 64 columns (each L entry is read once, rows coalesced), then warp 0
// solves the 64 x 64 diagonal block by substitution with shuffles.  x lives in shared memory.
constexpr int BS_THREADS = 256;
constexpr int BS_NB = 64;
constexpr int BS_SMEM = (TGP_BATCH_MAX_N + BS_NB * (BS_NB + 1) + 4 * BS_NB) * 8;

__global__ void __launch_bounds__(BS_THREADS)
backward_batch_kernel(const TgpBatchProb* __restrict__ pr) {
  extern __shared__ double bsm[];
  double* x = bsm;                                 // N unknowns
  double* Ld = bsm + TGP_BATCH_MAX_N;              // diagonal block, pitch BS_NB + 1
  double* part = Ld + BS_NB * (BS_NB + 1);         // 4 partial sums per column
  const TgpBatchProb& p = pr[blockIdx.x];
  const int64_t N = p.N, ld = p.ld;
  const double* L = p.A;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = tid & (BS_NB - 1), g = tid / BS_NB;
  for (int64_t i = tid; i < N; i += BS_THREADS) x[i] = p.alpha[i];
  __syncthreads();
  for (int64_t j0 = (N - 1) / BS_NB * BS_NB; j0 >= 0; j0 -= BS_NB) {
    const int nb = (int)(N - j0 < BS_NB ? N - j0 : BS_NB);
    const int64_t j1 = j0 + nb;
    double s = 0.0;
    if (c < nb) {
#pragma unroll 4
      for (int64_t i = j1 + g; i < N; i += 4) s = fma(L[i * ld + j0 + c], x[i], s);
    }
    part[g * BS_NB + c] = s;
    for (int idx = tid; idx < BS_NB * BS_NB; idx += BS_THREADS) {
      const int r = idx / BS_NB, cc = idx % BS_NB;
      Ld[r * (BS_NB + 1) + cc] = (r < nb && cc <= r) ? L[(j0 + r) * ld + j0 + cc] : 0.0;
    }
    __syncthreads();
    if (warp == 0) {
      // lane owns unknowns j0 + lane (r0) and j0 + 32 + lane (r1)
      double r0 = 0.0, r1 = 0.0;
      if (lane < nb)
        r0 = x[j0 + lane] - (((part[lane] + part[BS_NB + lane]) + part[2 * BS_NB + lane]) + part[3 * BS_NB + lane]);
      if (lane + 32 < nb) {
        const int l = lane + 32;
        r1 = x[j0 + l] - (((part[l] + part[BS_NB + l]) + part[2 * BS_NB + l]) + part[3 * BS_NB + l]);
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
      if (lane < nb) x[j0 + lane] = r0;
      if (lane + 32 < nb) x[j0 + lane + 32] = r1;
    }
    __syncthreads();
  }
  for (int64_t i = tid; i < N; i += BS_THREADS) p.alpha[i] = x[i];
}

// The chain of tgp_loglike_batch on checked arguments, with the tables staged into T (plus `extra` bytes) and their
// host copy in prob.  out: 3 B doubles, or nullptr for T.extra's first 3 B doubles.
static int loglike_batch_run(const double* X, const double* y, const double* yerr2, const int64_t* off, int32_t B,
                             const tgp_kernel_sum* ks, double* work, double* alpha, int want_alpha, double* out,
                             int32_t* info, cudaStream_t st, BatchTables& T, std::vector<TgpBatchProb>& prob,
                             const std::vector<unsigned char>& extra) {
  int rc;
  const int ndim = ks[0].ndim;
  prob.assign(B, TgpBatchProb{});
  std::vector<int> cls(B);
  std::vector<int64_t> Nh(B);
  int64_t woff = 0;
  for (int32_t b = 0; b < B; ++b) {
    const int64_t r0 = off[b], n = off[b + 1] - off[b];
    TgpBatchProb& p = prob[b];
    p = TgpBatchProb{};
    p.X = X + r0 * ndim;
    p.y = y + r0;
    p.yerr2 = yerr2 + r0;
    p.A = work + woff;
    p.alpha = alpha + r0;
    p.N = Nh[b] = n;
    p.ld = even_ld(n);
    woff += (n + 1) * p.ld;
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
  rc = tgp_batch_potrf_rows(T.pr, Nh.data(), B, info, T.flags, st);
  if (rc) return rc;
  batch_yrow_kernel<<<(unsigned)B, 256, 0, st>>>(T.pr, 1);
  TGP_LAUNCH_CHECK();
  if (want_alpha) {
    static TgpPerDeviceOnce attr_once;
    if (tgp_first_use_on_device(attr_once))
      TGP_CUDA(cudaFuncSetAttribute(backward_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BS_SMEM));
    backward_batch_kernel<<<(unsigned)B, BS_THREADS, BS_SMEM, st>>>(T.pr);
    TGP_LAUNCH_CHECK();
  }
  return tgp_batch_loglike_finish(T.pr, B, want_alpha, info, out, st);
}

extern "C" int tgp_loglike_batch(const double* X, const double* y, const double* yerr2, const int64_t* off, int32_t B,
                                 const tgp_kernel_sum* ks, double* work, double* alpha, int want_alpha, double* out,
                                 int32_t* info, void* stream) {
  const char* fn = __func__;
  int rc = check_batch(fn, off, B, ks);
  if (rc) return rc;
  BATCH_CHECK(X && y && yerr2 && work && alpha && out && info, "null pointer (X, y, yerr2, work, alpha, out, info)");
  BATCH_CHECK(((uintptr_t)work & 15) == 0, "work must be 16-byte aligned");
  BatchTables T;
  std::vector<TgpBatchProb> prob;
  return loglike_batch_run(X, y, yerr2, off, B, ks, work, alpha, want_alpha, out, info, (cudaStream_t)stream, T, prob,
                           std::vector<unsigned char>());
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

extern "C" int tgp_loglike_grad_batch(const double* X, const double* y, const double* yerr2, const int64_t* off,
                                      int32_t B, const tgp_kernel_sum* ks, double* work, double* alpha, double* out,
                                      int32_t* info, double* scratch, void* stream) {
  const char* fn = __func__;
  int rc = check_batch(fn, off, B, ks);
  if (rc) return rc;
  BATCH_CHECK(X && y && yerr2 && work && alpha && out && info && scratch,
              "null pointer (X, y, yerr2, work, alpha, out, info, scratch)");
  BATCH_CHECK(((uintptr_t)work & 15) == 0, "work must be 16-byte aligned");
  BATCH_CHECK(((uintptr_t)scratch & 15) == 0, "scratch must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  // extra tables: {logL, chi2, logdet} per problem, then the scratch block of every problem
  const size_t o_scr = align16((size_t)B * 3 * sizeof(double));
  std::vector<unsigned char> extra(o_scr + (size_t)B * sizeof(double*), 0);
  double** scr_h = reinterpret_cast<double**>(extra.data() + o_scr);
  int64_t soff = 0;
  for (int32_t b = 0; b < B; ++b) {
    scr_h[b] = scratch + soff;
    soff += tgp_loglike_grad_sum_work_doubles(off[b + 1] - off[b], TGP_MAX_TERMS);
  }
  BatchTables T;
  std::vector<TgpBatchProb> prob;
  rc = loglike_batch_run(X, y, yerr2, off, B, ks, work, alpha, 1, nullptr, info, st, T, prob, extra);
  if (rc) return rc;
  const double* ll = reinterpret_cast<const double*>(T.extra);
  double* const* scr = reinterpret_cast<double* const*>(T.extra + o_scr);
  rc = tgp_batch_selinv(T.pr, scr, prob.data(), scr_h, B, st);
  if (rc) return rc;
  for (int c = 0; c < TGP_BATCH_NCLASS; ++c) {
    if (T.start[c + 1] == T.start[c]) continue;
    int max_terms = 1;   // a sum's CTAs of terms beyond its own exit
    if (c == TGP_BATCH_SUM) {
      for (int32_t b = 0; b < B; ++b) max_terms = ks[b].nterms > max_terms ? ks[b].nterms : max_terms;
    }
    rc = tgp_batch_grad_contract(T.pr, T.kd, T.list + T.start[c], T.start[c + 1] - T.start[c], c, scr, T.max_n[c],
                                 max_terms, st);
    if (rc) return rc;
  }
  return tgp_batch_grad_finish(T.pr, T.kd, scr, B, info, ll, out, st);
}

extern "C" int tgp_predict_mean_batch(const double* Xs, const int64_t* soff, const double* X, const int64_t* off,
                                      int32_t B, const tgp_kernel_sum* ks, const double* alpha, double* mean,
                                      void* stream) {
  const char* fn = __func__;
  int rc = check_batch(fn, off, B, ks);
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
    p.alpha = const_cast<double*>(alpha) + off[b];
    p.N = off[b + 1] - off[b];
    p.Xs = Xs + soff[b] * ndim;
    p.mean = mean + soff[b];
    p.M = soff[b + 1] - soff[b];
    // tgp_predict_mean_sum: the single-term kernel for any one-term sum (no white term in K(Xs, X))
    cls[b] = ks[b].nterms == 1 ? ks[b].term[0].family : TGP_BATCH_SUM;
  }
  BatchTables T;
  rc = stage_tables(T, prob, ks, cls, st);
  if (rc) return rc;
  for (int c = 0; c < TGP_BATCH_NCLASS; ++c) {
    if (T.start[c + 1] == T.start[c] || T.max_m[c] == 0) continue;
    rc = tgp_batch_predict_mean(T.pr, T.kd, T.list + T.start[c], T.start[c + 1] - T.start[c], c, T.max_m[c], st);
    if (rc) return rc;
  }
  return TGP_OK;
}
