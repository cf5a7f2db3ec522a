// GP prediction: fused, never-materialised K(Xs, X) . alpha, and the diagonal predictive variance.
//
// Replaces /root/reference/treegp/gp_interp.py:177 + :183 (HT = kernel(X2, Y=X1); HT . alpha) and the
// diagonal of :187-191 (v = cho_solve(L, HT^T); K** - HT v).  The reference materialises the M x N
// matrix HT (320 GB at M = 1e6, N = 4e4); here each thread owns one test point, the training
// coordinates and alpha stream through shared memory, and only M doubles are written.
#include "tgp_common.cuh"
#include "profile_policy.cuh"
#include "batch.cuh"

constexpr int PM_THREADS = 256;   // test points per CTA
constexpr int PM_TILE = 1024;     // training points per shared-memory tile

// grid: (ceil(M / PM_THREADS), nsplit).  Split s handles training tiles s, s + nsplit, ...
// nsplit == 1 writes mean directly; otherwise partial sums are added with red.global.add.f64 into a
// zeroed output (used only when M alone cannot fill the machine).
// Several outputs (P = MultiOut<..., R>): alpha and mean are row-major (N, r) and (M, r); each thread keeps R pairs of
// accumulators, evaluates every pair's profile once and applies it to all columns -- each column in the order of the
// single-output kernel.  The tile shrinks with R so that the staged alpha stays at 16 KB.
// BATCH (tgp_predict_mean_batch): grid (problems of one profile class, test-point blocks of the largest of them); the
// problem's slices and descriptor replace the arguments, and every CTA sums all training tiles of its problem in order
// (one split): the single call's sum whenever that call runs unsplit, independent of the other problems.
template <class P, bool BATCH = false>
__global__ void __launch_bounds__(PM_THREADS)
predict_mean_kernel(const double* __restrict__ Xs, int64_t M, const double* __restrict__ X, int64_t N,
                    P prof, const double* __restrict__ alpha, double* __restrict__ mean,
                    const double* __restrict__ phi_g, const TgpBatchProb* __restrict__ pr = nullptr,
                    const KSumDesc* __restrict__ kd = nullptr, const int32_t* __restrict__ list = nullptr) {
  unsigned bx = blockIdx.x, by = blockIdx.y;
  int nsplit = gridDim.y;
  if constexpr (BATCH) {
    const int b = list[blockIdx.x];
    M = pr[b].M;
    if ((int64_t)blockIdx.y * PM_THREADS >= M) return;
    Xs = pr[b].Xs;
    X = pr[b].X;
    N = pr[b].N;
    alpha = pr[b].alpha;
    mean = pr[b].mean;
    prof = tgp_batch_profile<P>(kd[b]);
    bx = blockIdx.y;
    by = 0;
    nsplit = 1;
  }
  constexpr int R = OutputsOf<P>::kR;
  constexpr int TILE = R == 1 ? PM_TILE : 2048 / R;
  __shared__ double2 pxy[TILE];
  __shared__ double pa[TILE * R];
  __shared__ double phi_s[P::kPhiSize];
  const int tid = threadIdx.x;
  if (prof.stage_phi()) tgp_stage_phi(phi_s, phi_g);
  const int64_t m = (int64_t)bx * PM_THREADS + tid;
  const bool live = m < M;
  const double sx = live ? Xs[m * prof.desc.ndim] : 0.0;
  const double sy = (live && prof.desc.ndim == 2) ? Xs[m * 2 + 1] : 0.0;
  const int64_t ntile = (N + TILE - 1) / TILE;
  double acc0 = 0.0, acc1 = 0.0;
  double accm0[R], accm1[R];
#pragma unroll
  for (int c = 0; c < R; ++c) accm0[c] = accm1[c] = 0.0;
  for (int64_t tl = by; tl < ntile; tl += nsplit) {
    const int64_t n0 = tl * TILE;
    __syncthreads();
    for (int i = tid; i < TILE; i += PM_THREADS) {
      const int64_t n = n0 + i;
      const bool ok = n < N;
      double2 p;
      p.x = ok ? X[n * prof.desc.ndim] : 0.0;
      p.y = (ok && prof.desc.ndim == 2) ? X[n * 2 + 1] : 0.0;
      pxy[i] = p;
      if constexpr (R == 1) {
        pa[i] = ok ? prof.weight() * alpha[n] : 0.0;  // padded points carry zero weight
      } else {
#pragma unroll
        for (int c = 0; c < R; ++c) pa[i * R + c] = (ok && c < prof.nrhs) ? prof.weight() * alpha[n * prof.nrhs + c] : 0.0;
      }
    }
    __syncthreads();
    if constexpr (R > 1) {
      for (int i = 0; i < TILE; i += 2) prof.mean2_multi(sx, sy, pxy, pa, i, phi_s, accm0, accm1);
    } else if constexpr (P::kSum) {
      for (int i = 0; i < PM_TILE; i += 2) prof.mean2(sx, sy, pxy, pa, i, phi_s, acc0, acc1);
    } else {
      const KDesc& kd = prof.desc;
#pragma unroll 2
      for (int i = 0; i < PM_TILE; i += 2) {
        const double2 p0 = pxy[i], p1 = pxy[i + 1];
        const double q0 = tgp_qform(kd, sx - p0.x, sy - p0.y);
        const double q1 = tgp_qform(kd, sx - p1.x, sy - p1.y);
        acc0 = fma(tgp_profile<P::kFam>(q0, phi_s), pa[i], acc0);
        acc1 = fma(tgp_profile<P::kFam>(q1, phi_s), pa[i + 1], acc1);
      }
    }
  }
  if (live) {
    if constexpr (R == 1) {
      const double v = acc0 + acc1;
      if (nsplit == 1) mean[m] = v;
      else atomicAdd(mean + m, v);
    } else {
#pragma unroll
      for (int c = 0; c < R; ++c) {
        if (c < prof.nrhs) {
          const double v = accm0[c] + accm1[c];
          if (nsplit == 1) mean[m * prof.nrhs + c] = v;
          else atomicAdd(mean + m * prof.nrhs + c, v);
        }
      }
    }
  }
}

template <class P>
static int predict_mean_launch(const double* Xs, int64_t M, const double* X, int64_t N, const P& prof,
                               const double* alpha, double* mean, void* stream) {
  TGP_CHECK_ARG(M >= 0 && N >= 0, "M/N");
  if (M == 0) return TGP_OK;
  TGP_CHECK_ARG(Xs && mean && (N == 0 || (X && alpha)), "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t gx = tgp_cdiv(M, PM_THREADS);
  constexpr int R = OutputsOf<P>::kR;
  int64_t nout = 1;
  if constexpr (R > 1) nout = prof.nrhs;
  const int64_t ntile = tgp_cdiv(N, (int64_t)(R == 1 ? PM_TILE : 2048 / R));
  int64_t nsplit = 1;
  const int64_t target = 4ll * tgp_num_sms();
  if (gx < target) nsplit = tgp_cdiv(target, gx);
  if (nsplit > ntile) nsplit = ntile > 0 ? ntile : 1;
  if (nsplit > 65535) nsplit = 65535;
  if (nsplit > 1 || N == 0) TGP_CUDA(cudaMemsetAsync(mean, 0, M * nout * sizeof(double), st));
  if (N == 0) return TGP_OK;
  dim3 grid((unsigned)gx, (unsigned)nsplit);
  predict_mean_kernel<P><<<grid, PM_THREADS, 0, st>>>(Xs, M, X, N, prof, alpha, mean, tgp_phi_device());
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

extern "C" int tgp_predict_mean(const double* Xs, int64_t M, const double* X, int64_t N,
                                const tgp_kernel* k, const double* alpha, double* mean, void* stream) {
  TGP_CHECK_ARG(kdesc_ok(k), "kernel descriptor");
  const KDesc kd = make_kdesc(k);
  TGP_FAMILY_SWITCH(k->family, return predict_mean_launch(Xs, M, X, N, FamilyProfile<FAM>{kd}, alpha, mean, stream));
  return TGP_OK;
}

extern "C" int tgp_predict_mean_sum(const double* Xs, int64_t M, const double* X, int64_t N, const tgp_kernel_sum* k,
                                    const double* alpha, double* mean, void* stream) {
  TGP_CHECK_ARG(ksum_ok(k), "kernel sum descriptor");
  if (k->nterms == 1) return tgp_predict_mean(Xs, M, X, N, &k->term[0], alpha, mean, stream);
  return predict_mean_launch(Xs, M, X, N, SumProfile{make_ksumdesc(k)}, alpha, mean, stream);
}

int tgp_batch_predict_mean(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list, int32_t count, int cls,
                           int64_t max_m, cudaStream_t st) {
  const int64_t gy = tgp_cdiv(max_m, PM_THREADS);
  TGP_CHECK_ARG(gy <= 65535, "too many test points in one problem (at most 65535 * 256)");
  const dim3 grid((unsigned)count, (unsigned)gy);
  const double* phi = tgp_phi_device();
  if (cls == TGP_BATCH_SUM) {
    predict_mean_kernel<SumProfile, true><<<grid, PM_THREADS, 0, st>>>(nullptr, 0, nullptr, 0, SumProfile{}, nullptr,
                                                                      nullptr, phi, pr, kd, list);
  } else {
    TGP_FAMILY_SWITCH(cls, (predict_mean_kernel<FamilyProfile<FAM>, true><<<grid, PM_THREADS, 0, st>>>(
                               nullptr, 0, nullptr, 0, FamilyProfile<FAM>{}, nullptr, nullptr, phi, pr, kd, list)));
  }
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

// ---------------------------------------------------------------------------------------------
// Truncated-support variant.  Every profile f(q) decays (at least) exponentially, so the terms of
// sum_n K(x*, x_n) alpha_n with q beyond q_cut, f(q_cut) = 1e-40, change the sum by at most
// 1e-40 * sum_n |amp alpha_n| -- forty orders of magnitude below FP64 rounding of the sum itself.  The kernel
// skips whole groups of PG training points whose bounding box is provably farther than that from the bounding
// box of the CTA's 256 test points (q >= lambda_min(M) |delta|^2).  The rule is exact for ANY point order; it
// only pays when both point sets are stored in a space-filling-curve order (the host sorts them with
// tgp_hilbert_keys), where at the reference's field sizes >90 % of the N x M evaluations disappear.
// Groups that survive are evaluated in full, pair by pair, exactly as predict_mean_kernel does.
// ---------------------------------------------------------------------------------------------
constexpr int PG = 128;   // training points per bounding box

static double profile_qcut(int family) {
  // smallest q with f(q) <= 1e-40 (tools/gen_vk_tables.py conventions; checked in tests/test_cpu_host.py)
  switch (family) {
    case TGP_FAM_RBF: return 185.0;
    case TGP_FAM_VONKARMAN: return 224.0;
    case TGP_FAM_MATERN12: return 8484.0;
    case TGP_FAM_MATERN32: return 3117.0;
    default: return 2011.0;
  }
}

extern "C" int64_t tgp_predict_work_doubles(int64_t N) { return 4 * tgp_cdiv(N > 0 ? N : 1, PG); }
extern "C" double tgp_profile_qcut(int32_t family) { return profile_qcut(family); }

// boxes[4 g .. 4 g + 3] = {xmin, xmax, ymin, ymax} of training points [g PG, (g+1) PG).  Warp per group.
__global__ void __launch_bounds__(256)
point_boxes_kernel(const double* __restrict__ X, int64_t N, int ndim, double* __restrict__ boxes, int64_t ngroups) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t g = (int64_t)blockIdx.x * 8 + warp;
  if (g >= ngroups) return;
  double x0 = INFINITY, x1 = -INFINITY, y0 = INFINITY, y1 = -INFINITY;
  for (int i = lane; i < PG; i += 32) {
    const int64_t n = g * PG + i;
    if (n < N) {
      const double x = X[n * ndim], y = (ndim == 2) ? X[n * 2 + 1] : 0.0;
      x0 = fmin(x0, x); x1 = fmax(x1, x);
      y0 = fmin(y0, y); y1 = fmax(y1, y);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    x0 = fmin(x0, __shfl_xor_sync(0xffffffffu, x0, o));
    x1 = fmax(x1, __shfl_xor_sync(0xffffffffu, x1, o));
    y0 = fmin(y0, __shfl_xor_sync(0xffffffffu, y0, o));
    y1 = fmax(y1, __shfl_xor_sync(0xffffffffu, y1, o));
  }
  if (lane == 0) {
    boxes[4 * g + 0] = x0; boxes[4 * g + 1] = x1; boxes[4 * g + 2] = y0; boxes[4 * g + 3] = y1;
  }
}

template <class P>
__global__ void __launch_bounds__(PM_THREADS, OutputsOf<P>::kR > 1 ? 1 : 0)
predict_mean_trunc_kernel(const double* __restrict__ Xs, int64_t M, const double* __restrict__ X, int64_t N,
                          P prof, const double* __restrict__ alpha, double* __restrict__ mean,
                          const double* __restrict__ phi_g, const double* __restrict__ boxes, int64_t ngroups,
                          double r2cut) {
  constexpr int R = OutputsOf<P>::kR;
  __shared__ double2 pxy[PG];
  __shared__ double pa[PG * R];
  __shared__ double phi_s[P::kPhiSize];
  __shared__ double red[8][4];
  __shared__ int list[PM_THREADS];
  __shared__ int wcount[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (prof.stage_phi()) tgp_stage_phi(phi_s, phi_g);
  const int64_t m = (int64_t)blockIdx.x * PM_THREADS + tid;
  const bool live = m < M;
  const double sx = live ? Xs[m * prof.desc.ndim] : 0.0;
  const double sy = (live && prof.desc.ndim == 2) ? Xs[m * 2 + 1] : 0.0;
  // bounding box of this CTA's test points
  double bx0 = live ? sx : INFINITY, bx1 = live ? sx : -INFINITY, by0 = live ? sy : INFINITY, by1 = live ? sy : -INFINITY;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    bx0 = fmin(bx0, __shfl_xor_sync(0xffffffffu, bx0, o));
    bx1 = fmax(bx1, __shfl_xor_sync(0xffffffffu, bx1, o));
    by0 = fmin(by0, __shfl_xor_sync(0xffffffffu, by0, o));
    by1 = fmax(by1, __shfl_xor_sync(0xffffffffu, by1, o));
  }
  if (lane == 0) { red[warp][0] = bx0; red[warp][1] = bx1; red[warp][2] = by0; red[warp][3] = by1; }
  __syncthreads();
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    bx0 = fmin(bx0, red[w][0]); bx1 = fmax(bx1, red[w][1]);
    by0 = fmin(by0, red[w][2]); by1 = fmax(by1, red[w][3]);
  }
  double acc0 = 0.0, acc1 = 0.0;
  double accm0[R], accm1[R];
#pragma unroll
  for (int c = 0; c < R; ++c) accm0[c] = accm1[c] = 0.0;
  for (int64_t g0 = 0; g0 < ngroups; g0 += PM_THREADS) {
    // which of the next 256 groups can hold a point within the cut-off of any of our test points?
    const int64_t g = g0 + tid;
    bool active = false;
    if (g < ngroups) {
      const double tx0 = boxes[4 * g + 0], tx1 = boxes[4 * g + 1], ty0 = boxes[4 * g + 2], ty1 = boxes[4 * g + 3];
      const double gx = fmax(0.0, fmax(tx0 - bx1, bx0 - tx1));
      const double gy = fmax(0.0, fmax(ty0 - by1, by0 - ty1));
      active = !(gx * gx + gy * gy > r2cut);
    }
    const unsigned bal = __ballot_sync(0xffffffffu, active);
    __syncthreads();                      // previous list fully consumed
    if (lane == 0) wcount[warp] = __popc(bal);
    __syncthreads();
    int base = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const int c = wcount[w];
      if (w < warp) base += c;
      total += c;
    }
    if (active) list[base + __popc(bal & ((1u << lane) - 1u))] = (int)tid;   // ascending group order
    for (int li = 0; li < total; ++li) {
      __syncthreads();                    // list visible / previous tile consumed
      const int64_t n0 = (g0 + list[li]) * PG;
      if (tid < PG) {
        const int64_t n = n0 + tid;
        const bool ok = n < N;
        double2 p;
        p.x = ok ? X[n * prof.desc.ndim] : 0.0;
        p.y = (ok && prof.desc.ndim == 2) ? X[n * 2 + 1] : 0.0;
        pxy[tid] = p;
        if constexpr (R == 1) {
          pa[tid] = ok ? prof.weight() * alpha[n] : 0.0;
        } else {
#pragma unroll
          for (int c = 0; c < R; ++c)
            pa[tid * R + c] = (ok && c < prof.nrhs) ? prof.weight() * alpha[n * prof.nrhs + c] : 0.0;
        }
      }
      __syncthreads();
      if constexpr (R > 1) {
        for (int i = 0; i < PG; i += 2) prof.mean2_multi(sx, sy, pxy, pa, i, phi_s, accm0, accm1);
      } else if constexpr (P::kSum) {
        for (int i = 0; i < PG; i += 2) prof.mean2(sx, sy, pxy, pa, i, phi_s, acc0, acc1);
      } else {
#pragma unroll 2
        for (int i = 0; i < PG; i += 2) {
          const double2 p0 = pxy[i], p1 = pxy[i + 1];
          const double q0 = tgp_qform(prof.desc, sx - p0.x, sy - p0.y);
          const double q1 = tgp_qform(prof.desc, sx - p1.x, sy - p1.y);
          acc0 = fma(tgp_profile<P::kFam>(q0, phi_s), pa[i], acc0);
          acc1 = fma(tgp_profile<P::kFam>(q1, phi_s), pa[i + 1], acc1);
        }
      }
    }
  }
  if constexpr (R == 1) {
    if (live) mean[m] = acc0 + acc1;
  } else {
#pragma unroll
    for (int c = 0; c < R; ++c)
      if (live && c < prof.nrhs) mean[m * prof.nrhs + c] = accm0[c] + accm1[c];
  }
}

// smallest eigenvalue of the inverse metric: q >= lmin |delta|^2
static double metric_lmin(const tgp_kernel* k) {
  double lmin = k->m00;
  if (k->ndim == 2) {
    const double h = 0.5 * (k->m00 - k->m11);
    lmin = 0.5 * (k->m00 + k->m11) - sqrt(h * h + k->m01 * k->m01);
  }
  return lmin;
}

// r2cut: squared Euclidean distance beyond which every pair is below the cut-off (caller: > 0)
template <class P>
static int predict_mean_trunc_launch(const double* Xs, int64_t M, const double* X, int64_t N, const P& prof,
                                     double r2cut, const double* alpha, double* mean, double* work, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t ngroups = tgp_cdiv(N, PG);
  point_boxes_kernel<<<(unsigned)tgp_cdiv(ngroups, 8), 256, 0, st>>>(X, N, prof.desc.ndim, work, ngroups);
  TGP_LAUNCH_CHECK();
  const double* phi = tgp_phi_device();
  const int64_t gx = tgp_cdiv(M, PM_THREADS);
  TGP_CHECK_ARG(gx < (1ll << 31), "M too large for one launch");
  predict_mean_trunc_kernel<P><<<(unsigned)gx, PM_THREADS, 0, st>>>(Xs, M, X, N, prof, alpha, mean, phi, work,
                                                                      ngroups, r2cut);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

static int predict_mean_trunc_args(const double* Xs, int64_t M, const double* X, int64_t N, const double* alpha,
                                   double* mean, double* work, void* stream) {
  TGP_CHECK_ARG(M >= 0 && N >= 0, "M/N");
  if (M == 0) return TGP_OK;
  TGP_CHECK_ARG(Xs && mean && (N == 0 || (X && alpha && work)), "null pointer");
  if (N == 0) TGP_CUDA(cudaMemsetAsync(mean, 0, M * sizeof(double), (cudaStream_t)stream));
  return TGP_OK;
}

extern "C" int tgp_predict_mean_trunc(const double* Xs, int64_t M, const double* X, int64_t N,
                                      const tgp_kernel* k, const double* alpha, double* mean, double* work,
                                      void* stream) {
  TGP_CHECK_ARG(kdesc_ok(k), "kernel descriptor");
  const int rc = predict_mean_trunc_args(Xs, M, X, N, alpha, mean, work, stream);
  if (rc || M == 0 || N == 0) return rc;
  const double lmin = metric_lmin(k);
  TGP_CHECK_ARG(lmin > 0.0, "inverse metric must be positive definite");
  const double r2cut = profile_qcut(k->family) / lmin;
  const KDesc kd = make_kdesc(k);
  TGP_FAMILY_SWITCH(k->family, return predict_mean_trunc_launch(Xs, M, X, N, FamilyProfile<FAM>{kd}, r2cut, alpha,
                                                                mean, work, stream));
  return TGP_OK;
}

// A group is skipped only when it is beyond the cut-off of every term: the union of the supports is the largest
// per-term qcut_c / lmin(M_c).  Each skipped pair is below 1e-40 |amp_c| for every term, so the mean changes by at
// most 1e-40 sum_c |amp_c| sum_n |alpha_n|.
extern "C" int tgp_predict_mean_trunc_sum(const double* Xs, int64_t M, const double* X, int64_t N,
                                          const tgp_kernel_sum* k, const double* alpha, double* mean, double* work,
                                          void* stream) {
  TGP_CHECK_ARG(ksum_ok(k), "kernel sum descriptor");
  if (k->nterms == 1) return tgp_predict_mean_trunc(Xs, M, X, N, &k->term[0], alpha, mean, work, stream);
  const int rc = predict_mean_trunc_args(Xs, M, X, N, alpha, mean, work, stream);
  if (rc || M == 0 || N == 0) return rc;
  double r2cut = 0.0;
  for (int c = 0; c < k->nterms; ++c) {
    const double lmin = metric_lmin(&k->term[c]);
    TGP_CHECK_ARG(lmin > 0.0, "inverse metric must be positive definite");
    const double r2 = profile_qcut(k->term[c].family) / lmin;
    if (r2 > r2cut) r2cut = r2;
  }
  return predict_mean_trunc_launch(Xs, M, X, N, SumProfile{make_ksumdesc(k)}, r2cut, alpha, mean, work, stream);
}

// ---- several outputs ----------------------------------------------------------------------------------------------
// r is padded to R = 2, 4 or 8 accumulator columns; a one-term sum without white uses the single-term profile.
template <int R, class Q>
static int mean_multi_launch_r(const double* Xs, int64_t M, const double* X, int64_t N, const Q& prof, int r,
                               double r2cut, const double* alpha, double* mean, double* work, void* stream) {
  const MultiOut<Q, R> mp{prof, r};
  if (work) return predict_mean_trunc_launch(Xs, M, X, N, mp, r2cut, alpha, mean, work, stream);
  return predict_mean_launch(Xs, M, X, N, mp, alpha, mean, stream);
}

template <class Q>
static int mean_multi_launch(const double* Xs, int64_t M, const double* X, int64_t N, const Q& prof, int r,
                             double r2cut, const double* alpha, double* mean, double* work, void* stream) {
  if (r <= 2) return mean_multi_launch_r<2>(Xs, M, X, N, prof, r, r2cut, alpha, mean, work, stream);
  if (r <= 4) return mean_multi_launch_r<4>(Xs, M, X, N, prof, r, r2cut, alpha, mean, work, stream);
  return mean_multi_launch_r<8>(Xs, M, X, N, prof, r, r2cut, alpha, mean, work, stream);
}

// work == nullptr: the full sum; otherwise the truncated one with the cut-off of tgp_predict_mean_trunc_sum
static int predict_mean_multi_impl(const double* Xs, int64_t M, const double* X, int64_t N, const tgp_kernel_sum* k,
                                   const double* alpha, int r, double* mean, double* work, void* stream) {
  TGP_CHECK_ARG(r >= 1 && r <= TGP_MAX_RHS, "number of outputs must be 1 .. TGP_MAX_RHS");
  TGP_CHECK_ARG(ksum_ok(k), "kernel sum descriptor");
  if (r == 1)   // (N, 1) and (M, 1) are vectors: the single-output entries, bit for bit
    return work ? tgp_predict_mean_trunc_sum(Xs, M, X, N, k, alpha, mean, work, stream)
                : tgp_predict_mean_sum(Xs, M, X, N, k, alpha, mean, stream);
  TGP_CHECK_ARG(M >= 0 && N >= 0, "M/N");
  if (M == 0) return TGP_OK;
  TGP_CHECK_ARG(Xs && mean && (N == 0 || (X && alpha)), "null pointer");
  if (N == 0) {
    TGP_CUDA(cudaMemsetAsync(mean, 0, M * r * sizeof(double), (cudaStream_t)stream));
    return TGP_OK;
  }
  double r2cut = 0.0;
  if (work) {
    for (int c = 0; c < k->nterms; ++c) {
      const double lmin = metric_lmin(&k->term[c]);
      TGP_CHECK_ARG(lmin > 0.0, "inverse metric must be positive definite");
      const double r2 = profile_qcut(k->term[c].family) / lmin;
      if (r2 > r2cut) r2cut = r2;
    }
  }
  if (k->nterms == 1) {
    const KDesc kd = make_kdesc(&k->term[0]);
    TGP_FAMILY_SWITCH(k->term[0].family, return mean_multi_launch(Xs, M, X, N, FamilyProfile<FAM>{kd}, r, r2cut, alpha,
                                                                  mean, work, stream));
    return TGP_OK;
  }
  return mean_multi_launch(Xs, M, X, N, SumProfile{make_ksumdesc(k)}, r, r2cut, alpha, mean, work, stream);
}

extern "C" int tgp_predict_mean_multi(const double* Xs, int64_t M, const double* X, int64_t N, const tgp_kernel_sum* k,
                                      const double* alpha, int32_t r, double* mean, void* stream) {
  return predict_mean_multi_impl(Xs, M, X, N, k, alpha, r, mean, nullptr, stream);
}

extern "C" int tgp_predict_mean_trunc_multi(const double* Xs, int64_t M, const double* X, int64_t N,
                                            const tgp_kernel_sum* k, const double* alpha, int32_t r, double* mean,
                                            double* work, void* stream) {
  TGP_CHECK_ARG(work != nullptr || M == 0 || N == 0, "work");
  return predict_mean_multi_impl(Xs, M, X, N, k, alpha, r, mean, work, stream);
}

// var[m] = amp - sum_n V[m][n]^2, V = K(Xs, X) L^-T (row m = L^-1 k*_m).  Warp per row.
__global__ void __launch_bounds__(256)
var_from_rows_kernel(const double* __restrict__ V, int64_t M, int64_t N, int64_t ldv, double amp,
                     double* __restrict__ var) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t m = (int64_t)blockIdx.x * 8 + warp;
  if (m >= M) return;
  const double* row = V + m * ldv;
  double s0 = 0.0, s1 = 0.0;
  int64_t n = lane;
  for (; n + 32 < N; n += 64) {
    const double a = row[n], b = row[n + 32];
    s0 = fma(a, a, s0);
    s1 = fma(b, b, s1);
  }
  if (n < N) { const double a = row[n]; s0 = fma(a, a, s0); }
  double s = s0 + s1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) var[m] = amp - s;
}

// k or ks (the other NULL): single-term or sum kernel; the prior variance is amp, or sum_c amp_c + white
static int predict_var_impl(const double* Xs, int64_t M, const double* X, int64_t N,
                            const tgp_kernel* k, const tgp_kernel_sum* ks, const double* L, int64_t ld,
                            const int64_t* row_end, int64_t nblocks, double* work, int64_t chunk, double* var,
                            void* stream) {
  if (ks) TGP_CHECK_ARG(ksum_ok(ks), "kernel sum descriptor");
  else TGP_CHECK_ARG(kdesc_ok(k), "kernel descriptor");
  TGP_CHECK_ARG(M >= 0 && N > 0 && ld >= N && chunk > 0, "shape");
  if (M == 0) return TGP_OK;
  TGP_CHECK_ARG(Xs && X && L && work && var, "null pointer");
  const int64_t ldw = (N + 1) & ~1ll;  // even row pitch for the DMMA operand loads
  TGP_CHECK_ARG(((uintptr_t)work % 16) == 0, "work must be 16-byte aligned");
  const int ndim = ks ? ks->ndim : k->ndim;
  double prior = ks ? ks->white : k->amp;
  if (ks)
    for (int c = 0; c < ks->nterms; ++c) prior += ks->term[c].amp;
  for (int64_t m0 = 0; m0 < M; m0 += chunk) {
    const int64_t mc = (M - m0 < chunk) ? (M - m0) : chunk;
    int rc = ks ? tgp_kmat_cross_sum(Xs + m0 * ndim, mc, X, N, ks, work, ldw, stream)
                : tgp_kmat_cross(Xs + m0 * ndim, mc, X, N, k, work, ldw, stream);
    if (rc) return rc;
    rc = row_end ? tgp_trsm_rows_env(L, N, ld, row_end, nblocks, work, mc, ldw, stream)
                 : tgp_trsm_rows(L, N, ld, work, mc, ldw, stream);
    if (rc) return rc;
    var_from_rows_kernel<<<(unsigned)tgp_cdiv(mc, 8), 256, 0, (cudaStream_t)stream>>>(work, mc, N, ldw, prior,
                                                                                      var + m0);
    TGP_LAUNCH_CHECK();
  }
  return TGP_OK;
}

extern "C" int tgp_predict_var(const double* Xs, int64_t M, const double* X, int64_t N,
                               const tgp_kernel* k, const double* L, int64_t ld, double* work,
                               int64_t chunk, double* var, void* stream) {
  return predict_var_impl(Xs, M, X, N, k, nullptr, L, ld, nullptr, 0, work, chunk, var, stream);
}

// The same with a factor whose envelope is known (tgp_potrf_env): the multi-right-hand-side forward substitution
// only propagates every solved block of unknowns to the rows inside the envelope.
extern "C" int tgp_predict_var_env(const double* Xs, int64_t M, const double* X, int64_t N,
                                   const tgp_kernel* k, const double* L, int64_t ld, const int64_t* row_end,
                                   int64_t nblocks, double* work, int64_t chunk, double* var, void* stream) {
  TGP_CHECK_ARG(row_end != nullptr, "row_end");
  return predict_var_impl(Xs, M, X, N, k, nullptr, L, ld, row_end, nblocks, work, chunk, var, stream);
}

extern "C" int tgp_predict_var_sum(const double* Xs, int64_t M, const double* X, int64_t N, const tgp_kernel_sum* k,
                                   const double* L, int64_t ld, const int64_t* row_end, int64_t nblocks, double* work,
                                   int64_t chunk, double* var, void* stream) {
  TGP_CHECK_ARG(k != nullptr, "kernel sum descriptor");
  return predict_var_impl(Xs, M, X, N, nullptr, k, L, ld, row_end, nblocks, work, chunk, var, stream);
}

// ---------------------------------------------------------------------------------------------
// Mean-function lookup: uniform mean of the k nearest points of the meanify grid.
// Replaces sklearn's KNeighborsRegressor(n_neighbors).fit(X0, y0).predict(X) at
// /root/reference/treegp/gp_interp.py:236-238 (SURVEY section 8f-1: with the GP algebra on the device this
// KD-tree query of every training / test point is the host-side tail of predict()).  The grid is small
// (a few thousand points), so every query scans all of it: thread per query, grid tiles broadcast from
// shared memory, the K best kept sorted in registers.  Distances are squared Euclidean in FP64; exact ties
// are resolved towards the lower grid index (sklearn's KD-tree leaves them unspecified); the values are
// summed in order of increasing distance, as numpy.mean does over sklearn's sorted neighbour list.
// ---------------------------------------------------------------------------------------------
constexpr int KNN_TILE = 1024;
template <int K>
__global__ void __launch_bounds__(256)
knn_mean_kernel(const double* __restrict__ Xq, int64_t M, const double* __restrict__ X0,
                const double* __restrict__ y0, int64_t n0, int ndim, int k, double* __restrict__ out) {
  __shared__ double2 gxy[KNN_TILE];
  __shared__ double gv[KNN_TILE];
  const int tid = threadIdx.x;
  const int64_t m = (int64_t)blockIdx.x * 256 + tid;
  const bool live = m < M;
  const double qx = live ? Xq[m * ndim] : 0.0;
  const double qy = (live && ndim == 2) ? Xq[m * 2 + 1] : 0.0;
  double bd[K], bv[K];
#pragma unroll
  for (int j = 0; j < K; ++j) { bd[j] = INFINITY; bv[j] = 0.0; }
  for (int64_t n00 = 0; n00 < n0; n00 += KNN_TILE) {
    __syncthreads();
    for (int i = tid; i < KNN_TILE; i += 256) {
      const int64_t n = n00 + i;
      const bool ok = n < n0;
      gxy[i] = make_double2(ok ? X0[n * ndim] : INFINITY, (ok && ndim == 2) ? X0[n * 2 + 1] : 0.0);
      gv[i] = ok ? y0[n] : 0.0;
    }
    __syncthreads();
    const int cnt = (int)((n0 - n00 < KNN_TILE) ? (n0 - n00) : KNN_TILE);
    for (int i = 0; i < cnt; ++i) {
      const double2 p = gxy[i];
      const double dx = p.x - qx, dy = p.y - qy;
      double d = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
      if (d < bd[K - 1]) {       // strict: an equal distance later in index order does not displace an earlier one
        double v = gv[i];
#pragma unroll
        for (int j = 0; j < K; ++j) {   // insertion into the ascending list, stable for ties
          if (d < bd[j]) {
            const double td = bd[j], tv = bv[j];
            bd[j] = d; bv[j] = v;
            d = td; v = tv;
          }
        }
      }
    }
  }
  if (live) {
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < K; ++j)
      if (j < k) s += bv[j];
    out[m] = s / (double)k;
  }
}

// Any k (n_neighbors > 32): selection by k passes over the grid -- pass t picks the smallest (distance, index) pair
// that is lexicographically greater than the one picked in pass t - 1.  O(k n0) per query, no per-thread list; the
// same neighbours, the same order of summation and the same tie rule as the register-list kernel.
__global__ void __launch_bounds__(256)
knn_mean_passes_kernel(const double* __restrict__ Xq, int64_t M, const double* __restrict__ X0,
                       const double* __restrict__ y0, int64_t n0, int ndim, int k, double* __restrict__ out) {
  const int64_t m = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (m >= M) return;
  const double qx = Xq[m * ndim];
  const double qy = (ndim == 2) ? Xq[m * 2 + 1] : 0.0;
  double pd = -1.0, s = 0.0;
  int64_t pi = -1;
  for (int t = 0; t < k; ++t) {
    double bd = INFINITY;
    int64_t bi = -1;
    for (int64_t n = 0; n < n0; ++n) {
      const double dx = X0[n * ndim] - qx, dy = ((ndim == 2) ? X0[n * 2 + 1] : 0.0) - qy;
      const double d = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
      const bool after_prev = (d > pd) || (d == pd && n > pi);
      if (after_prev && d < bd) { bd = d; bi = n; }   // first index wins among equal distances
    }
    if (bi < 0) break;
    s += y0[bi];
    pd = bd;
    pi = bi;
  }
  out[m] = s / (double)k;
}

extern "C" int tgp_knn_mean(const double* Xq, int64_t M, const double* X0, const double* y0, int64_t n0,
                            int32_t ndim, int32_t k, double* out, void* stream) {
  TGP_CHECK_ARG(M >= 0 && n0 >= 1 && (ndim == 1 || ndim == 2), "M/n0/ndim");
  TGP_CHECK_ARG(k >= 1 && k <= n0, "need 1 <= n_neighbors <= number of grid points");
  if (M == 0) return TGP_OK;
  TGP_CHECK_ARG(Xq && X0 && y0 && out, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)tgp_cdiv(M, 256);
  // K = list length compiled in (entries beyond k stay +inf and are never summed... they are: cap by j < k)
  if (k <= 4) knn_mean_kernel<4><<<grid, 256, 0, st>>>(Xq, M, X0, y0, n0, ndim, k, out);
  else if (k <= 8) knn_mean_kernel<8><<<grid, 256, 0, st>>>(Xq, M, X0, y0, n0, ndim, k, out);
  else if (k <= 16) knn_mean_kernel<16><<<grid, 256, 0, st>>>(Xq, M, X0, y0, n0, ndim, k, out);
  else if (k <= 32) knn_mean_kernel<32><<<grid, 256, 0, st>>>(Xq, M, X0, y0, n0, ndim, k, out);
  else knn_mean_passes_kernel<<<grid, 256, 0, st>>>(Xq, M, X0, y0, n0, ndim, k, out);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}
