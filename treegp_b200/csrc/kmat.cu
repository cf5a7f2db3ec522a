// Covariance-matrix construction: K(X,X) + diag, K(Xs,X).
//
// Replaces the pdist/cdist + exp / scipy.special.kv + squareform pipelines of
// /root/reference/treegp/kernels.py:114-126 (AnisotropicRBF), :251-277 (VonKarman),
// :358-381 (AnisotropicVonKarman) and sklearn RBF/Matern reached through eval_kernel
// (kernels.py:17-59), plus the `+ np.eye(N) * y_err**2` of gp_interp.py:180 / log_likelihood.py:29.
//
// Design (B200): the build is store-bound for RBF (8 N^2 bytes) and FP64-ALU-bound for von Karman,
// so the symmetric kernel evaluates each off-diagonal 64x64 tile ONCE and writes it twice: directly
// (16-byte st.global.v2.f64, 512 B per warp-row) and transposed through a padded shared-memory
// tile.  Coordinates of the row/column tiles are staged in shared memory; the von Karman table
// lives in shared memory as well.  `lower_only` drops the mirrored write when the consumer is the
// Cholesky (halves HBM traffic).
#include <stdarg.h>
#include <string.h>
#include "tgp_common.cuh"
#include "profile_policy.cuh"
#include "batch.cuh"

// ---- error state / misc host helpers --------------------------------------------------------
static thread_local char g_err[512] = "";
void tgp_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}
extern "C" const char* tgp_last_error(void) { return g_err; }
extern "C" int tgp_abi_version(void) { return TGP_ABI_VERSION; }

int tgp_num_sms() {
  static int sms[TGP_MAX_DEVICES] = {};
  const int dev = tgp_current_device();
  if (!sms[dev]) {
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    sms[dev] = v > 0 ? v : 148;
  }
  return sms[dev];
}

__device__ const double g_vk_phi_dev[TGP_VK_PHI_SIZE] = TGP_VK_PHI_TABLE;
const double* tgp_phi_device() {
  static const double* p[TGP_MAX_DEVICES] = {};
  const int dev = tgp_current_device();
  if (!p[dev]) {
    void* q = nullptr;
    if (cudaGetSymbolAddress(&q, g_vk_phi_dev) == cudaSuccess) p[dev] = (const double*)q;
  }
  return p[dev];
}

// ---- kernels -----------------------------------------------------------------------------------
constexpr int KT = 64;          // tile edge
constexpr int KT_THREADS = 256; // 8 warps; lane -> 2 adjacent columns, warp -> rows w, w+8, ...
constexpr int KT_PITCH = KT + 1;

__device__ __forceinline__ void store2(double* p, double a, double b, bool vec, bool ok0, bool ok1) {
  if (vec && ok1) {
    double2 v = make_double2(a, b);
    *reinterpret_cast<double2*>(p) = v;
  } else {
    if (ok0) p[0] = a;
    if (ok1) p[1] = b;
  }
}

// Symmetric build of the lower-triangular tile pair number t (I >= J, linearised).
template <class P>
__device__ __forceinline__ void kmat_sym_tile(const double* __restrict__ X, int64_t N, const P& prof,
                                              const double* __restrict__ diag_add, double* __restrict__ out,
                                              int64_t ld, int lower_only, int vec_ok,
                                              const double* __restrict__ phi_g, const int64_t t) {
  __shared__ double xr[KT], yr[KT], xc[KT], yc[KT];
  __shared__ double tile[KT * KT_PITCH];
  __shared__ double phi_s[P::kPhiSize];

  // linear tile id -> (I, J), I >= J
  int64_t I = (int64_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while (I * (I + 1) / 2 > t) --I;
  while ((I + 1) * (I + 2) / 2 <= t) ++I;
  const int64_t J = t - I * (I + 1) / 2;
  const int64_t r0 = I * KT, c0 = J * KT;
  const int tid = threadIdx.x;

  if (prof.stage_phi()) tgp_stage_phi(phi_s, phi_g);
  if (tid < KT) {
    const int64_t r = r0 + tid;
    const bool ok = r < N;
    xr[tid] = ok ? X[r * prof.desc.ndim] : 0.0;
    yr[tid] = (ok && prof.desc.ndim == 2) ? X[r * 2 + 1] : 0.0;
  } else if (tid < 2 * KT) {
    const int l = tid - KT;
    const int64_t c = c0 + l;
    const bool ok = c < N;
    xc[l] = ok ? X[c * prof.desc.ndim] : 0.0;
    yc[l] = (ok && prof.desc.ndim == 2) ? X[c * 2 + 1] : 0.0;
  }
  __syncthreads();

  const int lane = tid & 31, warp = tid >> 5;
  const int cl = 2 * lane;
  const double cx0 = xc[cl], cy0 = yc[cl], cx1 = xc[cl + 1], cy1 = yc[cl + 1];
  const int64_t cg = c0 + cl;
  const bool diag_tile = (I == J);
  const bool mirror = !diag_tile && !lower_only;

  // von Karman: the profile (series / per-binade polynomial, sqrt, cbrt, exp) is ~350 instructions per evaluation;
  // unrolled 8 x 2 times the kernel was 94 KB of SASS and stalled on instruction fetch (no_instruction 4.4 per
  // issue, profiles/r2_start_kmat_vk.ncu.txt) -- two rows per trip keep it inside the instruction cache
#pragma unroll(P::kHeavy ? 2 : KT / 8)
  for (int rr = 0; rr < KT / 8; ++rr) {
    const int rl = warp + 8 * rr;
    const int64_t rg = r0 + rl;
    const double rx = xr[rl], ry = yr[rl];
    double v0, v1;
    prof.sym2(rx, ry, cx0, cy0, cx1, cy1, rg, cg, phi_s, v0, v1);
    if (diag_tile && diag_add != nullptr) {
      if (rg == cg && rg < N) v0 += diag_add[rg];
      if (rg == cg + 1 && rg < N) v1 += diag_add[rg];
    }
    if (mirror) {
      tile[rl * KT_PITCH + cl] = v0;
      tile[rl * KT_PITCH + cl + 1] = v1;
    }
    if (rg < N) {
      bool ok0 = cg < N, ok1 = cg + 1 < N;
      if (lower_only && diag_tile) {  // keep j <= i only
        ok0 = ok0 && (cg <= rg);
        ok1 = ok1 && (cg + 1 <= rg);
      }
      store2(out + rg * ld + cg, v0, v1, vec_ok && ok0, ok0, ok1);
    }
  }
  if (mirror) {
    __syncthreads();
    // transposed write: out[c0 + c][r0 + r] = tile[r][c]; warp w handles c = w, w+8, ...;
    // lane l reads tile[l][c] and tile[l+32][c] (odd pitch: conflict-free per half-warp).
#pragma unroll
    for (int cc = 0; cc < KT / 8; ++cc) {
      const int c = warp + 8 * cc;
      const int64_t orow = c0 + c;
      if (orow >= N) continue;
      const double a = tile[lane * KT_PITCH + c];
      const double b = tile[(lane + 32) * KT_PITCH + c];
      double* dst = out + orow * ld + r0;
      if (r0 + lane < N) dst[lane] = a;
      if (r0 + lane + 32 < N) dst[lane + 32] = b;
    }
  }
}

// Grid: one CTA per lower-triangular tile pair.
template <class P>
__global__ void __launch_bounds__(KT_THREADS)
kmat_sym_kernel(const double* __restrict__ X, int64_t N, P prof, const double* __restrict__ diag_add,
                double* __restrict__ out, int64_t ld, int lower_only, int vec_ok,
                const double* __restrict__ phi_g) {
  kmat_sym_tile(X, N, prof, diag_add, out, ld, lower_only, vec_ok, phi_g, (int64_t)blockIdx.x);
}

// Rectangular build K(Xs, X): rows = test points, columns = training points.
template <class P>
__global__ void __launch_bounds__(KT_THREADS)
kmat_cross_kernel(const double* __restrict__ Xs, int64_t M, const double* __restrict__ X, int64_t N,
                  P prof, double* __restrict__ out, int64_t ld, int vec_ok,
                  const double* __restrict__ phi_g) {
  __shared__ double xr[KT], yr[KT], xc[KT], yc[KT];
  __shared__ double phi_s[P::kPhiSize];
  const int64_t r0 = (int64_t)blockIdx.x * KT, c0 = (int64_t)blockIdx.y * KT;
  const int tid = threadIdx.x;
  if (prof.stage_phi()) tgp_stage_phi(phi_s, phi_g);
  if (tid < KT) {
    const int64_t r = r0 + tid;
    const bool ok = r < M;
    xr[tid] = ok ? Xs[r * prof.desc.ndim] : 0.0;
    yr[tid] = (ok && prof.desc.ndim == 2) ? Xs[r * 2 + 1] : 0.0;
  } else if (tid < 2 * KT) {
    const int l = tid - KT;
    const int64_t c = c0 + l;
    const bool ok = c < N;
    xc[l] = ok ? X[c * prof.desc.ndim] : 0.0;
    yc[l] = (ok && prof.desc.ndim == 2) ? X[c * 2 + 1] : 0.0;
  }
  __syncthreads();
  const int lane = tid & 31, warp = tid >> 5;
  const int cl = 2 * lane;
  const double cx0 = xc[cl], cy0 = yc[cl], cx1 = xc[cl + 1], cy1 = yc[cl + 1];
  const int64_t cg = c0 + cl;
#pragma unroll(P::kHeavy ? 2 : KT / 8)
  for (int rr = 0; rr < KT / 8; ++rr) {
    const int rl = warp + 8 * rr;
    const int64_t rg = r0 + rl;
    if (rg >= M) continue;
    const double rx = xr[rl], ry = yr[rl];
    double v0, v1;
    prof.cross2(rx, ry, cx0, cy0, cx1, cy1, phi_s, v0, v1);
    const bool ok0 = cg < N, ok1 = cg + 1 < N;
    store2(out + rg * ld + cg, v0, v1, vec_ok && ok0, ok0, ok1);
  }
}

// ---- C ABI -----------------------------------------------------------------------------------
extern "C" int tgp_kmat_sym(const double* X, int64_t N, const tgp_kernel* k, const double* diag_add,
                            double* out, int64_t ld, int lower_only, void* stream) {
  TGP_CHECK_ARG(kdesc_ok(k), "kernel descriptor");
  TGP_CHECK_ARG(N >= 0 && ld >= N, "N/ld");
  if (N == 0) return TGP_OK;
  TGP_CHECK_ARG(X && out, "null pointer");
  const KDesc kd = make_kdesc(k);
  const int64_t nt = tgp_cdiv(N, KT);
  const int64_t ntiles = nt * (nt + 1) / 2;
  TGP_CHECK_ARG(ntiles < (1ll << 31), "matrix too large for one launch");
  const int vec_ok = (ld % 2 == 0) && (((uintptr_t)out & 15) == 0);
  cudaStream_t st = (cudaStream_t)stream;
  const double* phi = tgp_phi_device();
  TGP_FAMILY_SWITCH(k->family, (kmat_sym_kernel<FamilyProfile<FAM>><<<(unsigned)ntiles, KT_THREADS, 0, st>>>(
                                   X, N, FamilyProfile<FAM>{kd}, diag_add, out, ld, lower_only, vec_ok, phi)));
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

extern "C" int tgp_kmat_cross(const double* Xs, int64_t M, const double* X, int64_t N,
                              const tgp_kernel* k, double* out, int64_t ld, void* stream) {
  TGP_CHECK_ARG(kdesc_ok(k), "kernel descriptor");
  TGP_CHECK_ARG(M >= 0 && N >= 0 && ld >= N, "M/N/ld");
  if (M == 0 || N == 0) return TGP_OK;
  TGP_CHECK_ARG(Xs && X && out, "null pointer");
  const KDesc kd = make_kdesc(k);
  const int vec_ok = (ld % 2 == 0) && (((uintptr_t)out & 15) == 0);
  dim3 grid((unsigned)tgp_cdiv(M, KT), (unsigned)tgp_cdiv(N, KT));  // x: row tiles (M may be millions)
  TGP_CHECK_ARG(grid.y <= 65535u, "N too large for one launch");
  cudaStream_t st = (cudaStream_t)stream;
  const double* phi = tgp_phi_device();
  TGP_FAMILY_SWITCH(k->family, (kmat_cross_kernel<FamilyProfile<FAM>><<<grid, KT_THREADS, 0, st>>>(
                                   Xs, M, X, N, FamilyProfile<FAM>{kd}, out, ld, vec_ok, phi)));
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

extern "C" int tgp_kmat_sym_sum(const double* X, int64_t N, const tgp_kernel_sum* k, const double* diag_add,
                                double* out, int64_t ld, int lower_only, void* stream) {
  TGP_CHECK_ARG(ksum_ok(k), "kernel sum descriptor");
  if (k->nterms == 1 && k->white == 0.0)   // one term: the single-term kernel, bit for bit
    return tgp_kmat_sym(X, N, &k->term[0], diag_add, out, ld, lower_only, stream);
  TGP_CHECK_ARG(N >= 0 && ld >= N, "N/ld");
  if (N == 0) return TGP_OK;
  TGP_CHECK_ARG(X && out, "null pointer");
  const int64_t nt = tgp_cdiv(N, KT);
  const int64_t ntiles = nt * (nt + 1) / 2;
  TGP_CHECK_ARG(ntiles < (1ll << 31), "matrix too large for one launch");
  const int vec_ok = (ld % 2 == 0) && (((uintptr_t)out & 15) == 0);
  kmat_sym_kernel<SumProfile><<<(unsigned)ntiles, KT_THREADS, 0, (cudaStream_t)stream>>>(
      X, N, SumProfile{make_ksumdesc(k)}, diag_add, out, ld, lower_only, vec_ok, tgp_phi_device());
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

extern "C" int tgp_kmat_cross_sum(const double* Xs, int64_t M, const double* X, int64_t N,
                                  const tgp_kernel_sum* k, double* out, int64_t ld, void* stream) {
  TGP_CHECK_ARG(ksum_ok(k), "kernel sum descriptor");
  if (k->nterms == 1) return tgp_kmat_cross(Xs, M, X, N, &k->term[0], out, ld, stream);   // no white in K(Xs, X)
  TGP_CHECK_ARG(M >= 0 && N >= 0 && ld >= N, "M/N/ld");
  if (M == 0 || N == 0) return TGP_OK;
  TGP_CHECK_ARG(Xs && X && out, "null pointer");
  const int vec_ok = (ld % 2 == 0) && (((uintptr_t)out & 15) == 0);
  dim3 grid((unsigned)tgp_cdiv(M, KT), (unsigned)tgp_cdiv(N, KT));
  TGP_CHECK_ARG(grid.y <= 65535u, "N too large for one launch");
  kmat_cross_kernel<SumProfile><<<grid, KT_THREADS, 0, (cudaStream_t)stream>>>(
      Xs, M, X, N, SumProfile{make_ksumdesc(k)}, out, ld, vec_ok, tgp_phi_device());
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

// ---- batches of independent problems (tgp_loglike_batch) ---------------------------------------------------------
// K(X_b, X_b) + diag(yerr2_b), lower triangle, into problem b's block of the batch workspace.  Grid: (problems of
// this profile class, tiles of the largest of them); each CTA runs the tile body of the single build with the
// problem's descriptor, so every problem gets the single call's matrix bit for bit.
template <class P>
__global__ void __launch_bounds__(KT_THREADS)
kmat_sym_batch_kernel(const TgpBatchProb* __restrict__ pr, const KSumDesc* __restrict__ kd,
                      const int32_t* __restrict__ list, const double* __restrict__ phi_g) {
  const int b = list[blockIdx.x];
  const int64_t N = pr[b].N, nt = (N + KT - 1) / KT;
  if ((int64_t)blockIdx.y >= nt * (nt + 1) / 2) return;
  const P prof = tgp_batch_profile<P>(kd[b]);
  kmat_sym_tile(pr[b].X, N, prof, pr[b].yerr2, pr[b].A, pr[b].ld, /*lower_only=*/1, /*vec_ok=*/1, phi_g,
                (int64_t)blockIdx.y);
}

int tgp_batch_kmat_sym(const TgpBatchProb* pr, const KSumDesc* kd, const int32_t* list, int32_t count, int cls,
                       int64_t max_n, cudaStream_t st) {
  const int64_t nt = tgp_cdiv(max_n, KT);
  const dim3 grid((unsigned)count, (unsigned)(nt * (nt + 1) / 2));
  const double* phi = tgp_phi_device();
  if (cls == TGP_BATCH_SUM) {
    kmat_sym_batch_kernel<SumProfile><<<grid, KT_THREADS, 0, st>>>(pr, kd, list, phi);
  } else {
    TGP_FAMILY_SWITCH(cls, (kmat_sym_batch_kernel<FamilyProfile<FAM>><<<grid, KT_THREADS, 0, st>>>(pr, kd, list, phi)));
  }
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}
