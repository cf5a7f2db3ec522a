// FP64 dense linear algebra for the GP solve: blocked right-looking Cholesky, triangular solves,
// log-determinant and the marginal log-likelihood.
//
// Replaces scipy.linalg.cholesky / cho_solve / np.dot at
//   /root/reference/treegp/gp_interp.py:181-191 and /root/reference/treegp/log_likelihood.py:29-37.
//
// Layout: row-major, lower triangle (numpy's default layout for K, `lower=True` factor).
//
// Everything O(N^3) funnels into ONE contraction kernel, gemm_nt_sub (C -= A * B^T with both
// operands K-contiguous), which runs on the FP64 tensor pipe via mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4;
// there is no tcgen05/TMEM path for FP64 -- larger PTX shapes lower to the same DMMA.8x8x4).
//   * Cholesky trailing update      A22 -= L21 L21^T            (lower tiles only)
//   * panel / multi-RHS solves      B2  -= B1  L21^T
//   * predictive covariance         C   -= V   V^T
// Operand tiles are brought in by a 4-stage cp.async ring into XOR-swizzled shared memory so the
// fragment loads are conflict-free 16-byte LDS; the K order inside a 16-wide stage is permuted
// (even k's then odd k's) so one LDS.128 feeds two DMMAs.
//
// The O(N^2 nb) parts (64x64 potf2, 64-wide triangular panel solve) are FP64-ALU kernels.
#include <float.h>
#include <math.h>
#include <string.h>
#include <atomic>
#include "tgp_common.cuh"
#include "profile_policy.cuh"
#include "batch.cuh"

// ============================================================================================
// gemm_nt_sub
// ============================================================================================
constexpr int BM = 128, BK = 16, STAGES = 4, GEMM_THREADS = 256;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem_src), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

// Load one BK-wide stage of a (ROWS x BK) operand tile: 8 chunks of 16 B per row.
// Chunk c of row r is stored at physical chunk c ^ ((r & 1) << 2).
template <int ROWS>
__device__ __forceinline__ void load_operand_stage(double* smem, const double* __restrict__ G,
                                                   int64_t ldg, int64_t row0, int64_t nrows,
                                                   int64_t k0, int64_t Kd, int tid) {
  const int c = tid & 7;
  const int rbase = tid >> 3;  // 0..31
  const int64_t k = k0 + 2 * c;
  int kbytes = (int)((Kd - k) * 8);
  kbytes = kbytes < 0 ? 0 : (kbytes > 16 ? 16 : kbytes);
#pragma unroll
  for (int i = 0; i < ROWS / 32; ++i) {
    const int r = rbase + 32 * i;
    const int64_t gr = row0 + r;
    const bool ok = gr < nrows;
    const double* src = G + (ok ? gr : 0) * ldg + (kbytes ? k : 0);
    const int pc = c ^ ((r & 1) << 2);
    cp_async16(smem + (r * 8 + pc) * 2, src, ok ? kbytes : 0);
  }
}

// C (M x Nc) -= A (M x Kd) * B^T (Nc x Kd).  lower_only: skip tiles above the diagonal and mask n > m.
// CTA tile BM x BN_, 8 warps arranged WARPS_M x WARPS_N.  The launches use <64, 4, 2, 2>: 128 x 64 tile, warp tile
// 32 x 32, two CTAs per SM so that the epilogue (C read-modify-write) and the pipeline fill of one CTA hide under the
// DMMA work of the other.
// The CTA tile whose top-left corner is (m0, n0).
template <int BN_, int WARPS_M, int WARPS_N>
__device__ __forceinline__ void gemm_nt_sub_tile(double* __restrict__ C, int64_t M, int64_t Nc, int64_t ldc,
                                                 const double* __restrict__ A, int64_t lda,
                                                 const double* __restrict__ B, int64_t ldb, int64_t Kd,
                                                 int lower_only, const int64_t m0, const int64_t n0) {
  constexpr int WM = BM / WARPS_M, WN = BN_ / WARPS_N;   // warp tile
  constexpr int MB = WM / 8, NBK = WN / 8;                // 8x8 blocks per warp tile
  constexpr int STAGE_D = (BM + BN_) * BK;
  static_assert(WARPS_M * WARPS_N == 8, "8 warps");
  extern __shared__ __align__(16) double gsm[];
  if (lower_only && n0 > m0 + BM - 1) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm0 = (warp / WARPS_N) * WM, wn0 = (warp % WARPS_N) * WN;
  const int g = lane >> 2, t = lane & 3;

  double acc[MB][NBK][2];
#pragma unroll
  for (int i = 0; i < MB; ++i)
#pragma unroll
    for (int j = 0; j < NBK; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  const int KT_ = (int)((Kd + BK - 1) / BK);
  auto issue = [&](int kt) {
    if (kt < KT_) {
      double* sa = gsm + (kt % STAGES) * STAGE_D;
      double* sb = sa + BM * BK;
      load_operand_stage<BM>(sa, A, lda, m0, M, (int64_t)kt * BK, Kd, tid);
      load_operand_stage<BN_>(sb, B, ldb, n0, Nc, (int64_t)kt * BK, Kd, tid);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) issue(s);

  const int swz = (g & 1) << 2;
  for (int kt = 0; kt < KT_; ++kt) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    issue(kt + STAGES - 1);
    const double* sa = gsm + (kt % STAGES) * STAGE_D;
    const double* sb = sa + BM * BK;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int pc = (h * 4 + t) ^ swz;
      double2 af[MB], bf[NBK];
#pragma unroll
      for (int i = 0; i < MB; ++i)
        af[i] = *reinterpret_cast<const double2*>(sa + ((wm0 + i * 8 + g) * 8 + pc) * 2);
#pragma unroll
      for (int j = 0; j < NBK; ++j)
        bf[j] = *reinterpret_cast<const double2*>(sb + ((wn0 + j * 8 + g) * 8 + pc) * 2);
#pragma unroll
      for (int i = 0; i < MB; ++i)
#pragma unroll
        for (int j = 0; j < NBK; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i].x, bf[j].x);
#pragma unroll
      for (int i = 0; i < MB; ++i)
#pragma unroll
        for (int j = 0; j < NBK; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i].y, bf[j].y);
    }
  }
  cp_async_wait<0>();

  const bool vec = ((ldc & 1) == 0) && ((((uintptr_t)C) & 15) == 0);
#pragma unroll
  for (int i = 0; i < MB; ++i) {
    const int64_t r = m0 + wm0 + i * 8 + g;
    if (r >= M) continue;
#pragma unroll
    for (int j = 0; j < NBK; ++j) {
      const int64_t c = n0 + wn0 + j * 8 + 2 * t;
      bool ok0 = c < Nc, ok1 = c + 1 < Nc;
      if (lower_only) {
        ok0 = ok0 && (c <= r);
        ok1 = ok1 && (c + 1 <= r);
      }
      double* p = C + r * ldc + c;
      if (vec && ok0 && ok1) {
        double2 v = *reinterpret_cast<double2*>(p);
        v.x -= acc[i][j][0];
        v.y -= acc[i][j][1];
        *reinterpret_cast<double2*>(p) = v;
      } else {
        if (ok0) p[0] -= acc[i][j][0];
        if (ok1) p[1] -= acc[i][j][1];
      }
    }
  }
}

template <int BN_, int WARPS_M, int WARPS_N, int MIN_CTAS>
__global__ void __launch_bounds__(GEMM_THREADS, MIN_CTAS)
gemm_nt_sub_kernel(double* __restrict__ C, int64_t M, int64_t Nc, int64_t ldc,
                   const double* __restrict__ A, int64_t lda, const double* __restrict__ B, int64_t ldb,
                   int64_t Kd, int lower_only) {
  gemm_nt_sub_tile<BN_, WARPS_M, WARPS_N>(C, M, Nc, ldc, A, lda, B, ldb, Kd, lower_only, (int64_t)blockIdx.y * BM,
                                          (int64_t)blockIdx.x * BN_);
}

static int gemm_nt_sub_launch(double* C, int64_t M, int64_t Nc, int64_t ldc, const double* A, int64_t lda,
                              const double* B, int64_t ldb, int64_t Kd, int lower_only, cudaStream_t st) {
  if (M <= 0 || Nc <= 0 || Kd <= 0) return TGP_OK;
  TGP_CHECK_ARG((lda % 2 == 0) && (ldb % 2 == 0), "leading dimensions must be even (16-byte rows)");
  TGP_CHECK_ARG(((uintptr_t)A % 16 == 0) && ((uintptr_t)B % 16 == 0), "operands must be 16-byte aligned");
  constexpr int SMEM = STAGES * (BM + 64) * BK * 8;
  static TgpPerDeviceOnce attr_once;
  if (tgp_first_use_on_device(attr_once)) {
    TGP_CUDA(cudaFuncSetAttribute(gemm_nt_sub_kernel<64, 4, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    // same shared-memory carve-out for every kernel of the factorisation: no L1/shared reconfiguration
    // between the back-to-back small launches of a panel
    TGP_CUDA(cudaFuncSetAttribute(gemm_nt_sub_kernel<64, 4, 2, 2>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
  }
  dim3 grid((unsigned)tgp_cdiv(Nc, 64), (unsigned)tgp_cdiv(M, BM));
  TGP_CHECK_ARG(grid.y <= 65535u, "M too large for one launch");
  gemm_nt_sub_kernel<64, 4, 2, 2><<<grid, GEMM_THREADS, SMEM, st>>>(C, M, Nc, ldc, A, lda, B, ldb, Kd, lower_only);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

extern "C" int tgp_pairbin_set_block_sums(int on);
extern "C" int tgp_pairbin_set_fast_paths(int bits);
extern "C" int tgp_pairbin_set_record_cap(int n);
extern "C" int tgp_bootbin_set_paths(int bits);
extern "C" int tgp_set_option(const char* name, int value) {
  if (name && !strcmp(name, "pairbin_block_sums")) return tgp_pairbin_set_block_sums(value);
  if (name && !strcmp(name, "pairbin_fast_paths")) return tgp_pairbin_set_fast_paths(value);
  if (name && !strcmp(name, "pairbin_record_cap")) return tgp_pairbin_set_record_cap(value);
  if (name && !strcmp(name, "bootbin_paths")) return tgp_bootbin_set_paths(value);
  tgp_set_error("tgp_set_option: unknown option");
  return TGP_ERR_INVALID;
}

// ============================================================================================
// potf2: unblocked Cholesky of an n x n (n <= 64) diagonal block by one CTA (CTA 0 of the fused panel step below).
// ============================================================================================
constexpr int NB = 64;           // inner block
constexpr int NB_PITCH = NB + 1;

// 256 threads, the block in shared memory, factorised in four 16-column steps so that only 4 x 3
// CTA barriers separate the phases instead of 64 x 2:
//   (i)   warp 0 factorises the 16 x 16 diagonal sub-block in registers (lane = row, shuffles),
//   (ii)  one thread per row below solves its 16 entries against that sub-block,
//   (iii) all threads apply the rank-16 update to the trailing lower triangle.
constexpr int PF_B = 16;
#ifdef TGP_PANEL_TIMING
__device__ unsigned long long g_pf_cycles[4];   // accumulated cycles of potf2 phases (i), (ii), (iii)
#define PF_T(k) if (threadIdx.x == 0) { const long long t_ = clock64(); g_pf_cycles[k] += t_ - pf_t0; pf_t0 = t_; }
#else
#define PF_T(k)
#endif
// Factorise the NB x NB tile S (pitch NB_PITCH, identity-padded beyond n) in shared memory; all 256 threads
// of the CTA call this.  rdiag receives 1 / L[j][j].  Ends with a CTA barrier.
__device__ __forceinline__ void potf2_smem(double* __restrict__ S, double* __restrict__ rdiag, int n,
                                           int32_t* __restrict__ info, int64_t global_off) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef TGP_PANEL_TIMING
  long long pf_t0 = clock64();
  if (tid == 0) g_pf_cycles[0] = g_pf_cycles[1] = g_pf_cycles[2] = 0;
#endif
  for (int k0 = 0; k0 < NB; k0 += PF_B) {
    // (i) 16 x 16 diagonal sub-block, lanes 0..15 hold one row each.  Pivots in groups of four: inside a group
    // every pivot updates only the group's own columns (<= 3 shuffle + DFMA pairs on the critical path); the
    // columns to the right take the group's rank-4 update afterwards, as independent shuffle / DFMA pairs.
    if (warp == 0) {
      double a[PF_B];
      const int l15 = lane & 15;
      const int r = k0 + l15;
      unsigned badmask = 0u;       // the same in every lane (d is a broadcast)
#pragma unroll
      for (int c = 0; c < PF_B; ++c) a[c] = S[r * NB_PITCH + k0 + c];
#pragma unroll
      for (int grp = 0; grp < PF_B / 4; ++grp) {
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int j = 4 * grp + jj;
          const double d = __shfl_sync(0xffffffffu, a[j], j);           // pivot a_jj from lane j
          // not positive definite / not finite: remembered branch-free (bit j), reported once after the block
          badmask |= (k0 + j < n && (!(d > 0.0) || !isfinite(d))) ? (1u << j) : 0u;
          // one reciprocal square root per pivot: l_jj = d * rsqrt(d), l_ij = a_ij * rsqrt(d) (no FP64 divide or
          // square-root call on the critical path; results agree with sqrt/divide to ~1 ulp)
          const double rinv = rsqrt(d);
          a[j] = (l15 == j) ? d * rinv : ((l15 > j) ? a[j] * rinv : a[j]);
          if (lane == j) rdiag[k0 + j] = rinv;
#pragma unroll
          for (int c = 0; c < PF_B; ++c) {   // constant bounds + static predicate: keeps a[] in registers
            if (c > j && c < 4 * grp + 4) {
              const double lcj = __shfl_sync(0xffffffffu, a[j], c);     // l_cj from lane c
              a[c] = (l15 >= c) ? fma(-a[j], lcj, a[c]) : a[c];
            }
          }
        }
#pragma unroll
        for (int c = 0; c < PF_B; ++c) {
          if (c >= 4 * grp + 4) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const double lck = __shfl_sync(0xffffffffu, a[4 * grp + k], c);
              a[c] = (l15 >= c) ? fma(-a[4 * grp + k], lck, a[c]) : a[c];
            }
          }
        }
      }
      if (lane < 16) {
#pragma unroll
        for (int c = 0; c < PF_B; ++c) S[r * NB_PITCH + k0 + c] = a[c];
      }
      if (badmask && lane == 0)   // keep the first failure (LAPACK's info)
        atomicCAS(info, 0, (int32_t)(global_off + k0 + __ffs(badmask)));
    }
    __syncthreads();
    PF_T(0);
    // (ii) rows below: x <- x * L11^-T (thread per row)
    const int below = NB - k0 - PF_B;
    if (tid < below) {
      const int r = k0 + PF_B + tid;
      double x[PF_B];
#pragma unroll
      for (int c = 0; c < PF_B; ++c) x[c] = S[r * NB_PITCH + k0 + c];
#pragma unroll
      for (int j = 0; j < PF_B; ++j) {
        x[j] = x[j] * rdiag[k0 + j];
#pragma unroll
        for (int c = j + 1; c < PF_B; ++c) x[c] = fma(-x[j], S[(k0 + c) * NB_PITCH + k0 + j], x[c]);
      }
#pragma unroll
      for (int c = 0; c < PF_B; ++c) S[r * NB_PITCH + k0 + c] = x[c];
    }
    __syncthreads();
    PF_T(1);
    // (iii) trailing update S[i][c] -= sum_k S[i][k0+k] S[c][k0+k], k0+16 <= c <= i < 64, on the DMMA pipe:
    // the lower 8 x 8 blocks of the trailing square are dealt to the warps, K = 16 = four m8n8k4 steps each
    if (below > 0) {
      const int m0 = k0 + PF_B, nblk = below / 8, g8 = lane >> 2, t4 = lane & 3;
      for (int p = warp; p < nblk * (nblk + 1) / 2; p += 8) {
        int bi = 0, bj = p;
        while (bj > bi) { bj -= bi + 1; ++bi; }
        const double* Ar = S + (m0 + 8 * bi + g8) * NB_PITCH + k0 + t4;
        const double* Br = S + (m0 + 8 * bj + g8) * NB_PITCH + k0 + t4;
        double c0 = 0.0, c1 = 0.0;
#pragma unroll
        for (int ks = 0; ks < PF_B / 4; ++ks) dmma884(c0, c1, Ar[4 * ks], Br[4 * ks]);
        double* Cr = S + (m0 + 8 * bi + g8) * NB_PITCH + m0 + 8 * bj + 2 * t4;
        Cr[0] -= c0;
        Cr[1] -= c1;
      }
    }
    __syncthreads();
    PF_T(2);
  }
}

// Load / store the lower triangle of an n x n (n <= NB) global block into the identity-padded tile S.
__device__ __forceinline__ void potf2_load(double* __restrict__ S, const double* __restrict__ A, int n, int64_t ld) {
#pragma unroll 4
  for (int idx = threadIdx.x; idx < NB * NB; idx += 256) {
    const int r = idx / NB, c = idx % NB;  // coalesced along c
    S[r * NB_PITCH + c] = (r < n && c <= r) ? A[(int64_t)r * ld + c] : (r == c ? 1.0 : 0.0);
  }
}
__device__ __forceinline__ void potf2_store(const double* __restrict__ S, double* __restrict__ A, int n, int64_t ld) {
#pragma unroll 4
  for (int idx = threadIdx.x; idx < NB * NB; idx += 256) {
    const int r = idx / NB, c = idx % NB;
    if (r < n && c <= r) A[(int64_t)r * ld + c] = S[r * NB_PITCH + c];
  }
}

// ============================================================================================
// trsm panel: B (M x nb) <- B * L^-T for an nb x nb (nb <= 64) lower-triangular L.  Thread per row,
// right-looking over columns so the FMAs of one step are independent.
// ============================================================================================
constexpr int TRSM_ROWS = 64;   // rows per CTA: small CTAs spread short panels over many SMs
constexpr int TRSM_SMEM = (NB * NB + NB + TRSM_ROWS * NB_PITCH) * 8;

// FULL: nb == 64 and 16-byte aligned rows: every thread streams its own row with 32 independent 16-byte
// loads (no staging, nothing to wait for but the L tile), solves in registers and streams it back.
// Otherwise (edge panels): rows are staged through shared memory element by element.
template <bool FULL>
__global__ void __launch_bounds__(TRSM_ROWS)
trsm_panel_kernel(const double* __restrict__ L, int nb, int64_t ldl, double* __restrict__ B, int64_t M,
                  int64_t ldb) {
#include "trsm_panel_body.cuh"
}

static int trsm_panel_launch(const double* L, int nb, int64_t ldl, double* B, int64_t M, int64_t ldb,
                             cudaStream_t st) {
  if (M <= 0 || nb <= 0) return TGP_OK;
  static TgpPerDeviceOnce attr_once;
  if (tgp_first_use_on_device(attr_once)) {
    TGP_CUDA(cudaFuncSetAttribute(trsm_panel_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TRSM_SMEM));
    TGP_CUDA(cudaFuncSetAttribute(trsm_panel_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TRSM_SMEM));
    TGP_CUDA(cudaFuncSetAttribute(trsm_panel_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TGP_CUDA(cudaFuncSetAttribute(trsm_panel_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  }
  const bool full = (nb == NB) && ((ldb & 1) == 0) && (((uintptr_t)B & 15) == 0);
  const unsigned grid = (unsigned)tgp_cdiv(M, TRSM_ROWS);
  if (full) trsm_panel_kernel<true><<<grid, TRSM_ROWS, TRSM_SMEM, st>>>(L, nb, ldl, B, M, ldb);
  else trsm_panel_kernel<false><<<grid, TRSM_ROWS, TRSM_SMEM, st>>>(L, nb, ldl, B, M, ldb);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

// ============================================================================================
// Fused panel step.  A w-wide (w <= TGP_OB = 512) panel = the w x w diagonal block D at `Akk` plus `below` rows
// stored under it.  ONE launch per 64-wide block column j factorises D's diagonal block (j,j) and solves every
// row block under it, instead of the potf2 / trsm_panel / K=64 gemm chain (3 launches per block column inside D
// plus ~15 for the rows below).  Inside the panel the off-diagonal blocks are LEFT-looking and the diagonal
// blocks of D RIGHT-looking:
//   CTA 0 (row block j)      : load block (j,j) -- already fully updated --, potf2 in shared memory, store,
//                              publish a flag in global memory.
//   CTA i > 0 (row block r)  : T = A[r, j] - A[r, 0:j] A[j, 0:j]^T  on the DMMA pipe (K = 64 j <= 448; this
//                              overlaps with CTA 0's potf2), wait for the flag, X = T L_jj^-T by substitution
//                              (4 threads per row), store X; if r is a row block of D also apply its own rank-64
//                              update A[r, r] -= X X^T, so that block (j+1, j+1) is final when launch j+1 starts.
// Waiting CTAs spin on the flag; CTA 0 is always dispatched first, so the wait cannot deadlock; the spin is
// bounded anyway (info = -1 if it ever trips).
// ============================================================================================
constexpr int PL_THREADS = 256;
constexpr int PL_P = NB + 2;                                 // pitch of the T / L tiles (even: 16-byte LDS)
constexpr int PL_RING_D = STAGES * (NB + NB) * BK;            // operand ring, doubles
constexpr int PL_MP = 9;                                      // pitch of the 8 x 8 inverse blocks
constexpr int PL_TAIL_D = 2 * NB * PL_P + NB + 8 * 8 * PL_MP;  // T tile + L tile + 1/diag + 8 inverses (aliases the ring)
constexpr int PL_SMEM = (PL_RING_D > PL_TAIL_D ? PL_RING_D : PL_TAIL_D) * 8;
constexpr int PL_NFLAGS = 4096;
__device__ unsigned g_panel_flags[PL_NFLAGS];
// every flag-synchronised launch takes a fresh (slot, epoch) pair: a stale value in a reused slot never matches
static unsigned next_flag_epoch() {
  static std::atomic<unsigned> counter{0};
  unsigned e = counter.fetch_add(1u) + 1u;
  if (e == 0) e = counter.fetch_add(1u) + 1u;   // 0 is the value of a never-used flag
  return e;
}

#ifdef TGP_PANEL_TIMING   // phase timestamps of one launch (tools/panel_timing.py builds a private copy of the library)
__device__ unsigned long long g_pl_times[32];   // [0,16): globaltimer ns, [16,32): clock64 of the same stamps
__device__ __forceinline__ void pl_stamp(int i) {
  if (threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_pl_times[i] = t;
    g_pl_times[16 + i] = (unsigned long long)clock64();
  }
}
#define PL_T(i) pl_stamp(i)
extern "C" int tgp_debug_panel_times(unsigned long long* host32) {
  return cudaMemcpyFromSymbol(host32, g_pl_times, sizeof(unsigned long long) * 32) == cudaSuccess ? 0 : -2;
}
extern "C" int tgp_debug_potf2_cycles(unsigned long long* host4) {
  return cudaMemcpyFromSymbol(host4, g_pf_cycles, sizeof(unsigned long long) * 4) == cudaSuccess ? 0 : -2;
}
#else
#define PL_T(i)
#endif

// CTA number `cta` of one launch (flag: the launch's inter-CTA flag word).
__device__ __forceinline__ void panel_left_body(double* __restrict__ Akk, int64_t ld, int w, int64_t below, int j,
                                                int32_t* __restrict__ info, int64_t goff, unsigned* flag,
                                                unsigned epoch, const unsigned cta) {
  extern __shared__ __align__(16) double psm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ndiag = (w + NB - 1) / NB;
  const int c0 = j * NB;
  const int nbj = (w - c0 < NB) ? (w - c0) : NB;

  if (cta == 0) {
    double* S = psm;                       // NB x NB_PITCH
    double* rdiag = psm + NB * NB_PITCH;
    double* D = Akk + (int64_t)c0 * ld + c0;
    PL_T(0);
    potf2_load(S, D, nbj, ld);
    __syncthreads();
    PL_T(1);
    potf2_smem(S, rdiag, nbj, info, goff + c0);
    PL_T(2);
    potf2_store(S, D, nbj, ld);
    __threadfence();
    __syncthreads();
    if (tid == 0) atomicExch(flag, epoch);
    PL_T(3);
    return;
  }

  const int rb = j + cta;                  // row block: < ndiag inside D, else among the rows below
  const bool in_diag = rb < ndiag;
  int64_t r0;
  int nrows;
  if (in_diag) {
    r0 = (int64_t)rb * NB;
    nrows = (w - rb * NB < NB) ? (w - rb * NB) : NB;
  } else {
    r0 = w + (int64_t)(rb - ndiag) * NB;
    const int64_t left = w + below - r0;
    nrows = left < NB ? (int)left : NB;
  }
  const int g = lane >> 2, t = lane & 3;
  const int wm0 = (warp >> 2) * 32, wn0 = (warp & 3) * 16;   // warp tile 32 x 16 of the 64 x 64 block
#ifdef TGP_PANEL_TIMING
  const bool stamp = cta == 1;
#undef PL_T
#define PL_T(i) if (stamp) pl_stamp(i)
#endif
  PL_T(8);

  // ---- T = A[r, j] (prefetched) - A[r, 0:c0] A[j, 0:c0]^T ------------------------------------
  double cv[4][2][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = wm0 + i * 8 + g;
#pragma unroll
    for (int jn = 0; jn < 2; ++jn) {
      const int c = wn0 + jn * 8 + 2 * t;
      const double* p = Akk + (r0 + r) * ld + c0 + c;
      double v0 = 0.0, v1 = 0.0;
      if (r < nrows) {
        if (c + 1 < nbj) {
          const double2 v = *reinterpret_cast<const double2*>(p);
          v0 = v.x;
          v1 = v.y;
        } else if (c < nbj) {
          v0 = p[0];
        }
      }
      cv[i][jn][0] = v0;
      cv[i][jn][1] = v1;
    }
  }
  const int KT_ = c0 / BK;
  if (KT_ > 0) {
    double acc[4][2][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int jn = 0; jn < 2; ++jn) acc[i][jn][0] = acc[i][jn][1] = 0.0;
    constexpr int STAGE_D = (NB + NB) * BK;
    auto issue = [&](int kt) {
      if (kt < KT_) {
        double* sa = psm + (kt % STAGES) * STAGE_D;
        double* sb = sa + NB * BK;
        load_operand_stage<NB>(sa, Akk, ld, r0, r0 + nrows, (int64_t)kt * BK, c0, tid);
        load_operand_stage<NB>(sb, Akk, ld, c0, w, (int64_t)kt * BK, c0, tid);
      }
      cp_async_commit();
    };
#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) issue(s);
    const int swz = (g & 1) << 2;
    for (int kt = 0; kt < KT_; ++kt) {
      cp_async_wait<STAGES - 2>();
      __syncthreads();
      issue(kt + STAGES - 1);
      const double* sa = psm + (kt % STAGES) * STAGE_D;
      const double* sb = sa + NB * BK;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int pc = (h * 4 + t) ^ swz;
        double2 af[4], bf[2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
          af[i] = *reinterpret_cast<const double2*>(sa + ((wm0 + i * 8 + g) * 8 + pc) * 2);
#pragma unroll
        for (int jn = 0; jn < 2; ++jn)
          bf[jn] = *reinterpret_cast<const double2*>(sb + ((wn0 + jn * 8 + g) * 8 + pc) * 2);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int jn = 0; jn < 2; ++jn) dmma884(acc[i][jn][0], acc[i][jn][1], af[i].x, bf[jn].x);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int jn = 0; jn < 2; ++jn) dmma884(acc[i][jn][0], acc[i][jn][1], af[i].y, bf[jn].y);
      }
    }
    cp_async_wait<0>();
    __syncthreads();   // the ring is dead from here on; its storage becomes the T / L tiles
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int jn = 0; jn < 2; ++jn) {
        cv[i][jn][0] -= acc[i][jn][0];
        cv[i][jn][1] -= acc[i][jn][1];
      }
  }
  double* Ts = psm;                        // NB x PL_P
  double* Ls = psm + NB * PL_P;            // NB x PL_P, Ls[i][c] = L_jj[i][c]
  double* dinv = Ls + NB * PL_P;           // 1 / L_jj[c][c]
  double* Minv = dinv + NB;                // inverses of the 8 x 8 diagonal blocks of L_jj, pitch PL_MP
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int jn = 0; jn < 2; ++jn) {
      const int r = wm0 + i * 8 + g, c = wn0 + jn * 8 + 2 * t;
      *reinterpret_cast<double2*>(Ts + r * PL_P + c) = make_double2(cv[i][jn][0], cv[i][jn][1]);
    }

  PL_T(9);
  // ---- wait for the diagonal block ---------------------------------------------------------
  if (tid == 0) {
    unsigned spins = 0;
    while (*reinterpret_cast<volatile unsigned*>(flag) != epoch) {
      __nanosleep(40);
      if (++spins > (1u << 26)) {          // seconds: something is badly wrong, do not hang the GPU
        atomicExch(info, -1);
        break;
      }
    }
    __threadfence();
  }
  __syncthreads();
  PL_T(10);
  const double* Lg = Akk + (int64_t)c0 * ld + c0;
  {
    // Ls[i][c] = L[i][c] (strictly lower part), dinv[c] = 1 / L[c][c].  Every thread touches column tid % 64.
    const int c = tid & (NB - 1);
#pragma unroll 4
    for (int idx = tid; idx < NB * NB; idx += PL_THREADS) {
      const int i = idx / NB;
      Ls[i * PL_P + c] = (i < nbj && c < i) ? __ldcg(Lg + (int64_t)i * ld + c) : 0.0;
    }
    if (tid < NB) dinv[tid] = (tid < nbj) ? 1.0 / __ldcg(Lg + (int64_t)tid * ld + tid) : 1.0;
  }
  __syncthreads();
  // inverses of the eight 8 x 8 diagonal blocks of L (warp b, lane c < 8: column c of block b by forward
  // substitution); everything else of the solve is then DMMA work without a scalar dependency chain
  if (lane < 8) {
    const int o = warp * 8, c = lane;
    double z[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      double sacc = (i == c) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k)
        if (k < i) sacc = fma(-Ls[(o + i) * PL_P + o + k], (k >= c) ? z[k] : 0.0, sacc);
      z[i] = (i >= c) ? sacc * dinv[o + i] : 0.0;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) Minv[warp * PL_MP * 8 + i * PL_MP + c] = z[i];
  }
  __syncthreads();
  PL_T(11);

  // ---- X = T L^-T by 8-column blocks: X_b = (T_b - sum_{b' < b} X_b' L_bb'^T) L_bb^-T.  Warp w owns rows
  // 8 w .. 8 w + 7 of the tile, so every dependency stays inside the warp (syncwarp only); right-looking: as
  // soon as X_b exists it is subtracted from all later column blocks (independent accumulators) -------------
  {
    double* Tw = Ts + (warp * 8 + g) * PL_P;      // this lane's row of the tile
    double acc[8][2];
#pragma unroll
    for (int bb = 0; bb < 8; ++bb) {
      const double2 v = *reinterpret_cast<const double2*>(Tw + 8 * bb + 2 * t);
      acc[bb][0] = v.x;
      acc[bb][1] = v.y;
    }
#pragma unroll
    for (int bb = 0; bb < 8; ++bb) {
      // R_b from the accumulator layout (row g, columns 2t, 2t+1) to the A-operand layout (row g, k = t)
      __syncwarp();
      *reinterpret_cast<double2*>(Tw + 8 * bb + 2 * t) = make_double2(acc[bb][0], acc[bb][1]);
      __syncwarp();
      const double a0 = Tw[8 * bb + t], a1 = Tw[8 * bb + 4 + t];
      const double* Mi = Minv + bb * PL_MP * 8 + g * PL_MP;
      double x0 = 0.0, x1 = 0.0;
      dmma884(x0, x1, a0, Mi[t]);
      dmma884(x0, x1, a1, Mi[4 + t]);
      __syncwarp();
      *reinterpret_cast<double2*>(Tw + 8 * bb + 2 * t) = make_double2(x0, x1);     // X_b, final
      if (bb < 7) {
        __syncwarp();
        const double na0 = -Tw[8 * bb + t], na1 = -Tw[8 * bb + 4 + t];
#pragma unroll
        for (int b2 = bb + 1; b2 < 8; ++b2) {
          const double* Lr = Ls + (8 * b2 + g) * PL_P + 8 * bb;
          dmma884(acc[b2][0], acc[b2][1], na0, Lr[t]);
          dmma884(acc[b2][0], acc[b2][1], na1, Lr[4 + t]);
        }
      }
    }
  }
  __syncthreads();
  PL_T(12);

  // ---- own rank-64 update of the diagonal block (r, r) of D (prefetch, DMMA, write back) -----------------
  // warps 0..3 take block rows (warp, 7 - warp) of the 8 x 8 grid of 8x8 blocks: 9 lower blocks each.
  if (in_diag && warp < 4) {
    double* Dg = Akk + r0 * ld + r0;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int bi = pass ? 7 - warp : warp;
      const int r = bi * 8 + g;
      double d[8][2], acc[8][2];
#pragma unroll
      for (int bj = 0; bj < 8; ++bj) {
        acc[bj][0] = acc[bj][1] = 0.0;
        d[bj][0] = d[bj][1] = 0.0;
        if (bj <= bi && r < nrows) {
          const int c = bj * 8 + 2 * t;
          const double* p = Dg + (int64_t)r * ld + c;
          if (c + 1 <= r) {
            const double2 v = *reinterpret_cast<const double2*>(p);
            d[bj][0] = v.x;
            d[bj][1] = v.y;
          } else if (c <= r) {
            d[bj][0] = p[0];
          }
        }
      }
#pragma unroll 4
      for (int k4 = 0; k4 < NB / 4; ++k4) {
        const double a = Ts[r * PL_P + k4 * 4 + t];
#pragma unroll
        for (int bj = 0; bj < 8; ++bj) {
          if (bj <= bi) {
            const double b = Ts[(bj * 8 + g) * PL_P + k4 * 4 + t];
            dmma884(acc[bj][0], acc[bj][1], a, b);
          }
        }
      }
#pragma unroll
      for (int bj = 0; bj < 8; ++bj) {
        if (bj <= bi && r < nrows) {
          const int c = bj * 8 + 2 * t;
          double* p = Dg + (int64_t)r * ld + c;
          if (c + 1 <= r) *reinterpret_cast<double2*>(p) = make_double2(d[bj][0] - acc[bj][0], d[bj][1] - acc[bj][1]);
          else if (c <= r) p[0] = d[bj][0] - acc[bj][0];
        }
      }
    }
  }

  PL_T(13);
  // ---- store X -----------------------------------------------------------------------------
#pragma unroll 4
  for (int idx = tid; idx < NB * NB; idx += PL_THREADS) {
    const int r = idx / NB, c = idx % NB;
    if (r < nrows && c < nbj) Akk[(r0 + r) * ld + c0 + c] = Ts[r * PL_P + c];
  }
  PL_T(14);
}

__global__ void __launch_bounds__(PL_THREADS, 2)
panel_left_kernel(double* __restrict__ Akk, int64_t ld, int w, int64_t below, int j, int32_t* __restrict__ info,
                  int64_t goff, unsigned slot, unsigned epoch) {
  panel_left_body(Akk, ld, w, below, j, info, goff, &g_panel_flags[slot], epoch, blockIdx.x);
}


// Factorise the w x w (w <= TGP_OB) diagonal block at Akk and solve the `below` rows under it (L21 = A21 L11^-T).
static int panel_factor(double* Akk, int64_t w, int64_t ld, int64_t below, int32_t* info, int64_t goff,
                        cudaStream_t st) {
  static TgpPerDeviceOnce attr_once;
  if (tgp_first_use_on_device(attr_once)) {
    TGP_CUDA(cudaFuncSetAttribute(panel_left_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PL_SMEM));
    TGP_CUDA(cudaFuncSetAttribute(panel_left_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
  }
  const int ndiag = (int)tgp_cdiv(w, NB);
  const int64_t nbelow = tgp_cdiv(below, NB);
  for (int j = 0; j < ndiag; ++j) {
    const unsigned epoch = next_flag_epoch();
    const unsigned grid = (unsigned)((ndiag - j) + nbelow);
    panel_left_kernel<<<grid, PL_THREADS, PL_SMEM, st>>>(Akk, ld, (int)w, below, j, info, goff,
                                                         epoch % PL_NFLAGS, epoch);
    TGP_LAUNCH_CHECK();
  }
  return TGP_OK;
}

// ============================================================================================
// Blocked drivers (two levels: TGP_OB-wide block columns whose updates run on DMMA with Kd = TGP_OB, NB-wide
// inner blocks handled by the kernels above).  A dense factor is the envelope factor whose row ends
// (tgp_envelope_ends) are n in every block column.
// ============================================================================================

// B (M x n) <- B * L^-T for an n x n (n <= TGP_OB) lower-triangular L, by recursive halving of the columns:
//   [B1 B2] <- [B1 L11^-T,  (B2 - B1 L21^T) L22^-T]
// so the updates are GEMMs with K = n/2, n/4, ... (large K, each C column block touched once per level)
// and only the 64-wide leaves run the FP64-ALU substitution kernel.
static int trsm_rows_halving(const double* L, int64_t n, int64_t ldl, double* B, int64_t M, int64_t ldb,
                             cudaStream_t st) {
  if (n <= NB) return trsm_panel_launch(L, (int)n, ldl, B, M, ldb, st);
  const int64_t h = ((n / 2 + NB - 1) / NB) * NB;  // split at a multiple of 64
  int rc = trsm_rows_halving(L, h, ldl, B, M, ldb, st);
  if (rc) return rc;
  // B2 -= B1 * L21^T, L21 = L[h:n, 0:h]
  rc = gemm_nt_sub_launch(B + h, M, n - h, ldb, B, ldb, L + h * ldl, ldl, h, 0, st);
  if (rc) return rc;
  return trsm_rows_halving(L + h * ldl + h, n - h, ldl, B + h, M, ldb, st);
}

// B (M x n) <- B * L^-T, right-looking over TGP_OB-wide block columns: the unknowns [k, c1) of block column b are
// solved by halving, then enter only the unknowns [c1, ends[b]) -- 2 M n bw flop instead of M n^2 for an envelope.
static int trsm_rows_blocked(const double* L, int64_t n, int64_t ld, const std::vector<int64_t>& ends, double* B,
                             int64_t M, int64_t ldb, cudaStream_t st) {
  for (int64_t k = 0, b = 0; k < n; k += TGP_OB, ++b) {
    const int64_t w = (n - k < TGP_OB) ? (n - k) : TGP_OB;
    const int64_t c1 = k + w;
    int rc = trsm_rows_halving(L + k * ld + k, w, ld, B + k, M, ldb, st);
    if (rc) return rc;
    rc = gemm_nt_sub_launch(B + c1, M, ends[b] - c1, ldb, B + k, ldb, L + c1 * ld + k, ld, w, 0, st);
    if (rc) return rc;
  }
  return TGP_OK;
}

// Per TGP_OB-wide block column b: the fused panel step factorises the diagonal block and solves the rows
// [c1, ends[b]) inside the envelope, then one lower-triangular DMMA update applies them to the trailing matrix inside
// the envelope.  The rows [ends[b], n) of block column b are neither read nor written (they keep whatever the K build
// left there: entries below 1e-40 amp for an envelope).  `extra` right-hand-side rows stored below the matrix (rows
// n .. n + extra - 1) end as Y L^-T (= L^-1 y per row): the forward substitution at DMMA speed.  Where the envelope
// reaches n they are contiguous with its rows and ride inside the panel solve and the update; elsewhere they take
// their own row solve and update.  (Empty updates launch nothing.)
static int potrf_blocked(double* A, int64_t n, int64_t ld, const std::vector<int64_t>& ends, int64_t extra,
                         int32_t* info, cudaStream_t st) {
  for (int64_t k = 0, b = 0; k < n; k += TGP_OB, ++b) {
    const int64_t w = (n - k < TGP_OB) ? (n - k) : TGP_OB;
    const int64_t c1 = k + w, below = ends[b] - c1;
    const int64_t ride = (ends[b] == n) ? extra : 0;
    double* Akk = A + k * ld + k;
    double* Ark = A + c1 * ld + k;      // the rows of this block column inside the envelope (+ the riding rows)
    int rc = panel_factor(Akk, w, ld, below + ride, info, k, st);
    if (rc) return rc;
    rc = gemm_nt_sub_launch(A + c1 * ld + c1, below + ride, below, ld, Ark, ld, Ark, ld, w, 1, st);
    if (rc) return rc;
    if (extra > ride) {
      double* Aek = A + n * ld + k;
      rc = trsm_rows_halving(Akk, w, ld, Aek, extra, ld, st);
      if (rc) return rc;
      rc = gemm_nt_sub_launch(A + n * ld + c1, extra, below, ld, Aek, ld, Ark, ld, w, 0, st);
      if (rc) return rc;
    }
  }
  return TGP_OK;
}

// --------------------------------------------------------------------------------------------
// Look-ahead driver for large N.  The panel of an outer block (diagonal factorisation + solve of the rows below) is
// a chain of small, latency-bound launches; run on its own high-priority stream it hides under the previous step's
// big trailing update:
//   panel stream P : panel(b) .. wait U2(b-1) .. U1(b) = update of the NEXT panel's column block only
//   caller stream U: wait panel(b) .. U2(b) = update of everything right of the next panel
// U1(b) and U2(b) write disjoint blocks; panel(b+1) needs U1(b) and U2(b-1) only, so U2(b) overlaps
// with panel(b+1).  The caller's stream is joined with P before returning.
// --------------------------------------------------------------------------------------------
// Helper stream + events of the look-ahead schedule: one set per host thread AND device (streams and events
// belong to the device that was current when they were created).
struct LookaheadCtx {
  cudaStream_t panel = nullptr;
  std::vector<cudaEvent_t> ev;
  bool ensure(size_t n) {
    while (ev.size() < n) {
      cudaEvent_t e;
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return false;
      ev.push_back(e);
    }
    return true;
  }
  cudaEvent_t get(size_t i) { return ev[i]; }
};
static LookaheadCtx* lookahead_ctx() {
  static thread_local LookaheadCtx c[TGP_MAX_DEVICES];
  LookaheadCtx& L = c[tgp_current_device()];
  if (!L.panel) {
    int lo = 0, hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithPriority(&L.panel, cudaStreamNonBlocking, hi) != cudaSuccess) {
      L.panel = nullptr;
      return nullptr;
    }
  }
  return &L;
}

// Outer blocks of width obl (a multiple of TGP_OB), each factorised as TGP_OB-wide sub-panels solved against all rows
// below them, with one K = TGP_OB update of the outer block's later columns in between.  The rows of an outer block
// end at the envelope of its first TGP_OB block column, and the `extra` rows ride through every panel and update: so
// an envelope runs with obl = TGP_OB and extra = 0, and only a dense factor (ends n everywhere) takes wider blocks or
// extra rows.
static int potrf_lookahead(double* A, int64_t n, int64_t ld, const std::vector<int64_t>& ends, int64_t extra,
                           int64_t obl, int32_t* info, cudaStream_t U) {
  LookaheadCtx* Lp = lookahead_ctx();
  if (!Lp) {
    tgp_set_error("potrf: could not create the look-ahead stream: %s", cudaGetErrorString(cudaGetLastError()));
    return TGP_ERR_CUDA;
  }
  LookaheadCtx& L = *Lp;
  cudaStream_t P = L.panel;
  const int64_t nblk = tgp_cdiv(n, obl);
  if (!L.ensure((size_t)(2 + 2 * nblk))) {
    tgp_set_error("potrf: cudaEventCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
    return TGP_ERR_CUDA;
  }
  TGP_CUDA(cudaEventRecord(L.get(0), U));
  TGP_CUDA(cudaStreamWaitEvent(P, L.get(0), 0));
  // event slots: 1 + 2 b = panel(b) done (on P), 2 + 2 b = U2(b) done (on U), 1 + 2 nblk = the join
  for (int64_t b = 0; b < nblk; ++b) {
    const int64_t k = b * obl;
    const int64_t w = (n - k < obl) ? (n - k) : obl;
    const int64_t c1 = k + w, below = ends[k / TGP_OB] - c1;
    int rc;
    for (int64_t s = 0; s < w; s += TGP_OB) {
      const int64_t ws = (w - s < TGP_OB) ? (w - s) : TGP_OB;
      double* Ass = A + (k + s) * ld + (k + s);
      const int64_t below_s = (c1 - (k + s) - ws) + below + extra;
      rc = panel_factor(Ass, ws, ld, below_s, info, k + s, P);
      if (rc) return rc;
      double* Aop = A + (k + s + ws) * ld + (k + s);
      rc = gemm_nt_sub_launch(A + (k + s + ws) * ld + (k + s + ws), below_s, w - s - ws, ld, Aop, ld, Aop, ld, ws, 1,
                              P);
      if (rc) return rc;
    }
    TGP_CUDA(cudaEventRecord(L.get(1 + 2 * b), P));
    TGP_CUDA(cudaStreamWaitEvent(U, L.get(1 + 2 * b), 0));
    // everything the next panel reads must be final: the U2 updates up to block b-1 (stream order on U covers the
    // earlier ones)
    if (b >= 1) TGP_CUDA(cudaStreamWaitEvent(P, L.get(2 + 2 * (b - 1)), 0));
    double* Ark = A + c1 * ld + k;
    const int64_t w2 = (below < obl) ? below : obl, rest2 = below - w2;
    rc = gemm_nt_sub_launch(A + c1 * ld + c1, below + extra, w2, ld, Ark, ld, Ark, ld, w, 1, P);   // U1(b)
    if (rc) return rc;
    rc = gemm_nt_sub_launch(A + (c1 + w2) * ld + (c1 + w2), rest2 + extra, rest2, ld, Ark + w2 * ld, ld, Ark + w2 * ld,
                            ld, w, 1, U);                                                            // U2(b)
    if (rc) return rc;
    TGP_CUDA(cudaEventRecord(L.get(2 + 2 * b), U));
  }
  TGP_CUDA(cudaEventRecord(L.get(1 + 2 * nblk), P));
  TGP_CUDA(cudaStreamWaitEvent(U, L.get(1 + 2 * nblk), 0));
  return TGP_OK;
}

static int check_mat(const double* A, int64_t N, int64_t ld) {
  if (N < 0 || ld < N) return 1;
  if (N > 0 && (!A || (ld & 1) || ((uintptr_t)A & 15))) return 1;
  return 0;
}

// The look-ahead schedule from N = 3 TGP_OB, for a dense factor or an envelope factor without extra rows; the
// sequential one otherwise.
static int potrf_run(double* A, int64_t N, int64_t ld, const int64_t* row_end, int64_t extra, int32_t* info,
                     cudaStream_t st) {
  TGP_CUDA(cudaMemsetAsync(info, 0, sizeof(int32_t), st));
  if (N == 0) return TGP_OK;
  const std::vector<int64_t> ends = tgp_envelope_ends(row_end, N);
  if (N >= 3 * TGP_OB && (!row_end || extra == 0)) {
    // K = 1024 trailing updates amortise the C read-modify-write better once the updates dominate (measured: K = 1024
    // from N ~ 14k, 2048 from ~ 28k)
    const int64_t obl = row_end ? TGP_OB : (N >= 28000 ? 2048 : (N >= 14000 ? 1024 : TGP_OB));
    return potrf_lookahead(A, N, ld, ends, extra, obl, info, st);
  }
  return potrf_blocked(A, N, ld, ends, extra, info, st);
}

extern "C" int tgp_potrf(double* A, int64_t N, int64_t ld, int32_t* info, void* stream) {
  TGP_CHECK_ARG(!check_mat(A, N, ld), "A must be 16-byte aligned with even ld >= N");
  TGP_CHECK_ARG(info != nullptr, "info");
  return potrf_run(A, N, ld, nullptr, 0, info, (cudaStream_t)stream);
}

extern "C" int tgp_potrf_rows(double* A, int64_t N, int64_t ld, int64_t nrows, int32_t* info, void* stream) {
  TGP_CHECK_ARG(!check_mat(A, N, ld), "A must be 16-byte aligned with even ld >= N");
  TGP_CHECK_ARG(info != nullptr && nrows >= 0, "info/nrows");
  return potrf_run(A, N, ld, nullptr, nrows, info, (cudaStream_t)stream);
}

// --------------------------------------------------------------------------------------------
// Envelope (variable-band) Cholesky.  With the points sorted along one axis, a kernel that is below 1e-40 of its
// amplitude beyond a coordinate difference d_cut gives a matrix whose row i starts (to 1e-40) at the first point
// within d_cut of point i; a Cholesky factor keeps the envelope of its matrix.  Per TGP_OB-wide block column b the
// caller states row_end[b]: the rows [row_end[b], N) of that block column are (numerically) zero in K and therefore in
// L, so the panel solve and the trailing update stop there: N bw^2 flop instead of N^3 / 3 for a band of bw rows.
// --------------------------------------------------------------------------------------------
extern "C" int tgp_envelope_block(void) { return TGP_OB; }

extern "C" int tgp_potrf_env(double* A, int64_t N, int64_t ld, const int64_t* row_end, int64_t nblocks,
                             int64_t nrows, int32_t* info, void* stream) {
  TGP_CHECK_ARG(!check_mat(A, N, ld), "A must be 16-byte aligned with even ld >= N");
  TGP_CHECK_ARG(info != nullptr && nrows >= 0, "info/nrows");
  TGP_CHECK_ARG(row_end && tgp_envelope_ok(row_end, nblocks, N),
                "row_end must hold one entry per tgp_envelope_block() columns");
  return potrf_run(A, N, ld, row_end, nrows, info, (cudaStream_t)stream);
}

extern "C" int tgp_trsm_rows_env(const double* L, int64_t N, int64_t ld, const int64_t* row_end, int64_t nblocks,
                                 double* B, int64_t M, int64_t ldb, void* stream) {
  TGP_CHECK_ARG(!check_mat(L, N, ld), "L must be 16-byte aligned with even ld >= N");
  TGP_CHECK_ARG(M >= 0 && ldb >= N, "M/ldb");
  TGP_CHECK_ARG(row_end && tgp_envelope_ok(row_end, nblocks, N),
                "row_end must hold one entry per tgp_envelope_block() columns");
  if (M == 0 || N == 0) return TGP_OK;
  TGP_CHECK_ARG(B && (ldb % 2 == 0) && ((uintptr_t)B % 16 == 0), "B must be 16-byte aligned with even ldb");
  return trsm_rows_blocked(L, N, ld, tgp_envelope_ends(row_end, N), B, M, ldb, (cudaStream_t)stream);
}

extern "C" int tgp_trsm_rows(const double* L, int64_t N, int64_t ld, double* B, int64_t M, int64_t ldb,
                             void* stream) {
  TGP_CHECK_ARG(!check_mat(L, N, ld), "L must be 16-byte aligned with even ld >= N");
  TGP_CHECK_ARG(M >= 0 && ldb >= N, "M/ldb");
  if (M == 0 || N == 0) return TGP_OK;
  TGP_CHECK_ARG(B && (ldb % 2 == 0) && ((uintptr_t)B % 16 == 0), "B must be 16-byte aligned with even ldb");
  return trsm_rows_blocked(L, N, ld, tgp_envelope_ends(nullptr, N), B, M, ldb, (cudaStream_t)stream);
}

extern "C" int tgp_gemm_nt_sub(double* C, int64_t M, int64_t Nc, int64_t ldc, const double* A, int64_t lda,
                               const double* B, int64_t ldb, int64_t Kd, int lower_only, void* stream) {
  TGP_CHECK_ARG(M >= 0 && Nc >= 0 && Kd >= 0 && ldc >= Nc && lda >= Kd && ldb >= Kd, "shape");
  if (M == 0 || Nc == 0 || Kd == 0) return TGP_OK;
  TGP_CHECK_ARG(C && A && B, "null pointer");
  return gemm_nt_sub_launch(C, M, Nc, ldc, A, lda, B, ldb, Kd, lower_only, (cudaStream_t)stream);
}

// ============================================================================================
// Single right-hand-side solves  L w = b  (forward) and  L^T x = w  (backward): persistent sweep kernels in trsv.cu.
// ============================================================================================
int tgp_trsv_sweeps(const double* L, int64_t N, int64_t ld, double* b, int which, cudaStream_t st);
int tgp_trsv_sweeps_multi(const double* L, int64_t N, int64_t ld, double* b, int r, int which, cudaStream_t st);
static int trsv_backward(const double* L, int64_t N, int64_t ld, double* b, cudaStream_t st) {
  return tgp_trsv_sweeps(L, N, ld, b, 2, st);
}

extern "C" int tgp_potrs_multi(const double* L, int64_t N, int64_t ld, double* B, int32_t r, void* stream) {
  TGP_CHECK_ARG(r >= 1 && r <= TGP_MAX_RHS, "number of right-hand sides must be 1 .. TGP_MAX_RHS");
  TGP_CHECK_ARG(N >= 0 && ld >= N, "N/ld");
  if (N == 0) return TGP_OK;
  TGP_CHECK_ARG(L && B, "null pointer");
  return tgp_trsv_sweeps_multi(L, N, ld, B, r, 3, (cudaStream_t)stream);
}

extern "C" int tgp_potrs_vec(const double* L, int64_t N, int64_t ld, double* b, void* stream) {
  TGP_CHECK_ARG(N >= 0 && ld >= N, "N/ld");
  if (N == 0) return TGP_OK;
  TGP_CHECK_ARG(L && b, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  return tgp_trsv_sweeps(L, N, ld, b, 3, st);   // forward, then backward (one workspace, one set of inverses)
}

// ============================================================================================
// Reductions: log-determinant, chi2 = y . alpha, final log-likelihood.
// ============================================================================================
// out[0] = sum 2 log L_ii ; out[1] = y . alpha (if given).  Single CTA, deterministic order.
__device__ __forceinline__ void logdet_chi2_body(const double* __restrict__ L, int64_t N, int64_t ld,
                                                 const double* __restrict__ y, const double* __restrict__ alpha,
                                                 double* __restrict__ out) {
  __shared__ double s0[32], s1[32];
  double a = 0.0, c = 0.0;
  for (int64_t i = threadIdx.x; i < N; i += blockDim.x) {
    a += 2.0 * log(L[i * ld + i]);
    if (y) c = fma(y[i], alpha[i], c);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    c += __shfl_xor_sync(0xffffffffu, c, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { s0[warp] = a; s1[warp] = c; }
  __syncthreads();
  if (warp == 0) {
    a = s0[lane];
    c = s1[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    if (lane == 0) {
      out[0] = a;
      if (y) out[1] = c;
    }
  }
}
__global__ void __launch_bounds__(1024)
logdet_chi2_kernel(const double* __restrict__ L, int64_t N, int64_t ld, const double* __restrict__ y,
                   const double* __restrict__ alpha, double* __restrict__ out) {
  logdet_chi2_body(L, N, ld, y, alpha, out);
}

extern "C" int tgp_logdet_chi2(const double* L, int64_t N, int64_t ld, const double* y, const double* alpha,
                               double* out, void* stream) {
  TGP_CHECK_ARG(N >= 0 && ld >= N && out, "N/ld/out");
  TGP_CHECK_ARG((y == nullptr) == (alpha == nullptr), "y and alpha go together");
  logdet_chi2_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(L, N, ld, y, alpha, out);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

// out = {logL, chi2, logdet}; tmp = {logdet, chi2}.
__device__ __forceinline__ void loglike_finish_body(const double* tmp, int64_t N, const int32_t* __restrict__ info,
                                                    double* out) {
  const double logdet = tmp[0], chi2 = tmp[1];
  double ll = -0.5 * chi2 - 0.5 * (double)N * log(2.0 * TGP_PI) - 0.5 * logdet;
  // info > 0: leading minor not positive definite -> -inf (log_likelihood.py:38-39).  info < 0: an internal
  // flag wait timed out -- NOT a property of the matrix: NaN here, and the host raises when it sees info < 0.
  if (*info > 0 || isnan(ll)) ll = -INFINITY;
  if (*info < 0) ll = NAN;
  out[0] = ll;
  out[1] = chi2;
  out[2] = logdet;
}
__global__ void loglike_finish_kernel(const double* tmp, int64_t N, const int32_t* __restrict__ info, double* out) {
  loglike_finish_body(tmp, N, info, out);
}

// chi2 = ||w||^2 with w = L^-1 y (forward sweep only) -- y^T K^-1 y without the backward solve.
__device__ __forceinline__ void sumsq_body(const double* __restrict__ w, int64_t N, double* __restrict__ out1) {
  __shared__ double s0[32];
  double a = 0.0;
  for (int64_t i = threadIdx.x; i < N; i += blockDim.x) a = fma(w[i], w[i], a);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) s0[warp] = a;
  __syncthreads();
  if (warp == 0) {
    a = s0[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) *out1 = a;
  }
}
__global__ void __launch_bounds__(1024)
sumsq_kernel(const double* __restrict__ w, int64_t N, double* __restrict__ out1) {
  sumsq_body(w, N, out1);
}

static int loglike_args(const double* X, const double* y, int64_t N, const double* work, const double* alpha,
                        const double* out, const int32_t* info, const int64_t* row_end, int64_t nblocks) {
  TGP_CHECK_ARG(N > 0 && X && y && work && alpha && out && info, "null pointer / N");
  TGP_CHECK_ARG(tgp_envelope_ok(row_end, nblocks, N), "row_end must hold one entry per tgp_envelope_block() columns");
  return TGP_OK;
}

// Everything after the K build (lower triangle of K + diag in `work`): factorisation, sweeps, reductions.
static int loglike_after_build(const double* y, int64_t N, double* work, int64_t ld, double* alpha, int want_alpha,
                               double* out, int32_t* info, const int64_t* row_end, int64_t nblocks, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  // out[1], out[2] double as scratch {logdet, chi2} until the finishing kernel reorders them
  double* tmp = out + 1;
  if (row_end) {
    // Envelope: a row riding through the factorisation would cost two more (one-row) launches chains per block column;
    // the persistent sweep kernels read the factor once instead (w = L^-1 y, and alpha = L^-T w in the same call).
    rc = tgp_potrf_env(work, N, ld, row_end, nblocks, 0, info, stream);
    if (rc) return rc;
    TGP_CUDA(cudaMemcpyAsync(alpha, y, N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    rc = tgp_trsv_sweeps(work, N, ld, alpha, want_alpha ? 3 : 1, st);
    if (rc) return rc;
  } else {
    // y rides along as row N of the workspace: the factorisation's panel solves turn it into w = L^-1 y
    double* wrow = work + N * ld;
    TGP_CUDA(cudaMemcpyAsync(wrow, y, N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    rc = tgp_potrf_rows(work, N, ld, 1, info, stream);
    if (rc) return rc;
    TGP_CUDA(cudaMemcpyAsync(alpha, wrow, N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (want_alpha) {
      rc = trsv_backward(work, N, ld, alpha, st);   // alpha = L^-T w
      if (rc) return rc;
    }
  }
  if (want_alpha) {
    logdet_chi2_kernel<<<1, 1024, 0, st>>>(work, N, ld, y, alpha, tmp);  // chi2 = y . alpha
    TGP_LAUNCH_CHECK();
  } else {
    // y^T K^-1 y = ||L^-1 y||^2: the backward sweep is not needed for the likelihood alone
    logdet_chi2_kernel<<<1, 1024, 0, st>>>(work, N, ld, nullptr, nullptr, tmp);
    TGP_LAUNCH_CHECK();
    sumsq_kernel<<<1, 1024, 0, st>>>(alpha, N, tmp + 1);
    TGP_LAUNCH_CHECK();
  }
  loglike_finish_kernel<<<1, 1, 0, st>>>(tmp, N, info, out);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

static int loglike_impl(const double* X, const double* y, const double* yerr2, int64_t N,
                        const tgp_kernel* k, double* work, int64_t ld, double* alpha, int want_alpha,
                        double* out, int32_t* info, const int64_t* row_end, int64_t nblocks, void* stream) {
  int rc = loglike_args(X, y, N, work, alpha, out, info, row_end, nblocks);
  if (rc) return rc;
  rc = tgp_kmat_sym(X, N, k, yerr2, work, ld, /*lower_only=*/1, stream);
  if (rc) return rc;
  return loglike_after_build(y, N, work, ld, alpha, want_alpha, out, info, row_end, nblocks, stream);
}

extern "C" int tgp_loglike(const double* X, const double* y, const double* yerr2, int64_t N,
                           const tgp_kernel* k, double* work, int64_t ld, double* alpha, int want_alpha,
                           double* out, int32_t* info, void* stream) {
  return loglike_impl(X, y, yerr2, N, k, work, ld, alpha, want_alpha, out, info, nullptr, 0, stream);
}

extern "C" int tgp_loglike_env(const double* X, const double* y, const double* yerr2, int64_t N,
                               const tgp_kernel* k, double* work, int64_t ld, double* alpha, int want_alpha,
                               double* out, int32_t* info, const int64_t* row_end, int64_t nblocks, void* stream) {
  TGP_CHECK_ARG(row_end != nullptr, "row_end");
  return loglike_impl(X, y, yerr2, N, k, work, ld, alpha, want_alpha, out, info, row_end, nblocks, stream);
}

extern "C" int tgp_loglike_sum(const double* X, const double* y, const double* yerr2, int64_t N,
                               const tgp_kernel_sum* k, double* work, int64_t ld, double* alpha, int want_alpha,
                               double* out, int32_t* info, const int64_t* row_end, int64_t nblocks, void* stream) {
  int rc = loglike_args(X, y, N, work, alpha, out, info, row_end, nblocks);
  if (rc) return rc;
  rc = tgp_kmat_sym_sum(X, N, k, yerr2, work, ld, /*lower_only=*/1, stream);
  if (rc) return rc;
  return loglike_after_build(y, N, work, ld, alpha, want_alpha, out, info, row_end, nblocks, stream);
}

// ============================================================================================
// Several outputs with one covariance (tgp_loglike_multi): K is built and factorised once; the r outputs ride
// through the dense factorisation as r extra rows (rows N .. N + r - 1 of `work`, one output per row), and the sweeps
// stream the factor once for all outputs (tgp_trsv_sweeps_multi), each column in the single-output order, so each
// column of alpha is the single-output alpha of that column bit for bit.
// ============================================================================================
// rows[c][i] = Y[i][c] (to_rows) or Y[i][c] = rows[c][i]
__global__ void __launch_bounds__(256)
multi_transpose_kernel(double* __restrict__ Y, int r, double* __restrict__ rows, int64_t ld, int64_t N, int to_rows) {
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < N * r;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = idx / r;
    const int c = (int)(idx - i * r);
    if (to_rows) rows[c * ld + i] = Y[idx];
    else Y[idx] = rows[c * ld + i];
  }
}

// sum over the 1024 threads in the order of logdet_chi2_kernel; the result is valid in every thread
__device__ double block_sum_1024(double a, double* s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();                                 // s is free
  if (lane == 0) s[warp] = a;
  __syncthreads();
  a = s[lane];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  return a;
}

// out = {sum_c logL_c, sum_c chi2_c, logdet}: logdet once; chi2_c = y_c . alpha_c (want_alpha) or |L^-1 y_c|^2,
// each in the order of the single-output reductions, then added up column by column.  Single CTA of 1024 threads.
__global__ void __launch_bounds__(1024)
loglike_multi_finish_kernel(const double* __restrict__ L, int64_t N, int64_t ld, const double* __restrict__ Y, int r,
                            const double* __restrict__ W, int want_alpha, const int32_t* __restrict__ info,
                            double* __restrict__ out) {
  __shared__ double s[32];
  double a = 0.0;
  for (int64_t i = threadIdx.x; i < N; i += blockDim.x) a += 2.0 * log(L[i * ld + i]);
  const double logdet = block_sum_1024(a, s);
  double chi2 = 0.0;
  for (int c = 0; c < r; ++c) {
    const double* w = W + c * ld;
    double v = 0.0;
    for (int64_t i = threadIdx.x; i < N; i += blockDim.x) v = want_alpha ? fma(Y[i * r + c], w[i], v) : fma(w[i], w[i], v);
    chi2 += block_sum_1024(v, s);
  }
  if (threadIdx.x == 0) {
    double ll = -0.5 * chi2 - 0.5 * (double)r * (double)N * log(2.0 * TGP_PI) - 0.5 * (double)r * logdet;
    if (*info > 0 || isnan(ll)) ll = -INFINITY;   // as loglike_finish_kernel
    if (*info < 0) ll = NAN;
    out[0] = ll;
    out[1] = chi2;
    out[2] = logdet;
  }
}

extern "C" int tgp_loglike_multi(const double* X, const double* Y, int32_t r, const double* yerr2, int64_t N,
                                 const tgp_kernel_sum* k, double* work, int64_t ld, double* alpha, int want_alpha,
                                 double* out, int32_t* info, const int64_t* row_end, int64_t nblocks, void* stream) {
  TGP_CHECK_ARG(r >= 1 && r <= TGP_MAX_RHS, "number of outputs must be 1 .. TGP_MAX_RHS");
  TGP_CHECK_ARG(ksum_ok(k), "kernel sum descriptor");
  int rc = loglike_args(X, Y, N, work, alpha, out, info, row_end, nblocks);
  if (rc) return rc;
  TGP_CHECK_ARG(!check_mat(work, N, ld), "work must be 16-byte aligned with even ld >= N");
  if (r == 1)   // (N, 1) is an N-vector: the single-output entry, bit for bit
    return tgp_loglike_sum(X, Y, yerr2, N, k, work, ld, alpha, want_alpha, out, info, row_end, nblocks, stream);
  cudaStream_t st = (cudaStream_t)stream;
  rc = tgp_kmat_sym_sum(X, N, k, yerr2, work, ld, /*lower_only=*/1, stream);
  if (rc) return rc;
  double* rows = work + N * ld;                    // output c in row N + c
  const unsigned tg = (unsigned)tgp_cdiv(N * r, (int64_t)256) < 4096u ? (unsigned)tgp_cdiv(N * r, (int64_t)256) : 4096u;
  multi_transpose_kernel<<<tg, 256, 0, st>>>(const_cast<double*>(Y), r, rows, ld, N, 1);
  TGP_LAUNCH_CHECK();
  if (row_end) {
    // as loglike_after_build: the envelope factorisation, then both sweeps per output
    rc = tgp_potrf_env(work, N, ld, row_end, nblocks, 0, info, stream);
    if (rc) return rc;
    rc = tgp_trsv_sweeps_multi(work, N, ld, rows, r, want_alpha ? 3 : 1, st);
    if (rc) return rc;
  } else {
    rc = tgp_potrf_rows(work, N, ld, r, info, stream);   // rows <- L^-1 Y^T
    if (rc) return rc;
    if (want_alpha) {
      rc = tgp_trsv_sweeps_multi(work, N, ld, rows, r, 2, st);
      if (rc) return rc;
    }
  }
  loglike_multi_finish_kernel<<<1, 1024, 0, st>>>(work, N, ld, Y, r, rows, want_alpha, info, out);
  TGP_LAUNCH_CHECK();
  multi_transpose_kernel<<<tg, 256, 0, st>>>(alpha, r, rows, ld, N, 0);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

// ============================================================================================
// Batches of independent problems (tgp_loglike_batch).  The schedule of potrf_blocked with y riding along as row N,
// run once over the panel steps of the largest problem: every launch covers each problem that still has columns at
// that step (CTAs of the others exit), and each CTA runs the body of the single-problem kernel on its problem's block.
// For N >= 3 TGP_OB the single call takes the look-ahead driver, whose U1 / U2 updates split the same K = TGP_OB update
// by columns: per element the same DMMA chain, so the factor is the same bit for bit.
// ============================================================================================
// grid: (problem, CTA of the panel launch); the CTAs 0 of all problems are dispatched before any CTA that waits.
__global__ void __launch_bounds__(PL_THREADS, 2)
panel_left_batch_kernel(const TgpBatchProb* __restrict__ pr, int64_t k, int j, int32_t* __restrict__ info,
                        unsigned* __restrict__ flags, unsigned epoch) {
  const int b = blockIdx.x;
  const int64_t N = pr[b].N;
  if (k >= N) return;
  const int w = (int)(N - k < TGP_OB ? N - k : TGP_OB);
  const int ndiag = (w + NB - 1) / NB;
  if (j >= ndiag) return;
  const int64_t below = N - k - w + 1;
  if ((int64_t)blockIdx.y >= (ndiag - j) + (below + NB - 1) / NB) return;
  const int64_t ld = pr[b].ld;
  panel_left_body(pr[b].A + k * ld + k, ld, w, below, j, info + b, k, flags + b, epoch, blockIdx.y);
}

// The trailing update of outer step k: C (rest + 1 x rest) -= L21 L21^T (lower), the y row included.
// grid: (problem, row tile * tiles_n + column tile).
__global__ void __launch_bounds__(GEMM_THREADS, 2)
gemm_trail_batch_kernel(const TgpBatchProb* __restrict__ pr, int64_t k, int tiles_n) {
  const int b = blockIdx.x;
  const int64_t N = pr[b].N;
  const int64_t w = N - k < TGP_OB ? N - k : TGP_OB, rest = N - k - w;
  if (rest <= 0) return;
  const int64_t m0 = (int64_t)(blockIdx.y / tiles_n) * BM, n0 = (int64_t)(blockIdx.y % tiles_n) * 64;
  if (m0 >= rest + 1 || n0 >= rest) return;
  const int64_t ld = pr[b].ld;
  double* Ark = pr[b].A + (k + w) * ld + k;
  gemm_nt_sub_tile<64, 4, 2>(Ark + w, rest + 1, rest, ld, Ark, ld, Ark, ld, w, 1, m0, n0);
}

int tgp_batch_potrf_rows(const TgpBatchProb* pr, const int64_t* Nh, int32_t B, int32_t* info, unsigned* flags,
                         cudaStream_t st) {
  static TgpPerDeviceOnce attr_once;
  if (tgp_first_use_on_device(attr_once)) {
    constexpr int GSMEM = STAGES * (BM + 64) * BK * 8;
    TGP_CUDA(cudaFuncSetAttribute(panel_left_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PL_SMEM));
    TGP_CUDA(cudaFuncSetAttribute(panel_left_batch_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
    TGP_CUDA(cudaFuncSetAttribute(gemm_trail_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GSMEM));
    TGP_CUDA(cudaFuncSetAttribute(gemm_trail_batch_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
  }
  TGP_CUDA(cudaMemsetAsync(info, 0, sizeof(int32_t) * B, st));
  int64_t nmax = 0;
  for (int32_t b = 0; b < B; ++b) nmax = Nh[b] > nmax ? Nh[b] : nmax;
  unsigned epoch = 0;   // the flags start at 0 and every panel launch of this call takes the next epoch
  for (int64_t k = 0; k < nmax; k += TGP_OB) {
    const int64_t wmax = nmax - k < TGP_OB ? nmax - k : TGP_OB;
    for (int j = 0; j < (int)tgp_cdiv(wmax, NB); ++j) {
      int64_t ctas = 0;   // the largest launch of a problem at this step
      for (int32_t b = 0; b < B; ++b) {
        if (Nh[b] <= k) continue;
        const int64_t w = Nh[b] - k < TGP_OB ? Nh[b] - k : TGP_OB, ndiag = tgp_cdiv(w, NB);
        if (j >= ndiag) continue;
        const int64_t c = (ndiag - j) + tgp_cdiv(Nh[b] - k - w + 1, NB);
        ctas = c > ctas ? c : ctas;
      }
      panel_left_batch_kernel<<<dim3((unsigned)B, (unsigned)ctas), PL_THREADS, PL_SMEM, st>>>(pr, k, j, info, flags,
                                                                                             ++epoch);
      TGP_LAUNCH_CHECK();
    }
    const int64_t rest = nmax - k - wmax;   // the largest trailing update belongs to the largest problem
    if (rest > 0) {
      const int tiles_n = (int)tgp_cdiv(rest, 64);
      const int64_t tiles = tgp_cdiv(rest + 1, BM) * tiles_n;
      gemm_trail_batch_kernel<<<dim3((unsigned)B, (unsigned)tiles), GEMM_THREADS, STAGES * (BM + 64) * BK * 8, st>>>(
          pr, k, tiles_n);
      TGP_LAUNCH_CHECK();
    }
  }
  return TGP_OK;
}

// One CTA per problem: the reductions of loglike_after_build and loglike_finish_kernel, same bodies, same order.
__global__ void __launch_bounds__(1024)
loglike_batch_finish_kernel(const TgpBatchProb* __restrict__ pr, int want_alpha, const int32_t* __restrict__ info,
                            double* __restrict__ out) {
  __shared__ double tmp[2];   // {logdet, chi2}
  const TgpBatchProb& p = pr[blockIdx.x];
  if (want_alpha) {
    logdet_chi2_body(p.A, p.N, p.ld, p.y, p.alpha, tmp);   // chi2 = y . alpha
  } else {
    logdet_chi2_body(p.A, p.N, p.ld, nullptr, nullptr, tmp);
    __syncthreads();
    sumsq_body(p.alpha, p.N, tmp + 1);                      // chi2 = ||L^-1 y||^2
  }
  __syncthreads();
  if (threadIdx.x == 0) loglike_finish_body(tmp, p.N, info + blockIdx.x, out + 3 * (int64_t)blockIdx.x);
}

int tgp_batch_loglike_finish(const TgpBatchProb* pr, int32_t B, int want_alpha, const int32_t* info, double* out,
                             cudaStream_t st) {
  loglike_batch_finish_kernel<<<(unsigned)B, 1024, 0, st>>>(pr, want_alpha, info, out);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

// ============================================================================================
// Selected inverse of a batch (tgp_batch_selinv in selinv.cu): the halving leaves and the DMMA products of step s of
// selinv_run, on a grid of (problem, CTA of the single launch); CTAs of problems without that launch exit.  Scratch
// of a problem as selinv_run lays it out: -W^T, W^T (TGP_OB x TGP_OB each), T^T (TGP_OB x even(N)).
// ============================================================================================
// grid: (CTA of the single launch, leaf blockIdx.y of the launch's table).  The operands come from the parameter bank,
// as the single kernel's do: that keeps them out of the registers, which the row solve of the FULL path fills.
template <bool FULL>
__global__ void __launch_bounds__(TRSM_ROWS)
selinv_leaf_batch_kernel(const __grid_constant__ TgpLeafLaunch p) {
  const TgpLeafArgs& a = p.a[blockIdx.y];
  if ((int64_t)blockIdx.x * TRSM_ROWS >= a.M) return;
  const double* const L = a.L;
  double* const B = a.B;
  const int64_t ldl = a.ldl, M = a.M, ldb = a.ldb;
  const int nb = a.nb;
#include "trsm_panel_body.cuh"
}

int tgp_batch_selinv_leaves(const TgpLeafArgs* leaves, int32_t n, bool full, cudaStream_t st) {
  static TgpPerDeviceOnce attr_once;
  if (tgp_first_use_on_device(attr_once)) {
    TGP_CUDA(cudaFuncSetAttribute(selinv_leaf_batch_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  TRSM_SMEM));
    TGP_CUDA(cudaFuncSetAttribute(selinv_leaf_batch_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  TRSM_SMEM));
  }
  for (int32_t i0 = 0; i0 < n; i0 += TGP_LEAF_GROUP) {
    TgpLeafLaunch p;
    const int32_t cnt = std::min(n - i0, TGP_LEAF_GROUP);
    int64_t mmax = 0;
    for (int32_t i = 0; i < cnt; ++i) {
      p.a[i] = leaves[i0 + i];
      mmax = std::max(mmax, p.a[i].M);
    }
    const dim3 grid((unsigned)tgp_cdiv(mmax, TRSM_ROWS), (unsigned)cnt);
    if (full) selinv_leaf_batch_kernel<true><<<grid, TRSM_ROWS, TRSM_SMEM, st>>>(p);
    else selinv_leaf_batch_kernel<false><<<grid, TRSM_ROWS, TRSM_SMEM, st>>>(p);
    TGP_LAUNCH_CHECK();
  }
  return TGP_OK;
}

// grid: (problem, row tile * tiles_n + column tile) of the product `op` (batch.cuh) of step s
__global__ void __launch_bounds__(GEMM_THREADS, 2)
selinv_gemm_batch_kernel(const TgpBatchProb* __restrict__ pr, double* const* __restrict__ scr, int s, int op,
                         int leaf, int tiles_n) {
  const int b = blockIdx.x;
  TgpSelStep g;
  if (!tgp_selinv_step(pr[b].N, s, g)) return;
  int64_t M, Nc, Kd;
  if (!tgp_selinv_gemm_shape(g, op, leaf, M, Nc, Kd)) return;
  const int64_t m0 = (int64_t)(blockIdx.y / tiles_n) * BM, n0 = (int64_t)(blockIdx.y % tiles_n) * 64;
  if (m0 >= M || n0 >= Nc) return;
  const int64_t ld = pr[b].ld, ldt = (pr[b].N + 1) & ~(int64_t)1;
  double* A = pr[b].A;
  double* NWT = scr[b];
  double* WT = NWT + TGP_OB * TGP_OB;
  double* TT = NWT + 2 * TGP_OB * TGP_OB;
  double* Akk = A + g.k * ld + g.k;
  double* L21 = A + g.c1 * ld + g.k;
  double* C;
  const double *X, *Y;
  int64_t ldc = ld, ldx = TGP_OB, ldy = ld;
  int lower = 0;
  switch (op) {
    case TGP_SEL_TT: C = TT; ldc = ldt; X = NWT; Y = L21; break;                                       // T^T = W^T L21^T
    case TGP_SEL_ZRJ: C = L21; X = A + g.c1 * ld + g.c1; ldx = ld; Y = TT; ldy = ldt; break;           // -Z[R, R] T
    case TGP_SEL_WTW: C = Akk; X = NWT; Y = WT; ldy = TGP_OB; lower = 1; break;                          // + W^T W
    case TGP_SEL_TZ: C = Akk; X = TT; ldx = ldt; Y = A + g.k * ld + g.c1; lower = 1; break;           // - T^T Z[J, R]
    default: {   // B2 -= B1 L21^T of trsm_rows_halving on the node [o, o + n) split at h
      int64_t o, h, n;
      tgp_halving_node(g.w, leaf, o, h, n);
      C = NWT + o + h;
      ldc = TGP_OB;
      X = NWT + o;
      Y = Akk + (o + h) * ld + o;
    }
  }
  gemm_nt_sub_tile<64, 4, 2>(C, M, Nc, ldc, X, ldx, Y, ldy, Kd, lower, m0, n0);
}

int tgp_batch_selinv_gemm(const TgpBatchProb* pr, double* const* scr, int32_t B, int s, int op, int leaf,
                          int tiles_n, int64_t tiles, cudaStream_t st) {
  constexpr int GSMEM = STAGES * (BM + 64) * BK * 8;
  static TgpPerDeviceOnce attr_once;
  if (tgp_first_use_on_device(attr_once)) {
    TGP_CUDA(cudaFuncSetAttribute(selinv_gemm_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GSMEM));
    TGP_CUDA(cudaFuncSetAttribute(selinv_gemm_batch_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  cudaSharedmemCarveoutMaxShared));
  }
  TGP_CHECK_ARG(tiles <= 65535, "too many tiles for one launch");
  selinv_gemm_batch_kernel<<<dim3((unsigned)B, (unsigned)tiles), GEMM_THREADS, GSMEM, st>>>(pr, scr, s, op, leaf,
                                                                                          tiles_n);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}
