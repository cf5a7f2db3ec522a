// Single right-hand-side triangular solves  L w = b  (forward) and  L^T x = w  (backward): the alpha solve of
// /root/reference/treegp/gp_interp.py:182 and log_likelihood.py:31 (scipy cho_solve -> LAPACK dpotrs).
//
// The operation is HBM-bound: each sweep reads the 4 N^2-byte triangle once (SURVEY.md section 8d).  ONE
// persistent kernel per sweep, one CTA per SM, launched cooperatively (all CTAs co-resident, so waiting on
// another CTA's result always makes progress -- no assumption about dispatch order):
//
//  * the triangle is cut into 64 x 64 tiles; block row k ("slab") is owned by CTA k mod G, which keeps the slab's
//    64 partial sums in shared memory and accumulates them in a FIXED order (column blocks ascending): the
//    result is deterministic, bit-identical from run to run;
//  * a CTA walks the column blocks in windows of up to four (256 unknowns, fetched with one wait) and applies each
//    window to all of its unsolved slabs.  The matrix is streamed straight from global memory into registers, GEMV
//    style: every warp owns eight rows of each slab and reads up to 2 KB contiguous per row with 16-byte loads (32
//    independent loads in flight per lane), so there is no per-tile barrier and no shared-memory staging on the
//    streaming path; the warps of a CTA only meet when a new window of unknowns is fetched;
//  * the serial chain.  For every diagonal block a pre-pass (trsv_prep_kernel) computes D_k = L_kk^-1 and the
//    product W_k = D_k L_{k,k-1} (forward; M_k = L_{k+1,k} D_k for the backward sweep), so that
//        x_k = D_k (b_k - sum_{j<k-1} L_kj x_j)  -  W_k x_{k-1} :
//    the first term is ready before x_{k-1} exists, and the step on the critical path is ONE 64 x 64 mat-vec
//    between "x_{k-1} seen" and "x_k published" instead of a 64-step substitution;
//  * publication is the payload itself: the 64 unknowns are stored into a buffer pre-filled with an all-ones
//    pattern and the waiting threads poll their own words, i.e. one L2 round trip per chain step (no flag + fence
//    + second load).  Only the CTA whose slab is next polls with all 64 threads; the others poll with one.
//
// The backward sweep is the same kernel on the mirrored index set (block i' = nb-1-i) with transposed tile
// products.  Workspace (inverses, products, publication buffers) comes from a library-private stream-ordered
// memory pool and is returned to it on the stream.  A wait that times out (cannot happen with co-resident CTAs;
// guards against a lost launch) sets a sticky device error word that tgp_device_error() reports.
#include <cuda_runtime.h>
#include <stdint.h>
#include "tgp_common.cuh"

constexpr int TS = 64;                 // tile edge = diagonal block = unknowns per chain step
constexpr int TS_P = TS + 2;           // shared-memory row pitch in doubles (528 B: 16-byte aligned rows)
constexpr int TS_THREADS = 256;
constexpr int TS_TILE_D = TS * TS_P;   // doubles per staged tile
constexpr int TS_WIN = 4;              // column blocks of unknowns fetched per wait
constexpr int TS_HAND = 1;             // distances (blocks before a slab's diagonal) handed over through distributed shared
                                       // memory inside a cluster.  1 = the chain step only.  Measured with 5 (the near blocks
                                       // too): hop 0.37 us instead of 0.9 us, but five remote stores per unknown cost the
                                       // publisher as much again -- no gain, so the near blocks keep the global path
constexpr int TS_NEAR = 4;              // blocks before its own diagonal from which a slab is fed one block at a time

__device__ int g_tgp_device_error = 0;

#ifdef TGP_TRSV_TIMING
// debug build (tools/trsv_timing.py): globaltimer stamps of the serial chain, per block: [0] unknowns of the
// previous block seen, [1] (unused), [2] own unknowns published
__device__ unsigned long long g_trsv_stamps[3 * 4096];
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
extern "C" int tgp_debug_trsv_stamps(unsigned long long* host, int n) {
  return cudaMemcpyFromSymbol(host, g_trsv_stamps, sizeof(unsigned long long) * n) == cudaSuccess ? 0 : -1;
}
#define TRSV_STAMP(kp, which) do { if (tid == 0 && (kp) < 4096) g_trsv_stamps[3 * (kp) + (which)] = gtime(); } while (0)
#else
#define TRSV_STAMP(kp, which) do { } while (0)
#endif

extern "C" int tgp_device_error(int reset) {
  int v = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;
  if (cudaMemcpyFromSymbol(&v, g_tgp_device_error, sizeof(int)) != cudaSuccess) return -1;
  if (reset && v) {
    int z = 0;
    cudaMemcpyToSymbol(g_tgp_device_error, &z, sizeof(int));
  }
  return v;
}

// ---- mbarrier / bulk-copy primitives (PTX) -----------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_addr(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_addr(dst)),
               "l"(src), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}
__device__ __forceinline__ double ld_relaxed_f64(const double* p) {
  double v;
  asm volatile("ld.relaxed.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_f64(double* p, double v) {
  asm volatile("st.relaxed.gpu.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ bool unpublished(double v) { return __double_as_longlong(v) == -1ll; }

// ---- pre-pass: inverse of every 64 x 64 diagonal block and its product with the neighbouring tile -------
// One CTA (256 threads) per block k.  dinv[k] = L_kk^-1 (dense 64 x 64 row-major, zero above the diagonal,
// identity in the padding of a short last block); wf[k] = dinv[k] . L[blk k, blk k-1] (k >= 1, forward sweep);
// wb[k] = L[blk k+1, blk k] . dinv[k] (k <= nb-2, backward sweep; rows beyond N are zero).
constexpr int TP_P = TS + 1;
constexpr int TP_SMEM = 3 * TS * TP_P * 8;
__global__ void __launch_bounds__(256)
trsv_prep_kernel(const double* __restrict__ L, int64_t ld, int64_t N, int nb, double* __restrict__ dinv,
                 double* __restrict__ wf, double* __restrict__ wb) {
  extern __shared__ __align__(16) double psm[];
  double (*Lk)[TP_P] = reinterpret_cast<double (*)[TP_P]>(psm);
  double (*Z)[TP_P] = reinterpret_cast<double (*)[TP_P]>(psm + TS * TP_P);
  double (*T)[TP_P] = reinterpret_cast<double (*)[TP_P]>(psm + 2 * TS * TP_P);
  const int tid = threadIdx.x;
  const int k = blockIdx.x;
  const int64_t k0 = (int64_t)k * TS;
  const int w = (int)((N - k0 < TS) ? (N - k0) : TS);
  for (int i = tid; i < TS * TS; i += 256) {
    const int r = i >> 6, c = i & 63;
    double v = (r == c) ? 1.0 : 0.0;
    if (r < w && c <= r) v = L[(k0 + r) * ld + k0 + c];
    Lk[r][c] = v;
    Z[r][c] = 0.0;
  }
  __syncthreads();
  // Z = Lk^-1, column by column: Z[r][c] = (delta_rc - sum_{c<=m<r} Lk[r][m] Z[m][c]) / Lk[r][r].  The four lanes that
  // share column c sit in one warp and nobody else touches that column, so the rows are separated by __syncwarp only.
  {
    double* rdiag = &T[0][0];                      // T is not in use yet
    if (tid < TS) rdiag[tid] = 1.0 / Lk[tid][tid];
    __syncthreads();
    const int c = tid >> 2, part = tid & 3;
    const int m0 = c + ((part - c) & 3);           // first m >= c with m = part (mod 4)
    for (int r = 0; r < TS; ++r) {
      double s0 = 0.0, s1 = 0.0;
      int m = m0;
      for (; m + 4 < r; m += 8) {
        s0 = fma(Lk[r][m], Z[m][c], s0);
        s1 = fma(Lk[r][m + 4], Z[m + 4][c], s1);
      }
      if (m < r) s0 = fma(Lk[r][m], Z[m][c], s0);
      double sv = s0 + s1;
      sv += __shfl_xor_sync(0xffffffffu, sv, 1);
      sv += __shfl_xor_sync(0xffffffffu, sv, 2);
      if (part == 0 && c <= r) Z[r][c] = (((r == c) ? 1.0 : 0.0) - sv) * rdiag[r];
      __syncwarp();
    }
    __syncthreads();
  }
  double* out = dinv + (int64_t)k * TS * TS;
  for (int i = tid; i < TS * TS; i += 256) out[i] = Z[i >> 6][i & 63];
  const int r4 = (tid >> 4) * 4, c4 = (tid & 15) * 4;
  if (wf != nullptr && k >= 1) {
    // T = L[blk k, blk k-1] (rows beyond N zero);  W = Z T
    for (int i = tid; i < TS * TS; i += 256) {
      const int r = i >> 6, c = i & 63;
      T[r][c] = (r < w) ? L[(k0 + r) * ld + (k0 - TS) + c] : 0.0;
    }
    __syncthreads();
    double a[4][4] = {};
    for (int m = 0; m < TS; ++m) {
      double zr[4], tc[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { zr[i] = Z[r4 + i][m]; tc[i] = T[m][c4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) a[i][j] = fma(zr[i], tc[j], a[i][j]);
    }
    double* o = wf + (int64_t)k * TS * TS;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) o[(r4 + i) * TS + c4 + j] = a[i][j];
    __syncthreads();
  }
  if (wb != nullptr && k + 1 < nb) {
    // T = L[blk k+1, blk k] (rows beyond N zero);  M = T Z
    const int w1 = (int)((N - (k0 + TS) < TS) ? (N - (k0 + TS)) : TS);
    for (int i = tid; i < TS * TS; i += 256) {
      const int r = i >> 6, c = i & 63;
      T[r][c] = (r < w1) ? L[(k0 + TS + r) * ld + k0 + c] : 0.0;
    }
    __syncthreads();
    double a[4][4] = {};
    for (int m = 0; m < TS; ++m) {
      double tr[4], zc[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { tr[i] = T[r4 + i][m]; zc[i] = Z[m][c4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) a[i][j] = fma(tr[i], zc[j], a[i][j]);
    }
    double* o = wb + (int64_t)k * TS * TS;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) o[(r4 + i) * TS + c4 + j] = a[i][j];
  }
}

// ---- the sweep ---------------------------------------------------------------------------------
struct TrsvParams {
  const double* L;
  int64_t ld, N;
  double* b;             // right-hand side in, unknowns out
  const double* dinv;    // nb blocks of 64 x 64: inverse diagonal blocks
  const double* wmat;    // nb blocks of 64 x 64: W_k (forward) or M_k (backward)
  double* xpub;          // nb * 64 words, all-ones on entry: block kp's unknowns are published at xpub + 64 kp
  int nb, G, aligned;
  int CS;                // thread-block cluster size (1: none).  G is a multiple of CS
};

// ---- cluster primitives: the chain hop between CTAs of one cluster goes through distributed shared memory ----
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta_rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta_rank));
  return r;
}
__device__ __forceinline__ void st_remote_f64(uint32_t cluster_addr, double v) {
  asm volatile("st.relaxed.cluster.shared::cluster.f64 [%0], %1;" ::"r"(cluster_addr), "d"(v) : "memory");
}
__device__ __forceinline__ double ld_shared_relaxed_f64(const double* p) {
  double v;
  asm volatile("ld.relaxed.cluster.shared::cta.f64 %0, [%1];" : "=d"(v) : "r"(smem_addr(p)) : "memory");
  return v;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ double2 ldg2(const double* p, bool vec) {
  if (vec) return __ldcs(reinterpret_cast<const double2*>(p));      // streamed once: evict-first
  return make_double2(__ldcs(p), __ldcs(p + 1));
}

// R right-hand sides (columns b + c ld, c < R) in one sweep: the factor is streamed once for all of them.  Everything
// that holds unknowns gets R columns of 64 -- a window block [g][c][64], a published block [c][64], acc [slab][c][64]
// (backward [slab][warp][c][64]) -- and every column is accumulated and solved in the order of the R = 1 sweep, so each
// column equals its own single right-hand-side run bit for bit when the grid is the same.
template <bool FWD, int R>
__global__ void __launch_bounds__(TS_THREADS, 1)
trsv_sweep_kernel(TrsvParams P) {
  extern __shared__ __align__(128) unsigned char smraw[];
  double* dtile = reinterpret_cast<double*>(smraw);                // D_k of the next chain step
  double* wtile = dtile + TS_TILE_D;                               // W_k / M_k of the next chain step
  double* xs = wtile + TS_TILE_D;                                  // window of unknowns: TS_WIN column blocks
  double* xh = xs + TS_WIN * TS * R;                               // hand-over buffers [slab parity][distance 1..TS_HAND][64]:
  double* vs = xh + 2 * TS_HAND * TS * R;                          // unknowns of the TS_NEAR blocks before a slab's diagonal; vs = b_k - partial sums
  double* bs = vs + TS * R;                                        // b of the next chain step (prefetched)
  double* red = bs + TS * R;                                       // 4 x 64 partials (backward chain step)
  uint64_t* full = reinterpret_cast<uint64_t*>(red + 4 * TS);      // [0] D/W tiles landed, [1] xc filled by a cluster peer
  double* acc = reinterpret_cast<double*>(full + 2);               // forward [slab][64]; backward [slab][warp][64]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.x, G = P.G, nb = P.nb;
  const int M = (nb - c + G - 1) / G;                              // slabs owned: k = c + m G (primed indices)
  const int64_t ld = P.ld, N = P.N;
  const bool vec = P.aligned != 0;
  const int CS = P.CS;
  constexpr int ACC_PER_SLAB = (FWD ? TS : 8 * TS) * R;

  // primed block index -> first row / column of the block in the matrix, and its height
  auto blk0 = [&](int kp) -> int64_t { return (int64_t)(FWD ? kp : nb - 1 - kp) * TS; };
  auto blkw = [&](int kp) -> int { const int64_t r0 = blk0(kp); return (int)((N - r0 < TS) ? (N - r0) : TS); };

  if (tid == 0) {
    mbar_init(&full[0], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < M * ACC_PER_SLAB; i += TS_THREADS) acc[i] = 0.0;
  for (int i = tid; i < 2 * TS_HAND * TS * R; i += TS_THREADS) xh[i] = __longlong_as_double(-1ll);   // "nothing handed over yet"
  __syncthreads();
  if (CS > 1) cluster_sync_all();                  // every peer's xc is initialised before anyone stores into it
  // The owner of slab k + 1 is CTA (c + 1) mod G, that of slab k - 1 CTA (c - 1) mod G: inside one cluster the
  // unknowns are handed over through distributed shared memory -- stored straight into the peer's xc, which the peer
  // polls word by word, the same payload-is-the-flag protocol as the global publication but without the L2 round
  // trip (~1 us); the global publication stays for everybody else.
  // The same hand-over serves the TS_NEAR blocks before a slab's diagonal (distance d = 1 is the chain step itself,
  // d = 2 .. TS_NEAR the block-by-block feeding of the urgent slab): the owner of slab k pushes its unknowns to the
  // owners of slabs k + 1 .. k + TS_NEAR that sit in its cluster.  local_from(d): is the owner of (my slab - d) a peer?
  auto peer_ahead = [&](int d) -> int { return (c + d) % G; };
  auto local_to = [&](int d) -> bool { return CS > 1 && G >= 2 * TS_HAND && (peer_ahead(d) / CS == c / CS); };
  auto local_from = [&](int d) -> bool { return CS > 1 && G >= 2 * TS_HAND && (((c + G - d) % G) / CS == c / CS); };
  const bool fed_by_prev_local = local_from(1);

  // prefetch what the next chain step (slab index ms) needs: D_k, W_k (bulk async copies) and its right-hand side
  auto prefetch_solve = [&](int ms) {
    if (ms >= M) return;
    const int kp = c + ms * G;
    const int64_t r0 = blk0(kp);
    const int w = blkw(kp);
    const int64_t blk = (int64_t)(FWD ? kp : nb - 1 - kp) * TS * TS;
    if (tid == 0) mbar_expect_tx(&full[0], (kp >= 1 ? 2u : 1u) * TS * TS * 8);
    if (tid < TS) {
      bulk_g2s(dtile + tid * TS_P, P.dinv + blk + tid * TS, TS * 8, &full[0]);
      if (kp >= 1) bulk_g2s(wtile + tid * TS_P, P.wmat + blk + tid * TS, TS * 8, &full[0]);
      if constexpr (R == 1) {
        bs[tid] = (tid < w) ? P.b[r0 + tid] : 0.0;
      } else {
#pragma unroll
        for (int c = 0; c < R; ++c) bs[c * TS + tid] = (tid < w) ? P.b[c * P.ld + r0 + tid] : 0.0;
      }
    }
  };

  // Product of a staged 64 x 64 block `T` (pitch TS_P) with `xvec` in the chain step: forward sum_c T[r][c] x[c] for
  // row r, backward sum_r T[r][c] x[r] for column c.  The result is returned in the register of the element's
  // OWNER thread (forward: the q == 0 lane of row r = tid / 4; backward: thread tid < 64 for column tid).
  const bool owner = FWD ? ((tid & 3) == 0) : (tid < TS);
  const int idx = FWD ? (tid >> 2) : tid;
  auto matvec = [&](const double* T, const double* xvec, int rows_valid) -> double {
    if (FWD) {
      const int r = tid >> 2, q = tid & 3;
      const double* row = T + r * TS_P + q * 16;
      const double* xv = xvec + q * 16;
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        const int c0 = (i + (q & 1)) & 15, c1 = (i + 1 + (q & 1)) & 15;   // rotation: conflict-free LDS.64
        const int c2 = (i + 2 + (q & 1)) & 15, c3 = (i + 3 + (q & 1)) & 15;
        s0 = fma(row[c0], xv[c0], s0);
        s1 = fma(row[c1], xv[c1], s1);
        s2 = fma(row[c2], xv[c2], s2);
        s3 = fma(row[c3], xv[c3], s3);
      }
      double sv = (s0 + s1) + (s2 + s3);
      sv += __shfl_xor_sync(0xffffffffu, sv, 1);
      sv += __shfl_xor_sync(0xffffffffu, sv, 2);
      return sv;
    } else {
      const int cc = tid & 63, q = tid >> 6;
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
      for (int i = 0; i < 16; i += 4) {
        const int r0 = q * 16 + i;
        if (r0 < rows_valid) s0 = fma(T[r0 * TS_P + cc], xvec[r0], s0);
        if (r0 + 1 < rows_valid) s1 = fma(T[(r0 + 1) * TS_P + cc], xvec[r0 + 1], s1);
        if (r0 + 2 < rows_valid) s2 = fma(T[(r0 + 2) * TS_P + cc], xvec[r0 + 2], s2);
        if (r0 + 3 < rows_valid) s3 = fma(T[(r0 + 3) * TS_P + cc], xvec[r0 + 3], s3);
      }
      red[q * TS + cc] = (s0 + s1) + (s2 + s3);
      __syncthreads();
      const double sv = (tid < TS) ? (red[tid] + red[TS + tid]) + (red[2 * TS + tid] + red[3 * TS + tid]) : 0.0;
      __syncthreads();                             // red may be rewritten by the next product
      return sv;
    }
  };

  uint32_t dphase = 0;
  // Chain step of slab index ms (block kp): x_k = D_k (b_k - acc) - W_k x_{k-1}.  The first term is formed before
  // x_{k-1} is waited for; between "x_{k-1} seen" and "x_k published" there is one mat-vec.
  auto chain_step = [&](int ms) {
    const int kp = c + ms * G;
    const int64_t r0 = blk0(kp);
    const int w = blkw(kp);
    __syncthreads();                               // every warp has booked its part of acc
    if constexpr (R == 1) {
      if (owner) {
        double a;
        if (FWD) {
          a = acc[ms * TS + idx];
        } else {                                     // the eight warps' partial sums, in a fixed order
          const double* p = acc + ms * 8 * TS + idx;
          a = ((p[0] + p[TS]) + (p[2 * TS] + p[3 * TS])) + ((p[4 * TS] + p[5 * TS]) + (p[6 * TS] + p[7 * TS]));
        }
        vs[idx] = (idx < w) ? bs[idx] - a : 0.0;
      }
      mbar_wait(&full[0], dphase);
      dphase ^= 1;
      __syncthreads();
      double xv = matvec(dtile, vs, TS);
      double* xc = xh + ((ms & 1) * TS_HAND + 0) * TS;   // hand-over buffer of this slab, distance 1
      if (kp >= 1) {
        if (fed_by_prev_local) {
          if (tid < TS) {                            // the peer stores the 64 unknowns straight into xc
            unsigned spins = 0;
            while (unpublished(ld_shared_relaxed_f64(xc + tid))) {
              if (++spins > (1u << 26)) { atomicExch(&g_tgp_device_error, 2); break; }
            }
          }
        } else {
          const double* src = P.xpub + (int64_t)(kp - 1) * TS;
          if (tid < TS) {
            double v = ld_relaxed_f64(src + tid);
            unsigned spins = 0;
            while (unpublished(v)) {
              if (++spins > (1u << 25)) { atomicExch(&g_tgp_device_error, 1); break; }
              v = ld_relaxed_f64(src + tid);
            }
            xc[tid] = v;
          }
        }
        __syncthreads();
        TRSV_STAMP(kp, 0);
        xv -= matvec(wtile, xc, FWD ? TS : blkw(kp - 1));
      }
      if (owner) {
        if (unpublished(xv)) xv = __longlong_as_double(0x7ff8000000000000ll);   // never publish the sentinel
  #pragma unroll
        for (int d = 1; d <= TS_HAND; ++d) {         // first the hops that are on (or next to) the serial chain
          if (local_to(d) && kp + d < nb) {
            // the peer's slab kp + d is its slab number (kp + d) / G: that parity selects its buffer set
            double* dst = xh + ((((kp + d) / G) & 1) * TS_HAND + (d - 1)) * TS + idx;
            st_remote_f64(map_to_cta(smem_addr(dst), (uint32_t)(peer_ahead(d) % CS)), xv);
          }
        }
        st_relaxed_f64(P.xpub + (int64_t)kp * TS + idx, xv);
        if (idx < w) P.b[r0 + idx] = xv;
      }
    } else {
      if (owner) {
  #pragma unroll
        for (int c = 0; c < R; ++c) {
          double a;
          if (FWD) {
            a = acc[(ms * R + c) * TS + idx];
          } else {                                   // the eight warps' partial sums, in a fixed order
            const double* p = acc + (ms * 8 * R + c) * TS + idx;
            constexpr int W = R * TS;                // from one warp's partials to the next
            a = ((p[0] + p[W]) + (p[2 * W] + p[3 * W])) + ((p[4 * W] + p[5 * W]) + (p[6 * W] + p[7 * W]));
          }
          vs[c * TS + idx] = (idx < w) ? bs[c * TS + idx] - a : 0.0;
        }
      }
      mbar_wait(&full[0], dphase);
      dphase ^= 1;
      __syncthreads();
      double xv[R];
  #pragma unroll
      for (int c = 0; c < R; ++c) xv[c] = matvec(dtile, vs + c * TS, TS);
      double* xc = xh + ((ms & 1) * TS_HAND + 0) * TS * R;   // hand-over buffer of this slab, distance 1
      if (kp >= 1) {
        if (fed_by_prev_local) {
          if (tid < TS) {                            // the peer stores the 64 unknowns straight into xc
  #pragma unroll
            for (int c = 0; c < R; ++c) {
              unsigned spins = 0;
              while (unpublished(ld_shared_relaxed_f64(xc + c * TS + tid))) {
                if (++spins > (1u << 26)) { atomicExch(&g_tgp_device_error, 2); break; }
              }
            }
          }
        } else {
          const double* src = P.xpub + (int64_t)(kp - 1) * TS * R;
          if (tid < TS) {
  #pragma unroll
            for (int c = 0; c < R; ++c) {
              double v = ld_relaxed_f64(src + c * TS + tid);
              unsigned spins = 0;
              while (unpublished(v)) {
                if (++spins > (1u << 25)) { atomicExch(&g_tgp_device_error, 1); break; }
                v = ld_relaxed_f64(src + c * TS + tid);
              }
              xc[c * TS + tid] = v;
            }
          }
        }
        __syncthreads();
        TRSV_STAMP(kp, 0);
  #pragma unroll
        for (int c = 0; c < R; ++c) xv[c] -= matvec(wtile, xc + c * TS, FWD ? TS : blkw(kp - 1));
      }
      if (owner) {
  #pragma unroll
        for (int c = 0; c < R; ++c) {
          if (unpublished(xv[c])) xv[c] = __longlong_as_double(0x7ff8000000000000ll);   // never publish the sentinel
  #pragma unroll
          for (int d = 1; d <= TS_HAND; ++d) {       // first the hops that are on (or next to) the serial chain
            if (local_to(d) && kp + d < nb) {
              // the peer's slab kp + d is its slab number (kp + d) / G: that parity selects its buffer set
              double* dst = xh + ((((kp + d) / G) & 1) * TS_HAND + (d - 1)) * TS * R + c * TS + idx;
              st_remote_f64(map_to_cta(smem_addr(dst), (uint32_t)(peer_ahead(d) % CS)), xv[c]);
            }
          }
          st_relaxed_f64(P.xpub + (int64_t)kp * TS * R + c * TS + idx, xv[c]);
          if (idx < w) P.b[c * P.ld + r0 + idx] = xv[c];
        }
      }
    }
    TRSV_STAMP(kp, 2);
    __syncthreads();                               // dtile, wtile, bs, vs, xc are free again
    // re-arm this slab's hand-over buffer: the next store into it (slab ms + 2) causally follows the publication of
    // slab ms + 1 by this CTA, which follows this line in program order
    if (CS > 1) {
      double* mine = xh + (ms & 1) * TS_HAND * TS * R;
      for (int i = tid; i < TS_HAND * TS * R; i += TS_THREADS) mine[i] = __longlong_as_double(-1ll);
    }
    prefetch_solve(ms + 1);
  };

  // ---- streaming part: one (slab, window) visit per warp, straight from global memory into registers ----------
  // Forward: the warp owns rows 8 warp .. 8 warp + 7 of every slab; a lane reads the 16-byte column pair 2 lane,
  // 2 lane + 1 of each 64-column block of the window (512 contiguous bytes per instruction, up to 2 KB per row)
  // and the eight row sums are completed with shuffles.  Backward (transposed product): the warp owns every
  // eighth row of the window's blocks, a lane accumulates the two columns 2 lane, 2 lane + 1 of the slab -- no
  // shuffles; the eight warps' partial sums stay separate in shared memory until the chain step.
  auto visit_fwd = [&](int m, int j0, int cnt) {
    const int kp = c + m * G;
    const int64_t r0 = blk0(kp) + warp * 8;
    const double* base = P.L + r0 * ld + (int64_t)j0 * TS + 2 * lane;
    double2 v[8][TS_WIN];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int g = 0; g < TS_WIN; ++g)
        v[i][g] = (g < cnt && r0 + i < N) ? ldg2(base + (int64_t)i * ld + g * TS, vec) : make_double2(0.0, 0.0);
    if constexpr (R == 1) {
      double s[8];
  #pragma unroll
      for (int i = 0; i < 8; ++i) {
        double a0 = 0.0, a1 = 0.0;
  #pragma unroll
        for (int g = 0; g < TS_WIN; ++g) {
          if (g < cnt) {
            a0 = fma(v[i][g].x, xs[g * TS + 2 * lane], a0);
            a1 = fma(v[i][g].y, xs[g * TS + 2 * lane + 1], a1);
          }
        }
        s[i] = a0 + a1;
      }
  #pragma unroll
      for (int o = 16; o > 0; o >>= 1)
  #pragma unroll
        for (int i = 0; i < 8; ++i) s[i] += __shfl_xor_sync(0xffffffffu, s[i], o);
      if (lane < 8) {
        double sv = s[0];
  #pragma unroll
        for (int i = 1; i < 8; ++i) sv = (lane == i) ? s[i] : sv;
        acc[m * TS + warp * 8 + lane] += sv;
      }
    } else {
  #pragma unroll
      for (int c = 0; c < R; ++c) {                  // the rows are read once; the columns are accumulated one by one
        double s[8];
  #pragma unroll
        for (int i = 0; i < 8; ++i) {
          double a0 = 0.0, a1 = 0.0;
  #pragma unroll
          for (int g = 0; g < TS_WIN; ++g) {
            if (g < cnt) {
              a0 = fma(v[i][g].x, xs[(g * R + c) * TS + 2 * lane], a0);
              a1 = fma(v[i][g].y, xs[(g * R + c) * TS + 2 * lane + 1], a1);
            }
          }
          s[i] = a0 + a1;
        }
  #pragma unroll
        for (int o = 16; o > 0; o >>= 1)
  #pragma unroll
          for (int i = 0; i < 8; ++i) s[i] += __shfl_xor_sync(0xffffffffu, s[i], o);
        if (lane < 8) {
          double sv = s[0];
  #pragma unroll
          for (int i = 1; i < 8; ++i) sv = (lane == i) ? s[i] : sv;
          acc[(m * R + c) * TS + warp * 8 + lane] += sv;
        }
      }
    }
  };
  auto visit_bwd = [&](int m, int j0, int cnt) {
    const int kp = c + m * G;
    const int64_t c0 = blk0(kp) + 2 * lane;          // the slab's columns
    if constexpr (R == 1) {
      double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0;
      for (int g = 0; g < cnt; ++g) {
        const int64_t rb = blk0(j0 + g);               // rows of window block g (primed j0 + g)
        const int rows = blkw(j0 + g);
        double2 v[8];
  #pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = warp * 8 + i;
          v[i] = (r < rows) ? ldg2(P.L + (rb + r) * ld + c0, vec) : make_double2(0.0, 0.0);
        }
  #pragma unroll
        for (int i = 0; i < 8; i += 2) {
          const double x0 = xs[g * TS + warp * 8 + i], x1 = xs[g * TS + warp * 8 + i + 1];
          a0 = fma(v[i].x, x0, a0);
          a1 = fma(v[i].y, x0, a1);
          b0 = fma(v[i + 1].x, x1, b0);
          b1 = fma(v[i + 1].y, x1, b1);
        }
      }
      double* p = acc + (m * 8 + warp) * TS + 2 * lane;
      p[0] += a0 + b0;
      p[1] += a1 + b1;
    } else {
      double a0[R], a1[R], b0[R], b1[R];
  #pragma unroll
      for (int c = 0; c < R; ++c) a0[c] = a1[c] = b0[c] = b1[c] = 0.0;
      for (int g = 0; g < cnt; ++g) {
        const int64_t rb = blk0(j0 + g);               // rows of window block g (primed j0 + g)
        const int rows = blkw(j0 + g);
        double2 v[8];
  #pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = warp * 8 + i;
          v[i] = (r < rows) ? ldg2(P.L + (rb + r) * ld + c0, vec) : make_double2(0.0, 0.0);
        }
  #pragma unroll
        for (int c = 0; c < R; ++c) {
          const double* xg = xs + (g * R + c) * TS + warp * 8;
  #pragma unroll
          for (int i = 0; i < 8; i += 2) {
            const double x0 = xg[i], x1 = xg[i + 1];
            a0[c] = fma(v[i].x, x0, a0[c]);
            a1[c] = fma(v[i].y, x0, a1[c]);
            b0[c] = fma(v[i + 1].x, x1, b0[c]);
            b1[c] = fma(v[i + 1].y, x1, b1[c]);
          }
        }
      }
  #pragma unroll
      for (int c = 0; c < R; ++c) {
        double* p = acc + ((m * 8 + warp) * R + c) * TS + 2 * lane;
        p[0] += a0[c] + b0[c];
        p[1] += a1[c] + b1[c];
      }
    }
  };

  // L2 prefetch of the 64-row tiles of slab index ms against column blocks j0 .. j0 + cnt - 1: near the chain front
  // a tile is needed the moment its unknowns appear, and an HBM round trip would then sit on the serial chain
  auto prefetch_l2 = [&](int ms, int j0, int cnt) {
    const int kp = c + ms * G;
    if (FWD) {
      const int rows = blkw(kp);
      const int lines = cnt * 4;                   // 128-byte lines per row
      for (int i = tid; i < rows * lines; i += TS_THREADS) {
        const double* p = P.L + (blk0(kp) + i / lines) * ld + (int64_t)j0 * TS + (i % lines) * 16;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
      }
    } else {
      for (int i = tid; i < cnt * TS * 4; i += TS_THREADS) {
        const int g = i / (TS * 4), r = (i / 4) % TS;
        if (r < blkw(j0 + g)) {
          const double* p = P.L + (blk0(j0 + g) + r) * ld + blk0(kp) + (i % 4) * 16;
          asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
        }
      }
    }
  };
  // fetch the unknowns of column blocks j0 .. j0 + cnt - 1 into xs (urgent: all 64 threads poll from the start)
  auto fetch_window = [&](int j0, int cnt, bool urgent) {
    __syncthreads();                               // everyone is done with the previous window
    if constexpr (R == 1) {
      const double* src = P.xpub + (int64_t)j0 * TS;
      if (!urgent) {
        if (tid == 0) {                              // blocks are published in order: wait for the last one, lazily
          unsigned spins = 0;
          while (unpublished(ld_relaxed_f64(src + (cnt - 1) * TS))) {
            if (spins > 16u) __nanosleep(32);
            if (++spins > (1u << 23)) { atomicExch(&g_tgp_device_error, 1); break; }
          }
        }
        __syncthreads();
      }
      if (tid < cnt * TS) {
        double v = ld_relaxed_f64(src + tid);
        unsigned spins = 0;
        while (unpublished(v)) {
          if (++spins > (1u << 25)) { atomicExch(&g_tgp_device_error, 1); break; }
          v = ld_relaxed_f64(src + tid);
        }
        if (!FWD && (tid & 63) >= blkw(j0 + (tid >> 6))) v = 0.0;    // padding rows of a short block
        xs[tid] = v;
      }
      __syncthreads();
    } else {
      const double* src = P.xpub + (int64_t)j0 * TS * R;
      if (!urgent) {
        if (tid == 0) {                              // blocks are published in order: wait for the last one, lazily
          unsigned spins = 0;
          while (unpublished(ld_relaxed_f64(src + (cnt - 1) * TS * R))) {
            if (spins > 16u) __nanosleep(32);
            if (++spins > (1u << 23)) { atomicExch(&g_tgp_device_error, 1); break; }
          }
        }
        __syncthreads();
      }
      for (int i = tid; i < cnt * TS * R; i += TS_THREADS) {
        double v = ld_relaxed_f64(src + i);
        unsigned spins = 0;
        while (unpublished(v)) {
          if (++spins > (1u << 25)) { atomicExch(&g_tgp_device_error, 1); break; }
          v = ld_relaxed_f64(src + i);
        }
        if (!FWD && (i & 63) >= blkw(j0 + i / (TS * R))) v = 0.0;    // padding rows of a short block
        xs[i] = v;
      }
      __syncthreads();
    }
  };

  // the unknowns of the block at distance d before slab index ms's diagonal, handed over by a cluster peer
  auto fetch_handover = [&](int ms, int d) {
    __syncthreads();                               // everyone is done with the previous window
    if constexpr (R == 1) {
      const double* src = xh + ((ms & 1) * TS_HAND + (d - 1)) * TS;
      if (tid < TS) {
        unsigned spins = 0;
        double v = ld_shared_relaxed_f64(src + tid);
        while (unpublished(v)) {
          if (++spins > (1u << 26)) { atomicExch(&g_tgp_device_error, 2); break; }
          v = ld_shared_relaxed_f64(src + tid);
        }
        xs[tid] = v;                                 // (a short block's padding rows are published as zeros)
      }
    } else {
      const double* src = xh + ((ms & 1) * TS_HAND + (d - 1)) * TS * R;
      for (int i = tid; i < TS * R; i += TS_THREADS) {
        unsigned spins = 0;
        double v = ld_shared_relaxed_f64(src + i);
        while (unpublished(v)) {
          if (++spins > (1u << 26)) { atomicExch(&g_tgp_device_error, 2); break; }
          v = ld_shared_relaxed_f64(src + i);
        }
        xs[i] = v;                                   // (a short block's padding rows are published as zeros)
      }
    }
    __syncthreads();
  };

  prefetch_solve(0);
  __syncthreads();

  // Progress: column blocks < j_rest are applied to every unsolved slab; the slab whose chain step comes next
  // ("urgent", index ms_next) may be ahead, at j_urg >= j_rest: within TS_NEAR blocks of its own diagonal it is fed
  // one block at a time, as soon as that block's unknowns exist and before the CTA's other slabs, so that it is
  // already waiting when the unknowns of the last block before its diagonal are published.
  int ms_next = 0;
  int j_rest = 0, j_urg = 0;
  for (;;) {
    if (ms_next >= M) break;
    const int k_next = c + ms_next * G;
    if (j_urg >= k_next - 1) {                     // blocks 0 .. k_next - 2 are in: the slab's chain step is due
      chain_step(ms_next);
      ++ms_next;
      j_urg = j_rest;
      continue;
    }
    const int left = k_next - 1 - j_urg;           // blocks still to apply to the urgent slab, >= 1
    if (left <= TS_NEAR) {
      if (left == TS_NEAR || j_urg == j_rest) prefetch_l2(ms_next, j_urg, left);
      if (left + 1 <= TS_HAND && local_from(left + 1)) {   // block j_urg sits left + 1 blocks before the slab's diagonal
        fetch_handover(ms_next, left + 1);
      } else {
        fetch_window(j_urg, 1, true);
      }
      if (FWD) visit_fwd(ms_next, j_urg, 1); else visit_bwd(ms_next, j_urg, 1);
      ++j_urg;
      continue;
    }
    // far from any diagonal of ours: a window of up to TS_WIN blocks for all unsolved slabs
    int cnt = left - TS_NEAR;
    cnt = cnt < TS_WIN ? cnt : TS_WIN;
    fetch_window(j_rest, cnt, false);
    for (int m = ms_next; m < M; ++m) {
      if (FWD) visit_fwd(m, j_rest, cnt); else visit_bwd(m, j_rest, cnt);
    }
    j_rest += cnt;
    j_urg = j_rest;
  }
  if (CS > 1) cluster_sync_all();                  // shared memory of a CTA stays valid while peers may still write
}

static size_t trsv_smem_bytes(bool fwd, int slabs_per_cta, int R = 1) {
  return (size_t)2 * TS_TILE_D * 8 + (size_t)((TS_WIN * TS + 2 * TS_HAND * TS + 2 * TS) * R + 4 * TS) * 8 + 2 * 8 +
         (size_t)slabs_per_cta * TS * 8 * (fwd ? 1 : 8) * R;
}

static bool g_clusters_refused = false;   // set when a cooperative launch with clusters is refused: none from then on

// CTAs of one cooperative launch: as many as are co-resident (one per SM: the kernel takes most of the shared
// memory), in clusters of CS when a cluster size is in use.
template <bool FWD, int R>
static int trsv_grid(int nb, int cs, size_t smem) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)cs);
  cfg.blockDim = dim3(TS_THREADS);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)cs;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  int nclusters = 0;
  if (cudaOccupancyMaxActiveClusters(&nclusters, trsv_sweep_kernel<FWD, R>, &cfg) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int g = nclusters * cs;
  const int want = (nb / cs) * cs;
  return g < want ? g : want;
}

template <bool FWD, int R>
static void trsv_max_smem() {
  static TgpPerDeviceOnce once;
  if (tgp_first_use_on_device(once))
    cudaFuncSetAttribute(trsv_sweep_kernel<FWD, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

// Grid of the single right-hand-side sweep: cluster size CS and CTA count G.
template <bool FWD>
static void trsv_config(const TrsvParams& P, int& cs, int& G) {
  trsv_max_smem<FWD, 1>();
  // cluster size: the largest of 8 / 4 / 2 that still keeps (nearly) all SMs busy; none for tiny matrices
  cs = 1;
  G = P.G;
  const size_t smem1 = trsv_smem_bytes(FWD, (P.nb + P.G - 1) / P.G);
  if (!g_clusters_refused && P.nb >= 4) {
    for (const int c2 : {8, 4, 2}) {
      if (P.nb < c2) continue;
      const int g = trsv_grid<FWD, 1>(P.nb, c2, smem1 + 4096);
      if (g >= c2 && 10 * g >= 9 * (P.nb < P.G ? (P.nb / c2) * c2 : P.G)) {
        cs = c2;
        G = g;
        break;
      }
    }
  }
}

// R > 1 runs on exactly the grid of R = 1 (the caller checks trsv_fits first): the slabs, their windows and hence every
// column's order of accumulation are those of the single right-hand-side sweep.
template <bool FWD, int R>
static int trsv_launch(const TrsvParams& P0, cudaStream_t st) {
  TrsvParams P = P0;
  int cs, G;
  trsv_config<FWD>(P, cs, G);
  P.CS = cs;
  P.G = G;
  const size_t smem = trsv_smem_bytes(FWD, (P.nb + P.G - 1) / P.G, R);
  if (R > 1) trsv_max_smem<FWD, R>();
  TGP_CHECK_ARG(smem <= 227 * 1024, "matrix too large for the sweep kernel's per-CTA accumulators");
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)P.G);
  cfg.blockDim = dim3(TS_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeCooperative;
  at[0].val.cooperative = 1;
  at[1].id = cudaLaunchAttributeClusterDimension;
  at[1].val.clusterDim.x = (unsigned)cs;
  at[1].val.clusterDim.y = 1;
  at[1].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = cs > 1 ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, trsv_sweep_kernel<FWD, R>, P);
  if (e != cudaSuccess && cs > 1) {                // clusters + cooperative launch refused: go on without clusters
    cudaGetLastError();
    g_clusters_refused = true;
    return trsv_launch<FWD, R>(P0, st);
  }
  TGP_CUDA(e);
  return TGP_OK;
}

// Library-private stream-ordered pool (one per device) that keeps what it was given: the sweeps' workspace is
// allocated and freed on the caller's stream at every call without going back to the driver.
static cudaMemPool_t trsv_pool() {
  static cudaMemPool_t pools[TGP_MAX_DEVICES] = {};
  const int dev = tgp_current_device();
  if (!pools[dev]) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t p = nullptr;
    if (cudaMemPoolCreate(&p, &props) != cudaSuccess) return nullptr;
    uint64_t keep = UINT64_MAX;
    cudaMemPoolSetAttribute(p, cudaMemPoolAttrReleaseThreshold, &keep);
    pools[dev] = p;
  }
  return pools[dev];
}

// Can R columns run on the grid of the single-column sweep (shared memory, co-residency)?
template <bool FWD, int R>
static bool trsv_fits(const TrsvParams& P) {
  int cs, G;
  trsv_config<FWD>(P, cs, G);
  const size_t smem = trsv_smem_bytes(FWD, (P.nb + G - 1) / G, R);
  if (smem > 227 * 1024) return false;
  trsv_max_smem<FWD, R>();
  return trsv_grid<FWD, R>(P.nb, cs, smem) >= G;
}

template <bool FWD>
static bool trsv_fits_r(const TrsvParams& P, int R) {
  switch (R) {
    case 2: return trsv_fits<FWD, 2>(P);
    case 4: return trsv_fits<FWD, 4>(P);
    case 8: return trsv_fits<FWD, 8>(P);
    default: return true;
  }
}

template <bool FWD>
static int trsv_launch_r(const TrsvParams& P, int R, cudaStream_t st) {
  switch (R) {
    case 1: return trsv_launch<FWD, 1>(P, st);
    case 2: return trsv_launch<FWD, 2>(P, st);
    case 4: return trsv_launch<FWD, 4>(P, st);
    default: return trsv_launch<FWD, 8>(P, st);
  }
}

// Workspace layout: [nb * 4096 doubles: inverse diagonal blocks][nb * 4096: W (forward)][nb * 4096: M (backward)]
// [2 * nb * 64 * Rmax doubles: published unknowns of the forward and of the backward sweep, filled with 0xFF bytes =
// "not yet published"][Rmax * ld: the right-hand sides of a multi-column sweep, padded with zero columns].
// which = 1: forward only, 2: backward only, 3: both (forward then backward).
// r columns b + c ld (c < r <= TGP_MAX_RHS) are swept in groups of R = 8, 4 or 2 columns (the largest that holds them
// and fits the single-column grid, else fewer), one column at a time when r == 1.  The diagonal-block inverses are
// computed once for all of them.
static int trsv_sweeps_impl(const double* L, int64_t N, int64_t ld, double* b, int r, int which, cudaStream_t st) {
  if (N <= 0) return TGP_OK;
  const int nb = (int)tgp_cdiv(N, TS);
  const int sms = tgp_num_sms();
  TrsvParams P;
  P.L = L; P.ld = ld; P.N = N; P.b = b; P.nb = nb;
  P.G = nb < sms ? nb : sms;
  P.CS = 1;
  P.aligned = ((ld & 1) == 0) && ((((uintptr_t)L) & 15) == 0);
  int rmax = 1;
  while (rmax < r) rmax *= 2;
  const size_t blk_d = (size_t)nb * TS * TS;
  const size_t pub_d = (size_t)2 * nb * TS * rmax;
  const size_t rhs_d = rmax > 1 ? (size_t)rmax * ld : 0;
  cudaMemPool_t pool = trsv_pool();
  if (!pool) {
    tgp_set_error("tgp_trsv_sweeps: cudaMemPoolCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
    return TGP_ERR_CUDA;
  }
  void* ws = nullptr;
  TGP_CUDA(cudaMallocFromPoolAsync(&ws, (3 * blk_d + pub_d + rhs_d) * sizeof(double), pool, st));
  double* dinv = reinterpret_cast<double*>(ws);
  double* wf = dinv + blk_d;
  double* wb = wf + blk_d;
  double* xpub = wb + blk_d;
  double* rhs = xpub + pub_d;
  int rc = TGP_OK;
  do {
    static TgpPerDeviceOnce prep_once;
    if (tgp_first_use_on_device(prep_once) &&
        cudaFuncSetAttribute(trsv_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TP_SMEM) != cudaSuccess) {
      rc = TGP_ERR_CUDA;
      break;
    }
    trsv_prep_kernel<<<(unsigned)nb, 256, TP_SMEM, st>>>(L, ld, N, nb, dinv, (which & 1) ? wf : nullptr,
                                                         (which & 2) ? wb : nullptr);
    if (cudaGetLastError() != cudaSuccess) { rc = TGP_ERR_CUDA; break; }
    P.dinv = dinv;
    // the widest group of columns whose sweeps run on the single-column grid
    int rfit = rmax;
    while (rfit > 1 && !(((which & 1) == 0 || trsv_fits_r<true>(P, rfit)) &&
                         ((which & 2) == 0 || trsv_fits_r<false>(P, rfit))))
      rfit /= 2;
    for (int c0 = 0, R = 1; c0 < r; c0 += R) {
      R = 1;
      while (R < r - c0 && R < rfit) R *= 2;
      const int nc = (r - c0 < R) ? r - c0 : R;
      if (R > 1) {                                 // the group's columns, padded with zero columns, at pitch ld
        if (cudaMemsetAsync(rhs, 0, (size_t)R * ld * sizeof(double), st) != cudaSuccess ||
            cudaMemcpy2DAsync(rhs, ld * sizeof(double), b + (size_t)c0 * ld, ld * sizeof(double), N * sizeof(double),
                              nc, cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
          rc = TGP_ERR_CUDA;
          break;
        }
      }
      P.b = R > 1 ? rhs : b + (size_t)c0 * ld;
#ifdef TGP_TRSV_TIMING
      // which & 4 (debug): pretend every block is already published -> no dependency waits, pure streaming rate
      if (cudaMemsetAsync(xpub, (which & 4) ? 0 : 0xFF, pub_d * sizeof(double), st) != cudaSuccess) { rc = TGP_ERR_CUDA; break; }
#else
      if (cudaMemsetAsync(xpub, 0xFF, pub_d * sizeof(double), st) != cudaSuccess) { rc = TGP_ERR_CUDA; break; }
#endif
      if (which & 1) {
        P.wmat = wf;
        P.xpub = xpub;
        rc = trsv_launch_r<true>(P, R, st);
        if (rc) break;
      }
      if (which & 2) {
        P.wmat = wb;
        P.xpub = xpub + (size_t)nb * TS * R;
        rc = trsv_launch_r<false>(P, R, st);
        if (rc) break;
      }
      if (R > 1 && cudaMemcpy2DAsync(b + (size_t)c0 * ld, ld * sizeof(double), rhs, ld * sizeof(double),
                                     N * sizeof(double), nc, cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
        rc = TGP_ERR_CUDA;
        break;
      }
    }
  } while (0);
  if (rc == TGP_ERR_CUDA) tgp_set_error("tgp_trsv_sweeps: %s", cudaGetErrorString(cudaGetLastError()));
  cudaFreeAsync(ws, st);
  return rc;
}

int tgp_trsv_sweeps(const double* L, int64_t N, int64_t ld, double* b, int which, cudaStream_t st) {
  return trsv_sweeps_impl(L, N, ld, b, 1, which, st);
}

// r right-hand sides b + c ld, c < r (1 <= r <= TGP_MAX_RHS): one pass over the factor per group of columns.
int tgp_trsv_sweeps_multi(const double* L, int64_t N, int64_t ld, double* b, int r, int which, cudaStream_t st) {
  return trsv_sweeps_impl(L, N, ld, b, r, which, st);
}

#ifdef TGP_TRSV_TIMING
extern "C" int tgp_trsv_only(const double* L, int64_t N, int64_t ld, double* b, int which, void* stream) {
  return tgp_trsv_sweeps(L, N, ld, b, which, (cudaStream_t)stream);
}
#endif
