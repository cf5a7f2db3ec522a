// Two-point correlation function by brute-force pair binning.
//
// Replaces the TreeCorr call of /root/reference/treegp/two_pcf.py:297-305 (KKCorrelation,
// bin_type="TwoD", bin_slop=0) and :330-338 (default Log binning, meanr), and -- launched over a batch
// of resampled catalogues -- the bootstrap loop of two_pcf.py:342-362.
//
// TreeCorr itself is not vendored in the reference; the semantics implemented here are the ones
// restated in oracle/pairbin_oracle.c (documented TreeCorr >= 4.2 behaviour, SURVEY.md section 8c):
//   TwoD: keep a pair iff r2 != 0, r2 >= min_sep^2 and max(|dx|,|dy|) < max_sep; column
//         floor((dx+max_sep)/bin_size), row floor((dy+max_sep)/bin_size); each unordered pair is entered
//         at (dx,dy) and at (-dx,-dy).
//   Log : keep iff min_sep^2 <= r2 < max_sep^2; bin floor((0.5 ln r2 - ln min_sep)/bin_size); once per
//         unordered pair; also accumulates sum w r for meanr.
// Bin decisions are made by comparing against host-supplied *thresholds* (the smallest double that
// the formula above sends to bin >= k), so counts are bit-exact with the oracle without FP64
// division or logarithms on the device; r2 is formed with un-fused mul/add for the same reason.
//
// Kernel shape (warp-centric, no CTA barriers in the main loop).  The pair matrix is cut into
// blocks of 32 row points x 32 column points.  A work item is one row block times a run of column
// chunks; warps of persistent CTAs pull items from a global counter (dynamic load balance: blocks
// that are provably out of range are skipped, so items differ in cost).  A lane owns one row point in
// registers; the warp stages one column chunk at a time in its private slice of shared memory and
// reads it back as broadcasts.
//
// TwoD with block forms runs as TWO kernels per round of items (tgp_pairbin): pairbin_classify_kernel classifies every
// block from the chunk boxes, books the closed-form blocks and records the others; pairbin_kernel<TwoD, W, true> then
// runs the paths below over the recorded blocks only.  The classification needs none of the per-row register state
// of the residual paths, so it runs at more warps per SM and the residual kernel's warm code no longer contains it.
// Before the rounds, pairbin_super_kernel books the pairs of super-chunks (PB_SUPER chunks) that are out of range, sit
// in one bin, or vary along one axis only (one rank query per row point on the super-chunk's sorted copy), and lists
// those that span at most 2 x 2 bins; pairbin_super_leaves_kernel decides the listed pairs in one launch, without
// records: per row point against the column super-chunk staged in shared memory (the list grouped by column
// super-chunk), or block by block.  The classification pass skips the blocks of all of them and descends to the
// 32-point blocks only for the other super pairs.
//
// Two instantiations per bin type (template parameter BS):
//   BS = false  the pair-by-pair kernel: every pair of every in-range block is evaluated individually
//               (tgp_set_option("pairbin_block_sums", 0)); the 10-FP64-ops-per-pair roofline is stated for it.
//               Blocks that provably sit in one bin per axis whose mirrored window is the mirror image skip the
//               per-pair mirrored bits (the forward bits are still evaluated for every pair).
//   BS = true   (default) block forms on top of the same classification, all exact (TwoD: pass B, see above):
//               * TwoD, block in ONE forward bin whose mirrored window is its mirror image: booked whole by the
//                 classifying lane from the chunk sums of the pre-pass (points never loaded);
//               * TwoD, one varying axis: rank query (4-ary search, 8 probes per row point) on the chunk's copy
//                 sorted along that axis with suffix sums (pre-pass); the exact mirrored bits need only the two
//                 neighbours of the split, a failed check hands the block back to the pair-by-pair loop.  Blocks
//                 that the open window already covers take a short cut in front of the general dispatch;
//               * TwoD, two bins along both axes: column-bit and row-bit sums from two rank queries on the x- and
//                 y-sorted copies, only the "both bits" quadrant summed per pair;
//               * Log, block in one radial bin or two adjacent ones: counts / k-sums from row and chunk sums,
//                 one square root per pair for sum w r, no atomics.
//
// For 32 chunks at a time each lane derives the bounding box of "its" chunk and classifies the
// block against the warp's row bounding box (FP subtraction is monotone, so the box gives exact bounds
// on dx, dy):
//   OUT        every pair fails the range test                          -> skipped, not even loaded
//   REG_FULL   every pair passes it and the displacements span <= 2 x 2 bins (both entries)
//   REG_CHECK  same window, range test needed per pair
//   GENERIC    wider window (unsorted input), Log bins, the diagonal block
// REG blocks accumulate in registers (see RegAcc): no atomics in the inner loop; the registers are
// flushed to the warp's private shared-memory histogram only when the window moves.  When the points
// are sorted along a Hilbert curve (tgp_hilbert_keys) nearly all blocks are REG; a GENERIC block is
// first retried as four 8-column sub-blocks.  The GENERIC path does a per-pair bin search and
// shared-memory atomics.  Histograms go to global memory with red.global when the warp changes
// catalogue.  Multi-GPU: items are dealt round-robin to ranks; the caller all-reduces the bin sums.
#include <float.h>
#include <math.h>
#include <atomic>
#include "tgp_common.cuh"

constexpr int PB_CHUNK = 32;          // column points per block (= row points per warp)
constexpr int PB_MAX_WARPS = 8;       // warps per CTA (each owns a private histogram)
constexpr int PB_FLUSH_ITEMS = 2048;  // keeps the 32-bit private counters from overflowing
constexpr int PB_SLOT = 8;            // doubles per chunk slot of the pre-pass: box + sums
constexpr int PB_SORTED = 6 * PB_CHUNK;  // + {sorted x, suffix k w, suffix w, sorted y, suffix k w, suffix w}
constexpr int PB_STRIDE = PB_SLOT + PB_SORTED;   // the two records of a chunk are stored back to back
// Super-chunks (TwoD block forms): PB_SUPER consecutive chunks of a catalogue, aligned to chunk 0.  Only full ones
// (PB_SUPER_PTS points) get a record: {box, sum k w, sum w, -, -} + the points sorted by x and by y, each with suffix
// sums of k w and w.  8 was the fastest admissible size at the bench size (DESIGN section 5, v10).
#ifndef PB_SUPER
#define PB_SUPER 8
#endif
constexpr int PB_SUPER_PTS = PB_SUPER * PB_CHUNK;
constexpr int PB_SUPER_STRIDE = PB_SLOT + 6 * PB_SUPER_PTS;
// the warp histogram of the super kernel takes <= 32 x PB_SUPER_PTS^2 pairs per item: flush before 2^31
constexpr int PB_SUPER_FLUSH_ITEMS = (int)((1u << 31) / (32u * PB_SUPER_PTS * PB_SUPER_PTS));

struct PBParams {
  const double *px, *py, *pk, *pw;
  const int64_t* cat_off;
  const double* edges;
  int64_t* npairs;
  double *sumw, *sumwkk, *sumwr;
  unsigned long long* counter;  // dynamic work counter (zeroed before the launch)
  const double* boxes;          // optional precomputed chunk boxes + sums (8 doubles per slot) or NULL
  const double* sorted;         // optional per-chunk sorted coordinates + suffix sums (PB_SORTED doubles per slot)
  double lo2;       // pairs need r2 >= lo2 (= max(min_sep^2, DBL_TRUE_MIN) for TwoD; min_sep^2 for Log)
  double hi;        // TwoD: max_sep (|dx|,|dy| < hi);  Log: max_sep^2 (r2 < hi)
  double inv_bin;   // TwoD: nbins / (2 max_sep)
  int64_t items_per_cat;  // upper bound from max_cat_len
  int64_t my_items;       // number of work items of this rank
  int32_t run;            // column chunks per work item (multiple of 32)
  int32_t ncat, nbins, nb, warps, rank, nranks;
  int32_t block_sums;     // 1: blocks whose pairs provably share a window bit use the block forms (default); 2 (TwoD
                          // classification pass only): and the super pairs that are not DESCEND go to the super kernel
  int32_t fast_paths;     // bit 0: short-cut dispatch of one-axis blocks that fit the open window; bit 1: 2 x 2-window
                          // blocks with marginal sums from rank queries; bit 2: pair-by-pair kernel, no mirrored bits
                          // per pair in blocks that provably sit in one bin and its mirror image (default: all)
  // TwoD block forms, two passes per round (pairbin_classify_kernel, then pairbin_kernel<TwoD, W, true>): this
  // round's items q in [q_begin, q_end) of this rank; the records of item q at recs + (q - q_begin) * run, their
  // number at rec_cnt[q - q_begin]; counter_next = the other pass's work counter, zeroed for its next launch
  int64_t q_begin, q_end;
  int4* recs;
  int* rec_cnt;
  unsigned long long* counter_next;
  unsigned long long* slist_len;   // super kernel / leaf kernel: length of the super pair list (pb_super_list)
  int32_t list_one_axis;           // super kernel: ONE_AXIS super pairs are listed for the staged leaf kernel (1) or
                                   // decided by the super kernel itself (0)
};

// Which path the pairs of all launches since the last reset took (in pairs): [0] closed form (block in one bin; TwoD:
// tallied by the classification pass, the others by the pass over the recorded blocks),
// [1] one varying axis, pair by pair, [2] pair by pair (2 x 2 window with or without the per-pair range test,
// generic sub-blocks), [3] one varying axis answered by a rank query on the sorted chunk, [4] 2 x 2 window with the
// marginal sums from rank queries (one quadrant pair by pair), [5] super pair in one bin, [6] super pair with one
// varying axis (rank queries on the super-chunk's sorted copy).  Diagnostics.
__device__ unsigned long long g_pb_stats[8];

__device__ __forceinline__ int pb_bin_twod(double d, double hi, double inv_bin, int nbins,
                                           const double* __restrict__ ed) {
  int i = (int)((d + hi) * inv_bin);
  i = max(0, min(i, nbins - 1));
  // exact fix-up: ed[0] = -inf, ed[nbins] = +inf, ed[k] = smallest d that belongs to bin >= k
  if (d < ed[i]) --i;
  else if (d >= ed[i + 1]) ++i;
  return i;
}

// Robust version for window end points (the estimate may be off by more than one there).
__device__ __forceinline__ int pb_bin_twod_search(double d, int nbins, const double* __restrict__ ed) {
  int lo = 0, hi = nbins - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (d >= ed[mid]) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// The same search out of line (rarely reached), and the bin of d given a guess g in [0, nbins-1]: two compares
// when the guess is right (ed[0] = -inf, ed[nbins] = +inf, thresholds ascending: the bin is unique).
__device__ __noinline__ int pb_bin_twod_search_cold(double d, int nbins, const double* ed) {
  return pb_bin_twod_search(d, nbins, ed);
}
__device__ __forceinline__ int pb_bin_twod_guess(double d, int g, int nbins, const double* __restrict__ ed) {
  if (d >= ed[g] && d < ed[g + 1]) return g;
  return pb_bin_twod_search_cold(d, nbins, ed);
}

__device__ __forceinline__ int pb_bin_log(double r2, int nbins, const double* __restrict__ ed) {
  // number of interior thresholds ed[1..nbins-1] that are <= r2 (binary search)
  int lo = 0, hi = nbins - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (r2 >= ed[mid]) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ unsigned warp_sum_u(unsigned v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Per-lane register accumulators of the 2 x 2 window.
// With px = "column bit" and py = "row bit" of a pair inside the window, the lane keeps
//   tot = sum kk,  sx = sum kk [px],  sy = sum kk [py],  sxy = sum kk [px & py]
// (masks applied as a multiplication by 0.0 / 1.0 inside one FMA: no branch, no 64-bit select) and the same
// three counters as integers; the four window bins follow by inclusion-exclusion at flush time (exact for
// the counts, of the size of ordinary summation rounding for the FP64 sums).
//
// Mirrored entry.  Every pair is also entered at (-dx,-dy).  The grid is point symmetric, so the mirrored
// bin of a pair is "almost always" the mirror image (nbins-1-ix, nbins-1-iy) of its forward bin; it can
// differ only when a displacement sits within rounding of a bin edge, because the thresholds of the
// TreeCorr formula are not exactly symmetric in floating point.  The window of the mirrored entry is
// therefore fixed to the mirror image of the forward window, the exact mirrored bits qx, qy are still
// evaluated for every pair, and `mmc` counts the pairs for which (qx, qy) != (!px, !py).  The forward
// registers are flushed into both the forward bins and their mirror images; blocks with mmc != 0 are
// rescanned and the (rare) inconsistent pairs moved from the assumed to the exact mirrored bin.
template <bool WEIGHTED>
struct RegAcc {
  double tot, fsx, fsy, fsxy;
  double wtot, fwx, fwy, fwxy;   // weights (WEIGHTED only)
  unsigned fcx, fcy, fcxy, nin, mmc;
  int fx0, fy0;              // forward window origin (bins); fx0 == -1: no open window.  Mirrored window
                             // origin: (nbins-2-fx0, nbins-2-fy0)
  long long ownerI;          // row block the per-lane thresholds were derived for
  double rki, rwi;           // this lane's row-point factors k_i w_i and w_i, applied to the sums at flush time
  // Per-lane thresholds on the COLUMN point's coordinates, equivalent to the bin thresholds on the
  // displacement because rounding is monotone:  fl(xj - xi) >= t  <=>  xj >= Tx(xi, t).
  double Tx, Ty, RTx, RTy;   // forward: px = xj >= Tx ; mirrored: qx = xj <= RTx
  __device__ __forceinline__ void zero() {
    tot = fsx = fsy = fsxy = 0.0;
    wtot = fwx = fwy = fwxy = 0.0;
    fcx = fcy = fcxy = nin = mmc = 0u;
  }
};

// Monotone map between doubles and signed integers (order-preserving; -0.0 and +0.0 share key 0).
__device__ __forceinline__ long long pb_key(double d) {
  const long long b = __double_as_longlong(d);
  return b >= 0 ? b : -(b & 0x7fffffffffffffffll);
}
__device__ __forceinline__ double pb_unkey(long long k) {
  return __longlong_as_double(k >= 0 ? k : (long long)(0x8000000000000000ull | (unsigned long long)(-k)));
}

// Smallest X with fl(X - xi) >= t.  X -> fl(X - xi) is monotone, so the answer is found by bisection over
// the ordered doubles inside a bracket of a few ulp(t) + ulp(t + xi) around t + xi.  `ok` is cleared if no
// bracket was found (the caller then uses the generic path).  NaN xi -> NaN (dead lanes: every comparison
// false); infinite t is returned unchanged (nbins == 1: the bit is constant).
__device__ __noinline__ double pb_coord_ge(double xi, double t, bool& ok) {
  if (isinf(t) || isnan(xi)) return isnan(xi) ? xi : t;
  const double c = t + xi;
  double e = (fabs(t) + fabs(c)) * 0x1p-50 + 0x1p-1060;
  double lo = c - e, hi = c + e;
  for (int it = 0; it < 8 && (!((hi - xi) >= t) || ((lo - xi) >= t)); ++it) { e *= 8.0; lo = c - e; hi = c + e; }
  if (!((hi - xi) >= t) || ((lo - xi) >= t)) { ok = false; return c; }
  long long klo = pb_key(lo), khi = pb_key(hi);  // pred(lo) false, pred(hi) true
  while (khi - klo > 1) {
    const long long mid = klo + ((khi - klo) >> 1);
    if ((pb_unkey(mid) - xi) >= t) khi = mid; else klo = mid;
  }
  return pb_unkey(khi);
}
// Largest X with fl(X - xi) <= t.
__device__ __noinline__ double pb_coord_le(double xi, double t, bool& ok) {
  if (isinf(t) || isnan(xi)) return isnan(xi) ? xi : t;
  const double c = t + xi;
  double e = (fabs(t) + fabs(c)) * 0x1p-50 + 0x1p-1060;
  double lo = c - e, hi = c + e;
  for (int it = 0; it < 8 && (!((lo - xi) <= t) || ((hi - xi) <= t)); ++it) { e *= 8.0; lo = c - e; hi = c + e; }
  if (!((lo - xi) <= t) || ((hi - xi) <= t)) { ok = false; return c; }
  long long klo = pb_key(lo), khi = pb_key(hi);  // pred(lo) true, pred(hi) false
  while (khi - klo > 1) {
    const long long mid = klo + ((khi - klo) >> 1);
    if ((pb_unkey(mid) - xi) <= t) klo = mid; else khi = mid;
  }
  return pb_unkey(klo);
}

// One pair into the window registers.  Written in PTX: four compares give the window bits of the
// forward entry and the exact bits of the mirrored entry, each masked sum is one FMA with a 0.0 / 1.0
// mask, each counter one predicated integer add (nvcc's code for the equivalent C++ needs ~2x the
// instructions; ptxas turns a predicated FP64 add into add + two selects, so the mask form is the shortest).
// What is summed is the COLUMN point's value k_j w_j (and w_j): the row point's factor k_i w_i (w_i) is
// constant for a lane while a window is open and is applied once, when the registers are flushed.
// TOT = "add.f64 tot, tot, kj" for blocks that need the range test per pair; blocks that are entirely in
// range add the chunk sum once instead.
#define PB_ONE "0d3FF0000000000000"
#define PB_ZERO "0d0000000000000000"
#define PB_PAIR_BODY(TOT)                                                                           \
      "{\n\t"                                                                                       \
      ".reg .pred px, py, qx, qy, pxy, cx, cy, mm;\n\t"                                             \
      ".reg .f64 m0, m1, m2;\n\t"                                                                   \
      "setp.ge.f64 px, %9, %11;\n\t"                                                                \
      "setp.ge.f64 py, %10, %12;\n\t"                                                               \
      "setp.le.f64 qx, %9, %13;\n\t"                                                                \
      "setp.le.f64 qy, %10, %14;\n\t"                                                               \
      "and.pred pxy, px, py;\n\t"                                                                   \
      "xor.pred cx, px, qx;\n\t"                                                                    \
      "xor.pred cy, py, qy;\n\t"                                                                    \
      "and.pred mm, cx, cy;\n\t"                                                                    \
      "not.pred mm, mm;\n\t"                                                                        \
      "selp.f64 m0, " PB_ONE ", " PB_ZERO ", px;\n\t"                                               \
      "selp.f64 m1, " PB_ONE ", " PB_ZERO ", py;\n\t"                                               \
      "selp.f64 m2, " PB_ONE ", " PB_ZERO ", pxy;\n\t"                                              \
      TOT                                                                                           \
      "fma.rn.f64 %1, %8, m0, %1;\n\t"                                                              \
      "fma.rn.f64 %2, %8, m1, %2;\n\t"                                                              \
      "fma.rn.f64 %3, %8, m2, %3;\n\t"                                                              \
      "@px add.u32 %4, %4, 1;\n\t"                                                                  \
      "@py add.u32 %5, %5, 1;\n\t"                                                                  \
      "@pxy add.u32 %6, %6, 1;\n\t"                                                                 \
      "@mm add.u32 %7, %7, 1;\n\t"                                                                  \
      "}\n"
#define PB_PAIR_OPS(A, XJ, YJ, KJ)                                                                  \
      : "+d"(A.tot), "+d"(A.fsx), "+d"(A.fsy), "+d"(A.fsxy), "+r"(A.fcx), "+r"(A.fcy), "+r"(A.fcxy), \
        "+r"(A.mmc)                                                                                 \
      : "d"(KJ), "d"(XJ), "d"(YJ), "d"(A.Tx), "d"(A.Ty), "d"(A.RTx), "d"(A.RTy)
#define PB_PAIR(A, XJ, YJ, KJ) asm volatile(PB_PAIR_BODY("add.f64 %0, %0, %8;\n\t") PB_PAIR_OPS(A, XJ, YJ, KJ))
#define PB_PAIR_NT(A, XJ, YJ, KJ) asm volatile(PB_PAIR_BODY("") PB_PAIR_OPS(A, XJ, YJ, KJ))

#define PB_PAIR_W_BODY(TOT)                                                                         \
      "{\n\t"                                                                                       \
      ".reg .pred px, py, qx, qy, pxy, cx, cy, mm;\n\t"                                             \
      ".reg .f64 m0, m1, m2;\n\t"                                                                   \
      "setp.ge.f64 px, %14, %16;\n\t"                                                               \
      "setp.ge.f64 py, %15, %17;\n\t"                                                               \
      "setp.le.f64 qx, %14, %18;\n\t"                                                               \
      "setp.le.f64 qy, %15, %19;\n\t"                                                               \
      "and.pred pxy, px, py;\n\t"                                                                   \
      "xor.pred cx, px, qx;\n\t"                                                                    \
      "xor.pred cy, py, qy;\n\t"                                                                    \
      "and.pred mm, cx, cy;\n\t"                                                                    \
      "not.pred mm, mm;\n\t"                                                                        \
      "selp.f64 m0, " PB_ONE ", " PB_ZERO ", px;\n\t"                                               \
      "selp.f64 m1, " PB_ONE ", " PB_ZERO ", py;\n\t"                                               \
      "selp.f64 m2, " PB_ONE ", " PB_ZERO ", pxy;\n\t"                                              \
      TOT                                                                                           \
      "fma.rn.f64 %1, %12, m0, %1;\n\t"                                                             \
      "fma.rn.f64 %2, %12, m1, %2;\n\t"                                                             \
      "fma.rn.f64 %3, %12, m2, %3;\n\t"                                                             \
      "fma.rn.f64 %5, %13, m0, %5;\n\t"                                                             \
      "fma.rn.f64 %6, %13, m1, %6;\n\t"                                                             \
      "fma.rn.f64 %7, %13, m2, %7;\n\t"                                                             \
      "@px add.u32 %8, %8, 1;\n\t"                                                                  \
      "@py add.u32 %9, %9, 1;\n\t"                                                                  \
      "@pxy add.u32 %10, %10, 1;\n\t"                                                               \
      "@mm add.u32 %11, %11, 1;\n\t"                                                                \
      "}\n"
#define PB_PAIR_W_OPS(A, XJ, YJ, KJ, WJ)                                                            \
      : "+d"(A.tot), "+d"(A.fsx), "+d"(A.fsy), "+d"(A.fsxy), "+d"(A.wtot), "+d"(A.fwx), "+d"(A.fwy), \
        "+d"(A.fwxy), "+r"(A.fcx), "+r"(A.fcy), "+r"(A.fcxy), "+r"(A.mmc)                           \
      : "d"(KJ), "d"(WJ), "d"(XJ), "d"(YJ), "d"(A.Tx), "d"(A.Ty), "d"(A.RTx), "d"(A.RTy)
#define PB_PAIR_W(A, XJ, YJ, KJ, WJ)                                                                \
  asm volatile(PB_PAIR_W_BODY("add.f64 %0, %0, %12;\n\tadd.f64 %4, %4, %13;\n\t") PB_PAIR_W_OPS(A, XJ, YJ, KJ, WJ))
#define PB_PAIR_W_NT(A, XJ, YJ, KJ, WJ) asm volatile(PB_PAIR_W_BODY("") PB_PAIR_W_OPS(A, XJ, YJ, KJ, WJ))

// The same pair without the mirrored bits (no mismatch counter): for blocks whose bounding boxes prove that the
// mirrored bin of every pair is the mirror image of its forward bin.
#define PB_PAIR_NM_BODY(TOT)                                                                        \
      "{\n\t"                                                                                       \
      ".reg .pred px, py, pxy;\n\t"                                                                 \
      ".reg .f64 m0, m1, m2;\n\t"                                                                   \
      "setp.ge.f64 px, %8, %10;\n\t"                                                                \
      "setp.ge.f64 py, %9, %11;\n\t"                                                                \
      "and.pred pxy, px, py;\n\t"                                                                   \
      "selp.f64 m0, " PB_ONE ", " PB_ZERO ", px;\n\t"                                               \
      "selp.f64 m1, " PB_ONE ", " PB_ZERO ", py;\n\t"                                               \
      "selp.f64 m2, " PB_ONE ", " PB_ZERO ", pxy;\n\t"                                              \
      TOT                                                                                           \
      "fma.rn.f64 %1, %7, m0, %1;\n\t"                                                              \
      "fma.rn.f64 %2, %7, m1, %2;\n\t"                                                              \
      "fma.rn.f64 %3, %7, m2, %3;\n\t"                                                              \
      "@px add.u32 %4, %4, 1;\n\t"                                                                  \
      "@py add.u32 %5, %5, 1;\n\t"                                                                  \
      "@pxy add.u32 %6, %6, 1;\n\t"                                                                 \
      "}\n"
#define PB_PAIR_NM_OPS(A, XJ, YJ, KJ)                                                               \
      : "+d"(A.tot), "+d"(A.fsx), "+d"(A.fsy), "+d"(A.fsxy), "+r"(A.fcx), "+r"(A.fcy), "+r"(A.fcxy) \
      : "d"(KJ), "d"(XJ), "d"(YJ), "d"(A.Tx), "d"(A.Ty)
#define PB_PAIR_NM(A, XJ, YJ, KJ) asm volatile(PB_PAIR_NM_BODY("add.f64 %0, %0, %7;\n\t") PB_PAIR_NM_OPS(A, XJ, YJ, KJ))
#define PB_PAIR_NM_NT(A, XJ, YJ, KJ) asm volatile(PB_PAIR_NM_BODY("") PB_PAIR_NM_OPS(A, XJ, YJ, KJ))
#define PB_PAIR_NM_W_BODY(TOT)                                                                      \
      "{\n\t"                                                                                       \
      ".reg .pred px, py, pxy;\n\t"                                                                 \
      ".reg .f64 m0, m1, m2;\n\t"                                                                   \
      "setp.ge.f64 px, %13, %15;\n\t"                                                               \
      "setp.ge.f64 py, %14, %16;\n\t"                                                               \
      "and.pred pxy, px, py;\n\t"                                                                   \
      "selp.f64 m0, " PB_ONE ", " PB_ZERO ", px;\n\t"                                               \
      "selp.f64 m1, " PB_ONE ", " PB_ZERO ", py;\n\t"                                               \
      "selp.f64 m2, " PB_ONE ", " PB_ZERO ", pxy;\n\t"                                              \
      TOT                                                                                           \
      "fma.rn.f64 %1, %11, m0, %1;\n\t"                                                             \
      "fma.rn.f64 %2, %11, m1, %2;\n\t"                                                             \
      "fma.rn.f64 %3, %11, m2, %3;\n\t"                                                             \
      "fma.rn.f64 %5, %12, m0, %5;\n\t"                                                             \
      "fma.rn.f64 %6, %12, m1, %6;\n\t"                                                             \
      "fma.rn.f64 %7, %12, m2, %7;\n\t"                                                             \
      "@px add.u32 %8, %8, 1;\n\t"                                                                  \
      "@py add.u32 %9, %9, 1;\n\t"                                                                  \
      "@pxy add.u32 %10, %10, 1;\n\t"                                                               \
      "}\n"
#define PB_PAIR_NM_W_OPS(A, XJ, YJ, KJ, WJ)                                                         \
      : "+d"(A.tot), "+d"(A.fsx), "+d"(A.fsy), "+d"(A.fsxy), "+d"(A.wtot), "+d"(A.fwx), "+d"(A.fwy), \
        "+d"(A.fwxy), "+r"(A.fcx), "+r"(A.fcy), "+r"(A.fcxy)                                        \
      : "d"(KJ), "d"(WJ), "d"(XJ), "d"(YJ), "d"(A.Tx), "d"(A.Ty)
#define PB_PAIR_NM_W(A, XJ, YJ, KJ, WJ)                                                             \
  asm volatile(PB_PAIR_NM_W_BODY("add.f64 %0, %0, %11;\n\tadd.f64 %4, %4, %12;\n\t") PB_PAIR_NM_W_OPS(A, XJ, YJ, KJ, WJ))
#define PB_PAIR_NM_W_NT(A, XJ, YJ, KJ, WJ) asm volatile(PB_PAIR_NM_W_BODY("") PB_PAIR_NM_W_OPS(A, XJ, YJ, KJ, WJ))

// One pair of a block whose displacements span two bins along ONE axis only (the other window bit is the same
// for every pair of the block): CJ = the column point's coordinate on the varying axis, T / RT the lane's
// forward / mirrored thresholds on it.  bs / bw / bc = block-local masked sums and count of the "upper bin" pairs.
#define PB_PAIR_1D(BS, BC, MMC, CJ, KJ, T, RT)                                                      \
  asm volatile(                                                                                     \
      "{\n\t"                                                                                       \
      ".reg .pred p, c;\n\t"                                                                        \
      ".reg .f64 m;\n\t"                                                                            \
      "setp.ge.f64 p, %3, %5;\n\t"                                                                  \
      "setp.le.f64 c, %3, %6;\n\t"                                                                  \
      "xor.pred c, c, p;\n\t"                                                                       \
      "selp.f64 m, " PB_ONE ", " PB_ZERO ", p;\n\t"                                                 \
      "fma.rn.f64 %0, %4, m, %0;\n\t"                                                               \
      "@p add.u32 %1, %1, 1;\n\t"                                                                   \
      "@!c add.u32 %2, %2, 1;\n\t"                                                                  \
      "}\n"                                                                                         \
      : "+d"(BS), "+r"(BC), "+r"(MMC)                                                               \
      : "d"(CJ), "d"(KJ), "d"(T), "d"(RT))
#define PB_PAIR_1D_W(BS, BW, BC, MMC, CJ, KJ, WJ, T, RT)                                            \
  asm volatile(                                                                                     \
      "{\n\t"                                                                                       \
      ".reg .pred p, c;\n\t"                                                                        \
      ".reg .f64 m;\n\t"                                                                            \
      "setp.ge.f64 p, %4, %7;\n\t"                                                                  \
      "setp.le.f64 c, %4, %8;\n\t"                                                                  \
      "xor.pred c, c, p;\n\t"                                                                       \
      "selp.f64 m, " PB_ONE ", " PB_ZERO ", p;\n\t"                                                 \
      "fma.rn.f64 %0, %5, m, %0;\n\t"                                                               \
      "fma.rn.f64 %1, %6, m, %1;\n\t"                                                               \
      "@p add.u32 %2, %2, 1;\n\t"                                                                   \
      "@!c add.u32 %3, %3, 1;\n\t"                                                                  \
      "}\n"                                                                                         \
      : "+d"(BS), "+d"(BW), "+r"(BC), "+r"(MMC)                                                     \
      : "d"(CJ), "d"(KJ), "d"(WJ), "d"(T), "d"(RT))

// One pair of a 2 x 2-window block whose marginal sums (column bit, row bit) come from rank queries on the sorted
// copies of the chunk: only the "both bits set" quadrant is accumulated per pair.
#define PB_PAIR_Q(BS, BC, XJ, YJ, KJ, TX, TY)                                                       \
  asm volatile(                                                                                     \
      "{\n\t"                                                                                       \
      ".reg .pred p, q;\n\t"                                                                        \
      ".reg .f64 m;\n\t"                                                                            \
      "setp.ge.f64 q, %2, %5;\n\t"                                                                  \
      "setp.ge.and.f64 p, %3, %6, q;\n\t"                                                           \
      "selp.f64 m, " PB_ONE ", " PB_ZERO ", p;\n\t"                                                 \
      "fma.rn.f64 %0, %4, m, %0;\n\t"                                                               \
      "@p add.u32 %1, %1, 1;\n\t"                                                                   \
      "}\n"                                                                                         \
      : "+d"(BS), "+r"(BC)                                                                          \
      : "d"(XJ), "d"(YJ), "d"(KJ), "d"(TX), "d"(TY))
#define PB_PAIR_Q_W(BS, BW, BC, XJ, YJ, KJ, WJ, TX, TY)                                             \
  asm volatile(                                                                                     \
      "{\n\t"                                                                                       \
      ".reg .pred p, q;\n\t"                                                                        \
      ".reg .f64 m;\n\t"                                                                            \
      "setp.ge.f64 q, %3, %7;\n\t"                                                                  \
      "setp.ge.and.f64 p, %4, %8, q;\n\t"                                                           \
      "selp.f64 m, " PB_ONE ", " PB_ZERO ", p;\n\t"                                                 \
      "fma.rn.f64 %0, %5, m, %0;\n\t"                                                               \
      "fma.rn.f64 %1, %6, m, %1;\n\t"                                                               \
      "@p add.u32 %2, %2, 1;\n\t"                                                                   \
      "}\n"                                                                                         \
      : "+d"(BS), "+d"(BW), "+r"(BC)                                                                \
      : "d"(XJ), "d"(YJ), "d"(KJ), "d"(WJ), "d"(TX), "d"(TY))

// Rank query in a chunk's sorted copy read straight from global memory (L1-resident after the first-level probes
// p7, p15, p23 = xs[7], xs[15], xs[23], which the caller issues early): pos = number of columns with c_j < T;
// returns whether the exact mirrored bits agree for this lane (see rank_query in the kernel).
__device__ __forceinline__ bool pb_rank_query_g(const double* __restrict__ xs, double p7, double p15, double p23,
                                                double T, double RT, bool live, int& pos) {
  const int b = 8 * ((p7 < T ? 1 : 0) + (p15 < T ? 1 : 0) + (p23 < T ? 1 : 0));
  const int sp = b + 2 * ((xs[b + 1] < T ? 1 : 0) + (xs[b + 3] < T ? 1 : 0) + (xs[b + 5] < T ? 1 : 0));
  pos = sp + (xs[sp] < T ? 1 : 0) + (xs[sp + 1] < T ? 1 : 0);
  return !live || ((pos == 0 || xs[pos - 1] <= RT) && (pos == PB_CHUNK || xs[pos] > RT));
}
__device__ __forceinline__ void pb_prefetch_l1(const void* p) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(__cvta_generic_to_global(p)));
}

enum { PB_OUT = 0, PB_REG_FULL = 1, PB_REG_CHECK = 2, PB_GENERIC = 3 };

// Classification of one (row block, column block) pair from the two bounding boxes.
// Returns the class; for REG classes w[0..3] receive the packed windows (origin | extent << 16) of the
// forward x, forward y, mirrored x and mirrored y bins.  INLINE_SEARCH: the rare fallback search of the mirrored ends
// is inlined instead of called (no call, so no registers saved around it: the small classification kernel).
template <bool INLINE_SEARCH = false>
__device__ __forceinline__ int pb_classify_twod(double iminx, double imaxx, double iminy, double imaxy,
                                                double cminx, double cmaxx, double cminy, double cmaxy,
                                                double M, double lo2, int nbins, const double* __restrict__ ed,
                                                int (&w)[4]) {
  // every dx = x_j - x_i of the block lies in [dx0, dx1] (rounding is monotone)
  const double dx0 = cminx - imaxx, dx1 = cmaxx - iminx;
  const double dy0 = cminy - imaxy, dy1 = cmaxy - iminy;
  const double ax = fmax(fabs(dx0), fabs(dx1)), ay = fmax(fabs(dy0), fabs(dy1));   // max |dx|, |dy|
  const double nx = dx0 > 0.0 ? dx0 : (dx1 < 0.0 ? -dx1 : 0.0);                    // min |dx|
  const double ny = dy0 > 0.0 ? dy0 : (dy1 < 0.0 ? -dy1 : 0.0);
  const double r2max = __dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay));
  const double r2min = __dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny));
  if (nx >= M || ny >= M || r2max < lo2) return PB_OUT;
  const int x0 = pb_bin_twod_search(dx0, nbins, ed), x1 = pb_bin_twod_search(dx1, nbins, ed);
  const int y0 = pb_bin_twod_search(dy0, nbins, ed), y1 = pb_bin_twod_search(dy1, nbins, ed);
  // mirrored ends: the grid is point symmetric up to rounding of the thresholds, so bin(-d) is nbins-1-bin(d)
  // unless d sits within a few ulp of an edge; the guess is verified against the thresholds (exact either way)
  auto guess = [&](double d, int g) {
    if (INLINE_SEARCH) return (d >= ed[g] && d < ed[g + 1]) ? g : pb_bin_twod_search(d, nbins, ed);
    return pb_bin_twod_guess(d, g, nbins, ed);
  };
  const int rx0 = guess(-dx1, nbins - 1 - x1), rx1 = guess(-dx0, nbins - 1 - x0);
  const int ry0 = guess(-dy1, nbins - 1 - y1), ry1 = guess(-dy0, nbins - 1 - y0);
  if (x1 - x0 > 1 || y1 - y0 > 1 || rx1 - rx0 > 1 || ry1 - ry0 > 1) return PB_GENERIC;
  w[0] = x0 | ((x1 - x0) << 16);
  w[1] = y0 | ((y1 - y0) << 16);
  w[2] = rx0 | ((rx1 - rx0) << 16);
  w[3] = ry0 | ((ry1 - ry0) << 16);
  return (ax < M && ay < M && r2min >= lo2) ? PB_REG_FULL : PB_REG_CHECK;
}

// Work item q of this rank -> catalogue, row block ib and column chunks [c_lo, c_hi).  Returns false for an empty
// item (past the end of a shorter catalogue); stop = true once q is past the last catalogue.  pairbin_kernel keeps
// the same decode inline: calling this helper there changes the register allocation of its pair-by-pair and Log
// instantiations, whose code is the reference the timings are stated for.
struct PBItem {
  int cat;
  int64_t off, n, ib, c_lo, c_hi;
};
__device__ __forceinline__ bool pb_decode_item(const PBParams& P, int64_t q, PBItem& it, bool& stop) {
  const int64_t item = q * P.nranks + P.rank;
  const int R = P.run;
  const int cat = (int)(item / P.items_per_cat);
  stop = cat >= P.ncat;
  if (stop) return false;
  const int64_t lq = item % P.items_per_cat;
  const int64_t off = P.cat_off[cat];
  const int64_t n = P.cat_off[cat + 1] - off;
  const int64_t nblk = (n + PB_CHUNK - 1) / PB_CHUNK;
  if (nblk == 0) return false;
  const int64_t nruns = (nblk + R - 1) / R;
  // decode lq -> (row block ib, run r): rows of group g = ib / R pair with runs g .. nruns-1;
  // items before group g: R * (g*nruns - g*(g-1)/2)
  const double tn = 2.0 * (double)nruns + 1.0;
  const double disc = tn * tn - 8.0 * (double)lq / (double)R;
  int64_t g = (int64_t)((tn - sqrt(disc > 0.0 ? disc : 0.0)) * 0.5);
  if (g < 0) g = 0;
  if (g >= nruns) g = nruns - 1;
  while (g > 0 && (int64_t)R * (g * nruns - g * (g - 1) / 2) > lq) --g;
  while (g + 1 < nruns && (int64_t)R * ((g + 1) * nruns - (g + 1) * g / 2) <= lq) ++g;
  const int64_t rem = lq - (int64_t)R * (g * nruns - g * (g - 1) / 2);
  const int64_t per_row = nruns - g;
  const int64_t row_in_g = rem / per_row;
  const int64_t ib = g * R + row_in_g;
  const int64_t r = g + rem % per_row;
  if (row_in_g >= R || ib >= nblk) return false;  // past the end of this (shorter) catalogue
  it.cat = cat;
  it.off = off;
  it.n = n;
  it.ib = ib;
  it.c_lo = (r * R > ib) ? r * R : ib;
  it.c_hi = ((r + 1) * R < nblk) ? (r + 1) * R : nblk;
  return it.c_lo < it.c_hi;
}

// A window of pb_classify_twod (origin < 4096 | extent <= 1 << 16) in the 13 bits of a record field, and back.
__device__ __forceinline__ int pb_pack_win(int w) { return (w & 0xfff) | ((w >> 16) << 12); }
__device__ __forceinline__ int pb_unpack_win(int v) { return (v & 0xfff) | (((v >> 12) & 1) << 16); }

#ifndef PB_MIN_CTAS
#define PB_MIN_CTAS 2
#endif
// BS: block forms on (closed-form / one-axis blocks).  BS = false is the pair-by-pair kernel: every pair of every
// in-range block goes through the compare / masked-FMA loop (TwoD) -- the kernel the 10-FP64-ops-per-pair
// roofline is stated for; it is compiled without any of the block-form code.
template <int BT, bool WEIGHTED, bool BS>
__global__ void __launch_bounds__(PB_MAX_WARPS * 32, PB_MIN_CTAS)
pairbin_kernel(PBParams P) {
  // TwoD with block forms is pass B of the two-pass count: the blocks come from the records of pass A
  constexpr bool PASS_B = BS && BT == TGP_BIN_TWOD;
  extern __shared__ __align__(16) unsigned char pb_smem[];
  const int nb = P.nb, nbins = P.nbins, nwarps = P.warps;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // ---- shared memory: thresholds (CTA), then per warp: column chunk buffer + private histogram ----
  double* ed = reinterpret_cast<double*>(pb_smem);                          // nbins + 1 (padded to even)
  double2* cxy_all = reinterpret_cast<double2*>(ed + ((nbins + 2) & ~1));   // [warps][32]
  double* ck_all = reinterpret_cast<double*>(cxy_all + nwarps * PB_CHUNK);  // [warps][32]
  double* cw_all = ck_all + nwarps * PB_CHUNK;                              // [warps][32]
  double* hs_all = cw_all + nwarps * PB_CHUNK;                              // [warps][nb]  sum wk wk
  double* hw_all = hs_all + (size_t)nwarps * nb;                            // [warps][nb]  sum w w     (WEIGHTED)
  double* hr_all = hw_all + (WEIGHTED ? (size_t)nwarps * nb : 0);           // [warps][nb]  sum w w r   (LOG)
  unsigned* hc_all = reinterpret_cast<unsigned*>(hr_all + (BT == TGP_BIN_LOG ? (size_t)nwarps * nb : 0));
  double2* cxy = cxy_all + warp * PB_CHUNK;
  double* ck = ck_all + warp * PB_CHUNK;
  double* cw = cw_all + warp * PB_CHUNK;
  double* my_s = hs_all + (size_t)warp * nb;
  double* my_w = hw_all + (size_t)warp * nb;
  double* my_r = hr_all + (size_t)warp * nb;
  unsigned* my_c = hc_all + (size_t)warp * nb;

  for (int i = tid; i <= nbins; i += blockDim.x) ed[i] = P.edges[i];
  for (int i = lane; i < nb; i += 32) {
    my_s[i] = 0.0;
    my_c[i] = 0u;
    if constexpr (WEIGHTED) my_w[i] = 0.0;
    if (BT == TGP_BIN_LOG) my_r[i] = 0.0;
  }
  __syncthreads();  // the only CTA-wide barrier
  if constexpr (PASS_B) {
    if (blockIdx.x == 0 && tid == 0) *P.counter_next = 0ull;   // pass A of the next round starts from zero
  }

  RegAcc<WEIGHTED> A;
  A.zero();
  A.fx0 = -1;
  A.ownerI = -1;
  // TwoD: the warp histogram holds the FORWARD entries only; every booking is point symmetric, so flush_hist adds
  // the mirror image (bin nb-1-b) when it writes a bin out.  The rare pair whose exact mirrored bin is not the
  // mirror image of its forward bin is corrected directly in global memory: -1 at the assumed bin, +1 at the exact.
  int cur_cat = -1;
  auto move_mirrored = [&](int assumed, int exact, double kk, double ww) {
    const size_t g = (size_t)cur_cat * nb;
    atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + g + assumed, ~0ull);   // -1 (mod 2^64)
    atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + g + exact, 1ull);
    atomicAdd(P.sumwkk + g + assumed, -kk);
    atomicAdd(P.sumwkk + g + exact, kk);
    atomicAdd(P.sumw + g + assumed, -ww);
    atomicAdd(P.sumw + g + exact, ww);
  };
  // Move the lane registers of the open window into the warp's shared histogram.
  auto flush_regs = [&]() {
    if (BT != TGP_BIN_TWOD) return;
    if (A.fx0 >= 0) {
      const unsigned n_in = warp_sum_u(A.nin);
      const unsigned fcx = warp_sum_u(A.fcx), fcy = warp_sum_u(A.fcy), fcxy = warp_sum_u(A.fcxy);
      // the lane sums hold sum_j k_j w_j [mask]: times the row point's k_i w_i they are the pair sums
      const double tot = warp_sum(A.tot * A.rki);
      const double fsx = warp_sum(A.fsx * A.rki), fsy = warp_sum(A.fsy * A.rki), fsxy = warp_sum(A.fsxy * A.rki);
      double wtot = 0, fwx = 0, fwy = 0, fwxy = 0;
      if constexpr (WEIGHTED) {
        wtot = warp_sum(A.wtot * A.rwi);
        fwx = warp_sum(A.fwx * A.rwi); fwy = warp_sum(A.fwy * A.rwi); fwxy = warp_sum(A.fwxy * A.rwi);
      }
      if (lane == 0 && n_in) {
        // inclusion-exclusion per window bin (index = bx + 2*by)
        const unsigned fc[4] = {n_in - fcx - fcy + fcxy, fcx - fcxy, fcy - fcxy, fcxy};
        const double fs[4] = {(tot - fsx) - (fsy - fsxy), fsx - fsxy, fsy - fsxy, fsxy};
        const double fw[4] = {(wtot - fwx) - (fwy - fwxy), fwx - fwxy, fwy - fwxy, fwxy};
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          if (fc[b]) {  // a non-empty bin is always inside the grid; the histogram is private to this warp
            const int bx = A.fx0 + (b & 1), by = A.fy0 + (b >> 1);
            const int o = by * nbins + bx;       // forward entry; flush_hist adds the mirror image
            my_c[o] += fc[b];
            my_s[o] += fs[b];
            if constexpr (WEIGHTED) my_w[o] += fw[b];
          }
        }
      }
      __syncwarp();
      A.zero();
      A.fx0 = -1;
    }
  };
  // Rare: some pair of the block just processed has a mirrored bin that is not the mirror image of its
  // forward bin.  Rescan the block and move those pairs from the assumed to the exact mirrored bin.
  auto fix_mirror = [&](int j0, int jn, bool check, double xi, double yi, double ki, double wi) {
    if (!__any_sync(0xffffffffu, A.mmc != 0u)) return;
    if (A.mmc) {
      const int rx0 = nbins - 2 - A.fx0, ry0 = nbins - 2 - A.fy0;
      for (int jj = j0; jj < j0 + jn; ++jj) {
        const double2 pj = cxy[jj];
        if (check) {
          const double dx = pj.x - xi, dy = pj.y - yi;
          const double r2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
          if (!(r2 >= P.lo2 && fabs(dx) < P.hi && fabs(dy) < P.hi)) continue;
        }
        const bool px = pj.x >= A.Tx, py = pj.y >= A.Ty, qx = pj.x <= A.RTx, qy = pj.y <= A.RTy;
        if ((px != qx) && (py != qy)) continue;  // consistent
        const int assumed = (nbins - 1 - (A.fy0 + (py ? 1 : 0))) * nbins + (nbins - 1 - (A.fx0 + (px ? 1 : 0)));
        const int exact = (ry0 + (qy ? 1 : 0)) * nbins + (rx0 + (qx ? 1 : 0));
        double ww = 1.0;
        if constexpr (WEIGHTED) ww = wi * cw[jj];
        move_mirrored(assumed, exact, ki * ck[jj], ww);
      }
      A.mmc = 0u;
    }
    __syncwarp();
  };
  // Warp-private shared histogram -> global (red.global), then clear.
  auto flush_hist = [&](int cat) {   // the window registers were flushed at the end of the last item
    __syncwarp();
    if (cat >= 0) {
      if (BT == TGP_BIN_TWOD) {
        for (int b = lane; b < nb; b += 32) {       // forward entries of bin b + those of its mirror image
          const int bm = nb - 1 - b;
          const unsigned long long c = (unsigned long long)my_c[b] + (unsigned long long)my_c[bm];
          if (c) {
            const size_t o = (size_t)cat * nb + b;
            atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + o, c);
            atomicAdd(P.sumwkk + o, my_s[b] + my_s[bm]);
            atomicAdd(P.sumw + o, WEIGHTED ? my_w[b] + my_w[bm] : (double)c);
          }
        }
        __syncwarp();   // every bin is read twice: clear after all reads
        for (int b = lane; b < nb; b += 32) {
          my_c[b] = 0u;
          my_s[b] = 0.0;
          if constexpr (WEIGHTED) my_w[b] = 0.0;
        }
      } else {
        for (int b = lane; b < nb; b += 32) {
          const unsigned c = my_c[b];
          if (c) {
            const size_t o = (size_t)cat * nb + b;
            atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + o, (unsigned long long)c);
            atomicAdd(P.sumwkk + o, my_s[b]);
            atomicAdd(P.sumw + o, WEIGHTED ? my_w[b] : (double)c);
            if (P.sumwr) atomicAdd(P.sumwr + o, my_r[b]);
            my_c[b] = 0u;
            my_s[b] = 0.0;
            if constexpr (WEIGHTED) my_w[b] = 0.0;
            my_r[b] = 0.0;
          }
        }
      }
    }
    __syncwarp();
  };

  // per-pair generic accumulation of columns [j0, j0+jn) of the staged chunk; `jfirst` = first column this
  // lane may pair with (diagonal block: j > i)
  auto generic_block = [&](int j0, int jn, int jfirst, double xi, double yi, double ki, double wi, bool live) {
    if (live) {
      for (int jj = max(j0, jfirst); jj < j0 + jn; ++jj) {
        const double2 pj = cxy[jj];
        const double dx = pj.x - xi, dy = pj.y - yi;
        const double r2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));  // no FMA: matches the oracle bit for bit
        if (BT == TGP_BIN_TWOD) {
          if (r2 >= P.lo2 && fabs(dx) < P.hi && fabs(dy) < P.hi) {
            const int b1 = pb_bin_twod(dy, P.hi, P.inv_bin, nbins, ed) * nbins + pb_bin_twod(dx, P.hi, P.inv_bin, nbins, ed);
            const int b2 = pb_bin_twod(-dy, P.hi, P.inv_bin, nbins, ed) * nbins + pb_bin_twod(-dx, P.hi, P.inv_bin, nbins, ed);
            const double kk = ki * ck[jj];
            double ww = 1.0;
            if constexpr (WEIGHTED) ww = wi * cw[jj];
            atomicAdd(my_c + b1, 1u);
            atomicAdd(my_s + b1, kk);
            if constexpr (WEIGHTED) atomicAdd(my_w + b1, ww);
            if (b2 != nb - 1 - b1) move_mirrored(nb - 1 - b1, b2, kk, ww);   // displacement on a bin edge
          }
        } else {
          if (r2 >= P.lo2 && r2 < P.hi) {
            const int b = pb_bin_log(r2, nbins, ed);
            double ww = 1.0;
            if constexpr (WEIGHTED) ww = wi * cw[jj];
            atomicAdd(my_c + b, 1u);
            atomicAdd(my_s + b, ki * ck[jj]);
            if constexpr (WEIGHTED) atomicAdd(my_w + b, ww);
            atomicAdd(my_r + b, ww * sqrt(r2));
          }
        }
      }
    }
    __syncwarp();
  };

  // Rank query of this lane's threshold T in the staged sorted copy of a chunk (cxy[].x = the coordinates along the
  // varying axis in ascending order, cxy[].y = suffix sums of k w, cw[] = suffix sums of w): pos = number of columns
  // with c_j < T, found by a 4-ary search -- 3 + 3 + 2 probes in three dependent steps instead of six dependent
  // probes (the kernel is latency-bound here).  Returns whether the exact mirrored bits agree for this lane: columns
  // below the split need c_j <= RT, columns from it on need c_j > RT, and in ascending order only the two
  // neighbours of the split can fail.
  auto rank_query = [&](double T, double RT, bool live, int& pos) -> bool {
    const int b = 8 * ((cxy[7].x < T ? 1 : 0) + (cxy[15].x < T ? 1 : 0) + (cxy[23].x < T ? 1 : 0));
    const int sp = b + 2 * ((cxy[b + 1].x < T ? 1 : 0) + (cxy[b + 3].x < T ? 1 : 0) + (cxy[b + 5].x < T ? 1 : 0));
    pos = sp + (cxy[sp].x < T ? 1 : 0) + (cxy[sp + 1].x < T ? 1 : 0);          // 0 .. 32
    return !live || ((pos == 0 || cxy[pos - 1].x <= RT) && (pos == PB_CHUNK || cxy[pos].x > RT));
  };

  const double M = P.hi, lo2 = P.lo2;
  const int R = P.run;
  unsigned st_closed = 0, st_1d = 0, st_pw = 0, st_sorted = 0, st_quad = 0;   // column counts (x 32 rows = pairs) per path
  int since_flush = 0;
  while (true) {
    // ---- next work item for this warp ----
    unsigned long long q = 0;
    int nrec = 0;
    if constexpr (PASS_B) {
      if (lane == 0) q = atomicAdd(P.counter, 1ull);
      q = __shfl_sync(0xffffffffu, q, 0) + (unsigned long long)P.q_begin;
      if ((int64_t)q >= P.q_end) break;
      nrec = P.rec_cnt[q - P.q_begin];
      if (nrec == 0) continue;
    } else {
      if (lane == 0) q = atomicAdd(P.counter, 1ull);
      q = __shfl_sync(0xffffffffu, q, 0);
      if ((int64_t)q >= P.my_items) break;
    }
    const int64_t item = (int64_t)q * P.nranks + P.rank;
    const int cat = (int)(item / P.items_per_cat);
    if (cat >= P.ncat) break;
    const int64_t lq = item % P.items_per_cat;
    const int64_t off = P.cat_off[cat];
    const int64_t n = P.cat_off[cat + 1] - off;
    const int64_t nblk = (n + PB_CHUNK - 1) / PB_CHUNK;
    if (nblk == 0) continue;
    const int64_t nruns = (nblk + R - 1) / R;
    // decode lq -> (row block ib, run r): rows of group g = ib / R pair with runs g .. nruns-1;
    // items before group g: R * (g*nruns - g*(g-1)/2)
    const double tn = 2.0 * (double)nruns + 1.0;
    const double disc = tn * tn - 8.0 * (double)lq / (double)R;
    int64_t g = (int64_t)((tn - sqrt(disc > 0.0 ? disc : 0.0)) * 0.5);
    if (g < 0) g = 0;
    if (g >= nruns) g = nruns - 1;
    while (g > 0 && (int64_t)R * (g * nruns - g * (g - 1) / 2) > lq) --g;
    while (g + 1 < nruns && (int64_t)R * ((g + 1) * nruns - (g + 1) * g / 2) <= lq) ++g;
    const int64_t rem = lq - (int64_t)R * (g * nruns - g * (g - 1) / 2);
    const int64_t per_row = nruns - g;
    const int64_t row_in_g = rem / per_row;
    const int64_t ib = g * R + row_in_g;
    const int64_t r = g + rem % per_row;
    if (row_in_g >= R || ib >= nblk) continue;  // past the end of this (shorter) catalogue
    const int64_t c_lo = (r * R > ib) ? r * R : ib;
    const int64_t c_hi = ((r + 1) * R < nblk) ? (r + 1) * R : nblk;
    if (c_lo >= c_hi) continue;

    if (cat != cur_cat || since_flush >= PB_FLUSH_ITEMS) {
      flush_hist(cur_cat);
      cur_cat = cat;
      since_flush = 0;
    }
    ++since_flush;

    // ---- this warp's row points ----
    const int64_t ig = ib * PB_CHUNK + lane;
    const bool live = ig < n;
    // dead lanes: NaN coordinates make every comparison false, zero field/weight adds nothing
    const double xi = live ? P.px[off + ig] : __longlong_as_double(0x7ff8000000000000ll);
    const double yi = live ? P.py[off + ig] : __longlong_as_double(0x7ff8000000000000ll);
    double wi = live ? 1.0 : 0.0;
    if constexpr (WEIGHTED) wi = live ? P.pw[off + ig] : 0.0;
    const double ki = live ? P.pk[off + ig] * wi : 0.0;
    const double iminx = warp_min(live ? xi : INFINITY), imaxx = warp_max(live ? xi : -INFINITY);
    const double iminy = warp_min(live ? yi : INFINITY), imaxy = warp_max(live ? yi : -INFINITY);
    const long long owner = (long long)(off + ib * PB_CHUNK);
    // pre-pass record of chunk c of this catalogue: slot (off + 32 c) / 32 + cat = off / 32 + c + cat
    const double* rec0 = P.boxes ? P.boxes + (size_t)PB_STRIDE * (size_t)(off / PB_CHUNK + cat) : nullptr;
    // row-block aggregates for the Log blocks that are booked whole
    const double rowK = warp_sum(ki);
    double rowW = 0.0;
    if constexpr (WEIGHTED) rowW = warp_sum(wi);
    const int nlive = __popc(__ballot_sync(0xffffffffu, live));
    // pass B: the records of this item, in chunk order
    const int4* irec = PASS_B ? P.recs + (size_t)(q - P.q_begin) * (size_t)P.run : nullptr;

    // pass B walks the item's records, 32 at a time; otherwise 32 column chunks at a time
    for (int64_t sc = PASS_B ? 0 : c_lo; sc < (PASS_B ? (int64_t)nrec : c_hi); sc += 32) {
      // ---- lane l classifies column chunk sc + l (pass B: loads record sc + l) ----
      const int64_t mychunk = sc + lane;
      int cls = PB_OUT;
      int kind = 0;   // 0: raw points; 1 / 2: one-axis block answered from the x- / y-sorted copy of the chunk
      // kind != 0 and the varying axis spans exactly two forward bins [v0, v0+1] whose mirrored window is the mirror
      // image (the usual case): 1 | kind << 1 | x0 << 3 | y0 << 15, everything the warp needs to see whether the
      // open window covers the block; 0 otherwise
      int fastw = 0;
      int win[4] = {0, 0, 0, 0};
      int roff = 0;   // pass B: the record's chunk, relative to c_lo
      if (PASS_B) {
        if (mychunk < nrec) {
          const int4 rr = irec[mychunk];
          roff = rr.x & 0xff;
          cls = (rr.x >> 8) & 3;
          kind = (rr.x >> 10) & 3;
          fastw = rr.y;
          win[0] = pb_unpack_win(rr.z);
          win[1] = pb_unpack_win(rr.z >> 16);
          win[2] = pb_unpack_win(rr.w);
          win[3] = pb_unpack_win(rr.w >> 16);
        }
      } else if (mychunk < c_hi) {
        const int64_t j0g = mychunk * PB_CHUNK;
        const int cnt = (int)((n - j0g < PB_CHUNK) ? (n - j0g) : PB_CHUNK);
        double cminx = INFINITY, cmaxx = -INFINITY, cminy = INFINITY, cmaxy = -INFINITY;
        if (P.boxes) {
          const double4 bb = *reinterpret_cast<const double4*>(rec0 + (size_t)PB_STRIDE * (size_t)mychunk);
          cminx = bb.x; cmaxx = bb.y; cminy = bb.z; cmaxy = bb.w;
        } else {
          const double* xs = P.px + off + j0g;
          const double* ys = P.py + off + j0g;
#pragma unroll 1
          for (int t = 0; t < PB_CHUNK; ++t) {   // only without a pre-pass (work == NULL): kept small
            if (t < cnt) {
              const double x = xs[t], y = ys[t];
              cminx = fmin(cminx, x); cmaxx = fmax(cmaxx, x);
              cminy = fmin(cminy, y); cmaxy = fmax(cmaxy, y);
            }
          }
        }
        if (BT == TGP_BIN_TWOD) {
          if (mychunk == ib) {
            cls = PB_GENERIC;  // diagonal block: needs j > i
          } else {
            cls = pb_classify_twod(iminx, imaxx, iminy, imaxy, cminx, cmaxx, cminy, cmaxy, M, lo2, nbins, ed, win);
          }
        } else {
          const double dx0 = cminx - imaxx, dx1 = cmaxx - iminx, dy0 = cminy - imaxy, dy1 = cmaxy - iminy;
          const double ax = fmax(fabs(dx0), fabs(dx1)), ay = fmax(fabs(dy0), fabs(dy1));
          const double nx = dx0 > 0.0 ? dx0 : (dx1 < 0.0 ? -dx1 : 0.0), ny = dy0 > 0.0 ? dy0 : (dy1 < 0.0 ? -dy1 : 0.0);
          const double r2max = __dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay));
          const double r2min = __dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny));
          cls = (r2max < lo2 || r2min >= M) ? PB_OUT : PB_GENERIC;  // M = max_sep^2 for Log
          if (BS && cls == PB_GENERIC && mychunk != ib && r2min >= lo2 && r2max < M) {
            // every pair in range; if the smallest and the largest r^2 of the block share a bin, all pairs do
            const int k0 = pb_bin_log(r2min, nbins, ed), k1 = pb_bin_log(r2max, nbins, ed);
            if (k0 == k1) { cls = PB_REG_FULL; win[0] = k0; }
            else if (k1 == k0 + 1) { cls = PB_REG_CHECK; win[0] = k0; }     // two adjacent bins: one compare per pair
          }
          if (mychunk == ib) cls = PB_GENERIC;
        }
        if (!(iminx <= imaxx)) cls = PB_OUT;  // no live row in this warp
      }
      const unsigned todo = __ballot_sync(0xffffffffu, cls != PB_OUT);
      // ---- process the non-OUT chunks; the next chunk's points are prefetched into registers ----
      unsigned rest = todo;
      double nx_ = 0.0, ny_ = 0.0, nk_ = 0.0, nw_ = 1.0;
      double2 nsum_ = make_double2(0.0, 0.0);
      int nkind_ = 0;
      // the column chunk of lane c's block
      auto chunk_of = [&](int c) -> int64_t {
        if constexpr (PASS_B) return c_lo + __shfl_sync(0xffffffffu, roff, c);
        else return sc + c;
      };
      auto fetch_raw = [&](int c) {
        const int64_t jg = chunk_of(c) * PB_CHUNK + lane;
        const bool ok = jg < n;
        nx_ = ok ? P.px[off + jg] : 0.0;
        ny_ = ok ? P.py[off + jg] : 0.0;
        if constexpr (WEIGHTED) nw_ = ok ? P.pw[off + jg] : 0.0;
        nk_ = ok ? P.pk[off + jg] * nw_ : 0.0;
      };
      auto fetch = [&](int c) {
        const double* rec = rec0 + (size_t)PB_STRIDE * (size_t)chunk_of(c);
        if (P.boxes) nsum_ = *reinterpret_cast<const double2*>(rec + 4);   // chunk sums of k w and w (pre-pass)
        if constexpr (!BS) {
          fetch_raw(c);
          return;
        }
        nkind_ = __shfl_sync(0xffffffffu, kind, c);
        if (nkind_ == 0) {
          fetch_raw(c);
        } else {
          // sorted copy: coordinate along the varying axis, suffix sums of k w (and w) in that order
          const double* sp = rec + PB_SLOT + (nkind_ == 1 ? 0 : 3 * PB_CHUNK) + lane;
          nx_ = sp[0];
          ny_ = sp[PB_CHUNK];
          if constexpr (WEIGHTED) nw_ = sp[2 * PB_CHUNK];
        }
      };
      if (rest) fetch(__ffs(rest) - 1);
      while (rest) {
        const int c = __ffs(rest) - 1;
        rest &= rest - 1;
        __syncwarp();  // previous chunk fully consumed
        cxy[lane] = make_double2(nx_, ny_);
        ck[lane] = nk_;
        if constexpr (WEIGHTED) cw[lane] = nw_;
        int ckind = nkind_;
        const double2 csum = nsum_;
        __syncwarp();
        if (rest) fetch(__ffs(rest) - 1);
        // a block staged from the sorted copy that ends up on a pair-by-pair path needs the raw points after all
        auto ensure_raw = [&]() {
          if (ckind == 0) return;
          __syncwarp();
          fetch_raw(c);
          cxy[lane] = make_double2(nx_, ny_);
          ck[lane] = nk_;
          if constexpr (WEIGHTED) cw[lane] = nw_;
          __syncwarp();
          if (rest) fetch(__ffs(rest) - 1);   // fetch_raw clobbered the prefetch registers
          ckind = 0;
        };
        if constexpr (BS && BT == TGP_BIN_TWOD) {
          // Short cut for the bulk of the one-axis blocks: a full chunk, every pair in range, two bins along the
          // varying axis, and the OPEN window already covers it (one shuffle and four integer compares instead of
          // the general dispatch below).  Anything else -- no open window, a window that has to move, a column
          // within rounding of a bin edge -- falls through to the general path, which decides again from scratch.
          const int fw = __shfl_sync(0xffffffffu, fastw, c);
          if (fw != 0 && A.fx0 >= 0 && A.ownerI == owner) {
            const bool vx = ((fw >> 1) & 3) == 1;
            const int bx0 = (fw >> 3) & 0xfff, by0 = (fw >> 15) & 0xfff;
            if (((fw >> 1) & 3) == 3) {
              // 2 x 2 window, every pair in range, and the open window is exactly the block's: the column-bit and
              // row-bit sums are rank queries on the x- / y-sorted copies (read from global memory: their lines
              // are pulled in while the pair loop runs); only the "both bits" quadrant is summed pair by pair.
              if (bx0 == A.fx0 && by0 == A.fy0) {
                const double* srt = rec0 + (size_t)PB_STRIDE * (size_t)chunk_of(c) + PB_SLOT;
                const double* srty = srt + 3 * PB_CHUNK;
                const double x7 = srt[7], x15 = srt[15], x23 = srt[23];
                const double y7 = srty[7], y15 = srty[15], y23 = srty[23];
                pb_prefetch_l1(srt + PB_CHUNK + 8); pb_prefetch_l1(srt + PB_CHUNK + 24);
                pb_prefetch_l1(srty + PB_CHUNK + 8); pb_prefetch_l1(srty + PB_CHUNK + 24);
                if constexpr (WEIGHTED) {
                  pb_prefetch_l1(srt + 2 * PB_CHUNK + 8); pb_prefetch_l1(srt + 2 * PB_CHUNK + 24);
                  pb_prefetch_l1(srty + 2 * PB_CHUNK + 8); pb_prefetch_l1(srty + 2 * PB_CHUNK + 24);
                }
                double bsq = 0.0, bwq = 0.0;
                unsigned bcq = 0u;
#pragma unroll 4
                for (int jj = 0; jj < PB_CHUNK; ++jj) {
                  const double2 pj = cxy[jj];
                  const double kj = ck[jj];
                  if constexpr (WEIGHTED) { const double wj = cw[jj]; PB_PAIR_Q_W(bsq, bwq, bcq, pj.x, pj.y, kj, wj, A.Tx, A.Ty); }
                  else PB_PAIR_Q(bsq, bcq, pj.x, pj.y, kj, A.Tx, A.Ty);
                }
                int posx, posy;
                const bool okx = pb_rank_query_g(srt, x7, x15, x23, A.Tx, A.RTx, live, posx);
                const bool oky = pb_rank_query_g(srty, y7, y15, y23, A.Ty, A.RTy, live, posy);
                if (__all_sync(0xffffffffu, okx && oky)) {
                  const unsigned n_add = live ? (unsigned)PB_CHUNK : 0u;
                  A.tot += csum.x;
                  A.nin += n_add;
                  A.fsx += (posx < PB_CHUNK) ? srt[PB_CHUNK + posx] : 0.0;
                  A.fsy += (posy < PB_CHUNK) ? srty[PB_CHUNK + posy] : 0.0;
                  A.fcx += live ? (unsigned)(PB_CHUNK - posx) : 0u;
                  A.fcy += live ? (unsigned)(PB_CHUNK - posy) : 0u;
                  A.fsxy += bsq;
                  A.fcxy += bcq;          // dead lanes: NaN thresholds, no compare is true
                  if constexpr (WEIGHTED) {
                    A.wtot += csum.y;
                    A.fwx += (posx < PB_CHUNK) ? srt[2 * PB_CHUNK + posx] : 0.0;
                    A.fwy += (posy < PB_CHUNK) ? srty[2 * PB_CHUNK + posy] : 0.0;
                    A.fwxy += bwq;
                  }
                  st_quad += (unsigned)PB_CHUNK;
                  continue;
                }
              }
            } else {
            const int dvar = vx ? bx0 - A.fx0 : by0 - A.fy0;      // varying axis: the window must start at its lower bin
            const int dcon = vx ? by0 - A.fy0 : bx0 - A.fx0;      // constant axis: either bin of the window
            if (dvar == 0 && (unsigned)dcon <= 1u) {
              int pos;
              const bool okl = rank_query(vx ? A.Tx : A.Ty, vx ? A.RTx : A.RTy, live, pos);
              if (__all_sync(0xffffffffu, okl)) {
                const unsigned n_add = live ? (unsigned)PB_CHUNK : 0u;
                const unsigned bc = live ? (unsigned)(PB_CHUNK - pos) : 0u;
                const double bs = (pos < PB_CHUNK) ? cxy[pos].y : 0.0;
                double bw_ = 0.0;
                if constexpr (WEIGHTED) bw_ = (pos < PB_CHUNK) ? cw[pos] : 0.0;
                const bool other = dcon != 0;
                A.tot += csum.x;
                A.nin += n_add;
                if constexpr (WEIGHTED) A.wtot += csum.y;
                if (vx) {
                  A.fsx += bs; A.fcx += bc;
                  if constexpr (WEIGHTED) A.fwx += bw_;
                  if (other) { A.fsy += csum.x; A.fcy += n_add; if constexpr (WEIGHTED) A.fwy += csum.y; }
                } else {
                  A.fsy += bs; A.fcy += bc;
                  if constexpr (WEIGHTED) A.fwy += bw_;
                  if (other) { A.fsx += csum.x; A.fcx += n_add; if constexpr (WEIGHTED) A.fwx += csum.y; }
                }
                if (other) { A.fsxy += bs; A.fcxy += bc; if constexpr (WEIGHTED) A.fwxy += bw_; }
                st_sorted += (unsigned)PB_CHUNK;
                continue;
              }
            }
            }
          }
        }
        const int64_t j0g = chunk_of(c) * PB_CHUNK;
        const int jcount = (int)((n - j0g < PB_CHUNK) ? (n - j0g) : PB_CHUNK);
        int ccls = __shfl_sync(0xffffffffu, cls, c);
        // Log bins and the diagonal block (needs j > i) go pair by pair through the generic path -- which has ONE
        // call site, at the top of the sub-block loop below, so that its code exists once in the kernel
        const bool whole_generic = (BT != TGP_BIN_TWOD && ccls == PB_GENERIC) || chunk_of(c) == ib;
        const int gfirst = (chunk_of(c) == ib) ? lane + 1 : 0;
        int cw4[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) cw4[k] = __shfl_sync(0xffffffffu, win[k], c);
        if (BT == TGP_BIN_LOG && !whole_generic) {
          // Log bins, every pair of the block in range and in ONE radial bin (or in two adjacent ones): counts and
          // the k-weighted sums of the block are products of the row and chunk sums; sum w_i w_j r needs the pairs
          // (one square root each); with two bins one compare per pair splits off the upper bin's share.  No
          // per-pair bin search, no atomics.
          const int kb = cw4[0];
          const bool two = (ccls == PB_REG_CHECK);
          double accr = 0.0, hr = 0.0, hk = 0.0, hw = 0.0;
          unsigned hcn = 0u;
          if (!two) {
#pragma unroll 4
            for (int jj = 0; jj < jcount; ++jj) {
              const double2 pj = cxy[jj];
              const double dx = pj.x - xi, dy = pj.y - yi;
              const double r = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
              if constexpr (WEIGHTED) accr = fma(cw[jj], r, accr);
              else accr += r;
            }
          } else {
            const double tsplit = ed[kb + 1];          // r2 >= tsplit <=> bin kb + 1
#pragma unroll 2
            for (int jj = 0; jj < jcount; ++jj) {
              const double2 pj = cxy[jj];
              const double dx = pj.x - xi, dy = pj.y - yi;
              const double r2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
              double wr = sqrt(r2);
              if constexpr (WEIGHTED) wr *= cw[jj];
              accr += wr;
              const double m = (r2 >= tsplit) ? 1.0 : 0.0;
              hr = fma(wr, m, hr);
              hk = fma(ck[jj], m, hk);
              if constexpr (WEIGHTED) hw = fma(cw[jj], m, hw);
              hcn += (r2 >= tsplit) ? 1u : 0u;
            }
          }
          const double tot_r = warp_sum(live ? accr * wi : 0.0);
          double S, Sw = 0.0;
          if (P.boxes) {
            S = csum.x;
            Sw = csum.y;
          } else {
            S = warp_sum(ck[lane]);
            if constexpr (WEIGHTED) Sw = warp_sum(cw[lane]);
          }
          double up_r = 0.0, up_k = 0.0, up_w = 0.0;
          unsigned up_c = 0u;
          if (two) {
            up_r = warp_sum(live ? hr * wi : 0.0);
            up_k = warp_sum(live ? hk * ki : 0.0);
            if constexpr (WEIGHTED) up_w = warp_sum(live ? hw * wi : 0.0);
            up_c = warp_sum_u(live ? hcn : 0u);
          }
          if (lane == 0) {       // the histogram is private to this warp
            my_c[kb] += (unsigned)(nlive * jcount) - up_c;
            my_s[kb] += rowK * S - up_k;
            if constexpr (WEIGHTED) my_w[kb] += rowW * Sw - up_w;
            my_r[kb] += tot_r - up_r;
            if (two) {
              my_c[kb + 1] += up_c;
              my_s[kb + 1] += up_k;
              if constexpr (WEIGHTED) my_w[kb + 1] += up_w;
              my_r[kb + 1] += up_r;
              st_1d += (unsigned)jcount;
            } else {
              st_closed += (unsigned)jcount;
            }
          }
          __syncwarp();
          continue;
        }
        // a block whose window is too wide is retried as four 8-column sub-blocks
        const int nsub = (ccls == PB_GENERIC && !whole_generic) ? 4 : 1;
        int scls = ccls;
        int sw[4] = {cw4[0], cw4[1], cw4[2], cw4[3]};
        if (nsub == 4) {
          scls = PB_OUT;
          if (lane < 4 && lane * 8 < jcount) {
            double cminx = INFINITY, cmaxx = -INFINITY, cminy = INFINITY, cmaxy = -INFINITY;
#pragma unroll 1
            for (int t = lane * 8; t < min(lane * 8 + 8, jcount); ++t) {
              const double2 pj = cxy[t];
              cminx = fmin(cminx, pj.x); cmaxx = fmax(cmaxx, pj.x);
              cminy = fmin(cminy, pj.y); cmaxy = fmax(cmaxy, pj.y);
            }
            scls = pb_classify_twod(iminx, imaxx, iminy, imaxy, cminx, cmaxx, cminy, cmaxy, M, lo2, nbins, ed, sw);
          }
        }
        for (int sb = 0; sb < nsub; ++sb) {
          int bcls = scls, bw[4] = {sw[0], sw[1], sw[2], sw[3]};
          int j0 = 0, jn = jcount;
          if (nsub == 4) {
            bcls = __shfl_sync(0xffffffffu, scls, sb);
#pragma unroll
            for (int k = 0; k < 4; ++k) bw[k] = __shfl_sync(0xffffffffu, sw[k], sb);
            j0 = sb * 8;
            jn = min(8, jcount - j0);
            if (jn <= 0) bcls = PB_OUT;
          }
          if (bcls == PB_OUT) continue;
          bool gen = (bcls == PB_GENERIC);
          // ---- register path: make sure the open window covers this block ----
          const int x0 = bw[0] & 0xffff, x1 = x0 + (bw[0] >> 16), y0 = bw[1] & 0xffff, y1 = y0 + (bw[1] >> 16);
          const int rx0 = bw[2] & 0xffff, rx1 = rx0 + (bw[2] >> 16), ry0 = bw[3] & 0xffff, ry1 = ry0 + (bw[3] >> 16);
          // the mirrored window is the mirror image [n-2-f0, n-1-f0] of the forward window [f0, f0+1]
          auto covers = [&](int fx0, int fy0) {
            return fx0 >= 0 && fy0 >= 0 && x0 >= fx0 && x1 <= fx0 + 1 && y0 >= fy0 && y1 <= fy0 + 1 &&
                   rx0 >= nbins - 2 - fx0 && rx1 <= nbins - 1 - fx0 && ry0 >= nbins - 2 - fy0 && ry1 <= nbins - 1 - fy0;
          };
          const bool fits = A.fx0 >= 0 && A.ownerI == owner && covers(A.fx0, A.fy0);
          if (!fits && !gen) {
            flush_regs();
            // candidate origins: the block's lowest bin, or one below it (a window must stay inside the grid
            // unless nbins == 1)
            const int hi0 = max(nbins - 2, 0);
            int fx0 = min(x0, hi0), fy0 = min(y0, hi0);
            if (!covers(fx0, fy0)) {
              const int ax = (x1 == x0 && x0 >= 1) ? x0 - 1 : fx0, ay = (y1 == y0 && y0 >= 1) ? y0 - 1 : fy0;
              if (covers(ax, fy0)) fx0 = ax;
              else if (covers(fx0, ay)) fy0 = ay;
              else if (covers(ax, ay)) { fx0 = ax; fy0 = ay; }
              else gen = true;   // edge asymmetry: exact path
            }
            if (!gen) {
            A.fx0 = fx0; A.fy0 = fy0;
            A.ownerI = owner;
            A.rki = ki;
            A.rwi = wi;
            // bit = (bin >= b0 + 1): forward dx >= ed[b0+1]; mirrored -dx >= ed[r0+1] <=> dx <= -ed[r0+1] with
            // r0 = nbins-2-b0; turned into thresholds on the column coordinate for this lane's row point
            const double tx = (nbins > 1) ? ed[fx0 + 1] : INFINITY, ty = (nbins > 1) ? ed[fy0 + 1] : INFINITY;
            const double ntx = -ed[nbins - 1 - fx0], nty = -ed[nbins - 1 - fy0];   // ed[0] = -inf when nbins == 1
            bool okl = true;
            A.Tx = pb_coord_ge(xi, tx, okl);
            A.Ty = pb_coord_ge(yi, ty, okl);
            A.RTx = pb_coord_le(xi, ntx, okl);
            A.RTy = pb_coord_le(yi, nty, okl);
            if (!__all_sync(0xffffffffu, okl)) {
              // (never seen in practice) the per-lane thresholds did not settle: generic path for this block
              A.fx0 = -1;
              gen = true;
            }
            }
          }
          if (gen) {
            ensure_raw();
            generic_block(j0, jn, gfirst, xi, yi, ki, wi, live);
            if (!whole_generic) st_pw += (unsigned)jn;
            continue;
          }
          if (bcls == PB_REG_FULL) {
            // Every pair of the block is in range.  How many bins do its displacements span?  one_x: all dx in ONE
            // forward bin, all -dx in ONE mirrored bin, and that bin is the mirror image (the usual case: bins are
            // much wider than a 32-point chunk of a sorted catalogue).  Such an axis needs no per-pair decision:
            // the window bit is the same for the whole block.
            const bool whole = BS && (nsub == 1);
            const bool one_x = whole && x1 == x0 && rx1 == rx0 && rx0 == nbins - 1 - x0;
            const bool one_y = whole && y1 == y0 && ry1 == ry0 && ry0 == nbins - 1 - y0;
            // Pair-by-pair kernel: when the bounding boxes put the whole block into ONE forward bin per axis and its
            // mirrored window is that bin's mirror image, the mirrored bits of every pair are the complement of the
            // forward bits by construction; the pair loop then evaluates the forward bits only (every pair is still
            // binned individually).
            const bool nm = !BS && (P.fast_paths & 4) && x1 == x0 && rx1 == rx0 && rx0 == nbins - 1 - x0 &&
                            y1 == y0 && ry1 == ry0 && ry0 == nbins - 1 - y0;
            const unsigned n_add = live ? (unsigned)jn : 0u;
            if (one_x || one_y) {
              // chunk sums of the column values (dead columns were staged as zero)
              double S, Sw = 0.0;
              if (P.boxes) {
                S = csum.x;
                Sw = csum.y;
              } else {
                S = warp_sum(ck[lane]);
                if constexpr (WEIGHTED) Sw = warp_sum(cw[lane]);
              }
              const bool bx = (x0 - A.fx0) != 0, by = (y0 - A.fy0) != 0;   // window bits of the constant axes
              double bs = 0.0, bw_ = 0.0;     // block-local sums / count of the pairs in the upper bin of the varying axis
              unsigned bc = 0u;
              bool done = false;
              if (ckind != 0) {
                // Staged: the chunk's coordinates along the varying axis in ascending order (cxy[].x) with the
                // suffix sums of k w (cxy[].y) and w (cw[]).  The lane's bit "c_j >= T" is a rank query: lower
                // bound by bisection (6 probes instead of 32 compares), count and sum read off the suffix arrays.
                const double T = (ckind == 1) ? A.Tx : A.Ty, RT = (ckind == 1) ? A.RTx : A.RTy;
                int pos;
                const bool okl = rank_query(T, RT, live, pos);
                if (__all_sync(0xffffffffu, okl)) {
                  bc = live ? (unsigned)(PB_CHUNK - pos) : 0u;
                  bs = (pos < PB_CHUNK) ? cxy[pos].y : 0.0;
                  if constexpr (WEIGHTED) bw_ = (pos < PB_CHUNK) ? cw[pos] : 0.0;
                  done = true;
                } else {
                  // (rare) a column within rounding of a bin edge: redo the block pair by pair from the raw points
                  ensure_raw();
                }
              }
              const bool vary_x = one_y;                 // (one_x && one_y): treated as "x varies" with a constant bit
              if (done) {
              } else if (one_x && one_y) {
                // all 32 x jn pairs in one bin (and its mirror image): closed form, no per-pair work at all
                bs = bx ? S : 0.0;
                bw_ = bx ? Sw : 0.0;
                bc = bx ? n_add : 0u;
              } else if (one_y) {
#pragma unroll 2
                for (int jj = 0; jj < jn; ++jj) {
                  const double cj = cxy[jj].x, kj = ck[jj];
                  if constexpr (WEIGHTED) { const double wj = cw[jj]; PB_PAIR_1D_W(bs, bw_, bc, A.mmc, cj, kj, wj, A.Tx, A.RTx); }
                  else PB_PAIR_1D(bs, bc, A.mmc, cj, kj, A.Tx, A.RTx);
                }
              } else {
#pragma unroll 2
                for (int jj = 0; jj < jn; ++jj) {
                  const double cj = cxy[jj].y, kj = ck[jj];
                  if constexpr (WEIGHTED) { const double wj = cw[jj]; PB_PAIR_1D_W(bs, bw_, bc, A.mmc, cj, kj, wj, A.Ty, A.RTy); }
                  else PB_PAIR_1D(bs, bc, A.mmc, cj, kj, A.Ty, A.RTy);
                }
              }
              // fold into the window registers.  v = the varying axis (x unless only x is constant):
              // sum[v bit] += bs; sum[other bit] += S if that bit is set; sum[both] += bs if the other bit is set.
              const bool other = vary_x ? by : bx;
              A.tot += S;
              if constexpr (WEIGHTED) A.wtot += Sw;
              A.nin += n_add;
              if (vary_x) {
                A.fsx += bs; A.fcx += bc;
                if constexpr (WEIGHTED) A.fwx += bw_;
                if (other) { A.fsy += S; A.fcy += n_add; if constexpr (WEIGHTED) A.fwy += Sw; }
              } else {
                A.fsy += bs; A.fcy += bc;
                if constexpr (WEIGHTED) A.fwy += bw_;
                if (other) { A.fsx += S; A.fcx += n_add; if constexpr (WEIGHTED) A.fwx += Sw; }
              }
              if (other) { A.fsxy += bs; A.fcxy += bc; if constexpr (WEIGHTED) A.fwxy += bw_; }
              if (!live) A.mmc = 0u;
              if (one_x && one_y) { if (lane == 0) st_closed += (unsigned)jn; }
              else if (done) st_sorted += (unsigned)jn;
              else st_1d += (unsigned)jn;
              if ((one_x && one_y) || done) continue;   // nothing can be inconsistent
            } else {
            // all pairs of the block are in range: the unmasked sums (sum of k w, of w) are the chunk sums of the
            // pre-pass when the whole chunk is processed, so only the masked sums are accumulated per pair
            const bool tot_from_sums = P.boxes && nsub == 1;
            if (!BS && tot_from_sums && nm) {
#pragma unroll 4
              for (int jj = j0; jj < j0 + jn; ++jj) {
                const double2 pj = cxy[jj];
                const double kj = ck[jj];
                if constexpr (WEIGHTED) {
                  const double wj = cw[jj];
                  PB_PAIR_NM_W_NT(A, pj.x, pj.y, kj, wj);
                } else {
                  PB_PAIR_NM_NT(A, pj.x, pj.y, kj);
                }
              }
              A.tot += csum.x;
              if constexpr (WEIGHTED) A.wtot += csum.y;
            } else if (tot_from_sums) {
#pragma unroll 4
              for (int jj = j0; jj < j0 + jn; ++jj) {
                const double2 pj = cxy[jj];
                const double kj = ck[jj];
                if constexpr (WEIGHTED) {
                  const double wj = cw[jj];
                  PB_PAIR_W_NT(A, pj.x, pj.y, kj, wj);
                } else {
                  PB_PAIR_NT(A, pj.x, pj.y, kj);
                }
              }
              A.tot += csum.x;
              if constexpr (WEIGHTED) A.wtot += csum.y;
            } else {
#pragma unroll 4
              for (int jj = j0; jj < j0 + jn; ++jj) {
                const double2 pj = cxy[jj];
                const double kj = ck[jj];
                if constexpr (WEIGHTED) {
                  const double wj = cw[jj];
                  PB_PAIR_W(A, pj.x, pj.y, kj, wj);
                } else {
                  PB_PAIR(A, pj.x, pj.y, kj);
                }
              }
            }
            A.nin += n_add;
            if (!live) A.mmc = 0u;  // dead lanes (NaN coordinates) compare false everywhere: not a mismatch
            st_pw += (unsigned)jn;
            }
          } else {
            st_pw += (unsigned)jn;
#pragma unroll 2
            for (int jj = j0; jj < j0 + jn; ++jj) {
              const double2 pj = cxy[jj];
              const double dx = pj.x - xi, dy = pj.y - yi;
              const double r2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
              const bool ok = r2 >= lo2 && fabs(dx) < M && fabs(dy) < M;  // false for dead lanes (NaN)
              if (ok) {
                const double kj = ck[jj];
                if constexpr (WEIGHTED) {
                  const double wj = cw[jj];
                  PB_PAIR_W(A, pj.x, pj.y, kj, wj);
                } else {
                  PB_PAIR(A, pj.x, pj.y, kj);
                }
                A.nin += 1u;
              }
            }
          }
          fix_mirror(j0, jn, bcls != PB_REG_FULL, xi, yi, ki, wi);
        }
      }
    }
    // bound the per-lane 32-bit counters: registers go to shared memory at the end of every item
    __syncwarp();
    flush_regs();
  }
  flush_hist(cur_cat);
  {  // blocks booked at classification time are tallied by the classifying lane
    if (st_closed) atomicAdd(&g_pb_stats[0], 32ull * st_closed);
  }
  if (lane == 0) {
    if (st_1d) atomicAdd(&g_pb_stats[1], 32ull * st_1d);
    if (st_pw) atomicAdd(&g_pb_stats[2], 32ull * st_pw);
    if (st_sorted) atomicAdd(&g_pb_stats[3], 32ull * st_sorted);
    if (st_quad) atomicAdd(&g_pb_stats[4], 32ull * st_quad);
  }
}

// Pass A of the TwoD block forms: classify and book.  Same items and dealing as pairbin_kernel; a warp takes an item
// of this round, reads the row block's box, sums and live count from the pre-pass record of chunk ib (no point is
// loaded), and lane l classifies chunk sc + l from the boxes exactly as the fused kernel did:
//   * a block in ONE forward bin whose mirrored window is its mirror image is booked whole from the chunk sums
//     (count = rows x columns, sum = (rows' sum of k w) x (columns' sum of k w)); consecutive chunks of a lane mostly hit
//     the same bin, so the lane keeps one open bin in registers and spills to the warp histogram on a change;
//   * every other block that is not OUT (the diagonal block as GENERIC) is appended to the item's records in chunk
//     order: {chunk - c_lo | class << 8 | kind << 10, fastw, packed forward windows, packed mirrored windows}.
// kind 1 / 2: one varying axis, answered from the x- / y-sorted copy of the chunk; fastw != 0: the block may take
// one of pass B's short cuts (see there).  The warp histograms hold forward entries; the mirror image is added
// when they are written out.
#ifndef PB_CLASSIFY_MIN_CTAS
#define PB_CLASSIFY_MIN_CTAS 2
#endif

// The super records follow the chunk records; their start depends on the total point count cat_off[ncat].
__device__ __forceinline__ const double* pb_super_records(const PBParams& P) {
  return P.boxes + (size_t)PB_STRIDE * (size_t)(P.cat_off[P.ncat] / PB_CHUNK + P.ncat + 2);
}

// Status of super pair (R, C) of one catalogue from the super boxes (srec = record of super-chunk 0 of the catalogue,
// nsf = its number of full super-chunks).  Exact for the reason the chunk classification is: FP subtraction is
// monotone, so the boxes bound every displacement.
//   OUT       every pair fails the range test;
//   CLOSED    every pair in range, in ONE forward bin per axis, and the mirrored window is its mirror image;
//   ONE_AXIS  every pair in range, one such bin on one axis, exactly two forward bins [v0, v0 + 1] on the other whose
//             mirrored window is the mirror image [nbins-2-v0, nbins-1-v0]; vx: x is the varying axis;
//   TWO_AXIS  neither of the above, but every pair passes r2 >= lo2 and each axis spans at most two "bins", where the
//             out-of-range region |d| >= max_sep counts as one, and its in-range mirrored window is the mirror image of
//             the forward one (the range test is the same for both entries: fl(x_i - x_j) = -fl(x_j - x_i)).  x0, y0 =
//             origin of the fixed 2 x 2 forward window [x0, x0 + 1] x [y0, y0 + 1] that holds every in-range pair;
//   DESCEND   anything else, the diagonal (R == C) and short super-chunks: the chunks are classified one by one.
// The super kernel books CLOSED and ONE_AXIS and lists TWO_AXIS for the leaf kernel; the classification pass skips
// every block of a super pair that is not DESCEND.
enum { PB_S_OUT = 0, PB_S_CLOSED = 1, PB_S_ONE_AXIS = 2, PB_S_DESCEND = 3, PB_S_TWO_AXIS = 4 };
__device__ __forceinline__ int pb_super_status(const double* __restrict__ srec, int64_t nsf, int64_t R, int64_t C,
                                               double M, double lo2, int nbins, const double* __restrict__ ed,
                                               int& x0, int& y0, bool& vx) {
  if (R == C || R >= nsf || C >= nsf) return PB_S_DESCEND;
  const double4 a = *reinterpret_cast<const double4*>(srec + (size_t)PB_SUPER_STRIDE * (size_t)R);
  const double4 b = *reinterpret_cast<const double4*>(srec + (size_t)PB_SUPER_STRIDE * (size_t)C);
  int w[4];
  const int cls = pb_classify_twod<true>(a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, M, lo2, nbins, ed, w);
  if (cls == PB_OUT || cls == PB_GENERIC) return cls == PB_OUT ? PB_S_OUT : PB_S_DESCEND;
  x0 = w[0] & 0xffff;
  y0 = w[1] & 0xffff;
  const int rx0 = w[2] & 0xffff, ry0 = w[3] & 0xffff;
  const int ex = w[0] >> 16, ey = w[1] >> 16;
  if (cls == PB_REG_FULL) {
    const bool one_x = ex == 0 && (w[2] >> 16) == 0 && rx0 == nbins - 1 - x0;
    const bool one_y = ey == 0 && (w[3] >> 16) == 0 && ry0 == nbins - 1 - y0;
    const bool clean_x = ex == 1 && (w[2] >> 16) == 1 && rx0 == nbins - 2 - x0;
    const bool clean_y = ey == 1 && (w[3] >> 16) == 1 && ry0 == nbins - 2 - y0;
    vx = one_y;
    if (one_x && one_y) return PB_S_CLOSED;
    if ((one_y && clean_x) || (one_x && clean_y)) return PB_S_ONE_AXIS;
  }
  if (nbins < 2) return PB_S_DESCEND;
  // in-range windows [x0, x0 + ex] (mirrored: the mirror image) plus the out-of-range ends, at most two slots per axis
  const double dx0 = b.x - a.y, dx1 = b.y - a.x, dy0 = b.z - a.w, dy1 = b.w - a.z;
  const double nx = dx0 > 0.0 ? dx0 : (dx1 < 0.0 ? -dx1 : 0.0), ny = dy0 > 0.0 ? dy0 : (dy1 < 0.0 ? -dy1 : 0.0);
  const bool mirror_x = (w[2] >> 16) == ex && rx0 == nbins - 1 - x0 - ex;
  const bool mirror_y = (w[3] >> 16) == ey && ry0 == nbins - 1 - y0 - ey;
  const int sx = ex + 1 + (dx1 >= M ? 1 : 0) + (dx0 <= -M ? 1 : 0);
  const int sy = ey + 1 + (dy1 >= M ? 1 : 0) + (dy0 <= -M ? 1 : 0);
  if (!mirror_x || !mirror_y || sx > 2 || sy > 2 || __dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny)) < lo2)
    return PB_S_DESCEND;
  x0 = min(x0, nbins - 2);   // one in-range bin (nbins - 1 when the upper range edge is the other slot): either bit
  y0 = min(y0, nbins - 2);
  return PB_S_TWO_AXIS;
}

// The list of super pairs for the leaf kernel follows the super records: {length, work counter of the leaf kernel} at
// `work` words 3 and 4, entries {cat, R, C, x0 | y0 << 16} here, room for every super pair of every catalogue.  TWO_AXIS
// entries carry the origin of their 2 x 2 window; ONE_AXIS entries (listed when the staged leaf kernel runs) carry
// the two bins of pb_super_status with PB_E_ONE set and PB_E_VX set when x is the varying axis (nbins <= 4096 leaves
// the top bits of each half free).
constexpr int PB_E_ONE = 1 << 15, PB_E_VX = 1 << 14;
__device__ __forceinline__ int4* pb_super_list(const PBParams& P) {
  return reinterpret_cast<int4*>(const_cast<double*>(pb_super_records(P)) +
                                 (size_t)PB_SUPER_STRIDE * (size_t)(P.cat_off[P.ncat] / PB_SUPER_PTS + P.ncat + 2));
}

// Super pairs per work item of the staged leaf kernel: a slice of the pairs of one kind that share a column super-chunk.
// 128 measured best overall on a B200 (DESIGN section 5, v13): 256 builds fewer tables but balances worse at N = 2e5.
constexpr int PB_LEAF_SLICE = 128;
// Entries of the list (every super pair of every catalogue), super-chunk slots, and work items of the grouped list (at
// most one partial slice per slot and kind), from the total point count.
__host__ __device__ __forceinline__ int64_t pb_super_list_cap(int64_t total) {
  const int64_t nsup = total / PB_SUPER_PTS;
  return nsup * (nsup > 0 ? nsup - 1 : 0) / 2;
}
__host__ __device__ __forceinline__ int64_t pb_super_slots(int64_t total, int32_t ncat) {
  return total / PB_SUPER_PTS + ncat + 2;
}
__host__ __device__ __forceinline__ int64_t pb_super_items_cap(int64_t total, int32_t ncat) {
  return (pb_super_list_cap(total) / PB_LEAF_SLICE + 2 * pb_super_slots(total, ncat) + 1) & ~(int64_t)1;
}
// Words per row of the DESCEND bitmap: one bit per super column of the longest catalogue, and more.
__host__ __device__ __forceinline__ int64_t pb_super_desc_words(int64_t total) { return total / PB_SUPER_PTS / 32 + 1; }
// Behind the list: the links of the super-chunk records (PB_SUPER_PTS halfwords per slot: for every x-sorted position,
// the point's index in the super-chunk | its position in the stored y-sorted copy << 8), two words per slot (the
// TWO_AXIS and the ONE_AXIS pairs with that column super-chunk, then their offsets in the grouped list), the work items
// {first entry << 16 | entries}, the list grouped by column super-chunk and kind, and the DESCEND bitmap: bit C % 32 of
// word desc[(slot of super row R) x pb_super_desc_words + C / 32] is set iff super pair (R, C) is DESCEND (written by
// the super kernel for R < C < the catalogue's full super-chunks; one spare word at the end).  `boxes` = the chunk
// records.
struct PBSuperGroups {
  unsigned short* links;
  unsigned long long *goff, *items;
  int4* glist;
  unsigned* desc;
};
__device__ __forceinline__ PBSuperGroups pb_super_groups(const double* boxes, const int64_t* cat_off, int32_t ncat) {
  const int64_t total = cat_off[ncat], nslot = pb_super_slots(total, ncat);
  const double* rec = boxes + (size_t)PB_STRIDE * (size_t)(total / PB_CHUNK + ncat + 2);
  PBSuperGroups g;
  g.links = reinterpret_cast<unsigned short*>(const_cast<int4*>(
      reinterpret_cast<const int4*>(rec + (size_t)PB_SUPER_STRIDE * (size_t)nslot) + pb_super_list_cap(total)));
  g.goff = reinterpret_cast<unsigned long long*>(g.links + (size_t)PB_SUPER_PTS * nslot);
  g.items = g.goff + 2 * nslot;
  g.glist = reinterpret_cast<int4*>(g.items + pb_super_items_cap(total, ncat));
  g.desc = reinterpret_cast<unsigned*>(g.glist + pb_super_list_cap(total));
  return g;
}

// One row point i of a ONE_AXIS super pair against the column super-chunk's copy sorted along the varying axis (sc:
// PB_SUPER_PTS ascending coordinates, ss / sw: their suffix sums of k w and w), in shared memory.  pos = #{j : fl(c_j -
// c_i) < t} by bisection with that predicate (monotone in c_j); the upper bin v0 + 1 gets PB_SUPER_PTS - pos pairs and
// k_i w_i x suffix(pos) (w_i x suffix(pos)), added to up_c, up_s, up_w; the caller books the lower bin v0 as the rest.
// The exact mirrored bits differ from the mirror image only for the columns between pos and pos_m = #{j : fl(c_j - c_i)
// <= tm}, nearly always none; those pairs are moved in global memory (cb: the bin of the constant axis, vx: x varies).
// Serves the staged leaf kernel and, where it does not run, the super kernel.
template <bool WEIGHTED>
__device__ __forceinline__ void pb_one_axis_row(const double* sc, const double* ss, const double* sw, double ci,
                                                double ki, double wi, double t, double tm, int v0, int cb, bool vx,
                                                int cat, const PBParams& P, unsigned& up_c, double& up_s,
                                                double& up_w) {
  const int nbins = P.nbins;
  // pos = #{j : fl(c_j - c_i) < t} (branch-free lower bound over the ascending copy)
  int pos = 0;
#pragma unroll
  for (int step = PB_SUPER_PTS / 2; step >= 1; step >>= 1)
    if (__dsub_rn(sc[pos + step - 1], ci) < t) pos += step;
  if (pos == PB_SUPER_PTS - 1 && __dsub_rn(sc[pos], ci) < t) pos = PB_SUPER_PTS;
  up_c += (unsigned)(PB_SUPER_PTS - pos);
  const double sk = pos < PB_SUPER_PTS ? ss[pos] : 0.0;
  up_s = fma(ki, sk, up_s);
  double swp = 0.0;
  if constexpr (WEIGHTED) { swp = pos < PB_SUPER_PTS ? sw[pos] : 0.0; up_w = fma(wi, swp, up_w); }
  // exact mirrored bits: consistent iff pos_m == pos, i.e. column pos - 1 has the mirrored upper bit and column
  // pos has not
  const bool ok = (pos == 0 || __dsub_rn(sc[pos - 1], ci) <= tm) &&
                  (pos == PB_SUPER_PTS || !(__dsub_rn(sc[pos], ci) <= tm));
  if (!ok) {   // (rare) a column within rounding of a bin edge
    int pm = 0;
    for (int step = PB_SUPER_PTS / 2; step >= 1; step >>= 1)
      if (__dsub_rn(sc[pm + step - 1], ci) <= tm) pm += step;
    if (pm == PB_SUPER_PTS - 1 && __dsub_rn(sc[pm], ci) <= tm) pm = PB_SUPER_PTS;
    // columns [lo, hi) have a mirrored bin that is not the mirror image of their forward bin: pm > pos, forward
    // upper bin whose mirrored entry is the upper mirrored bin; pm < pos, forward lower bin, mirrored lower bin
    const int a = min(pos, pm), b = max(pos, pm);
    const double kk = ki * ((a < PB_SUPER_PTS ? ss[a] : 0.0) - (b < PB_SUPER_PTS ? ss[b] : 0.0));
    double ww = (double)(b - a);
    if constexpr (WEIGHTED) ww = wi * ((a < PB_SUPER_PTS ? sw[a] : 0.0) - (b < PB_SUPER_PTS ? sw[b] : 0.0));
    const int fv = pm > pos ? v0 + 1 : v0;                   // forward bin on the varying axis
    const int av = nbins - 1 - fv;                           // assumed mirrored bin: the mirror image
    const int xv = pm > pos ? nbins - 1 - v0 : nbins - 2 - v0;   // exact mirrored bin
    const int mc = nbins - 1 - cb;                           // mirrored bin on the constant axis (exact)
    const int assumed = vx ? mc * nbins + av : av * nbins + mc;
    const int exact = vx ? mc * nbins + xv : xv * nbins + mc;
    const size_t g = (size_t)cat * P.nb;
    unsigned long long* cnt = reinterpret_cast<unsigned long long*>(P.npairs) + g;
    atomicAdd(cnt + assumed, (unsigned long long)(-(long long)(b - a)));   // -(b - a) (mod 2^64)
    atomicAdd(cnt + exact, (unsigned long long)(b - a));
    atomicAdd(P.sumwkk + g + assumed, -kk);
    atomicAdd(P.sumwkk + g + exact, kk);
    atomicAdd(P.sumw + g + assumed, -ww);
    atomicAdd(P.sumw + g + exact, ww);
  }
}
template <bool WEIGHTED>
__global__ void __launch_bounds__(PB_MAX_WARPS * 32, PB_CLASSIFY_MIN_CTAS)
pairbin_classify_kernel(PBParams P) {
  extern __shared__ __align__(16) unsigned char pb_smem[];
  const int nb = P.nb, nbins = P.nbins;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double* ed = reinterpret_cast<double*>(pb_smem);                        // nbins + 1 (padded to even)
  double* hs_all = ed + ((nbins + 2) & ~1);                               // [warps][nb]  sum wk wk
  double* hw_all = hs_all + (size_t)P.warps * nb;                         // [warps][nb]  sum w w     (WEIGHTED)
  unsigned* hc_all = reinterpret_cast<unsigned*>(hw_all + (WEIGHTED ? (size_t)P.warps * nb : 0));
  double* my_s = hs_all + (size_t)warp * nb;
  double* my_w = hw_all + (size_t)warp * nb;
  unsigned* my_c = hc_all + (size_t)warp * nb;
  for (int i = tid; i <= nbins; i += blockDim.x) ed[i] = P.edges[i];
  for (int i = lane; i < nb; i += 32) {
    my_s[i] = 0.0;
    my_c[i] = 0u;
    if constexpr (WEIGHTED) my_w[i] = 0.0;
  }
  __syncthreads();
  if (blockIdx.x == 0 && tid == 0) *P.counter_next = 0ull;   // pass B of this round starts from zero

  auto flush_hist = [&](int cat) {   // forward entries of bin b + those of its mirror image, then clear
    __syncwarp();
    if (cat >= 0) {
      for (int b = lane; b < nb; b += 32) {
        const int bm = nb - 1 - b;
        const unsigned long long c = (unsigned long long)my_c[b] + (unsigned long long)my_c[bm];
        if (c) {
          const size_t o = (size_t)cat * nb + b;
          atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + o, c);
          atomicAdd(P.sumwkk + o, my_s[b] + my_s[bm]);
          atomicAdd(P.sumw + o, WEIGHTED ? my_w[b] + my_w[bm] : (double)c);
        }
      }
      __syncwarp();
      for (int b = lane; b < nb; b += 32) {
        my_c[b] = 0u;
        my_s[b] = 0.0;
        if constexpr (WEIGHTED) my_w[b] = 0.0;
      }
    }
    __syncwarp();
  };
  int cf_bin = -1;   // this lane's open bin (forward entry)
  unsigned cf_cnt = 0u;
  double cf_s = 0.0, cf_w = 0.0;
  auto cf_spill = [&]() {
    if (cf_bin >= 0 && cf_cnt) {
      atomicAdd(my_c + cf_bin, cf_cnt);
      atomicAdd(my_s + cf_bin, cf_s);
      if constexpr (WEIGHTED) atomicAdd(my_w + cf_bin, cf_w);
    }
    cf_cnt = 0u;
    cf_s = 0.0;
    cf_w = 0.0;
  };

  const double M = P.hi, lo2 = P.lo2;
  unsigned st_closed = 0;
  int cur_cat = -1, since_flush = 0;
  while (true) {
    unsigned long long q = 0;
    if (lane == 0) q = atomicAdd(P.counter, 1ull);
    q = __shfl_sync(0xffffffffu, q, 0) + (unsigned long long)P.q_begin;
    if ((int64_t)q >= P.q_end) break;
    PBItem it;
    bool stop;
    int nrec = 0;
    if (pb_decode_item(P, (int64_t)q, it, stop)) {
      if (it.cat != cur_cat || since_flush >= PB_FLUSH_ITEMS) {
        flush_hist(cur_cat);
        cur_cat = it.cat;
        since_flush = 0;
      }
      ++since_flush;
      // 32-bit offsets from c_lo keep the register count low: the item spans <= 256 chunks, only the catalogue's last
      // chunk can be short, and the diagonal block is the first one when c_lo == ib
      const int64_t nblk = (it.n + PB_CHUNK - 1) / PB_CHUNK;
      const int span = (int)(it.c_hi - it.c_lo);
      const int tail = (int)(it.n - (nblk - 1) * PB_CHUNK);                    // points of the last chunk
      const int last = (nblk - 1 - it.c_lo < span) ? (int)(nblk - 1 - it.c_lo) : span;
      const bool diag = it.c_lo == it.ib;
      const double* rec0 = P.boxes + (size_t)PB_STRIDE * (size_t)(it.off / PB_CHUNK + it.cat);
      const double* recl = rec0 + (size_t)PB_STRIDE * (size_t)it.c_lo;
      // the row block is chunk ib: its box and sums are the pre-pass record (the same warp reductions)
      const double4 rb = *reinterpret_cast<const double4*>(rec0 + (size_t)PB_STRIDE * (size_t)it.ib);
      const double2 rsum = *reinterpret_cast<const double2*>(rec0 + (size_t)PB_STRIDE * (size_t)it.ib + 4);
      const int nlive = (it.ib == nblk - 1) ? tail : PB_CHUNK;
      int4* out = P.recs + (size_t)(q - P.q_begin) * (size_t)P.run;
      // the super kernel books or lists every super pair that is not DESCEND (on one rank); its blocks are skipped here
      // on every rank.  Lane l takes super column cw + l (cw >= sR: c_lo >= ib), whose status the super kernel left in
      // the DESCEND bitmap; the chunks of the DESCEND ones are then classified 32 at a time.
      const int64_t nsf = P.block_sums == 2 ? it.n / PB_SUPER_PTS : 0, sR = it.ib / PB_SUPER;
      const unsigned* drow = nullptr;   // bitmap row of super row sR (rows at or past nsf are all DESCEND)
      if (sR < nsf) {
        const PBSuperGroups grp = pb_super_groups(P.boxes, P.cat_off, P.ncat);
        drow = grp.desc + (size_t)pb_super_desc_words(P.cat_off[P.ncat]) * (size_t)(it.off / PB_SUPER_PTS + it.cat + sR);
      }
      for (int64_t cw = it.c_lo / PB_SUPER; cw * PB_SUPER < it.c_hi; cw += 32) {
        unsigned bits = ~0u;   // the 32 bits from super column cw on
        if (drow) bits = __funnelshift_r(drow[cw >> 5], drow[(cw >> 5) + 1], (unsigned)(cw & 31));
        const int64_t C = cw + lane;
        const unsigned dm = __ballot_sync(0xffffffffu, C * PB_SUPER < it.c_hi &&
                                                           (C <= sR || C >= nsf || ((bits >> lane) & 1u)));
        const int nd = __popc(dm) * PB_SUPER;
        const int base = (int)(cw * PB_SUPER - it.c_lo);   // negative only for the diagonal super-chunk
        for (int s0 = 0; s0 < nd; s0 += 32) {
          int ch = span;   // chunk c_lo + ch: the ((s0 + lane) % PB_SUPER)-th chunk of the ((s0 + lane) / PB_SUPER)-th
          if (s0 + lane < nd) {   // DESCEND super column: bit b of dm is its t-th set bit <=> popc(dm below b) == t
            const int t = (s0 + lane) / PB_SUPER;
            int b = 0;
#pragma unroll
            for (int step = 16; step > 0; step >>= 1)
              if (__popc(dm & ((1u << (b + step)) - 1u)) <= t) b += step;
            const int c = base + b * PB_SUPER + (s0 + lane) % PB_SUPER;
            if (c >= 0 && c < span) ch = c;
          }
          int cls = PB_OUT, kind = 0, fastw = 0;
          int win[4] = {0, 0, 0, 0};
          if (ch < span) {
            const double* rec = recl + (size_t)PB_STRIDE * (size_t)ch;
            const int cnt = (ch == last) ? tail : PB_CHUNK;
            const double4 bb = *reinterpret_cast<const double4*>(rec);
            if (diag && ch == 0) cls = PB_GENERIC;  // diagonal block: needs j > i
            else cls = pb_classify_twod<true>(rb.x, rb.y, rb.z, rb.w, bb.x, bb.y, bb.z, bb.w, M, lo2, nbins, ed, win);
            if (cls == PB_REG_FULL) {
              const int x0 = win[0] & 0xffff, y0 = win[1] & 0xffff, rx0 = win[2] & 0xffff, ry0 = win[3] & 0xffff;
              const bool one_x = (win[0] >> 16) == 0 && (win[2] >> 16) == 0 && rx0 == nbins - 1 - x0;
              const bool one_y = (win[1] >> 16) == 0 && (win[3] >> 16) == 0 && ry0 == nbins - 1 - y0;
              // exactly one varying axis: the block is answered from the chunk's points sorted along that axis
              if (cnt == PB_CHUNK) kind = (one_y && !one_x) ? 1 : ((one_x && !one_y) ? 2 : 0);
              // kind != 0 and the varying axis spans exactly two forward bins [v0, v0+1] whose mirrored window is the
              // mirror image (the usual case): 1 | kind << 1 | x0 << 3 | y0 << 15, everything pass B needs to see
              // whether its open window covers the block
              if (P.fast_paths & 1) {
                const bool clean_x = (win[0] >> 16) == 1 && (win[2] >> 16) == 1 && rx0 == nbins - 2 - x0;
                const bool clean_y = (win[1] >> 16) == 1 && (win[3] >> 16) == 1 && ry0 == nbins - 2 - y0;
                if ((kind == 1 && clean_x) || (kind == 2 && clean_y)) fastw = 1 | (kind << 1) | (x0 << 3) | (y0 << 15);
              }
              // two bins along BOTH axes: the raw points are staged (kind stays 0); field value 3
              if ((P.fast_paths & 2) && cnt == PB_CHUNK && (win[0] >> 16) == 1 && (win[2] >> 16) == 1 &&
                  rx0 == nbins - 2 - x0 && (win[1] >> 16) == 1 && (win[3] >> 16) == 1 && ry0 == nbins - 2 - y0)
                fastw = 1 | (3 << 1) | (x0 << 3) | (y0 << 15);
              if (one_x && one_y) {
                const double2 sums = *reinterpret_cast<const double2*>(rec + 4);
                const int o = y0 * nbins + x0;
                if (o != cf_bin) { cf_spill(); cf_bin = o; }
                cf_cnt += (unsigned)(nlive * cnt);
                cf_s = fma(rsum.x, sums.x, cf_s);
                if constexpr (WEIGHTED) cf_w = fma(rsum.y, sums.y, cf_w);
                st_closed += (unsigned)cnt;
                cls = PB_OUT;
              }
            }
          }
          const unsigned rm = __ballot_sync(0xffffffffu, cls != PB_OUT);
          if (cls != PB_OUT)
            out[nrec + __popc(rm & ((1u << lane) - 1u))] =
                make_int4(ch | (cls << 8) | (kind << 10), fastw,
                          pb_pack_win(win[0]) | (pb_pack_win(win[1]) << 16),
                          pb_pack_win(win[2]) | (pb_pack_win(win[3]) << 16));
          nrec += __popc(rm);
        }
      }
      cf_spill();   // bounds the per-lane 32-bit count
      cf_bin = -1;
    } else if (stop) {   // (not reached: q_end <= this rank's item count) pass B must still see an empty item
      if (lane == 0) P.rec_cnt[q - P.q_begin] = 0;
      break;
    }
    if (lane == 0) P.rec_cnt[q - P.q_begin] = nrec;
  }
  flush_hist(cur_cat);
  if (st_closed) atomicAdd(&g_pb_stats[0], 32ull * st_closed);
}

// Pre-pass: bounding box and sums of every 32-point chunk of every catalogue (one warp per chunk).
// Slot of chunk c of catalogue `cat`: (cat_off[cat] + 32 c) / 32 + cat  (distinct and monotone); PB_SLOT doubles
// per slot: {xmin, xmax, ymin, ymax, sum k w, sum w, -, -}.
__global__ void __launch_bounds__(256)
pairbin_boxes_kernel(const double* __restrict__ px, const double* __restrict__ py, const double* __restrict__ pk,
                     const double* __restrict__ pw, const int64_t* __restrict__ cat_off,
                     int32_t ncat, int64_t chunks_per_cat, double* __restrict__ boxes, double* __restrict__ sorted) {
  const int lane = threadIdx.x & 31;
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t cat = w / chunks_per_cat, c = w % chunks_per_cat;
  if (cat >= ncat) return;
  const int64_t off = cat_off[cat], n = cat_off[cat + 1] - off;
  const int64_t j = c * PB_CHUNK + lane;
  if (c * PB_CHUNK >= n) return;
  const bool ok = j < n;
  const double x = ok ? px[off + j] : 0.0, y = ok ? py[off + j] : 0.0;
  const double wj = ok ? (pw ? pw[off + j] : 1.0) : 0.0;
  const double kj = ok ? pk[off + j] * wj : 0.0;
  const double a = warp_min(ok ? x : INFINITY), b = warp_max(ok ? x : -INFINITY);
  const double cc = warp_min(ok ? y : INFINITY), d = warp_max(ok ? y : -INFINITY);
  const double sk = warp_sum(kj), sw = warp_sum(wj);
  const int64_t slot = (off + c * PB_CHUNK) / PB_CHUNK + cat;
  if (lane == 0) {
    double* o = boxes + PB_STRIDE * slot;
    o[0] = a; o[1] = b; o[2] = cc; o[3] = d;
    o[4] = sk; o[5] = sw; o[6] = 0.0; o[7] = 0.0;
  }
  if (sorted) {
    // the chunk sorted by x and by y (bitonic network over the 32 lanes; absent points sort last as +inf with
    // zero payload), each with the suffix sums of k w and w in that order
#pragma unroll
    for (int axis = 0; axis < 2; ++axis) {
      double key = ok ? (axis == 0 ? x : y) : INFINITY, vk = kj, vw = wj;
#pragma unroll
      for (int k2 = 2; k2 <= 32; k2 <<= 1) {
#pragma unroll
        for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
          const double okey = __shfl_xor_sync(0xffffffffu, key, j2);
          const double ovk = __shfl_xor_sync(0xffffffffu, vk, j2);
          const double ovw = __shfl_xor_sync(0xffffffffu, vw, j2);
          const bool take_min = ((lane & j2) == 0) == ((lane & k2) == 0);
          const bool swap = take_min ? (okey < key) : (okey > key);
          if (swap) { key = okey; vk = ovk; vw = ovw; }
        }
      }
#pragma unroll
      for (int o2 = 1; o2 < 32; o2 <<= 1) {
        const double tk = __shfl_down_sync(0xffffffffu, vk, o2), tw = __shfl_down_sync(0xffffffffu, vw, o2);
        if (lane + o2 < 32) { vk += tk; vw += tw; }
      }
      double* o = sorted + PB_STRIDE * slot + axis * 3 * PB_CHUNK + lane;
      o[0] = key;
      o[PB_CHUNK] = vk;
      o[2 * PB_CHUNK] = vw;
    }
  }
}

// Pre-pass of the super-chunks: one CTA of PB_SUPER_PTS threads per full super-chunk sorts its points by x and by y
// (bitonic network in shared memory) and stores them with the suffix sums of k w and w, the box (the sorted ends) and
// the sums (the first suffix sums of the x order).  Record of super-chunk s of catalogue `cat`:
// PB_SUPER_STRIDE x (cat_off[cat] / PB_SUPER_PTS + s + cat) doubles from the start of the super records, which
// follow the chunk records (`boxes`).  The point index is carried through both sorts, so the links (pb_super_groups)
// name, for every x-sorted position, the point and its position in the y-sorted copy as stored.  The CTAs also zero
// the group counts of every slot.
__global__ void __launch_bounds__(PB_SUPER_PTS)
pairbin_super_boxes_kernel(const double* __restrict__ px, const double* __restrict__ py, const double* __restrict__ pk,
                           const double* __restrict__ pw, const int64_t* __restrict__ cat_off, int32_t ncat,
                           int64_t supers_per_cat, double* __restrict__ boxes) {
  __shared__ double s_key[PB_SUPER_PTS], s_k[PB_SUPER_PTS], s_w[PB_SUPER_PTS], s_part[2][PB_SUPER_PTS / 32];
  __shared__ int s_idx[PB_SUPER_PTS];
  __shared__ unsigned char s_xi[PB_SUPER_PTS], s_yr[PB_SUPER_PTS];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  {
    unsigned long long* goff = pb_super_groups(boxes, cat_off, ncat).goff;
    const int64_t nslot = pb_super_slots(cat_off[ncat], ncat);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + t; i < 2 * nslot; i += (int64_t)gridDim.x * blockDim.x)
      goff[i] = 0ull;
  }
  const int64_t cat = blockIdx.x / supers_per_cat, s = blockIdx.x % supers_per_cat;
  if (cat >= ncat) return;
  const int64_t off = cat_off[cat], n = cat_off[cat + 1] - off;
  if ((s + 1) * PB_SUPER_PTS > n) return;   // only full super-chunks take a super form
  const int64_t j = off + s * PB_SUPER_PTS + t;
  const double wj = pw ? pw[j] : 1.0, kj = pk[j] * wj;
  double* o = boxes + (size_t)PB_STRIDE * (size_t)(cat_off[ncat] / PB_CHUNK + ncat + 2) +   // = pb_super_records
              (size_t)PB_SUPER_STRIDE * (size_t)(off / PB_SUPER_PTS + s + cat);
  for (int axis = 0; axis < 2; ++axis) {
    s_key[t] = axis == 0 ? px[j] : py[j];
    s_k[t] = kj;
    s_w[t] = wj;
    s_idx[t] = t;
    __syncthreads();
    for (int k2 = 2; k2 <= PB_SUPER_PTS; k2 <<= 1) {
      for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
        const int u = t ^ j2;
        if (u > t) {
          const bool up = (t & k2) == 0;
          if (up ? (s_key[t] > s_key[u]) : (s_key[t] < s_key[u])) {
            double v = s_key[t]; s_key[t] = s_key[u]; s_key[u] = v;
            v = s_k[t]; s_k[t] = s_k[u]; s_k[u] = v;
            v = s_w[t]; s_w[t] = s_w[u]; s_w[u] = v;
            const int iv = s_idx[t]; s_idx[t] = s_idx[u]; s_idx[u] = iv;
          }
        }
        __syncthreads();
      }
    }
    // suffix sums: within the warp, then the totals of the warps above
    double vk = s_k[t], vw = s_w[t];
#pragma unroll
    for (int o2 = 1; o2 < 32; o2 <<= 1) {
      const double tk = __shfl_down_sync(0xffffffffu, vk, o2), tw = __shfl_down_sync(0xffffffffu, vw, o2);
      if (lane + o2 < 32) { vk += tk; vw += tw; }
    }
    if (lane == 0) { s_part[0][warp] = vk; s_part[1][warp] = vw; }
    __syncthreads();
    for (int u = warp + 1; u < PB_SUPER_PTS / 32; ++u) { vk += s_part[0][u]; vw += s_part[1][u]; }
    double* so = o + PB_SLOT + axis * 3 * PB_SUPER_PTS + t;
    so[0] = s_key[t];
    so[PB_SUPER_PTS] = vk;
    so[2 * PB_SUPER_PTS] = vw;
    if (t == 0) {
      o[2 * axis] = s_key[0];
      o[2 * axis + 1] = s_key[PB_SUPER_PTS - 1];
      if (axis == 0) { o[4] = vk; o[5] = vw; o[6] = 0.0; o[7] = 0.0; }
    }
    if (axis == 0) {
      s_xi[t] = (unsigned char)s_idx[t];   // x position t holds point s_idx[t]
    } else {
      s_yr[s_idx[t]] = (unsigned char)t;   // point s_idx[t] sits at y position t
      __syncthreads();
      pb_super_groups(boxes, cat_off, ncat).links[(size_t)PB_SUPER_PTS * (size_t)(off / PB_SUPER_PTS + s + cat) + t] =
          (unsigned short)(s_xi[t] | (s_yr[s_xi[t]] << 8));
    }
    __syncthreads();   // the buffers are refilled for the y order
  }
}

// The super kernel: decides the status of every super pair once per count, before the rounds, and books or lists every
// one that is not DESCEND.  Items are (super row R, run of 32 super columns); lane l takes the status of super pair
// (R, 32 r + l), and the warp writes the run's word of the DESCEND bitmap that the classification pass reads.  Every
// rank sweeps all items (the classification pass of a rank reads super pairs of every item); the items q with
// q % nranks == rank are its own:
//   CLOSED    booked by its lane: count n_R n_C, sum (sum k w)_R (sum k w)_C (forward entry only);
//   ONE_AXIS  with list_one_axis: appended to the list of the staged leaf kernel like TWO_AXIS.  Otherwise one pair at a
//             time by the warp: the column super-chunk's copy sorted along the varying axis is staged in shared memory
//             and every row point takes pb_one_axis_row; the lower bin gets the rest of the pairs and sums;
//   TWO_AXIS  appended to the list of the leaf kernel (pairbin_super_leaves_kernel) and counted per column super-chunk.
// The warp histograms hold forward entries; the mirror image is added when they are written out.
template <bool WEIGHTED>
__global__ void __launch_bounds__(PB_MAX_WARPS * 32, 2)
pairbin_super_kernel(PBParams P) {
  extern __shared__ __align__(16) unsigned char pb_smem[];
  const int nb = P.nb, nbins = P.nbins;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double* ed = reinterpret_cast<double*>(pb_smem);                        // nbins + 1 (padded to even)
  double* stage_all = ed + ((nbins + 2) & ~1);                            // [warps][3][PB_SUPER_PTS]
  double* hs_all = stage_all + (size_t)P.warps * 3 * PB_SUPER_PTS;        // [warps][nb]  sum wk wk
  double* hw_all = hs_all + (size_t)P.warps * nb;                         // [warps][nb]  sum w w     (WEIGHTED)
  unsigned* hc_all = reinterpret_cast<unsigned*>(hw_all + (WEIGHTED ? (size_t)P.warps * nb : 0));
  double* sc = stage_all + (size_t)warp * 3 * PB_SUPER_PTS;   // sorted coordinates
  double* ss = sc + PB_SUPER_PTS;                             // suffix sums of k w
  double* sw = ss + PB_SUPER_PTS;                             // suffix sums of w
  double* my_s = hs_all + (size_t)warp * nb;
  double* my_w = hw_all + (size_t)warp * nb;
  unsigned* my_c = hc_all + (size_t)warp * nb;
  for (int i = tid; i <= nbins; i += blockDim.x) ed[i] = P.edges[i];
  for (int i = lane; i < nb; i += 32) {
    my_s[i] = 0.0;
    my_c[i] = 0u;
    if constexpr (WEIGHTED) my_w[i] = 0.0;
  }
  __syncthreads();

  auto flush_hist = [&](int cat) {   // forward entries of bin b + those of its mirror image, then clear
    __syncwarp();
    if (cat >= 0) {
      for (int b = lane; b < nb; b += 32) {
        const int bm = nb - 1 - b;
        const unsigned long long c = (unsigned long long)my_c[b] + (unsigned long long)my_c[bm];
        if (c) {
          const size_t o = (size_t)cat * nb + b;
          atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + o, c);
          atomicAdd(P.sumwkk + o, my_s[b] + my_s[bm]);
          atomicAdd(P.sumw + o, WEIGHTED ? my_w[b] + my_w[bm] : (double)c);
        }
      }
      __syncwarp();
      for (int b = lane; b < nb; b += 32) {
        my_c[b] = 0u;
        my_s[b] = 0.0;
        if constexpr (WEIGHTED) my_w[b] = 0.0;
      }
    }
    __syncwarp();
  };

  const double M = P.hi, lo2 = P.lo2;
  const double* sup0 = pb_super_records(P);
  int4* slist = pb_super_list(P);
  unsigned long long* goff = pb_super_groups(P.boxes, P.cat_off, P.ncat).goff;
  unsigned* desc = pb_super_groups(P.boxes, P.cat_off, P.ncat).desc;
  const int64_t dwords = pb_super_desc_words(P.cat_off[P.ncat]);
  const int64_t nruns = (P.items_per_cat + 31) / 32;   // items_per_cat: super-chunks of the longest catalogue
  unsigned st_closed = 0, st_one = 0;   // super pairs
  int cur_cat = -1, since_flush = 0;
  while (true) {
    unsigned long long q = 0;
    if (lane == 0) q = atomicAdd(P.counter, 1ull);
    q = __shfl_sync(0xffffffffu, q, 0);
    if ((int64_t)q >= P.my_items) break;
    // every rank sweeps the status of every super pair into the DESCEND bitmap (its classification pass reads super
    // pairs of every item); it books and lists only the items dealt to it
    const int64_t item = (int64_t)q;
    const bool mine = (int64_t)(q % (unsigned long long)P.nranks) == P.rank;
    const int cat = (int)(item / (P.items_per_cat * nruns));
    if (cat >= P.ncat) break;
    const int64_t R = (item % (P.items_per_cat * nruns)) / nruns, r = item % nruns;
    const int64_t off = P.cat_off[cat], n = P.cat_off[cat + 1] - off;
    const int64_t nsf = n / PB_SUPER_PTS;
    if (R >= nsf || (r + 1) * 32 <= R + 1 || r * 32 >= nsf) continue;   // no super column C > R in this run
    const double* srec = sup0 + (size_t)PB_SUPER_STRIDE * (size_t)(off / PB_SUPER_PTS + cat);
    const int64_t C = r * 32 + lane;
    int x0 = 0, y0 = 0;
    bool vx = false;
    const int st = C > R ? pb_super_status(srec, nsf, R, C, M, lo2, nbins, ed, x0, y0, vx) : PB_S_DESCEND;
    const unsigned dsc = __ballot_sync(0xffffffffu, st == PB_S_DESCEND);
    if (lane == 0) desc[(size_t)dwords * (size_t)(off / PB_SUPER_PTS + cat + R) + r] = dsc;
    if (!mine) continue;
    if (cat != cur_cat || since_flush >= PB_SUPER_FLUSH_ITEMS) {
      flush_hist(cur_cat);
      cur_cat = cat;
      since_flush = 0;
    }
    ++since_flush;
    const double2 rsum = *reinterpret_cast<const double2*>(srec + (size_t)PB_SUPER_STRIDE * (size_t)R + 4);
    const bool one = st == PB_S_ONE_AXIS;
    const bool listed = st == PB_S_TWO_AXIS || (one && P.list_one_axis);
    const unsigned lst = __ballot_sync(0xffffffffu, listed);
    if (lst) {   // appended for the leaf kernel: one atomic per warp step
      unsigned long long base = 0;
      if (lane == 0) base = atomicAdd(P.slist_len, (unsigned long long)__popc(lst));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (listed) {
        const int ew = one ? x0 | (y0 << 16) | PB_E_ONE | (vx ? PB_E_VX : 0) : x0 | (y0 << 16);
        slist[base + __popc(lst & ((1u << lane) - 1u))] = make_int4(cat, (int)R, (int)C, ew);
        atomicAdd(goff + 2 * (off / PB_SUPER_PTS + cat + C) + (one ? 1 : 0), 1ull);   // group size of (C, kind)
      }
    }
    if (st == PB_S_CLOSED) {
      const double2 csum = *reinterpret_cast<const double2*>(srec + (size_t)PB_SUPER_STRIDE * (size_t)C + 4);
      const int o = y0 * nbins + x0;
      atomicAdd(my_c + o, (unsigned)(PB_SUPER_PTS * PB_SUPER_PTS));
      atomicAdd(my_s + o, rsum.x * csum.x);
      if constexpr (WEIGHTED) atomicAdd(my_w + o, rsum.y * csum.y);
      ++st_closed;
    }
    unsigned todo = __ballot_sync(0xffffffffu, one && !P.list_one_axis);
    while (todo) {
      const int c = __ffs(todo) - 1;
      todo &= todo - 1;
      const bool cvx = __shfl_sync(0xffffffffu, vx, c);
      const int cx0 = __shfl_sync(0xffffffffu, x0, c), cy0 = __shfl_sync(0xffffffffu, y0, c);
      const double* crec = srec + (size_t)PB_SUPER_STRIDE * (size_t)(r * 32 + c);
      const double* srt = crec + PB_SLOT + (cvx ? 0 : 3 * PB_SUPER_PTS);
      __syncwarp();   // the previous pair's staging is consumed
      for (int u = lane; u < PB_SUPER_PTS; u += 32) {
        sc[u] = srt[u];
        ss[u] = srt[PB_SUPER_PTS + u];
        if constexpr (WEIGHTED) sw[u] = srt[2 * PB_SUPER_PTS + u];
      }
      __syncwarp();
      const int v0 = cvx ? cx0 : cy0, cb = cvx ? cy0 : cx0;   // varying axis: bins v0, v0 + 1; constant axis: bin cb
      const double t = ed[v0 + 1], tm = -ed[nbins - 1 - v0];   // forward upper bit: d >= t; mirrored upper bit: d <= tm
      const double* rc = (cvx ? P.px : P.py) + off + R * PB_SUPER_PTS;
      const double* rk = P.pk + off + R * PB_SUPER_PTS;
      const double* rw = WEIGHTED ? P.pw + off + R * PB_SUPER_PTS : nullptr;
      double up_s = 0.0, up_w = 0.0;
      unsigned up_c = 0u;
#pragma unroll 2
      for (int k = 0; k < PB_SUPER; ++k) {
        const int i = k * 32 + lane;
        const double ci = rc[i];
        double wi = 1.0;
        if constexpr (WEIGHTED) wi = rw[i];
        pb_one_axis_row<WEIGHTED>(sc, ss, sw, ci, rk[i] * wi, wi, t, tm, v0, cb, cvx, cat, P, up_c, up_s, up_w);
      }
      up_c = warp_sum_u(up_c);
      up_s = warp_sum(up_s);
      if constexpr (WEIGHTED) up_w = warp_sum(up_w);
      if (lane == 0) {   // the histogram is private to this warp
        const double2 csum = *reinterpret_cast<const double2*>(crec + 4);
        const int lo_b = cvx ? cb * nbins + v0 : v0 * nbins + cb;
        const int hi_b = cvx ? cb * nbins + v0 + 1 : (v0 + 1) * nbins + cb;
        my_c[lo_b] += (unsigned)(PB_SUPER_PTS * PB_SUPER_PTS) - up_c;
        my_s[lo_b] += rsum.x * csum.x - up_s;
        my_c[hi_b] += up_c;
        my_s[hi_b] += up_s;
        if constexpr (WEIGHTED) {
          my_w[lo_b] += rsum.y * csum.y - up_w;
          my_w[hi_b] += up_w;
        }
        ++st_one;
      }
    }
  }
  flush_hist(cur_cat);
  if (st_closed) atomicAdd(&g_pb_stats[5], (unsigned long long)PB_SUPER_PTS * PB_SUPER_PTS * st_closed);
  if (st_one) atomicAdd(&g_pb_stats[6], (unsigned long long)PB_SUPER_PTS * PB_SUPER_PTS * st_one);
}

// Super pairs taken by the leaf kernel since the last reset (tgp_pairbin_super_leaves), and those of them decided per row
// point against the staged column super-chunk (tgp_pairbin_super_rows).  Diagnostics.
__device__ unsigned long long g_pb_super_leaves;
__device__ unsigned long long g_pb_super_rows;
// ONE_AXIS super pairs decided by the staged leaf kernel since the last reset (tgp_pairbin_super_one_axis_rows): those
// not counted here were decided by the super kernel.  Diagnostics.
__device__ unsigned long long g_pb_super_one_rows;

// Grouping of the list by column super-chunk and kind, for the staged leaf kernel (one CTA): the group sizes counted by
// the super kernel (two per slot: TWO_AXIS, ONE_AXIS) become offsets (exclusive scan over the groups), and every group
// is cut into work items of at most PB_LEAF_SLICE entries, so that an item holds one kind only.  The number of items
// goes to work word 5 (P.slist_len[2]); the host never reads it.
__global__ void __launch_bounds__(1024) pairbin_super_group_kernel(PBParams P) {
  __shared__ unsigned long long s_part[2][32];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const PBSuperGroups grp = pb_super_groups(P.boxes, P.cat_off, P.ncat);
  const int64_t nslot = 2 * pb_super_slots(P.cat_off[P.ncat], P.ncat);   // groups
  const int64_t per = (nslot + blockDim.x - 1) / blockDim.x;
  const int64_t s0 = min((int64_t)t * per, nslot), s1 = min(s0 + per, nslot);
  unsigned long long c = 0, m = 0;
  for (int64_t s = s0; s < s1; ++s) {
    const unsigned long long v = grp.goff[s];
    c += v;
    m += (v + PB_LEAF_SLICE - 1) / PB_LEAF_SLICE;
  }
  unsigned long long ic = c, im = m;   // inclusive scans over the warp, then over the warps
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long tc = __shfl_up_sync(0xffffffffu, ic, o), tm = __shfl_up_sync(0xffffffffu, im, o);
    if (lane >= o) { ic += tc; im += tm; }
  }
  if (lane == 31) { s_part[0][warp] = ic; s_part[1][warp] = im; }
  __syncthreads();
  for (int u = 0; u < warp; ++u) { ic += s_part[0][u]; im += s_part[1][u]; }
  unsigned long long o = ic - c, io = im - m;
  for (int64_t s = s0; s < s1; ++s) {
    const unsigned long long v = grp.goff[s];
    grp.goff[s] = o;
    for (unsigned long long k = 0; k < v; k += PB_LEAF_SLICE)
      grp.items[io++] = ((o + k) << 16) | (v - k < PB_LEAF_SLICE ? v - k : (unsigned long long)PB_LEAF_SLICE);
    o += v;
  }
  if (t == (int)blockDim.x - 1) P.slist_len[2] = io;
}

// Scatter of the list into its groups (the order inside a group is immaterial).
__global__ void __launch_bounds__(256) pairbin_super_scatter_kernel(PBParams P) {
  const PBSuperGroups grp = pb_super_groups(P.boxes, P.cat_off, P.ncat);
  const int4* slist = pb_super_list(P);
  const unsigned long long n = *P.slist_len;
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const int4 e = slist[i];
    const int64_t g = 2 * (P.cat_off[e.x] / PB_SUPER_PTS + e.x + e.z) + ((e.w & PB_E_ONE) ? 1 : 0);
    grp.glist[atomicAdd(grp.goff + g, 1ull)] = e;
  }
}

// Rank query with the bin predicate on the displacement itself: pos = #{j : fl(c_j - ci) < t} in a chunk's ascending
// copy xs (4-ary search as pb_rank_query_g: 3 + 3 + 2 probes in three dependent steps).  fl(c_j - ci) is monotone in
// c_j, so the bisection is exact.  Returns whether the exact mirrored bits agree: columns below pos need
// fl(c_j - ci) <= tm (mirrored upper bit), columns from pos on need it false; only the neighbours of pos can fail.
__device__ __forceinline__ bool pb_rank_query_d(const double* __restrict__ xs, double ci, double t, double tm,
                                                int& pos) {
  const int b = 8 * ((xs[7] - ci < t ? 1 : 0) + (xs[15] - ci < t ? 1 : 0) + (xs[23] - ci < t ? 1 : 0));
  const int sp = b + 2 * ((xs[b + 1] - ci < t ? 1 : 0) + (xs[b + 3] - ci < t ? 1 : 0) + (xs[b + 5] - ci < t ? 1 : 0));
  pos = sp + (xs[sp] - ci < t ? 1 : 0) + (xs[sp + 1] - ci < t ? 1 : 0);
  return (pos == 0 || xs[pos - 1] - ci <= tm) && (pos == PB_CHUNK || !(xs[pos] - ci <= tm));
}

// Leaf classes inside a TWO_AXIS super pair (pairbin_super_leaves_kernel)
enum { PB_L_OUT = 0, PB_L_ONE_X = 2, PB_L_ONE_Y = 3, PB_L_QUAD = 4, PB_L_PAIRS = 5 };

// The bit of each axis of a TWO_AXIS super pair, fixed per super pair from the super-chunk boxes {xmin, xmax, ymin,
// ymax} of rows (rsb) and columns (csb), as pb_super_status decides: bin edge t = ed[x0 + 1] (bit 0 -> bin x0, bit 1
// -> bin x0 + 1); upper range edge t = max_sep (bit 0 -> bin nbins - 1, bit 1 -> out of range); lower range edge t =
// the smallest double above -max_sep (bit 0 -> out, bit 1 -> bin 0).  The mirrored entry's upper bit is d <= m: m =
// -ed[nbins-1-x0] for a bin edge; for a range edge m = the double below t, so the mirror check passes by construction
// (the range test is the same for both entries, fl(x_i - x_j) = -fl(x_j - x_i), and the in-range mirrored window is
// the mirror image).  b*0 / b*1 = forward bin of each bit value, -1 = out of range (dropped at booking).
struct PBLeafBits {
  double tx, ty, mx, my;
  int bx0, bx1, by0, by1;
  bool upx, lox, upy, loy;
};
__device__ __forceinline__ PBLeafBits pb_leaf_bits(const double4& rsb, const double4& csb, double M, int nbins,
                                                   const double* __restrict__ ed, int wx0, int wy0) {
  PBLeafBits b;
  b.upx = csb.y - rsb.x >= M;
  b.lox = csb.x - rsb.y <= -M;
  b.upy = csb.w - rsb.z >= M;
  b.loy = csb.z - rsb.w <= -M;
  b.tx = b.upx ? M : (b.lox ? nextafter(-M, 0.0) : ed[wx0 + 1]);
  b.ty = b.upy ? M : (b.loy ? nextafter(-M, 0.0) : ed[wy0 + 1]);
  b.mx = b.upx ? nextafter(M, 0.0) : (b.lox ? -M : -ed[nbins - 1 - wx0]);
  b.my = b.upy ? nextafter(M, 0.0) : (b.loy ? -M : -ed[nbins - 1 - wy0]);
  b.bx0 = b.upx ? nbins - 1 : (b.lox ? -1 : wx0);
  b.bx1 = b.upx ? -1 : (b.lox ? 0 : wx0 + 1);
  b.by0 = b.upy ? nbins - 1 : (b.loy ? -1 : wy0);
  b.by1 = b.upy ? -1 : (b.loy ? 0 : wy0 + 1);
  return b;
}

// The staged column super-chunk of the leaf kernel.  With p_x = #{j : x-bit 0} (a split of the x-sorted copy) and p_y
// the same on the y-sorted copy, the "both bits" quadrant {j : x position >= p_x, y position >= p_y} is read from a
// two-level dominance table over x-blocks of PB_LT_XB consecutive x positions:
//   U[b][p_y]      sum k w, sum w (uk, uw) and count (uc) over x-blocks >= b with y position >= p_y (row NB = 0);
//   Qr[b][p_y]     members of x-block b with y position < p_y;
//   V[b][xo][q]    sum k w, sum w over members of x-block b with in-block x offset >= xo and in-block y order >= q;
//   msk[b][q]      the members of x-block b with in-block y order >= q, as a bit mask over the x offsets;
// quadrant = U[b + 1][p_y] + V[b][p_x % XB][Qr[b][p_y]] with b = p_x / XB (empty for p_x = PB_SUPER_PTS), its count
// U[b + 1][p_y] + popc(msk[b][Qr[b][p_y]] >> (p_x % XB)).  Suffix sums of the two sorted copies give the x-bit and
// the y-bit sums; index PB_SUPER_PTS of every suffix array is 0.  kx, wx, yr, xp, yo: k w and w in x order, the y
// position of every x position and its inverse, the in-block y order (build only).
constexpr int PB_LT_XB = 16, PB_LT_NB = PB_SUPER_PTS / PB_LT_XB, PB_LT_N = PB_SUPER_PTS + 1;
constexpr int PB_LT_U = (PB_LT_NB + 1) * PB_LT_N, PB_LT_V = PB_LT_NB * PB_LT_XB * (PB_LT_XB + 1);
__host__ __device__ constexpr size_t pb_leaf_table_doubles(bool w) {
  return ((size_t)(w ? 2 : 1) * (2 * PB_LT_N + PB_LT_U + PB_LT_V + PB_SUPER_PTS) + 2 * PB_SUPER_PTS + 1) & ~(size_t)1;
}
constexpr size_t PB_LT_TAIL =   // msk, uc, qr, yr, xp, yo (bytes, 16-byte multiple)
    ((size_t)PB_LT_NB * (PB_LT_XB + 1) * 4 + ((size_t)PB_LT_U * 2 + 3) / 4 * 4 + (size_t)PB_LT_NB * PB_LT_N +
     3 * PB_SUPER_PTS + 15) / 16 * 16;
__host__ __device__ constexpr size_t pb_leaf_table_bytes(bool w) { return pb_leaf_table_doubles(w) * 8 + PB_LT_TAIL; }
struct PBLeafTable {
  double *xs, *ys, *sxk, *syk, *sxw, *syw, *uk, *uw, *vk, *vw, *kx, *wx;
  unsigned* msk;
  unsigned short* uc;
  unsigned char *qr, *yr, *xp, *yo;
  __device__ __forceinline__ void carve(double* p, bool w) {
    double* q = p;
    xs = q; q += PB_SUPER_PTS;
    ys = q; q += PB_SUPER_PTS;
    sxk = q; q += PB_LT_N;
    syk = q; q += PB_LT_N;
    uk = q; q += PB_LT_U;
    vk = q; q += PB_LT_V;
    kx = q; q += PB_SUPER_PTS;
    sxw = syw = uw = vw = wx = nullptr;
    if (w) {
      sxw = q; q += PB_LT_N;
      syw = q; q += PB_LT_N;
      uw = q; q += PB_LT_U;
      vw = q; q += PB_LT_V;
      wx = q;
    }
    msk = reinterpret_cast<unsigned*>(p + pb_leaf_table_doubles(w));
    uc = reinterpret_cast<unsigned short*>(msk + PB_LT_NB * (PB_LT_XB + 1));
    qr = reinterpret_cast<unsigned char*>(uc) + (PB_LT_U * 2 + 3) / 4 * 4;
    yr = qr + PB_LT_NB * PB_LT_N;
    xp = yr + PB_SUPER_PTS;
    yo = xp + PB_SUPER_PTS;
  }
};

// The leaf kernel: the TWO_AXIS super pairs of the list.  A super pair's window [x0, x0 + 1] x [y0, y0 + 1] holds every
// in-range pair and its mirrored window is the mirror image, so the lanes keep four forward bins in registers for the
// whole super pair (sums over all pairs, over the x-bit, the y-bit and both bits; inclusion-exclusion at the end).
// Each axis has one bit per pair, fixed per super pair (pb_leaf_bits).
//
// STAGED (the default when the tables fit in shared memory): work items are slices of the list grouped by column
// super-chunk C and kind (pairbin_super_group_kernel).  A CTA claims an item, stages C's sorted copies and, for a
// TWO_AXIS item, the dominance table (PBLeafTable) once, and its warps pull the slice's super pairs from a shared
// counter.  A ONE_AXIS super pair (the list holds them only in this form) takes pb_one_axis_row for each of its 256
// row points against the staged copy of its varying axis, and is booked like a TWO_AXIS pair; it needs no table and
// no per-block body, and its pairs go to path statistic [6] as the super kernel's did.  For each of the 256 row points
// of a super pair, p_x and p_y come from bisections on the staged copies and the four sums from the suffix sums and the
// table; the exact mirrored bits need only the neighbours of each split.  If any check fails (a column within rounding
// of a bin edge), the super pair goes through the per-block body below instead.  One histogram per CTA, booked with
// shared atomics once per super pair, written out when the catalogue changes and at the end.
//
// Otherwise one super pair per warp step from the list itself (device-side counter), warp histograms, per-block body.
//
// The per-block body decides the 64 leaf blocks (32 x 32 points) as pass B decides them, from pb_classify_twod on the
// chunk boxes of the pre-pass:
//   closed    in ONE bin whose mirrored window is its mirror image: booked by the classifying lane (2 blocks per lane)
//             from the chunk sums, no point loaded;
//   one axis  one rank query per row point on the chunk's copy sorted along the varying axis;
//   2 x 2     (both windows clean) the column-bit and row-bit sums from two rank queries, the "both bits" quadrant
//             pair by pair;
//   otherwise pair by pair over the staged chunk (an unclean mirrored window), with the range test where the range
//             edge runs through the block.
// A block the range edge runs through takes the one-axis or 2 x 2 form like any other block whose bit varies; the
// out-of-range slots are dropped at booking.  A failed mirrored-bit check at the split hands the block to the
// pair-by-pair loop, which counts the pairs whose exact mirrored bin is not the mirror image and moves them in global
// memory afterwards (as pass B's fix_mirror).  The blocks of a super pair decided per row point are classified all
// the same and attributed to the path statistics by their form class.
// The bit predicates compare the displacement fl(c_j - c_i) with the thresholds directly (no per-lane coordinate
// thresholds).  The histograms hold forward entries; the mirror image is added when they are written out.
#ifndef PB_LEAVES_MIN_CTAS
#define PB_LEAVES_MIN_CTAS 2
#endif
template <bool WEIGHTED, bool STAGED>
__global__ void __launch_bounds__(PB_MAX_WARPS * 32 * (STAGED ? 2 : 1), STAGED ? 1 : PB_LEAVES_MIN_CTAS)
pairbin_super_leaves_kernel(PBParams P) {
  extern __shared__ __align__(16) unsigned char pb_smem[];
  const int nb = P.nb, nbins = P.nbins;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double* ed = reinterpret_cast<double*>(pb_smem);                          // nbins + 1 (padded to even)
  double2* cxy_all = reinterpret_cast<double2*>(ed + ((nbins + 2) & ~1));   // [warps][32]
  double* ck_all = reinterpret_cast<double*>(cxy_all + P.warps * PB_CHUNK);  // [warps][32]
  double* cw_all = ck_all + P.warps * PB_CHUNK;                              // [warps][32]
  // !STAGED: [warps][nb] sum wk wk, sum w w (WEIGHTED), counts (32 bit); STAGED: [nb] of each, counts 64 bit
  double* hs_all = cw_all + P.warps * PB_CHUNK;
  double* hw_all = hs_all + (size_t)(STAGED ? 1 : P.warps) * nb;
  unsigned* hc_all = reinterpret_cast<unsigned*>(hw_all + (WEIGHTED ? (size_t)(STAGED ? 1 : P.warps) * nb : 0));
  unsigned long long* hc_cta = reinterpret_cast<unsigned long long*>(hc_all);
  double2* cxy = cxy_all + warp * PB_CHUNK;
  double* ck = ck_all + warp * PB_CHUNK;
  double* cw = cw_all + warp * PB_CHUNK;
  double* my_s = hs_all + (size_t)(STAGED ? 0 : warp) * nb;
  double* my_w = hw_all + (size_t)(STAGED ? 0 : warp) * nb;
  unsigned* my_c = hc_all + (size_t)warp * nb;
  PBLeafTable T;
  if constexpr (STAGED) T.carve(reinterpret_cast<double*>(hc_cta + nb), WEIGHTED);
  for (int i = tid; i <= nbins; i += blockDim.x) ed[i] = P.edges[i];
  if constexpr (STAGED) {
    for (int i = tid; i < nb; i += blockDim.x) {
      my_s[i] = 0.0;
      hc_cta[i] = 0ull;
      if constexpr (WEIGHTED) my_w[i] = 0.0;
    }
  } else {
    for (int i = lane; i < nb; i += 32) {
      my_s[i] = 0.0;
      my_c[i] = 0u;
      if constexpr (WEIGHTED) my_w[i] = 0.0;
    }
  }
  __syncthreads();

  auto flush_hist = [&](int cat) {   // forward entries of bin b + those of its mirror image, then clear
    __syncwarp();
    if (cat >= 0) {
      for (int b = lane; b < nb; b += 32) {
        const int bm = nb - 1 - b;
        const unsigned long long c = (unsigned long long)my_c[b] + (unsigned long long)my_c[bm];
        if (c) {
          const size_t o = (size_t)cat * nb + b;
          atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + o, c);
          atomicAdd(P.sumwkk + o, my_s[b] + my_s[bm]);
          atomicAdd(P.sumw + o, WEIGHTED ? my_w[b] + my_w[bm] : (double)c);
        }
      }
      __syncwarp();
      for (int b = lane; b < nb; b += 32) {
        my_c[b] = 0u;
        my_s[b] = 0.0;
        if constexpr (WEIGHTED) my_w[b] = 0.0;
      }
    }
    __syncwarp();
  };
  auto flush_cta = [&](int cat) {   // the same for the CTA histogram (all threads, after a CTA barrier)
    if (cat < 0) return;
    for (int b = tid; b < nb; b += blockDim.x) {
      const int bm = nb - 1 - b;
      const unsigned long long c = hc_cta[b] + hc_cta[bm];
      if (c) {
        const size_t o = (size_t)cat * nb + b;
        atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + o, c);
        atomicAdd(P.sumwkk + o, my_s[b] + my_s[bm]);
        atomicAdd(P.sumw + o, WEIGHTED ? my_w[b] + my_w[bm] : (double)c);
      }
    }
    __syncthreads();
    for (int b = tid; b < nb; b += blockDim.x) {
      hc_cta[b] = 0ull;
      my_s[b] = 0.0;
      if constexpr (WEIGHTED) my_w[b] = 0.0;
    }
  };

  const double M = P.hi, lo2 = P.lo2;
  const double* sup0 = pb_super_records(P);
  unsigned st_closed = 0, st_1d = 0, st_pw = 0, st_sorted = 0, st_quad = 0, st_pairs = 0, st_rows = 0, st_one = 0;

  // ---- one super pair (one warp) ----
  auto decide = [&](const int4 e) {
    const int cat = e.x, wx0 = e.w & 0xffff, wy0 = e.w >> 16;
    ++st_pairs;
    const int64_t off = P.cat_off[cat];
    const int64_t r0 = (int64_t)e.y * PB_SUPER, c0 = (int64_t)e.z * PB_SUPER;   // first row / column chunk
    const double* rec0 = P.boxes + (size_t)PB_STRIDE * (size_t)(off / PB_CHUNK + cat);
    const double4 rsb = *reinterpret_cast<const double4*>(sup0 + (size_t)PB_SUPER_STRIDE * (size_t)(off / PB_SUPER_PTS + cat + e.y));
    const double4 csb = *reinterpret_cast<const double4*>(sup0 + (size_t)PB_SUPER_STRIDE * (size_t)(off / PB_SUPER_PTS + cat + e.z));
    const PBLeafBits B = pb_leaf_bits(rsb, csb, M, nbins, ed, wx0, wy0);
    const double tx = B.tx, ty = B.ty, mx = B.mx, my = B.my;
    // the four forward bins of the super pair, per lane: all pairs, x-bit, y-bit, both bits
    unsigned n_t = 0u, n_x = 0u, n_y = 0u, n_xy = 0u;
    double s_t = 0.0, s_x = 0.0, s_y = 0.0, s_xy = 0.0, w_t = 0.0, w_x = 0.0, w_y = 0.0, w_xy = 0.0;

    // ---- classify the 64 leaf blocks: lane l takes column chunk l % 8 against row chunks l / 8 and l / 8 + 4 ----
    // BOOK: closed blocks into the four sums (the per-block body); otherwise only the form class is kept
    const double* crec = rec0 + (size_t)PB_STRIDE * (size_t)(c0 + (lane & 7));
    double2 cs = make_double2(0.0, 0.0);
    int code[2];
    auto classify = [&](bool book) {
      const double4 cb = *reinterpret_cast<const double4*>(crec);
      cs = *reinterpret_cast<const double2*>(crec + 4);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const double* rrec = rec0 + (size_t)PB_STRIDE * (size_t)(r0 + (lane >> 3) + 4 * h);
        const double4 rb = *reinterpret_cast<const double4*>(rrec);
        int win[4];
        const int cls = pb_classify_twod<true>(rb.x, rb.y, rb.z, rb.w, cb.x, cb.y, cb.z, cb.w, M, lo2, nbins, ed, win);
        // per axis: 0 / 1 = the bit is constant, 2 = it varies (bin edge with a clean mirrored window, or the range
        // edge runs through the block), 3 = neither (unclean mirrored window)
        auto axis = [&](bool up, bool lo, double d0, double d1, int w, int rw, int a) -> int {
          if (up || lo) return (up ? d1 >= M : d0 <= -M) ? 2 : (up ? 0 : 1);
          const int x0 = w & 0xffff, rx0 = rw & 0xffff;
          if ((w >> 16) == 0 && (rw >> 16) == 0 && rx0 == nbins - 1 - x0) return x0 - a;
          if ((w >> 16) == 1 && (rw >> 16) == 1 && rx0 == nbins - 2 - x0) return 2;
          return 3;
        };
        int bx = 3, by = 3;
        if (cls == PB_REG_FULL || cls == PB_REG_CHECK) {
          bx = axis(B.upx, B.lox, cb.x - rb.y, cb.y - rb.x, win[0], win[2], wx0);
          by = axis(B.upy, B.loy, cb.z - rb.w, cb.w - rb.z, win[1], win[3], wy0);
        }
        int c = PB_L_OUT;
        if (cls != PB_OUT) {
          if (bx < 2 && by < 2) {   // every pair in range, in one slot
            if (book) {
              const double2 rs = *reinterpret_cast<const double2*>(rrec + 4);
              const double s = rs.x * cs.x, w = WEIGHTED ? rs.y * cs.y : 0.0;
              const unsigned n = (unsigned)(PB_CHUNK * PB_CHUNK);
              n_t += n; s_t += s; w_t += w;
              if (bx) { n_x += n; s_x += s; w_x += w; }
              if (by) { n_y += n; s_y += s; w_y += w; }
              if (bx && by) { n_xy += n; s_xy += s; w_xy += w; }
            }
            ++st_closed;
          } else if (bx == 2 && by < 2) c = PB_L_ONE_X | (by << 3);   // x varies, the y bit is constant
          else if (by == 2 && bx < 2) c = PB_L_ONE_Y | (bx << 3);
          else c = (bx == 2 && by == 2 && (P.fast_paths & 2)) ? PB_L_QUAD : PB_L_PAIRS;
          if (cls != PB_REG_FULL && c != PB_L_OUT) c |= 16;   // the range edge runs through the block
        }
        code[h] = c;
      }
    };

    // ---- the leaf blocks that are not closed, one row chunk at a time: lane = row point ----
    auto per_block = [&]() {
      const unsigned act0 = __ballot_sync(0xffffffffu, code[0] != PB_L_OUT);
      const unsigned act1 = __ballot_sync(0xffffffffu, code[1] != PB_L_OUT);
      int staged = -1;   // column chunk staged in cxy / ck / cw
      auto stage = [&](int c) {
        if (c == staged) return;
        const int64_t j = off + (c0 + c) * PB_CHUNK + lane;
        double wj = 1.0;
        if constexpr (WEIGHTED) wj = P.pw[j];
        __syncwarp();
        cxy[lane] = make_double2(P.px[j], P.py[j]);
        ck[lane] = P.pk[j] * wj;
        if constexpr (WEIGHTED) cw[lane] = wj;
        __syncwarp();
        staged = c;
      };
#pragma unroll 1
      for (int rk = 0; rk < PB_SUPER; ++rk) {
        unsigned m = ((rk < 4 ? act0 : act1) >> ((rk & 3) * 8)) & 0xffu;
        if (!m) continue;
        const int codes = rk < 4 ? code[0] : code[1];
        const int64_t i = off + (r0 + rk) * PB_CHUNK + lane;
        const double xi = P.px[i], yi = P.py[i];
        double wi = 1.0;
        if constexpr (WEIGHTED) wi = P.pw[i];
        const double ki = P.pk[i] * wi;
        // a block's column sums of k_j w_j (w_j) over all pairs, the x-bit, the y-bit and both bits, times this row
        // point's k_i w_i (w_i)
        auto book = [&](double at, double ax, double ay, double axy, double bt, double bx, double by, double bxy) {
          s_t = fma(ki, at, s_t); s_x = fma(ki, ax, s_x); s_y = fma(ki, ay, s_y); s_xy = fma(ki, axy, s_xy);
          if constexpr (WEIGHTED) {
            w_t = fma(wi, bt, w_t); w_x = fma(wi, bx, w_x); w_y = fma(wi, by, w_y); w_xy = fma(wi, bxy, w_xy);
          }
        };
        while (m) {
          const int c = __ffs(m) - 1;
          m &= m - 1;
          const int lc = __shfl_sync(0xffffffffu, codes, (rk & 3) * 8 + c);
          const int cls = lc & 7, cbit = (lc >> 3) & 1;
          const bool check = (lc >> 4) & 1;
          const double csk = __shfl_sync(0xffffffffu, cs.x, c);
          double csw = 0.0;
          if constexpr (WEIGHTED) csw = __shfl_sync(0xffffffffu, cs.y, c);
          const double* srt = rec0 + (size_t)PB_STRIDE * (size_t)(c0 + c) + PB_SLOT;   // sorted copies of the chunk
          bool per_pair = cls == PB_L_PAIRS;
          if (cls == PB_L_ONE_X || cls == PB_L_ONE_Y) {
            const bool vx = cls == PB_L_ONE_X;
            const double* xs = vx ? srt : srt + 3 * PB_CHUNK;
            int pos;
            const bool ok = pb_rank_query_d(xs, vx ? xi : yi, vx ? tx : ty, vx ? mx : my, pos);
            if (__all_sync(0xffffffffu, ok)) {
              const unsigned bc = (unsigned)(PB_CHUNK - pos);
              const double bs = pos < PB_CHUNK ? xs[PB_CHUNK + pos] : 0.0;
              double bw = 0.0;
              if constexpr (WEIGHTED) bw = pos < PB_CHUNK ? xs[2 * PB_CHUNK + pos] : 0.0;
              // the varying axis' bit: the rank query; the constant axis' bit: cbit for every pair
              const unsigned cc = cbit ? (unsigned)PB_CHUNK : 0u;
              const double ck_ = cbit ? csk : 0.0, cw_ = cbit ? csw : 0.0;
              n_t += PB_CHUNK;
              n_x += vx ? bc : cc;
              n_y += vx ? cc : bc;
              n_xy += cbit ? bc : 0u;
              book(csk, vx ? bs : ck_, vx ? ck_ : bs, cbit ? bs : 0.0, csw, vx ? bw : cw_, vx ? cw_ : bw, cbit ? bw : 0.0);
              ++st_sorted;
              continue;
            }
            ++st_1d;   // (rare) a column within rounding of a bin edge: pair by pair
            per_pair = true;
          } else if (cls == PB_L_QUAD) {
            stage(c);
            double qs = 0.0, qw = 0.0;
            unsigned qc = 0u;
#pragma unroll 4
            for (int jj = 0; jj < PB_CHUNK; ++jj) {
              const double2 pj = cxy[jj];
              const bool p = (pj.x - xi >= tx) && (pj.y - yi >= ty);
              const double mk = p ? 1.0 : 0.0;
              qs = fma(ck[jj], mk, qs);
              if constexpr (WEIGHTED) qw = fma(cw[jj], mk, qw);
              qc += p ? 1u : 0u;
            }
            int posx, posy;
            const bool okx = pb_rank_query_d(srt, xi, tx, mx, posx);
            const bool oky = pb_rank_query_d(srt + 3 * PB_CHUNK, yi, ty, my, posy);
            if (__all_sync(0xffffffffu, okx && oky)) {
              n_t += PB_CHUNK;
              n_x += (unsigned)(PB_CHUNK - posx);
              n_y += (unsigned)(PB_CHUNK - posy);
              n_xy += qc;
              double bx = 0.0, by = 0.0;
              if constexpr (WEIGHTED) {
                bx = posx < PB_CHUNK ? srt[2 * PB_CHUNK + posx] : 0.0;
                by = posy < PB_CHUNK ? srt[5 * PB_CHUNK + posy] : 0.0;
              }
              book(csk, posx < PB_CHUNK ? srt[PB_CHUNK + posx] : 0.0, posy < PB_CHUNK ? srt[4 * PB_CHUNK + posy] : 0.0,
                   qs, csw, bx, by, qw);
              ++st_quad;
              continue;
            }
            per_pair = true;
          }
          if (!per_pair) continue;
          // pair by pair over the raw points of the chunk: every in-range pair sits in the window; blocks the range
          // edge runs through test the range per pair (r2 >= lo2 holds for every pair of a TWO_AXIS super pair)
          if (cls != PB_L_ONE_X && cls != PB_L_ONE_Y) ++st_pw;
          stage(c);
          unsigned mmc = 0u;
          double a_t = 0.0, a_x = 0.0, a_y = 0.0, a_xy = 0.0, b_t = 0.0, b_x = 0.0, b_y = 0.0, b_xy = 0.0;
#pragma unroll 2
          for (int jj = 0; jj < PB_CHUNK; ++jj) {
            const double2 pj = cxy[jj];
            const double dx = pj.x - xi, dy = pj.y - yi;
            if (check && !(fabs(dx) < M && fabs(dy) < M)) continue;
            const bool px = dx >= tx, py = dy >= ty, qx = dx <= mx, qy = dy <= my;
            const double kj = ck[jj];
            double wj = 0.0;
            if constexpr (WEIGHTED) wj = cw[jj];
            const double fx = px ? 1.0 : 0.0, fy = py ? 1.0 : 0.0, fxy = (px && py) ? 1.0 : 0.0;
            n_t += 1u; n_x += px ? 1u : 0u; n_y += py ? 1u : 0u; n_xy += (px && py) ? 1u : 0u;
            a_t += kj; a_x = fma(kj, fx, a_x); a_y = fma(kj, fy, a_y); a_xy = fma(kj, fxy, a_xy);
            if constexpr (WEIGHTED) { b_t += wj; b_x = fma(wj, fx, b_x); b_y = fma(wj, fy, b_y); b_xy = fma(wj, fxy, b_xy); }
            mmc += ((px != qx) && (py != qy)) ? 0u : 1u;
          }
          book(a_t, a_x, a_y, a_xy, b_t, b_x, b_y, b_xy);
          if (__any_sync(0xffffffffu, mmc != 0u) && mmc) {
            // (rare) pairs whose exact mirrored bin is not the mirror image of the forward bin: -1 at the assumed
            // bin, +1 at the exact one, directly in global memory
            const size_t g = (size_t)cat * nb;
            for (int jj = 0; jj < PB_CHUNK; ++jj) {
              const double2 pj = cxy[jj];
              const double dx = pj.x - xi, dy = pj.y - yi;
              if (check && !(fabs(dx) < M && fabs(dy) < M)) continue;
              const bool px = dx >= tx, py = dy >= ty, qx = dx <= mx, qy = dy <= my;
              if ((px != qx) && (py != qy)) continue;
              // only bin-edge bits can disagree; a range bit's mirrored bin is the mirror image
              const int fx = px ? B.bx1 : B.bx0, fy = py ? B.by1 : B.by0;
              const int ex = px != qx ? nbins - 1 - fx : nbins - 2 - wx0 + (qx ? 1 : 0);
              const int ey = py != qy ? nbins - 1 - fy : nbins - 2 - wy0 + (qy ? 1 : 0);
              const int assumed = (nbins - 1 - fy) * nbins + (nbins - 1 - fx), exact = ey * nbins + ex;
              const double kk = ki * ck[jj];
              double ww = 1.0;
              if constexpr (WEIGHTED) ww = wi * cw[jj];
              atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + g + assumed, ~0ull);   // -1 (mod 2^64)
              atomicAdd(reinterpret_cast<unsigned long long*>(P.npairs) + g + exact, 1ull);
              atomicAdd(P.sumwkk + g + assumed, -kk);
              atomicAdd(P.sumwkk + g + exact, kk);
              atomicAdd(P.sumw + g + assumed, -ww);
              atomicAdd(P.sumw + g + exact, ww);
            }
          }
        }
      }
    };

    bool rows_ok = false;
    if constexpr (STAGED) {
      // ---- per row point against the staged column super-chunk: p_x, p_y by bisection, the quadrant from the table
      const int SP = PB_SUPER_PTS, XB = PB_LT_XB, N = PB_LT_N;
      const int64_t rb = off + (int64_t)e.y * PB_SUPER_PTS + lane;
      const double csk = T.sxk[0];
      double csw = 0.0;
      if constexpr (WEIGHTED) csw = T.sxw[0];
      bool ok = true;
#pragma unroll 2
      for (int k = 0; k < PB_SUPER; ++k) {
        const int64_t i = rb + k * 32;
        const double xi = P.px[i], yi = P.py[i];
        double wi = 1.0;
        if constexpr (WEIGHTED) wi = P.pw[i];
        const double ki = P.pk[i] * wi;
        int px = 0, py = 0;   // #{j : fl(c_j - c_i) < t} (branch-free lower bounds over the ascending copies)
#pragma unroll
        for (int step = SP / 2; step >= 1; step >>= 1) {
          if (T.xs[px + step - 1] - xi < tx) px += step;
          if (T.ys[py + step - 1] - yi < ty) py += step;
        }
        if (px == SP - 1 && T.xs[px] - xi < tx) px = SP;
        if (py == SP - 1 && T.ys[py] - yi < ty) py = SP;
        // exact mirrored bits: consistent iff the column below each split has the mirrored upper bit and the column at
        // the split has not
        ok = ok && (px == 0 || T.xs[px - 1] - xi <= mx) && (px == SP || !(T.xs[px] - xi <= mx)) &&
             (py == 0 || T.ys[py - 1] - yi <= my) && (py == SP || !(T.ys[py] - yi <= my));
        const int b = min(px / XB, PB_LT_NB - 1), xo = px % XB;
        const int q = T.qr[b * N + py];
        unsigned qc = T.uc[(b + 1) * N + py] + __popc(T.msk[b * (XB + 1) + q] >> xo);
        double qs = T.uk[(b + 1) * N + py] + T.vk[(b * XB + xo) * (XB + 1) + q];
        if (px == SP) { qc = 0u; qs = 0.0; }
        n_t += (unsigned)SP;
        n_x += (unsigned)(SP - px);
        n_y += (unsigned)(SP - py);
        n_xy += qc;
        s_t = fma(ki, csk, s_t);
        s_x = fma(ki, T.sxk[px], s_x);
        s_y = fma(ki, T.syk[py], s_y);
        s_xy = fma(ki, qs, s_xy);
        if constexpr (WEIGHTED) {
          double qw = T.uw[(b + 1) * N + py] + T.vw[(b * XB + xo) * (XB + 1) + q];
          if (px == SP) qw = 0.0;
          w_t = fma(wi, csw, w_t);
          w_x = fma(wi, T.sxw[px], w_x);
          w_y = fma(wi, T.syw[py], w_y);
          w_xy = fma(wi, qw, w_xy);
        }
      }
      rows_ok = __all_sync(0xffffffffu, ok);
    }
    if (rows_ok) {   // the leaf blocks only for the path statistics, by form class
      classify(false);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int cls = code[h] & 7;
        st_sorted += __popc(__ballot_sync(0xffffffffu, cls == PB_L_ONE_X || cls == PB_L_ONE_Y));
        st_quad += __popc(__ballot_sync(0xffffffffu, cls == PB_L_QUAD));
        st_pw += __popc(__ballot_sync(0xffffffffu, cls == PB_L_PAIRS));
      }
      ++st_rows;
    } else {
      n_t = n_x = n_y = n_xy = 0u;
      s_t = s_x = s_y = s_xy = w_t = w_x = w_y = w_xy = 0.0;
      classify(true);
      per_block();
    }

    // ---- the four bins of the window into the histogram (forward entries) ----
    n_t = warp_sum_u(n_t); n_x = warp_sum_u(n_x); n_y = warp_sum_u(n_y); n_xy = warp_sum_u(n_xy);
    s_t = warp_sum(s_t); s_x = warp_sum(s_x); s_y = warp_sum(s_y); s_xy = warp_sum(s_xy);
    if constexpr (WEIGHTED) { w_t = warp_sum(w_t); w_x = warp_sum(w_x); w_y = warp_sum(w_y); w_xy = warp_sum(w_xy); }
    if (lane == 0) {   // inclusion-exclusion per slot (index = bx + 2 by), out-of-range slots dropped
      const unsigned fc[4] = {n_t - n_x - n_y + n_xy, n_x - n_xy, n_y - n_xy, n_xy};
      const double fs[4] = {(s_t - s_x) - (s_y - s_xy), s_x - s_xy, s_y - s_xy, s_xy};
      const double fw[4] = {(w_t - w_x) - (w_y - w_xy), w_x - w_xy, w_y - w_xy, w_xy};
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int fx = (b & 1) ? B.bx1 : B.bx0, fy = (b >> 1) ? B.by1 : B.by0;
        if (fc[b] && fx >= 0 && fy >= 0) {
          const int o = fy * nbins + fx;
          if constexpr (STAGED) {   // the CTA histogram
            atomicAdd(hc_cta + o, (unsigned long long)fc[b]);
            atomicAdd(my_s + o, fs[b]);
            if constexpr (WEIGHTED) atomicAdd(my_w + o, fw[b]);
          } else {                  // the private warp histogram
            my_c[o] += fc[b];
            my_s[o] += fs[b];
            if constexpr (WEIGHTED) my_w[o] += fw[b];
          }
        }
      }
    }
    __syncwarp();
  };

  // ---- one ONE_AXIS super pair (one warp, STAGED): per row point against the staged copy of the varying axis ----
  auto decide_one = [&](const int4 e) {
    const int cat = e.x, x0 = e.w & 0xfff, y0 = (e.w >> 16) & 0xfff;
    const bool vx = (e.w & PB_E_VX) != 0;
    const int v0 = vx ? x0 : y0, cb = vx ? y0 : x0;   // varying axis: bins v0, v0 + 1; constant axis: bin cb
    const double t = ed[v0 + 1], tm = -ed[nbins - 1 - v0];   // forward upper bit: d >= t; mirrored upper bit: d <= tm
    const int64_t off = P.cat_off[cat];
    const int64_t rb = off + (int64_t)e.y * PB_SUPER_PTS + lane;
    const double* rc = vx ? P.px : P.py;
    const double *sc = vx ? T.xs : T.ys, *ss = vx ? T.sxk : T.syk, *sw = vx ? T.sxw : T.syw;
    double up_s = 0.0, up_w = 0.0;
    unsigned up_c = 0u;
    // four row points at a time: their loads issued together, then four independent bisections (the pair is bound by
    // the latency of the loads and of the dependent probes, not by their number)
#pragma unroll 1
    for (int h = 0; h < PB_SUPER; h += 4) {
      double ci[4], ki[4], wi[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int64_t i = rb + (h + k) * 32;
        ci[k] = rc[i];
        wi[k] = 1.0;
        if constexpr (WEIGHTED) wi[k] = P.pw[i];
        ki[k] = P.pk[i];
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        pb_one_axis_row<WEIGHTED>(sc, ss, sw, ci[k], ki[k] * wi[k], wi[k], t, tm, v0, cb, vx, cat, P, up_c, up_s, up_w);
    }
    up_c = warp_sum_u(up_c);
    up_s = warp_sum(up_s);
    if constexpr (WEIGHTED) up_w = warp_sum(up_w);
    if (lane == 0) {   // the CTA histogram (forward entries)
      const double2 rsum = *reinterpret_cast<const double2*>(
          sup0 + (size_t)PB_SUPER_STRIDE * (size_t)(off / PB_SUPER_PTS + cat + e.y) + 4);
      const int lo_b = vx ? cb * nbins + v0 : v0 * nbins + cb;
      const int hi_b = vx ? cb * nbins + v0 + 1 : (v0 + 1) * nbins + cb;
      atomicAdd(hc_cta + lo_b, (unsigned long long)((unsigned)(PB_SUPER_PTS * PB_SUPER_PTS) - up_c));
      atomicAdd(my_s + lo_b, rsum.x * T.sxk[0] - up_s);
      atomicAdd(hc_cta + hi_b, (unsigned long long)up_c);
      atomicAdd(my_s + hi_b, up_s);
      if constexpr (WEIGHTED) {
        atomicAdd(my_w + lo_b, rsum.y * T.sxw[0] - up_w);
        atomicAdd(my_w + hi_b, up_w);
      }
    }
    ++st_one;
    __syncwarp();
  };

  if constexpr (STAGED) {
    __shared__ unsigned long long s_item;
    __shared__ unsigned s_next;
    const PBSuperGroups grp = pb_super_groups(P.boxes, P.cat_off, P.ncat);
    const unsigned long long nitems = P.slist_len[2];
    const int nthr = blockDim.x, nwarps = nthr >> 5;
    const int SP = PB_SUPER_PTS, XB = PB_LT_XB, N = PB_LT_N;
    int cur_cat = -1;
    while (true) {
      __syncthreads();   // the previous item's tables are consumed
      if (tid == 0) {
        const unsigned long long q = atomicAdd(P.counter, 1ull);
        s_item = q < nitems ? grp.items[q] : ~0ull;
        s_next = 0u;
      }
      __syncthreads();
      const unsigned long long item = s_item;
      if (item == ~0ull) break;
      const int4* slice = grp.glist + (item >> 16);
      const int len = (int)(item & 0xffff);
      const int4 e0 = slice[0];
      if (e0.x != cur_cat) {
        flush_cta(cur_cat);
        cur_cat = e0.x;
      }
      // ---- stage column super-chunk C: sorted copies, suffix sums; for TWO_AXIS items also k w and w in x order and
      // the links.  An item holds one kind only; ONE_AXIS items need no dominance table ----
      const bool one_item = (e0.w & PB_E_ONE) != 0;
      {
        const int64_t off = P.cat_off[e0.x], slot = off / PB_SUPER_PTS + e0.x + e0.z;
        const double* crec = sup0 + (size_t)PB_SUPER_STRIDE * (size_t)slot + PB_SLOT;
        const unsigned short* lk = grp.links + (size_t)PB_SUPER_PTS * (size_t)slot;
        const int64_t base = off + (int64_t)e0.z * PB_SUPER_PTS;
        for (int i = tid; i < SP; i += nthr) {
          T.xs[i] = crec[i];
          T.sxk[i] = crec[SP + i];
          T.ys[i] = crec[3 * SP + i];
          T.syk[i] = crec[4 * SP + i];
          if constexpr (WEIGHTED) {
            T.sxw[i] = crec[2 * SP + i];
            T.syw[i] = crec[5 * SP + i];
          }
          if (one_item) continue;
          const unsigned l = lk[i];
          const int j = (int)(l & 0xffu), r = (int)(l >> 8);
          double wj = 1.0;
          if constexpr (WEIGHTED) {
            wj = P.pw[base + j];
            T.wx[i] = wj;
          }
          T.kx[i] = P.pk[base + j] * wj;
          T.yr[i] = (unsigned char)r;
          T.xp[r] = (unsigned char)i;
        }
        if (tid == 0) {
          T.sxk[SP] = 0.0;
          T.syk[SP] = 0.0;
          if constexpr (WEIGHTED) { T.sxw[SP] = 0.0; T.syw[SP] = 0.0; }
        }
        for (int i = tid; i < N && !one_item; i += nthr) {   // row NB of U: no x-block
          T.uk[PB_LT_NB * N + i] = 0.0;
          T.uc[PB_LT_NB * N + i] = 0;
          if constexpr (WEIGHTED) T.uw[PB_LT_NB * N + i] = 0.0;
        }
      }
      __syncthreads();
      if (one_item) {   // ---- the slice's ONE_AXIS super pairs, one per warp step ----
        while (true) {
          unsigned k = 0;
          if (lane == 0) k = atomicAdd(&s_next, 1u);
          k = __shfl_sync(0xffffffffu, k, 0);
          if ((int)k >= len) break;
          decide_one(slice[k]);
        }
        continue;
      }
      // in-block y order of every x position; U row by row (one warp per x-block: suffix scans over the y order)
      for (int p = tid; p < SP; p += nthr) {
        const int b0 = p & ~(XB - 1), r = T.yr[p];
        int c = 0;
#pragma unroll
        for (int o = 0; o < XB; ++o) c += T.yr[b0 + o] < r ? 1 : 0;
        T.yo[p] = (unsigned char)c;
      }
      for (int b = warp; b < PB_LT_NB; b += nwarps) {
        double ak = 0.0, aw = 0.0;
        unsigned ac = 0u;
        for (int sg = SP / 32 - 1; sg >= 0; --sg) {
          const int q = sg * 32 + lane, p = T.xp[q];
          const bool in = p >= b * XB;
          double vk = in ? T.kx[p] : 0.0, vw = 0.0;
          if constexpr (WEIGHTED) vw = in ? T.wx[p] : 0.0;
          unsigned vc = in ? 1u : 0u;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const double tk = __shfl_down_sync(0xffffffffu, vk, o);
            const unsigned tc = __shfl_down_sync(0xffffffffu, vc, o);
            double tw = 0.0;
            if constexpr (WEIGHTED) tw = __shfl_down_sync(0xffffffffu, vw, o);
            if (lane + o < 32) { vk += tk; vc += tc; if constexpr (WEIGHTED) vw += tw; }
          }
          vk += ak; vc += ac;
          T.uk[b * N + q] = vk;
          T.uc[b * N + q] = (unsigned short)vc;
          if constexpr (WEIGHTED) { vw += aw; T.uw[b * N + q] = vw; aw = __shfl_sync(0xffffffffu, vw, 0); }
          ak = __shfl_sync(0xffffffffu, vk, 0);
          ac = __shfl_sync(0xffffffffu, vc, 0);
        }
        if (lane == 0) {
          T.uk[b * N + SP] = 0.0;
          T.uc[b * N + SP] = 0;
          if constexpr (WEIGHTED) T.uw[b * N + SP] = 0.0;
        }
      }
      __syncthreads();
      for (int i = tid; i < PB_LT_NB * N; i += nthr) T.qr[i] = (unsigned char)(XB - (T.uc[i] - T.uc[i + N]));
      for (int i = tid; i < PB_LT_NB * (XB + 1); i += nthr) {   // V and the masks: suffix over the in-block x offset
        const int b = i / (XB + 1), q = i % (XB + 1);
        double ak = 0.0, aw = 0.0;
        unsigned m = 0u;
        for (int xo = XB - 1; xo >= 0; --xo) {
          const int p = b * XB + xo;
          if (T.yo[p] >= q) {
            ak += T.kx[p];
            if constexpr (WEIGHTED) aw += T.wx[p];
            m |= 1u << xo;
          }
          T.vk[(b * XB + xo) * (XB + 1) + q] = ak;
          if constexpr (WEIGHTED) T.vw[(b * XB + xo) * (XB + 1) + q] = aw;
        }
        T.msk[i] = m;
      }
      __syncthreads();
      // ---- the slice's super pairs, one per warp step ----
      while (true) {
        unsigned k = 0;
        if (lane == 0) k = atomicAdd(&s_next, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if ((int)k >= len) break;
        decide(slice[k]);
      }
    }
    flush_cta(cur_cat);
  } else {
    const int4* slist = pb_super_list(P);
    const unsigned long long nlist = *P.slist_len;
    int cur_cat = -1, since_flush = 0;
    while (true) {
      unsigned long long q = 0;
      if (lane == 0) q = atomicAdd(P.counter, 1ull);
      q = __shfl_sync(0xffffffffu, q, 0);
      if (q >= nlist) break;
      const int4 e = slist[q];
      // <= 2^16 pairs per super pair and 2^31 / 2^16 super pairs per flush keep the 32-bit warp histogram counts exact
      if (e.x != cur_cat || since_flush >= (1 << 14)) {
        flush_hist(cur_cat);
        cur_cat = e.x;
        since_flush = 0;
      }
      ++since_flush;
      decide(e);
    }
    flush_hist(cur_cat);
  }
  const unsigned long long LEAF = (unsigned long long)PB_CHUNK * PB_CHUNK;
  if (st_closed) atomicAdd(&g_pb_stats[0], LEAF * st_closed);   // per classifying lane
  if (lane == 0) {
    if (st_1d) atomicAdd(&g_pb_stats[1], LEAF * st_1d);
    if (st_pw) atomicAdd(&g_pb_stats[2], LEAF * st_pw);
    if (st_sorted) atomicAdd(&g_pb_stats[3], LEAF * st_sorted);
    if (st_quad) atomicAdd(&g_pb_stats[4], LEAF * st_quad);
    if (st_pairs) atomicAdd(&g_pb_super_leaves, (unsigned long long)st_pairs);
    if (st_rows) atomicAdd(&g_pb_super_rows, (unsigned long long)st_rows);
    if (st_one) {
      atomicAdd(&g_pb_stats[6], (unsigned long long)PB_SUPER_PTS * PB_SUPER_PTS * st_one);
      atomicAdd(&g_pb_super_one_rows, (unsigned long long)st_one);
    }
  }
}

extern "C" int tgp_pairbin_tile(void) { return PB_CHUNK; }

// Records of one round of the two-pass TwoD count (16 bytes each): 2^26 = 1 GiB, about 8 rounds at N = 1e6.
constexpr int64_t PB_REC_CAP = 1ll << 26;
static int64_t g_pb_rec_cap = PB_REC_CAP;   // tgp_set_option("pairbin_record_cap", n): smaller rounds (tests)
extern "C" int tgp_pairbin_set_record_cap(int n) {
  g_pb_rec_cap = n <= 0 ? PB_REC_CAP : (n < 256 ? 256 : n);
  return TGP_OK;
}

// Record slots reserved in the work buffer for catalogues of up to `max_len` points: an item holds at most `run`
// records, and run x (items of one catalogue) <= (nblk + 512)^2 / 2 for run <= 256; capped at PB_REC_CAP.
// Non-decreasing in max_len, so the total point count of the caller's sizing bounds max_cat_len's.
static int64_t pb_rec_slots(int64_t max_len, int32_t ncat) {
  const double nblk = (double)((max_len + PB_CHUNK - 1) / PB_CHUNK);
  const double need = 0.5 * (double)ncat * (nblk + 512.0) * (nblk + 512.0);
  if (need >= (double)PB_REC_CAP) return PB_REC_CAP;
  return ((int64_t)need + 255) / 256 * 256;
}
// Work buffer of the two-pass count: {work counters of pass A, pass B, the super kernel; length of the TWO_AXIS list,
// work counter of the leaf kernel, its number of work items; 2 spare words} {record counts of a round: slots / 32 ints}
// {records: 2 doubles each} {pre-pass chunk records} {super-chunk records} {super pair list: 2 doubles per super pair}
// {the regions of pb_super_groups}.  The other paths keep the chunk records at the start.
static int64_t pb_rec_region_doubles(int64_t slots) { return 8 + slots / 64 + 2 * slots; }

extern "C" int64_t tgp_pairbin_work_doubles(int64_t total_points, int32_t ncat) {
  const int64_t nslot = pb_super_slots(total_points, ncat);
  return pb_rec_region_doubles(pb_rec_slots(total_points, ncat)) +
         (int64_t)PB_STRIDE * (total_points / PB_CHUNK + (int64_t)ncat + 2) + (int64_t)PB_SUPER_STRIDE * nslot +
         4 * pb_super_list_cap(total_points) + (int64_t)PB_SUPER_PTS / 4 * nslot + 2 * nslot +
         pb_super_items_cap(total_points, ncat) + (nslot * pb_super_desc_words(total_points) + 2) / 2;
}

static int g_pb_fast_paths = 7;   // tgp_set_option("pairbin_fast_paths", bits): see PBParams::fast_paths
extern "C" int tgp_pairbin_set_fast_paths(int bits) { g_pb_fast_paths = bits; return TGP_OK; }
static int g_pb_block_sums = 1;   // tgp_set_option("pairbin_block_sums", 0): every pair evaluated individually
extern "C" int tgp_pairbin_set_block_sums(int on) { g_pb_block_sums = on ? 1 : 0; return TGP_OK; }

extern "C" int tgp_pairbin_super_leaves(unsigned long long* host1, int reset) {
  TGP_CHECK_ARG(host1 != nullptr, "host1");
  TGP_CUDA(cudaMemcpyFromSymbol(host1, g_pb_super_leaves, sizeof(unsigned long long)));
  if (reset) {
    const unsigned long long z = 0;
    TGP_CUDA(cudaMemcpyToSymbol(g_pb_super_leaves, &z, sizeof(z)));
  }
  return TGP_OK;
}

extern "C" int tgp_pairbin_super_rows(unsigned long long* host1, int reset) {
  TGP_CHECK_ARG(host1 != nullptr, "host1");
  TGP_CUDA(cudaMemcpyFromSymbol(host1, g_pb_super_rows, sizeof(unsigned long long)));
  if (reset) {
    const unsigned long long z = 0;
    TGP_CUDA(cudaMemcpyToSymbol(g_pb_super_rows, &z, sizeof(z)));
  }
  return TGP_OK;
}

extern "C" int tgp_pairbin_super_one_axis_rows(unsigned long long* host1, int reset) {
  TGP_CHECK_ARG(host1 != nullptr, "host1");
  TGP_CUDA(cudaMemcpyFromSymbol(host1, g_pb_super_one_rows, sizeof(unsigned long long)));
  if (reset) {
    const unsigned long long z = 0;
    TGP_CUDA(cudaMemcpyToSymbol(g_pb_super_one_rows, &z, sizeof(z)));
  }
  return TGP_OK;
}

extern "C" int tgp_pairbin_stats(unsigned long long* host8, int reset) {
  TGP_CHECK_ARG(host8 != nullptr, "host8");
  TGP_CUDA(cudaMemcpyFromSymbol(host8, g_pb_stats, sizeof(unsigned long long) * 8));
  if (reset) {
    unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    TGP_CUDA(cudaMemcpyToSymbol(g_pb_stats, z, sizeof(z)));
  }
  return TGP_OK;
}

// ring of work counters so that launches on different streams do not share one
constexpr int PB_COUNTER_SLOTS = 64;
__device__ unsigned long long g_pb_counters[PB_COUNTER_SLOTS];

extern "C" int tgp_pairbin(const double* px, const double* py, const double* pk, const double* pw,
                           const int64_t* cat_off, int32_t ncat, int64_t max_cat_len, int32_t bin_type,
                           const double* edges, int32_t nbins, double min_sep2, double max_sep,
                           int32_t tile_rank, int32_t tile_nranks, int64_t* npairs, double* sumw,
                           double* sumwkk, double* sumwr, double* work, void* stream) {
  TGP_CHECK_ARG(bin_type == TGP_BIN_TWOD || bin_type == TGP_BIN_LOG, "bin_type");
  TGP_CHECK_ARG(ncat >= 0 && max_cat_len >= 0 && nbins >= 1, "ncat/max_cat_len/nbins");
  TGP_CHECK_ARG(tile_nranks >= 1 && tile_rank >= 0 && tile_rank < tile_nranks, "rank");
  TGP_CHECK_ARG(max_sep > 0.0 && min_sep2 >= 0.0, "separations");
  if (ncat == 0 || max_cat_len < 2) return TGP_OK;
  TGP_CHECK_ARG(px && py && pk && cat_off && edges && npairs && sumw && sumwkk, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;

  PBParams P;
  P.px = px; P.py = py; P.pk = pk; P.pw = pw; P.cat_off = cat_off; P.edges = edges;
  P.npairs = npairs; P.sumw = sumw; P.sumwkk = sumwkk; P.sumwr = sumwr;
  P.ncat = ncat; P.nbins = nbins; P.rank = tile_rank; P.nranks = tile_nranks;
  P.block_sums = g_pb_block_sums;
  P.fast_paths = g_pb_fast_paths;
  const bool twod = bin_type == TGP_BIN_TWOD;
  TGP_CHECK_ARG(!twod || nbins <= 4096, "nbins too large");
  P.nb = twod ? nbins * nbins : nbins;
  if (twod) {
    P.lo2 = min_sep2 > 0.0 ? min_sep2 : 4.9406564584124654e-324;  // r2 != 0
    P.hi = max_sep;
    P.inv_bin = (double)nbins / (2.0 * max_sep);
  } else {
    P.lo2 = min_sep2;
    P.hi = max_sep * max_sep;
    P.inv_bin = 0.0;
  }
  const bool weighted = pw != nullptr;

  // shared memory: every warp owns a private histogram; the budget decides the warps per CTA
  const size_t per_warp = (size_t)P.nb * (8 + 4 + (weighted ? 8 : 0) + (twod ? 0 : 8)) + PB_CHUNK * (16 + 8 + 8) + 16;
  const size_t fixed = (size_t)((nbins + 2) & ~1) * 8;
  const size_t budget = 200 * 1024;
  TGP_CHECK_ARG(fixed + per_warp <= budget, "too many bins for the shared-memory histogram");
  int warps = (int)((100 * 1024 - fixed) / per_warp);  // aim at two CTAs per SM
  if (warps < 1) warps = (int)((budget - fixed) / per_warp);
  if (warps > PB_MAX_WARPS) warps = PB_MAX_WARPS;
  if (warps < 1) warps = 1;
  P.warps = warps;
  const size_t smem = fixed + (size_t)warps * per_warp + 64;
  const int sms = tgp_num_sms();
  const int ctas_per_sm = (2 * smem <= 220 * 1024) ? 2 : 1;
  const int64_t grid_target = (int64_t)sms * ctas_per_sm;

  // work decomposition: item = 32 row points x a run of `run` column chunks
  const int64_t nblk = tgp_cdiv(max_cat_len, PB_CHUNK);
  const double chunk_pairs = 0.5 * (double)nblk * (double)nblk * (double)ncat;
  const double slots = (double)grid_target * warps * tile_nranks;
  int64_t run = (int64_t)(chunk_pairs / (slots * 32.0));  // >= ~32 items per warp slot
  run = (run / 32) * 32;
  if (run < 32) run = 32;
  if (run > 256) run = 256;
  P.run = (int32_t)run;
  const int64_t nruns = tgp_cdiv(nblk, run);
  // items of one catalogue: groups g of `run` rows pair with runs g..nruns-1
  int64_t items = 0;
  for (int64_t g = 0; g < nruns; ++g) {
    const int64_t rows = (nblk - g * run < run) ? (nblk - g * run) : run;
    items += rows * (nruns - g);
  }
  // the decode assumes full groups; the upper bound below covers the (shorter) last group too
  P.items_per_cat = run * (nruns * nruns - nruns * (nruns - 1) / 2);
  (void)items;
  const int64_t total_items = P.items_per_cat * ncat;
  P.my_items = (total_items - tile_rank + tile_nranks - 1) / tile_nranks;
  if (P.my_items <= 0) return TGP_OK;
  int64_t grid = tgp_cdiv(P.my_items, warps);
  if (grid > grid_target) grid = grid_target;

  // TwoD block forms need the pre-pass: two passes per round of items, records and counters in `work`
  const bool split = twod && P.block_sums && work;
  const int64_t rec_slots = split ? pb_rec_slots(max_cat_len, ncat) : 0;
  P.boxes = nullptr;
  P.sorted = nullptr;
  P.q_begin = 0;
  P.q_end = P.my_items;
  P.recs = nullptr;
  P.rec_cnt = nullptr;
  P.counter_next = nullptr;
  P.slist_len = nullptr;
  P.list_one_axis = 0;
  if (work) {
    TGP_CHECK_ARG(((uintptr_t)work % 32) == 0, "work must be 32-byte aligned");
    double* bx = work + (split ? pb_rec_region_doubles(rec_slots) : 0);
    const int64_t warps_needed = nblk * ncat;
    pairbin_boxes_kernel<<<(unsigned)tgp_cdiv(warps_needed * 32, 256), 256, 0, st>>>(px, py, pk, pw, cat_off, ncat, nblk,
                                                                                       bx, bx + PB_SLOT);
    TGP_LAUNCH_CHECK();
    P.boxes = bx;
    P.sorted = bx + PB_SLOT;
  }

  if (split) {
    // [0] pass A's work counter, [1] pass B's, [2] the super kernel's, [3] the TWO_AXIS list length, [4] the leaf
    // kernel's work counter, [5] its number of work items (staged; written by pairbin_super_group_kernel)
    unsigned long long* ctr = reinterpret_cast<unsigned long long*>(work);
    P.rec_cnt = reinterpret_cast<int*>(work + 8);
    P.recs = reinterpret_cast<int4*>(work + 8 + rec_slots / 64);
    const int64_t per_round = (rec_slots < g_pb_rec_cap ? rec_slots : g_pb_rec_cap) / run;   // items
    TGP_CUDA(cudaMemsetAsync(ctr, 0, 5 * sizeof(unsigned long long), st));
    // super-chunk records (they follow the chunk records; the kernels find them from cat_off[ncat]) and the super
    // kernel, which books the super pairs that the classification pass of every round skips
    // kernel, which books the super pairs that the classification pass of every round skips.  Off when the staging
    // buffer leaves no room for a warp histogram (the largest bin counts): then every super pair descends.
    const int64_t nsf_max = max_cat_len / PB_SUPER_PTS;
    const size_t per_warp_s = (size_t)P.nb * (8 + 4 + (weighted ? 8 : 0)) + 3 * PB_SUPER_PTS * 8;
    int warps_s = (int)((budget - fixed - 64) / per_warp_s);
    if (warps_s > PB_MAX_WARPS) warps_s = PB_MAX_WARPS;
    const bool supers = nsf_max >= 2 && warps_s >= 1;
    // the leaf kernel takes the super pairs the super kernel listed (the length stays on the device).  Staged (the
    // per-row form of the 2 x 2 window is on): the list grouped by column super-chunk and kind, the tables of one
    // super-chunk + a CTA histogram + one staged column chunk per warp, 2 CTAs of 8 warps per SM, or one of 16 if only
    // that fits; the ONE_AXIS super pairs are listed too.  Otherwise warp histograms + one staged column chunk per
    // warp, and the super kernel decides the ONE_AXIS super pairs itself.
    const size_t hist_t = (size_t)P.nb * (8 + 8 + (weighted ? 8 : 0));
    auto smem_t = [&](int w) {
      return fixed + (size_t)w * PB_CHUNK * (16 + 8 + 8) + hist_t + pb_leaf_table_bytes(weighted) + 64;
    };
    // what one CTA takes of the SM's 228 KB: dynamic + static shared memory (the item and pair claims) + the 1 KB the
    // driver reserves per CTA, in 128-byte allocation units
    auto cta_t = [&](int w) { return (smem_t(w) + 16 + 1024 + 127) / 128 * 128; };
    int warps_t = 0, ctas_t = 0;
    if (P.fast_paths & 2) {
      if (2 * cta_t(PB_MAX_WARPS) <= 228 * 1024) { warps_t = PB_MAX_WARPS; ctas_t = 2; }
      else if (smem_t(2 * PB_MAX_WARPS) <= 226 * 1024) { warps_t = 2 * PB_MAX_WARPS; ctas_t = 1; }
    }
    PBParams PS = P;
    const int64_t super_items = nsf_max * ((nsf_max + 31) / 32) * ncat;
    PS.items_per_cat = nsf_max;   // the super kernel's items of a catalogue: nsf_max rows x runs of 32 columns
    // every rank sweeps the statuses of all items (the DESCEND bitmap of its classification pass) and books or lists
    // those with item % nranks == rank
    PS.my_items = super_items;
    PS.counter = ctr + 2;
    PS.slist_len = ctr + 3;
    PS.warps = warps_s;
    PS.list_one_axis = warps_t ? 1 : 0;
    const size_t smem_s = fixed + (size_t)warps_s * per_warp_s + 64;
    if (supers) {
      pairbin_super_boxes_kernel<<<(unsigned)(nsf_max * ncat), PB_SUPER_PTS, 0, st>>>(
          px, py, pk, pw, cat_off, ncat, nsf_max, const_cast<double*>(P.boxes));
      TGP_LAUNCH_CHECK();
    }
    if (supers && PS.my_items > 0) {
      static TgpPerDeviceOnce once_s[2];
      const void* kern_s =
          weighted ? (const void*)pairbin_super_kernel<true> : (const void*)pairbin_super_kernel<false>;
      if (tgp_first_use_on_device(once_s[weighted ? 1 : 0]))
        TGP_CUDA(cudaFuncSetAttribute(kern_s, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget));
      int ctas_s = (int)((220 * 1024) / smem_s);
      if (ctas_s > 2) ctas_s = 2;
      if (ctas_s < 1) ctas_s = 1;
      int64_t grid_s = tgp_cdiv(PS.my_items, warps_s);
      if (grid_s > (int64_t)sms * ctas_s) grid_s = (int64_t)sms * ctas_s;
      if (weighted) pairbin_super_kernel<true><<<(unsigned)grid_s, warps_s * 32, smem_s, st>>>(PS);
      else pairbin_super_kernel<false><<<(unsigned)grid_s, warps_s * 32, smem_s, st>>>(PS);
      TGP_LAUNCH_CHECK();
      // the leaf kernel (per_warp_l < per_warp_s, so warps_l >= 1 when it is not staged)
      PBParams PL = P;
      PL.counter = ctr + 4;
      PL.slist_len = ctr + 3;
      if (warps_t) {
        pairbin_super_group_kernel<<<1, 1024, 0, st>>>(PL);
        TGP_LAUNCH_CHECK();
        pairbin_super_scatter_kernel<<<(unsigned)(sms * 4), 256, 0, st>>>(PL);
        TGP_LAUNCH_CHECK();
        PL.warps = warps_t;
        const size_t smem_l = smem_t(warps_t);
        static TgpPerDeviceOnce once_t[2];
        const void* kern_t = weighted ? (const void*)pairbin_super_leaves_kernel<true, true>
                                      : (const void*)pairbin_super_leaves_kernel<false, true>;
        if (tgp_first_use_on_device(once_t[weighted ? 1 : 0]))
          TGP_CUDA(cudaFuncSetAttribute(kern_t, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
        const unsigned grid_t = (unsigned)((int64_t)sms * ctas_t);
        if (weighted) pairbin_super_leaves_kernel<true, true><<<grid_t, warps_t * 32, smem_l, st>>>(PL);
        else pairbin_super_leaves_kernel<false, true><<<grid_t, warps_t * 32, smem_l, st>>>(PL);
        TGP_LAUNCH_CHECK();
      } else {
        const size_t per_warp_l = (size_t)P.nb * (8 + 4 + (weighted ? 8 : 0)) + PB_CHUNK * (16 + 8 + 8);
        int warps_l = (int)((budget - fixed - 64) / per_warp_l);
        if (warps_l > PB_MAX_WARPS) warps_l = PB_MAX_WARPS;
        PL.warps = warps_l;
        const size_t smem_l = fixed + (size_t)warps_l * per_warp_l + 64;
        int ctas_l = (int)((220 * 1024) / smem_l);
        if (ctas_l > PB_LEAVES_MIN_CTAS) ctas_l = PB_LEAVES_MIN_CTAS;
        if (ctas_l < 1) ctas_l = 1;
        static TgpPerDeviceOnce once_l[2];
        const void* kern_l = weighted ? (const void*)pairbin_super_leaves_kernel<true, false>
                                      : (const void*)pairbin_super_leaves_kernel<false, false>;
        if (tgp_first_use_on_device(once_l[weighted ? 1 : 0]))
          TGP_CUDA(cudaFuncSetAttribute(kern_l, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget));
        const unsigned grid_l = (unsigned)((int64_t)sms * ctas_l);
        if (weighted) pairbin_super_leaves_kernel<true, false><<<grid_l, warps_l * 32, smem_l, st>>>(PL);
        else pairbin_super_leaves_kernel<false, false><<<grid_l, warps_l * 32, smem_l, st>>>(PL);
        TGP_LAUNCH_CHECK();
      }
    }
    PBParams PA = P;
    PA.block_sums = supers ? 2 : 1;
    // pass A: warp histograms only (forward entries; bins x (count + sum [+ sum w])), as many warps per CTA as the
    // budget allows (up to 8): every nbins the residual kernel accepts runs
    const size_t per_warp_a = (size_t)P.nb * (8 + 4 + (weighted ? 8 : 0));
    int warps_a = (int)((budget - fixed - 64) / per_warp_a);
    if (warps_a > PB_MAX_WARPS) warps_a = PB_MAX_WARPS;
    PA.warps = warps_a;
    PA.counter = ctr;
    PA.counter_next = ctr + 1;
    const size_t smem_a = fixed + (size_t)warps_a * per_warp_a + 64;   // warps_a >= 1: per_warp_a < the checked per_warp
    int ctas_a = (int)((220 * 1024) / smem_a);
    if (ctas_a > PB_CLASSIFY_MIN_CTAS) ctas_a = PB_CLASSIFY_MIN_CTAS;
    if (ctas_a < 1) ctas_a = 1;
    P.counter = ctr + 1;
    P.counter_next = ctr;
    static TgpPerDeviceOnce once_[2];
    const void* kern_a = weighted ? (const void*)pairbin_classify_kernel<true> : (const void*)pairbin_classify_kernel<false>;
    const void* kern_b = weighted ? (const void*)pairbin_kernel<TGP_BIN_TWOD, true, true>
                                  : (const void*)pairbin_kernel<TGP_BIN_TWOD, false, true>;
    if (tgp_first_use_on_device(once_[weighted ? 1 : 0])) {
      TGP_CUDA(cudaFuncSetAttribute(kern_a, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget));
      TGP_CUDA(cudaFuncSetAttribute(kern_b, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)budget));
    }
    for (int64_t q0 = 0; q0 < P.my_items; q0 += per_round) {
      const int64_t q1 = (q0 + per_round < P.my_items) ? q0 + per_round : P.my_items;
      PA.q_begin = P.q_begin = q0;
      PA.q_end = P.q_end = q1;
      int64_t grid_a = tgp_cdiv(q1 - q0, warps_a), grid_b = tgp_cdiv(q1 - q0, warps);
      if (grid_a > (int64_t)sms * ctas_a) grid_a = (int64_t)sms * ctas_a;
      if (grid_b > grid_target) grid_b = grid_target;
      if (weighted) {
        pairbin_classify_kernel<true><<<(unsigned)grid_a, warps_a * 32, smem_a, st>>>(PA);
        pairbin_kernel<TGP_BIN_TWOD, true, true><<<(unsigned)grid_b, warps * 32, smem, st>>>(P);
      } else {
        pairbin_classify_kernel<false><<<(unsigned)grid_a, warps_a * 32, smem_a, st>>>(PA);
        pairbin_kernel<TGP_BIN_TWOD, false, true><<<(unsigned)grid_b, warps * 32, smem, st>>>(P);
      }
      TGP_LAUNCH_CHECK();
    }
    return TGP_OK;
  }

  static std::atomic<unsigned> launch_seq{0};   // host threads launching on different streams get different slots
  static void* cbase_dev[TGP_MAX_DEVICES] = {};
  void*& cbase = cbase_dev[tgp_current_device()];
  if (!cbase) TGP_CUDA(cudaGetSymbolAddress(&cbase, g_pb_counters));
  P.counter = reinterpret_cast<unsigned long long*>(cbase) + (launch_seq.fetch_add(1u) % PB_COUNTER_SLOTS);
  TGP_CUDA(cudaMemsetAsync(P.counter, 0, sizeof(unsigned long long), st));

#define TGP_PB_LAUNCH(BT, W, BS)                                                                          \
  do {                                                                                                    \
    static TgpPerDeviceOnce once_;                                                                        \
    if (tgp_first_use_on_device(once_))                                                                   \
      TGP_CUDA(cudaFuncSetAttribute(pairbin_kernel<BT, W, BS>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                    (int)budget));                                                        \
    pairbin_kernel<BT, W, BS><<<(unsigned)grid, warps * 32, smem, st>>>(P);                               \
  } while (0)
  if (twod) {   // pair by pair (block forms off, or no work buffer for the pre-pass)
    if (weighted) TGP_PB_LAUNCH(TGP_BIN_TWOD, true, false); else TGP_PB_LAUNCH(TGP_BIN_TWOD, false, false);
  } else {
    if (P.block_sums) {
      if (weighted) TGP_PB_LAUNCH(TGP_BIN_LOG, true, true); else TGP_PB_LAUNCH(TGP_BIN_LOG, false, true);
    } else {
      if (weighted) TGP_PB_LAUNCH(TGP_BIN_LOG, true, false); else TGP_PB_LAUNCH(TGP_BIN_LOG, false, false);
    }
  }
#undef TGP_PB_LAUNCH
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

// ============================================================================================
// Hilbert-curve keys: sorting the points by this key makes consecutive points spatial neighbours,
// which is what lets the pair-binning kernel keep whole 32 x 32 blocks inside a 2 x 2 bin window.
// ============================================================================================
__global__ void hilbert_keys_kernel(const double* __restrict__ x, const double* __restrict__ y, int64_t n,
                                    double x0, double y0, double inv_cell, int order, int64_t* __restrict__ keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned side = 1u << order;
  long long cx = (long long)floor((x[i] - x0) * inv_cell), cy = (long long)floor((y[i] - y0) * inv_cell);
  unsigned ux = (unsigned)(cx < 0 ? 0 : (cx >= (long long)side ? side - 1 : cx));
  unsigned uy = (unsigned)(cy < 0 ? 0 : (cy >= (long long)side ? side - 1 : cy));
  // classic xy -> d conversion
  unsigned long long d = 0;
  for (unsigned s = side >> 1; s > 0; s >>= 1) {
    const unsigned rx = (ux & s) ? 1u : 0u, ry = (uy & s) ? 1u : 0u;
    d += (unsigned long long)s * s * ((3u * rx) ^ ry);
    if (ry == 0) {
      if (rx == 1) { ux = side - 1 - ux; uy = side - 1 - uy; }
      const unsigned t = ux; ux = uy; uy = t;
    }
  }
  keys[i] = (int64_t)d;
}

// ---- the same keys with the bounding square found on the device: no host round trip in the middle of a call ----
__device__ __forceinline__ unsigned long long hb_key(double v) {   // order-preserving map double -> uint64
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double hb_unkey(unsigned long long k) {
  const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}
__global__ void hilbert_bounds_init_kernel(unsigned long long* b4) {
  if (threadIdx.x < 4) b4[threadIdx.x] = (threadIdx.x & 1) ? 0ull : ~0ull;   // {min x, max x, min y, max y}
}
__global__ void __launch_bounds__(256)
hilbert_bounds_kernel(const double* __restrict__ x, const double* __restrict__ y, int64_t n, unsigned long long* b4) {
  double xmin = INFINITY, xmax = -INFINITY, ymin = INFINITY, ymax = -INFINITY;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double a = x[i], b = y[i];
    xmin = fmin(xmin, a); xmax = fmax(xmax, a);
    ymin = fmin(ymin, b); ymax = fmax(ymax, b);
  }
  xmin = warp_min(xmin); xmax = warp_max(xmax);
  ymin = warp_min(ymin); ymax = warp_max(ymax);
  if ((threadIdx.x & 31) == 0 && xmin <= xmax) {
    atomicMin(b4 + 0, hb_key(xmin)); atomicMax(b4 + 1, hb_key(xmax));
    atomicMin(b4 + 2, hb_key(ymin)); atomicMax(b4 + 3, hb_key(ymax));
  }
}
__global__ void hilbert_keys_auto_kernel(const double* __restrict__ x, const double* __restrict__ y, int64_t n,
                                         const unsigned long long* __restrict__ b4, int order,
                                         int64_t* __restrict__ keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double x0 = hb_unkey(b4[0]), x1 = hb_unkey(b4[1]), y0 = hb_unkey(b4[2]), y1 = hb_unkey(b4[3]);
  // the formula of treegp_b200.backend.hilbert_order (same IEEE operations, so the same keys as tgp_hilbert_keys)
  double extent = fmax(__dsub_rn(x1, x0), __dsub_rn(y1, y0));
  extent = extent > 0.0 ? __dmul_rn(extent, 1.0 + 1e-9) : 1.0;
  const double inv_cell = __ddiv_rn((double)(1u << order), extent);
  const unsigned side = 1u << order;
  long long cx = (long long)floor(__dmul_rn(__dsub_rn(x[i], x0), inv_cell));
  long long cy = (long long)floor(__dmul_rn(__dsub_rn(y[i], y0), inv_cell));
  unsigned ux = (unsigned)(cx < 0 ? 0 : (cx >= (long long)side ? side - 1 : cx));
  unsigned uy = (unsigned)(cy < 0 ? 0 : (cy >= (long long)side ? side - 1 : cy));
  unsigned long long d = 0;
  for (unsigned s = side >> 1; s > 0; s >>= 1) {
    const unsigned rx = (ux & s) ? 1u : 0u, ry = (uy & s) ? 1u : 0u;
    d += (unsigned long long)s * s * ((3u * rx) ^ ry);
    if (ry == 0) {
      if (rx == 1) { ux = side - 1 - ux; uy = side - 1 - uy; }
      const unsigned t = ux; ux = uy; uy = t;
    }
  }
  keys[i] = (int64_t)d;
}

extern "C" int tgp_hilbert_keys_auto(const double* x, const double* y, int64_t n, int32_t order, void* scratch32,
                                     int64_t* keys, void* stream) {
  TGP_CHECK_ARG(n >= 0 && order >= 1 && order <= 30, "n/order");
  if (n == 0) return TGP_OK;
  TGP_CHECK_ARG(x && y && keys && scratch32 && ((uintptr_t)scratch32 % 8) == 0, "null / unaligned pointer");
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* b4 = reinterpret_cast<unsigned long long*>(scratch32);
  hilbert_bounds_init_kernel<<<1, 32, 0, st>>>(b4);
  int64_t blocks = tgp_cdiv(n, 256 * 8);
  if (blocks > 4 * tgp_num_sms()) blocks = 4 * tgp_num_sms();
  hilbert_bounds_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, y, n, b4);
  hilbert_keys_auto_kernel<<<(unsigned)tgp_cdiv(n, 256), 256, 0, st>>>(x, y, n, b4, order, keys);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}

extern "C" int tgp_hilbert_keys(const double* x, const double* y, int64_t n, double xmin, double ymin,
                                double extent, int32_t order, int64_t* keys, void* stream) {
  TGP_CHECK_ARG(n >= 0 && order >= 1 && order <= 30 && extent > 0.0, "n/order/extent");
  if (n == 0) return TGP_OK;
  TGP_CHECK_ARG(x && y && keys, "null pointer");
  const double inv_cell = (double)(1u << order) / extent;
  hilbert_keys_kernel<<<(unsigned)tgp_cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(x, y, n, xmin, ymin, inv_cell,
                                                                                  order, keys);
  TGP_LAUNCH_CHECK();
  return TGP_OK;
}
