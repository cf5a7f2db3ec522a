// Body of var_from_rows_kernel (predict.cu), included as statements by that kernel and by its batched twin
// var_rows_batch_kernel, so that both compile the same code: var[m] = amp - sum_n V[m][n]^2 for row
// m = 8 blockIdx.x + warp, one warp per row.  In scope: V, M, N, ldv, amp, var.
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
