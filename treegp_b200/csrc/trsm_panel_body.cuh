// Statement body of trsm_panel_kernel (dense.cu), included inside that kernel and inside selinv_leaf_batch_kernel,
// so that both compile from one text.  It is included rather than called because a device function loses what the
// kernel's launch bounds tell the compiler about threadIdx.x: the single kernel's code would change.  In scope: FULL
// and L, nb, ldl, B, M, ldb as in trsm_panel_kernel's parameters; blockIdx.x is the block of TRSM_ROWS rows.
  extern __shared__ __align__(16) double tsm[];
  double* LsT = tsm;                 // NB x NB, LsT[j*NB + i] = L[i][j] (column j contiguous), zero padded
  double* dinv = tsm + NB * NB;      // 1 / L[j][j]
  double* Bs = dinv + NB;            // TRSM_ROWS x NB_PITCH (edge path only)
  const int tid = threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.x * TRSM_ROWS;
  const int64_t gr = r0 + tid;
  double x[NB];
  if (FULL) {
    if (gr < M) {
      const double2* row = reinterpret_cast<const double2*>(B + gr * ldb);
#pragma unroll
      for (int j = 0; j < NB / 2; ++j) { const double2 v = row[j]; x[2 * j] = v.x; x[2 * j + 1] = v.y; }
    } else {
#pragma unroll
      for (int j = 0; j < NB; ++j) x[j] = 0.0;
    }
  }
  if (FULL && ((ldl & 1) == 0) && (((uintptr_t)L & 15) == 0)) {
    // one batch of 32 independent 16-byte loads per thread: element pairs (i, 2c), (i, 2c+1) of the L tile
    double2 lv[NB * NB / 2 / TRSM_ROWS];
#pragma unroll
    for (int q = 0; q < NB * NB / 2 / TRSM_ROWS; ++q) {
      const int idx = tid + q * TRSM_ROWS;       // pair index: row i = idx / 32, column pair c = idx % 32
      lv[q] = *reinterpret_cast<const double2*>(L + (int64_t)(idx >> 5) * ldl + 2 * (idx & 31));
    }
#pragma unroll
    for (int q = 0; q < NB * NB / 2 / TRSM_ROWS; ++q) {
      const int idx = tid + q * TRSM_ROWS;
      const int i = idx >> 5, j = 2 * (idx & 31);
      LsT[j * NB + i] = (j < i) ? lv[q].x : 0.0;
      LsT[(j + 1) * NB + i] = (j + 1 < i) ? lv[q].y : 0.0;
    }
  } else {
#pragma unroll 16
    for (int idx = tid; idx < NB * NB; idx += TRSM_ROWS) {
      const int i = idx / NB, j = idx % NB;  // coalesced along j
      double v = 0.0;
      if (i < nb && j < i) v = L[(int64_t)i * ldl + j];
      LsT[j * NB + i] = v;
    }
  }
  if (tid < NB) dinv[tid] = (tid < nb) ? 1.0 / L[(int64_t)tid * ldl + tid] : 1.0;
  if (!FULL) {
    for (int idx = tid; idx < TRSM_ROWS * NB; idx += TRSM_ROWS) {
      const int r = idx / NB, j = idx % NB;
      const int64_t g2 = r0 + r;
      Bs[r * NB_PITCH + j] = (g2 < M && j < nb) ? B[g2 * ldb + j] : 0.0;
    }
  }
  __syncthreads();
  if (!FULL) {
#pragma unroll
    for (int j = 0; j < NB; ++j) x[j] = Bs[tid * NB_PITCH + j];
  }
#pragma unroll
  for (int j = 0; j < NB; ++j) {
    x[j] *= dinv[j];
    const double nx = -x[j];
#pragma unroll
    for (int ip = ((j + 1) & ~1); ip < NB; ip += 2) {  // pairs (ip, ip+1); entries with i <= j are zero/skipped
      const double2 l = *reinterpret_cast<const double2*>(LsT + j * NB + ip);
      if (ip > j) x[ip] = fma(nx, l.x, x[ip]);
      x[ip + 1] = fma(nx, l.y, x[ip + 1]);
    }
  }
  if (FULL) {
    if (gr < M) {
      double2* row = reinterpret_cast<double2*>(B + gr * ldb);
#pragma unroll
      for (int j = 0; j < NB / 2; ++j) row[j] = make_double2(x[2 * j], x[2 * j + 1]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < NB; ++j) Bs[tid * NB_PITCH + j] = x[j];
    __syncthreads();
    for (int idx = tid; idx < TRSM_ROWS * NB; idx += TRSM_ROWS) {
      const int r = idx / NB, j = idx % NB;
      const int64_t g2 = r0 + r;
      if (g2 < M && j < nb) B[g2 * ldb + j] = Bs[r * NB_PITCH + j];
    }
  }
