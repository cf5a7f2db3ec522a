// Statement body of grad_contract_kernel (selinv.cu), included inside that kernel and inside
// grad_contract_batch_kernel, so that both compile from one text.  It is included rather than called because a device
// function loses what the kernel's launch bounds tell the compiler about threadIdx.x: the single kernel's code would
// change.  In scope: the profile type P and X, N, prof, Z, ld, alpha, re_dev, partials, phi_g as in
// grad_contract_kernel's parameters; blockIdx.x is the tile and blockIdx.y the term of a sum.
  constexpr int RM = OutputsOf<P>::kR;
  __shared__ double xr[GT], yr[GT], ar[GT * RM], xc[GT], yc[GT], ac[GT * RM];
  __shared__ double red[GT_THREADS / 32][P::kSum ? 5 : 4];
  __shared__ double phi_s[P::kPhiSize];
  const KDesc& kd = prof.grad_term();
  const int64_t t = blockIdx.x;
  int64_t I = (int64_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
  while (I * (I + 1) / 2 > t) --I;
  while ((I + 1) * (I + 2) / 2 <= t) ++I;
  const int64_t J = t - I * (I + 1) / 2;
  const int64_t r0 = I * GT, c0 = J * GT;
  const int64_t rend = re_dev ? re_dev[c0 / TGP_OB] : N;   // one past the last envelope row of this block column
  const int tid = threadIdx.x;
  if (r0 >= rend) {
    if (tid < 4) partials[prof.partial(t, tid)] = 0.0;
    if constexpr (P::kSum) {
      if (tid == 4 && blockIdx.y == 0) partials[prof.white_partial(t)] = 0.0;
    }
    return;
  }
  if (prof.stage_phi()) tgp_stage_phi(phi_s, phi_g);
  if (tid < GT) {
    const int64_t r = r0 + tid;
    const bool ok = r < N;
    xr[tid] = ok ? X[r * kd.ndim] : 0.0;
    yr[tid] = (ok && kd.ndim == 2) ? X[r * 2 + 1] : 0.0;
    if constexpr (RM > 1) {
      for (int c = 0; c < prof.nrhs; ++c) ar[tid * RM + c] = ok ? alpha[r * prof.nrhs + c] : 0.0;
    } else {
      ar[tid] = ok ? alpha[r] : 0.0;
    }
  } else if (tid < 2 * GT) {
    const int l = tid - GT;
    const int64_t c = c0 + l;
    const bool ok = c < N;
    xc[l] = ok ? X[c * kd.ndim] : 0.0;
    yc[l] = (ok && kd.ndim == 2) ? X[c * 2 + 1] : 0.0;
    if constexpr (RM > 1) {
      for (int j = 0; j < prof.nrhs; ++j) ac[l * RM + j] = ok ? alpha[c * prof.nrhs + j] : 0.0;
    } else {
      ac[l] = ok ? alpha[c] : 0.0;
    }
  }
  __syncthreads();
  const int lane = tid & 31, warp = tid >> 5;
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  double sw = 0.0;   // sums: the white column
#pragma unroll(P::kHeavy ? 1 : GT / 8)
  for (int rr = 0; rr < GT / 8; ++rr) {
    const int rl = warp + 8 * rr;
    const int64_t rg = r0 + rl;
    if (rg >= N || rg >= rend) continue;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int cl = 2 * lane + h;
      const int64_t cg = c0 + cl;
      if (cg > rg) continue;
      const double dx = xr[rl] - xc[cl], dy = yr[rl] - yc[cl];
      const double q = tgp_qform(kd, dx, dy);
      double wij;
      if constexpr (RM > 1) {
        const double* a = ar + rl * RM;
        const double* b = ac + cl * RM;
        double aa = a[0] * b[0];
        for (int c = 1; c < prof.nrhs; ++c) aa = fma(a[c], b[c], aa);
        wij = (rg == cg ? 1.0 : 2.0) * (aa - (double)prof.nrhs * Z[rg * ld + cg]);
      } else {
        wij = (rg == cg ? 1.0 : 2.0) * (ar[rl] * ac[cl] - Z[rg * ld + cg]);
      }
      double f = prof.f(kd, q, phi_s);
      // K(X, X) of the von Karman kernels is 0 between distinct coincident points (kmat.cu, kernels.py:253-262)
      if (prof.vk(kd) && q == 0.0 && rg != cg) f = 0.0;
      if constexpr (P::kSum) {
        if (rg == cg) sw += wij;
      }
      s[0] = fma(wij, kd.amp * f, s[0]);
      if (q > 0.0) {
        const double d = wij * kd.amp * prof.fdq(kd, q, phi_s);
        s[1] = fma(d, dx * dx, s[1]);
        s[2] = fma(d, 2.0 * dx * dy, s[2]);
        s[3] = fma(d, dy * dy, s[3]);
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[c] += __shfl_xor_sync(0xffffffffu, s[c], o);
  }
  if constexpr (P::kSum) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sw += __shfl_xor_sync(0xffffffffu, sw, o);
    if (lane == 0) red[warp][4] = sw;
  }
  if (lane == 0) {
#pragma unroll
    for (int c = 0; c < 4; ++c) red[warp][c] = s[c];
  }
  __syncthreads();
  if (tid < 4) {
    double v = 0.0;
    for (int wi = 0; wi < GT_THREADS / 32; ++wi) v += red[wi][tid];
    partials[prof.partial(t, tid)] = v;
  }
  if constexpr (P::kSum) {
    if (tid == 4 && blockIdx.y == 0) {
      double v = 0.0;
      for (int wi = 0; wi < GT_THREADS / 32; ++wi) v += red[wi][4];
      partials[prof.white_partial(t)] = prof.desc.white * v;
    }
  }
