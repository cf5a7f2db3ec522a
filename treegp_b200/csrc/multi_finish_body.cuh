// Statement body of loglike_multi_finish_kernel (dense.cu), included there and in loglike_multi_batch_finish_kernel,
// so that both compile from one text (as a device function it would not keep the single kernel's SASS).  In scope:
// L, N, ld (the factor), Y (N x r, row-major), r, W with value i of output c at W[c * wcol + i * wrow] (L^-1 y_c, or
// alpha_c with want_alpha), want_alpha, info and out (3 doubles).  1024 threads.
  __shared__ double s[32];
  double a = 0.0;
  for (int64_t i = threadIdx.x; i < N; i += blockDim.x) a += 2.0 * log(L[i * ld + i]);
  const double logdet = block_sum_1024(a, s);
  double chi2 = 0.0;
  for (int c = 0; c < r; ++c) {
    const double* w = W + c * wcol;
    double v = 0.0;
    for (int64_t i = threadIdx.x; i < N; i += blockDim.x)
      v = want_alpha ? fma(Y[i * r + c], w[i * wrow], v) : fma(w[i * wrow], w[i * wrow], v);
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
