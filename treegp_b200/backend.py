"""Device-side operators of the GP hot path: thin wrappers that hand torch CUDA tensors
(device memory + current stream: plumbing) to the C ABI in libtreegp_b200.so.

Every function here requires a CUDA device; nothing falls back to the CPU.
"""
import ctypes
import numpy as np
import torch

from . import _cabi
from ._cabi import TgpKernel, TgpKernelSum, check

F64 = torch.float64


def require_cuda():
    if not torch.cuda.is_available():
        raise _cabi.TgpError("treegp_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")
    return torch.device("cuda", torch.cuda.current_device())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def to_device(a, dtype=F64, non_blocking=False):
    """numpy / tensor -> contiguous CUDA tensor (no copy if already there).  non_blocking: the copy is only
    enqueued on the current stream -- it overlaps host work when the source is page-locked (a pageable source
    is staged before the call returns); the caller must not change the source before the stream has passed it."""
    dev = require_cuda()
    if isinstance(a, torch.Tensor):
        return a.to(device=dev, dtype=dtype, non_blocking=non_blocking).contiguous()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(dev, non_blocking=non_blocking)


def as_points(X):
    """(N,) or (N, d) host/device array -> (N, d) contiguous CUDA tensor, d in {1, 2}."""
    Xd = to_device(X)
    if Xd.dim() == 1:
        Xd = Xd.reshape(-1, 1)
    if Xd.dim() != 2 or Xd.shape[1] not in (1, 2):
        raise ValueError("coordinates must have shape (N, 1) or (N, 2); got %r" % (tuple(Xd.shape),))
    return Xd.contiguous()


def even(n):
    return (int(n) + 1) & ~1


def alloc_matrix(rows, cols, device=None):
    """rows x cols FP64 workspace with an even leading dimension (16-byte rows for the DMMA loads)."""
    dev = device or require_cuda()
    return torch.empty((int(rows), even(cols)), dtype=F64, device=dev)


def _check_dims(kdesc, X, Xs=None):
    """The device kernels index coordinates with the descriptor's ndim: a mismatch would read past the buffers
    (the reference raises from pdist / cdist in that case)."""
    if X.shape[1] != kdesc.ndim:
        raise ValueError("kernel is %d-dimensional but the coordinates have %d columns" % (kdesc.ndim, X.shape[1]))
    if Xs is not None and Xs.shape[1] != X.shape[1]:
        raise ValueError("XA and XB must have the same number of columns (%d vs %d)" % (Xs.shape[1], X.shape[1]))


def is_sum(kdesc):
    """True for a TgpKernelSum (the *_sum entry points), False for a single-term TgpKernel."""
    return isinstance(kdesc, TgpKernelSum)


def as_sum(kdesc):
    """The descriptor as a TgpKernelSum (the *_sum and multi-output entries): a TgpKernel becomes a one-term sum
    without white, which those entries hand to the single-term entries, bit for bit."""
    if is_sum(kdesc):
        return kdesc
    s = TgpKernelSum()
    s.nterms, s.ndim, s.white = 1, kdesc.ndim, 0.0
    s.term[0] = kdesc
    return s


def _outputs(v, N, name):
    """Number of outputs r of `v`: (N,) is one output, (N, r) r of them with 1 <= r <= MAX_RHS."""
    r = 1 if v.dim() == 1 else int(v.shape[1]) if v.dim() == 2 else 0
    if not (1 <= r <= _cabi.MAX_RHS and v.shape[0] == N):
        raise ValueError("%s must have shape (N,) or (N, r) = (%d, r) with 1 <= r <= %d; got %r"
                         % (name, N, _cabi.MAX_RHS, tuple(v.shape)))
    return r


def _envelope(row_end):
    """(pointer, block count) of an optional envelope (envelope_rows) for the C entries."""
    return (None, 0) if row_end is None else (_host_i64(row_end), len(row_end))


def kmat_sym(X, kdesc, diag_add=None, out=None, lower_only=False):
    """K(X,X) + diag(diag_add).  Returns the (N, ld) workspace; the matrix is out[:, :N].  kdesc: TgpKernel or
    TgpKernelSum (every function here that takes a descriptor accepts both)."""
    X = as_points(X)
    _check_dims(kdesc, X)
    N = X.shape[0]
    if out is None:
        out = alloc_matrix(N, N, X.device)
    check(_cabi.load().tgp_kmat_sym_sum(_p(X), N, ctypes.byref(as_sum(kdesc)), _p(diag_add), _p(out), out.stride(0),
                                        int(bool(lower_only)), _stream()), "tgp_kmat_sym_sum")
    return out


def kmat_cross(Xs, X, kdesc, out=None):
    Xs, X = as_points(Xs), as_points(X)
    _check_dims(kdesc, X, Xs)
    M, N = Xs.shape[0], X.shape[0]
    if out is None:
        out = alloc_matrix(M, N, X.device)
    check(_cabi.load().tgp_kmat_cross_sum(_p(Xs), M, _p(X), N, ctypes.byref(as_sum(kdesc)), _p(out), out.stride(0),
                                          _stream()), "tgp_kmat_cross_sum")
    return out


def potrf(A, N, row_end=None):
    """In-place lower Cholesky of the leading N x N block of the workspace A.  Returns info (device int32).
    row_end: restrict the factorisation to that envelope (envelope_rows; tgp_potrf_env)."""
    info = torch.zeros(1, dtype=torch.int32, device=A.device)
    if row_end is None:
        check(_cabi.load().tgp_potrf(_p(A), N, A.stride(0), _p(info), _stream()), "tgp_potrf")
    else:
        check(_cabi.load().tgp_potrf_env(_p(A), N, A.stride(0), _host_i64(row_end), len(row_end), 0, _p(info),
                                         _stream()), "tgp_potrf_env")
    return info


def _host_i64(a):
    """Pointer to a host int64 array the C side reads during the call (envelopes)."""
    if not (isinstance(a, np.ndarray) and a.dtype == np.int64 and a.flags["C_CONTIGUOUS"]):
        raise TypeError("envelope must be a contiguous int64 numpy array")
    return ctypes.c_void_p(a.ctypes.data)


# ---- envelopes: K(X, X) of points sorted along one axis is zero (below 1e-40 amp) beyond the kernel's support ----
def envelope_block():
    return int(_cabi.load().tgp_envelope_block())


def envelope_rows(x_sorted, dcut, start=0):
    """Envelope of K for the points x_sorted[start:] (ascending coordinates along the sorting axis, host array):
    per block of envelope_block() columns the first row that is farther than `dcut` from every point of the block
    (and of all earlier blocks).  int64 array for the *_env entry points."""
    x = np.asarray(x_sorted, dtype=np.float64)[int(start):]
    n, ob = len(x), envelope_block()
    c1 = np.minimum(np.arange(ob, n + ob, ob), n)          # one past the last column of every block
    reach = x[c1 - 1] + dcut * (1.0 + 1e-9)                 # a hair wider: the device forms fl(x_i - x_j)
    return np.ascontiguousarray(np.maximum(np.searchsorted(x, reach, side="left"), c1), dtype=np.int64)


def envelope_flops(row_end, n):
    """Flop count of tgp_potrf_env for that envelope (diagonal blocks + panel solves + trailing updates)."""
    ob = envelope_block()
    k = np.arange(0, n, ob, dtype=np.float64)
    w = np.minimum(ob, n - k)
    below = np.maximum.accumulate(np.clip(np.asarray(row_end, dtype=np.float64), k + w, n)) - (k + w)
    return float(np.sum(w ** 3 / 3.0 + w * w * below + w * below * below))


ENVELOPE_MIN_N = 4096      # below this the dense factorisation takes a few ms at most
ENVELOPE_MIN_GAIN = 2.0    # use the envelope when it needs at most 1/2 of the dense flops (its GEMMs are smaller)


def plan_envelope(X, kdesc, sorted_axes=None):
    """Decide whether K(X, X) for this kernel is worth factorising inside its envelope.  Returns None (dense), or a
    dict: axis, dcut, order (device index tensor: points ascending along `axis`), x (their coordinates along it, host),
    row_end, flops, flops_dense.  sorted_axes: optional cache {axis: (order, x_host)} filled / reused across calls with
    the same X (the likelihood search evaluates many kernels on one point set)."""
    N = int(X.shape[0])
    if N < ENVELOPE_MIN_N:
        return None
    dcut = np.asarray(support_cutoffs(kdesc), dtype=np.float64)
    if not np.all(np.isfinite(dcut)):
        return None
    cache = sorted_axes if sorted_axes is not None else {}
    if "extent" not in cache:
        lo_hi = torch.stack([X.amin(dim=0), X.amax(dim=0)]).cpu().numpy()
        cache["extent"] = np.maximum(lo_hi[1] - lo_hi[0], 1e-300)
    extent = cache["extent"]
    axis = int(np.argmin(dcut / extent))
    if dcut[axis] >= 0.7 * extent[axis]:
        return None
    if axis not in cache:
        order = torch.argsort(X[:, axis], stable=True)
        cache[axis] = (order, X[order, axis].cpu().numpy())
    order, x = cache[axis]
    row_end = envelope_rows(x, dcut[axis])
    f_env, f_dense = envelope_flops(row_end, N), float(N) ** 3 / 3.0
    if f_env * ENVELOPE_MIN_GAIN > f_dense:
        return None
    return {"axis": axis, "dcut": float(dcut[axis]), "order": order, "x": x, "row_end": row_end,
            "flops": f_env, "flops_dense": f_dense}


def potrs_vec(L, N, b):
    """Solve L L^T x = b in place (b: N-vector on the device)."""
    check(_cabi.load().tgp_potrs_vec(_p(L), N, L.stride(0), _p(b), _stream()), "tgp_potrs_vec")
    return b


def potrs_multi(L, N, B):
    """Solve L L^T X = B in place for the r rows of B (device tensor (r, >= N) with B.stride(0) == L.stride(0)); one
    pass over the factor per sweep for all rows (tgp_potrs_multi)."""
    if B.dim() != 2 or B.stride(0) != L.stride(0) or not 1 <= B.shape[0] <= _cabi.MAX_RHS:
        raise ValueError("B must be (r, ld) with the factor's row pitch and 1 <= r <= %d" % _cabi.MAX_RHS)
    check(_cabi.load().tgp_potrs_multi(_p(L), N, L.stride(0), _p(B), int(B.shape[0]), _stream()), "tgp_potrs_multi")
    return B


def trsm_rows(L, N, B, M, row_end=None):
    """B[:M, :N] <- B L^-T in place.  row_end: the factor's envelope (envelope_rows) -- solved blocks are only
    propagated to the rows inside it."""
    if row_end is None:
        check(_cabi.load().tgp_trsm_rows(_p(L), N, L.stride(0), _p(B), M, B.stride(0), _stream()), "tgp_trsm_rows")
    else:
        check(_cabi.load().tgp_trsm_rows_env(_p(L), N, L.stride(0), _host_i64(row_end), len(row_end), _p(B), M,
                                             B.stride(0), _stream()), "tgp_trsm_rows_env")
    return B


def gemm_nt_sub(C, M, Nc, A, B, Kd, lower_only=False):
    """C[:M, :Nc] -= A[:M, :Kd] @ B[:Nc, :Kd].T in place."""
    check(_cabi.load().tgp_gemm_nt_sub(_p(C), M, Nc, C.stride(0), _p(A), A.stride(0), _p(B), B.stride(0), Kd,
                                       int(bool(lower_only)), _stream()), "tgp_gemm_nt_sub")
    return C


def logdet_chi2(L, N, y=None, alpha=None):
    out = torch.zeros(2, dtype=F64, device=L.device)
    check(_cabi.load().tgp_logdet_chi2(_p(L), N, L.stride(0), _p(y), _p(alpha), _p(out), _stream()),
          "tgp_logdet_chi2")
    return out


def _solve_args(X, y, yerr2, work, name):
    """Points, N, the number of outputs r of y ((N,) or (N, r)) and a workspace of N + r rows (the outputs ride
    through the factorisation as extra rows)."""
    X = as_points(X)
    N = X.shape[0]
    r = _outputs(y, N, "y")
    if yerr2 is not None and tuple(yerr2.shape) != (N,):
        raise ValueError("yerr2 must have shape (N,) = (%d,); got %r" % (N, tuple(yerr2.shape)))
    if work is None:
        work = alloc_matrix(N + r, N, X.device)
    if work.shape[0] < N + r:
        raise ValueError("%s workspace needs N+%d rows" % (name, r))
    return X, N, r, work


def loglike(X, y, yerr2, kdesc, work=None, want_alpha=False, row_end=None):
    """One marginal-likelihood evaluation (tgp_loglike_multi).  y: (N,), or (N, r) for r outputs sharing the kernel,
    whose joint logL is the sum of theirs.  Returns (out[3] = logL, chi2, logdet; info; alpha, shaped as y; work,
    N + r rows).  row_end: X (with y, yerr2) is sorted along an axis and the factorisation stays inside that envelope
    (plan_envelope)."""
    X, N, r, work = _solve_args(X, y, yerr2, work, "loglike")
    y = y.contiguous()
    alpha = torch.empty(y.shape, dtype=F64, device=X.device)
    out = torch.zeros(3, dtype=F64, device=X.device)
    info = torch.zeros(1, dtype=torch.int32, device=X.device)
    re, nre = _envelope(row_end)
    check(_cabi.load().tgp_loglike_multi(_p(X), _p(y), r, _p(yerr2), N, ctypes.byref(as_sum(kdesc)), _p(work),
                                         work.stride(0), _p(alpha), int(bool(want_alpha)), _p(out), _p(info), re, nre,
                                         _stream()), "tgp_loglike_multi")
    return out, info, alpha, work


def _selinv_scratch(N, device):
    return torch.empty(int(_cabi.load().tgp_selinv_work_doubles(int(N))), dtype=F64, device=device)


def selinv(L, N, row_end=None):
    """In place on the factor L (workspace of potrf / loglike): Z = (L L^T)^-1 on every entry of the envelope row_end
    (None: the whole matrix), lower triangle mirrored into the upper one (tgp_selinv).  Returns L."""
    scratch = _selinv_scratch(N, L.device)
    re = None if row_end is None else _host_i64(row_end)
    check(_cabi.load().tgp_selinv(_p(L), int(N), L.stride(0), re, 0 if row_end is None else len(row_end), _p(scratch),
                                  _stream()), "tgp_selinv")
    return L


def selinv_flops(row_end, n):
    """Flop count of tgp_selinv for that envelope (None: dense): per block column of width w with m envelope rows
    below it, w^3 (the inverse of the diagonal block) + 2 w^2 m (T) + 2 w m^2 (Z[R, J]) + w^3 + w^2 m (Z[J, J])."""
    ob = envelope_block()
    k = np.arange(0, n, ob, dtype=np.float64)
    w = np.minimum(ob, n - k)
    re = np.full(len(k), float(n)) if row_end is None else np.asarray(row_end, dtype=np.float64)
    m = np.maximum.accumulate(np.clip(re, k + w, n)) - (k + w)
    return float(np.sum(2.0 * w ** 3 + 3.0 * w * w * m + 2.0 * w * m * m))


def loglike_grad(X, y, yerr2, kdesc, work=None, row_end=None):
    """Log-likelihood and its gradient in one call.  Returns (out; info; alpha = K^-1 y, shaped as y; work, which holds
    Z = K^-1 inside the envelope afterwards).  y and row_end as for loglike.  A TgpKernel with y of shape (N,)
    (tgp_loglike_grad): out[7] = logL, chi2, logdet, d logL / d ln amp, d logL / d m00, d m01, d m11.  A sum, or r
    outputs (tgp_loglike_grad_multi: the joint logL): out has 4 + 4 nterms entries, the four derivatives per term,
    then d logL / d ln white; a TgpKernel counts as one term."""
    X, N, r, work = _solve_args(X, y, yerr2, work, "loglike_grad")
    _check_dims(kdesc, X)
    y = y.contiguous()
    alpha = torch.empty(y.shape, dtype=F64, device=X.device)
    info = torch.zeros(1, dtype=torch.int32, device=X.device)
    re, nre = _envelope(row_end)
    lib = _cabi.load()
    if y.dim() == 1 and not is_sum(kdesc):
        # the single-term entry: as a one-term sum it would take one more launch (clearing d / d ln white) and a
        # larger scratch
        out = torch.zeros(7, dtype=F64, device=X.device)
        check(lib.tgp_loglike_grad(_p(X), _p(y), _p(yerr2), N, ctypes.byref(kdesc), _p(work), work.stride(0),
                                   _p(alpha), _p(out), _p(info), re, nre, _p(_selinv_scratch(N, X.device)), _stream()),
              "tgp_loglike_grad")
        return out, info, alpha, work
    ks = as_sum(kdesc)
    out = torch.zeros(4 + 4 * ks.nterms, dtype=F64, device=X.device)
    scratch = torch.empty(int(lib.tgp_loglike_grad_multi_work_doubles(int(N), int(ks.nterms), r)), dtype=F64,
                          device=X.device)
    check(lib.tgp_loglike_grad_multi(_p(X), _p(y), r, _p(yerr2), N, ctypes.byref(ks), _p(work), work.stride(0),
                                     _p(alpha), _p(out), _p(info), re, nre, _p(scratch), _stream()),
          "tgp_loglike_grad_multi")
    return out, info, alpha, work


# ---- batches of independent problems (tgp_loglike_batch / tgp_predict_mean_batch) ----------------------------------
def batch_offsets(sizes):
    """Host int64 offsets [0, n_0, n_0 + n_1, ...] of problems with `sizes` points."""
    return np.ascontiguousarray(np.concatenate([[0], np.cumsum(np.asarray(sizes, dtype=np.int64))]), dtype=np.int64)


def batch_work_doubles(sizes, r=1):
    """Workspace of tgp_loglike_batch_multi with r outputs: sum_b (N_b + r) * ld_b doubles, ld_b = N_b rounded up to
    even."""
    n = np.asarray(sizes, dtype=np.int64)
    return int(np.sum((n + r) * ((n + 1) & ~1)))


def grad_batch_scratch_doubles(sizes):
    """Scratch of tgp_loglike_grad_batch: sum_b of tgp_loglike_grad_sum_work_doubles(N_b, TGP_MAX_TERMS), i.e. the
    larger of the selected-inverse blocks (2 OB^2 + OB even(N)) and 4 TGP_MAX_TERMS + 1 partial sums per 64 x 64
    contraction tile, plus even(ceil(N / OB)) for the envelope copy (OB = 512)."""
    n = np.asarray(sizes, dtype=np.int64)
    ob, ev = 512, (n + 1) & ~1
    nt = (n + 63) // 64
    selinv = 2 * ob * ob + ob * ev
    partials = (4 * _cabi.MAX_TERMS + 1) * (nt * (nt + 1) // 2)
    nblk = (n + ob - 1) // ob
    return int(np.sum(np.maximum(selinv, partials) + ((nblk + 1) & ~1)))


def plan_batch_chunks(sizes, budget_bytes, scratch=False, r=1):
    """Split problems with `sizes` points, in order, into consecutive chunks whose loglike_batch workspace for r
    outputs (plus, with scratch=True, the loglike_grad_batch scratch) fits `budget_bytes`; a problem larger than the
    budget gets a chunk of its own.  Pure host function: returns a list of (start, stop) index pairs covering
    range(len(sizes))."""
    chunks, start, used = [], 0, 0
    for b, n in enumerate(sizes):
        need = 8 * batch_work_doubles([n], r) + (8 * grad_batch_scratch_doubles([n]) if scratch else 0)
        if b > start and used + need > budget_bytes:
            chunks.append((start, b))
            start, used = b, 0
        used += need
    if len(sizes):
        chunks.append((start, len(sizes)))
    return chunks


def _ksum_array(descs):
    arr = (TgpKernelSum * len(descs))()
    for b, d in enumerate(descs):
        arr[b] = as_sum(d)
    return arr


def _check_batch_inputs(X, sizes, descs):
    if len(sizes) != len(descs) or len(sizes) == 0:
        raise ValueError("need one kernel descriptor per problem (%d sizes, %d descriptors)" % (len(sizes), len(descs)))
    if X.shape[0] != int(np.sum(sizes)):
        raise ValueError("X has %d rows but the problems have %d points" % (X.shape[0], int(np.sum(sizes))))
    for d in descs:
        _check_dims(d, X)


def loglike_batch(X, y, yerr2, sizes, descs, want_alpha=False, budget_bytes=4 << 30):
    """tgp_loglike_batch_multi over B problems: X (sum N_b, ndim), y (sum N_b,) or (sum N_b, r) for r outputs sharing
    each problem's kernel, and yerr2 (sum N_b,) concatenated device tensors, problem b owning `sizes[b]` consecutive
    rows; descs: B descriptors (TgpKernel or TgpKernelSum).  The problems are put through in chunks whose workspace
    fits `budget_bytes` (plan_batch_chunks); the results do not depend on the chunking.  Returns (out (B, 3) = logL,
    chi2, logdet per problem, joint over the outputs; info (B,); alpha, shaped as y: K^-1 y with want_alpha, else
    L^-1 y)."""
    X = as_points(X)
    sizes = [int(n) for n in sizes]
    _check_batch_inputs(X, sizes, descs)
    r = _outputs(y, X.shape[0], "y")
    y = y.contiguous()
    off = batch_offsets(sizes)
    B = len(sizes)
    out = torch.empty((B, 3), dtype=F64, device=X.device)
    info = torch.empty(B, dtype=torch.int32, device=X.device)
    alpha = torch.empty(y.shape, dtype=F64, device=X.device)
    lib = _cabi.load()
    for b0, b1 in plan_batch_chunks(sizes, budget_bytes, r=r):
        r0, r1 = int(off[b0]), int(off[b1])
        o = np.ascontiguousarray(off[b0:b1 + 1] - off[b0])
        work = torch.empty(batch_work_doubles(sizes[b0:b1], r), dtype=F64, device=X.device)
        ks = _ksum_array(descs[b0:b1])
        check(lib.tgp_loglike_batch_multi(_p(X[r0:r1]), _p(y[r0:r1]), r, _p(yerr2[r0:r1]), _host_i64(o), b1 - b0,
                                          ctypes.cast(ks, ctypes.c_void_p), _p(work), _p(alpha[r0:r1]),
                                          int(bool(want_alpha)), _p(out[b0:b1]), _p(info[b0:b1]), _stream()),
              "tgp_loglike_batch_multi")
    return out, info, alpha


def loglike_grad_batch(X, y, yerr2, sizes, descs, budget_bytes=4 << 30):
    """tgp_loglike_grad_batch_multi over B problems, arguments as loglike_batch: each problem's (joint) log-likelihood
    and its gradient in one pass, in chunks whose workspace plus scratch fit `budget_bytes`
    (plan_batch_chunks(scratch=True)); the results do not depend on the chunking.  Returns (out (B,
    TGP_GRAD_BATCH_OUT): per problem the layout of loglike_grad for a sum, {logL, chi2, logdet, 4 derivatives per term,
    d / d ln white}, zero-padded; info (B,); alpha = K^-1 y, shaped as y)."""
    X = as_points(X)
    sizes = [int(n) for n in sizes]
    _check_batch_inputs(X, sizes, descs)
    r = _outputs(y, X.shape[0], "y")
    y = y.contiguous()
    off = batch_offsets(sizes)
    B = len(sizes)
    out = torch.empty((B, _cabi.GRAD_BATCH_OUT), dtype=F64, device=X.device)
    info = torch.empty(B, dtype=torch.int32, device=X.device)
    alpha = torch.empty(y.shape, dtype=F64, device=X.device)
    lib = _cabi.load()
    for b0, b1 in plan_batch_chunks(sizes, budget_bytes, scratch=True, r=r):
        r0, r1 = int(off[b0]), int(off[b1])
        o = np.ascontiguousarray(off[b0:b1 + 1] - off[b0])
        work = torch.empty(batch_work_doubles(sizes[b0:b1], r), dtype=F64, device=X.device)
        scratch = torch.empty(grad_batch_scratch_doubles(sizes[b0:b1]), dtype=F64, device=X.device)
        ks = _ksum_array(descs[b0:b1])
        check(lib.tgp_loglike_grad_batch_multi(_p(X[r0:r1]), _p(y[r0:r1]), r, _p(yerr2[r0:r1]), _host_i64(o),
                                               b1 - b0, ctypes.cast(ks, ctypes.c_void_p), _p(work), _p(alpha[r0:r1]),
                                               _p(out[b0:b1]), _p(info[b0:b1]), _p(scratch), _stream()),
              "tgp_loglike_grad_batch_multi")
    return out, info, alpha


def predict_mean_batch(Xs, ssizes, X, sizes, descs, alpha):
    """tgp_predict_mean_batch_multi: mean rows of problem b = K_b(Xs_b, X_b) alpha_b (the full sum), with Xs
    (sum M_b, ndim) and X, alpha ((sum N_b,) or (sum N_b, r)) concatenated as for loglike_batch.  Returns the device
    tensor of means, (sum M_b,) or (sum M_b, r) as alpha."""
    Xs, X = as_points(Xs), as_points(X)
    sizes, ssizes = [int(n) for n in sizes], [int(m) for m in ssizes]
    _check_batch_inputs(X, sizes, descs)
    if len(ssizes) != len(sizes) or Xs.shape[0] != int(np.sum(ssizes)):
        raise ValueError("need one test-point count per problem, adding up to the rows of Xs")
    _check_dims(descs[0], X, Xs)
    r = _outputs(alpha, X.shape[0], "alpha")
    alpha = alpha.contiguous()
    mean = torch.empty((Xs.shape[0],) + tuple(alpha.shape[1:]), dtype=F64, device=X.device)
    soff, off, ks = batch_offsets(ssizes), batch_offsets(sizes), _ksum_array(descs)   # alive during the call
    check(_cabi.load().tgp_predict_mean_batch_multi(_p(Xs), _host_i64(soff), _p(X), _host_i64(off), len(sizes),
                                                    ctypes.cast(ks, ctypes.c_void_p), _p(alpha), r, _p(mean),
                                                    _stream()), "tgp_predict_mean_batch_multi")
    return mean


def var_batch_chunk_limit(sizes):
    """The largest `chunk` tgp_predict_var_batch accepts for problems with `sizes` points: its gemm grid (row tiles of
    128 times column tiles of 64 of the largest problem) and the K build's row tiles stay within 65535."""
    return min(65535 // ((max(int(n) for n in sizes) + 63) // 64) * 128, 65535 * 64)


def var_batch_chunk(ssizes, sizes, budget_bytes):
    """Test points per problem per pass of tgp_predict_var_batch: the largest count whose V rows
    (sum_b min(M_b, chunk) ld_b doubles) fit what `budget_bytes` leaves after the factors (batch_work_doubles(sizes)),
    at least 1, at most max(M_b) and var_batch_chunk_limit(sizes).  Pure host function."""
    m = np.asarray(ssizes, dtype=np.int64)
    ld = (np.asarray(sizes, dtype=np.int64) + 1) & ~1
    avail = budget_bytes - 8 * batch_work_doubles(sizes)
    lo, hi = 1, max(1, min(int(m.max()) if len(m) else 1, var_batch_chunk_limit(sizes)))
    while lo < hi:   # the V bytes grow with the chunk: the largest that fits
        mid = (lo + hi + 1) // 2
        if 8 * int(np.sum(np.minimum(m, mid) * ld)) <= avail:
            lo = mid
        else:
            hi = mid - 1
    return lo


def predict_var_batch(Xs, ssizes, X, y, yerr2, sizes, descs, budget_bytes=4 << 30):
    """Diagonal predictive variance of every problem (tgp_predict_var_batch), arguments as loglike_batch and
    predict_mean_batch: rows [soff[b], soff[b+1]) are sum_c amp_c + white - |L_b^-1 k*|^2.  Each chunk of problems
    (plan_batch_chunks) is factorised into a workspace of its own (tgp_loglike_batch, want_alpha = 0), then its test
    points go through in passes of var_batch_chunk rows per problem; rows are solved independently, so the results
    do not depend on either chunking.  Returns (var (sum M_b,), info (B,))."""
    Xs, X = as_points(Xs), as_points(X)
    sizes, ssizes = [int(n) for n in sizes], [int(m) for m in ssizes]
    _check_batch_inputs(X, sizes, descs)
    if len(ssizes) != len(sizes) or Xs.shape[0] != int(np.sum(ssizes)):
        raise ValueError("need one test-point count per problem, adding up to the rows of Xs")
    _check_dims(descs[0], X, Xs)
    off, soff = batch_offsets(sizes), batch_offsets(ssizes)
    B = len(sizes)
    var = torch.empty(Xs.shape[0], dtype=F64, device=X.device)
    info = torch.empty(B, dtype=torch.int32, device=X.device)
    lib = _cabi.load()
    for b0, b1 in plan_batch_chunks(sizes, budget_bytes):
        r0, r1, s0, s1 = int(off[b0]), int(off[b1]), int(soff[b0]), int(soff[b1])
        o = np.ascontiguousarray(off[b0:b1 + 1] - off[b0])
        so = np.ascontiguousarray(soff[b0:b1 + 1] - soff[b0])
        ks = _ksum_array(descs[b0:b1])
        work = torch.empty(batch_work_doubles(sizes[b0:b1]), dtype=F64, device=X.device)
        alpha = torch.empty(r1 - r0, dtype=F64, device=X.device)
        out = torch.empty((b1 - b0, 3), dtype=F64, device=X.device)
        check(lib.tgp_loglike_batch(_p(X[r0:r1]), _p(y[r0:r1]), _p(yerr2[r0:r1]), _host_i64(o), b1 - b0,
                                    ctypes.cast(ks, ctypes.c_void_p), _p(work), _p(alpha), 0, _p(out),
                                    _p(info[b0:b1]), _stream()), "tgp_loglike_batch")
        if s1 == s0:
            continue
        chunk = var_batch_chunk(ssizes[b0:b1], sizes[b0:b1], budget_bytes)
        nv = int(lib.tgp_predict_var_batch_work_doubles(_host_i64(so), _host_i64(o), b1 - b0, chunk))
        check(min(nv, 0), "tgp_predict_var_batch_work_doubles")
        vwork = torch.empty(nv, dtype=F64, device=X.device)
        check(lib.tgp_predict_var_batch(_p(Xs[s0:s1]), _host_i64(so), _p(X[r0:r1]), _host_i64(o), b1 - b0,
                                        ctypes.cast(ks, ctypes.c_void_p), _p(work), _p(vwork), chunk, _p(var[s0:s1]),
                                        _stream()), "tgp_predict_var_batch")
    return var, info


def loo_batch(X, y, yerr2, sizes, descs, budget_bytes=4 << 30):
    """Leave-one-out predictions of every problem (tgp_loo_batch_multi), arguments as loglike_batch, in chunks whose
    workspace plus scratch fit `budget_bytes` (plan_batch_chunks(scratch=True)): mean_ic = y_ic - alpha_ic / Z_ii and
    var_i = 1 / Z_ii - yerr2_i in residual space, Z = K^-1.  Returns (mean, shaped as y; var (sum N_b,); info (B,));
    the rows of a problem with info != 0 are NaN."""
    X = as_points(X)
    sizes = [int(n) for n in sizes]
    _check_batch_inputs(X, sizes, descs)
    r = _outputs(y, X.shape[0], "y")
    y = y.contiguous()
    off = batch_offsets(sizes)
    B = len(sizes)
    mean = torch.empty(y.shape, dtype=F64, device=X.device)
    var = torch.empty(int(off[-1]), dtype=F64, device=X.device)
    info = torch.empty(B, dtype=torch.int32, device=X.device)
    lib = _cabi.load()
    for b0, b1 in plan_batch_chunks(sizes, budget_bytes, scratch=True, r=r):
        r0, r1 = int(off[b0]), int(off[b1])
        o = np.ascontiguousarray(off[b0:b1 + 1] - off[b0])
        work = torch.empty(batch_work_doubles(sizes[b0:b1], r), dtype=F64, device=X.device)
        scratch = torch.empty(grad_batch_scratch_doubles(sizes[b0:b1]), dtype=F64, device=X.device)
        alpha = torch.empty(y[r0:r1].shape, dtype=F64, device=X.device)
        ks = _ksum_array(descs[b0:b1])
        check(lib.tgp_loo_batch_multi(_p(X[r0:r1]), _p(y[r0:r1]), r, _p(yerr2[r0:r1]), _host_i64(o), b1 - b0,
                                      ctypes.cast(ks, ctypes.c_void_p), _p(work), _p(alpha), _p(scratch),
                                      _p(mean[r0:r1]), _p(var[r0:r1]), _p(info[b0:b1]), _stream()),
              "tgp_loo_batch_multi")
    return mean, var, info


TRUNC_MIN_M, TRUNC_MIN_N = 16384, 2048   # below this the plain kernel is launch-bound anyway


def predict_mean(Xs, X, kdesc, alpha, out=None, truncate=None):
    """mean = K(Xs, X) . alpha without materialising K(Xs, X) (gp_interp.py:177,183); alpha (N,) gives mean (M,),
    alpha (N, r) of r outputs mean (M, r), every pair's profile evaluated once for all outputs
    (tgp_predict_mean[_trunc]_multi).

    truncate=True (default for large problems): both point sets are put in Hilbert-curve order (torch argsort /
    gather: plumbing) and the truncated entry skips blocks of pairs whose correlation is provably below
    1e-40; the result differs from the full sum by at most 1e-40 * sum|amp alpha| (and by summation order)."""
    Xs, X = as_points(Xs), as_points(X)
    _check_dims(kdesc, X, Xs)
    M, N = Xs.shape[0], X.shape[0]
    r = _outputs(alpha, N, "alpha")
    alpha = alpha.contiguous()
    shape = (M,) + tuple(alpha.shape[1:])
    if out is None:
        out = torch.empty(shape, dtype=F64, device=X.device)
    ks = as_sum(kdesc)
    lib = _cabi.load()
    if truncate is None:
        truncate = M >= TRUNC_MIN_M and N >= TRUNC_MIN_N
    if not truncate:
        check(lib.tgp_predict_mean_multi(_p(Xs), M, _p(X), N, ctypes.byref(ks), _p(alpha), r, _p(out), _stream()),
              "tgp_predict_mean_multi")
        return out
    two_d = X.shape[1] == 2
    zt, zs = torch.zeros(N, dtype=F64, device=X.device), torch.zeros(M, dtype=F64, device=X.device)
    ot = hilbert_order(X[:, 0].contiguous(), X[:, 1].contiguous() if two_d else zt)
    os_ = hilbert_order(Xs[:, 0].contiguous(), Xs[:, 1].contiguous() if two_d else zs)
    Xt, at, Xss = X[ot].contiguous(), alpha[ot].contiguous(), Xs[os_].contiguous()
    work = torch.empty(int(lib.tgp_predict_work_doubles(N)), dtype=F64, device=X.device)
    tmp = torch.empty(shape, dtype=F64, device=X.device)
    check(lib.tgp_predict_mean_trunc_multi(_p(Xss), M, _p(Xt), N, ctypes.byref(ks), _p(at), r, _p(tmp), _p(work),
                                           _stream()), "tgp_predict_mean_trunc_multi")
    out[os_] = tmp
    return out


def knn_mean(X0, y0, Xq, k):
    """Uniform mean of the k nearest grid values for every query point (gp_interp.py:236-238); y0 (n0,) or
    (n0, ncols).  Returns a device tensor (M,) or (M, ncols)."""
    X0, Xq = as_points(X0), as_points(Xq)
    n0, M = X0.shape[0], Xq.shape[0]
    if X0.shape[1] != Xq.shape[1]:
        raise ValueError("query and grid dimensions differ")
    if k > n0:
        # what sklearn's KNeighborsRegressor raises
        raise ValueError("Expected n_neighbors <= n_samples_fit, but n_neighbors = %d, n_samples_fit = %d" % (k, n0))
    y0 = to_device(y0)
    cols = [y0] if y0.dim() == 1 else [y0[:, j].contiguous() for j in range(y0.shape[1])]
    outs = []
    for col in cols:
        out = torch.empty(M, dtype=F64, device=X0.device)
        check(_cabi.load().tgp_knn_mean(_p(Xq), M, _p(X0), _p(col), n0, int(X0.shape[1]), int(k), _p(out), _stream()),
              "tgp_knn_mean")
        outs.append(out)
    return outs[0] if y0.dim() == 1 else torch.stack(outs, dim=1)


def predict_var(Xs, X, kdesc, L, chunk=None, out=None, work=None, row_end=None):
    """Diagonal predictive variance amp - |L^-1 k*|^2 (a sum: sum_c amp_c + white - |L^-1 k*|^2; tgp_predict_var_sum);
    row_end: the factor's envelope, X in the factor's (sorted) order."""
    Xs, X = as_points(Xs), as_points(X)
    _check_dims(kdesc, X, Xs)
    M, N = Xs.shape[0], X.shape[0]
    if chunk is None:
        # keep the K(Xs_chunk, X) workspace around 2 GiB
        chunk = max(128, min(M, (1 << 28) // max(N, 1)))
        chunk = (chunk + 127) // 128 * 128
    if work is None:
        work = torch.empty(chunk * (N + 1), dtype=F64, device=X.device)
    if out is None:
        out = torch.empty(M, dtype=F64, device=X.device)
    re, nre = _envelope(row_end)
    check(_cabi.load().tgp_predict_var_sum(_p(Xs), M, _p(X), N, ctypes.byref(as_sum(kdesc)), _p(L), L.stride(0), re,
                                           nre, _p(work), chunk, _p(out), _stream()), "tgp_predict_var_sum")
    return out


def var_chunk(N, M):
    """Test points per pass of tgp_predict_var: a K(Xs_chunk, X) workspace of about 2 GiB."""
    chunk = max(128, min(int(M), (1 << 28) // max(int(N), 1)))
    return (chunk + 127) // 128 * 128


def support_cutoffs(kdesc):
    """Per axis, the coordinate difference beyond which the kernel is below 1e-40 of its amplitude whatever the
    other coordinate: q = d^T M d >= d_a^2 / (M^-1)_aa, and f(q) <= 1e-40 for q >= tgp_profile_qcut(family).
    NaN / inf for a metric that is not positive definite (callers then keep the dense path).  A sum: per axis the
    largest cut-off of its terms (the white level has no off-diagonal support)."""
    if is_sum(kdesc):
        return [float(v) for v in np.max([support_cutoffs(kdesc.term[c]) for c in range(kdesc.nterms)], axis=0)]
    qcut = float(_cabi.load().tgp_profile_qcut(int(kdesc.family)))
    with np.errstate(invalid="ignore", divide="ignore"):
        if kdesc.ndim == 1:
            return [float(np.sqrt(np.float64(qcut) / kdesc.m00))]
        det = np.float64(kdesc.m00 * kdesc.m11 - kdesc.m01 * kdesc.m01)
        if not det > 0:
            return [float("nan"), float("nan")]
        return [float(np.sqrt(qcut * kdesc.m11 / det)), float(np.sqrt(qcut * kdesc.m00 / det))]


def envelope_trsm_flops(row_end, n):
    """Flops per right-hand side of tgp_trsm_rows_env for that envelope."""
    ob = envelope_block()
    k = np.arange(0, n, ob, dtype=np.float64)
    w = np.minimum(ob, n - k)
    below = np.maximum.accumulate(np.clip(np.asarray(row_end, dtype=np.float64), k + w, n)) - (k + w)
    return float(np.sum(w * w + 2.0 * w * below))


def plan_var_windows(x_train_sorted, a, b, dcut, chunk_sizes, align=64):
    """Host-side plan of the windowed variance (pure numpy: no device needed).  Training coordinates ascending in
    `x_train_sorted`; chunk c of the (sorted) test points spans [a[c], b[c]].  A training point further than `dcut`
    from that span is uncorrelated with the whole chunk, so the chunk's K* has a leading block of zeros in the
    ascending order (points below a - dcut) and in the descending order (points above b + dcut); forward substitution
    keeps leading zeros, so only the trailing sub-system L[lo:, lo:] is solved.  Returns (skip_asc, skip_desc,
    use_desc, flops_windowed, flops_full): the leading unknowns skipped in either order (multiples of `align`: the
    DMMA operand loads need 16-byte rows, and whole 64-blocks keep the solver's blocking), the cheaper order per chunk,
    and the N^2-per-test-point flop counts with and without the windows."""
    n = len(x_train_sorted)
    a, b, sizes = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64), np.asarray(chunk_sizes, dtype=np.float64)
    skip_asc = np.searchsorted(x_train_sorted, a - dcut, side="left") // align * align
    skip_desc = (n - np.searchsorted(x_train_sorted, b + dcut, side="right")) // align * align
    # keep at least one block of unknowns so that every call has a non-empty system
    cap = max(0, (n - 1) // align * align)
    skip_asc, skip_desc = np.minimum(skip_asc, cap), np.minimum(skip_desc, cap)
    use_desc = skip_desc > skip_asc
    left = n - np.where(use_desc, skip_desc, skip_asc)
    return (skip_asc.astype(np.int64), skip_desc.astype(np.int64), use_desc,
            float(np.sum(sizes * left.astype(np.float64) ** 2)), float(np.sum(sizes) * float(n) ** 2))


def predict_var_windowed(Xs, X, kdesc, yerr2, chunk=None, min_gain=1.25, stats=None):
    """Diagonal predictive variance k** - |L^-1 k*|^2 for MANY test points with a kernel whose support (correlation
    >= 1e-40 amp) is small against the field -- the regime of configs[2]: N = 4e4 training points, correlation length
    1.5 in a field of 160.  Training and test points are sorted along the axis with the shortest support; a chunk of
    neighbouring test points then sees zeros in K* for every training point before (ascending order) or after
    (descending order) its support, and forward substitution L v = k* leaves leading zeros in place: the chunk solves
    the trailing sub-system of ONE of two factorisations (points ascending / descending), whichever is shorter.
    Work per test point falls from N^2 to (N - skipped)^2 -- about 1/5 on average for a support of 1/6 of the field
    -- for two extra factorisations (2 N^3 / 3 flop).  The only approximation is the one predict_mean makes:
    correlations below 1e-40 amp count as zero.

    Returns None when the plan does not pay (support too wide, too few test points: fewer than `min_gain` times
    cheaper including the two factorisations, or the workspaces do not fit) -- the caller then runs the plain
    tgp_predict_var on its existing factor.  `stats` (a dict) receives the plan's figures."""
    Xs, X = as_points(Xs), as_points(X)
    _check_dims(kdesc, X, Xs)
    M, N = int(Xs.shape[0]), int(X.shape[0])
    if M == 0 or N < 128:
        return None
    dcut = support_cutoffs(kdesc)
    lo_hi = torch.stack([X.amin(dim=0), X.amax(dim=0)]).cpu().numpy()
    extent = np.maximum(lo_hi[1] - lo_hi[0], 1e-300)
    axis = int(np.argmin(np.asarray(dcut) / extent))
    if chunk is None:
        chunk = var_chunk(N, M)
    order_t = torch.argsort(X[:, axis], stable=True)
    order_s = torch.argsort(Xs[:, axis], stable=True)
    xs_sorted = Xs[order_s, axis]
    starts = torch.arange(0, M, chunk, device=X.device)
    ends = torch.clamp(starts + chunk, max=M) - 1
    a, b = xs_sorted[starts].cpu().numpy(), xs_sorted[ends].cpu().numpy()
    sizes = (ends - starts + 1).cpu().numpy()
    xt = X[order_t, axis].cpu().numpy()
    skip_asc, skip_desc, use_desc, f_win, f_full = plan_var_windows(xt, a, b, dcut[axis], sizes)
    need_asc, need_desc = bool(np.any(~use_desc)), bool(np.any(use_desc))
    # the two factors are Cholesky factors of matrices sorted along the axis: they live inside an envelope
    # (tgp_potrf_env), and so does the forward substitution of every window (tgp_predict_var_env)
    coords = {False: xt, True: np.ascontiguousarray(-xt[::-1])}
    env_full = envelope_rows(xt, dcut[axis])
    use_env = N >= ENVELOPE_MIN_N and envelope_flops(env_full, N) * ENVELOPE_MIN_GAIN <= float(N) ** 3 / 3.0
    f_factor = (need_asc + need_desc) * (envelope_flops(env_full, N) if use_env else float(N) ** 3 / 3.0)
    envs = None
    if use_env:
        envs = [envelope_rows(coords[bool(use_desc[c])], dcut[axis], start=int(skip_desc[c] if use_desc[c] else skip_asc[c]))
                for c in range(len(a))]
        f_win = float(sum(sizes[c] * envelope_trsm_flops(envs[c], N - int(skip_desc[c] if use_desc[c] else skip_asc[c]))
                          for c in range(len(a))))
    if stats is not None:
        stats.update({"axis": axis, "dcut": float(dcut[axis]), "extent": float(extent[axis]), "chunks": int(len(a)),
                      "flops_windowed": f_win, "flops_full": f_full, "flops_factors": f_factor,
                      "chunks_descending": int(np.sum(use_desc)), "envelope": bool(use_env), "used": False})
    if (f_win + f_factor) * min_gain > f_full:
        return None
    ld = even(N)
    bytes_needed = 8 * ((need_asc + need_desc) * N * ld + chunk * (N + 1) + 2 * M)
    free, _ = torch.cuda.mem_get_info(X.device)
    if bytes_needed > 0.9 * (free + torch.cuda.memory_reserved(X.device) - torch.cuda.memory_allocated(X.device)):
        return None
    e2 = None if yerr2 is None else yerr2[order_t].contiguous()
    Xa = X[order_t].contiguous()
    factors = {}
    for desc_order in ([False] if need_asc else []) + ([True] if need_desc else []):
        Xo = Xa.flip(0).contiguous() if desc_order else Xa
        eo = None if e2 is None else (e2.flip(0).contiguous() if desc_order else e2)
        L = kmat_sym(Xo, kdesc, eo, lower_only=True)
        info = int(potrf(L, N, row_end=envelope_rows(coords[desc_order], dcut[axis]) if use_env else None).item())
        if info < 0:
            raise _cabi.TgpError("tgp_potrf: internal synchronisation timed out (info = %d)" % info)
        if info != 0:
            raise np.linalg.LinAlgError("%d-th leading minor of the array is not positive definite" % info)
        factors[desc_order] = (Xo, L)
    Xss = Xs[order_s].contiguous()
    work = torch.empty(chunk * (N + 1), dtype=F64, device=X.device)
    out_sorted = torch.empty(M, dtype=F64, device=X.device)
    for c in range(len(a)):
        c0, c1 = c * chunk, min(M, (c + 1) * chunk)
        d = bool(use_desc[c])
        s = int(skip_desc[c] if d else skip_asc[c])
        Xo, L = factors[d]
        predict_var(Xss[c0:c1], Xo[s:], kdesc, L[s:, s:], chunk=chunk, out=out_sorted[c0:c1], work=work,
                    row_end=None if envs is None else envs[c])
    var = torch.empty(M, dtype=F64, device=X.device)
    var[order_s] = out_sorted
    if stats is not None:
        stats["used"] = True
    return var


_PB_SCRATCH = {}


def _pairbin_scratch(dev, doubles):
    """The workspace of tgp_pairbin (chunk boxes + sorted chunk copies, ~50 MB at N = 1e6, the super-chunk records, the
    list of super pairs for the leaf kernel and the same list grouped by column super-chunk, ~300 MB, plus the block
    records of one round of the two-pass TwoD count, at most 1 GiB), kept per
    (device, stream) and grown on demand: launches on one stream are ordered, so they can share it; launches on
    different streams get different buffers."""
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    buf = _PB_SCRATCH.get(key)
    if buf is None or buf.numel() < doubles:
        buf = torch.empty(int(doubles), dtype=F64, device=dev)
        _PB_SCRATCH[key] = buf
    return buf


def pairbin_packed(px, py, pk, pw, cat_off, max_cat_len, bin_type, edges, nbins, min_sep, max_sep,
                   rank=0, nranks=1):
    """Accumulate pair bins for `ncat` catalogues into ONE zeroed device buffer of shape (3 | 4, ncat, nb), FP64:
    plane 0 holds the int64 pair counts (raw 8-byte words), plane 1 sum w, plane 2 sum w k k, plane 3 (Log
    binning only) sum w r -- one allocation, and later one all-reduce / one device->host copy for all of them."""
    ncat = int(cat_off.numel()) - 1
    nb = nbins * nbins if bin_type == _cabi.BIN_TWOD else nbins
    dev = px.device
    planes = 4 if bin_type == _cabi.BIN_LOG else 3
    out = torch.zeros((planes, ncat, nb), dtype=F64, device=dev)
    lib = _cabi.load()
    work = _pairbin_scratch(dev, lib.tgp_pairbin_work_doubles(int(px.numel()), ncat))
    check(lib.tgp_pairbin(_p(px), _p(py), _p(pk), _p(pw), _p(cat_off), ncat, int(max_cat_len),
                          int(bin_type), _p(edges), int(nbins), float(min_sep) ** 2, float(max_sep),
                          int(rank), int(nranks), _p(out[0]), _p(out[1]), _p(out[2]),
                          _p(out[3]) if planes == 4 else _p(None), _p(work), _stream()), "tgp_pairbin")
    return out


def pairbin(px, py, pk, pw, cat_off, max_cat_len, bin_type, edges, nbins, min_sep, max_sep,
            rank=0, nranks=1):
    """Accumulate pair bins for `ncat` catalogues.  Returns (npairs int64, sumw, sumwkk, sumwr|None),
    each shaped (ncat, nb) (views of one packed buffer, see pairbin_packed)."""
    out = pairbin_packed(px, py, pk, pw, cat_off, max_cat_len, bin_type, edges, nbins, min_sep, max_sep,
                         rank=rank, nranks=nranks)
    return out[0].view(torch.int64), out[1], out[2], (out[3] if out.shape[0] == 4 else None)


def bootbin_sums(px, py, pz, pw, mult, edges, nbins, min_sep, max_sep, rank=0, nranks=1):
    """Pair sums of a bootstrap batch with shared geometry (tgp_bootbin_twod).  px, py, pz, pw|None: the base
    catalogue on the device (Hilbert order); mult: (nboot, n) uint8 device tensor of multiplicities.  Returns
    (sums, delta): the packed (6 * nb * bpad) forward / correction sums of this rank and the resample means."""
    n = int(px.numel())
    nboot = int(mult.shape[0])
    dev = px.device
    lib = _cabi.load()
    bpad = (nboot + 31) // 32 * 32
    sums = torch.empty(int(lib.tgp_bootbin_sums_doubles(int(nbins), nboot)), dtype=F64, device=dev)
    delta = torch.empty(bpad, dtype=F64, device=dev)
    nbytes = int(lib.tgp_bootbin_work_bytes(n, nboot))
    work = _pairbin_scratch(dev, nbytes // 8 + 64)
    off = (-work.data_ptr()) % 256          # torch allocations are 512-byte aligned; kept general
    check(lib.tgp_bootbin_twod(_p(px), _p(py), _p(pz), _p(pw), n, _p(mult), nboot, _p(edges), int(nbins),
                               float(min_sep) ** 2, float(max_sep), int(rank), int(nranks), _p(sums), _p(delta),
                               ctypes.c_void_p(work.data_ptr() + off), _stream()), "tgp_bootbin_twod")
    return sums, delta


def bootbin_xi(sums, delta, nbins, nboot, want_sumw=False):
    """xi (nboot, nbins^2) [and sumw] from the (all-reduced) sums of bootbin_sums."""
    xi = torch.empty((int(nboot), int(nbins) ** 2), dtype=F64, device=sums.device)
    sw = torch.empty_like(xi) if want_sumw else None
    check(_cabi.load().tgp_bootbin_xi(_p(sums), _p(delta), int(nbins), int(nboot), _p(xi), _p(sw), _stream()),
          "tgp_bootbin_xi")
    return (xi, sw) if want_sumw else xi


def bootbin_stats(reset=True):
    """Blocks per path of tgp_bootbin_twod since the last reset; synchronises the device."""
    buf = (ctypes.c_ulonglong * 8)()
    check(_cabi.load().tgp_bootbin_stats(buf, int(bool(reset))), "tgp_bootbin_stats")
    keys = ("closed_form", "sweeps", "pairwise", "exact_per_pair", "flushes", "sweeps_handed_back", "bin_by_bin")
    return {k: int(buf[i]) for i, k in enumerate(keys)}


def vcorr_sums(x, y, dx, dy, logrmin, dlogr, bins):
    """Pair sums of the vector-field correlation functions (utils.py:5-74) as numpy arrays:
    counts, sum ln r, sum Re(v1 conj v2), sum v1 v2 (complex), sum v1 v2 conj(d)^2/|d|^2 (complex).

    The device bins by thresholds on r^2; the pairs it reports as undecided (r^2 within 1e-14 of a threshold,
    where hypot and sqrt(r^2) may round apart: none for generic inputs) are placed here with the reference's own
    expression np.log(np.absolute(d)), so the counts equal np.histogram's bit for bit."""
    from . import binning

    x, y, dx, dy = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, dx, dy))
    xd, yd, vxd, vyd = (to_device(a) for a in (x, y, dx, dy))
    n = int(xd.numel())
    edges = to_device(binning.hist_thresholds_r2(logrmin, dlogr, bins))
    cap = 1 << 16
    while True:
        counts = torch.zeros(bins, dtype=torch.int64, device=xd.device)
        sums = torch.zeros((6, bins), dtype=F64, device=xd.device)
        amb = torch.empty((cap, 2), dtype=torch.int64, device=xd.device)
        namb = torch.zeros(1, dtype=torch.int32, device=xd.device)
        check(_cabi.load().tgp_vcorr(_p(xd), _p(yd), _p(vxd), _p(vyd), n, _p(edges), int(bins), _p(counts), _p(sums),
                                     _p(amb), cap, _p(namb), _stream()), "tgp_vcorr")
        na = int(namb.item())
        if na <= cap:
            break
        cap = 1 << int(np.ceil(np.log2(na)))
    s = sums.cpu().numpy()
    c = counts.cpu().numpy().astype(np.float64)
    if na:
        i1, i2 = amb[:na].cpu().numpy().T
        dr = 1j * (y[i2] - y[i1])
        dr += x[i2] - x[i1]
        with np.errstate(divide="ignore"):
            logdr = np.log(np.absolute(dr))
        k = binning.hist_bin(logdr, binning.hist_edges(logrmin, dlogr, bins))
        ok = k >= 0
        k, dr, logdr, i1, i2 = k[ok], dr[ok], logdr[ok], i1[ok], i2[ok]
        v = dx + 1j * dy
        vv = v[i1] * v[i2]
        rot = vv * np.conj(dr) ** 2 / (dr.real * dr.real + dr.imag * dr.imag)
        c += np.bincount(k, minlength=bins)
        for row, wgt in enumerate((logdr, dx[i1] * dx[i2] + dy[i1] * dy[i2], vv.real, vv.imag, rot.real, rot.imag)):
            s[row] += np.bincount(k, weights=wgt, minlength=bins)
    return (c, s[0], s[1], s[2] + 1j * s[3], s[4] + 1j * s[5])


def robust_chi2_batch(coord_d, y_d, W_d, family, params):
    """chi2, |amplitude|, offset of robust_2dfit.chi2 (two_pcf.py:115-148) for every row (size, g1, g2) of `params`
    in ONE launch (tgp_robust_chi2_batch).  coord_d (P, 2), y_d (P,), W_d (P, P): device tensors of the masked pixels.
    Returns a (len(params), 4) numpy array; chi2 = inf where the reference returns inf."""
    params = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 3)
    pd = to_device(params)
    out = torch.empty((params.shape[0], 4), dtype=F64, device=coord_d.device)
    check(_cabi.load().tgp_robust_chi2_batch(_p(coord_d), _p(y_d), _p(W_d), int(y_d.numel()), int(family), _p(pd),
                                             int(params.shape[0]), _p(out), _stream()), "tgp_robust_chi2_batch")
    return out.cpu().numpy()


def hilbert_order(px, py):
    """Permutation (device int64) that sorts the points along a Hilbert curve; makes tgp_pairbin's
    register path applicable.  The argsort is torch plumbing; the keys come from the C ABI."""
    n = int(px.numel())
    if n == 0:
        return torch.zeros(0, dtype=torch.int64, device=px.device)
    # the bounding square is found on the device (tgp_hilbert_keys_auto): nothing is read back, so the host keeps
    # enqueueing while the uploads and the sort run
    order = int(min(16, max(1, np.ceil(np.log2(max(np.sqrt(n), 2.0))) + 1)))
    keys = torch.empty(n, dtype=torch.int64, device=px.device)
    scratch = torch.empty(4, dtype=torch.int64, device=px.device)
    check(_cabi.load().tgp_hilbert_keys_auto(_p(px), _p(py), n, order, _p(scratch), _p(keys), _stream()),
          "tgp_hilbert_keys_auto")
    return torch.argsort(keys)


def pairbin_stats(reset=True):
    """Pairs per kernel path since the last reset (see tgp_pairbin_stats); synchronises the device."""
    buf = (ctypes.c_ulonglong * 8)()
    check(_cabi.load().tgp_pairbin_stats(buf, int(bool(reset))), "tgp_pairbin_stats")
    keys = ("closed_form", "one_axis", "pairwise", "one_axis_sorted", "two_axis_sorted", "super_closed_form",
            "super_one_axis")
    return {k: int(buf[i]) for i, k in enumerate(keys)}


def pairbin_super_leaves(reset=True):
    """Super-chunk pairs decided by the TwoD leaf kernel since the last reset (see tgp_pairbin_super_leaves); kept
    apart from pairbin_stats, whose values are pair counts that add up to the total."""
    v = ctypes.c_ulonglong(0)
    check(_cabi.load().tgp_pairbin_super_leaves(ctypes.byref(v), int(bool(reset))), "tgp_pairbin_super_leaves")
    return int(v.value)


def pairbin_super_rows(reset=True):
    """Of the super-chunk pairs of pairbin_super_leaves, those decided per row point against the staged column
    super-chunk (see tgp_pairbin_super_rows)."""
    v = ctypes.c_ulonglong(0)
    check(_cabi.load().tgp_pairbin_super_rows(ctypes.byref(v), int(bool(reset))), "tgp_pairbin_super_rows")
    return int(v.value)


def pairbin_super_one_axis_rows(reset=True):
    """Super-chunk pairs with one varying axis (pairbin_stats' super_one_axis, in super pairs) decided by the TwoD
    leaf kernel against a column super-chunk staged for many of them (see tgp_pairbin_super_one_axis_rows)."""
    v = ctypes.c_ulonglong(0)
    check(_cabi.load().tgp_pairbin_super_one_axis_rows(ctypes.byref(v), int(bool(reset))),
          "tgp_pairbin_super_one_axis_rows")
    return int(v.value)


def set_option(name, value):
    check(_cabi.load().tgp_set_option(name.encode(), int(value)), "tgp_set_option")


def microbench_fp64(kind, iters=20000):
    require_cuda()
    v = ctypes.c_double(0.0)
    check(_cabi.load().tgp_microbench_fp64(int(kind), int(iters), ctypes.byref(v)), "tgp_microbench_fp64")
    return v.value
