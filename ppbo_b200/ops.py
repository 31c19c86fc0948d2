"""Thin host wrappers: torch CUDA tensors in, C-ABI calls on the current stream, torch CUDA tensors out.

Every function here ends in a call into libppbo_b200.so; nothing is computed with torch ops or numpy.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import KERNEL_KINDS, PPBOError, check

F64 = torch.float64


def device(index=None):
    if not torch.cuda.is_available():
        raise PPBOError("ppbo_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device() if index is None else index)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


_SCRATCH = {}


def _scratch(purpose, nbytes, dev):
    """Workspace of at least nbytes for `purpose`: one buffer per (purpose, device, host thread, stream), kept between calls and
    grown with 25 % headroom.  A model that grows by one comparison set per iteration asks for a slightly larger workspace every
    time; fresh allocations would miss the caching allocator's pool each iteration (a cudaMalloc of up to hundreds of MB, and the
    cached smaller block is never reused).  Calls with the same key are ordered on their stream, so reuse is safe."""
    import threading
    key = (purpose, dev.index, threading.get_ident(), torch.cuda.current_stream(dev).cuda_stream)
    buf = _SCRATCH.get(key)
    need = nbytes // 8 + 2
    if buf is None or buf.numel() < need:
        buf = _SCRATCH[key] = torch.empty(int(need * 1.25) + 16, dtype=F64, device=dev)
    return buf


def to_dev(a, dev=None):
    """host array-like -> contiguous float64 CUDA tensor"""
    if isinstance(a, torch.Tensor):
        return a.to(device=dev or device(), dtype=F64).contiguous()
    return torch.as_tensor(np.ascontiguousarray(np.asarray(a, dtype=np.float64)), device=dev or device())


def _ls(lengthscales, D):
    ls = np.broadcast_to(np.asarray(lengthscales, dtype=np.float64), (D,))
    return _lib.host_doubles(ls)


def _kind(kernel):
    if isinstance(kernel, int):
        return kernel
    name = kernel if isinstance(kernel, str) else getattr(kernel, "__name__", str(kernel))
    if name not in KERNEL_KINDS:
        raise PPBOError("unknown kernel %r" % (name,))
    return KERNEL_KINDS[name]


# ------------------------------------------------------------------------------------------- K1
def kernel_matrix(kernel, X1, X2, lengthscales, sigma_f, out=None):
    n1, D = X1.shape
    n2 = X2.shape[0]
    out = torch.empty((n1, n2), dtype=F64, device=X1.device) if out is None else out
    check(_lib.load().ppbo_kernel_matrix(_kind(kernel), _p(X1), n1, _p(X2), n2, D, _ls(lengthscales, D), float(sigma_f),
                                         _p(out), out.stride(0) if n1 else max(n2, 1), _stream()), "ppbo_kernel_matrix")
    return out


def sqdist(X1, X2):
    """squared Euclidean distances between the rows of X1 and X2"""
    n1, D = X1.shape
    n2 = X2.shape[0]
    out = torch.empty((n1, n2), dtype=F64, device=X1.device)
    check(_lib.load().ppbo_sqdist(_p(X1), n1, _p(X2), n2, D, _p(out), max(n2, 1), _stream()), "ppbo_sqdist")
    return out


def gram_regularized(kernel, X, lengthscales, sigma_f, shrinkage, out=None):
    n, D = X.shape
    out = torch.empty((n, n), dtype=F64, device=X.device) if out is None else out
    check(_lib.load().ppbo_gram_regularized(_kind(kernel), _p(X), n, D, _ls(lengthscales, D), float(sigma_f),
                                            float(shrinkage), _p(out), max(out.stride(0), 1), _stream()), "ppbo_gram_regularized")
    return out


def kernel_se_grad(X1, X2, lengthscales, sigma_f):
    n1, D = X1.shape
    n2 = X2.shape[0]
    dK = torch.empty((D + 1, n1, n2), dtype=F64, device=X1.device)
    check(_lib.load().ppbo_kernel_se_grad(_p(X1), n1, _p(X2), n2, D, _ls(lengthscales, D), float(sigma_f), _p(dK), n2,
                                          n1 * n2, _stream()), "ppbo_kernel_se_grad")
    return dK


# ------------------------------------------------------------------------------------------- K2
def lik_terms(f, Q, m, sigma, want_sum=True, want_beta=True, want_arrow=True):
    dev = f.device
    s = torch.empty(1, dtype=F64, device=dev) if want_sum else None
    beta = torch.empty(Q * (m + 1), dtype=F64, device=dev) if want_beta else None
    arrow = torch.empty(Q * m, dtype=F64, device=dev) if want_arrow else None
    check(_lib.load().ppbo_lik_terms(_p(f), Q, m, float(sigma), _p(s), _p(beta), _p(arrow), _stream()), "ppbo_lik_terms")
    return s, beta, arrow


def lik_set_sums(f, Q, m, sigma):
    out = torch.empty(Q, dtype=F64, device=f.device)
    check(_lib.load().ppbo_lik_set_sums(_p(f), Q, m, float(sigma), _p(out), _stream()), "ppbo_lik_set_sums")
    return out


def lambda_dense(arrow, Q, m):
    N = Q * (m + 1)
    out = torch.empty((N, N), dtype=F64, device=arrow.device)
    check(_lib.load().ppbo_lambda_dense(_p(arrow), Q, m, _p(out), N, _stream()), "ppbo_lambda_dense")
    return out


def diffspace_gram(Sigma, Q, m):
    M = Q * m
    G = torch.empty((M, M), dtype=F64, device=Sigma.device)
    check(_lib.load().ppbo_diffspace_gram(_p(Sigma), Sigma.stride(0), Q, m, _p(G), M, _stream()), "ppbo_diffspace_gram")
    return G


class LaplaceFit:
    """Device-resident products of the MAP fit (everything prediction / acquisition needs).

    G and the factor object may have a capacity larger than the problem (`cap` >= Q m, leading dimensions `ldg`, `cap`), so that
    a model can grow in place (ModelState in iteration.py).  The factor AT the mode is only needed by prediction with covariance:
    it is built on first read of `Lfac` when the fit skipped it (`factor_state` < 2)."""
    __slots__ = ("Q", "m", "sigma", "f_map", "alpha", "arrow", "G", "ldg", "cap", "_Lfac", "sa_fac", "factor_state", "stats",
                 "n_neg", "_neg_idx", "_neg_corr", "info", "binv_cache", "binv_state")

    @property
    def M(self):
        return self.Q * self.m

    @property
    def Lfac(self):
        """factor object holding chol(I + a+^1/2 G a+^1/2) at the mode"""
        if self.factor_state < 2 and self.info == 0:
            rc = check(_lib.load().ppbo_laplace_refactor(_p(self.G), self.ldg, self.M, _p(self.arrow), _p(self._Lfac), self.cap,
                                                         _p(self.sa_fac), _stream()), "ppbo_laplace_refactor")
            if rc > 0:
                self.info = rc
                raise PPBOError("mode system not positive definite (pivot %d)" % rc)
            self.factor_state = 2
        return self._Lfac

    @property
    def L(self):
        """the M x M lower factor at the mode as a strided view"""
        buf = self.Lfac
        return buf[:self.cap * self.cap].view(self.cap, self.cap)[:self.M, :self.M]

    def count_negative(self):
        """number (and indices) of negative likelihood-curvature coefficients at the mode; host sync"""
        if self._neg_idx is None:
            idx = (ctypes.c_int * self.M)()
            self.n_neg = check(_lib.load().ppbo_neg_count(_p(self.arrow), self.M, idx, self.M, _stream()), "ppbo_neg_count")
            self._neg_idx = idx
        return self.n_neg

    @property
    def neg_corr(self):
        """Exact rank-r Woodbury correction of the posterior covariance for the r observations with a negative likelihood
        curvature (W indefinite there; the factor carries a+ only).  Only prediction WITH covariance needs it, so it is
        built on first use (r solves with the factor) instead of inside every fit."""
        self.count_negative()
        if self._neg_corr is None and self.n_neg > 0 and self.info == 0:
            lib = _lib.load()
            M = self.M
            Lf = self.Lfac
            self._neg_corr = torch.empty(lib.ppbo_neg_corr_doubles(M, self.n_neg), dtype=F64, device=self.G.device)
            rc2 = check(lib.ppbo_neg_corr_build(_p(self.G), self.ldg, M, _p(self.arrow), _p(Lf), self.cap, self._neg_idx,
                                                self.n_neg, _p(self._neg_corr), _stream()), "ppbo_neg_corr_build")
            if rc2 > 0:
                self.info = rc2
        return self._neg_corr


_STATS = ("iterations", "last_step", "last_rel_step", "T", "halvings", "info", "factorizations", "chord_steps", "factor_state",
          "converged", "warm_first_rel", "border_rows")


def laplace_fit(Sigma, Q, m, sigma, f_init=None, max_iter=100, tol=1e-10, factor_at_mode=False, into=None, g_ready=False,
                warm_rows=0, alpha_init=None):
    """MAP fit.  `into`: a LaplaceFit whose (capacity) buffers G / factor / sa_fac are reused -- with g_ready the grown G is
    taken as is; warm_rows > 0: the factor object holds the factor of the leading warm_rows x warm_rows system (the previous
    iteration's) and the chord iteration starts from (f_init, alpha_init) with the appended rows carried as a border."""
    warm_factor = warm_rows > 0
    lib = _lib.load()
    dev = Sigma.device
    N, M = Q * (m + 1), Q * m
    if into is None:
        fit = LaplaceFit()
        fit.cap = fit.ldg = M
        fit.binv_cache, fit.binv_state = None, None
        fit.G = torch.empty((M, M), dtype=F64, device=dev)
        fit._Lfac = torch.empty(lib.ppbo_factor_doubles(M), dtype=F64, device=dev)
        fit.sa_fac = torch.empty(M, dtype=F64, device=dev)
        fit.f_map = torch.empty(N, dtype=F64, device=dev)
        fit.alpha = torch.empty(N, dtype=F64, device=dev)
        fit.arrow = torch.empty(M, dtype=F64, device=dev)
    else:
        fit = into
        if fit.cap < M:
            raise PPBOError("model capacity %d below Q m = %d" % (fit.cap, M))
    fit.Q, fit.m, fit.sigma = Q, m, float(sigma)
    flags = (_lib.FIT_G_READY if g_ready else 0) | (_lib.FIT_FACTOR_WARM if warm_factor else 0) | \
            (_lib.FIT_FACTOR_AT_MODE if factor_at_mode else 0)
    wbytes = lib.ppbo_laplace_workspace_bytes(Q, m)
    ws = _scratch("laplace", wbytes, dev)
    stats = (ctypes.c_double * 12)()
    binv_cache = getattr(fit, "binv_cache", None)
    rc = check(lib.ppbo_laplace_fit(_p(Sigma), Sigma.stride(0), Q, m, float(sigma), _p(f_init), _p(alpha_init), int(max_iter),
                                    float(tol), flags, _p(fit.G), fit.ldg, _p(fit._Lfac), fit.cap, _p(fit.sa_fac), int(warm_rows),
                                    _p(binv_cache), fit.binv_state if binv_cache is not None else None,
                                    _p(fit.f_map), _p(fit.alpha), _p(fit.arrow), _p(ws), wbytes, stats, _stream()),
               "ppbo_laplace_fit")
    fit.info = rc
    fit.stats = {k: stats[i] for i, k in enumerate(_STATS)}
    for k in ("iterations", "halvings", "factorizations", "chord_steps", "converged", "border_rows"):
        fit.stats[k] = int(fit.stats[k])
    fit.factor_state = int(stats[8]) if rc == 0 else 0
    fit.n_neg, fit._neg_corr, fit._neg_idx = 0, None, None
    return fit


def gram_append(kernel, X, n_old, lengthscales, sigma_f, shrinkage, Sigma_cap):
    """rows / columns [n_old, n) of the regularised covariance of X [n x D] written into the capacity buffer Sigma_cap in place"""
    n, D = X.shape
    check(_lib.load().ppbo_gram_append(_kind(kernel), _p(X), int(n_old), n, D, _ls(lengthscales, D), float(sigma_f), float(shrinkage),
                                       _p(Sigma_cap), Sigma_cap.stride(0), _stream()), "ppbo_gram_append")
    return Sigma_cap


def diffspace_gram_append(Sigma, Q_old, Q_new, m, G_cap):
    check(_lib.load().ppbo_diffspace_gram_append(_p(Sigma), Sigma.stride(0), int(Q_old), int(Q_new), m, _p(G_cap), G_cap.stride(0),
                                                 _stream()), "ppbo_diffspace_gram_append")
    return G_cap


def factor_extend(fit, M_old, M_new, f_new_sets=None, sigma=None):
    """grow fit's factor object from M_old to M_new rows; the coefficients of the new rows come from the warm-start values
    f_new_sets of the appended comparison sets (or are already in fit.sa_fac[M_old:M_new]); returns LAPACK-style info"""
    return check(_lib.load().ppbo_factor_extend(_p(fit.G), fit.ldg, int(M_old), int(M_new), _p(fit.sa_fac), _p(f_new_sets), fit.m,
                                                float(fit.sigma if sigma is None else sigma), _p(fit._Lfac), fit.cap, _stream()),
                 "ppbo_factor_extend")


# ------------------------------------------------------------------------------------------- dense linear algebra
def gemm_nt(A, B, C=None, alpha=1.0, beta=0.0):
    M, K = A.shape
    N = B.shape[0]
    C = torch.empty((M, N), dtype=F64, device=A.device) if C is None else C
    check(_lib.load().ppbo_gemm_nt(_p(A), A.stride(0), _p(B), B.stride(0), _p(C), C.stride(0), M, N, K, float(alpha),
                                   float(beta), _stream()), "ppbo_gemm_nt")
    return C


def gemm_nt_lower(A, B, C, alpha=1.0, beta=0.0):
    """lower tiles of C = alpha A B^T + beta C (square C); the lower triangle has the bits of gemm_nt"""
    N, K = A.shape
    check(_lib.load().ppbo_gemm_nt_lower(_p(A), A.stride(0), _p(B), B.stride(0), _p(C), C.stride(0), N, K, float(alpha),
                                         float(beta), _stream()), "ppbo_gemm_nt_lower")
    return C


def gemm_nt_cfg(cfg, A, B, C, alpha=1.0, beta=0.0):
    M, K = A.shape
    N = B.shape[0]
    check(_lib.load().ppbo_gemm_nt_cfg(int(cfg), _p(A), A.stride(0), _p(B), B.stride(0), _p(C), C.stride(0), M, N, K,
                                       float(alpha), float(beta), _stream()), "ppbo_gemm_nt_cfg")
    return C


def potrf_lower(A):
    """in-place lower Cholesky; returns (info, workspace holding the inverted diagonal blocks)"""
    lib = _lib.load()
    n = A.shape[0]
    wbytes = lib.ppbo_potrf_workspace_bytes(n)
    ws = torch.empty(wbytes // 8 + 1, dtype=F64, device=A.device)
    info = ctypes.c_int(0)
    rc = check(lib.ppbo_potrf_lower(_p(A), A.stride(0), n, _p(ws), wbytes, ctypes.byref(info), _stream()), "ppbo_potrf_lower")
    return rc, ws


def trsm_right_lower(L, ws, X):
    """X[nrhs x n] <- X L^-T in place"""
    lib = _lib.load()
    n = L.shape[0]
    check(lib.ppbo_trsm_right_lower(_p(L), L.stride(0), n, _p(X), X.stride(0), X.shape[0], 0, _p(ws),
                                    lib.ppbo_potrf_workspace_bytes(n), _stream()), "ppbo_trsm_right_lower")
    return X


def potrs_vec(L, ws, b):
    """solve (L L^T) x = b for one right-hand side; returns x (new tensor)"""
    lib = _lib.load()
    n = L.shape[0]
    x = torch.empty(n + 128, dtype=F64, device=L.device)
    x[:n].copy_(b)
    check(lib.ppbo_potrs_vec(_p(L), L.stride(0), n, _p(x), _p(ws), lib.ppbo_potrf_workspace_bytes(n), _stream()),
          "ppbo_potrs_vec")
    return x[:n]


def blockinv_build(L, ws):
    """1024 x 1024 block inverses of a factor from potrf_lower (for many solves with the same factor)"""
    lib = _lib.load()
    n = L.shape[0]
    nbytes = lib.ppbo_blockinv_bytes(n)
    W = torch.empty(nbytes // 8, dtype=F64, device=L.device)
    check(lib.ppbo_blockinv_build(_p(L), L.stride(0), n, _p(ws), _p(W), nbytes, _stream()), "ppbo_blockinv_build")
    return W


def potrs_vec_blockinv(L, W, b):
    """solve (L L^T) x = b with the block inverses W of blockinv_build; returns x (new tensor)"""
    n = L.shape[0]
    x = b.clone()
    check(_lib.load().ppbo_potrs_vec_blockinv(_p(L), L.stride(0), n, _p(W), W.numel() * 8, _p(x), _stream()),
          "ppbo_potrs_vec_blockinv")
    return x


def potri_lower(L, ws):
    """dense (L L^T)^-1 from a factor produced by potrf_lower"""
    lib = _lib.load()
    n = L.shape[0]
    work = torch.empty((n, n), dtype=F64, device=L.device)
    out = torch.empty((n, n), dtype=F64, device=L.device)
    check(lib.ppbo_potri_lower(_p(L), L.stride(0), n, _p(ws), lib.ppbo_potrf_workspace_bytes(n), _p(work), _p(out), n,
                               _stream()), "ppbo_potri_lower")
    return out


def lu_logdet(A):
    """LU with partial pivoting of the square device matrix A (overwritten): (sign det U, log|det A|, sign of the row permutation)"""
    lib = _lib.load()
    n = A.shape[0]
    wbytes = lib.ppbo_lu_workspace_bytes(n)
    ws = torch.empty(wbytes // 8 + 1, dtype=F64, device=A.device)
    res = (ctypes.c_double * 3)()
    rc = check(lib.ppbo_lu_logdet(_p(A), A.stride(0), n, _p(ws), wbytes, res, _stream()), "ppbo_lu_logdet")
    return res[0], res[1], res[2], rc


def evidence_logdet(Sigma, Q, m, arrow, reference=True):
    """LU log-determinant of I + Sigma Lambda (reference=True: the matrix GPModel.evidence factors, src/gp_model.py:301-308)
    or of I + Sigma W (the Laplace normaliser) for the signed coefficients `arrow`"""
    N = Q * (m + 1)
    A = torch.empty((N, N), dtype=F64, device=Sigma.device)
    check(_lib.load().ppbo_evidence_matrix(_p(Sigma), Sigma.stride(0), Q, m, _p(arrow), 1 if reference else 0, _p(A), N, _stream()),
          "ppbo_evidence_matrix")
    return lu_logdet(A)


def shrink_inplace(K, shrinkage):
    n = K.shape[0]
    scratch = torch.empty(1, dtype=F64, device=K.device)
    check(_lib.load().ppbo_shrink_inplace(_p(K), K.stride(0), n, float(shrinkage), _p(scratch), _stream()),
          "ppbo_shrink_inplace")
    return K


def gemv(A, x, out=None):
    y = torch.empty(A.shape[0], dtype=F64, device=A.device) if out is None else out
    check(_lib.load().ppbo_gemv(_p(A), A.stride(0), A.shape[0], A.shape[1], _p(x), _p(y), _stream()), "ppbo_gemv")
    return y


def symv_lower(A, x, out=None):
    """y = A x for a symmetric A, reading only its lower triangle"""
    n = A.shape[0]
    y = torch.empty(n, dtype=F64, device=A.device) if out is None else out
    check(_lib.load().ppbo_symv_lower(_p(A), A.stride(0), n, _p(x), _p(y), _stream()), "ppbo_symv_lower")
    return y


# ------------------------------------------------------------------------------------------- K4
def predict(kernel, X, lengthscales, sigma_f, shrinkage, fit, Xp, P, batch, want_cov=True):
    lib = _lib.load()
    N, D = X.shape
    dev = X.device
    mu = torch.empty(P * batch, dtype=F64, device=dev)
    Sp = torch.empty((batch, P, P), dtype=F64, device=dev) if want_cov else None
    wbytes = (lib.ppbo_predict_workspace_bytes(N, fit.Q, fit.m, P, batch) if want_cov else
              lib.ppbo_predict_mean_workspace_bytes(_kind(kernel), N, P, batch))
    ws = _scratch("predict" if want_cov else "predict_mean", wbytes, dev)
    neg_corr = fit.neg_corr if want_cov else None            # the mean needs alpha only (no factor, no Woodbury term)
    if want_cov and fit.info > 0:
        # the Woodbury block of the negative coefficients has no Cholesky factor: there is no covariance to return
        raise PPBOError("posterior precision not positive definite (info %d): no predictive covariance" % fit.info)
    Lfac = fit.Lfac if want_cov else None
    check(lib.ppbo_predict(_kind(kernel), _p(X), N, D, _ls(lengthscales, D), float(sigma_f), float(shrinkage), fit.Q, fit.m,
                           _p(fit.alpha), _p(fit.arrow), _p(Lfac), fit.cap, _p(neg_corr), fit.n_neg if want_cov else 0, _p(Xp), P,
                           batch, _p(mu), _p(Sp), _p(ws), wbytes, _stream()), "ppbo_predict")
    return mu.view(batch, P), Sp


def posterior_mean(kernel, X, lengthscales, sigma_f, alpha, Xp):
    """mu(Xp) = k(Xp, X) alpha without a fit object (GPModel.mu_pred batched, src/gp_model.py:454-458)"""
    lib = _lib.load()
    N, D = X.shape
    P = Xp.shape[0]
    mu = torch.empty(P, dtype=F64, device=X.device)
    wbytes = lib.ppbo_predict_mean_workspace_bytes(_kind(kernel), N, P, 1)
    ws = _scratch("predict_mean", wbytes, X.device)
    check(lib.ppbo_predict(_kind(kernel), _p(X), N, D, _ls(lengthscales, D), float(sigma_f), 0.0, N, 0, _p(alpha), None, None, 0,
                           None, 0, _p(Xp), P, 1, _p(mu), None, _p(ws), wbytes, _stream()), "ppbo_predict")
    return mu


class PointMean:
    """mu(x) = k(x, X) alpha for one host point per call (ppbo_mu_pred_point): the objective of GPModel.mu_star's sequential
    search.  Everything that does not change between calls is prepared once."""

    def __init__(self, kernel, X, lengthscales, sigma_f, alpha):
        self.lib = _lib.load()
        self.kind, self.X, self.alpha = _kind(kernel), X, alpha
        self.N, self.D = X.shape
        self.ls, self.sigma_f = _ls(lengthscales, self.D), float(sigma_f)
        self.out = ctypes.c_double(0.0)
        self.out_ref = ctypes.byref(self.out)
        self.buf = (ctypes.c_double * self.D)()
        self.Xp, self.ap = _p(X), _p(alpha)
        self.calls = 0

    def __call__(self, x):
        self.buf[:] = x
        rc = self.lib.ppbo_mu_pred_point(self.kind, self.Xp, self.N, self.D, self.ls, self.sigma_f, self.ap, self.buf,
                                         ctypes.cast(self.out_ref, ctypes.POINTER(ctypes.c_double)), _stream())
        if rc:
            check(rc, "ppbo_mu_pred_point")
        self.calls += 1
        return self.out.value


# --- GPModel.mu_star's sequential differential evolution with the loop in C++ (csrc/de.cu) -----------------------------------
_OBJECTIVE_FN = ctypes.CFUNCTYPE(ctypes.c_double, ctypes.POINTER(ctypes.c_double), ctypes.c_int, ctypes.c_void_p)
_OBJECTIVE_BATCH_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.c_int, ctypes.c_int,
                                       ctypes.POINTER(ctypes.c_double), ctypes.c_void_p)
DE_MAX_WINDOW = 64                                                                                             # PPBO_MAX_POINTS


class DEResult:
    """x, fun: best member (problem units) and its value at the end of the evolution (before any polish); nit, nfev, converged,
    population_size as scipy reports them; discarded: evaluations of speculative windows whose results were never looked at;
    calls: calls of the objective (one per window, i.e. launches on the device)"""

    def __init__(self, x, fun, stats):
        self.x, self.fun = x, fun
        self.nit, self.nfev, self.converged, self.population_size = int(stats[0]), int(stats[1]), bool(stats[2]), int(stats[3])
        self.discarded, self.calls = int(stats[4]), int(stats[5])


def _de_call(entry, bounds, popsize, maxiter, tol, atol, mutation, recombination, what):
    """shared part of the two entries: numpy's global MT19937 state in, the same stream advanced by exactly scipy's draws out.
    entry(D, lo, hi, popsize, maxiter, tol, atol, mutation_lo, mutation_hi, recombination, key, pos, x, fun, stats) -> status"""
    bounds = np.asarray(bounds, dtype=np.float64)
    D = bounds.shape[0]
    lo, hi = _lib.host_doubles(bounds[:, 0]), _lib.host_doubles(bounds[:, 1])
    name, key, pos, has_gauss, cached = np.random.get_state()
    if name != "MT19937":
        raise PPBOError("numpy's global generator is not the legacy MT19937")
    key = np.ascontiguousarray(key, dtype=np.uint32).copy()
    pos_c = ctypes.c_int(int(pos))
    x = (ctypes.c_double * D)()
    fun = ctypes.c_double(0.0)
    stats = (ctypes.c_int * 6)()
    mut = sorted(float(v) for v in np.atleast_1d(mutation))
    if len(mut) != 2:
        raise PPBOError("mutation must be a (min, max) pair (dither), as in the reference's default call")
    rc = entry(D, lo, hi, int(popsize), int(maxiter), float(tol), float(atol), mut[0], mut[1], float(recombination),
               key.ctypes.data_as(ctypes.POINTER(ctypes.c_uint)), ctypes.byref(pos_c), x, ctypes.byref(fun), stats)
    np.random.set_state((name, key, int(pos_c.value), has_gauss, cached))
    if rc:
        raise PPBOError("%s failed (%d): %s" % (what, rc, _lib.last_error()))
    return DEResult(np.array(x[:], dtype=np.float64), float(fun.value), stats)


def de_minimize(func, bounds, popsize=15, maxiter=1000, tol=0.01, atol=0.0, mutation=(0.5, 1.0), recombination=0.7, window=1):
    """scipy.optimize.differential_evolution(func, bounds, updating='immediate', polish=False) on numpy's GLOBAL legacy stream,
    replayed draw for draw by ppbo_de_minimize: same result bits, same state of np.random afterwards.  func: x (D,) -> float.
    window > 1: evaluations issued in speculative windows of that many trials (same result; func is called on discarded trials too)."""
    failure = []

    def one(xp, d, _ctx):
        try:
            return float(func(np.ctypeslib.as_array(xp, shape=(d,)).copy()))
        except BaseException as e:                    # an exception must not unwind through the C frames
            failure.append(e)
            return float("nan")

    def many(xp, b, d, fp, _ctx):
        try:
            X = np.ctypeslib.as_array(xp, shape=(b, d)).copy()
            for k in range(b):
                fp[k] = float(func(X[k]))
            return 0
        except BaseException as e:
            failure.append(e)
            return -1
    f1, fb = _OBJECTIVE_FN(one), _OBJECTIVE_BATCH_FN(many)
    lib = _lib.load()

    def entry(D, *rest):
        return lib.ppbo_de_minimize(f1, fb, int(window), None, D, *rest)
    try:
        return _de_call(entry, bounds, popsize, maxiter, tol, atol, mutation, recombination, "ppbo_de_minimize")
    except PPBOError:
        if failure:
            raise failure[0]
        raise


def de_polish(func, de, bounds):
    """the L-BFGS-B polish that ends scipy.optimize.differential_evolution(..., polish=True), made exactly as
    scipy/optimize/_differentialevolution.py (1.18: solve(), 'if self.polish') makes it: from the best member, inside the bounds,
    accepted only if it improves.  de: DEResult of the evolution; returns a scipy OptimizeResult (x, fun, nit, nfev, success)."""
    import scipy.optimize
    limits = np.array(bounds, dtype=float).T
    res = scipy.optimize.OptimizeResult(x=de.x, fun=de.fun, nit=de.nit, nfev=de.nfev, success=de.converged)
    polished = scipy.optimize.minimize(lambda x: func(np.atleast_2d(x)[0]), np.copy(de.x), method='L-BFGS-B',
                                       bounds=scipy.optimize.Bounds(lb=limits[0], ub=limits[1]), constraints=())
    res.nfev += polished.get("nfev", 0)
    if polished.fun < res.fun and polished.success and np.all(polished.x <= limits[1]) and np.all(limits[0] <= polished.x):
        res.fun, res.x = polished.fun, polished.x
    return res


def mu_star_de(kernel, X, lengthscales, sigma_f, alpha, bounds, popsize=15, maxiter=1000, tol=0.01, atol=0.0, mutation=(0.5, 1.0),
               recombination=0.7, window=1):
    """the same search with the objective -mu(x) = -k(x, X) alpha evaluated on the device: one ppbo_mu_pred_point launch per trial
    (window = 1) or one ppbo_mu_pred_points launch per speculative window; bit-identical to a scipy call over PointMean either
    way.  Returns a DEResult with fun = -mu(x)."""
    N, Dx = X.shape
    lib = _lib.load()
    kind, ls, st = _kind(kernel), _ls(lengthscales, Dx), _stream()

    def entry(D, lo, hi, popsize_, maxiter_, tol_, atol_, m0, m1, rec, key, pos, x, fun, stats):
        return lib.ppbo_mu_star_de(kind, _p(X), N, D, ls, float(sigma_f), _p(alpha), lo, hi, popsize_, maxiter_, tol_, atol_, m0, m1,
                                   rec, int(window), key, pos, x, fun, stats, st)
    return _de_call(entry, bounds, popsize, maxiter, tol, atol, mutation, recombination, "ppbo_mu_star_de")


def mu_pred_points(kernel, X, lengthscales, sigma_f, alpha, points):
    """posterior means of up to 64 host points in one launch, host result (ppbo_mu_pred_points)"""
    pts = np.ascontiguousarray(np.atleast_2d(np.asarray(points, dtype=np.float64)))
    B, D = pts.shape
    out = np.empty(B, dtype=np.float64)
    check(_lib.load().ppbo_mu_pred_points(_kind(kernel), _p(X), X.shape[0], D, _ls(lengthscales, D), float(sigma_f), _p(alpha),
                                          pts.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), B,
                                          out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), _stream()), "ppbo_mu_pred_points")
    return out


MU_MAXIMIZE_MAX_ITER = 100      # step cap of the posterior-mean ascent (DESIGN.md 7 item 16)
MU_MAXIMIZE_GTOL = 1e-10        # its stationarity tolerance, relative to sigma_f^2 sum |alpha| (the bound on |mu|)


def mu_maximize(kernel, X, lengthscales, sigma_f, alpha, X0, max_iter=MU_MAXIMIZE_MAX_ITER, gtol=MU_MAXIMIZE_GTOL, periodic_mask=0):
    """Multi-start ascent of mu(x) = k(x, X) alpha over [0,1]^D from the starts X0 [R, D] (ppbo_mu_maximize, one CTA per start).
    Device tensors, no synchronisation: (xbest [D], fbest [1], xout [R, D], fout [R], gout [R, D], iters [R] int32) -- the best end
    point (lowest start index on ties) and its mean, then per start the end point, the mean and its gradient there and the steps
    taken.  max_iter = 0: the mean and its gradient at the starts.  periodic_mask: spectral.periodic_mask of the kernel."""
    R, D = X0.shape
    dev = X0.device
    xout = torch.empty((R, D), dtype=F64, device=dev)
    gout = torch.empty((R, D), dtype=F64, device=dev)
    fout = torch.empty(R, dtype=F64, device=dev)
    iters = torch.empty(R, dtype=torch.int32, device=dev)
    xbest = torch.empty(D, dtype=F64, device=dev)
    fbest = torch.empty(1, dtype=F64, device=dev)
    check(_lib.load().ppbo_mu_maximize(_kind(kernel), _p(X), X.shape[0], D, _ls(lengthscales, D), float(sigma_f), _p(alpha),
                                       _p(X0.contiguous()), R, int(max_iter), float(gtol), int(periodic_mask), _p(xout), _p(fout),
                                       _p(gout), _p(iters), _p(xbest), _p(fbest), _stream()), "ppbo_mu_maximize")
    return xbest, fbest, xout, fout, gout, iters


def mvn_rowmax(Z, Fac, mu):
    """Z: [B,S,K], Fac: [B,P,K], mu: [B,P] -> fmax [B,S], arg [B,S] (int32)"""
    B, S, K = Z.shape
    P = Fac.shape[1]
    fmax = torch.empty((B, S), dtype=F64, device=Z.device)
    arg = torch.empty((B, S), dtype=torch.int32, device=Z.device)
    check(_lib.load().ppbo_mvn_rowmax(_p(Z), Z.stride(1), Z.stride(0), _p(Fac), Fac.stride(1), Fac.stride(0), _p(mu),
                                      mu.stride(0), S, P, K, B, _p(fmax), _p(arg), _stream()), "ppbo_mvn_rowmax")
    return fmax, arg


def acq_reduce(fmax, mustar):
    B, S = fmax.shape
    out = torch.empty((B, 3), dtype=F64, device=fmax.device)
    check(_lib.load().ppbo_acq_reduce(_p(fmax), S, B, float(mustar), _p(out), _stream()), "ppbo_acq_reduce")
    return out


# ------------------------------------------------------------------------------------------- K3
def rff_features(W, b, X, sigma_f, feature_major, out=None):
    F, D = W.shape
    n = X.shape[0]
    if out is None:
        out = torch.empty((F, n) if feature_major else (n, F), dtype=F64, device=W.device)
    check(_lib.load().ppbo_rff_features(_p(W), _p(b), F, D, _p(X), n, float(sigma_f), _p(out), out.stride(0),
                                        1 if feature_major else 0, _stream()), "ppbo_rff_features")
    return out


def rff_jacobian(W, b, x, sigma_f):
    F, D = W.shape
    J = torch.empty((F, D), dtype=F64, device=W.device)
    check(_lib.load().ppbo_rff_jacobian(_p(W), _p(b), F, D, _p(x), float(sigma_f), _p(J), _stream()), "ppbo_rff_jacobian")
    return J


def rff_maximize(W, b, sigma_f, Omega, X0, max_iter=500, gtol=1e-9, periodic_mask=0):
    """Omega [S,F], starts X0 [S,R,D] -> (xbest [S,D], fbest [S]): maximisers of the sampled functions phi(x)' Omega[s] on [0,1]^D.
    Coordinates whose bit is set in `periodic_mask` (spectral.periodic_mask of the basis' kernel) wrap modulo 1 instead of being
    projected onto [0, 1]."""
    Fdim, D = W.shape
    S, R, _ = X0.shape
    dev = W.device
    xbest = torch.empty((S, D), dtype=F64, device=dev)
    fbest = torch.empty(S, dtype=F64, device=dev)
    work = _scratch("rff_maximize", S * R * (D + 1) * 8, dev)
    check(_lib.load().ppbo_rff_maximize(_p(W), _p(b), Fdim, D, float(sigma_f), _p(Omega), Omega.stride(0), S, _p(X0.contiguous()), R,
                                        int(max_iter), float(gtol), int(periodic_mask), _p(xbest), _p(fbest), _p(work), _stream()),
          "ppbo_rff_maximize")
    return xbest, fbest


def _rff_ws(F, Q, m, dev):
    wbytes = _lib.load().ppbo_rff_workspace_bytes(F, Q, m)
    return _scratch("rff", wbytes, dev), wbytes


def rff_objective(Phi_X, Q, m, sigma, omega, want_S=True, want_grad=True, want_hess=True):
    F = Phi_X.shape[0]
    ws, wbytes = _rff_ws(F, Q, m, Phi_X.device)
    S = ctypes.c_double(0.0)
    grad = torch.empty(F, dtype=F64, device=Phi_X.device) if want_grad else None
    hd = torch.empty(F, dtype=F64, device=Phi_X.device) if want_hess else None
    check(_lib.load().ppbo_rff_objective(_p(Phi_X), Phi_X.stride(0), F, Q, m, float(sigma), _p(omega),
                                         ctypes.byref(S) if want_S else None, _p(grad), _p(hd), _p(ws), wbytes, _stream()),
          "ppbo_rff_objective")
    return (S.value if want_S else None), grad, hd


def rff_factor_cache(F, dev):
    """persistent buffer for the weight-space Hessian factor (rff_fit(..., factor_cache=..., warm=True) reuses it between fits)"""
    return torch.empty(_lib.load().ppbo_rff_factor_cache_doubles(F) + 2, dtype=F64, device=dev)


def rff_fit(Phi_X, Q, m, sigma, omega0=None, max_iter=100, tol=1e-10, factor_cache=None, warm=False):
    F = Phi_X.shape[0]
    ws, wbytes = _rff_ws(F, Q, m, Phi_X.device)
    omega = torch.empty(F, dtype=F64, device=Phi_X.device)
    hd = torch.empty(F, dtype=F64, device=Phi_X.device)
    stats = (ctypes.c_double * 8)()
    warm_flag = (int(warm) if warm in (1, 2) else 1) if (warm and factor_cache is not None) else 0      # 2: block inverses cached too
    rc = check(_lib.load().ppbo_rff_fit(_p(Phi_X), Phi_X.stride(0), F, Q, m, float(sigma), _p(omega0), int(max_iter),
                                        float(tol), _p(factor_cache), warm_flag, _p(omega), _p(hd),
                                        _p(ws), wbytes, stats, _stream()), "ppbo_rff_fit")
    return omega, hd, dict(iterations=int(stats[0]), last_rel_step=stats[1], S=stats[2], info=rc,
                           factorizations=int(stats[3]), chord_steps=int(round((stats[3] - int(stats[3])) * 1000)),
                           binv_cached=bool(stats[4]))


def rff_hessian_factor_buffer(F, dev):
    """flat buffer for rff_hessian_factor: the F x F factor followed by the inverted 128-blocks its solves read"""
    return torch.empty(_lib.load().ppbo_rff_hessian_factor_doubles(F, F), dtype=F64, device=dev)


def hessian_factor_views(Lbuf, F):
    """(L [F x F] view, the solve workspace behind it) of a rff_hessian_factor buffer, as potrf_lower returns them"""
    return Lbuf[:F * F].view(F, F), Lbuf[F * F:]


def rff_hessian_factor(Phi_X, Q, m, sigma, omega, out, sync=True):
    """Cholesky factor of the exact weight-space Hessian I + Psi' diag(a) Psi (signed a at omega) into `out`
    (rff_hessian_factor_buffer); returns info (0, or the first non-positive pivot; sync=False: no host synchronisation, 0)"""
    lib = _lib.load()
    F = Phi_X.shape[0]
    wbytes = lib.ppbo_rff_hessian_factor_workspace_bytes(F, Q, m)
    ws = _scratch("rff_hessian", wbytes, Phi_X.device)
    info = ctypes.c_int(0)
    return check(lib.ppbo_rff_hessian_factor(_p(Phi_X), Phi_X.stride(0), F, Q, m, float(sigma), _p(omega), _p(out), F, _p(ws), wbytes,
                                             ctypes.byref(info) if sync else None, _stream()), "ppbo_rff_hessian_factor")


def rff_sample_omega_full(omega_map, Lbuf, S, Z=None, seed=0, stream_id=0, sample0=0):
    """Omega [S,F] ~ N(omega_map, H^-1) with H = L L' from rff_hessian_factor: omega_map + Z L^-1 (Z injected or Philox)"""
    lib = _lib.load()
    Fdim = omega_map.shape[0]
    Om = torch.empty((S, Fdim), dtype=F64, device=omega_map.device)
    for s0 in range(0, S, 65535):
        n = min(65535, S - s0)
        wbytes = lib.ppbo_rff_sample_omega_full_workspace_bytes(n, Fdim)
        ws = _scratch("rff_sample_full", wbytes, omega_map.device)
        check(lib.ppbo_rff_sample_omega_full(_p(omega_map), _p(Lbuf), Fdim, _p(None if Z is None else Z[s0:s0 + n]),
                                             Z.stride(0) if Z is not None else 0, int(seed), int(stream_id), int(sample0) + s0, n, Fdim,
                                             _p(Om[s0:s0 + n]), Fdim, _p(ws), wbytes, _stream()), "ppbo_rff_sample_omega_full")
    return Om


def rff_eval_argmax(Omega, PhiT_grid, want_full=False):
    """Omega [S,F]; PhiT_grid [B,P,F] -> fmax [B,S], arg [B,S], optional dense Fs [B,S,P]"""
    S, F = Omega.shape
    B, P, _ = PhiT_grid.shape
    fmax = torch.empty((B, S), dtype=F64, device=Omega.device)
    arg = torch.empty((B, S), dtype=torch.int32, device=Omega.device)
    full = torch.empty((B, S, P), dtype=F64, device=Omega.device) if want_full else None
    check(_lib.load().ppbo_rff_eval_argmax(_p(Omega), Omega.stride(0), S, F, _p(PhiT_grid), PhiT_grid.stride(1),
                                           PhiT_grid.stride(0), P, B, _p(fmax), _p(arg), _p(full), _stream()),
          "ppbo_rff_eval_argmax")
    return fmax, arg, full


def ozaki_slice(X, operand, slices=6):
    """X [rows,K] (operand 0: samples) or [B,rows,K] (operand 1: grid points) -> (digit planes int8, row scales) in the
    tensor-core operand layout of csrc/ozaki.cu"""
    lib = _lib.load()
    if X.dim() == 2:
        X = X.unsqueeze(0)
    B, rows, K = X.shape
    if X.stride(2) != 1:
        raise PPBOError("ozaki_slice: K must be contiguous")
    tr = lib.ppbo_ozaki_tile_rows(operand)
    planes = torch.empty(lib.ppbo_ozaki_plane_bytes(rows, K, tr, B, slices), dtype=torch.int8, device=X.device)
    scale = torch.empty(lib.ppbo_ozaki_scale_doubles(rows, tr, B), dtype=F64, device=X.device)
    check(lib.ppbo_ozaki_slice(_p(X), X.stride(1), X.stride(0), rows, K, tr, B, slices, _p(scale), _p(planes), _stream()),
          "ppbo_ozaki_slice")
    return planes, scale


def ozaki_sample_slice(omega_map, hess_diag, S, seed=0, stream_id=0, sample0=0, slices=6):
    """(digit planes, row scales) of the S Philox draws Omega ~ N(omega_map, diag(1 / -hess_diag)) without materialising Omega"""
    lib = _lib.load()
    Fdim = omega_map.shape[0]
    tr = lib.ppbo_ozaki_tile_rows(0)
    planes = torch.empty(lib.ppbo_ozaki_plane_bytes(S, Fdim, tr, 1, slices), dtype=torch.int8, device=omega_map.device)
    scale = torch.empty(lib.ppbo_ozaki_scale_doubles(S, tr, 1), dtype=F64, device=omega_map.device)
    check(lib.ppbo_ozaki_sample_slice(_p(omega_map), _p(hess_diag), int(seed), int(stream_id), int(sample0), S, Fdim, slices,
                                      _p(scale), _p(planes), _stream()), "ppbo_ozaki_sample_slice")
    return planes, scale


def ozaki_normal_slice(S, Fdim, dev, seed=0, stream_id=0, sample0=0, slices=6):
    """(digit planes, row scales) of the standard normals z[s][f] = Philox number (sample0 + s) F + f (ppbo_ozaki_normal_slice)"""
    lib = _lib.load()
    tr = lib.ppbo_ozaki_tile_rows(0)
    planes = torch.empty(lib.ppbo_ozaki_plane_bytes(S, Fdim, tr, 1, slices), dtype=torch.int8, device=dev)
    scale = torch.empty(lib.ppbo_ozaki_scale_doubles(S, tr, 1), dtype=F64, device=dev)
    check(lib.ppbo_ozaki_normal_slice(int(seed), int(stream_id), int(sample0), S, Fdim, slices, _p(scale), _p(planes), _stream()),
          "ppbo_ozaki_normal_slice")
    return planes, scale


def ozaki_rowmax(ap, asc, S, bp, bsc, P, B, F, slices, fmax=None, arg=None, want_full=False, err=None, bias=None):
    """fused INT8 GEMM + per-sample max / first arg-max from digit planes (ppbo_ozaki_rowmax); bias [B, P]: max over
    bias[b][p] + product (ppbo_ozaki_rowmax_bias)"""
    lib = _lib.load()
    dev = ap.device
    fmax = torch.empty((B, S), dtype=F64, device=dev) if fmax is None else fmax
    arg = torch.empty((B, S), dtype=torch.int32, device=dev) if arg is None else arg
    full = torch.empty((B, S, P), dtype=F64, device=dev) if want_full else None
    wbytes = lib.ppbo_ozaki_rowmax_workspace_bytes(S, P, B)
    ws = _scratch("ozaki_rowmax", wbytes, dev) if wbytes > 0 else None
    if bias is None:
        check(lib.ppbo_ozaki_rowmax(_p(ap), _p(asc), S, _p(bp), _p(bsc), P, B, F, slices, _p(fmax), _p(arg), _p(full), _p(ws), wbytes,
                                    _p(err), _stream()), "ppbo_ozaki_rowmax")
    else:
        if tuple(bias.shape) != (B, P) or not bias.is_contiguous():
            raise PPBOError("bias must be a contiguous [B, P] tensor")
        check(lib.ppbo_ozaki_rowmax_bias(_p(ap), _p(asc), S, _p(bp), _p(bsc), _p(bias), P, B, F, slices, _p(fmax), _p(arg), _p(full),
                                         _p(ws), wbytes, _p(err), _stream()), "ppbo_ozaki_rowmax_bias")
    return fmax, arg, full


def rff_eval_argmax_i8(Omega, PhiT_grid, slices=6, want_full=False, sliced_grid=None):
    """rff_eval_argmax on the tcgen05 INT8 tensor pipe (error-free splitting into `slices` digit planes per operand).
    sliced_grid: (planes, scale) of PhiT_grid from ozaki_slice(PhiT_grid, 1, slices) when the caller reuses them."""
    S, F = Omega.shape
    B, P, _ = PhiT_grid.shape
    ap, asc = ozaki_slice(Omega, 0, slices)
    bp, bsc = sliced_grid if sliced_grid is not None else ozaki_slice(PhiT_grid, 1, slices)
    err = torch.zeros(1, dtype=torch.int32, device=Omega.device)
    return ozaki_rowmax(ap, asc, S, bp, bsc, P, B, F, slices, want_full=want_full, err=err)


def normal_fill(seed, stream_id, offset, n, dev=None):
    """n standard normals: numbers offset .. offset+n-1 of Philox stream `stream_id` under `seed` (device-side RNG)."""
    out = torch.empty(n, dtype=F64, device=dev or device())
    check(_lib.load().ppbo_normal_fill(int(seed), int(stream_id), int(offset), _p(out), n, _stream()), "ppbo_normal_fill")
    return out


def rff_sample_omega(omega_map, hess_diag, S, Z=None, seed=0, stream_id=0, sample0=0):
    """Omega [S,F] ~ N(omega_map, diag(1 / -hess_diag)); Z [S,F] injects the standard normals, else Philox."""
    Fdim = omega_map.shape[0]
    Om = torch.empty((S, Fdim), dtype=F64, device=omega_map.device)
    check(_lib.load().ppbo_rff_sample_omega(_p(omega_map), _p(hess_diag), _p(Z), Z.stride(0) if Z is not None else 0,
                                            int(seed), int(stream_id), int(sample0), S, Fdim, _p(Om), Fdim, _stream()),
          "ppbo_rff_sample_omega")
    return Om


def acq_reduce_dev(fmax, mustar_dev):
    B, S = fmax.shape
    out = torch.empty((B, 3), dtype=F64, device=fmax.device)
    check(_lib.load().ppbo_acq_reduce_dev(_p(fmax), S, B, _p(mustar_dev), _p(out), _stream()), "ppbo_acq_reduce_dev")
    return out


def acq_batch_gain(fmax, mustar_dev, cur, k, q, out=None):
    """gains [B + 1] of greedy step k over this rank's samples: gain[b] = sum_s max(max(cur[s], fmax[b][s]) - mu*, 0), gain[B] = S"""
    B, S = fmax.shape
    out = torch.empty(B + 1, dtype=F64, device=fmax.device) if out is None else out
    check(_lib.load().ppbo_acq_batch_gain(_p(fmax), S, B, _p(mustar_dev), _p(cur), int(k), int(q), _p(out), _stream()),
          "ppbo_acq_batch_gain")
    return out


def acq_batch_pick(gain, fmax, k, q, idx, val, cur):
    """step k: idx[k] = best candidate not in idx[:k] (lowest index on ties), val[k] = gain[idx[k]] / gain[B], cur updated with its
    maxima.  fmax None: a rank without samples (picks only)."""
    B = gain.shape[0] - 1
    S = 0 if fmax is None else fmax.shape[1]
    check(_lib.load().ppbo_acq_batch_pick(_p(gain), B, _p(fmax), S, int(k), int(q), _p(idx), _p(val), _p(cur), _stream()),
          "ppbo_acq_batch_pick")


def vec_max(x, out=None, accumulate=False):
    out = torch.empty(1, dtype=F64, device=x.device) if out is None else out
    check(_lib.load().ppbo_vec_max(_p(x), x.numel(), 1 if accumulate else 0, _p(out), _stream()), "ppbo_vec_max")
    return out


def rff_value_grad(W, b, omega, x, sigma_f):
    """(phi(x)' omega, gradient in x) as one [1 + D] device tensor"""
    Fdim, D = W.shape
    out = torch.empty(1 + D, dtype=F64, device=W.device)
    check(_lib.load().ppbo_rff_value_grad(_p(W), _p(b), Fdim, D, _p(omega), _p(x), float(sigma_f), _p(out), _stream()),
          "ppbo_rff_value_grad")
    return out
