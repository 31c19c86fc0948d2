"""One PPBO iteration on the device: GP Laplace fit  ->  RFF weight-space fit  ->  sampled acquisition over the
projected xi-grids of every query direction (BASELINE.json north_star; reference call stack SURVEY.md 3.1-3.4).

Host side is Python/torch for memory, streams and torch.distributed only; all arithmetic goes through the C ABI
(`ops`).  Data layout in HBM (all row-major float64):

    X        [N x D]      design matrix, N = Q (m+1), comparison set q = rows q(m+1)..q(m+1)+m, winner first
    Sigma    [N x N]      regularised prior covariance                      (GPModel.Sigma)
    G, Lfac  [M x M]      difference-space Gram B'Sigma B and the Cholesky factor at the mode, M = Q m
    Phi_X    [F x N]      RFF features of the design (feature-major, the reference's Hsampler.phi_X layout)
    Omega    [S_loc x F]  this rank's posterior weight samples (K-contiguous A operand of the sampling GEMM)
    PhiT     [B][P x F]   RFF features of grid b, point-major (K-contiguous B operand)
    fmax,arg [B][S_loc]   per-sample max / first arg-max over the grid (the S x P product never reaches HBM)

Multi-GPU (SURVEY.md 8e): only the Monte-Carlo samples are partitioned.  Rank 0 fits and broadcasts the small fit
products (omega_MAP, hess_diag, mu*: 8(2F+1) bytes); every rank draws its own slice of the counter-based normal stream,
evaluates its S/R samples on all B grids and one all-reduce(sum) of the 3B partial sums follows.
"""
import threading

import numpy as np
import torch

from . import ops
from ._lib import PPBOError

F64 = torch.float64
SHRINKAGE = 1e-6          # GPModel.COVARIANCE_SHRINKAGE, src/gp_model.py:26
# Sampling contraction Omega . PhiT^T: "i8" = tcgen05 INT8 tensor pipe with error-free splitting into SLICES base-256 digit
# planes per operand (csrc/ozaki.cu; 6 planes: ~1e-13 relative, i.e. the accuracy of an FP64 GEMM of this depth), "f64" = the
# FP64 DMMA kernel.  Small contractions (reference-size grids) stay on the FP64 kernel: a 128 x 64 INT8 tile would be mostly
# padding there.
SAMPLING_ENGINE = "i8"
SAMPLING_SLICES = 6
I8_MIN_WORK = 1 << 24     # S * P * F below which the FP64 kernel is used
# Covariance of the weight-space Laplace posterior the draws come from: "diag" = the reference's 1 / -hess_diag
# (src/random_fourier_sampler.py:134-137), "full" = the inverse of the exact Hessian I + Psi' diag(a) Psi (opt-in).  With "full" the
# draws stay standard normals z_s and the covariance moves into the grid operand: f_s(x_p) = mu_p + z_s . Phi~_p with
# mu_p = phi(x_p)' omega_MAP and Phi~ = Phi L^-T, H = L L'.
WEIGHT_COVARIANCES = ("diag", "full")


# The GP fit and the weight-space (RFF) fit only share their input X: both are chains of small, latency-bound launches with one
# host decision per Newton step, so rank 0 drives them from two host threads on two streams and the shorter one (RFF) hides
# behind the longer.  The RFF fit then starts from omega = 0 (or the caller's omega0) instead of the projection of the GP mode,
# which costs one extra Newton step (20 against 19 on the Ackley-20D bench problem).
CONCURRENT_FITS = True
# One GPU: the sampling contraction needs the weight-space fit only (mu* enters at the reduction), so the background thread goes
# on from the weight-space fit to the draws and the INT8 contraction on its lowest-priority stream WHILE the GP fit -- a chain of
# small, latency-bound kernels that leaves most SMs idle -- runs beside it.  The contraction's persistent grid then leaves
# OVERLAP_RESERVED_SMS(_COLD) SMs to the fit (tuning key 14); a contraction CTA fills its SM, so the two never share one.
# PPBO_OVERLAP_SAMPLING=0 restores the sequential order (diagnostics).
import os as _os
# Reserved SMs: an appended iteration's GP chain is short (it still ends before the contraction on 8 SMs); a cold fit has 13
# chord steps with one 100 MB half-triangle mat-vec of G each plus the factorisation and is the longer chain, so it gets more
# (sweeps in DESIGN.md 5.1).
_RESERVE_ENV = _os.environ.get("PPBO_OVERLAP_RESERVE")
OVERLAP_RESERVED_SMS = int(_RESERVE_ENV) if _RESERVE_ENV else 12            # appended iterations
OVERLAP_RESERVED_SMS_COLD = int(_RESERVE_ENV) if _RESERVE_ENV else 24       # cold iterations
# Steady state of the overlapped pipeline, opt-in: refresh the weight-space Hessian factor at each new optimum while the contraction
# runs (RFFState.refresh_factor).  The next fit then needs 10 chord steps and never a mid-fit refactorisation (7-13 steps and a
# refactorisation in 6 of 13 iterations with the stale factor, tests/test_steady_state.py), but the refresh (10 GFLOP of Hessian GEMM + a Cholesky) shares
# the reserved SMs with the GP chain, which then ends AFTER the contraction: 14.05 ms per appended iteration against 13.09 without
# (measured), so it is off.
REFRESH_RFF_FACTOR = _os.environ.get("PPBO_RFF_REFRESH", "0") != "0"
OVERLAP_SAMPLING = _os.environ.get("PPBO_OVERLAP_SAMPLING", "1") != "0"


def sampling_engine(S, P, Fdim):
    return "i8" if (SAMPLING_ENGINE == "i8" and S * P * Fdim >= I8_MIN_WORK) else "f64"


class SlicedGrids:
    """PhiT [B, P, F] together with its INT8 digit planes (computed once per iteration, before the fit is known)."""
    __slots__ = ("PhiT", "planes", "scale", "slices")

    def __init__(self, PhiT, slices=None):
        self.PhiT, self.slices = PhiT, SAMPLING_SLICES if slices is None else slices
        self.planes, self.scale = ops.ozaki_slice(PhiT, 1, self.slices)

    @property
    def shape(self):
        return self.PhiT.shape


class Shard:
    """Which slice of the S Monte-Carlo samples this process owns (rank r of R: samples [lo, hi))."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist if (dist.is_available() and dist.is_initialized()) else None
        self.group = group
        self.rank = self.dist.get_rank(group) if self.dist else 0
        self.world = self.dist.get_world_size(group) if self.dist else 1

    def bounds(self, S):
        lo = (S * self.rank) // self.world
        hi = (S * (self.rank + 1)) // self.world
        return lo, hi

    def sample_bounds(self, S, shares=None):
        """Partition of the Monte-Carlo samples inside run_iteration.  shares: one non-negative weight per rank (plan_shares);
        the default gives the rank that runs the GP fit (rank 0) none: the sampling contraction does not depend on the GP fit
        -- only the final reduction needs mu* -- so the other ranks evaluate all samples WHILE rank 0 fits.  For large S the
        boundaries are multiples of 128 samples (one row tile of the tensor-core kernel) except the last."""
        if self.world == 1:
            return 0, S
        if shares is None:
            shares = [0.0] + [1.0] * (self.world - 1)
        tot = float(sum(shares))
        align = 128 if S >= 512 * self.world else 1
        cum, edges = 0.0, [0]
        for w in shares:
            cum += w
            e = int(round(S * cum / tot / align)) * align
            edges.append(min(S, max(edges[-1], e)))
        edges[-1] = S
        return edges[self.rank], edges[self.rank + 1]

    def broadcast(self, t, src=0):
        if self.dist and self.world > 1:
            self.dist.broadcast(t, src=src, group=self.group)
        return t

    def all_reduce_sum(self, t):
        if self.dist and self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return t

    def all_reduce_max(self, t):
        if self.dist and self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
        return t


def plan_shares(world, t_gp, t_rff, t_sampling, rff_rank=1):
    """Sample shares per rank from measured stage times (ms): rank 0 is busy with the GP fit + mu* for t_gp, every other rank can
    start sampling when the weight-space fit (t_rff, on rff_rank) has been broadcast, and the whole sample set costs t_sampling
    on one GPU.  Water-filling: all ranks that sample finish together at time t with sum_r max(0, t - start_r) = t_sampling."""
    if world == 1:
        return [1.0]
    starts = [t_gp if r == 0 else t_rff for r in range(world)]
    order = sorted(range(world), key=lambda r: starts[r])
    t = starts[order[0]]
    for k in range(1, world + 1):
        active = order[:k]
        t = (t_sampling + sum(starts[r] for r in active)) / k
        if k == world or t <= starts[order[k]]:
            break
    return [max(0.0, t - starts[r]) for r in range(world)]


class GPFit:
    """Device-resident products of GPModel.update_model (src/gp_model.py:87-132)."""
    __slots__ = ("X", "kernel", "theta", "lengthscales", "Q", "m", "Sigma", "lap")

    @property
    def f_map(self):
        return self.lap.f_map

    @property
    def alpha(self):
        return self.lap.alpha


def gp_fit(X, kernel, theta, Q, m, f_init=None, lengthscales=None, max_iter=100, tol=1e-10, shrinkage=SHRINKAGE,
           factor_at_mode=False):
    """Sigma = reg(K(X,X)) and the Laplace mode of T (update_Sigma + update_fMAP + Lambda_MAP, src/gp_model.py:157,354,111).
    factor_at_mode: also leave the Cholesky factor of the Newton matrix AT the mode behind (prediction with covariance needs it;
    the RFF acquisition and mu* do not -- LaplaceFit builds it on first use otherwise)."""
    g = GPFit()
    g.X, g.kernel, g.theta, g.Q, g.m = X, kernel, [float(t) for t in theta], Q, m
    g.lengthscales = theta[1] if lengthscales is None else lengthscales
    if X.shape[0] != Q * (m + 1):
        raise PPBOError("X must have Q (m+1) rows")
    g.Sigma = ops.gram_regularized(kernel, X, g.lengthscales, theta[2], shrinkage)
    g.lap = ops.laplace_fit(g.Sigma, Q, m, theta[0], f_init=f_init, max_iter=max_iter, tol=tol, factor_at_mode=factor_at_mode)
    if g.lap.info != 0:
        raise PPBOError("Laplace fit: system not positive definite (info=%d)" % g.lap.info)
    return g


class GPState(GPFit):
    """A GP model that grows in place (SURVEY.md 8f rank 2; FeedbackProcessing.update_X appends one (m+1)-row block per
    iteration, src/feedback_processing.py:133-154).  Capacity buffers for X, Sigma, G = B' Sigma B and the factor object; `append`
    adds comparison sets in O(N^2 m): new rows of Sigma and G, the factor of the previous iteration grown by the new rows, and
    a chord iteration from the previous mode (new points start at their posterior mean) -- no O(N^3) factorisation unless the
    chord steps contract too slowly (ppbo_laplace_fit falls back to a Newton step by itself)."""
    __slots__ = ("Q_cap", "X_cap", "Sigma_cap", "f_buf", "alpha_buf", "arrow_buf", "f_init_buf", "alpha_init_buf", "shrinkage",
                 "max_iter", "tol")

    def __init__(self, kernel, theta, D, m, Q_cap, dev, lengthscales=None, max_iter=100, tol=1e-8, shrinkage=SHRINKAGE):
        lib = ops._lib.load()
        self.kernel, self.theta, self.m, self.Q, self.Q_cap = kernel, [float(t) for t in theta], m, 0, Q_cap
        self.lengthscales = theta[1] if lengthscales is None else lengthscales
        self.shrinkage, self.max_iter, self.tol = shrinkage, max_iter, tol
        Nr, Mc = Q_cap * (m + 1), (Q_cap * m + 15) // 16 * 16     # leading dimensions: multiples of 16 doubles (the specialised
        Nc = (Nr + 15) // 16 * 16                                   # Cholesky / GEMM kernels want 16-byte aligned rows)
        self.X_cap = torch.empty((Nr, D), dtype=F64, device=dev)
        self.Sigma_cap = torch.empty((Nc, Nc), dtype=F64, device=dev)
        self.f_buf, self.alpha_buf, self.f_init_buf, self.alpha_init_buf = (torch.empty(Nc, dtype=F64, device=dev) for _ in range(4))
        self.arrow_buf = torch.empty(Mc, dtype=F64, device=dev)
        lap = ops.LaplaceFit()
        lap.cap = lap.ldg = Mc
        lap.G = torch.empty((Mc, Mc), dtype=F64, device=dev)
        lap._Lfac = torch.empty(lib.ppbo_factor_doubles(Mc), dtype=F64, device=dev)
        lap.sa_fac = torch.empty(Mc, dtype=F64, device=dev)
        lap.binv_cache = torch.empty(lib.ppbo_blockinv_bytes(Mc) // 8 + 2, dtype=F64, device=dev)
        import ctypes
        lap.binv_state = (ctypes.c_int * 2)(0, 0)
        lap.m, lap.Q, lap.sigma, lap.info, lap.factor_state = m, 0, float(theta[0]), 0, 0
        self.lap = lap
        self.X = self.Sigma = None

    def _views(self, Q):
        N, M = Q * (self.m + 1), Q * self.m
        self.X, self.Sigma = self.X_cap[:N], self.Sigma_cap[:N, :N]
        self.lap.f_map, self.lap.alpha, self.lap.arrow = self.f_buf[:N], self.alpha_buf[:N], self.arrow_buf[:M]
        return N, M

    def cold(self, X, f_init=None, factor_at_mode=False):
        """fit from scratch on X [Q (m+1) x D] (device)"""
        Q = X.shape[0] // (self.m + 1)
        if Q > self.Q_cap or Q * (self.m + 1) != X.shape[0]:
            raise PPBOError("X must have Q (m+1) rows with Q <= capacity")
        N, _ = self._views(Q)
        self.X_cap[:N].copy_(X)
        ops.gram_regularized(self.kernel, self.X, self.lengthscales, self.theta[2], self.shrinkage, out=self.Sigma)
        ops.laplace_fit(self.Sigma, Q, self.m, self.theta[0], f_init=f_init, max_iter=self.max_iter, tol=self.tol,
                        factor_at_mode=factor_at_mode, into=self.lap)
        if self.lap.info != 0:
            raise PPBOError("Laplace fit: system not positive definite (info=%d)" % self.lap.info)
        self.Q = Q
        return self

    def append(self, X_block, factor_at_mode=False):
        """add the comparison sets X_block [q (m+1) x D] (device) and refit from the previous mode"""
        if self.Q == 0:
            return self.cold(X_block, factor_at_mode=factor_at_mode)
        m, Q_old = self.m, self.Q
        Q_new = Q_old + X_block.shape[0] // (m + 1)
        if Q_new > self.Q_cap or X_block.shape[0] % (m + 1):
            raise PPBOError("appended rows must be whole comparison sets within the capacity")
        N_old, M_old = Q_old * (m + 1), Q_old * m
        alpha_old = self.alpha_buf[:N_old]
        warm = self.lap.factor_state >= 1 and self.lap.info == 0
        N, M = self._views(Q_new)
        self.X_cap[N_old:N].copy_(X_block)
        ops.gram_append(self.kernel, self.X, N_old, self.lengthscales, self.theta[2], self.shrinkage, self.Sigma_cap)
        ops.diffspace_gram_append(self.Sigma, Q_old, Q_new, m, self.lap.G)
        # warm start: alpha = [alpha_old, 0] and f = Sigma_new alpha, i.e. the previous mode on the old rows and the posterior mean
        # k(x_new, X_old) alpha_old on the new ones -- consistent by construction, so the chord iteration (with its acceptance
        # test) starts at once.  (The reference pads fMAP with its mean, src/gp_model.py:375-377; both are starts for the same
        # fixed point.)
        f_init, alpha_init = self.f_init_buf[:N], self.alpha_init_buf[:N]
        f_init[:N_old].copy_(self.f_buf[:N_old])
        ops.gemv(self.Sigma_cap[N_old:N, :N_old], alpha_old, out=f_init[N_old:])
        alpha_init[:N_old].copy_(alpha_old)
        alpha_init[N_old:].zero_()
        self.lap.Q = Q_new
        ops.laplace_fit(self.Sigma, Q_new, m, self.theta[0], f_init=f_init, alpha_init=alpha_init, max_iter=self.max_iter,
                        tol=self.tol, factor_at_mode=factor_at_mode, into=self.lap, g_ready=True, warm_rows=M_old if warm else 0)
        if self.lap.info != 0:
            raise PPBOError("Laplace fit: system not positive definite (info=%d)" % self.lap.info)
        self.Q = Q_new
        return self


def posterior_mean(g, Xp):
    """mu(Xp) = k(Xp, X) alpha  (GPModel.mu_pred, src/gp_model.py:454-458, batched over the rows of Xp)."""
    mu, _ = ops.predict(g.kernel, g.X, g.lengthscales, g.theta[2], SHRINKAGE, g.lap, Xp, Xp.shape[0], 1, want_cov=False)
    return mu.view(-1)


def mustar_over_candidates(g, candidates=None):
    """mu* = max posterior mean over the design rows (= max f_MAP) and optional candidate points; stays on the device.
    Batched stand-in for the sequential differential evolution of GPModel.mu_star (src/gp_model.py:415-437)."""
    out = ops.vec_max(g.f_map)
    if candidates is not None and candidates.shape[0] > 0:
        ops.vec_max(posterior_mean(g, candidates), out=out, accumulate=True)
    return out


class RFFFit:
    """Device-resident state of Hsampler after update_phi_X / update_omega_MAP / update_covariancematrix.  L: buffer of the exact
    Hessian factor (ops.rff_hessian_factor_buffer) for the full covariance, None for the diagonal one."""
    __slots__ = ("W", "b", "sigma_f", "Phi_X", "omega_map", "hess_diag", "stats", "L")

    def __init__(self):
        self.L = None


def rff_full_factor(r, Q, m, sigma, out=None):
    """r.L <- factor of the exact weight-space Hessian at r.omega_map (into `out`, a rff_hessian_factor_buffer, or a new one)"""
    Fdim = r.omega_map.shape[0]
    out = ops.rff_hessian_factor_buffer(Fdim, r.omega_map.device) if out is None else out
    info = ops.rff_hessian_factor(r.Phi_X, Q, m, sigma, r.omega_map, out)
    if info != 0:
        raise PPBOError("exact weight-space Hessian not positive definite (pivot %d)" % info)
    r.L = out
    return r


def rff_fit(X, W, b, theta, Q, m, omega0=None, max_iter=100, tol=1e-10, f_map=None):
    """omega0=None with f_map given: start from the projection of the GP mode (rff_start_from_gp); else from omega0 / zero"""
    r = RFFFit()
    r.W, r.b, r.sigma_f = W, b, float(theta[2])
    r.Phi_X = ops.rff_features(W, b, X, theta[2], feature_major=True)
    if omega0 is None and f_map is not None:
        omega0 = rff_start_from_gp(r.Phi_X, f_map)
    r.omega_map, r.hess_diag, r.stats = ops.rff_fit(r.Phi_X, Q, m, theta[0], omega0=omega0, max_iter=max_iter, tol=tol)
    if r.stats["info"] != 0:
        raise PPBOError("RFF fit: weight-space Hessian not positive definite (info=%d)" % r.stats["info"])
    return r


class RFFState:
    """Weight-space model that grows with the design: capacity buffer for Phi_X [F x N_cap]; `append` adds the features of the new
    rows and refits from the previous omega_MAP."""

    def __init__(self, W, b, theta, m, Q_cap, max_iter=100, tol=1e-8):
        self.W, self.b, self.theta, self.m, self.Q, self.Q_cap = W, b, [float(t) for t in theta], m, 0, Q_cap
        self.max_iter, self.tol = max_iter, tol
        self.Phi_cap = torch.empty((W.shape[0], Q_cap * (m + 1)), dtype=F64, device=W.device)
        self.factor_cache = ops.rff_factor_cache(W.shape[0], W.device)
        self.L_buf = None            # exact-Hessian factor of the full covariance: its own buffer, never the fit's factor_cache
        self.fit = None
        self.pending = None          # stream of an asynchronous refresh of the factor (refresh_factor): the next fit waits for it

    def _fit(self, Q, omega0, warm=False):
        r = RFFFit()
        r.W, r.b, r.sigma_f = self.W, self.b, self.theta[2]
        r.Phi_X = self.Phi_cap[:, :Q * (self.m + 1)]
        r.omega_map, r.hess_diag, r.stats = ops.rff_fit(r.Phi_X, Q, self.m, self.theta[0], omega0=omega0, max_iter=self.max_iter,
                                                        tol=self.tol, factor_cache=self.factor_cache, warm=warm)
        if r.stats["info"] != 0:
            raise PPBOError("RFF fit: weight-space Hessian not positive definite (info=%d)" % r.stats["info"])
        self.Q, self.fit = Q, r
        return r

    def hessian_factor(self):
        """exact-Hessian factor of the current fit (full covariance) into this model's own buffer"""
        if self.L_buf is None:
            self.L_buf = ops.rff_hessian_factor_buffer(self.W.shape[0], self.W.device)
        return rff_full_factor(self.fit, self.Q, self.m, self.theta[0], out=self.L_buf)

    def _wait_refresh(self):
        if self.pending is not None:
            torch.cuda.current_stream().wait_stream(self.pending)
            self.pending = None

    def refresh_factor(self):
        """Rebuild the Hessian factor (and its block inverses) at the optimum just found, asynchronously on the CURRENT stream: the
        next append then starts its chord steps from a factor built at its own starting point (ppbo_rff_refactor).  The caller
        runs this off the critical path and leaves the stream in self.pending."""
        r = self.fit
        ops.rff_refactor(r.Phi_X, self.Q, self.m, self.theta[0], r.omega_map, self.factor_cache)
        r.stats["warm"] = True
        r.stats["binv_cached"] = True
        self.pending = torch.cuda.current_stream()

    def cold(self, X, omega0=None):
        self._wait_refresh()
        Q = X.shape[0] // (self.m + 1)
        ops.rff_features(self.W, self.b, X, self.theta[2], True, out=self.Phi_cap[:, :X.shape[0]])
        return self._fit(Q, omega0)

    def append(self, X_block):
        if self.Q == 0:
            return self.cold(X_block)
        self._wait_refresh()
        N_old = self.Q * (self.m + 1)
        ops.rff_features(self.W, self.b, X_block, self.theta[2], True, out=self.Phi_cap[:, N_old:N_old + X_block.shape[0]])
        warm = self.fit.stats.get("factorizations", 0) > 0 or self.fit.stats.get("warm", False)
        if warm and self.fit.stats.get("binv_cached", False):
            warm = 2                            # the cache also holds the block inverses of its factor
        r = self._fit(self.Q + X_block.shape[0] // (self.m + 1), self.fit.omega_map, warm=warm)
        r.stats["warm"] = True              # the cache holds a factor from now on
        return r


def rff_start_from_gp(Phi_X, f_map, ridge=1e-3):
    """omega0 = argmin |Phi_X' omega - f_MAP|^2 + lambda |omega|^2: the weight vector whose function is closest to the GP mode.
    The reference starts its weight-space optimiser at a random omega0 ~ N(0, I) (src/random_fourier_sampler.py:125); S is
    not concave, so the start decides which optimum is reached -- this one is deterministic and a few Newton steps away."""
    A = ops.gemm_nt(Phi_X, Phi_X)                      # F x F, contraction over the N design rows
    ops.shrink_inplace(A, ridge)
    info, ws = ops.potrf_lower(A)
    if info != 0:
        raise PPBOError("feature Gram matrix not positive definite (info=%d)" % info)
    return ops.potrs_vec(A, ws, ops.gemv(Phi_X, f_map))


def line_grids(xis, xs, alphas):
    """grids[b][p] = alphas[b][p] * xi[b] + x[b]  (FeedbackProcessing.xi_grid with is_scaled=True,
    src/feedback_processing.py:47-108).  Host arrays in, [B, P, D] host array out (tiny: the jitter of the alphas
    consumes the host RNG in reference order, so this stays on the host)."""
    xis, xs, alphas = np.asarray(xis, float), np.asarray(xs, float), np.asarray(alphas, float)
    return alphas[:, :, None] * xis[:, None, :] + xs[:, None, :]


def rff_grid_features(W, b, sigma_f, grids):
    """PhiT [B, P, F] for device grids [B, P, D]"""
    B, P, D = grids.shape
    return ops.rff_features(W, b, grids.reshape(B * P, D), sigma_f, feature_major=False).view(B, P, -1)


class SlicedSamples:
    """Digit planes of the posterior weight draws [lo, hi) (the A operand of the INT8 sampling contraction)."""
    __slots__ = ("planes", "scale", "count", "slices")

    def __init__(self, Omega=None, slices=None, drawn=None, count=None):
        self.slices = SAMPLING_SLICES if slices is None else slices
        if drawn is not None:                       # (planes, scale) straight from the fused draw
            self.planes, self.scale = drawn
            self.count = count
        else:
            self.count = Omega.shape[0]
            self.planes, self.scale = ops.ozaki_slice(Omega, 0, self.slices)


def rff_prepare_normals(Fdim, lo, hi, P, dev, Z=None, seed=0, stream_id=0):
    """Standard normals [lo, hi) of the sample stream (the draws of the full covariance) in the form the contraction consumes: digit
    planes for the INT8 engine, the FP64 matrix otherwise.  Independent of every fit."""
    if hi <= lo:
        return None
    i8 = sampling_engine(hi - lo, P, Fdim) == "i8"
    if Z is None and i8 and Fdim * 64 <= 200 * 1024:
        return SlicedSamples(drawn=ops.ozaki_normal_slice(hi - lo, Fdim, dev, seed=seed, stream_id=stream_id, sample0=lo,
                                                          slices=SAMPLING_SLICES), count=hi - lo)
    Zloc = Z[lo:hi] if Z is not None else ops.normal_fill(seed, stream_id, lo * Fdim, (hi - lo) * Fdim, dev).view(hi - lo, Fdim)
    return SlicedSamples(Zloc) if i8 else Zloc


def rff_transform_grids(r, PhiT, slices=None):
    """(mu [B, P], Phi~): the posterior mean phi(x_p)' omega_MAP and the grid features Phi L^-T of the full covariance, Phi~ cut
    into `slices` digit planes (SlicedGrids) when given.  The triangular solve treats all B P rows in one call: same bits on
    every rank."""
    G = PhiT.PhiT if isinstance(PhiT, SlicedGrids) else PhiT
    B, P, Fdim = G.shape
    mu = ops.gemv(G.reshape(B * P, Fdim), r.omega_map).view(B, P)
    L, ws = ops.hessian_factor_views(r.L, Fdim)
    Gt = G.reshape(B * P, Fdim).clone()
    ops.trsm_right_lower(L, ws, Gt)                    # rows phi_p' L^-T = (L^-1 phi_p)'
    Gt = Gt.view(B, P, Fdim)
    return mu, (SlicedGrids(Gt, slices) if slices is not None else Gt)


def rff_prepare_samples(r, lo, hi, P, Z=None, seed=0, stream_id=0, covariance="diag"):
    """Draws [lo, hi) of the sample stream, already in the form the contraction consumes (digit planes for the INT8 engine, the
    FP64 matrix otherwise).  Needs the weight-space fit only, so run_iteration does this while the GP fit is still running.
    covariance="full": the standard normals themselves (rff_prepare_normals)."""
    if hi <= lo:
        return None
    Fdim = r.omega_map.shape[0]
    if covariance == "full":
        return rff_prepare_normals(Fdim, lo, hi, P, r.omega_map.device, Z=Z, seed=seed, stream_id=stream_id)
    if Z is None and sampling_engine(hi - lo, P, Fdim) == "i8" and Fdim * 64 <= 200 * 1024:
        # draws and digit planes in one kernel: the S x F matrix of draws never reaches HBM
        return SlicedSamples(drawn=ops.ozaki_sample_slice(r.omega_map, r.hess_diag, hi - lo, seed=seed, stream_id=stream_id, sample0=lo,
                                                          slices=SAMPLING_SLICES), count=hi - lo)
    Zloc = None if Z is None else Z[lo:hi]
    Omega = ops.rff_sample_omega(r.omega_map, r.hess_diag, hi - lo, Z=Zloc, seed=seed, stream_id=stream_id, sample0=lo)
    return SlicedSamples(Omega) if sampling_engine(hi - lo, P, Fdim) == "i8" else Omega


def rff_sampled_maxima(r, PhiT, lo, hi, Z=None, seed=0, stream_id=0, prepared=None, covariance="diag", transformed=None):
    """Posterior weight draws [lo, hi) of the sample stream evaluated on every grid: per-sample max and first arg-max over the grid
    points, (fmax [B, hi-lo], arg [B, hi-lo]); (None, None) for an empty slice.  Needs the weight-space fit only -- not mu*.
    prepared: the result of rff_prepare_samples for the same slice.  covariance="full" (r.L set): max_p (mu_p + z_s . Phi~_p);
    transformed: rff_transform_grids(r, PhiT) when the caller has it already."""
    if hi <= lo:
        return None, None
    if covariance == "full":
        return _sampled_maxima_full(r, PhiT, lo, hi, Z, seed, stream_id, prepared, transformed)
    sliced = PhiT if isinstance(PhiT, SlicedGrids) else None
    PhiT = sliced.PhiT if sliced is not None else PhiT
    B, P, Fdim = PhiT.shape
    if prepared is None:
        prepared = rff_prepare_samples(r, lo, hi, P, Z=Z, seed=seed, stream_id=stream_id)
    if isinstance(prepared, SlicedSamples):
        bp, bsc = (sliced.planes, sliced.scale) if sliced is not None else ops.ozaki_slice(PhiT, 1, prepared.slices)
        err = torch.zeros(1, dtype=torch.int32, device=PhiT.device)
        fmax, arg, _ = ops.ozaki_rowmax(prepared.planes, prepared.scale, prepared.count, bp, bsc, P, B, Fdim, prepared.slices, err=err)
    else:
        fmax, arg, _ = ops.rff_eval_argmax(prepared, PhiT)
    return fmax, arg


def _sampled_maxima_full(r, PhiT, lo, hi, Z, seed, stream_id, prepared, transformed):
    G = PhiT.PhiT if isinstance(PhiT, SlicedGrids) else PhiT
    B, P, Fdim = G.shape
    if prepared is None:
        prepared = rff_prepare_normals(Fdim, lo, hi, P, G.device, Z=Z, seed=seed, stream_id=stream_id)
    if transformed is None:
        transformed = rff_transform_grids(r, G, slices=prepared.slices if isinstance(prepared, SlicedSamples) else None)
    mu, Gt = transformed
    if isinstance(prepared, SlicedSamples):
        err = torch.zeros(1, dtype=torch.int32, device=G.device)
        fmax, arg, _ = ops.ozaki_rowmax(prepared.planes, prepared.scale, prepared.count, Gt.planes, Gt.scale, P, B, Fdim, prepared.slices,
                                        err=err, bias=mu)
    else:                                              # FP64 engine: the mean-offset row max of the exact-GP sampler
        fmax, arg = ops.mvn_rowmax(prepared.unsqueeze(0).expand(B, -1, -1), Gt, mu)
    return fmax, arg


def rff_reduce(fmax, mustar_dev, n_grids, shard=None):
    """sums [B, 3] over all ranks' samples of max(fmax - mu*, 0), fmax, fmax^2 (one all-reduce of 3 B doubles)"""
    shard = shard or Shard()
    if fmax is not None:
        sums = ops.acq_reduce_dev(fmax, mustar_dev)
    else:
        sums = torch.zeros((n_grids, 3), dtype=F64, device=mustar_dev.device)
    shard.all_reduce_sum(sums)
    return sums


def rff_acquisition(r, PhiT, S, mustar_dev, shard=None, Z=None, seed=0, stream_id=0, bounds=None, prepared=None, n_grids=None,
                    covariance="diag"):
    """Sampled acquisition on B grids: per grid b the sums over the S samples of max(fmax - mu*, 0), fmax and fmax^2
    (acquisition.EI / varmax, src/acquisition.py:78-81,176-178, with RFF posterior draws in place of the exact-GP MVN).
    Returns (sums [B,3] reduced over all ranks, fmax [B,S_loc], arg [B,S_loc]); bounds: this rank's samples (default: even split)."""
    shard = shard or Shard()
    lo, hi = bounds if bounds is not None else shard.bounds(S)
    fmax, arg = rff_sampled_maxima(r, PhiT, lo, hi, Z=Z, seed=seed, stream_id=stream_id, prepared=prepared, covariance=covariance)
    if n_grids is None:                 # (a rank without samples has no grid features: the caller passes the count)
        n_grids = (PhiT.PhiT if isinstance(PhiT, SlicedGrids) else PhiT).shape[0]
    return rff_reduce(fmax, mustar_dev, n_grids, shard), fmax, arg


def acquisition_values(sums, S):
    """host: EI and variance-of-max per grid from the reduced sums (src/acquisition.py:81,178)."""
    s = np.asarray(sums, dtype=float)
    ei = s[:, 0] / S
    mean = s[:, 1] / S
    var = np.maximum(s[:, 2] / S - mean * mean, 0.0)          # one-pass form: clamp the round-off of the cancellation
    return ei, var


class IterationInputs:
    """Host-side (pinned) inputs of one iteration; `to_device` is the H2D leg measured by bench.py's e2e."""
    FIELDS = ("X", "f_init", "W", "b", "omega0", "grids")

    def __init__(self, X, f_init, W, b, omega0, grids):
        self.host = {}
        for k, v in zip(self.FIELDS, (X, f_init, W, b, omega0, grids)):
            if v is None:
                continue
            t = torch.from_numpy(np.ascontiguousarray(np.asarray(v, dtype=np.float64)))
            self.host[k] = t.pin_memory() if torch.cuda.is_available() else t

    def nbytes(self):
        return sum(t.numel() * 8 for t in self.host.values())

    def to_device(self, dev):
        return {k: t.to(dev, non_blocking=True) for k, t in self.host.items()}


_SIDE_STREAMS = {}
# The GP fit is the critical path of the iteration: its launches go to a stream one level above the default priority, its
# Cholesky bulk (library-internal side stream) sits at the same level, and the background weight-space fit keeps the default
# (lowest) priority for everything (ppbo_set_thread_background), so it only fills the SMs the GP fit leaves idle.
# None / 0: stay on the caller's stream.
GP_STREAM_PRIORITY = int(_os.environ.get("PPBO_FG_PRIORITY", "-1"))
_WORKER = None


def _background_worker():
    """One persistent host thread for the concurrent weight-space fit (the library keeps per-thread streams: a fresh thread per
    iteration would create new ones every time).  Marked as background before its first launch."""
    global _WORKER
    if _WORKER is None:
        from concurrent.futures import ThreadPoolExecutor
        from . import _lib
        _WORKER = ThreadPoolExecutor(max_workers=1, thread_name_prefix="ppbo-rff-fit",
                                     initializer=lambda: _lib.load().ppbo_set_thread_background(1))
    return _WORKER


def _side_stream(dev, priority=0, tag=""):
    key = (dev.type, dev.index, priority, tag)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=dev, priority=priority)
    return _SIDE_STREAMS[key]


class IterationState:
    """What persists between the iterations of one PPBO run on this rank: the growing GP model (rank 0) and the growing
    weight-space model (the rank that runs the weight-space fit)."""

    def __init__(self, kernel, theta, D, m, Q_cap, dev, W, b, shard=None, fit_iters=100, tol=1e-8):
        shard = shard or Shard()
        rff_rank = 1 if (CONCURRENT_FITS and shard.world > 1) else 0
        self.gp = GPState(kernel, theta, D, m, Q_cap, dev, max_iter=fit_iters, tol=tol) if shard.rank == 0 else None
        self.rff = RFFState(W, b, theta, m, Q_cap, max_iter=fit_iters, tol=tol) if shard.rank == rff_rank else None
        self.Q, self.m = 0, m
        self.X_cap = torch.empty((Q_cap * (m + 1), D), dtype=F64, device=dev)       # the design, on every rank (mu* slices)

    def design(self, Q):
        return self.X_cap[:Q * (self.m + 1)]


def run_iteration(d, kernel, theta, Q, m, S, shard=None, seed=0, fit_iters=100, tol=1e-8, timers=None, state=None, shares=None,
                  factor_at_mode=False, shard_mustar=None, weight_covariance="diag"):
    """d: dict of device tensors (IterationInputs.to_device).  Returns (sums [B,3] device, gp, rff).
    Rank 0 fits; the others receive (omega_MAP, hess_diag, mu*) by broadcast while they compute the grid features.
    tol: both Newton iterations stop when the last full step is below tol relative to the iterate.  The chord steps contract
    by ~5x per step, so the distance to the mode is ~tol/4 = 2.5e-9 at the default: 400x inside the 1e-6 parity bound of
    BASELINE.json and far below the reference's own stopping rule (|grad T| < 1e-4, src/gp_model.py:382).
    state: an IterationState makes the models persistent: the first call fits from scratch into its capacity buffers (d["X"]),
    later calls APPEND the comparison sets d["block"] (Q is the new total) and refit from the previous modes.
    shares: sample share per rank (plan_shares); default: rank 0 of several takes none.
    factor_at_mode: also produce the Cholesky factor at the GP mode (only prediction with covariance needs it).
    shard_mustar: split the mu* candidates over the ranks (alpha by broadcast, one all-reduce(max)).  Pays when the other ranks are
    idle by the time the GP fit ends (default: 3 or more ranks and a cold fit); when they are still sampling, rank 0 would wait for
    them inside the collective.
    weight_covariance: "diag" (the reference's) or "full" (WEIGHT_COVARIANCES): the rank that fits the weight space also factors the
    exact Hessian at omega_MAP and sends the factor with (omega_MAP, hess_diag); the draws are standard normals and every sampling
    rank transforms its grid features once (rff_transform_grids)."""
    if weight_covariance not in WEIGHT_COVARIANCES:
        raise PPBOError("weight_covariance must be one of %s" % (WEIGHT_COVARIANCES,))
    full = weight_covariance == "full"
    shard = shard or Shard()
    W, b, grids = d["W"], d["b"], d["grids"]
    dev = W.device
    Fdim = W.shape[0]
    B, P, D = grids.shape
    warm = state is not None and state.Q > 0
    if shard_mustar is None:
        shard_mustar = shard.world >= 3 and not warm
    X = None if warm else d["X"]
    block = d["block"] if warm else None
    if state is not None:
        if warm:
            state.X_cap[state.Q * (m + 1):Q * (m + 1)].copy_(block)
        else:
            state.X_cap[:Q * (m + 1)].copy_(X)

    def mark(name):
        if timers is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            timers.append((name, ev))

    def fit_gp():
        if state is None:
            return gp_fit(X, kernel, theta, Q, m, f_init=d.get("f_init"), max_iter=fit_iters, tol=tol, factor_at_mode=factor_at_mode)
        if warm:
            return state.gp.append(block, factor_at_mode=factor_at_mode)
        return state.gp.cold(X, f_init=d.get("f_init"), factor_at_mode=factor_at_mode)

    def fit_rff():
        if state is None:
            r = rff_fit(X, W, b, theta, Q, m, omega0=d.get("omega0"), max_iter=fit_iters, tol=tol)
            return rff_full_factor(r, Q, m, theta[0]) if full else r
        r = state.rff.append(block) if warm else state.rff.cold(X, omega0=d.get("omega0"))
        return state.rff.hessian_factor() if full else r

    def mu_star(gp, cand):
        """max posterior mean over the design rows and the candidate points; with >= 3 ranks every rank takes a slice of the
        candidates (alpha travels by broadcast) and one all-reduce(max) follows"""
        if not shard_mustar:
            return mustar_over_candidates(gp, cand) if shard.rank == 0 else None
        Qn = Q
        N = Qn * (m + 1)
        pack_a = torch.empty(N + 1, dtype=F64, device=dev)          # alpha and max f_MAP
        if shard.rank == 0:
            pack_a[:N].copy_(gp.alpha)
            ops.vec_max(gp.f_map, out=pack_a[N:])
        shard.broadcast(pack_a, src=0)
        lo_c, hi_c = shard.bounds(cand.shape[0])
        out = pack_a[N:].clone()
        if hi_c > lo_c:
            Xd = state.design(Q) if state is not None else X
            mu = ops.posterior_mean(kernel, Xd, theta[1], theta[2], pack_a[:N], cand[lo_c:hi_c])
            ops.vec_max(mu, out=out, accumulate=True)
        shard.all_reduce_max(out)
        return out
    mark("start")
    lo, hi = shard.sample_bounds(S, shares)
    # The grid features (and their digit planes) do not depend on the fit.  On the rank that runs the latency-bound GP fit they
    # go to the side stream and fill SMs the fit leaves idle; the other ranks compute them while they wait for the broadcast.
    main = torch.cuda.current_stream()
    grid_stream = _side_stream(dev, tag="grid") if shard.rank == 0 else main
    if grid_stream is not main:
        grid_stream.wait_stream(main)
    PhiT = normals = None
    i8 = hi > lo and sampling_engine(hi - lo, P, Fdim) == "i8"
    with torch.cuda.stream(grid_stream):
        if hi > lo:                                           # a rank without samples (rank 0 of several) needs no grid features
            PhiT = rff_grid_features(W, b, theta[2], grids)
            if full:
                # the draws of the full covariance are plain standard normals: cut into digit planes before any fit ends; the grid
                # features are sliced after their transform by the Hessian factor
                normals = rff_prepare_normals(Fdim, lo, hi, P, dev, seed=seed)
            elif i8:
                PhiT = SlicedGrids(PhiT)                      # digit planes of the grid features
    mark("grid_features")

    def grid_tensors():
        if PhiT is None:
            return ()
        out = (PhiT.PhiT, PhiT.planes, PhiT.scale) if isinstance(PhiT, SlicedGrids) else (PhiT,)
        if isinstance(normals, SlicedSamples):
            out += (normals.planes, normals.scale)
        elif normals is not None:
            out += (normals,)
        return out
    pack = torch.empty(2 * Fdim + 1, dtype=F64, device=dev)
    gp = rff = prepared = None
    cand = grids.reshape(B * P, D)
    rff_rank = 1 if (CONCURRENT_FITS and shard.world > 1) else 0      # with more than one GPU the two fits run on two of them
    if shard.rank == 0 and CONCURRENT_FITS and shard.world == 1 and OVERLAP_SAMPLING and i8:
        # One GPU, INT8 engine.  Two chains that only share X:
        #   A  GP fit -> mu*                                   latency-bound, short (8.7 ms cold / 5 ms appended when alone)
        #   B  weight-space fit -> draws -> contraction        the contraction alone keeps every tensor pipe busy for ~9 ms
        # B is the longer one and its head (the weight-space fit) is as latency-bound as A, so B runs in the FOREGROUND (this
        # thread, streams above the default priority) and A on the persistent background thread whose streams all sit at the
        # lowest priority; the contraction's persistent grid leaves OVERLAP_RESERVED_SMS SMs free, where A finishes while the
        # tensor pipes of the other SMs are busy.  Only the reduction (3 B sums) needs both chains.
        bg = _side_stream(dev)
        bg.wait_stream(main)
        fg = _side_stream(dev, priority=GP_STREAM_PRIORITY, tag="gp") if GP_STREAM_PRIORITY else main
        if fg is not main:
            fg.wait_stream(main)

        def gp_chain():
            torch.cuda.set_device(dev)
            with torch.cuda.stream(bg):
                g = fit_gp()
                return g, mustar_over_candidates(g, cand)
        fut = _background_worker().submit(gp_chain)
        lib = ops._lib.load()
        fmax = None
        try:
            with torch.cuda.stream(fg):
                rff = fit_rff()
                mark("rff_fit")
                fit_done = torch.cuda.Event()
                fit_done.record(fg)
                transformed = None
                if full:
                    fg.wait_stream(grid_stream)
                    for t in grid_tensors():
                        t.record_stream(fg)
                    prepared = normals
                    transformed = rff_transform_grids(rff, PhiT, slices=SAMPLING_SLICES)
                    mark("grid_transform")
                else:
                    prepared = rff_prepare_samples(rff, lo, hi, P, seed=seed)
                    fg.wait_stream(grid_stream)
                    for t in grid_tensors():
                        t.record_stream(fg)
                lib.ppbo_set_tuning(14, OVERLAP_RESERVED_SMS if warm else OVERLAP_RESERVED_SMS_COLD)
                try:
                    fmax, _ = rff_sampled_maxima(rff, PhiT, lo, hi, seed=seed, prepared=prepared, covariance=weight_covariance,
                                                 transformed=transformed)
                finally:
                    lib.ppbo_set_tuning(14, 0)
                mark("sampling")
            if warm and REFRESH_RFF_FACTOR:
                # while the contraction runs: the weight-space Hessian factor at the new optimum, for the NEXT iteration's fit
                # (lowest priority, on the SMs the contraction leaves free; it only waits for this iteration's fit)
                rf = _side_stream(dev, tag="rff_refresh")
                rf.wait_event(fit_done)
                rff.omega_map.record_stream(rf)
                with torch.cuda.stream(rf):
                    state.rff.refresh_factor()
        finally:
            gp, mustar = fut.result()          # re-raises on this thread
        main.wait_stream(bg)
        for t in (gp.Sigma, gp.lap.G, gp.lap._Lfac, gp.lap.f_map, gp.lap.alpha, gp.lap.arrow, mustar):
            t.record_stream(main)
        if fg is not main:
            main.wait_stream(fg)
            for t in (rff.omega_map, rff.hess_diag, rff.Phi_X, fmax) + ((rff.L,) if full else ()):
                t.record_stream(main)
        mark("gp_tail")                        # what is left of the GP fit + mu* after the contraction has finished
        sums = rff_reduce(fmax, mustar, B, shard)
        mark("acquisition")
        if state is not None:
            state.Q = Q
        return sums, gp, rff
    if shard.rank == 0 and CONCURRENT_FITS and shard.world == 1:
        # (FP64 engine / PPBO_OVERLAP_SAMPLING=0.)  GP fit: foreground, on a stream one priority level above the default;
        # weight-space fit: a persistent background host thread whose streams all sit at the lowest priority, so it only takes the
        # SMs the GP fit leaves idle.
        side = _side_stream(dev)
        side.wait_stream(main)
        gp_stream = _side_stream(dev, priority=GP_STREAM_PRIORITY, tag="gp") if GP_STREAM_PRIORITY else main
        if gp_stream is not main:
            gp_stream.wait_stream(main)

        def weight_space_fit():
            torch.cuda.set_device(dev)
            with torch.cuda.stream(side):
                fit = fit_rff()
                # the draws and their digit planes need this fit only: done here, behind the GP fit (the standard normals of the
                # full covariance are already on the grid stream)
                return fit, (normals if full else rff_prepare_samples(fit, lo, hi, P, seed=seed))
        fut = _background_worker().submit(weight_space_fit)
        try:
            with torch.cuda.stream(gp_stream):
                gp = fit_gp()
                mark("gp_fit")
                mustar = mustar_over_candidates(gp, cand)
                mark("mustar")
        finally:
            rff, prepared = fut.result()       # re-raises on this thread
        if gp_stream is not main:
            main.wait_stream(gp_stream)
            for t in (gp.Sigma, gp.lap.G, gp.lap._Lfac, gp.lap.f_map, gp.lap.alpha, gp.lap.arrow, mustar):
                t.record_stream(main)
        main.wait_stream(side)
        for t in (rff.omega_map, rff.hess_diag, rff.Phi_X) + ((prepared.planes, prepared.scale) if isinstance(prepared, SlicedSamples)
                                                              else ((prepared,) if prepared is not None else ())) + \
                ((rff.L,) if full else ()):
            t.record_stream(main)
        mark("rff_fit")                        # what is left of the weight-space fit after the GP fit has finished
    elif shard.world > 1 and CONCURRENT_FITS:
        # Several ranks: rank 0 runs the GP fit; rank 1 runs the weight-space fit and broadcasts it; every rank with a sample share
        # draws and evaluates its samples as soon as the weight-space fit has arrived (the contraction needs that fit only) --
        # rank 0 after its GP fit; when mu* is known only the reduction and the all-reduce of 3 B doubles are left.
        pack_rff, mu_t = pack[:2 * Fdim], pack[2 * Fdim:]
        fmax = None
        Lbuf = ops.rff_hessian_factor_buffer(Fdim, dev) if full and shard.rank != rff_rank else None
        if shard.rank == 0:
            bstream = _side_stream(dev, tag="bcast")     # rank 0 joins the first broadcast off its critical path
            bstream.wait_stream(main)
            pack.record_stream(bstream)
            with torch.cuda.stream(bstream):
                shard.broadcast(pack_rff, src=rff_rank)
                if full:
                    Lbuf.record_stream(bstream)
                    shard.broadcast(Lbuf, src=rff_rank)
            gp = fit_gp()
            mark("gp_fit")
            main.wait_stream(bstream)
        else:
            if shard.rank == rff_rank:
                rff = fit_rff()
                mark("rff_fit")
                pack_rff[:Fdim].copy_(rff.omega_map)
                pack_rff[Fdim:].copy_(rff.hess_diag)
                Lbuf = rff.L
            shard.broadcast(pack_rff, src=rff_rank)
            if full:
                shard.broadcast(Lbuf, src=rff_rank)
            mark("rff_received")
        if rff is None:
            rff = RFFFit()
            rff.W, rff.b, rff.sigma_f, rff.Phi_X, rff.stats = W, b, float(theta[2]), None, None
        rff.omega_map, rff.hess_diag, rff.L = pack_rff[:Fdim], pack_rff[Fdim:], Lbuf
        if shard.rank != 0 and hi > lo:
            fmax, _ = rff_sampled_maxima(rff, PhiT, lo, hi, seed=seed, prepared=normals, covariance=weight_covariance)
            mark("sampling")
        if shard_mustar:
            mustar = mu_star(gp, cand)
            mu_t.copy_(mustar)
        else:
            if shard.rank == 0:
                mu_t.copy_(mustar_over_candidates(gp, cand))
            shard.broadcast(mu_t, src=0)
        mark("mustar")
        if shard.rank == 0 and hi > lo:
            if grid_stream is not main:
                main.wait_stream(grid_stream)
                for t in grid_tensors():
                    t.record_stream(main)
            fmax, _ = rff_sampled_maxima(rff, PhiT, lo, hi, seed=seed, prepared=normals, covariance=weight_covariance)
            mark("sampling")
        sums = rff_reduce(fmax, mu_t, B, shard)
        mark("acquisition")
        if state is not None:
            state.Q = Q
        return sums, gp, rff
    else:
        if shard.rank == 0:
            gp = fit_gp()
            mark("gp_fit")
            mustar = mustar_over_candidates(gp, cand)
            mark("mustar")
        if shard.rank == rff_rank:
            rff = fit_rff()
            mark("rff_fit")
    if shard.rank == rff_rank:
        pack[:Fdim].copy_(rff.omega_map)
        pack[Fdim:2 * Fdim].copy_(rff.hess_diag)
    if shard.rank == 0:
        pack[2 * Fdim:].copy_(mustar)
    if rff_rank == 0:
        shard.broadcast(pack, src=0)
    else:
        shard.broadcast(pack[:2 * Fdim], src=rff_rank)
        shard.broadcast(pack[2 * Fdim:], src=0)
    Lbuf = None
    if full:
        Lbuf = rff.L if shard.rank == rff_rank else ops.rff_hessian_factor_buffer(Fdim, dev)
        shard.broadcast(Lbuf, src=rff_rank)
        prepared = normals
    if rff is None:
        rff = RFFFit()
        rff.W, rff.b, rff.sigma_f, rff.Phi_X, rff.stats = W, b, float(theta[2]), None, None
    rff.omega_map, rff.hess_diag, rff.L = pack[:Fdim], pack[Fdim:2 * Fdim], Lbuf
    if grid_stream is not main:
        main.wait_stream(grid_stream)
        for t in grid_tensors():
            t.record_stream(main)
    sums, fmax, arg = rff_acquisition(rff, PhiT, S, pack[2 * Fdim:], shard=shard, seed=seed, bounds=(lo, hi), prepared=prepared,
                                      n_grids=B, covariance=weight_covariance)
    mark("acquisition")
    if state is not None:
        state.Q = Q
    return sums, gp, rff
