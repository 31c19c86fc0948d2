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
products (omega_MAP, hess_diag, mu*: 8(2F+1) bytes, 8(2F+D+1) with the x* of an incumbent); every rank draws its own slice of the counter-based normal stream,
evaluates its S/R samples on all B grids and one all-reduce(sum) of the 3B partial sums follows.
"""
import threading

import numpy as np
import torch

from . import ops
from ._lib import PPBOError
from .spectral import periodic_mask

F64 = torch.float64
SHRINKAGE = 1e-6          # GPModel.COVARIANCE_SHRINKAGE, src/gp_model.py:26
# Sampling contraction Omega . PhiT^T (sampling_engine): "i8" = tcgen05 INT8 tensor pipe with error-free splitting into
# SAMPLING_SLICES base-256 digit planes per operand (csrc/ozaki.cu; 6 planes: ~1e-13 relative, i.e. the accuracy of an FP64 GEMM
# of this depth), "f64" = the FP64 DMMA kernel.  Small contractions (reference-size grids) stay on the FP64 kernel: a 128 x 64
# INT8 tile would be mostly padding there.
SAMPLING_SLICES = 6
I8_MIN_WORK = 1 << 24     # S * P * F below which the FP64 kernel is used
# Covariance of the weight-space Laplace posterior the draws come from: "diag" = the reference's 1 / -hess_diag
# (src/random_fourier_sampler.py:134-137), "full" = the inverse of the exact Hessian I + Psi' diag(a) Psi (opt-in).  With "full" the
# draws stay standard normals z_s and the covariance moves into the grid operand: f_s(x_p) = mu_p + z_s . Phi~_p with
# mu_p = phi(x_p)' omega_MAP and Phi~ = Phi L^-T, H = L L'.
WEIGHT_COVARIANCES = ("diag", "full")


# One GPU: the sampling contraction needs the weight-space fit only (mu* enters at the reduction), so the weight-space fit, the
# draws and the INT8 contraction run in the foreground WHILE the GP fit -- a chain of small, latency-bound kernels that leaves most
# SMs idle -- runs beside them on the background thread.  The contraction's persistent grid then leaves OVERLAP_RESERVED_SMS(_COLD)
# SMs to the GP fit (tuning key 14); a contraction CTA fills its SM, so the two never share one.  OVERLAP_SAMPLING = False runs the
# contraction after both fits instead: the same bits, which makes that order the reference of the overlapped one.
OVERLAP_SAMPLING = True
# Reserved SMs: an appended iteration's GP chain is short (it still ends before the contraction on 8 SMs); a cold fit has 13
# chord steps with one 100 MB half-triangle mat-vec of G each plus the factorisation and is the longer chain, so it gets more
# (sweeps in DESIGN.md 5.1).
OVERLAP_RESERVED_SMS = 12            # appended iterations
OVERLAP_RESERVED_SMS_COLD = 24       # cold iterations


def sampling_engine(S, P, Fdim):
    return "i8" if S * P * Fdim >= I8_MIN_WORK else "f64"


def _fused_draw(Fdim):
    """whether the draws and their digit planes fit one kernel: it holds 8 rows of F doubles in at most 200 KB of shared memory"""
    return Fdim * 64 <= 200 * 1024


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


# Starts of the continuous mu* search: the MUSTAR_STARTS design rows with the largest f_MAP (DESIGN.md 7 item 16 and
# profiles/r04_mustar_ascent_probe.txt for the choice), plus the best candidate of this iteration's lines and the previous x*.
MUSTAR_STARTS = 128


def mustar_starts(f_map, X, cand_mu=None, candidates=None, n_starts=MUSTAR_STARTS, prev=None):
    """Starts [R, D] of mustar_ascent: the n_starts rows of X with the largest f_map (stable descending sort: the lowest index
    first among equal values), the candidate with the largest posterior mean cand_mu (the first one on ties) and prev (the last
    x*), in this order.  Device or host tensors alike."""
    order = torch.sort(f_map, descending=True, stable=True).indices[:min(n_starts, X.shape[0])]
    parts = [X[order]]
    if candidates is not None and candidates.shape[0] > 0:
        parts.append(candidates[torch.argmax(cand_mu)].view(1, -1))
    if prev is not None:
        parts.append(prev.reshape(1, -1).to(X.dtype))
    return torch.cat(parts)


def mustar_ascent(g, candidates=None, n_starts=MUSTAR_STARTS, prev=None, max_iter=ops.MU_MAXIMIZE_MAX_ITER, gtol=ops.MU_MAXIMIZE_GTOL):
    """Continuous mu* and x* of the GP fit g on the device: multi-start ascent of the posterior mean (ops.mu_maximize) from
    mustar_starts.  Returns (mu* [1], x* [D], the end point of every start [R, D]); mu* = mu(x*) as the ascent kernel evaluates
    it (the reference's GPModel.mu_star returns mu_pred(xstar) as well).  No synchronisation."""
    cand_mu = posterior_mean(g, candidates) if candidates is not None and candidates.shape[0] > 0 else None
    X0 = mustar_starts(g.f_map, g.X, cand_mu, candidates, n_starts, prev)
    xbest, fbest, xout, _, _, _ = ops.mu_maximize(g.kernel, g.X, g.lengthscales, g.theta[2], g.alpha, X0, max_iter=max_iter, gtol=gtol,
                                                  periodic_mask=periodic_mask(g.kernel))
    return fbest, xbest, xout


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

    def cold(self, X, omega0=None):
        Q = X.shape[0] // (self.m + 1)
        ops.rff_features(self.W, self.b, X, self.theta[2], True, out=self.Phi_cap[:, :X.shape[0]])
        return self._fit(Q, omega0)

    def append(self, X_block):
        if self.Q == 0:
            return self.cold(X_block)
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
    if Z is None and i8 and _fused_draw(Fdim):
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
    if Z is None and sampling_engine(hi - lo, P, Fdim) == "i8" and _fused_draw(Fdim):
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


def select_batch(fmax, mustar_dev, q, n_grids, shard=None):
    """q query lines by greedy joint expected improvement over the draws behind fmax [B, S_loc] (this rank's samples; None on a
    rank without samples): step k adds the line that raises E_s[max(max_{b in chosen} fmax[b][s] - mu*, 0)] most, lowest index on
    ties.  The maxima of all lines in one sample come from the same sampled function, so a line that reaches the same peak as a
    chosen one adds nothing.  Returns (idx [q] int32, qei [q]) on the device, qei[k] = the joint EI of the first k+1 picks.
    With several ranks every step's gains go through one all-reduce of B + 1 doubles (the last one counts the samples), so all
    ranks pick the same lines; every rank joins every collective."""
    shard = shard or Shard()
    if not 1 <= q <= n_grids:
        raise PPBOError("batch size q must be in [1, %d], not %r" % (n_grids, q))
    dev = mustar_dev.device
    idx = torch.empty(q, dtype=torch.int32, device=dev)
    qei = torch.empty(q, dtype=F64, device=dev)
    gain = torch.zeros(n_grids + 1, dtype=F64, device=dev)
    cur = None if fmax is None else torch.empty(fmax.shape[1], dtype=F64, device=dev)
    for k in range(q):
        if fmax is not None:
            ops.acq_batch_gain(fmax, mustar_dev, cur, k, q, out=gain)
        shard.all_reduce_sum(gain)
        ops.acq_batch_pick(gain, fmax, k, q, idx, qei, cur)
        if fmax is None:
            gain.zero_()                 # this rank's share of the next step's sums
    return idx, qei


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
# The foreground chain of the one-GPU schedules goes to a stream one level above the default priority, where this thread's
# Cholesky bulk (library-internal side stream) sits too; the background thread keeps the default (lowest) priority for everything
# (ppbo_set_thread_background), so its chain only fills the SMs the foreground leaves idle.
FOREGROUND_PRIORITY = -1
_WORKER = None


def _background_worker():
    """One persistent host thread for the chain beside the foreground one (the library keeps per-thread streams: a fresh thread per
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


def _join(dst, src, tensors):
    """dst waits for the work queued on src so far; the tensors src made stay allocated until dst's work on them is done"""
    dst.wait_stream(src)
    for t in tensors:
        t.record_stream(dst)


def _device_tensors(*parts):
    """the tensors behind grid features and prepared draws (SlicedGrids, SlicedSamples, a tensor or None)"""
    out = []
    for p in parts:
        if isinstance(p, SlicedGrids):
            out += [p.PhiT, p.planes, p.scale]
        elif isinstance(p, SlicedSamples):
            out += [p.planes, p.scale]
        elif p is not None:
            out.append(p)
    return out


def _gp_tensors(gp):
    return [gp.Sigma, gp.lap.G, gp.lap._Lfac, gp.lap.f_map, gp.lap.alpha, gp.lap.arrow]


def _rff_tensors(rff):
    return [rff.omega_map, rff.hess_diag, rff.Phi_X] + ([rff.L] if rff.L is not None else [])


def _weight_space_rank(world):
    """the rank that runs the weight-space fit: with more than one GPU the two fits run on two of them"""
    return 1 if world > 1 else 0


class IterationState:
    """What persists between the iterations of one PPBO run on this rank: the growing GP model (rank 0) and the growing
    weight-space model (the rank that runs the weight-space fit)."""

    def __init__(self, kernel, theta, D, m, Q_cap, dev, W, b, shard=None, fit_iters=100, tol=1e-8):
        shard = shard or Shard()
        rff_rank = _weight_space_rank(shard.world)
        self.gp = GPState(kernel, theta, D, m, Q_cap, dev, max_iter=fit_iters, tol=tol) if shard.rank == 0 else None
        self.rff = RFFState(W, b, theta, m, Q_cap, max_iter=fit_iters, tol=tol) if shard.rank == rff_rank else None
        self.Q, self.m = 0, m
        self.X_cap = torch.empty((Q_cap * (m + 1), D), dtype=F64, device=dev)       # the design, on every rank (mu* slices)
        self.xstar = None            # x* of the last iteration run with an incumbent: one more start of the next search

    def design(self, Q):
        return self.X_cap[:Q * (self.m + 1)]


class _Iteration:
    """One call of run_iteration: its arguments and what follows from them, the two fits and the timer marks."""

    def __init__(self, d, kernel, theta, Q, m, S, shard, seed, fit_iters, tol, timers, state, shares, factor_at_mode, shard_mustar,
                 weight_covariance, incumbent):
        self.d, self.kernel, self.theta, self.Q, self.m, self.S, self.seed = d, kernel, theta, Q, m, S, seed
        self.shard, self.fit_iters, self.tol, self.timers, self.state = shard, fit_iters, tol, timers, state
        self.factor_at_mode, self.covariance, self.full = factor_at_mode, weight_covariance, weight_covariance == "full"
        self.W, self.b, self.grids = d["W"], d["b"], d["grids"]
        self.dev, self.Fdim = self.W.device, self.W.shape[0]
        self.B, self.P, D = self.grids.shape
        self.cand = self.grids.reshape(self.B * self.P, D)
        self.warm = state is not None and state.Q > 0
        self.X = None if self.warm else d["X"]
        self.block = d["block"] if self.warm else None
        self.incumbent = incumbent
        if shard_mustar is None:
            shard_mustar = shard.world >= 3 and not self.warm and incumbent is None
        self.shard_mustar = shard_mustar
        self.lo, self.hi = shard.sample_bounds(S, shares)
        self.i8 = self.hi > self.lo and sampling_engine(self.hi - self.lo, self.P, self.Fdim) == "i8"

    def mark(self, name):
        """timing event on the current stream"""
        if self.timers is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.timers.append((name, ev))

    def fit_gp(self):
        if self.state is None:
            return gp_fit(self.X, self.kernel, self.theta, self.Q, self.m, f_init=self.d.get("f_init"), max_iter=self.fit_iters,
                          tol=self.tol, factor_at_mode=self.factor_at_mode)
        if self.warm:
            return self.state.gp.append(self.block, factor_at_mode=self.factor_at_mode)
        return self.state.gp.cold(self.X, f_init=self.d.get("f_init"), factor_at_mode=self.factor_at_mode)

    def mustar(self, g):
        """mu* of the GP fit g on the device: the discrete stand-in (1 double), or with an incumbent the continuous search, written
        into the incumbent (mu*, x*: 1 + D doubles, which the reductions read as mu* through its first element)"""
        if self.incumbent is None:
            return mustar_over_candidates(g, self.cand)
        prev = self.state.xstar if self.warm else None
        mu, x, _ = mustar_ascent(g, self.cand, prev=prev)
        self.incumbent[:1].copy_(mu)
        self.incumbent[1:].copy_(x)
        return self.incumbent

    def fit_rff(self):
        if self.state is None:
            r = rff_fit(self.X, self.W, self.b, self.theta, self.Q, self.m, omega0=self.d.get("omega0"), max_iter=self.fit_iters,
                        tol=self.tol)
            return rff_full_factor(r, self.Q, self.m, self.theta[0]) if self.full else r
        st = self.state.rff
        r = st.append(self.block) if self.warm else st.cold(self.X, omega0=self.d.get("omega0"))
        return st.hessian_factor() if self.full else r


def run_iteration(d, kernel, theta, Q, m, S, shard=None, seed=0, fit_iters=100, tol=1e-8, timers=None, state=None, shares=None,
                  factor_at_mode=False, shard_mustar=None, weight_covariance="diag", batch=None, incumbent=None):
    """d: dict of device tensors (IterationInputs.to_device).  Returns (sums [B,3] device, gp, rff); with batch=q also the q query
    lines chosen by greedy joint expected improvement over the same draws (select_batch): (sums, gp, rff, (idx [q], qei [q])).
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
    rank transforms its grid features once (rff_transform_grids).
    timers: a list that receives (name, CUDA event) marks between the stages of the schedule that ran.
    batch: q >= 1 keeps this rank's per-sample maxima and runs the greedy selection after the reduction on every rank (inside the
    "acquisition" stage); without it nothing of the result changes.
    incumbent: a float64 device tensor of D + 1 elements turns on the continuous mu* search (mustar_ascent, on rank 0 right after
    the GP fit) in place of the discrete stand-in mustar_over_candidates: the EI sums and the batch selection use its mu*, and
    every rank's incumbent receives (mu*, x*).  With a state, x* is kept there and starts the next appended iteration's search.
    Not with shard_mustar=True.  incumbent=None changes nothing."""
    if weight_covariance not in WEIGHT_COVARIANCES:
        raise PPBOError("weight_covariance must be one of %s" % (WEIGHT_COVARIANCES,))
    if batch is not None and not 1 <= batch <= d["grids"].shape[0]:
        raise PPBOError("batch must be in [1, %d], not %r" % (d["grids"].shape[0], batch))
    if incumbent is not None:
        D = d["grids"].shape[2]
        if not (isinstance(incumbent, torch.Tensor) and incumbent.dtype == F64 and incumbent.is_cuda and incumbent.is_contiguous()
                and incumbent.numel() == D + 1):
            raise PPBOError("incumbent must be a contiguous float64 device tensor of D + 1 = %d elements" % (D + 1))
        if shard_mustar:
            raise PPBOError("the continuous mu* search runs on rank 0: shard_mustar=True cannot be combined with an incumbent")
    it = _Iteration(d, kernel, theta, Q, m, S, shard or Shard(), seed, fit_iters, tol, timers, state, shares, factor_at_mode,
                    shard_mustar, weight_covariance, incumbent)
    if state is not None:
        if it.warm:
            state.X_cap[state.Q * (m + 1):Q * (m + 1)].copy_(it.block)
        else:
            state.X_cap[:Q * (m + 1)].copy_(it.X)
    it.mark("start")
    main = torch.cuda.current_stream()
    grid = _grid_stage(it, main)
    it.mark("grid_features")
    if it.shard.world > 1:
        sums, gp, rff, fmax, mustar = _several_ranks(it, main, grid)
    elif it.i8 and OVERLAP_SAMPLING:
        sums, gp, rff, fmax, mustar = _one_gpu_overlapped(it, main, grid)
    else:
        sums, gp, rff, fmax, mustar = _one_gpu_sequential(it, main, grid)
    picks = select_batch(fmax, mustar, batch, it.B, it.shard) if batch is not None else None
    it.mark("acquisition")
    if state is not None:
        state.Q = Q
        if incumbent is not None:
            state.xstar = incumbent[1:].clone()
    return (sums, gp, rff) if batch is None else (sums, gp, rff, picks)


def _grid_stage(it, main):
    """The grid features (and their digit planes, or the standard normals of the full covariance) of this rank's samples: they do
    not depend on the fit.  On the rank that runs the latency-bound GP fit they go to a side stream and fill SMs the fit leaves
    idle; the other ranks compute them while they wait for the broadcast.
    Returns (stream, PhiT, normals, the tensors a stream that reads them must record)."""
    stream = _side_stream(it.dev, tag="grid") if it.shard.rank == 0 else main
    if stream is not main:
        stream.wait_stream(main)
    PhiT = normals = None
    with torch.cuda.stream(stream):
        if it.hi > it.lo:                                     # a rank without samples (rank 0 of several) needs no grid features
            PhiT = rff_grid_features(it.W, it.b, it.theta[2], it.grids)
            if it.full:
                # the draws of the full covariance are plain standard normals: cut into digit planes before any fit ends; the grid
                # features are sliced after their transform by the Hessian factor
                normals = rff_prepare_normals(it.Fdim, it.lo, it.hi, it.P, it.dev, seed=it.seed)
            elif it.i8:
                PhiT = SlicedGrids(PhiT)                      # digit planes of the grid features
    return stream, PhiT, normals, _device_tensors(PhiT, normals)


def _one_gpu_overlapped(it, main, grid):
    """One GPU, INT8 engine.  Two chains that only share X:
      A  GP fit -> mu*                                   latency-bound, short (8.7 ms cold / 5 ms appended when alone)
      B  weight-space fit -> draws -> contraction        the contraction alone keeps every tensor pipe busy for ~9 ms
    B is the longer one and its head (the weight-space fit) is as latency-bound as A, so B runs in the FOREGROUND (this thread, on a
    stream above the default priority) and A on the persistent background thread whose streams all sit at the lowest priority; the
    contraction's persistent grid leaves OVERLAP_RESERVED_SMS SMs free, where A finishes while the tensor pipes of the other SMs are
    busy.  Only the reduction (3 B sums) needs both chains."""
    grid_stream, PhiT, normals, grid_tensors = grid
    bg = _side_stream(it.dev)
    bg.wait_stream(main)
    fg = _side_stream(it.dev, priority=FOREGROUND_PRIORITY, tag="fg")
    fg.wait_stream(main)

    def gp_chain():
        torch.cuda.set_device(it.dev)
        with torch.cuda.stream(bg):
            g = it.fit_gp()
            return g, it.mustar(g)
    fut = _background_worker().submit(gp_chain)
    lib = ops._lib.load()
    try:
        with torch.cuda.stream(fg):
            rff = it.fit_rff()
            it.mark("rff_fit")
            transformed = None
            if it.full:
                _join(fg, grid_stream, grid_tensors)
                prepared = normals
                transformed = rff_transform_grids(rff, PhiT, slices=SAMPLING_SLICES)
                it.mark("grid_transform")
            else:
                prepared = rff_prepare_samples(rff, it.lo, it.hi, it.P, seed=it.seed)
                _join(fg, grid_stream, grid_tensors)
            lib.ppbo_set_tuning(14, OVERLAP_RESERVED_SMS if it.warm else OVERLAP_RESERVED_SMS_COLD)
            try:
                fmax, _ = rff_sampled_maxima(rff, PhiT, it.lo, it.hi, seed=it.seed, prepared=prepared, covariance=it.covariance,
                                             transformed=transformed)
            finally:
                lib.ppbo_set_tuning(14, 0)
            it.mark("sampling")
    finally:
        gp, mustar = fut.result()          # re-raises on this thread
    _join(main, bg, _gp_tensors(gp) + [mustar])
    _join(main, fg, _rff_tensors(rff) + [fmax])
    it.mark("gp_tail")                     # what is left of the GP fit + mu* after the contraction has finished
    return rff_reduce(fmax, mustar, it.B, it.shard), gp, rff, fmax, mustar


def _one_gpu_sequential(it, main, grid):
    """One GPU, FP64 engine (or OVERLAP_SAMPLING off): the two fits only share X and are both chains of small, latency-bound launches
    with one host decision per Newton step.  The GP fit runs in the foreground; the weight-space fit and its draws on the
    background thread, whose streams all sit at the lowest priority, so they only take the SMs the GP fit leaves idle.  The
    weight-space fit then starts from omega = 0 (or the caller's omega0) instead of the projection of the GP mode, which costs one
    extra Newton step (20 against 19 on the Ackley-20D bench problem).  The contraction follows both fits."""
    grid_stream, PhiT, normals, grid_tensors = grid
    side = _side_stream(it.dev)
    side.wait_stream(main)
    fg = _side_stream(it.dev, priority=FOREGROUND_PRIORITY, tag="fg")
    fg.wait_stream(main)

    def weight_space_fit():
        torch.cuda.set_device(it.dev)
        with torch.cuda.stream(side):
            fit = it.fit_rff()
            # the draws and their digit planes need this fit only: done here, behind the GP fit (the standard normals of the
            # full covariance are already on the grid stream)
            return fit, (normals if it.full else rff_prepare_samples(fit, it.lo, it.hi, it.P, seed=it.seed))
    fut = _background_worker().submit(weight_space_fit)
    try:
        with torch.cuda.stream(fg):
            gp = it.fit_gp()
            it.mark("gp_fit")
            mustar = it.mustar(gp)
            it.mark("mustar")
    finally:
        rff, prepared = fut.result()       # re-raises on this thread
    _join(main, fg, _gp_tensors(gp) + [mustar])
    _join(main, side, _rff_tensors(rff) + _device_tensors(prepared))
    it.mark("rff_fit")                     # what is left of the weight-space fit after the GP fit has finished
    _join(main, grid_stream, grid_tensors)
    sums, fmax, _ = rff_acquisition(rff, PhiT, it.S, mustar, shard=it.shard, seed=it.seed, bounds=(it.lo, it.hi), prepared=prepared,
                                    n_grids=it.B, covariance=it.covariance)
    return sums, gp, rff, fmax, mustar


def _several_ranks(it, main, grid):
    """Several ranks: rank 0 runs the GP fit; rank 1 runs the weight-space fit and broadcasts it; every rank with a sample share
    draws and evaluates its samples as soon as the weight-space fit has arrived (the contraction needs that fit only) -- rank 0
    after its GP fit; when mu* is known only the reduction and the all-reduce of 3 B doubles are left."""
    grid_stream, PhiT, normals, grid_tensors = grid
    shard, Fdim, full = it.shard, it.Fdim, it.full
    rff_rank = _weight_space_rank(shard.world)
    pack = torch.empty(2 * Fdim + (1 if it.incumbent is None else it.incumbent.numel()), dtype=F64, device=it.dev)
    pack_rff, mu_t = pack[:2 * Fdim], pack[2 * Fdim:]
    gp = rff = fmax = None
    Lbuf = ops.rff_hessian_factor_buffer(Fdim, it.dev) if full and shard.rank != rff_rank else None
    if shard.rank == 0:
        bstream = _side_stream(it.dev, tag="bcast")     # rank 0 joins the first broadcast off its critical path
        bstream.wait_stream(main)
        pack.record_stream(bstream)
        with torch.cuda.stream(bstream):
            shard.broadcast(pack_rff, src=rff_rank)
            if full:
                Lbuf.record_stream(bstream)
                shard.broadcast(Lbuf, src=rff_rank)
        gp = it.fit_gp()
        it.mark("gp_fit")
        main.wait_stream(bstream)
    else:
        if shard.rank == rff_rank:
            rff = it.fit_rff()
            it.mark("rff_fit")
            pack_rff[:Fdim].copy_(rff.omega_map)
            pack_rff[Fdim:].copy_(rff.hess_diag)
            Lbuf = rff.L
        shard.broadcast(pack_rff, src=rff_rank)
        if full:
            shard.broadcast(Lbuf, src=rff_rank)
        it.mark("rff_received")
    if rff is None:                                     # the weight-space fit as received: no features of the design, no statistics
        rff = RFFFit()
        rff.W, rff.b, rff.sigma_f, rff.Phi_X, rff.stats = it.W, it.b, float(it.theta[2]), None, None
    rff.omega_map, rff.hess_diag, rff.L = pack_rff[:Fdim], pack_rff[Fdim:], Lbuf
    if shard.rank != 0 and it.hi > it.lo:
        fmax, _ = rff_sampled_maxima(rff, PhiT, it.lo, it.hi, seed=it.seed, prepared=normals, covariance=it.covariance)
        it.mark("sampling")
    if it.shard_mustar:
        mu_t.copy_(_sharded_mustar(it, gp))
    else:
        if shard.rank == 0:
            mu_t.copy_(it.mustar(gp))
        shard.broadcast(mu_t, src=0)
        if it.incumbent is not None and shard.rank != 0:
            it.incumbent.copy_(mu_t)
    it.mark("mustar")
    if shard.rank == 0 and it.hi > it.lo:
        _join(main, grid_stream, grid_tensors)
        fmax, _ = rff_sampled_maxima(rff, PhiT, it.lo, it.hi, seed=it.seed, prepared=normals, covariance=it.covariance)
        it.mark("sampling")
    return rff_reduce(fmax, mu_t, it.B, shard), gp, rff, fmax, mu_t


def _sharded_mustar(it, gp):
    """max posterior mean over the design rows and the candidate points, every rank taking a slice of the candidates: alpha and
    max f_MAP travel by broadcast from rank 0 and one all-reduce(max) follows"""
    shard, N = it.shard, it.Q * (it.m + 1)
    pack_a = torch.empty(N + 1, dtype=F64, device=it.dev)          # alpha and max f_MAP
    if shard.rank == 0:
        pack_a[:N].copy_(gp.alpha)
        ops.vec_max(gp.f_map, out=pack_a[N:])
    shard.broadcast(pack_a, src=0)
    lo_c, hi_c = shard.bounds(it.cand.shape[0])
    out = pack_a[N:].clone()
    if hi_c > lo_c:
        Xd = it.state.design(it.Q) if it.state is not None else it.X
        mu = ops.posterior_mean(it.kernel, Xd, it.theta[1], it.theta[2], pack_a[:N], it.cand[lo_c:hi_c])
        ops.vec_max(mu, out=out, accumulate=True)
    shard.all_reduce_max(out)
    return out
