"""Next-query selection -- host-side mirror of the reference's src/acquisition.py (same function names and signatures).

The Monte-Carlo acquisition values (EI, varmax) are evaluated on the GPU, all candidate (xi, x) pairs of a strategy in ONE
batched pass: posterior mean/covariance on every projected xi-grid (ppbo_predict), S draws per grid as a GEMM with a fused
per-sample max (ppbo_mvn_rowmax), fixed-order reductions (ppbo_acq_reduce).  Everything random is still drawn from the
global legacy numpy RNG on the host in exactly the order the reference consumes it (grid jitter, then S x 70 standard
normals, per candidate), so a seeded run selects the same query as the reference.

Sampling factor: numpy's legacy multivariate_normal draws x = mu + z . (sqrt(s) * V) with (u, s, V) = svd(cov).  With
`mvn_factor='svd-host'` (default) that 70 x 70 factor is formed by the same LAPACK call on the host from the device-computed
covariance -- the only way to reproduce the reference's draws from the same z, since the factor's sign/rotation convention is
LAPACK's.  `mvn_factor='device'` uses a Cholesky factor computed on the GPU instead (same distribution, different draws).
"""
import os
import sys
import time

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

from ppbo_b200 import ops  # noqa: E402

GRID_POINTS = 70          # hard-coded in the reference (src/acquisition.py:73,171)


# ------------------------------------------------------------------------------------------------ batched MC engine
try:
    from threadpoolctl import ThreadpoolController as _ThreadpoolController
except Exception:        # pragma: no cover
    _ThreadpoolController = None
_blas_controller = None


def _svd_factor(cov):
    """cov: (P x P) or a stack (B x P x P) -> F with F[..., p, k] = sqrt(s_k) V[k][p]: numpy's legacy multivariate_normal factor,
    transposed for the GEMM.  One LAPACK call per matrix (numpy's gufunc loops over the stack in C: the same calls, the same bits
    as matrix-by-matrix), on ONE BLAS thread: a 70 x 70 SVD on a many-core host otherwise spends its time waking and parking the
    thread pool.  The thread limit goes through one ThreadpoolController kept for the process (a fresh threadpool_limits context
    re-scans the loaded libraries, ~0.4 ms per use)."""
    global _blas_controller
    if _ThreadpoolController is not None:
        if _blas_controller is None:
            _blas_controller = _ThreadpoolController()
        with _blas_controller.limit(limits=1):
            _, s, v = np.linalg.svd(cov)
    else:
        _, s, v = np.linalg.svd(cov)
    return np.ascontiguousarray(np.swapaxes(np.sqrt(s)[..., :, None] * v, -1, -2))


def _device_factor(Sp_dev):
    """lower Cholesky factors of a [B, P, P] stack on the device (jitter retry on round-off indefiniteness)"""
    B, P, _ = Sp_dev.shape
    out = Sp_dev.clone()
    for b in range(B):
        jitter = 0.0
        for _ in range(6):
            A = Sp_dev[b].clone()
            if jitter:
                A.diagonal().add_(jitter)
            info, _ws = ops.potrf_lower(A)
            if info == 0:
                break
            jitter = max(10 * jitter, 1e-12 * float(Sp_dev[b].diagonal().max()))
        else:
            raise np.linalg.LinAlgError("predictive covariance of grid %d is not positive definite even with jitter %g" % (b, jitter))
        out[b] = A.tril()
    return out


def sampled_max_batch(pairs, GP_model, mc_samples):
    """For every (xi, x) in `pairs`: f_max of `mc_samples` posterior draws on the 70-point projected grid.
    Returns fmax [B, S] on the device.  RNG order per pair = reference order inside EI / varmax (:73-79)."""
    B, S, P = len(pairs), int(mc_samples), GRID_POINTS
    t0 = time.time()
    grids = np.empty((B, P, GP_model.D))
    Z = np.empty((B, S, P))
    for b, (xi, x) in enumerate(pairs):
        grids[b] = GP_model.FP.xi_grid(xi=xi, x=x, alpha_grid_distribution='equispaced', alpha_star=None, m=P, is_scaled=True)
        Z[b] = np.random.standard_normal((S, P))            # == S successive multivariate_normal draws of size P
    t1 = time.time()
    mu, Sp = GP_model._predict_dev(ops.to_dev(grids.reshape(B * P, -1)), P, B)
    if getattr(GP_model, "mvn_factor", "svd-host") == "device":
        Fac = _device_factor(Sp)
        t2 = t3 = time.time()
    else:
        Sp_h = Sp.cpu().numpy()
        t2 = time.time()
        Fac = ops.to_dev(_svd_factor(Sp_h))
        t3 = time.time()
    fmax, _arg = ops.mvn_rowmax(ops.to_dev(Z), Fac, mu)
    tm = getattr(GP_model, "timing", None)
    if tm is not None:       # seconds: host draws / device prediction (incl. the factor at the mode on first use) / host SVD factors
        tm["acq_draws"], tm["acq_predict"], tm["acq_svd"] = t1 - t0, t2 - t1, t3 - t2
    return fmax


def _ei_values(pairs, GP_model, mc_samples):
    fmax = sampled_max_batch(pairs, GP_model, mc_samples)
    sums = ops.acq_reduce(fmax, float(GP_model.mustar)).cpu().numpy()
    return sums[:, 0] / mc_samples


def _varmax_values(pairs, GP_model, mc_samples):
    fmax = sampled_max_batch(pairs, GP_model, mc_samples)
    sums = ops.acq_reduce(fmax, 0.0).cpu().numpy()
    mean = sums[:, 1] / mc_samples
    # (one-pass form E[x^2] - mean^2 from the device sums; the reference's mean((x - mean)^2) is >= 0 by construction, so clamp
    # the round-off of the cancellation)
    return np.maximum(sums[:, 2] / mc_samples - mean * mean, 0.0)


# ------------------------------------------------------------------------------------------------ reference API
def next_query(PPBO_settings, GP_model, unscale=True):
    """dispatch on the strategy name (src/acquisition.py:9-65); mutates the cyclic state on PPBO_settings like the reference"""
    start = time.time()
    name = PPBO_settings.xi_acquisition_function
    if name in ('EI', 'EXR', 'EI-FIXEDX'):
        xi_dims = list((np.array(PPBO_settings.xi_dims_prev_iter) + 1) % PPBO_settings.D)
        PPBO_settings.xi_dims_prev_iter = xi_dims
    if name == 'EI':
        xi_next, x_next = maximize_EI(xi_dims, GP_model, PPBO_settings)
    elif name == 'EI-FIXEDX':
        xi_next, x_next = maximize_EI_fixed_x(xi_dims, GP_model, PPBO_settings)
    elif name == 'EXR':
        xi_next, x_next = maximize_varmax(xi_dims, GP_model, PPBO_settings)
    else:
        if name in ('EI-EXT-FAST', 'EI-VARMAX-FAST'):
            xi_next = EId_xstar(GP_model, PPBO_settings.mc_samples)
        elif name in ('EI-EXT', 'EI-VARMAX'):
            xi_next = EId_integrate(GP_model, PPBO_settings.mc_samples)
        elif name in ('COORDINATE-VARMAX', 'PCD'):
            xi_next = PCD_next_xi(PPBO_settings)
        elif name == 'RAND':
            xi_next = random_next_xi(PPBO_settings)
        elif name == 'EXT':
            xi_next = EXT_next_xi(PPBO_settings, GP_model)
        else:
            print('Invalid acquisition function name!')
            return 0
        x_next = next_x_given_xi(xi_next, GP_model, PPBO_settings)
    if GP_model.verbose:
        print("Evaluation of the acquisition function took " + str(time.time() - start) + " seconds.")
    xi_next = np.abs(xi_next) / np.max(np.abs(xi_next))           # normalise before unscaling (:58)
    if unscale:
        xi_next = GP_model.FP.unscale(xi_next, retain_0_values=True)
        x_next = GP_model.FP.unscale(x_next, retain_0_values=True)
        if GP_model.verbose:
            print("Next query: (xi,x) = " + str((xi_next, x_next)))
    return (xi_next, x_next)


BATCH_STRATEGIES = ('EI-EXT-FAST', 'EI-VARMAX-FAST')


def sampled_max_joint(pairs, GP_model, mc_samples):
    """f_max on the 70-point grid of every (xi, x) in `pairs` from JOINT posterior draws over all B grids: one prediction of the
    B*70 points with their cross-covariance, one device Cholesky factor L (jitter retry: lines through x* nearly share points),
    f = mu + L z with z = np.random.standard_normal((S, B*70)) in one call.  RNG: the B grid jitters in order, then the S x B*70
    normals.  Returns fmax [B, S] and, for checking, the grids [B, 70, D], Z [S, B*70], mu [B*70] and L (device)."""
    B, S, P = len(pairs), int(mc_samples), GRID_POINTS
    grids = np.empty((B, P, GP_model.D))
    for b, (xi, x) in enumerate(pairs):
        grids[b] = GP_model.FP.xi_grid(xi=xi, x=x, alpha_grid_distribution='equispaced', alpha_star=None, m=P, is_scaled=True)
    Z = np.random.standard_normal((S, B * P))
    mu, Sp = GP_model._predict_dev(ops.to_dev(grids.reshape(B * P, -1)), B * P, 1)
    L = _device_factor(Sp)[0]
    Zd = ops.to_dev(Z)
    # grid b's rows of L are its points' coefficients on the B*70 joint normals: one row-max per grid over the shared draws
    fmax, _arg = ops.mvn_rowmax(Zd.unsqueeze(0).expand(B, -1, -1), L.view(B, P, B * P), mu.view(B, P))
    return fmax, grids, Z, mu.view(-1), L


def next_query_batch(PPBO_settings, GP_model, q, unscale=True):
    """q queries for evaluators who answer in parallel (no counterpart in the reference, which proposes one).  For the strategies
    whose xi is a coordinate direction through x* ('EI-EXT-FAST', 'EI-VARMAX-FAST'): the D lines of EId_xstar, joint posterior
    draws on all of them (sampled_max_joint), and q lines chosen greedily by joint expected improvement over those draws
    (ppbo_b200.iteration.select_batch): a line that reaches the same peak as a chosen one adds nothing, where the top q by marginal
    EI would take both.  Each chosen xi then gets its x from next_x_given_xi, in pick order.  Returns a list of q (xi, x) pairs,
    normalised and unscaled as next_query does.
    RNG consumption: the D grid jitters (reference order of _coordinate_pairs), one standard_normal((mc_samples, D*70)) call, then
    whatever next_x_given_xi draws for each pick in turn (nothing for x_acquisition_function 'exploit')."""
    from ppbo_b200 import iteration
    name = PPBO_settings.xi_acquisition_function
    if name not in BATCH_STRATEGIES:
        raise ValueError("next_query_batch serves %s, not %r" % (BATCH_STRATEGIES, name))
    xis, pairs = _coordinate_pairs(GP_model)
    if not 1 <= q <= len(pairs):
        raise ValueError("q must be in [1, %d], not %r" % (len(pairs), q))
    fmax = sampled_max_joint(pairs, GP_model, PPBO_settings.mc_samples)[0]
    mustar = ops.to_dev(np.array([float(GP_model.mustar)]))
    idx, _qei = iteration.select_batch(fmax, mustar, q, len(pairs))
    out = []
    for b in idx.cpu().numpy():
        xi_next = xis[int(b)].copy()
        x_next = next_x_given_xi(xi_next, GP_model, PPBO_settings)
        xi_next = np.abs(xi_next) / np.max(np.abs(xi_next))
        if unscale:
            xi_next = GP_model.FP.unscale(xi_next, retain_0_values=True)
            x_next = GP_model.FP.unscale(x_next, retain_0_values=True)
        out.append((xi_next, x_next))
    return out


def EI(xi, x, GP_model, mc_samples):
    """expected improvement of the projective query (xi, x) (src/acquisition.py:72-81)"""
    return float(_ei_values([(xi, x)], GP_model, mc_samples)[0])


def varmax(xi, x, GP_model, mc_samples):
    """variance over posterior draws of the maximum along the query line (src/acquisition.py:170-178)"""
    return float(_varmax_values([(xi, x)], GP_model, mc_samples)[0])


def _coordinate_pairs(GP_model):
    xis = np.eye(GP_model.D)
    pairs = []
    for d in range(GP_model.D):
        x = GP_model.xstar.copy()
        x[d] = 0
        pairs.append((xis[d], x))
    return xis, pairs


def EId_xstar(GP_model, mc_samples):
    """unit vector e_d maximising EI(e_d, xstar with coordinate d freed) (src/acquisition.py:132-145); the D evaluations
    are one batched device pass"""
    xis, pairs = _coordinate_pairs(GP_model)
    EIvals = _ei_values(pairs, GP_model, mc_samples)
    return xis[int(np.argmax(EIvals))]


def EId_integrate(GP_model, mc_samples):
    """as EId_xstar with x integrated out over 50 uniform draws per coordinate (src/acquisition.py:146-163)"""
    mc_samples2 = 50
    D = GP_model.D
    xis = np.eye(D)
    EIvals = np.zeros(D)
    for d in range(D):
        xs = np.random.uniform(0, 1, (mc_samples2, D))
        xs[:, d] = 0
        EIvals[d] = np.sum(_ei_values([(xis[d], x) for x in xs], GP_model, mc_samples)) / mc_samples2
    return xis[int(np.argmax(EIvals))]


# ---- outer searches over (xi, x).  The reference runs GPyOpt's Bayesian optimisation (5 initial + BO_maxiter sequential
# evaluations) around the EI / varmax callbacks; GPyOpt is not installable here, so the same evaluation budget is spent on a
# uniform candidate set scored in one batched device pass.  If GPyOpt is importable it is used exactly as in the reference.
def _maximise(score_batch, score_one, n_free, budget):
    try:
        from GPyOpt.methods import BayesianOptimization
    except Exception:
        BayesianOptimization = None
    if BayesianOptimization is not None:
        bounds = [{'name': 'var_' + str(d), 'type': 'continuous', 'domain': (0, 1)} for d in range(1, n_free + 1)]
        BO = BayesianOptimization(lambda v: -score_one(v[0]), domain=bounds, optimize_restarts=0, normalize_Y=True)
        BO.run_optimization(max_iter=budget)
        return np.asarray(BO.x_opt, dtype=float)
    cand = np.random.uniform(0, 1, (5 + int(budget), n_free))
    return cand[int(np.argmax(score_batch(cand)))]


def _split(v, xi_dims, x_dims, D):
    xi, x = np.zeros(D), np.zeros(D)
    xi[xi_dims] = v[xi_dims]
    x[x_dims] = v[x_dims]
    return xi, x


def EI_to_maximize(xi_plus_x, xi_dims, x_dims, GP_model, mc_samples):
    xi, x = _split(np.asarray(xi_plus_x)[0], xi_dims, x_dims, GP_model.D)
    return EI(xi, x, GP_model, mc_samples)


def varmax_to_maximize(xi_plus_x, xi_dims, x_dims, GP_model, mc_samples):
    xi, x = _split(np.asarray(xi_plus_x)[0], xi_dims, x_dims, GP_model.D)
    return varmax(xi, x, GP_model, mc_samples)


def _maximise_over_xi_x(values, xi_dims, GP_model, PPBO_settings):
    D, S = GP_model.D, PPBO_settings.mc_samples
    x_dims = [i for i in range(D) if i not in xi_dims]
    res = _maximise(lambda C: values([_split(c, xi_dims, x_dims, D) for c in C], GP_model, S),
                    lambda v: values([_split(np.asarray(v), xi_dims, x_dims, D)], GP_model, S)[0], D, PPBO_settings.BO_maxiter)
    xi, x = _split(res, xi_dims, x_dims, D)
    return perturbate_zerocoordinates(xi, xi_dims), perturbate_zerocoordinates(x, x_dims)


def maximize_EI(xi_dims, GP_model, PPBO_settings):
    """src/acquisition.py:91-113"""
    return _maximise_over_xi_x(_ei_values, xi_dims, GP_model, PPBO_settings)


def maximize_varmax(xi_dims, GP_model, PPBO_settings):
    """src/acquisition.py:189-206"""
    return _maximise_over_xi_x(_varmax_values, xi_dims, GP_model, PPBO_settings)


def EI_fixed_x_to_maximize(xi, xstar, xi_dims, GP_model, mc_samples):
    xi_ = xstar.copy()
    xi_[xi_dims] = np.asarray(xi)[0]
    return EI(xi_, xstar, GP_model, mc_samples)


def maximize_EI_fixed_x(xi_dims, GP_model, PPBO_settings):
    """src/acquisition.py:114-131: EI over the xi coordinates with x pinned to xstar"""
    D, S = GP_model.D, PPBO_settings.mc_samples
    xstar = GP_model.xstar.copy()
    x_dims = [i for i in range(D) if i not in xi_dims]

    def pair(v):
        xi_ = xstar.copy()
        xi_[xi_dims] = v
        return (xi_, xstar)
    res = _maximise(lambda C: _ei_values([pair(c) for c in C], GP_model, S),
                    lambda v: _ei_values([pair(np.asarray(v))], GP_model, S)[0], len(xi_dims), PPBO_settings.BO_maxiter)
    xi, x = np.zeros(D), np.zeros(D)
    xi[xi_dims] = res
    x[x_dims] = xstar[x_dims]
    return perturbate_zerocoordinates(xi, xi_dims), perturbate_zerocoordinates(x, x_dims)


def maximize_varmax_given_xi(xi, GP_model, PPBO_settings):
    """src/acquisition.py:208-218"""
    D, S = GP_model.D, PPBO_settings.mc_samples
    x_next = _maximise(lambda C: _varmax_values([(xi, c) for c in C], GP_model, S),
                       lambda v: _varmax_values([(xi, np.asarray(v))], GP_model, S)[0], D, PPBO_settings.BO_maxiter)
    x_next = np.array(x_next, dtype=float)
    x_next[np.where(np.asarray(xi) != 0)[0]] = 0
    return x_next


# ------------------------------------------------------------------------------------------------ coordinate rules (host glue)
def random_next_xi(PPBO_settings):
    D = PPBO_settings.D
    coords = list(set(np.random.choice(D, D - 1, replace=True)))
    xi_next = np.zeros(D)
    xi_next[coords] = np.random.uniform(0, 1, (1, len(coords)))[0]
    return xi_next


def _advance_dim(PPBO_settings):
    d = int(PPBO_settings.dim_query_prev_iter + 1)
    if d > PPBO_settings.D:
        d = 1
    PPBO_settings.dim_query_prev_iter = d
    return d


def PCD_next_xi(PPBO_settings):
    return np.eye(PPBO_settings.D)[:, _advance_dim(PPBO_settings) - 1]


def EXT_next_xi(PPBO_settings, GP_model):
    xi_next = GP_model.xstar.copy()
    xi_next[xi_next == 0] = 1e-7
    xi_next[_advance_dim(PPBO_settings) - 1] = 0
    return xi_next


def next_x_given_xi(xi, GP_model, PPBO_settings):
    free = list(np.where(xi == 0)[0])
    x_next = np.zeros(PPBO_settings.D)
    rule = PPBO_settings.x_acquisition_function
    if rule == "exploit":
        x_next[free] = GP_model.xstar.copy()[free]
    elif rule == "varmax":
        x_next = maximize_varmax_given_xi(xi, GP_model, PPBO_settings)
    elif rule == "random":
        x_next[free] = np.random.uniform(0, 1, (1, len(free)))[0]
    else:
        print("Invalid acquisition function selected!")
        return None
    return perturbate_zerocoordinates(x_next, free)


def perturbate_zerocoordinates(x, nonzero_coords):
    x_ = x[nonzero_coords].copy()
    x_[x_ == 0] = 1e-7
    x[nonzero_coords] = x_
    return x
