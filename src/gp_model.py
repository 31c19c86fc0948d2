"""GP utility model with the preference likelihood -- host-side mirror of the reference's src/gp_model.py (same class,
method and attribute names) whose arithmetic runs on the GPU through the C ABI of ppbo_b200.

What differs from the reference, on purpose (DESIGN.md "Laplace fit"):
  * The mode is found by a damped Newton iteration in the space of latent differences (one Cholesky of size Q m per step,
    no Sigma^-1), not by scipy's trust-exact on the N x N Hessian.  Both stop at a stationary point of the same T; the
    reference stops at |grad T| < 1e-4, this path at a relative step of 1e-10.
  * The reference starts the optimiser from a random draw f ~ N(0, Sigma) (SVD of Sigma).  The draw is still consumed from
    the global numpy RNG (so later draws -- DE, grid jitter, MVN normals -- stay aligned with a reference run), but the
    Newton iteration starts from the previous mode padded with its mean (the reference's own warm-start rule,
    src/gp_model.py:375-377) or from zero.
  * Sigma_inv, Lambda_MAP, posterior_covariance(_inv) and Sigma are materialised on the host only when read.
"""
import os
import sys
import time

import numpy as np
import scipy.optimize

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

from feedback_processing import FeedbackProcessing  # noqa: E402
from kernels import SE_kernel, RQ_kernel, camphor_copper_kernel, Matern32_kernel, Matern52_kernel  # noqa: E402,F401
from misc import pd_inverse, regularize_covariance, var2_normal_pdf  # noqa: E402,F401
from ppbo_b200 import ops  # noqa: E402
from ppbo_b200 import device_linalg as _dl  # noqa: E402

_KERNELS = {"SE_kernel": SE_kernel, "RQ_kernel": RQ_kernel, "camphor_copper_kernel": camphor_copper_kernel,
            "Matern32_kernel": Matern32_kernel, "Matern52_kernel": Matern52_kernel}


class _Lazy:
    """Attribute computed on the device, copied to the host on first read, overridable by assignment."""

    def __init__(self, name):
        self.slot = "_lazy_" + name
        self.maker = "_make_" + name

    def __get__(self, obj, owner=None):
        if obj is None:
            return self
        val = obj.__dict__.get(self.slot)
        if val is None:
            val = getattr(obj, self.maker)()
            obj.__dict__[self.slot] = val
        return val

    def __set__(self, obj, value):
        obj.__dict__[self.slot] = value


class GPModel:
    Sigma = _Lazy("Sigma")
    Sigma_inv = _Lazy("Sigma_inv")
    Lambda_MAP = _Lazy("Lambda_MAP")
    posterior_covariance = _Lazy("posterior_covariance")
    posterior_covariance_inv = _Lazy("posterior_covariance_inv")

    def __init__(self, PPBO_settings):
        self.COVARIANCE_SHRINKAGE = 1e-6                     # src/gp_model.py:26
        self.verbose = PPBO_settings.verbose
        self.FP = None
        self.D = PPBO_settings.D
        self.original_bounds = PPBO_settings.original_bounds
        self.bounds = ((0, 1),) * self.D
        self.X = None
        self.N = None
        self.m = PPBO_settings.n_pseudoobservations
        self.obs_indices = self.pseudobs_indices = self.latest_obs_indices = None
        self.alpha_grid_distribution = PPBO_settings.alpha_grid_distribution
        self.TGN_speed = PPBO_settings.TGN_speed
        self.n_gausshermite_sample_points = PPBO_settings.n_gausshermite_sample_points
        self.xi_acquisition_function = PPBO_settings.xi_acquisition_function
        self.kernel = _KERNELS[PPBO_settings.kernel]
        self.theta_initial = PPBO_settings.theta_initial
        self.theta = None
        self.fMAP = None
        self.fMAP_finding_trials = 1
        self.fMAP_optimizer = PPBO_settings.fMAP_optimizer
        self.fMAP_random_initial_vector = True
        self.mustar_finding_trials = PPBO_settings.mustar_finding_trials
        self.mustar_previous_iteration = 0
        self.mustar = None
        self.xstar = None
        self.xstars_local = None
        self.initialization_running = True
        self.last_iteration = False
        self.skip_computations_during_initialization = PPBO_settings.skip_computations_during_initialization
        self.skip_xstaroptimization_during_initialization = PPBO_settings.skip_xstaroptimization_during_initialization
        # B200-path knobs (additive, see PPBO_settings)
        self.mvn_factor = getattr(PPBO_settings, "mvn_factor", "svd-host")
        self.mustar_method = getattr(PPBO_settings, "mustar_method", "de")
        self.mustar_window = getattr(PPBO_settings, "mustar_window", 16)
        self.newton_max_iter, self.newton_tol = 100, 1e-10
        # device state
        self._X_dev = None           # [N x D]
        self._Sigma_dev = None       # [N x N]
        self._fit = None             # ops.LaplaceFit (f_map, alpha, arrow, G, Lfac, neg_corr)
        self.fit_stats = None
        self.timing = {}             # seconds spent in the last update_model: 'fit' (covariance + MAP), 'mu_star' 

    # ------------------------------------------------------------------ wrappers (src/gp_model.py:73-85)
    def update_feedback_processing_object(self, X_obs):
        if self.FP is None:
            self.FP = FeedbackProcessing(self.D, self.m, self.original_bounds, self.alpha_grid_distribution, self.TGN_speed)
            self.FP.initialize_data(X_obs)
        else:
            self.FP.update_data(X_obs)

    def update_data(self):
        self.X = self.FP.X
        self.N = self.FP.N
        self.obs_indices = self.FP.obs_indices
        self.pseudobs_indices = self.FP.pseudobs_indices
        self.latest_obs_indices = self.FP.latest_obs_indices
        self._X_dev = None

    def turn_initialization_off(self):
        self.initialization_running = False
        self.FP.alpha_grid_distribution = self.alpha_grid_distribution

    def set_last_iteration(self):
        self.last_iteration = True

    def is_pseudobs(self, i):
        return self.FP.is_pseudobs(i)

    def set_theta(self):
        """defaults for missing hyper-parameters; mutates the caller's list like the reference (src/gp_model.py:164-171)"""
        self.theta = self.theta_initial
        for idx, default in ((1, 1), (2, 0.1), (0, 8)):
            if self.theta[idx] is None:
                self.theta[idx] = default

    # ------------------------------------------------------------------ device plumbing
    def _Q(self):
        Q, rem = divmod(int(self.N), self.m + 1)
        if rem:
            raise ValueError("N must be a multiple of m + 1")
        return Q

    def _Xd(self):
        if self._X_dev is None or self._X_dev.shape[0] != self.N:
            self._X_dev = ops.to_dev(self.X)
        return self._X_dev

    def _invalidate(self, *names):
        for n in names:
            self.__dict__.pop("_lazy_" + n, None)

    def _kernel_name(self, kernel=None):
        k = self.kernel if kernel is None else kernel
        return k if isinstance(k, str) else k.__name__

    # ------------------------------------------------------------------ covariance (src/gp_model.py:147-162)
    def create_Gramian(self, X1, X2, kernel, *args):
        """regularised square covariance: kernel + fused shrinkage on the device when X1 is X2, else kernel then shrink"""
        theta = args[0]
        X1 = np.atleast_2d(np.asarray(X1, dtype=np.float64))
        if X1 is X2 or (np.shape(X1) == np.shape(X2) and np.array_equal(X1, X2)):
            Xd = ops.to_dev(X1)
            return ops.gram_regularized(self._kernel_name(kernel), Xd, theta[1], theta[2], self.COVARIANCE_SHRINKAGE).cpu().numpy()
        return regularize_covariance(kernel(X1, X2, *args), self.COVARIANCE_SHRINKAGE)

    def create_Gramian_nonsquare(self, X1, X2, kernel, *args):
        return kernel(X1, X2, *args)

    def update_Sigma(self, theta):
        self._Sigma_dev = ops.gram_regularized(self._kernel_name(), self._Xd(), theta[1], theta[2], self.COVARIANCE_SHRINKAGE)
        self._invalidate("Sigma", "Sigma_inv")

    def update_Sigma_inv(self, theta):
        """The device path never needs Sigma^-1; the public attribute is built on first read (_make_Sigma_inv)."""
        self._invalidate("Sigma_inv")

    def _make_Sigma(self):
        return None if self._Sigma_dev is None else self._Sigma_dev.cpu().numpy()

    def _make_Sigma_inv(self):
        if self._Sigma_dev is None:
            return None
        return _dl.spd_inverse_dev(self._Sigma_dev.clone()).cpu().numpy()

    # ------------------------------------------------------------------ functional T (src/gp_model.py:176-274)
    def _lik(self, f, sigma, want_sum=False, want_beta=False, want_arrow=False):
        fd = ops.to_dev(np.asarray(f, dtype=np.float64).ravel())
        return ops.lik_terms(fd, self._Q(), self.m, sigma, want_sum, want_beta, want_arrow)

    def sum_Phi_vec(self, order_of_derivative, f, sigma, over_all_indices=False):
        """per comparison set: sum_j Phi~(Delta), sum_j phi~(Delta) or sum_j -Delta phi~(Delta)/2 (src/gp_model.py:206-218)"""
        Q, m = self._Q(), self.m
        fd = ops.to_dev(np.asarray(f, dtype=np.float64).ravel())
        if order_of_derivative == 0:
            out = ops.lik_set_sums(fd, Q, m, sigma).cpu().numpy()          # all comparison sets in one launch
        elif order_of_derivative == 1:
            _, beta, _ = ops.lik_terms(fd, Q, m, sigma, False, True, False)
            out = beta.cpu().numpy().reshape(Q, m + 1)[:, 0] * (sigma * m)
        elif order_of_derivative == 2:
            _, _, arrow = ops.lik_terms(fd, Q, m, sigma, False, False, True)
            out = arrow.cpu().numpy().reshape(Q, m).sum(axis=1) * (m * sigma ** 2)
        else:
            print("The derivatives of an order higher than 2 are not needed!")
            return None
        if over_all_indices:
            return np.repeat(out, m + 1)
        return out

    def _Sigma_inv_times(self, f, Sigma_inv_):
        f = np.asarray(f, dtype=np.float64).ravel()
        if Sigma_inv_ is not None:
            return ops.gemv(ops.to_dev(Sigma_inv_), ops.to_dev(f)).cpu().numpy()
        A = self._Sigma_dev.clone()
        info, ws = ops.potrf_lower(A)
        if info:
            raise np.linalg.LinAlgError("Sigma is not positive definite (pivot %d)" % info)
        return ops.potrs_vec(A, ws, ops.to_dev(f)).cpu().numpy()

    def T(self, f, theta, Sigma_inv_=None):
        """-1/2 f' Sigma^-1 f - (1/m) sum Phi~(Delta)   (src/gp_model.py:221-226)"""
        f = np.asarray(f, dtype=np.float64).ravel()
        s, _, _ = self._lik(f, theta[0], want_sum=True)
        return float(-0.5 * f @ self._Sigma_inv_times(f, Sigma_inv_) - float(s) / self.m)

    def T_grad(self, f, theta, Sigma_inv_=None):
        """-Sigma^-1 f + beta   (src/gp_model.py:228-240)"""
        f = np.asarray(f, dtype=np.float64).ravel()
        _, beta, _ = self._lik(f, theta[0], want_beta=True)
        return -self._Sigma_inv_times(f, Sigma_inv_) + beta.cpu().numpy()

    def T_hessian(self, f, theta, Sigma_inv_=None):
        """-Sigma^-1 + Lambda   (src/gp_model.py:242-247)"""
        Sinv = self.Sigma_inv if Sigma_inv_ is None else Sigma_inv_
        return -Sinv + self.create_Lambda(f, theta[0])

    def create_Lambda(self, f, sigma):
        """dense likelihood Hessian: one arrow block per comparison set (src/gp_model.py:249-274)"""
        _, _, arrow = self._lik(f, sigma, want_arrow=True)
        return ops.lambda_dense(arrow, self._Q(), self.m).cpu().numpy()

    # ------------------------------------------------------------------ MAP (src/gp_model.py:354-389)
    def update_fMAP(self, random_initial_vector=None, fmap_finding_trials=None, approx_optimization=False):
        if fmap_finding_trials is None:
            fmap_finding_trials = self.fMAP_finding_trials
        if random_initial_vector is None:
            random_initial_vector = self.fMAP_random_initial_vector
        if self.verbose:
            print("MAP-estimation begins...")
        start = time.time()
        Q, N = self._Q(), int(self.N)
        best = None
        Lsig = None
        for trial in range(fmap_finding_trials):
            prev = None if self.fMAP is None else np.asarray(self.fMAP, dtype=np.float64).ravel()
            draws_random = prev is None or random_initial_vector or len(prev) > N
            z = None
            if draws_random:
                z = np.random.standard_normal(N)    # the reference's N(0, Sigma) start consumes N normals here (:374,:381)
            if prev is None or len(prev) > N:
                f0 = None
            elif len(prev) < N:
                f0 = np.concatenate([prev, np.full(N - len(prev), prev.mean())])        # :375-377
            else:
                f0 = prev
            f0_dev = None if f0 is None else ops.to_dev(f0)
            if trial > 0 and z is not None:
                # multi-start (the reference's last iteration runs 10 random starts on a non-concave T, :96-97): trials after the
                # first start from the consumed draw, f0 = chol(Sigma) z ~ N(0, Sigma) (the reference uses an SVD factor)
                if Lsig is None:
                    Lsig = self._Sigma_dev.clone()
                    info, _ws = ops.potrf_lower(Lsig)
                    Lsig = Lsig.tril_() if info == 0 else False
                if Lsig is not False:
                    f0_dev = ops.gemv(Lsig, ops.to_dev(z))
            # approx_optimization (gtol=100 in the reference ~ a single Newton step, :365-366)
            iters = 2 if approx_optimization else self.newton_max_iter
            fit = ops.laplace_fit(self._Sigma_dev, Q, self.m, self.theta[0], f_init=f0_dev, max_iter=iters, tol=self.newton_tol)
            if fit.info != 0:
                print('---!!!--- Newton system is not positive definite (info=%d) ---!!!---' % fit.info)
            elif not approx_optimization and not fit.stats["converged"]:
                print('---!!!--- MAP iteration stopped at max_iter with relative step %.2e ---!!!---' % fit.stats["last_rel_step"])
            if self.verbose:
                print('... this took ' + str(time.time() - start) + ' seconds.')
            if best is None or fit.stats["T"] > best.stats["T"]:
                best = fit
        self._fit = best
        self.fit_stats = best.stats
        self._point_mean = None
        self.fMAP = best.f_map.cpu().numpy()
        self._invalidate("Lambda_MAP", "posterior_covariance", "posterior_covariance_inv")

    def _make_Lambda_MAP(self):
        if self._fit is None:
            return None
        return ops.lambda_dense(self._fit.arrow, self._Q(), self.m).cpu().numpy()

    def _make_posterior_covariance_inv(self):
        if self._fit is None:
            return None
        return self.Sigma_inv - self.Lambda_MAP

    def _make_posterior_covariance(self):
        """(Sigma^-1 - Lambda_MAP)^-1 (src/gp_model.py:116-117) evaluated as Sigma - Sigma W^1/2 (I + W^1/2 Sigma W^1/2)^-1 W^1/2 Sigma
        through the prediction kernel with the design itself as the prediction set (no explicit inverse)."""
        if self._fit is None:
            return None
        try:
            theta = self.theta
            _, Sp = ops.predict(self._kernel_name(), self._Xd(), theta[1], theta[2], self.COVARIANCE_SHRINKAGE, self._fit,
                                self._Xd(), int(self.N), 1)
            return Sp[0].cpu().numpy()
        except Exception:
            print('---!!!--- Posterior covariance matrix is not PSD ---!!!---')
            return None

    # ------------------------------------------------------------------ model update (src/gp_model.py:87-132)
    def update_model(self, optimize_theta=False):
        t_fit = time.time()
        if self.theta is None:
            self.set_theta()
        self.update_Sigma(self.theta)
        self.update_Sigma_inv(self.theta)
        init_light = self.initialization_running and self.skip_computations_during_initialization
        if init_light:
            self.FP.alpha_grid_distribution = 'equispaced'
            self.update_fMAP(random_initial_vector=False, fmap_finding_trials=1, approx_optimization=True)
        elif self.last_iteration:
            self.update_fMAP(random_initial_vector=True, fmap_finding_trials=10)
        else:
            self.update_fMAP()
        if optimize_theta:
            self.optimize_theta()
            self.update_fMAP()
            self.update_Sigma(self.theta)
            self.update_Sigma_inv(self.theta)
        if self.verbose:
            print("Current theta is: " + str(self.theta) + ' (Acq. = ' + str(self.xi_acquisition_function) + ')')
        # Lambda_MAP / posterior covariance are products of the fit (arrow coefficients + factor) and materialise lazily
        if self.verbose:
            print("Computing mu_star and x_star ...")
        start = time.time()
        self.timing["fit"] = start - t_fit
        if init_light and not self.skip_xstaroptimization_during_initialization:
            self.xstar, self.mustar, self.xstars_local = self.mu_star(mustar_finding_trials=1)
        elif self.initialization_running and self.skip_xstaroptimization_during_initialization:
            pass
        elif self.last_iteration:
            self.xstar, self.mustar, self.xstars_local = self.mu_star(mustar_finding_trials=20)
        else:
            self.xstar, self.mustar, self.xstars_local = self.mu_star()
        self.timing["mu_star"] = time.time() - start
        if self.verbose:
            print("... this took " + str(time.time() - start) + " seconds.")

    # ------------------------------------------------------------------ evidence (src/gp_model.py:278-413)
    def _evidence_terms(self, theta, f=None):
        """(T(f), sign of det U, log|det|, sign of the row permutation, info) at hyper-parameters theta; f: the mode to evaluate
        at (None: found here by the device Newton iteration from f = 0).  `evidence_formula`:
          'reference' (default): LU of I + Sigma Lambda_MAP exactly as the reference (src/gp_model.py:301-308) -- with
                       Lambda = -W this is det(I - Sigma W), not the Laplace normaliser; reproduced for drop-in parity
          'laplace'  : LU of I + Sigma W, the determinant the Laplace approximation of the evidence calls for."""
        Q = self._Q()
        Sigma_ = ops.gram_regularized(self._kernel_name(), self._Xd(), theta[1], theta[2], self.COVARIANCE_SHRINKAGE)
        if f is None:
            fit = ops.laplace_fit(Sigma_, Q, self.m, theta[0], max_iter=self.newton_max_iter, tol=self.newton_tol)
            if fit.info != 0:
                return np.nan, 1.0, np.nan, 1.0, fit.info
            T_map, arrow = fit.stats["T"], fit.arrow
        else:
            fd = ops.to_dev(np.asarray(f, dtype=np.float64).ravel())
            s, _, arrow = ops.lik_terms(fd, Q, self.m, theta[0], True, False, True)
            A = Sigma_.clone()
            info, ws = ops.potrf_lower(A)
            if info:
                return np.nan, 1.0, np.nan, 1.0, info
            fh = np.asarray(f, dtype=np.float64).ravel()
            T_map = float(-0.5 * fh @ ops.potrs_vec(A, ws, fd).cpu().numpy() - float(s) / self.m)
        sign_u, logabs, sign_p, info = ops.evidence_logdet(Sigma_, Q, self.m, arrow,
                                                            reference=getattr(self, "evidence_formula", "reference") == "reference")
        return T_map, sign_u, logabs, sign_p, info

    def evidence(self, theta, f_initial=None):
        """log-evidence + log-prior of theta (src/gp_model.py:278-319): T(fMAP) - 1/2 (sign U) log|det(I + Sigma Lambda_MAP)| with
        the determinant from an LU with partial pivoting on the device.  The reference's random start consumes N normals from the
        global RNG (:294, `f_initial` is ignored there too); the mode itself is found deterministically from f = 0."""
        import scipy.stats
        np.random.standard_normal(int(self.N))                 # RNG alignment with the reference's random start (:294)
        T_map, sign_u, logabs, _, info = self._evidence_terms(theta)
        lp = (np.log(scipy.stats.lognorm.pdf(theta[0], s=1, scale=np.exp(1))) +
              np.log(scipy.stats.lognorm.pdf(theta[1], s=0.5, scale=np.exp(-1.4))) +
              np.log(scipy.stats.lognorm.pdf(theta[2], s=0.5, scale=np.exp(1.7))))
        value = T_map - 0.5 * sign_u * logabs + lp
        if info != 0 or np.isnan(value) or not np.isfinite(value):
            if self.verbose:
                print('Nan log-evidence!')
            return -500
        if self.verbose:
            print('(scaled) Log-evidence + Log-prior: ' + str(value))
        return float(value)

    def optimize_theta(self):
        """Hyper-parameter search by maximising `evidence` (src/gp_model.py:391-413): sigma pinned to 1, l in (0.01, 2),
        sigma_f in (0.1, 15) as in the reference.  The reference drives this with GPyOpt (20 initial + 40 sequential evaluations);
        GPyOpt is used when importable, otherwise the same bounds and a comparable evaluation budget go to scipy's differential
        evolution."""
        if self.verbose:
            print("Hyperparameter optimization begins...")
        start = time.time()
        try:
            from GPyOpt.methods import BayesianOptimization
        except Exception:
            BayesianOptimization = None
        if BayesianOptimization is not None:
            bounds = [{'name': 'sigma', 'type': 'continuous', 'domain': (1, 1)},
                      {'name': 'leghtscale', 'type': 'continuous', 'domain': (0.01, 2)},
                      {'name': 'sigma_f', 'type': 'continuous', 'domain': (0.1, 15)}]
            BO = BayesianOptimization(lambda theta: -self.evidence(theta[0], self.fMAP), domain=bounds, optimize_restarts=3,
                                      normalize_Y=True, initial_design_numdata=20)
            BO.run_optimization(max_iter=40)
            self.theta = BO.x_opt
        else:
            res = scipy.optimize.differential_evolution(lambda t: -self.evidence([1.0, t[0], t[1]], None),
                                                        [(0.01, 2), (0.1, 15)], maxiter=5, popsize=5, polish=False)
            self.theta = [1.0, float(res.x[0]), float(res.x[1])]
        if self.verbose:
            print('Optimization of hyperparameters took ' + str(time.time() - start) + ' seconds.')
            print("The optimized theta is " + str(self.theta))

    # ------------------------------------------------------------------ maximiser of the posterior mean (src/gp_model.py:415-437)
    def mu_star(self, mustar_finding_trials=None):
        if mustar_finding_trials is None:
            mustar_finding_trials = self.mustar_finding_trials
        method = self.mustar_method
        if method not in ("de", "de-scipy", "batched"):
            raise ValueError("mustar_method must be 'de', 'de-scipy' or 'batched', not %r" % (method,))
        xstar = xstars_local = None
        best = np.inf
        for i in range(mustar_finding_trials):
            if method == "batched":
                res = scipy.optimize.differential_evolution(self._mu_pred_neq_population, self.bounds, updating='deferred',
                                                            vectorized=True, disp=False, maxiter=2000)
            elif method == "de-scipy":   # literally the reference's call: sequential 'immediate' updating on the global RNG
                res = scipy.optimize.differential_evolution(self.mu_pred_neq, self.bounds, updating='immediate', disp=False,
                                                            maxiter=2000)
            else:                        # 'de': the same search, same draws, same bits, with the loop in C++ (ppbo_mu_star_de)
                res = self._mu_star_de()
            if i == 0:
                xstars_local = np.array(res.x, dtype=float).reshape(1, self.D)
            elif all(np.linalg.norm(x - res.x) > 1e-1 for x in xstars_local):
                xstars_local = np.vstack([xstars_local, res.x])
            if res.fun < best:
                best, xstar = res.fun, np.array(res.x, dtype=float)
        xstar = xstar.reshape(self.D,)
        return xstar, self.mu_pred(xstar), xstars_local

    def _mu_star_de(self):
        """scipy.optimize.differential_evolution(self.mu_pred_neq, self.bounds, updating='immediate', maxiter=2000) with the
        evolution replayed by ppbo_mu_star_de (csrc/de.cu): numpy's global stream is consumed draw for draw as scipy would, every
        trial is one device evaluation of the posterior mean, and the result equals the scipy call's bit for bit (tests/
        test_de_replay.py on the CPU, test_src_gpu.py::test_mu_star_native_equals_scipy on the GPU).  The evaluations are
        issued in speculative windows of `mustar_window` trials, one launch each (1: one launch per trial); the bits do not
        depend on it.  The L-BFGS-B polish that ends scipy's call is made by ops.de_polish exactly as scipy makes it."""
        theta = self.theta
        de = ops.mu_star_de(self._kernel_name(), self._Xd(), theta[1], theta[2], self._fit.alpha, self.bounds, maxiter=2000,
                            window=self.mustar_window)
        self.mu_pred_calls = getattr(self, "mu_pred_calls", 0) + de.nfev
        self.mu_star_launches = getattr(self, "mu_star_launches", 0) + de.calls
        return ops.de_polish(self.mu_pred_neq, de, self.bounds)

    # ------------------------------------------------------------------ predictions (src/gp_model.py:441-461)
    def _predict_dev(self, X_pred_dev, P, batch, want_cov=True):
        theta = self.theta
        return ops.predict(self._kernel_name(), self._Xd(), theta[1], theta[2], self.COVARIANCE_SHRINKAGE, self._fit,
                           X_pred_dev, P, batch, want_cov=want_cov)

    def mu_Sigma_pred(self, X_pred):
        X_pred = np.atleast_2d(np.asarray(X_pred, dtype=np.float64))
        mu, Sp = self._predict_dev(ops.to_dev(X_pred), X_pred.shape[0], 1)
        return mu[0].cpu().numpy(), Sp[0].cpu().numpy()

    def mu_pred(self, X_pred):
        """posterior mean at one point: one launch with the point and the result in mapped host memory (ops.PointMean) -- the
        objective of mu_star's sequential search, ~10^4 evaluations per model update"""
        pm = self.__dict__.get("_point_mean")
        if pm is None or pm.alpha is not self._fit.alpha:
            theta = self.theta
            pm = self._point_mean = ops.PointMean(self._kernel_name(), self._Xd(), theta[1], theta[2], self._fit.alpha)
        self.mu_pred_calls = getattr(self, "mu_pred_calls", 0) + 1
        return pm(np.asarray(X_pred, dtype=np.float64).reshape(self.D))

    def mu_pred_neq(self, X_pred):
        return -self.mu_pred(X_pred)

    def _mu_pred_neq_population(self, Xt):
        """vectorised objective for scipy's DE: Xt is (D, S) -> (S,) negative posterior means, one device call"""
        Xp = np.ascontiguousarray(np.asarray(Xt, dtype=np.float64).T)
        mu, _ = self._predict_dev(ops.to_dev(Xp), Xp.shape[0], 1, want_cov=False)
        return -mu.cpu().numpy().ravel()
