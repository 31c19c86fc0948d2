"""Random-Fourier-feature posterior sampler -- host-side mirror of the reference's src/random_fourier_sampler.py (class
Hsampler, same method and attribute names).  Feature maps, the weight-space objective and its derivatives, the MAP fit,
posterior weight draws and the evaluation of sampled functions run on the GPU through the C ABI of ppbo_b200.

Additions for the B200 path (north_star piece 3): `sample_omegas`, `sample_max_over_grids` -- S posterior functions
evaluated on B projected xi-grids as one dense contraction Omega[S x F] . Phi_grid[F x P] with a fused per-sample
max / arg-max, optionally sharded over the GPUs of a box.

Random numbers: every draw comes from the global legacy numpy RNG on the host, in the reference's order (generate_basis:
W then b -- for the Matern kernels, an addition, W's normals, its chi-square draws, then b; update_omega_MAP: omega0; sample_omega: F normals through numpy's SVD-factor rule, which for the diagonal Laplace
covariance is a permutation by decreasing variance).
"""
import os
import sys
import time

import numpy as np
import scipy.optimize

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

from misc import pd_inverse, var2_normal_pdf  # noqa: E402,F401
from ppbo_b200 import ops  # noqa: E402
from ppbo_b200 import iteration as _it  # noqa: E402
from ppbo_b200.spectral import draw_rff_basis  # noqa: E402


def legacy_mvn_draw(mean, cov, n, rng=np.random):
    """n draws of numpy's legacy multivariate_normal(mean, cov) for a dense covariance, computed as numpy computes them: n F
    standard normals from `rng` in row order, times the SVD factor sqrt(s) V, plus the mean (same values, same generator state)."""
    mean = np.asarray(mean, dtype=np.float64)
    x = rng.standard_normal((n, mean.shape[0]))
    (_, s, v) = np.linalg.svd(cov)
    x = np.dot(x, np.sqrt(s)[:, None] * v)
    x += mean
    return x


class Hsampler:
    def __init__(self, gp_model, nFeatures=1000):
        self.nFeatures = nFeatures
        self.b = None
        self.W = None
        self.D = gp_model.D
        self.m = gp_model.m
        self.X = gp_model.X
        self.GP_xstar = gp_model.xstar
        self.GP_xstars_local = gp_model.xstars_local
        self.n_gausshermite_sample_points = gp_model.n_gausshermite_sample_points
        self.obs_indices = gp_model.obs_indices
        self.kernel = str(gp_model.kernel.__name__)
        self.theta = gp_model.theta
        self.phi_X = None
        self.omega_MAP = None
        self.covariance = None
        self.covariance_inv = None
        # Laplace covariance of the weight posterior: "diag" = the reference's 1 / -hess_diag; "full" = the inverse of the exact
        # Hessian I + Psi' diag(a) Psi (opt-in addition; iteration.WEIGHT_COVARIANCES)
        self.covariance_form = "diag"
        self.verbose = False
        self.newton_max_iter, self.newton_tol = 100, 1e-10
        self.fit_stats = None
        self._dev = {}                     # device copies: W, b, X, phi_X, omega_MAP, hess_diag

    # ------------------------------------------------------------------ basis and feature maps (:38-58)
    def generate_basis(self):
        # SE: the reference's draws; Matern: z, u, b (ppbo_b200/spectral.py); RQ / camphor: b only, no W
        self.W, b = draw_rff_basis(self.kernel, self.nFeatures, self.D, self.theta[1], np.random)
        self.b = b[:, None]
        self._dev.clear()

    def _d(self, name):
        if name not in self._dev:
            if name == "W":
                if self.W is None:
                    raise ValueError("random Fourier basis exists for the SE kernel only (generate_basis)")
                self._dev[name] = ops.to_dev(self.W)
            elif name == "b":
                self._dev[name] = ops.to_dev(np.asarray(self.b).reshape(-1))
            elif name == "X":
                self._dev[name] = ops.to_dev(self.X)
            elif name == "phi_X":
                self._dev[name] = ops.rff_features(self._d("W"), self._d("b"), self._d("X"), self.theta[2], feature_major=True)
        return self._dev[name]

    def _Q(self):
        return self.X.shape[0] // (self.m + 1)

    def phiVec(self, x):
        """F x n feature matrix of the rows of x"""
        x = np.atleast_2d(np.asarray(x, dtype=np.float64))
        return ops.rff_features(self._d("W"), self._d("b"), ops.to_dev(x), self.theta[2], feature_major=True).cpu().numpy()

    def phi(self, x):
        """feature vector (F,) of one point"""
        return self.phiVec(np.asarray(x, dtype=np.float64).reshape(1, self.D))[:, 0]

    def Dphi(self, x):
        """Jacobian d phi / d x, F x D"""
        return ops.rff_jacobian(self._d("W"), self._d("b"), ops.to_dev(np.asarray(x, dtype=np.float64).reshape(self.D)),
                                self.theta[2]).cpu().numpy()

    def DDphi(self, x):
        raise NotImplementedError

    def update_phi_X(self):
        self._dev.pop("phi_X", None)
        self._dev.pop("X", None)
        self.phi_X = self._d("phi_X").cpu().numpy()

    # ------------------------------------------------------------------ objective S and derivatives (:62-122)
    def _objective(self, omega, theta, want_S=False, want_grad=False, want_hess=False):
        return ops.rff_objective(self._d("phi_X"), self._Q(), self.m, theta[0], ops.to_dev(np.asarray(omega, dtype=np.float64)),
                                 want_S=want_S, want_grad=want_grad, want_hess=want_hess)

    def sum_Phi(self, i, order_of_derivative, f, sigma, sample_points=None, weights=None):
        """per comparison set i (an element of obs_indices): scalar (order 0) or F-vector (orders 1, 2) exactly as :62-96;
        thin host loop kept for API parity -- S / S_grad / S_hessian below evaluate all sets in one device pass"""
        m = self.m
        f = np.asarray(f, dtype=float).ravel()
        blk = ops.to_dev(f[i:i + m + 1])
        if order_of_derivative == 0:
            return float(ops.lik_terms(blk, 1, m, sigma, True, False, False)[0])
        Delta = (f[i + 1:i + m + 1] - f[i]) / sigma
        dphi = self.phi_X[:, i + 1:i + m + 1] - self.phi_X[:, [i]]
        if order_of_derivative == 1:
            return dphi @ var2_normal_pdf(Delta)
        if order_of_derivative == 2:
            return -(dphi ** 2) @ (0.5 * Delta * var2_normal_pdf(Delta))
        print("The derivatives of an order higher than 2 are not needed!")
        return None

    def sum_Phi_vec(self, order_of_derivative, f, sigma):
        return np.array([self.sum_Phi(i, order_of_derivative, f, sigma) for i in self.obs_indices])

    def S(self, omega, theta):
        return self._objective(omega, theta, want_S=True)[0]

    def S_grad(self, omega, theta):
        return self._objective(omega, theta, want_grad=True)[1].cpu().numpy()

    def S_hessian(self, omega, theta):
        """the reference's Hessian is diagonal; returned dense (F x F) as there"""
        return np.diag(self._objective(omega, theta, want_hess=True)[2].cpu().numpy())

    # ------------------------------------------------------------------ MAP and Laplace covariance (:124-140)
    def update_omega_MAP(self, omega_initial=None):
        """weight-space MAP.  The reference starts trust-exact from omega0 ~ N(0, I); the same draw is consumed and used as
        the start of the device Newton iteration (exact Hessian, clamped; backtracking)."""
        omega0 = np.random.randn(self.nFeatures)
        if omega_initial is not None:
            omega0 = np.asarray(omega_initial, dtype=np.float64)
        start = time.time()
        omega, hd, stats = ops.rff_fit(self._d("phi_X"), self._Q(), self.m, self.theta[0], omega0=ops.to_dev(omega0),
                                       max_iter=self.newton_max_iter, tol=self.newton_tol)
        if self.verbose:
            print('... this took ' + str(time.time() - start) + ' seconds.')
        self._dev["omega_MAP"], self._dev["hess_diag"] = omega, hd
        self.fit_stats = stats
        self.omega_MAP = omega.cpu().numpy()

    def update_covariancematrix(self):
        if "hess_diag" not in self._dev or self._dev.get("omega_MAP") is None:
            _, _, hd = self._objective(self.omega_MAP, self.theta, want_hess=True)
            self._dev["hess_diag"] = hd
            self._dev["omega_MAP"] = ops.to_dev(self.omega_MAP)
        if self.covariance_form == "full":
            F = self.nFeatures
            Lbuf = ops.rff_hessian_factor_buffer(F, self._dev["omega_MAP"].device)
            info = ops.rff_hessian_factor(self._d("phi_X"), self._Q(), self.m, self.theta[0], self._dev["omega_MAP"], Lbuf)
            if info != 0:
                print('---!!!--- Posterior covariance matrix is not PSD ---!!!---')
                return
            L, ws = ops.hessian_factor_views(Lbuf, F)
            self._dev["L"] = Lbuf
            Lh = np.tril(L.cpu().numpy())
            self.covariance_inv = Lh @ Lh.T
            self.covariance = ops.potri_lower(L, ws).cpu().numpy()
            return
        if self.covariance_form != "diag":
            raise ValueError("covariance_form must be 'diag' or 'full'")
        h = -self._dev["hess_diag"].cpu().numpy()
        if not np.all(h > 0):
            print('---!!!--- Posterior covariance matrix is not PSD ---!!!---')
            return
        self.covariance_inv = np.diag(h)
        self.covariance = np.diag(1.0 / h)

    # ------------------------------------------------------------------ posterior draws (:207-213)
    def _legacy_mvn_normals(self, n):
        """standard normals arranged so that omega_MAP + z / sqrt(h) equals numpy's legacy multivariate_normal draw for the
        diagonal covariance: its SVD factor is the permutation sorting the variances in decreasing order."""
        var = np.diag(self.covariance)
        order = np.argsort(-var, kind="stable")
        z = np.random.standard_normal((n, self.nFeatures))
        out = np.empty_like(z)
        out[:, order] = z
        return out

    def sample_omega(self):
        try:
            return self.sample_omegas(1)[0]
        except Exception:
            print("Omega sampler error! Omega MAP-estimate was used instead.")
            return self.omega_MAP

    def sample_omegas(self, n, seed=None, on_device=False):
        """n draws omega ~ N(omega_MAP, covariance).  seed=None: host RNG in reference order; seed=int: counter-based device RNG"""
        if self.covariance is None:
            raise ValueError("update_covariancematrix() first")
        if self.covariance_form == "full":
            if seed is None:
                Om = ops.to_dev(legacy_mvn_draw(self.omega_MAP, self.covariance, n))
            else:
                Om = ops.rff_sample_omega_full(self._dev["omega_MAP"], self._dev["L"], n, seed=seed)
            return Om if on_device else Om.cpu().numpy()
        if seed is None:
            Om = ops.rff_sample_omega(self._dev["omega_MAP"], self._dev["hess_diag"], n, Z=ops.to_dev(self._legacy_mvn_normals(n)))
        else:
            Om = ops.rff_sample_omega(self._dev["omega_MAP"], self._dev["hess_diag"], n, seed=seed)
        return Om if on_device else Om.cpu().numpy()

    # ------------------------------------------------------------------ batched evaluation (north_star piece 3)
    def evaluate_on_grids(self, Omega, grids):
        """Omega [S, F], grids [B, P, D] (host arrays) -> (fmax [B, S], argmax [B, S]) : per-sample maximum over each grid"""
        grids = np.asarray(grids, dtype=np.float64)
        PhiT = _it.rff_grid_features(self._d("W"), self._d("b"), self.theta[2], ops.to_dev(grids))
        Om = Omega if hasattr(Omega, "data_ptr") else ops.to_dev(Omega)
        fmax, arg, _ = ops.rff_eval_argmax(Om, PhiT)
        return fmax.cpu().numpy(), arg.cpu().numpy()

    def sample_max_over_grids(self, grids, n_samples, mustar, seed=0, shard=None):
        """EI / varmax ingredients from RFF posterior draws: sums over the samples of max(fmax - mu*, 0), fmax, fmax^2 per grid
        (reduced over all ranks of `shard`)."""
        rff = _it.RFFFit()
        rff.W, rff.b, rff.sigma_f = self._d("W"), self._d("b"), float(self.theta[2])
        rff.omega_map, rff.hess_diag = self._dev["omega_MAP"], self._dev["hess_diag"]
        if self.covariance_form == "full":
            if "L" not in self._dev:
                raise ValueError("update_covariancematrix() first")
            rff.L = self._dev["L"]
        PhiT = _it.rff_grid_features(rff.W, rff.b, rff.sigma_f, ops.to_dev(np.asarray(grids, dtype=np.float64)))
        sums, _, _ = _it.rff_acquisition(rff, PhiT, n_samples, ops.to_dev(np.array([float(mustar)])), shard=shard, seed=seed,
                                         covariance=self.covariance_form)
        return sums.cpu().numpy()

    # ------------------------------------------------------------------ batched maximiser (north_star piece 3; SURVEY.md 8f rank 4)
    def return_xstar_batch(self, omegas, n_restarts=16, max_iter=500, gtol=1e-9):
        """maximisers of many sampled functions at once: omegas [S, F] -> (xstars [S, D], values [S]).  Starts per sample (drawn from
        the global RNG, sample by sample): a quarter like return_xstar -- a random GP local maximiser + 0.01 U(0,1) jitter; a quarter
        on the diagonal, (c, ..., c) + jitter with c a random coordinate of a local maximiser (what the reference's return_xstar
        actually starts from: its mu_star leaves xstars_local one-dimensional, src/gp_model.py:425-435, so indexing it yields a
        scalar); the rest uniform in the box.  Every (sample, restart) is one CTA of ppbo_rff_maximize."""
        omegas = np.atleast_2d(np.asarray(omegas, dtype=np.float64))
        S, D = omegas.shape[0], self.D
        n_local = max(1, n_restarts // 4)
        X0 = np.empty((S, n_restarts, D))
        loc = np.atleast_2d(self.GP_xstars_local)
        for s in range(S):
            for r in range(n_restarts):
                if r < n_local:
                    X0[s, r] = np.clip(loc[np.random.randint(loc.shape[0])] + 0.01 * np.random.uniform(0, 1, size=D), 0, 1)
                elif r < 2 * n_local:
                    X0[s, r] = np.clip(loc.ravel()[np.random.randint(loc.size)] + 0.01 * np.random.uniform(0, 1, size=D), 0, 1)
                else:
                    X0[s, r] = np.random.uniform(0, 1, size=D)
        xb, fb = ops.rff_maximize(self._d("W"), self._d("b"), self.theta[2], ops.to_dev(omegas), ops.to_dev(X0), max_iter=max_iter, gtol=gtol)
        return xb.cpu().numpy(), fb.cpu().numpy()

    def sample_xstars(self, n, n_restarts=16):
        """n posterior draws of the maximiser location (batched sample_xstar): omega ~ N(omega_MAP, covariance), x* = argmax phi(x)' omega"""
        return self.return_xstar_batch(self.sample_omegas(n), n_restarts=n_restarts)[0]

    # ------------------------------------------------------------------ maximiser of one sampled function (:143-204)
    def _value_grad(self, omega_dev, x):
        out = ops.rff_value_grad(self._d("W"), self._d("b"), omega_dev, ops.to_dev(np.asarray(x, dtype=np.float64)), self.theta[2])
        out = out.cpu().numpy()
        return out[0], out[1:]

    def return_xstar(self, omega):
        start = time.time()
        min_trials, max_trials = 5, 30
        fval, xstar, i = -1e+10, None, 0
        om = ops.to_dev(np.asarray(omega, dtype=np.float64))

        def neg(x):
            v, g = self._value_grad(om, x)
            return -v, -g
        while xstar is None or i < min_trials:
            if i > max_trials:
                print('Bad omega sample: unable to find f_approx maximizer')
                break
            i += 1
            x_initial = self.GP_xstars_local[np.random.randint(self.GP_xstars_local.shape[0])]
            x_initial = np.clip(x_initial + 0.01 * np.random.uniform(0, 1, size=self.D), 0, 1)
            res = scipy.optimize.minimize(neg, x0=x_initial, method='L-BFGS-B', jac=True, bounds=((0, 1),) * self.D,
                                          options={'disp': False, 'maxiter': 5000})
            cand = res.x
            fval_ = self._value_grad(om, cand)[0]
            if fval_ > fval and np.all((cand >= 0) & (cand <= 1)):
                fval, xstar = fval_, cand
        if self.verbose:
            print('Optimization of f_approx took ' + str(time.time() - start) + ' seconds.')
        return xstar

    def return_xstar_for_dim(self, omega, dim, x_ref):
        start = time.time()
        min_trials, max_trials = 5, 30
        fval, xstar, i = -1e+10, None, 0
        om = ops.to_dev(np.asarray(omega, dtype=np.float64))

        def x(x_dim):
            x_ref[dim - 1] = x_dim[0]
            return x_ref
        while xstar is None or i < min_trials:
            if i > max_trials:
                print('Bad omega sample: unable to find f_approx maximizer')
                break
            i += 1
            x_initial = np.array(self.GP_xstar[dim - 1])
            res = scipy.optimize.minimize(lambda x_dim: -self._value_grad(om, x(x_dim))[0], x0=x_initial, method='Nelder-Mead',
                                          bounds=((0, 1),), options={'disp': False, 'maxiter': 5000})
            cand = x(res.x)
            fval_ = self._value_grad(om, cand)[0]
            if fval_ > fval and np.all((cand >= 0) & (cand <= 1)):
                fval, xstar = fval_, cand
        if self.verbose:
            print('Optimization of f_approx took ' + str(time.time() - start) + ' seconds.')
        return xstar

    def sample_xstar(self):
        xstar = None
        while xstar is None:
            xstar = self.return_xstar(self.sample_omega())
        return xstar

    def sample_xstar_for_dim(self, dim, x_ref):
        xstar = None
        while xstar is None:
            xstar = self.return_xstar_for_dim(self.sample_omega(), dim, x_ref)
        return xstar
