"""Synthetic PPBO problems of the BASELINE.json shapes (SURVEY.md 8, table of configs and 8d "Synthetic inputs").

Everything is generated on the host with a private numpy RandomState (never the global legacy RNG, which belongs to the
caller as in the reference).  The design matrix is produced already scaled to [0,1]^D, in the layout
FeedbackProcessing.create_X builds (src/feedback_processing.py:110-130): one block of m+1 rows per query, the chosen
point first, then the m pseudo-observations alpha_k xi + x on a jittered equispaced alpha grid (:66-74).
"""
import numpy as np

from .spectral import draw_rff_basis

# name: D, Q, m, kernel, theta=[sigma, l, sigma_f], S (MC samples), P (grid points per direction), F (RFF features)
CONFIGS = {
    "camel2d": dict(D=2, Q=39, m=25, kernel="SE_kernel", theta=[0.01, 0.26, 0.1], S=150, P=70, F=1000),
    "hartmann6d": dict(D=6, Q=41, m=25, kernel="SE_kernel", theta=[0.001, 0.26, 0.1], S=150, P=70, F=1000),
    "camphor6d": dict(D=6, Q=20, m=25, kernel="camphor_copper_kernel", theta=[0.001, 0.26, 0.1], S=150, P=70, F=0),
    "levy10d": dict(D=10, Q=80, m=25, kernel="SE_kernel", theta=[0.001, 0.4, 0.15], S=4096, P=1024, F=1000),
    "ackley20d": dict(D=20, Q=200, m=25, kernel="SE_kernel", theta=[0.09, 0.3, 0.5], S=32768, P=1024, F=1000),
}


def jittered_alphas(rng, n, lo=0.0, hi=1.0, noise=0.01):
    """jittered linspace of src/feedback_processing.py:66-74 (retry until n distinct values)"""
    eps_b = (hi - lo) * (noise / 2)
    eps_n = abs(hi - lo) * noise
    while True:
        a = np.unique(np.clip(np.linspace(lo + eps_b, hi - eps_b, n) + rng.normal(0, eps_n, n), lo, hi))
        if len(a) == n:
            return a


def utility(points, centre):
    """smooth synthetic utility on [0,1]^D with its maximum at `centre`"""
    return -np.sum((points - centre) ** 2, axis=-1)


def make_design(D, Q, m, seed=0, answer_noise=1e-3):
    """X [Q(m+1) x D] in [0,1]^D plus the query log (xi, x, alpha*) it came from."""
    rng = np.random.RandomState(seed)
    centre = rng.uniform(0.25, 0.75, D)
    X = np.empty((Q * (m + 1), D))
    log = []
    for q in range(Q):
        xi = np.zeros(D)
        if q < D or q % 3:
            xi[q % D] = 1.0                                   # coordinate queries (ppbo_numerical_main.py:136,152,165,177)
        else:                                                 # some genuinely projective ones
            dims = rng.choice(D, size=min(D, 2), replace=False)
            xi[dims] = rng.uniform(0.3, 1.0, len(dims))
            xi /= xi.max()
        x = rng.uniform(0, 1, D)
        x[xi != 0] = 0
        fine = np.linspace(0, 1, 401)
        a_star = fine[np.argmax(utility(fine[:, None] * xi + x, centre))] + answer_noise * rng.randn()
        a_star = float(np.clip(a_star, 0, 1))
        alphas = jittered_alphas(rng, m)
        blk = X[q * (m + 1):(q + 1) * (m + 1)]
        blk[0] = a_star * xi + x
        blk[1:] = alphas[:, None] * xi + x
        log.append((xi, x, a_star))
    return np.clip(X, 0, 1), log, centre


def make_problem(name, seed=0, Q=None, S=None, P=None, F=None, kernel=None):
    """All host inputs of one iteration for config `name` (sizes overridable for small parity cases).  `kernel` overrides the
    config's covariance function; the RFF basis is then drawn from that kernel's spectral density (draw_rff_basis).  The design,
    the grids and, for the configs' own kernels, every draw are the same as without the override."""
    cfg = dict(CONFIGS[name])
    for k, v in (("Q", Q), ("S", S), ("P", P), ("F", F), ("kernel", kernel)):
        if v is not None:
            cfg[k] = v
    D, Qn, m = cfg["D"], cfg["Q"], cfg["m"]
    X, log, centre = make_design(D, Qn, m, seed)
    rng = np.random.RandomState(seed + 1)
    N = Qn * (m + 1)
    prob = dict(cfg, name=name, N=N, X=X, centre=centre, f_init=np.zeros(N))
    # query directions of EId_xstar (src/acquisition.py:132-145): e_d with x = incumbent, coordinate d zeroed
    inc = np.clip(centre + 0.05 * rng.randn(D), 0, 1)
    xis = np.eye(D)
    xs = np.tile(inc, (D, 1))
    xs[np.arange(D), np.arange(D)] = 0.0
    alphas = np.stack([jittered_alphas(rng, cfg["P"]) for _ in range(D)])
    prob.update(xis=xis, xs=xs, alphas=alphas, grids=alphas[:, :, None] * xis[:, None, :] + xs[:, None, :])
    if cfg["F"]:
        W, b = draw_rff_basis(cfg["kernel"], cfg["F"], D, cfg["theta"][1], rng)       # src/random_fourier_sampler.py:42-43
        if W is None:
            raise ValueError("random Fourier basis exists for the SE, Matern and camphor kernels only, not %s (use F=0)" % cfg["kernel"])
        prob["W"], prob["b"] = W, b
        prob["omega0"] = np.zeros(cfg["F"])
    return prob
