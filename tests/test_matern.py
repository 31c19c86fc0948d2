"""Matern-3/2 and Matern-5/2 covariance functions end to end: FP64 closed-form references (difference form, in this file), the random Fourier basis drawn from their
spectral density (a multivariate Student-t), the tensor-pipe and difference-form covariance kernels in all modes, the incremental
growth, the posterior mean paths, the Laplace fit and the one-GPU iteration at the bench shape.

Bounds of the tensor-pipe covariance: the |x|^2 + |y|^2 - 2 x.y form carries a cancellation error of a few ulp of the squared norms
in r^2.  Near r = 0 the kernel turns it into an error of |dk/d(r^2)| / sf^2 times that: 1/2 for SE, 3/2 for Matern-3/2 and 5/6 for
Matern-5/2.  The SE bound of 1e-12 (max-norm relative) is therefore scaled by 3 and 5/3 for the two Matern kernels."""
from fractions import Fraction
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import load_golden, relerr

MATERN = {"Matern32_kernel": 1.5, "Matern52_kernel": 2.5}
KM_BOUND = {"Matern32_kernel": 3e-12, "Matern52_kernel": 5e-12 / 3}
RFF_F = 1 << 16


# ------------------------------------------------------------------------------------------------ FP64 references (host)
def _scaled_dist(X1, X2, theta):
    """r = |(x - y) / l| in difference form (no cancellation near r = 0); theta[1] scalar or per dimension (ARD)"""
    l = np.asarray(theta[1], dtype=float)
    X1, X2 = np.atleast_2d(np.asarray(X1, dtype=float)), np.atleast_2d(np.asarray(X2, dtype=float))
    r = np.empty((X1.shape[0], X2.shape[0]))
    for i in range(0, X1.shape[0], 256):                     # row blocks: the difference tensor stays small
        diff = (X1[i:i + 256, None, :] - X2[None, :, :]) / l
        r[i:i + 256] = np.sqrt(np.einsum("ijk,ijk->ij", diff, diff))
    return r


def matern32_ref(X1, X2, theta):
    """sf^2 (1 + sqrt3 r) exp(-sqrt3 r)"""
    a = np.sqrt(3.0) * _scaled_dist(X1, X2, theta)
    return theta[2] ** 2 * (1.0 + a) * np.exp(-a)


def matern52_ref(X1, X2, theta):
    """sf^2 (1 + sqrt5 r + 5 r^2 / 3) exp(-sqrt5 r)"""
    r = _scaled_dist(X1, X2, theta)
    a = np.sqrt(5.0) * r
    return theta[2] ** 2 * (1.0 + a + 5.0 * r * r / 3.0) * np.exp(-a)


REFS = {"Matern32_kernel": matern32_ref, "Matern52_kernel": matern52_ref}




# ------------------------------------------------------------------------------------------------ host (no GPU)
@pytest.mark.parametrize("name", sorted(MATERN))
def test_reference_closed_form_equals_bessel_form(name):
    """sf^2 2^(1-nu) / Gamma(nu) (sqrt(2 nu) r)^nu K_nu(sqrt(2 nu) r) at nu = 3/2, 5/2, with ARD length-scales"""
    from scipy.special import gamma, kv
    nu, sf = MATERN[name], 1.3
    rng = np.random.RandomState(0)
    l = np.array([0.2, 0.5, 0.9])
    r = np.concatenate([np.logspace(-6, 0, 40), np.linspace(1.0, 12.0, 60)])
    u = rng.randn(r.size, 3)
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    x = rng.rand(r.size, 3)
    y = x + r[:, None] * l * u
    got = np.array([REFS[name](x[i:i + 1], y[i:i + 1], [0.0, l, sf])[0, 0] for i in range(r.size)])
    z = np.sqrt(2 * nu) * np.linalg.norm((x - y) / l, axis=1)
    ref = sf ** 2 * 2 ** (1 - nu) / gamma(nu) * z ** nu * kv(nu, z)
    assert np.abs(got - ref).max() <= 1e-14 * sf ** 2
    assert np.all(REFS[name](x, x, [0.0, l, sf]).diagonal() == sf ** 2)


def _rff_pairs(D, l, n=64, seed=0):
    """x in [0,1]^D and y = x + r l u (u a random unit vector): scaled distance exactly r, r on 64 values in [0.05, 2.5]"""
    rng = np.random.RandomState(seed)
    r = np.linspace(0.05, 2.5, n)
    x = rng.rand(n, D)
    u = rng.randn(n, D)
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    return x, x + r[:, None] * l * u


def _rff_errors(name, D, l, sf, features):
    """phi(x)' phi(y) - k(x, y) over the pairs, in units of sf^2; features(points) -> F x n"""
    x, y = _rff_pairs(D, l)
    got = np.einsum("fi,fi->i", features(x), features(y))
    k = np.array([REFS[name](x[i:i + 1], y[i:i + 1], [0.0, l, sf])[0, 0] for i in range(len(x))])
    return (got - k) / sf ** 2


def _check_rff_errors(e):
    # the basis of draw_rff_basis: max 0.007-0.010, mean <= 4e-4 (F = 2^16).  A u per entry, the SE basis, the other nu or a basis
    # without the ARD scaling: max 0.05-0.35, mean 0.011-0.10
    assert np.abs(e).max() <= 0.03, np.abs(e).max()
    assert abs(e.mean()) <= 0.006, e.mean()


@pytest.mark.parametrize("D", [6, 20])
@pytest.mark.parametrize("name", sorted(MATERN))
def test_rff_basis_statistics(name, D):
    """E[phi(x)' phi(y)] = k(x, y) for the Matern basis: one Student-t row per feature, ARD length-scales"""
    from oracle import ppbo_oracle as O
    from ppbo_b200.spectral import draw_rff_basis
    l = np.random.RandomState(D).uniform(0.2, 0.8, D)
    sf = 0.8
    W, b = draw_rff_basis(name, RFF_F, D, l, np.random.RandomState(7))
    _check_rff_errors(_rff_errors(name, D, l, sf, lambda P: O.rff_features(W, b, P, sf)))


def _hsampler(kernel_name, D, F, theta):
    from random_fourier_sampler import Hsampler

    def kernel():
        pass
    kernel.__name__ = kernel_name
    gp = SimpleNamespace(D=D, m=3, X=np.zeros((4, D)), xstar=None, xstars_local=None, n_gausshermite_sample_points=200,
                         obs_indices=[0], kernel=kernel, theta=theta)
    return Hsampler(gp, nFeatures=F)


@pytest.mark.parametrize("name", ["SE_kernel", "Matern32_kernel", "Matern52_kernel", "RQ_kernel"])
def test_generate_basis_consumes_global_stream_in_order(name):
    """Hsampler.generate_basis draws from np.random: SE W = randn / l then b; Matern z, u (one per row), then b; RQ b only.  After
    the call the global generator is where the documented draws by hand leave it."""
    D, F = 5, 300
    l = [0.2, 0.3, 0.4, 0.5, 0.6] if name != "RQ_kernel" else 0.3
    h = _hsampler(name, D, F, [0.01, l, 0.7])
    np.random.seed(11)
    h.generate_basis()
    after = np.random.get_state()
    np.random.seed(11)
    if name == "SE_kernel":
        W = np.random.randn(F, D) / l
    elif name in MATERN:
        z = np.random.randn(F, D)
        u = np.random.chisquare(2 * MATERN[name], F)
        W = z / np.asarray(l) * np.sqrt(2 * MATERN[name] / u)[:, None]
    else:
        W = None
    b = np.random.uniform(low=0, high=2 * np.pi, size=F)[:, None]
    ref = np.random.get_state()
    assert after[0] == ref[0] and np.array_equal(after[1], ref[1]) and after[2:] == ref[2:]
    assert np.array_equal(h.b, b)
    if W is None:
        assert h.W is None
    else:
        assert np.array_equal(h.W, W)


# ------------------------------------------------------------------------------------------------ GPU
torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import ops as _ops
    return _ops


def _np(t):
    return t.detach().cpu().numpy()


def _fma_diag(scale, sf2, add):
    return float(Fraction(scale) * Fraction(sf2) + Fraction(add))      # one rounding, as fma(diag_scale, sf^2, diag_add)


@gpu
@pytest.mark.parametrize("ard", [False, True])
@pytest.mark.parametrize("name", sorted(MATERN))
def test_kernel_matrix_vs_reference_and_difference_form(ops, name, ard):
    """tensor-pipe kernels (symmetric with fused shrinkage, store) against the FP64 reference and against the difference-form kernels of
    tuning key 11, on ragged shapes; the symmetric matrix is bit-symmetric with the exact fused diagonal on both paths"""
    from ppbo_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(5)
    sf, s = 0.7, 1e-6
    diag = _fma_diag(1.0 - s, sf * sf, s * sf * sf)
    for n in (1, 63, 64, 65, 127, 128, 129, 700):
        for D in (1, 2, 6, 20, 64):
            ls = rng.uniform(0.2, 0.9, D) if ard else 0.3
            Xh, Yh = rng.rand(n, D), rng.rand(n + 3, D)
            X, Y = ops.to_dev(Xh), ops.to_dev(Yh)
            res = {}
            for key in (1, 0):
                lib.ppbo_set_tuning(11, key)
                try:
                    res[key] = (_np(ops.gram_regularized(name, X, ls, sf, s)), _np(ops.kernel_matrix(name, Y, X, ls, sf)))
                finally:
                    lib.ppbo_set_tuning(11, 0)
            what = (name, ard, n, D)
            Kref = REFS[name](Yh, Xh, [0.0, ls, sf])
            assert relerr(res[0][1], Kref) <= KM_BOUND[name], what
            assert relerr(res[1][1], Kref) <= 1e-13, what                   # difference form: no cancellation
            assert relerr(res[0][1], res[1][1]) <= KM_BOUND[name], what
            assert relerr(res[0][0], res[1][0]) <= KM_BOUND[name], what
            Sref = (1.0 - s) * REFS[name](Xh, Xh, [0.0, ls, sf]) + s * sf * sf * np.eye(n)
            assert relerr(res[0][0], Sref) <= KM_BOUND[name], what
            assert np.array_equal(res[0][0], res[0][0].T), what
            assert np.all(np.diag(res[0][0]) == diag) and np.all(np.diag(res[1][0]) == diag), what


@gpu
@pytest.mark.parametrize("D", [3, 20])
@pytest.mark.parametrize("name", sorted(MATERN))
def test_gram_append_bit_identical(ops, name, D):
    """appended rows / columns of Sigma and of G equal the from-scratch matrices bit for bit, on ragged sizes"""
    rng = np.random.RandomState(D)
    m = 7
    ls = rng.uniform(0.2, 0.6, D)
    for Q_old, Q_new in ((1, 2), (9, 10), (16, 19), (37, 38), (0, 3)):
        n_old, n_new = Q_old * (m + 1), Q_new * (m + 1)
        cap = n_new + 5
        X = ops.to_dev(rng.rand(n_new, D))
        ref = ops.gram_regularized(name, X, ls, 0.7, 1e-6)
        S = torch.full((cap, cap), float("nan"), dtype=torch.float64, device=X.device)
        if n_old:
            ops.gram_regularized(name, X[:n_old], ls, 0.7, 1e-6, out=S[:n_old, :n_old])
        ops.gram_append(name, X, n_old, ls, 0.7, 1e-6, S)
        assert torch.equal(S[:n_new, :n_new], ref)
        assert torch.isnan(S[n_new:]).all() and torch.isnan(S[:, n_new:]).all()
        Gref = ops.diffspace_gram(ref, Q_new, m)
        capM = Q_new * m + 3
        G = torch.full((capM, capM), float("nan"), dtype=torch.float64, device=X.device)
        if Q_old:
            G[:Q_old * m, :Q_old * m].copy_(ops.diffspace_gram(ref[:n_old, :n_old].contiguous(), Q_old, m))
        ops.diffspace_gram_append(S[:n_new, :n_new], Q_old, Q_new, m, G)
        assert torch.equal(G[:Q_new * m, :Q_new * m], Gref)


@gpu
@pytest.mark.parametrize("name", sorted(MATERN))
def test_posterior_mean_paths(ops, name):
    """mat-vec mode (mean without the cross-covariance) against the materialised product, within the SE bound; the one-CTA point
    kernel of the differential evolution (ppbo_mu_pred_points) against the mat-vec mean"""
    rng = np.random.RandomState(9)
    for N, P, D in ((1, 1, 1), (130, 67, 6), (1300, 517, 20), (700, 64, 64)):
        ls = rng.uniform(0.2, 0.8, D)
        X, Y = ops.to_dev(rng.rand(N, D)), ops.to_dev(rng.rand(P, D))
        alpha = rng.randn(N)
        ad = ops.to_dev(alpha)
        K = _np(ops.kernel_matrix(name, Y, X, ls, 0.7))
        ref = K @ alpha
        mu = _np(ops.posterior_mean(name, X, ls, 0.7, ad, Y)).ravel()
        assert np.abs(mu - ref).max() <= 1e-12 * max(np.abs(ref).max(), 1e-300) + 1e-13 * np.abs(alpha).sum(), (N, P, D)
        pts = _np(Y[:min(P, 32)])
        got = ops.mu_pred_points(name, X, ls, 0.7, ad, pts)
        r = mu[:len(pts)]
        assert np.abs(got - r).max() <= 1e-11 * max(np.abs(r).max(), 1e-300) + 1e-13 * np.abs(alpha).sum(), (N, P, D)


@gpu
def test_mu_star_native_equals_scipy_matern52(ops):
    """on a Matern-5/2 GPModel: ppbo_mu_star_de replays scipy's differential evolution bit for bit, np.random state included"""
    from test_src_gpu import _model
    g = load_golden("hartmann6d")
    g["kernel"] = "Matern52_kernel"
    st, gp = _model(g)
    assert gp._kernel_name() == "Matern52_kernel"
    out = {}
    for tag, method, window in (("scipy", "de-scipy", 1), ("w32", "de", 32)):
        gp.mustar_method, gp.mustar_window = method, window
        gp.mu_pred_calls = 0
        np.random.seed(int(g["seed_fit"]) + 1)
        xstar, mustar, local = gp.mu_star(mustar_finding_trials=2)
        out[tag] = (xstar, mustar, local, gp.mu_pred_calls, np.random.get_state())
    a, b = out["scipy"], out["w32"]
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]
    assert a[2].shape == b[2].shape and np.array_equal(a[2], b[2])
    assert a[3] == b[3] and a[3] > 0
    assert a[4][0] == b[4][0] and np.array_equal(a[4][1], b[4][1]) and a[4][2:] == b[4][2:]


@gpu
@pytest.mark.parametrize("name", sorted(MATERN))
def test_laplace_fit_vs_reference(ops, name):
    """N = 1300 (Q = 50, m = 25, D = 10): the device mode equals the oracle's Newton iteration from zero (fmap_tight) to 1e-6"""
    from oracle import ppbo_oracle as O
    from ppbo_b200 import iteration, synthetic
    Q, m, D = 50, 25, 10
    theta = [0.05, 0.4, 0.5]
    Xh, _, _ = synthetic.make_design(D, Q, m, seed=3)
    Sh = O.regularize_covariance(REFS[name](Xh, Xh, theta), svd_roundtrip=False)
    f_ref = O.fmap_tight(Sh, Q, m, theta[0], np.zeros(Xh.shape[0]), iters=100)
    assert np.linalg.norm(f_ref - Sh @ O.lik_beta(f_ref, Q, m, theta[0])) <= 1e-10 * np.linalg.norm(f_ref)
    fit = iteration.gp_fit(ops.to_dev(Xh), name, theta, Q, m, tol=1e-10)
    f = _np(fit.f_map)
    assert np.abs(f - f_ref).max() <= 1e-6 * np.abs(f_ref).max()


@gpu
def test_bench_shape_matern52_iterations(ops):
    """Ackley-20D with the Matern-5/2 kernel through the one-GPU pipeline: a cold iteration at Q = 200 and four appended ones.
    Overlapped and sequential pipelines give the same bits at every step; Sigma and G equal fresh builds; the GP mode solves
    f = Sigma beta(f) to 1e-8 (FP64 on the host); at the last step omega_MAP matches the oracle's weight-space optimum and the
    2048-sample sums match the FP64 contraction of that optimum."""
    from oracle import ppbo_oracle as O
    from oracle.make_full_fixtures import rff_tight
    from ppbo_b200 import iteration as it
    from ppbo_b200 import synthetic
    name, Q0, STEPS, S, seed = "Matern52_kernel", 200, 4, 2048, 0
    prob = synthetic.make_problem("ackley20d", Q=Q0 + STEPS, kernel=name)
    assert prob["kernel"] == name
    theta, m = prob["theta"], prob["m"]
    sigma = theta[0]
    B, P, D = prob["grids"].shape
    dev = torch.device("cuda", torch.cuda.current_device())
    Xh = prob["X"]
    X = ops.to_dev(Xh)
    W, b, grids = ops.to_dev(prob["W"]), ops.to_dev(prob["b"]), ops.to_dev(prob["grids"])
    Sigma_h = O.regularize_covariance(matern52_ref(Xh, Xh, theta), svd_roundtrip=False)

    def run(overlap, checks):
        saved = it.OVERLAP_SAMPLING
        out = []
        try:
            it.OVERLAP_SAMPLING = overlap
            state = it.IterationState(name, theta, D, m, Q0 + STEPS, dev, W, b)
            for k in range(STEPS + 1):
                Q = Q0 + k
                if k == 0:
                    d = {"X": X[:Q0 * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids}
                else:
                    d = {"block": X[(Q - 1) * (m + 1):Q * (m + 1)].contiguous(), "W": W, "b": b, "grids": grids}
                sums, gp, rff = it.run_iteration(d, name, theta, Q, m, S, seed=seed, state=state)
                torch.cuda.synchronize()
                out.append((sums.clone(), gp.f_map.clone(), rff.omega_map.clone()))
                if checks:
                    N, M = Q * (m + 1), Q * m
                    fresh = ops.gram_regularized(name, X[:N].contiguous(), theta[1], theta[2], it.SHRINKAGE)
                    assert torch.equal(gp.Sigma, fresh), Q
                    assert torch.equal(gp.lap.G[:M, :M], ops.diffspace_gram(fresh, Q, m)), Q
                    assert relerr(_np(gp.Sigma), Sigma_h[:N, :N]) <= KM_BOUND[name], Q
                    f = _np(gp.f_map)
                    res = f - Sigma_h[:N, :N] @ O.lik_beta(f, Q, m, sigma)
                    assert np.linalg.norm(res) <= 1e-8 * np.linalg.norm(f), (Q, np.linalg.norm(res) / np.linalg.norm(f))
        finally:
            it.OVERLAP_SAMPLING = saved
        return out

    seq = run(True, True)
    plain = run(False, False)
    for k, (a, b_) in enumerate(zip(seq, plain)):
        for x, y, what in zip(a, b_, ("sums", "f_map", "omega_map")):
            assert torch.equal(x, y), "overlapped and sequential pipelines differ in %s at Q = %d" % (what, Q0 + k)
    Q = Q0 + STEPS
    N = Q * (m + 1)
    PhiX = O.rff_features(prob["W"], prob["b"], Xh[:N], theta[2])
    w_te, _ = O.rff_omega_map(PhiX, Q, m, sigma, np.zeros(prob["F"]))
    w_ref = rff_tight(PhiX, Q, m, sigma, w_te)
    w = _np(seq[-1][2])
    assert np.abs(w - w_ref).max() <= 1e-6 * np.abs(w_ref).max()
    f_last = _np(seq[-1][1])
    hd = O.rff_S_hess_diag(w_ref, PhiX, Q, m, sigma)
    Z = O.philox_normals(seed, 0, 0, S * prob["F"]).reshape(S, prob["F"])
    Omega = ops.to_dev(O.rff_sample_omega(w_ref, hd, Z))
    beta = O.lik_beta(f_last, Q, m, sigma)
    mustar = f_last.max()
    fmax = []
    for g in prob["grids"]:
        mustar = max(mustar, float((matern52_ref(Xh[:N], g, theta).T @ beta).max()))
        fmax.append((Omega @ ops.to_dev(O.rff_features(prob["W"], prob["b"], g, theta[2]))).max(dim=1).values)
    fmax = torch.stack(fmax)
    ref_sums = _np(torch.stack([(fmax - mustar).clamp(min=0).sum(dim=1), fmax.sum(dim=1), (fmax * fmax).sum(dim=1)], dim=1))
    got = _np(seq[-1][0])
    scale = float(fmax.abs().max().item())
    for c in range(3):
        assert np.abs(got[:, c] - ref_sums[:, c]).max() <= 1e-6 * max(np.abs(ref_sums[:, c]).max(), S * 1e-3 * scale), c
    ei, _ = it.acquisition_values(got, S)
    ei_ref = ref_sums[:, 0] / S
    assert int(np.argmax(ei)) == int(np.argmax(ei_ref))


@gpu
@pytest.mark.parametrize("name", sorted(MATERN))
def test_device_rff_features_statistics(ops, name):
    """ops.rff_features (the feature kernel of the weight-space fit and the sampling) with a Matern basis: same bound as on the host.
    Point-major output, the layout of the sampling contraction's grid operand (the feature-major launch puts F on grid.y)."""
    from ppbo_b200.spectral import draw_rff_basis
    D, sf = 20, 0.8
    l = np.random.RandomState(D).uniform(0.2, 0.8, D)
    W, b = draw_rff_basis(name, RFF_F, D, l, np.random.RandomState(7))
    Wd, bd = ops.to_dev(W), ops.to_dev(b)
    e = _rff_errors(name, D, l, sf, lambda P: _np(ops.rff_features(Wd, bd, ops.to_dev(P), sf, feature_major=False)).T)
    _check_rff_errors(e)
