"""GPU tests of the incremental-growth entry points (SURVEY.md 8f rank 2: one (m+1)-row block is appended per PPBO iteration,
src/feedback_processing.py:133-154) and of the linear algebra added for the evidence (LU log-determinant) and for mu_star
(single-point posterior mean)."""
import numpy as np
import pytest

from conftest import relerr

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from ppbo_b200 import ops as _ops
    return _ops


def _np(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize("kernel,D", [("SE_kernel", 20), ("SE_kernel", 3), ("RQ_kernel", 5), ("camphor_copper_kernel", 6)])
def test_gram_append_bit_identical(ops, kernel, D):
    """appended rows / columns of Sigma and of G = B' Sigma B equal the from-scratch matrices bit for bit, on ragged sizes"""
    rng = np.random.RandomState(0)
    m = 7
    for Q_old, Q_new in ((1, 2), (9, 10), (16, 19), (37, 38), (0, 3)):
        n_old, n_new = Q_old * (m + 1), Q_new * (m + 1)
        cap = n_new + 5                                       # leading dimension larger than the matrix
        X = ops.to_dev(rng.rand(n_new, D))
        ref = ops.gram_regularized(kernel, X, 0.3, 0.7, 1e-6)
        S = torch.full((cap, cap), float("nan"), dtype=torch.float64, device=X.device)
        if n_old:
            ops.gram_regularized(kernel, X[:n_old], 0.3, 0.7, 1e-6, out=S[:n_old, :n_old])
            assert torch.equal(S[:n_old, :n_old], ref[:n_old, :n_old])           # the old matrix is the leading block
        ops.gram_append(kernel, X, n_old, 0.3, 0.7, 1e-6, S)
        assert torch.equal(S[:n_new, :n_new], ref)
        assert torch.isnan(S[n_new:]).all() and torch.isnan(S[:, n_new:]).all()   # nothing outside the matrix is written
        Gref = ops.diffspace_gram(ref, Q_new, m)
        capM = Q_new * m + 3
        G = torch.full((capM, capM), float("nan"), dtype=torch.float64, device=X.device)
        if Q_old:
            G[:Q_old * m, :Q_old * m].copy_(ops.diffspace_gram(ref[:n_old, :n_old].contiguous(), Q_old, m))
        ops.diffspace_gram_append(S[:n_new, :n_new], Q_old, Q_new, m, G)
        assert torch.equal(G[:Q_new * m, :Q_new * m], Gref)
        assert torch.isnan(G[Q_new * m:]).all()


@pytest.mark.parametrize("M_old,M_new", [(100, 125), (128, 153), (250, 275), (1000, 1025), (1270, 1295), (1279, 1281)])
def test_factor_extend(ops, M_old, M_new):
    """chol(I + s G s) grown from M_old to M_new rows equals (in the residual sense) the factor of the grown system"""
    from ppbo_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(M_old)
    cap = M_new + 11
    Z = rng.randn(M_new, 40)
    Gh = Z @ Z.T / 40 + 0.1 * np.eye(M_new)
    sa = np.sqrt(rng.rand(M_new) * (rng.rand(M_new) > 0.1))                # some exact zeros
    A = np.eye(M_new) + sa[:, None] * Gh * sa[None, :]
    fit = ops.LaplaceFit()
    fit.cap = fit.ldg = cap
    fit.Q, fit.m, fit.sigma, fit.info, fit.factor_state = M_new, 1, 1.0, 0, 1
    dev = ops.device()
    fit.G = torch.zeros((cap, cap), dtype=torch.float64, device=dev)
    fit.G[:M_new, :M_new].copy_(ops.to_dev(Gh))
    fit._Lfac = torch.zeros(lib.ppbo_factor_doubles(cap), dtype=torch.float64, device=dev)
    fit.sa_fac = torch.zeros(cap, dtype=torch.float64, device=dev)
    fit.sa_fac[:M_new].copy_(ops.to_dev(sa))
    # factor of the leading M_old system, written into the capacity buffer
    L = fit._Lfac[:cap * cap].view(cap, cap)
    Aold = ops.to_dev(A[:M_old, :M_old])
    info, ws = ops.potrf_lower(Aold)
    assert info == 0
    L[:M_old, :M_old].copy_(Aold)
    nb = (M_old + 127) // 128
    fit._Lfac[cap * cap:cap * cap + nb * 128 * 128].copy_(ws[:nb * 128 * 128])
    assert ops.factor_extend(fit, M_old, M_new) == 0
    Lh = np.tril(_np(L[:M_new, :M_new]))
    assert np.abs(Lh @ Lh.T - A).max() <= 1e-12 * np.abs(A).max() * np.sqrt(M_new)
    # and the grown factor object solves: (L L') x = b through the blocked kernels (uses the rebuilt inverted diagonal blocks)
    b = rng.randn(M_new)
    x = torch.zeros(M_new + 128, dtype=torch.float64, device=dev)
    x[:M_new].copy_(ops.to_dev(b))
    from ppbo_b200._lib import check
    check(lib.ppbo_potrs_vec(L.data_ptr(), cap, M_new, x.data_ptr(), fit._Lfac[cap * cap:].data_ptr(),
                             lib.ppbo_potrf_workspace_bytes(M_new), torch.cuda.current_stream().cuda_stream), "potrs")
    assert relerr(_np(x[:M_new]), np.linalg.solve(A, b)) < 1e-10


def test_state_append_equals_cold_fit(ops, golden):
    """GPState: cold fit on Q - 2 comparison sets, two appends -> same mode, same prediction as the from-scratch fit"""
    from ppbo_b200 import iteration
    g = golden
    Q, m, theta = g["Q"], g["m"], g["theta"]
    X = ops.to_dev(g["X"])
    cold = iteration.gp_fit(X, g["kernel"], theta, Q, m, tol=1e-10)
    st = iteration.GPState(g["kernel"], theta, g["D"], m, Q + 1, X.device, tol=1e-10)
    n2 = (Q - 2) * (m + 1)
    st.cold(X[:n2])
    st.append(X[n2:n2 + m + 1])
    st.append(X[n2 + m + 1:])
    assert torch.equal(st.Sigma, cold.Sigma)
    f, f_ref = _np(st.f_map), _np(cold.f_map)
    assert np.abs(f - f_ref).max() <= 1e-7 * np.abs(f_ref).max()
    assert st.lap.stats["converged"] == 1
    P = g["pred_grid"].shape[0]
    Xp = ops.to_dev(g["pred_grid"])
    mu0, Sp0 = ops.predict(g["kernel"], X, theta[1], theta[2], 1e-6, cold.lap, Xp, P, 1)
    mu1, Sp1 = ops.predict(g["kernel"], st.X, theta[1], theta[2], 1e-6, st.lap, Xp, P, 1)
    assert relerr(_np(mu1), _np(mu0)) < 1e-6
    assert np.abs(_np(Sp1) - _np(Sp0)).max() <= 1e-6 * theta[2] ** 2


def test_lazy_mode_factor(ops, golden):
    """a fit without the factor at the mode gives the same prediction as one with it (built on first use)"""
    g = golden
    Q, m, theta = g["Q"], g["m"], g["theta"]
    X, Sigma = ops.to_dev(g["X"]), ops.to_dev(g["Sigma"])
    a = ops.laplace_fit(Sigma, Q, m, theta[0], factor_at_mode=True)
    b = ops.laplace_fit(Sigma, Q, m, theta[0], factor_at_mode=False)
    assert a.factor_state == 2 and b.factor_state in (0, 1)
    assert a.stats["factorizations"] == b.stats["factorizations"] + 1
    P = g["pred_grid"].shape[0]
    Xp = ops.to_dev(g["pred_grid"])
    _, Sa = ops.predict(g["kernel"], X, theta[1], theta[2], 1e-6, a, Xp, P, 1)
    _, Sb = ops.predict(g["kernel"], X, theta[1], theta[2], 1e-6, b, Xp, P, 1)
    assert b.factor_state == 2
    assert np.abs(_np(Sa) - _np(Sb)).max() <= 1e-12 * theta[2] ** 2


@pytest.mark.parametrize("n", [1, 5, 64, 65, 200, 777])
def test_lu_logdet(ops, n):
    rng = np.random.RandomState(n)
    A = rng.randn(n, n)
    if n > 3:
        A[2] *= -3.0
    sign_u, logabs, sign_p, info = ops.lu_logdet(ops.to_dev(A).clone())
    s_ref, l_ref = np.linalg.slogdet(A)
    assert info == 0
    assert sign_u * sign_p == s_ref
    assert abs(logabs - l_ref) <= 1e-10 * max(1.0, abs(l_ref))
    import scipy.linalg
    P, L, U = scipy.linalg.lu(A)
    assert sign_u == np.sign(np.prod(np.sign(np.diag(U))))               # same pivoting rule as LAPACK: same split of the sign


def test_evidence_terms_match_reference(ops, golden):
    """GPModel.evidence (src/gp_model.py:278-319): log|det(I + Sigma Lambda)| and its sign at the mode the reference's own run found,
    and the value the reference returned (recorded by oracle/make_golden.py)"""
    import scipy.stats
    from test_src_gpu import _model
    g = golden
    if "evidence_value" not in g:
        pytest.skip("golden file predates the evidence recording")
    st, gp = _model(g)
    for k, th in enumerate(g["evidence_theta"]):
        th = [float(t) for t in th]
        T_map, sign_u, logabs, sign_p, info = gp._evidence_terms(th, f=g["evidence_fmap"][k])
        assert info == 0
        assert abs(T_map - g["evidence_T"][k]) <= 1e-6 * max(1.0, abs(g["evidence_T"][k]))
        assert sign_u * sign_p == g["evidence_det_sign"][k]
        assert abs(logabs - g["evidence_logabsdet"][k]) <= 1e-6 * max(1.0, abs(g["evidence_logabsdet"][k]))
        lp = (np.log(scipy.stats.lognorm.pdf(th[0], s=1, scale=np.exp(1))) + np.log(scipy.stats.lognorm.pdf(th[1], s=0.5, scale=np.exp(-1.4))) +
              np.log(scipy.stats.lognorm.pdf(th[2], s=0.5, scale=np.exp(1.7))))
        # the reference's value = T - 1/2 sign(U) log|det| + log prior: either sign of U reproduces it or the pivot order differed
        cand = [T_map - 0.5 * s * logabs + lp for s in (sign_u, -sign_u)]
        assert abs(cand[0] - g["evidence_value"][k]) <= 1e-5 * abs(g["evidence_value"][k]), (cand, g["evidence_value"][k])
    # end to end from our own deterministic start: finite, no -500 sentinel on a problem with negative curvature coefficients
    np.random.seed(3)
    v = gp.evidence([float(t) for t in g["evidence_theta"][0]], None)
    assert v != -500 and np.isfinite(v)
    gp.evidence_formula = "laplace"
    v2 = gp.evidence([float(t) for t in g["evidence_theta"][0]], None)
    assert v2 != -500 and np.isfinite(v2)


def test_mu_pred_point(ops, golden):
    """single-point posterior mean with host-resident argument / result against the batched device prediction"""
    g = golden
    Q, m, theta = g["Q"], g["m"], g["theta"]
    X = ops.to_dev(g["X"])
    fit = ops.laplace_fit(ops.to_dev(g["Sigma"]), Q, m, theta[0])
    pm = ops.PointMean(g["kernel"], X, theta[1], theta[2], fit.alpha)
    pts = np.vstack([g["pred_grid"][:5], g["xstar"][None]])
    ref = _np(ops.posterior_mean(g["kernel"], X, theta[1], theta[2], fit.alpha, ops.to_dev(pts)))
    got = np.array([pm(x) for x in pts])
    assert np.abs(got - ref).max() <= 1e-11 * max(np.abs(ref).max(), 1e-300) + 1e-13 * float(fit.alpha.abs().sum())
    assert pm.calls == len(pts)

